// Python module `CUDA_BACKEND`: the thin shim between DeepFlows' Python host code and the C ABI of
// libdfb200.so (include/dfb200.h). It is importable at the dotted path the reference hard-codes,
//   DeepFlows.backend.backend_src.build.Release.CUDA_BACKEND
//   (reference: DeepFlows/backend/backend_tensor.py:57),
// exports the same class/function names with the same argument order as the reference module
//   (reference: DeepFlows/backend/backend_src/ndarray_backend_cuda.cu:515-716),
// and adds the fused L1 entry points. No computation happens here: every function unpacks its
// arguments, calls one dfb_* function and maps the status to the Python exception class pybind
// would have produced for the reference's C++ exception.
#include <pybind11/numpy.h>
#include <pybind11/pybind11.h>
#include <pybind11/stl.h>

#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "../../include/dfb200.h"

namespace py = pybind11;

namespace {

void check(dfb_status st) {
  if (st == DFB_OK) return;
  std::string msg = dfb_last_error();
  switch (st) {
    case DFB_ERR_INVALID:
    case DFB_ERR_DOMAIN:
      throw py::value_error(msg);
    case DFB_ERR_OUT_OF_RANGE:
      throw py::index_error(msg);
    case DFB_ERR_NOMEM:
      PyErr_SetString(PyExc_MemoryError, msg.c_str());
      throw py::error_already_set();
    default:
      throw std::runtime_error(msg);
  }
}

// Owning 1-D float32 device buffer (reference: CudaArray, ndarray_backend_cuda.cu:48-83).
struct Array {
  float* ptr = nullptr;
  size_t size = 0;
  bool owned = true;   // false: a window on memory the library owns (the peer-memory gradient arena)
  explicit Array(size_t n) : size(n) { check(dfb_malloc(n, &ptr)); }
  Array(float* p, size_t n) : ptr(p), size(n), owned(false) {}
  Array(const Array&) = delete;
  Array& operator=(const Array&) = delete;
  ~Array() {
    if (ptr && owned) dfb_free(ptr);
  }
};

// A tensor argument is an Array, an (Array, element_offset) tuple, or None.
float* dptr(const py::handle& h) {
  if (h.is_none()) return nullptr;
  if (py::isinstance<Array>(h)) return h.cast<Array&>().ptr;
  if (py::isinstance<py::tuple>(h)) {
    py::tuple t = py::reinterpret_borrow<py::tuple>(h);
    if (t.size() == 2) return t[0].cast<Array&>().ptr + t[1].cast<long long>();
  }
  throw py::type_error("expected CUDA_BACKEND.Array, (Array, offset) or None");
}
Array& arr(const py::handle& h, const char* what) {
  if (h.is_none() || !py::isinstance<Array>(h)) throw py::value_error(std::string(what) + ": array cannot be null");
  return h.cast<Array&>();
}

struct View {
  int ndim;
  int32_t shape[DFB_MAX_DIMS];
  int32_t strides[DFB_MAX_DIMS];
};
View parse_view(const py::sequence& shape, const py::sequence& strides) {
  size_t n = py::len(shape);
  if (n > DFB_MAX_DIMS || py::len(strides) != n)
    throw py::value_error("CUDA dimension limit exceeded: max supported dimensions = " + std::to_string(DFB_MAX_DIMS) +
                          ", requested = " + std::to_string(n));
  View v;
  v.ndim = (int)n;
  for (size_t i = 0; i < n; ++i) {
    v.shape[i] = (int32_t)py::cast<long long>(shape[i]);
    v.strides[i] = (int32_t)py::cast<long long>(strides[i]);
  }
  return v;
}

int g_matmul_mode = DFB_MODE_FP32;

using BinFn = dfb_status (*)(const float*, const float*, float*, size_t);
using ScaFn = dfb_status (*)(const float*, float, float*, size_t);
using UnaFn = dfb_status (*)(const float*, float*, size_t);

template <BinFn F>
void ewise_binary(const py::object& a, const py::object& b, const py::object& out) {
  Array& A = arr(a, "a");
  Array& B = arr(b, "b");
  Array& O = arr(out, "out");
  if (A.size != B.size || A.size != O.size) throw py::value_error("Input arrays must have the same size");
  check(F(A.ptr, B.ptr, O.ptr, O.size));
}
template <ScaFn F>
void ewise_scalar(const py::object& a, float v, const py::object& out) {
  Array& A = arr(a, "a");
  Array& O = arr(out, "out");
  if (A.size != O.size) throw py::value_error("Input and output arrays must have the same size");
  check(F(A.ptr, v, O.ptr, O.size));
}
template <UnaFn F>
void ewise_unary(const py::object& a, const py::object& out) {
  Array& A = arr(a, "a");
  Array& O = arr(out, "out");
  if (A.size != O.size) throw py::value_error("Input and output arrays must have the same size");
  check(F(A.ptr, O.ptr, O.size));
}

// Int32Vector / SizeTVector: the two helper containers the reference module exports for shapes and strides
// (ndarray_backend_cuda.cu:526-556: default constructor, push_back, size(), indexing with negative indices, clear).
// backend_tensor.py passes tuples, so they are only here for scripts that build the containers by hand; every entry
// point that takes a shape accepts them because they are Python sequences.
template <typename T>
struct PyVector {
  std::vector<T> items;
};
template <typename T>
void bind_vector(py::module_& m, const char* name, const char* doc) {
  py::class_<PyVector<T>>(m, name, doc)
      .def(py::init<>())
      .def("push_back", [](PyVector<T>& v, T value) { v.items.push_back(value); }, py::arg("value"))
      .def("size", [](const PyVector<T>& v) { return v.items.size(); })
      .def("__len__", [](const PyVector<T>& v) { return v.items.size(); })
      .def("__getitem__",
           [name](const PyVector<T>& v, long long i) {
             const long long n = (long long)v.items.size();
             if (i < 0) i += n;
             if (i < 0 || i >= n) throw py::index_error(std::string(name) + " index out of range: " + std::to_string(i));
             return v.items[(size_t)i];
           },
           py::arg("index"))
      .def("clear", [](PyVector<T>& v) { v.items.clear(); });
}

}  // namespace

PYBIND11_MODULE(CUDA_BACKEND, m) {
  m.doc() = "DeepFlows CUDA backend for NVIDIA B200 (sm_100a), C ABI: libdfb200.so";
  m.attr("__version__") = dfb_version();
  m.attr("__device__name__") = "cuda";
  m.attr("__tile_size__") = 128;
  m.attr("__max_dimensions__") = DFB_MAX_DIMS;
  m.attr("MODE_FP32") = (int)DFB_MODE_FP32;
  m.attr("MODE_TF32") = (int)DFB_MODE_TF32;
  m.attr("MODE_BF16") = (int)DFB_MODE_BF16;
  m.attr("MODE_SIMT") = (int)DFB_MODE_SIMT;
  m.attr("LAYOUT_NCHW") = (int)DFB_LAYOUT_NCHW;
  m.attr("LAYOUT_NHWC") = (int)DFB_LAYOUT_NHWC;
  m.attr("WLAYOUT_KCRS") = (int)DFB_WLAYOUT_KCRS;
  m.attr("WLAYOUT_KRSC") = (int)DFB_WLAYOUT_KRSC;
  m.attr("DGRAD_REFERENCE") = (int)DFB_DGRAD_REFERENCE;
  m.attr("DGRAD_EXACT") = (int)DFB_DGRAD_EXACT;
  m.attr("UPSAMPLE_NEAREST") = (int)DFB_UPSAMPLE_NEAREST;
  m.attr("UPSAMPLE_BILINEAR") = (int)DFB_UPSAMPLE_BILINEAR;

  bind_vector<int32_t>(m, "Int32Vector", "Vector of int32 (shape / stride arguments)");
  bind_vector<size_t>(m, "SizeTVector", "Vector of size_t (numpy shape / stride arguments)");

  py::class_<Array>(m, "Array")
      .def(py::init<size_t>(), py::return_value_policy::take_ownership)
      .def_readonly("size", &Array::size)
      .def("ptr", [](const Array& a) { return (size_t)a.ptr; })
      .def("__repr__", [](const Array& a) {
        return "<CUDA_BACKEND.Array size=" + std::to_string(a.size) + " ptr=" + std::to_string((size_t)a.ptr) + ">";
      });

  // ---- runtime ------------------------------------------------------------------------------
  m.def("set_device", [](int d) { check(dfb_set_device(d)); });
  m.def("get_device", []() { int d = 0; check(dfb_get_device(&d)); return d; });
  m.def("device_count", []() { int n = 0; dfb_device_count(&n); return n; });
  m.def("device_info", []() {
    char name[256];
    int sms = 0, maj = 0, min = 0;
    size_t mem = 0;
    check(dfb_device_info(name, sizeof(name), &sms, &maj, &min, &mem));
    py::dict d;
    d["name"] = std::string(name);
    d["sm_count"] = sms;
    d["cc"] = py::make_tuple(maj, min);
    d["total_mem"] = mem;
    return d;
  });
  m.def("synchronize", []() { py::gil_scoped_release nogil; check(dfb_synchronize()); });
  m.def("empty_cache", []() { check(dfb_empty_cache()); });
  m.def("mem_stats", []() {
    size_t a = 0, b = 0, c = 0;
    check(dfb_mem_stats(&a, &b, &c));
    return py::make_tuple(a, b, c);
  });
  m.def("launch_count", []() { return (unsigned long long)dfb_launch_count(); });
  m.def("tc_launch_count", []() { return (unsigned long long)dfb_tc_launch_count(); });
  // step timeline (dfb_trace_*): trace_end() -> (records as an (n, 2) uint64 array, host launch lines)
  m.def("trace_begin", [](size_t capacity) { check(dfb_trace_begin(capacity)); });
  m.def("trace_reset", []() { check(dfb_trace_reset()); });
  m.def("trace_end", [](size_t capacity) {
    py::array_t<unsigned long long> rec({(py::ssize_t)capacity, (py::ssize_t)2});
    size_t n = 0;
    check(dfb_trace_end(rec.mutable_data(), capacity, &n));
    py::list lines;
    for (size_t i = 0; i < dfb_trace_host_count(); ++i) lines.append(py::str(dfb_trace_host_line(i)));
    return py::make_tuple(rec, n, lines);
  });
  m.def("set_matmul_mode", [](int mode) { g_matmul_mode = mode; });
  m.def("get_matmul_mode", []() { return g_matmul_mode; });
  m.def("event_create", []() { void* e = nullptr; check(dfb_event_create(&e)); return (size_t)e; });
  m.def("event_destroy", [](size_t e) { check(dfb_event_destroy((void*)e)); });
  m.def("event_record", [](size_t e) { check(dfb_event_record((void*)e)); });
  m.def("event_synchronize", [](size_t e) { py::gil_scoped_release nogil; check(dfb_event_synchronize((void*)e)); });
  m.def("event_elapsed_ms", [](size_t a, size_t b) { float ms = 0; check(dfb_event_elapsed_ms((void*)a, (void*)b, &ms)); return ms; });
  m.def("side_begin", []() { check(dfb_side_begin()); });
  m.def("side_end", []() { check(dfb_side_end()); });
  m.def("side_join", []() { check(dfb_side_join()); });
  m.def("side_join_lag", [](int lag) { check(dfb_side_join_lag(lag)); });
  m.def("graph_begin_capture", []() { check(dfb_graph_begin_capture()); });
  m.def("graph_end_capture", []() { void* g = nullptr; check(dfb_graph_end_capture(&g)); return (size_t)g; });
  m.def("graph_launch", [](size_t g) { check(dfb_graph_launch((void*)g)); });
  m.def("graph_destroy", [](size_t g) { check(dfb_graph_destroy((void*)g)); });
  m.def("graph_node_counts", [](size_t g) {
    int k = 0, n = 0;
    check(dfb_graph_node_counts((void*)g, &k, &n));
    return py::make_tuple(k, n);
  });
  m.def("graph_capturing", []() { int c = 0; check(dfb_graph_capturing(&c)); return c != 0; });
  m.def("graph_set_adam", [](size_t g, int index, double lr, double b1, double b2, double eps, double wd, int t, double gs) {
    check(dfb_graph_set_adam((void*)g, index, lr, b1, b2, eps, wd, t, gs));
  });
  m.def("graph_set_sgd", [](size_t g, int index, double lr, double mom, double wd, bool nesterov, double gs) {
    check(dfb_graph_set_sgd((void*)g, index, lr, mom, wd, nesterov ? 1 : 0, gs));
  });

  // ---- L0: the reference protocol -------------------------------------------------------------
  m.def("fill", [](const py::object& out, float v) {
    Array& O = arr(out, "Fill: out");
    check(dfb_fill(O.ptr, v, O.size));
  });
  m.def("from_numpy", [](py::array_t<float, py::array::c_style | py::array::forcecast> a, const py::object& out) {
    Array& O = arr(out, "from_numpy: out");
    if ((size_t)a.size() != O.size) throw py::value_error("Input numpy array size does not match output CudaArray size");
    check(dfb_from_host(a.data(), O.ptr, O.size));
  });
  m.def("to_numpy", [](const py::object& a, const py::sequence& shape, const py::sequence& strides, size_t offset) {
    Array& A = arr(a, "to_numpy: a");
    size_t n = py::len(shape);
    std::vector<py::ssize_t> sh(n), st(n);
    size_t extent = 0, count = 1;
    for (size_t i = 0; i < n; ++i) {
      long long s = py::cast<long long>(shape[i]), t = py::cast<long long>(strides[i]);
      if (s < 0 || t < 0) throw py::value_error("to_numpy: negative shape/stride");
      sh[i] = (py::ssize_t)s;
      st[i] = (py::ssize_t)(t * (long long)sizeof(float));
      count *= (size_t)s;
      if (s > 0) extent += (size_t)(s - 1) * (size_t)t;
    }
    if (count == 0) return py::array_t<float>(sh);
    if (offset + extent >= A.size + (A.size == 0)) throw py::index_error("to_numpy: view exceeds the array");
    // copy only the touched range [offset, offset + extent], then expose the strided view
    py::array_t<float> base((py::ssize_t)(extent + 1));
    check(dfb_to_host(A.ptr + offset, base.mutable_data(), extent + 1));
    return py::array_t<float>(sh, st, base.data(), base);
  });
  m.def("compact", [](const py::object& a, const py::object& out, const py::sequence& shape, const py::sequence& strides, size_t offset) {
    Array& A = arr(a, "Compact: a");
    Array& O = arr(out, "Compact: out");
    View v = parse_view(shape, strides);
    check(dfb_compact(A.ptr, O.ptr, O.size, v.ndim, v.shape, v.strides, offset));
  });
  m.def("compact_scale", [](const py::object& a, const py::object& out, const py::sequence& shape, const py::sequence& strides, size_t offset,
                            float scale) {
    Array& A = arr(a, "CompactScale: a");
    Array& O = arr(out, "CompactScale: out");
    View v = parse_view(shape, strides);
    check(dfb_compact_scale(A.ptr, O.ptr, O.size, v.ndim, v.shape, v.strides, offset, scale));
  });
  m.def("reduce_sum_view_div", [](const py::object& a, const py::object& out, const py::sequence& shape, const py::sequence& strides,
                                  size_t offset, float divisor) {
    Array& A = arr(a, "ReduceSumView: a");
    Array& O = arr(out, "ReduceSumView: out");
    View v = parse_view(shape, strides);
    check(dfb_reduce_sum_view_div(A.ptr, O.ptr, O.size, v.ndim, v.shape, v.strides, offset, divisor));
  });
  m.def("ewise_setitem", [](const py::object& a, const py::object& out, const py::sequence& shape, const py::sequence& strides, size_t offset) {
    Array& A = arr(a, "EwiseSetitem: a");
    Array& O = arr(out, "EwiseSetitem: out");
    View v = parse_view(shape, strides);
    check(dfb_ewise_setitem(A.ptr, A.size, O.ptr, v.ndim, v.shape, v.strides, offset));
  });
  m.def("scalar_setitem", [](size_t size, float val, const py::object& out, const py::sequence& shape, const py::sequence& strides, size_t offset) {
    Array& O = arr(out, "ScalarSetitem: out");
    View v = parse_view(shape, strides);
    check(dfb_scalar_setitem(size, val, O.ptr, O.size, v.ndim, v.shape, v.strides, offset));
  });
  m.def("ewise_add", &ewise_binary<dfb_ewise_add>);
  m.def("ewise_mul", &ewise_binary<dfb_ewise_mul>);
  m.def("ewise_div", &ewise_binary<dfb_ewise_div>);
  m.def("ewise_maximum", &ewise_binary<dfb_ewise_maximum>);
  m.def("ewise_eq", &ewise_binary<dfb_ewise_eq>);
  m.def("ewise_ge", &ewise_binary<dfb_ewise_ge>);
  m.def("scalar_add", &ewise_scalar<dfb_scalar_add>);
  m.def("scalar_mul", &ewise_scalar<dfb_scalar_mul>);
  m.def("scalar_div", &ewise_scalar<dfb_scalar_div>);
  m.def("scalar_power", &ewise_scalar<dfb_scalar_power>);
  m.def("scalar_maximum", &ewise_scalar<dfb_scalar_maximum>);
  m.def("scalar_eq", &ewise_scalar<dfb_scalar_eq>);
  m.def("scalar_ge", &ewise_scalar<dfb_scalar_ge>);
  m.def("ewise_log", &ewise_unary<dfb_ewise_log>);
  m.def("ewise_exp", &ewise_unary<dfb_ewise_exp>);
  m.def("ewise_tanh", &ewise_unary<dfb_ewise_tanh>);
  m.def("matmul", [](const py::object& a, const py::object& b, const py::object& out, uint32_t M, uint32_t N, uint32_t P) {
    Array& A = arr(a, "Matmul: a");
    Array& B = arr(b, "Matmul: b");
    Array& O = arr(out, "Matmul: out");
    if (A.size != (size_t)M * N || B.size != (size_t)N * P || O.size != (size_t)M * P)
      throw py::value_error("Matmul: array sizes do not match matrix dimensions");
    check(dfb_matmul(A.ptr, B.ptr, O.ptr, M, N, P, g_matmul_mode));
  });
  m.def("reduce_sum", [](const py::object& a, const py::object& out, size_t reduce_size) {
    Array& A = arr(a, "ReduceSum: a");
    Array& O = arr(out, "ReduceSum: out");
    if (reduce_size == 0) throw py::value_error("ReduceSum: reduce_size cannot be zero");
    if (A.size != O.size * reduce_size) throw py::value_error("ReduceSum: a.size != out.size * reduce_size");
    check(dfb_reduce_sum(A.ptr, O.ptr, O.size, reduce_size));
  });
  m.def("reduce_max", [](const py::object& a, const py::object& out, size_t reduce_size) {
    Array& A = arr(a, "ReduceMax: a");
    Array& O = arr(out, "ReduceMax: out");
    if (reduce_size == 0) throw py::value_error("ReduceMax: reduce_size cannot be zero");
    if (A.size != O.size * reduce_size) throw py::value_error("ReduceMax: a.size != out.size * reduce_size");
    check(dfb_reduce_max(A.ptr, O.ptr, O.size, reduce_size));
  });

  // ---- L1: fused entry points (tensor arguments: Array | (Array, offset) | None) ------------------
  m.def("copy", [](const py::object& src, const py::object& dst, size_t n) { check(dfb_copy(dptr(src), dptr(dst), n)); });
  m.def("add_n", [](const py::object& a, const py::object& b, const py::object& out, size_t n) {
    check(dfb_ewise_add(dptr(a), dptr(b), dptr(out), n));
  });
  m.def("mul_n", [](const py::object& a, const py::object& b, const py::object& out, size_t n) {
    check(dfb_ewise_mul(dptr(a), dptr(b), dptr(out), n));
  });
  m.def("scale_n", [](const py::object& a, float v, const py::object& out, size_t n) {
    check(dfb_scalar_mul(dptr(a), v, dptr(out), n));
  });
  m.def("fill_n", [](const py::object& out, float v, size_t n) { check(dfb_fill(dptr(out), v, n)); });
  m.def("gemm", [](const py::object& A, const py::object& B, const py::object& C, int M, int N, int K, int ta, int tb,
                   int lda, int ldb, int ldc, int accumulate, const py::object& bias, int mode) {
    check(dfb_gemm(dptr(A), dptr(B), dptr(C), M, N, K, ta, tb, lda, ldb, ldc, accumulate, dptr(bias), mode));
  });
  m.def("conv2d_workspace_floats", [](int N, int C, int H, int W, int K, int R, int pad, int stride) {
    size_t n = 0;
    check(dfb_conv2d_workspace_floats(N, C, H, W, K, R, pad, stride, &n));
    return n;
  });
  // the trailing w_layout (WLAYOUT_KCRS = 0 default, WLAYOUT_KRSC = 1) is optional: two overloads per op
  m.def("conv2d_fprop", [](const py::object& x, int x_layout, const py::object& w, const py::object& y, int N, int C, int H,
                           int W, int K, int R, int pad, int stride, int mode, const py::object& ws, size_t ws_floats) {
    check(dfb_conv2d_fprop(dptr(x), x_layout, dptr(w), DFB_WLAYOUT_KCRS, dptr(y), N, C, H, W, K, R, pad, stride, mode, dptr(ws), ws_floats));
  });
  m.def("conv2d_fprop", [](const py::object& x, int x_layout, const py::object& w, const py::object& y, int N, int C, int H,
                           int W, int K, int R, int pad, int stride, int mode, const py::object& ws, size_t ws_floats, int w_layout) {
    check(dfb_conv2d_fprop(dptr(x), x_layout, dptr(w), w_layout, dptr(y), N, C, H, W, K, R, pad, stride, mode, dptr(ws), ws_floats));
  });
  m.def("conv2d_dgrad", [](const py::object& dy, const py::object& w, const py::object& dx, int N, int C, int H, int W, int K,
                           int R, int pad, int stride, int mode, int dgrad_mode, const py::object& ws, size_t ws_floats) {
    check(dfb_conv2d_dgrad(dptr(dy), dptr(w), DFB_WLAYOUT_KCRS, dptr(dx), N, C, H, W, K, R, pad, stride, mode, dgrad_mode, dptr(ws), ws_floats));
  });
  m.def("conv2d_dgrad", [](const py::object& dy, const py::object& w, const py::object& dx, int N, int C, int H, int W, int K,
                           int R, int pad, int stride, int mode, int dgrad_mode, const py::object& ws, size_t ws_floats, int w_layout) {
    check(dfb_conv2d_dgrad(dptr(dy), dptr(w), w_layout, dptr(dx), N, C, H, W, K, R, pad, stride, mode, dgrad_mode, dptr(ws), ws_floats));
  });
  m.def("conv2d_wgrad", [](const py::object& x, int x_layout, const py::object& dy, const py::object& dw, int N, int C, int H,
                           int W, int K, int R, int pad, int stride, int mode, const py::object& ws, size_t ws_floats) {
    check(dfb_conv2d_wgrad(dptr(x), x_layout, dptr(dy), dptr(dw), DFB_WLAYOUT_KCRS, N, C, H, W, K, R, pad, stride, mode, dptr(ws), ws_floats));
  });
  m.def("conv2d_wgrad", [](const py::object& x, int x_layout, const py::object& dy, const py::object& dw, int N, int C, int H,
                           int W, int K, int R, int pad, int stride, int mode, const py::object& ws, size_t ws_floats, int w_layout) {
    check(dfb_conv2d_wgrad(dptr(x), x_layout, dptr(dy), dptr(dw), w_layout, N, C, H, W, K, R, pad, stride, mode, dptr(ws), ws_floats));
  });
  m.def("add_rowvec", [](const py::object& x, const py::object& v, const py::object& y, size_t rows, int cols) {
    check(dfb_add_rowvec(dptr(x), dptr(v), dptr(y), rows, cols));
  });
  m.def("colsum", [](const py::object& x, const py::object& out, size_t rows, int cols) {
    check(dfb_colsum(dptr(x), dptr(out), rows, cols));
  });
  m.def("bn_fwd_train", [](const py::object& x, const py::object& gamma, const py::object& beta, const py::object& y,
                           const py::object& save_mean, const py::object& save_invstd, const py::object& rmean,
                           const py::object& rvar, float momentum, float eps, size_t rows, int C) {
    check(dfb_bn_fwd_train(dptr(x), dptr(gamma), dptr(beta), dptr(y), dptr(save_mean), dptr(save_invstd), dptr(rmean),
                           dptr(rvar), momentum, eps, rows, C));
  });
  m.def("bn_fwd_eval", [](const py::object& x, const py::object& gamma, const py::object& beta, const py::object& rmean,
                          const py::object& rvar, const py::object& y, float eps, size_t rows, int C) {
    check(dfb_bn_fwd_eval(dptr(x), dptr(gamma), dptr(beta), dptr(rmean), dptr(rvar), dptr(y), eps, rows, C));
  });
  m.def("bn_bwd", [](const py::object& x, const py::object& dy, const py::object& gamma, const py::object& save_mean,
                     const py::object& save_invstd, const py::object& dx, const py::object& dgamma, const py::object& dbeta,
                     size_t rows, int C) {
    check(dfb_bn_bwd(dptr(x), dptr(dy), dptr(gamma), dptr(save_mean), dptr(save_invstd), dptr(dx), dptr(dgamma), dptr(dbeta),
                     rows, C));
  });
  // ---- fused epilogue / BatchNorm halves (include/dfb200.h: dfb_conv2d_fprop_stats ... dfb_bn_bwd_apply) ----
  // lazy = true: the statistics go only to bn_fwd_apply / bn_bwd_apply (dfb_conv2d_fprop_stats_lazy, dfb_conv2d_dgrad_fused_lazy)
  m.attr("STATS_LAZY") = 1;
  m.def("conv2d_fprop_stats", [](const py::object& x, int x_layout, const py::object& w, int w_layout, const py::object& y, int N,
                                 int C, int H, int W, int K, int R, int pad, int stride, int mode, const py::object& mean_var, bool lazy) {
    check((lazy ? dfb_conv2d_fprop_stats_lazy : dfb_conv2d_fprop_stats)(dptr(x), x_layout, dptr(w), w_layout, dptr(y), N, C, H, W, K, R, pad,
                                                                      stride, mode, dptr(mean_var)));
  }, py::arg("x"), py::arg("x_layout"), py::arg("w"), py::arg("w_layout"), py::arg("y"), py::arg("N"), py::arg("C"), py::arg("H"), py::arg("W"),
     py::arg("K"), py::arg("R"), py::arg("pad"), py::arg("stride"), py::arg("mode"), py::arg("mean_var"), py::arg("lazy") = false);
  // BatchNorms as 5-tuples (x, save_mean, save_invstd, gamma, beta), like relu_bwd_bn; n_bn = how many are given
  m.def("conv2d_dgrad_fused", [](const py::object& dy, const py::object& w, int w_layout, const py::object& dx, int N, int C, int H,
                                 int W, int K, int R, int pad, int stride, int mode, int dgrad_mode, const py::object& addend,
                                 const py::object& bn0, const py::object& bn1, const py::object& sums, bool relu,
                                 const py::object& relu_res, bool lazy) {
    float* b[2][5] = {{nullptr, nullptr, nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr, nullptr, nullptr}};
    int n_bn = 0;
    const py::object* bns[2] = {&bn0, &bn1};
    for (int i = 0; i < 2; ++i) {
      if (bns[i]->is_none()) break;
      py::tuple t = bns[i]->cast<py::tuple>();
      if (t.size() != 5) throw py::value_error("conv2d_dgrad_fused: a BatchNorm is a 5-tuple");
      for (int j = 0; j < 5; ++j) b[i][j] = dptr(t[j]);
      ++n_bn;
    }
    check((lazy ? dfb_conv2d_dgrad_fused_lazy : dfb_conv2d_dgrad_fused)(dptr(dy), dptr(w), w_layout, dptr(dx), N, C, H, W, K, R, pad, stride, mode,
                                                                        dgrad_mode, dptr(addend), n_bn, b[0][0], b[0][1], b[0][2], b[1][0], b[1][1],
                                                                        b[1][2], dptr(sums), relu ? 1 : 0, b[0][3], b[0][4], b[1][3], b[1][4],
                                                                        dptr(relu_res)));
  }, py::arg("dy"), py::arg("w"), py::arg("w_layout"), py::arg("dx"), py::arg("N"), py::arg("C"), py::arg("H"), py::arg("W"), py::arg("K"),
     py::arg("R"), py::arg("pad"), py::arg("stride"), py::arg("mode"), py::arg("dgrad_mode"), py::arg("addend"), py::arg("bn0"), py::arg("bn1"),
     py::arg("sums"), py::arg("relu"), py::arg("relu_res"), py::arg("lazy") = false);
  m.def("stem_cols", [](const py::object& x, int x_layout, const py::object& col, int N, int C, int H, int W, int R, int pad, int stride,
                        int w_layout) { check(dfb_stem_cols(dptr(x), x_layout, dptr(col), N, C, H, W, R, pad, stride, w_layout)); });
  m.def("stem_pad_weights", [](const py::object& w, const py::object& wp, int K, int cols) {
    check(dfb_stem_pad_weights(dptr(w), dptr(wp), K, cols));
  });
  m.def("conv2d_wgrad_cols", [](const py::object& col, const py::object& dy, const py::object& dw, int w_layout, int N, int OH, int OW,
                                int K, int cols, int mode) {
    check(dfb_conv2d_wgrad_cols(dptr(col), dptr(dy), dptr(dw), w_layout, N, OH, OW, K, cols, mode));
  });
  m.def("colstats_mean_var", [](const py::object& x, size_t rows, int C, const py::object& mean_var) {
    check(dfb_colstats_mean_var(dptr(x), rows, C, dptr(mean_var)));
  });
  // each BatchNorm is the tuple (x, mean_var, gamma, beta, save_mean, save_invstd, running_mean, running_var, momentum, eps)
  m.def("bn_fwd_apply", [](const py::tuple& a, const py::object& b_or_none, const py::object& residual, const py::object& y,
                           size_t rows, int C, bool relu) {
    auto f = [](const py::tuple& t, int i) { return dptr(t[i]); };
    if (a.size() != 10) throw py::value_error("bn_fwd_apply: a BatchNorm is a 10-tuple");
    if (b_or_none.is_none()) {
      check(dfb_bn_fwd_apply(f(a, 0), f(a, 1), f(a, 2), f(a, 3), f(a, 4), f(a, 5), f(a, 6), f(a, 7), a[8].cast<float>(), a[9].cast<float>(),
                             nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0.f, 0.f, dptr(residual), dptr(y),
                             rows, C, relu ? 1 : 0));
    } else {
      py::tuple b = b_or_none.cast<py::tuple>();
      if (b.size() != 10) throw py::value_error("bn_fwd_apply: a BatchNorm is a 10-tuple");
      check(dfb_bn_fwd_apply(f(a, 0), f(a, 1), f(a, 2), f(a, 3), f(a, 4), f(a, 5), f(a, 6), f(a, 7), a[8].cast<float>(), a[9].cast<float>(),
                             f(b, 0), f(b, 1), f(b, 2), f(b, 3), f(b, 4), f(b, 5), f(b, 6), f(b, 7), b[8].cast<float>(), b[9].cast<float>(),
                             dptr(residual), dptr(y), rows, C, relu ? 1 : 0));
    }
  });
  // each BatchNorm is the tuple (x, save_mean, save_invstd, gamma, beta)
  m.def("relu_bwd_bn", [](const py::tuple& a, const py::object& b_or_none, const py::object& residual, const py::object& dy,
                          const py::object& dx, size_t rows, int C) {
    auto f = [](const py::tuple& t, int i) { return dptr(t[i]); };
    if (a.size() != 5) throw py::value_error("relu_bwd_bn: a BatchNorm is a 5-tuple");
    if (b_or_none.is_none()) {
      check(dfb_relu_bwd_bn(f(a, 0), f(a, 1), f(a, 2), f(a, 3), f(a, 4), nullptr, nullptr, nullptr, nullptr, nullptr, dptr(residual),
                            dptr(dy), dptr(dx), rows, C));
    } else {
      py::tuple b = b_or_none.cast<py::tuple>();
      if (b.size() != 5) throw py::value_error("relu_bwd_bn: a BatchNorm is a 5-tuple");
      check(dfb_relu_bwd_bn(f(a, 0), f(a, 1), f(a, 2), f(a, 3), f(a, 4), f(b, 0), f(b, 1), f(b, 2), f(b, 3), f(b, 4), dptr(residual),
                            dptr(dy), dptr(dx), rows, C));
    }
  });
  m.def("bn_bwd_sums", [](const py::object& x, const py::object& dy, const py::object& save_mean, const py::object& save_invstd,
                          const py::object& dbeta, const py::object& dgamma, size_t rows, int C) {
    check(dfb_bn_bwd_sums(dptr(x), dptr(dy), dptr(save_mean), dptr(save_invstd), dptr(dbeta), dptr(dgamma), rows, C));
  });
  // bn = (x, save_mean, save_invstd, gamma, beta)
  m.def("maxpool_relu_bn_bwd", [](const py::tuple& bn, const py::object& pool_y, const py::object& pool_dy, const py::object& dy,
                                  const py::object& sums, int N, int H, int W, int C, int k) {
    if (bn.size() != 5) throw py::value_error("maxpool_relu_bn_bwd: a BatchNorm is a 5-tuple");
    check(dfb_maxpool_relu_bn_bwd(dptr(bn[0]), dptr(bn[1]), dptr(bn[2]), dptr(bn[3]), dptr(bn[4]), dptr(pool_y), dptr(pool_dy), dptr(dy),
                                  dptr(sums), N, H, W, C, k));
  });
  m.def("bn_bwd_apply", [](const py::object& x, const py::object& dy, const py::object& gamma, const py::object& save_mean,
                           const py::object& save_invstd, const py::object& dbeta, const py::object& dgamma, const py::object& dx,
                           size_t rows, int C) {
    check(dfb_bn_bwd_apply(dptr(x), dptr(dy), dptr(gamma), dptr(save_mean), dptr(save_invstd), dptr(dbeta), dptr(dgamma), dptr(dx), rows, C));
  });
  m.def("relu_fwd", [](const py::object& x, const py::object& y, size_t n) { check(dfb_relu_fwd(dptr(x), dptr(y), n)); });
  m.def("relu_bwd", [](const py::object& x, const py::object& dy, const py::object& dx, size_t n) {
    check(dfb_relu_bwd(dptr(x), dptr(dy), dptr(dx), n));
  });
  m.def("maxpool2d_fwd", [](const py::object& x, const py::object& y, const py::object& idx, int N, int H, int W, int C, int k) {
    check(dfb_maxpool2d_fwd(dptr(x), dptr(y), (int32_t*)dptr(idx), N, H, W, C, k));
  });
  m.def("maxpool2d_bwd", [](const py::object& x, const py::object& y, const py::object& dy, const py::object& dx, int N, int H,
                            int W, int C, int k) {
    check(dfb_maxpool2d_bwd(dptr(x), dptr(y), dptr(dy), dptr(dx), N, H, W, C, k));
  });
  m.def("maxpool2d_bwd_idx", [](const py::object& idx, const py::object& dy, const py::object& dx, int N, int H, int W, int C,
                                int k) {
    check(dfb_maxpool2d_bwd_idx((const int32_t*)dptr(idx), dptr(dy), dptr(dx), N, H, W, C, k));
  });
  m.def("avgpool2d_fwd", [](const py::object& x, const py::object& y, int N, int H, int W, int C, int k) {
    check(dfb_avgpool2d_fwd(dptr(x), dptr(y), N, H, W, C, k));
  });
  m.def("avgpool2d_bwd", [](const py::object& dy, const py::object& dx, int N, int H, int W, int C, int k) {
    check(dfb_avgpool2d_bwd(dptr(dy), dptr(dx), N, H, W, C, k));
  });
  m.def("upsample2d_fwd", [](const py::object& x, const py::object& y, int N, int H, int W, int C, int scale, int mode) {
    check(dfb_upsample2d_fwd(dptr(x), dptr(y), N, H, W, C, scale, mode));
  });
  m.def("upsample2d_bwd", [](const py::object& dy, const py::object& dx, int N, int H, int W, int C, int scale, int mode) {
    check(dfb_upsample2d_bwd(dptr(dy), dptr(dx), N, H, W, C, scale, mode));
  });
  m.def("linear_small_fwd", [](const py::object& x, const py::object& w, const py::object& bias, const py::object& y, int M, int K, int N) {
    check(dfb_linear_small_fwd(dptr(x), dptr(w), dptr(bias), dptr(y), M, K, N));
  });
  m.def("linear_small_bwd", [](const py::object& x, const py::object& w, const py::object& dy, const py::object& dx, const py::object& dw,
                               const py::object& db, int M, int K, int N) {
    check(dfb_linear_small_bwd(dptr(x), dptr(w), dptr(dy), dptr(dx), dptr(dw), dptr(db), M, K, N));
  });
  m.def("softmax_ce_fwd", [](const py::object& logits, const py::object& target, const py::object& loss, size_t rows, int cols,
                             float scale) {
    check(dfb_softmax_ce_fwd(dptr(logits), dptr(target), dptr(loss), rows, cols, scale));
  });
  m.def("softmax_ce_bwd", [](const py::object& logits, const py::object& target, const py::object& upstream,
                             const py::object& dlogits, size_t rows, int cols, float scale) {
    check(dfb_softmax_ce_bwd(dptr(logits), dptr(target), dptr(upstream), dptr(dlogits), rows, cols, scale));
  });
  m.def("to_numpy_i32", [](const py::object& a, size_t n) {
    py::array_t<int32_t> out((py::ssize_t)n);
    check(dfb_to_host(dptr(a), (float*)out.mutable_data(), n));
    return out;
  });

  auto ptr_table = [](const py::sequence& seq, std::vector<float*>* out, bool allow_none) {
    out->clear();
    for (auto h : seq) {
      float* p = dptr(h);
      if (!p && !allow_none) throw py::value_error("optimizer step: null tensor in table");
      out->push_back(p);
    }
  };
  m.def("multi_adam_step", [ptr_table](const py::sequence& params, const py::sequence& grads, const py::sequence& m1,
                                       const py::sequence& m2, const std::vector<size_t>& sizes, double lr, double beta1,
                                       double beta2, double eps, double weight_decay, int t, double grad_scale) {
    std::vector<float*> p, g, a, b;
    ptr_table(params, &p, false);
    ptr_table(grads, &g, false);
    ptr_table(m1, &a, false);
    ptr_table(m2, &b, false);
    if (p.size() != sizes.size() || g.size() != sizes.size() || a.size() != sizes.size() || b.size() != sizes.size())
      throw py::value_error("multi_adam_step: table lengths differ");
    check(dfb_multi_adam_step(p.data(), (const float* const*)g.data(), a.data(), b.data(), sizes.data(), (int)sizes.size(), lr,
                              beta1, beta2, eps, weight_decay, t, grad_scale));
  });
  m.def("multi_sgd_step", [ptr_table](const py::sequence& params, const py::sequence& grads, const py::sequence& vel,
                                      const std::vector<size_t>& sizes, double lr, double momentum, double weight_decay,
                                      bool nesterov, double grad_scale) {
    std::vector<float*> p, g, v;
    ptr_table(params, &p, false);
    ptr_table(grads, &g, false);
    ptr_table(vel, &v, true);
    if (p.size() != sizes.size() || g.size() != sizes.size() || v.size() != sizes.size())
      throw py::value_error("multi_sgd_step: table lengths differ");
    check(dfb_multi_sgd_step(p.data(), (const float* const*)g.data(), v.data(), sizes.data(), (int)sizes.size(), lr, momentum,
                             weight_decay, nesterov ? 1 : 0, grad_scale));
  });

  m.def("multi_copy", [ptr_table](const py::sequence& srcs, const py::sequence& dsts, const std::vector<size_t>& sizes) {
    std::vector<float*> s, d;
    ptr_table(srcs, &s, false);
    ptr_table(dsts, &d, false);
    if (s.size() != sizes.size() || d.size() != sizes.size()) throw py::value_error("multi_copy: table lengths differ");
    check(dfb_multi_copy((const float* const*)s.data(), d.data(), sizes.data(), (int)sizes.size()));
  });
  // the library checks the tables (count, null sources, widths)
  m.def("concat_channels_fwd", [ptr_table](const py::sequence& srcs, const std::vector<int>& widths, const py::object& y,
                                           long long rows) {
    std::vector<float*> s;
    ptr_table(srcs, &s, true);
    if (s.size() != widths.size()) throw py::value_error("concat_channels_fwd: table lengths differ");
    check(dfb_concat_channels_fwd((const float* const*)s.data(), widths.data(), (int)s.size(), dptr(y), rows));
  });
  m.def("concat_channels_bwd", [ptr_table](const py::object& dy, const py::sequence& dsrcs, const std::vector<int>& widths,
                                           long long rows) {
    std::vector<float*> d;
    ptr_table(dsrcs, &d, true);
    if (d.size() != widths.size()) throw py::value_error("concat_channels_bwd: table lengths differ");
    check(dfb_concat_channels_bwd(dptr(dy), d.data(), widths.data(), (int)d.size(), rows));
  });

  // ---- pinned host buffers + async copies (input pipeline / bench e2e) ------------------------------
  m.def("pinned_empty", [](size_t n) {
    float* p = nullptr;
    check(dfb_host_alloc_pinned(n, &p));
    py::capsule owner(p, [](void* q) { dfb_host_free_pinned((float*)q); });
    return py::array_t<float>({(py::ssize_t)n}, {(py::ssize_t)sizeof(float)}, p, owner);
  });
  m.def("from_pinned_async", [](py::array_t<float, py::array::c_style> a, const py::object& out, size_t n) {
    if ((size_t)a.size() < n) throw py::value_error("from_pinned_async: source too small");
    check(dfb_from_host_async(a.data(), dptr(out), n));
  });
  m.def("prefetch_from_pinned", [](py::array_t<float, py::array::c_style> a, const py::object& out, size_t n) {
    if ((size_t)a.size() < n) throw py::value_error("prefetch_from_pinned: source too small");
    check(dfb_prefetch_from_host(a.data(), dptr(out), n));
  });
  m.def("prefetch_wait", []() { check(dfb_prefetch_wait()); });
  m.def("to_pinned_async", [](const py::object& src, py::array_t<float, py::array::c_style> a, size_t n) {
    if ((size_t)a.size() < n) throw py::value_error("to_pinned_async: destination too small");
    check(dfb_to_host_async(dptr(src), a.mutable_data(), n));
  });

  // ---- per-batch preparation on the device (augmentation, one-hot + label smoothing) ----------------------
  m.attr("AUGMENT_FIELDS") = DFB_AUGMENT_FIELDS;
  m.def("augment_batch", [](const py::object& x, const py::object& y, const py::object& table, int N, int C, int H, int W, int pad,
                            bool clip, float lo, float hi) {
    check(dfb_augment_batch(dptr(x), dptr(y), dptr(table), N, C, H, W, pad, clip ? 1 : 0, lo, hi));
  });
  m.def("dropout_mask", [](const py::object& mask, size_t n, float keep_prob, const py::object& state) {
    check(dfb_dropout_mask(dptr(mask), n, keep_prob, dptr(state)));
  });
  m.def("onehot_smooth", [](const py::object& labels, const py::object& y, size_t n, int classes, float on_value, float off_value) {
    check(dfb_onehot_smooth(dptr(labels), dptr(y), n, classes, on_value, off_value));
  });

  // ---- data parallel ---------------------------------------------------------------------------------
  m.def("comm_unique_id", []() {
    unsigned char id[128];
    check(dfb_comm_unique_id(id));
    return py::bytes((const char*)id, 128);
  });
  m.def("comm_init", [](const py::bytes& id, int rank, int world) {
    std::string s = id;
    if (s.size() != 128) throw py::value_error("comm_init: id must be 128 bytes");
    py::gil_scoped_release nogil;
    check(dfb_comm_init((const unsigned char*)s.data(), rank, world));
  });
  m.def("comm_destroy", []() { check(dfb_comm_destroy()); });
  m.def("comm_rank", []() { int r = 0, w = 1; dfb_comm_rank(&r, &w); return py::make_tuple(r, w); });
  m.def("comm_allreduce_async", [](const py::object& buf, size_t n) { check(dfb_comm_allreduce_async(dptr(buf), n)); });
  m.def("comm_broadcast_async", [](const py::object& buf, size_t n, int root) { check(dfb_comm_broadcast_async(dptr(buf), n, root)); });
  m.def("comm_wait", []() { check(dfb_comm_wait()); });
  // peer-memory gradient exchange (csrc/peer.cu); peer_init -> an Array over the library-owned arena
  m.def("peer_init", [](size_t n) {
    float* a = nullptr;
    dfb_status st;
    {
      py::gil_scoped_release nogil;
      st = dfb_peer_init(n, &a);
    }
    check(st);
    return std::unique_ptr<Array>(new Array(a, (n + 3) & ~size_t(3)));
  });
  m.def("peer_allreduce_async", [](size_t offset, size_t n, int slot, bool exposed) {
    check(dfb_peer_allreduce_async(offset, n, slot, exposed ? 1 : 0));
  });
  m.def("peer_wait", []() { check(dfb_peer_wait()); });
  m.def("peer_status", []() { unsigned e = 0; dfb_peer_status(&e); return e; });
  m.def("peer_destroy", []() { check(dfb_peer_destroy()); });
}
