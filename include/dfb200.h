/*
 * dfb200.h — C ABI of libdfb200.so, the B200 (sm_100a) compute backend for DeepFlows.
 *
 * This header is the drop-in boundary. Everything the reference binds through its one
 * pybind module `CUDA_BACKEND`
 *   (reference: DeepFlows/backend/backend_src/ndarray_backend_cuda.cu:515-716)
 * has an `extern "C"` entry point here ("L0", same argument meaning and error behaviour),
 * plus the fused entry points ("L1") that replace what the reference composes in Python
 *   (DeepFlows/nn/functional.py, DeepFlows/nn/modules/batchnorm.py, DeepFlows/optim/*.py).
 *
 * Conventions
 *   - every function returns a dfb_status (0 = ok). On error the message is available from
 *     dfb_last_error() (thread local). The status classes mirror the C++ exception classes the
 *     reference throws through pybind (std::invalid_argument -> ValueError, ...), see
 *     ndarray_backend_cuda.cu:113-118,136,167,189,211-212,305.
 *   - all `float*` / `const float*` arguments are DEVICE pointers unless the name says `host`.
 *   - sizes are element counts (float32), not bytes.
 *   - all work is enqueued on the library's compute stream (dfb_stream()); results are visible
 *     to a subsequent dfb_to_host() without an explicit sync, like the reference's default
 *     stream + cudaMemcpy (ndarray_backend_cuda.cu:678,708).
 *   - no function falls back to the CPU. Without a usable CUDA device every call fails with
 *     DFB_ERR_RUNTIME.
 */
#ifndef DFB200_H_
#define DFB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DFB_API __attribute__((visibility("default")))

typedef int dfb_status;
enum {
  DFB_OK = 0,
  DFB_ERR_INVALID = 1,      /* std::invalid_argument -> ValueError   */
  DFB_ERR_RUNTIME = 2,      /* std::runtime_error    -> RuntimeError */
  DFB_ERR_OUT_OF_RANGE = 3, /* std::out_of_range     -> IndexError   */
  DFB_ERR_NOMEM = 4,        /* std::bad_alloc        -> MemoryError  */
  DFB_ERR_DOMAIN = 5        /* std::domain_error     -> ValueError   */
};

#define DFB_MAX_DIMS 8 /* reference: MAX_VEC_SIZE, ndarray_backend_cuda.cu:17 */

/* GEMM / conv operand precision modes (north star: fp32-accurate, TF32, BF16 operand modes;
 * accumulation is always fp32). */
enum {
  DFB_MODE_FP32 = 0,  /* fp32-accurate (parity within 1e-5 of the reference): tcgen05 with operands split into TF32 high and
                         low parts, three MMAs per k-step, fp32 accumulation in TMEM ("3xTF32"); FFMA kernels for shapes
                         the tensor-core path does not take, or for everything with DFB_FP32_TC=0                     */
  DFB_MODE_TF32 = 1,  /* tcgen05 kind::tf32: fp32 operands read as TF32, fp32 accumulation in TMEM (2e-2)      */
  DFB_MODE_BF16 = 2,  /* accepted for API completeness: no bf16 operand format exists, served by the exact FFMA kernels    */
  DFB_MODE_SIMT = 3   /* force the generic FFMA kernels (no first-layer / tensor-core specialisations; tests)  */
};

/* ---------------------------------------------------------------------------------------------
 * Runtime: device, streams, events, memory
 * ------------------------------------------------------------------------------------------- */
DFB_API const char* dfb_last_error(void);
DFB_API const char* dfb_version(void);
/* Select the CUDA device for this process (one process per GPU). Lazy default: device 0,
 * like the reference (it never calls cudaSetDevice). Must be called before the first
 * allocation to have an effect. */
DFB_API dfb_status dfb_set_device(int device);
DFB_API dfb_status dfb_get_device(int* device);
DFB_API dfb_status dfb_device_count(int* count);
DFB_API dfb_status dfb_device_info(char* name, size_t name_cap, int* sm_count, int* cc_major,
                                   int* cc_minor, size_t* total_mem_bytes);
DFB_API dfb_status dfb_synchronize(void);
/* cudaStream_t of the compute stream, as an opaque pointer (for event timing by callers). */
DFB_API void* dfb_stream(void);

/* CUDA events on the compute stream (bench.py times with these). */
DFB_API dfb_status dfb_event_create(void** ev);
DFB_API dfb_status dfb_event_destroy(void* ev);
DFB_API dfb_status dfb_event_record(void* ev);
DFB_API dfb_status dfb_event_synchronize(void* ev);
DFB_API dfb_status dfb_event_elapsed_ms(void* start, void* stop, float* ms);

/* Device buffers. Replaces CudaArray (ndarray_backend_cuda.cu:48-83): an owning 1-D float32
 * device buffer. Memory comes from a caching pool (no cudaMalloc/cudaFree per temporary). */
DFB_API dfb_status dfb_malloc(size_t n_floats, float** out_ptr);
DFB_API dfb_status dfb_free(float* ptr);
DFB_API dfb_status dfb_empty_cache(void);
DFB_API dfb_status dfb_mem_stats(size_t* bytes_in_use, size_t* bytes_reserved,
                                 size_t* n_cuda_malloc);
/* launches issued by this library since process start (kernels only; bench.py "gpu_launches") */
DFB_API uint64_t dfb_launch_count(void);
/* how many of those were tcgen05 (TMA + tensor-core) kernels: lets tests and bench.py prove that a
 * TF32/BF16-mode call really ran on the tensor pipe and did not fall back to the FFMA kernels */
DFB_API uint64_t dfb_tc_launch_count(void);
/* Step timeline (diagnostics; scripts/step_timeline.py): between dfb_trace_begin and dfb_trace_end every kernel of the
 * library records (%globaltimer in ns, grid / block fingerprint: grid.x | grid.y << 24 | grid.z << 40 | block.x << 52) when
 * its work starts - also inside a replayed CUDA graph - and the host notes "stream grid.x grid.y grid.z block name" of every
 * launch it makes (dfb_trace_host_count / dfb_trace_host_line). dfb_trace_reset forgets the device records so far. */
DFB_API dfb_status dfb_trace_begin(size_t capacity);
DFB_API dfb_status dfb_trace_reset(void);
DFB_API dfb_status dfb_trace_end(unsigned long long* records, size_t capacity, size_t* count);
DFB_API size_t dfb_trace_host_count(void);
DFB_API const char* dfb_trace_host_line(size_t i);

/* Host <-> device. Replaces from_numpy / to_numpy (ndarray_backend_cuda.cu:667-716). The copy
 * is staged through pinned memory owned by the library and is complete on return. */
DFB_API dfb_status dfb_from_host(const float* host_src, float* dst, size_t n);
DFB_API dfb_status dfb_to_host(const float* src, float* host_dst, size_t n);
/* Async variants on the compute stream for callers that own pinned memory (input pipeline). */
DFB_API dfb_status dfb_host_alloc_pinned(size_t n_floats, float** host_ptr);
DFB_API dfb_status dfb_host_free_pinned(float* host_ptr);
DFB_API dfb_status dfb_from_host_async(const float* pinned_src, float* dst, size_t n);
DFB_API dfb_status dfb_to_host_async(const float* src, float* pinned_dst, size_t n);
DFB_API dfb_status dfb_copy(const float* src, float* dst, size_t n); /* device to device */
/* Input pipeline (SURVEY 8f rank 2: the reference's DataLoader only hands numpy batches to a blocking
 * cudaMemcpy, utils/data/dataloader.py:60-139 + cu:700-716): the next batch is copied from pinned host memory
 * into a staging buffer on a copy stream WHILE the current step runs. dfb_prefetch_from_host orders the copy
 * after everything enqueued on the compute stream so far (the readers of the staging buffer's old contents);
 * dfb_prefetch_wait makes the compute stream wait for the prefetches issued so far. */
DFB_API dfb_status dfb_prefetch_from_host(const float* pinned_src, float* dst, size_t n);
DFB_API dfb_status dfb_prefetch_wait(void);
/* Per-batch preparation that the reference's training scripts do in numpy on the host before every step, here as
 * one pass on the device over the batch that the prefetch delivered; bit-identical to the numpy code.
 * dfb_augment_batch: augment_batch of test/ResNet_CIFAR10_cuda.py:129-148 on x, y = (N, C, H, W):
 *   reflect-pad by `pad` (numpy mode='reflect', pad < H, W), crop H x W at (crop_y, crop_x) of the padded image,
 *   mirror the crop horizontally where flip != 0, zero the rectangle [erase_y, +erase_h) x [erase_x, +erase_w) of
 *   the result (erase_h = 0 or erase_w = 0: none), then clip to [clip_lo, clip_hi] if `clip` (NaN stays NaN).
 *   `table` is a device array of N rows of DFB_AUGMENT_FIELDS floats holding the host's random draws as exact small
 *   integers: {crop_y, crop_x, flip, erase_y, erase_x, erase_h, erase_w, unused}. y must not alias x.
 * dfb_onehot_smooth: y[i][j] = (j == labels[i] ? 1 : 0) * on_value + off_value, the product and the sum rounded
 *   separately (test/ResNet_CIFAR10_cuda.py:181-183 with on_value = 1 - eps, off_value = eps / classes, both rounded
 *   to float as numpy rounds the Python scalars; 1, 0 gives the plain one-hot of the other scripts). labels are class
 *   indices stored as floats (the reference's buffers are float-only, cu:48-83). */
#define DFB_AUGMENT_FIELDS 8
DFB_API dfb_status dfb_augment_batch(const float* x, float* y, const float* table, int N, int C, int H, int W,
                                     int pad, int clip, float clip_lo, float clip_hi);
/* Dropout mask on the device (opt-in, DEEPFLOWS_DROPOUT=device): mask[i] = Philox4x32-10(key (seed, 0xCAFEF00D), counter
 * (i / 4, step, i >> 34, 0))[i % 4] * 2^-32 < keep_prob ? 1 : 0, with seed = state[0], step = state[1] read from device
 * memory (floats holding integers < 2^24), so a captured graph draws a new mask at every replay when the host bumps
 * state[1]. The reference draws the mask with numpy on the host (nn/modules/dropout.py:27-29): that remains the default. */
DFB_API dfb_status dfb_dropout_mask(float* mask, size_t n, float keep_prob, const float* state);
DFB_API dfb_status dfb_onehot_smooth(const float* labels, float* y, size_t n, int classes, float on_value,
                                     float off_value);

/* Side stream: work enqueued between dfb_side_begin() and dfb_side_end() runs on a second stream that is
 * ordered after everything enqueued on the compute stream so far, concurrently with what the compute
 * stream gets next (used for the wgrad of a convolution's backward, which nothing on the dgrad chain
 * depends on). Several such tasks may be outstanding (they run one after the other on the side stream):
 * dfb_side_join() makes the compute stream wait for all of them, dfb_side_join_lag(n) for all but the n most
 * recent ones - a backward pass joins with a lag of a few layers, so that a weight gradient overlaps the next
 * layers' data-gradient chain instead of sitting on it, and joins everything before anyone reads the weight
 * gradients. A buffer freed while a task is outstanding is recycled only when the compute stream has joined
 * that task. Call them from one thread; begin / end pair up. */
DFB_API dfb_status dfb_side_begin(void);
DFB_API dfb_status dfb_side_end(void);
DFB_API dfb_status dfb_side_join(void);
DFB_API dfb_status dfb_side_join_lag(int lag);

/* CUDA-graph capture of everything enqueued on the compute stream (and, through the comm events, on the
 * communication stream) between begin/end: a whole training step - forward, loss, backward, gradient
 * all-reduce, optimizer - replays as ONE graph launch, with no per-kernel host cost. The reference has
 * nothing comparable (one blocking launch per op, ndarray_backend_cuda.cu passim).
 *   - every block dfb_malloc hands out during the capture belongs to the graph until dfb_graph_destroy:
 *     freed blocks return to the graph's private pool, so replays never alias memory somebody else got.
 *   - host copies (dfb_from_host / dfb_to_host) fail with DFB_ERR_RUNTIME during a capture.
 *   - optimizer steps captured in the graph read their hyper-parameters from pinned host memory at each
 *     replay; dfb_graph_set_adam / dfb_graph_set_sgd set them for the next replay (index = order of the
 *     optimizer steps inside the capture). */
DFB_API dfb_status dfb_graph_begin_capture(void);
DFB_API dfb_status dfb_graph_end_capture(void** graph_exec);
DFB_API dfb_status dfb_graph_launch(void* graph_exec);
DFB_API dfb_status dfb_graph_destroy(void* graph_exec);
DFB_API dfb_status dfb_graph_capturing(int* capturing);
/* kernel nodes / all nodes (kernels, memcpys, NCCL, event waits) that one launch of the graph replays */
DFB_API dfb_status dfb_graph_node_counts(void* graph_exec, int* kernel_nodes, int* all_nodes);
DFB_API dfb_status dfb_graph_set_adam(void* graph_exec, int index, double lr, double beta1, double beta2,
                                      double eps, double weight_decay, int step_t, double grad_scale);
DFB_API dfb_status dfb_graph_set_sgd(void* graph_exec, int index, double lr, double momentum,
                                     double weight_decay, int nesterov, double grad_scale);

/* ---------------------------------------------------------------------------------------------
 * L0: the device-module protocol (one entry per binding of the reference module)
 * ------------------------------------------------------------------------------------------- */
/* fill: ndarray_backend_cuda.cu:127-144 */
DFB_API dfb_status dfb_fill(float* out, float value, size_t n);
/* compact (strided gather): cu:157-176. out[gid] = a[offset + sum_d idx_d*strides[d]] */
DFB_API dfb_status dfb_compact(const float* a, float* out, size_t out_size, int ndim,
                               const int32_t* shape, const int32_t* strides, size_t offset);
/* ewise_setitem (strided scatter): cu:178-198. out[idx(gid)] = a[gid], gid < a_size */
DFB_API dfb_status dfb_ewise_setitem(const float* a, size_t a_size, float* out, int ndim,
                                     const int32_t* shape, const int32_t* strides, size_t offset);
/* scalar_setitem: cu:200-221 */
DFB_API dfb_status dfb_scalar_setitem(size_t size, float value, float* out, size_t out_size,
                                      int ndim, const int32_t* shape, const int32_t* strides,
                                      size_t offset);
/* binary elementwise: cu:224-243,259-270,285-296,325-336,351-362,377-388 */
DFB_API dfb_status dfb_ewise_add(const float* a, const float* b, float* out, size_t n);
DFB_API dfb_status dfb_ewise_mul(const float* a, const float* b, float* out, size_t n);
DFB_API dfb_status dfb_ewise_div(const float* a, const float* b, float* out, size_t n);
DFB_API dfb_status dfb_ewise_maximum(const float* a, const float* b, float* out, size_t n);
DFB_API dfb_status dfb_ewise_eq(const float* a, const float* b, float* out, size_t n);
DFB_API dfb_status dfb_ewise_ge(const float* a, const float* b, float* out, size_t n);
/* tensor-scalar: cu:246-257,272-283,298-323,338-349,364-375,390-401.
 * dfb_scalar_div(value == 0) fails with DFB_ERR_DOMAIN (cu:305). */
DFB_API dfb_status dfb_scalar_add(const float* a, float value, float* out, size_t n);
DFB_API dfb_status dfb_scalar_mul(const float* a, float value, float* out, size_t n);
DFB_API dfb_status dfb_scalar_div(const float* a, float value, float* out, size_t n);
DFB_API dfb_status dfb_scalar_power(const float* a, float value, float* out, size_t n);
DFB_API dfb_status dfb_scalar_maximum(const float* a, float value, float* out, size_t n);
DFB_API dfb_status dfb_scalar_eq(const float* a, float value, float* out, size_t n);
DFB_API dfb_status dfb_scalar_ge(const float* a, float value, float* out, size_t n);
/* unary: cu:403-440. log(a <= 0) = -inf (cu:405). */
DFB_API dfb_status dfb_ewise_log(const float* a, float* out, size_t n);
DFB_API dfb_status dfb_ewise_exp(const float* a, float* out, size_t n);
DFB_API dfb_status dfb_ewise_tanh(const float* a, float* out, size_t n);
/* matmul: cu:443-466. out[M,P] = a[M,N] . b[N,P], row-major (inner dimension is called N). */
DFB_API dfb_status dfb_matmul(const float* a, const float* b, float* out, uint32_t M, uint32_t N,
                              uint32_t P, int mode);
/* reductions over trailing contiguous `reduce_size`: cu:469-509 */
DFB_API dfb_status dfb_reduce_sum(const float* a, float* out, size_t out_size, size_t reduce_size);
/* Fused forms of what backend_tensor.py composes for `sum` / `mean` over one axis (bt.py:624-662) and for the backward
 * of `mean` (tensor.py:763-766); same values bit for bit, fewer passes.
 * reduce_sum_view_div: the view (shape / strides / offset as in dfb_compact, at most DFB_MAX_DIMS dims) has the reduced
 *   axis LAST (1..32 elements); out[i] = (a[view(i, 0)] + a[view(i, 1)] + ... in ascending order) / divisor
 *   = compact + reduce_sum + scalar_div without the compact copy. divisor == 0 -> DFB_ERR_DOMAIN like scalar_div.
 * compact_scale: out[i] = a[view(i)] * scale = scalar_mul + compact of a (broadcast) view in one pass. */
DFB_API dfb_status dfb_reduce_sum_view_div(const float* a, float* out, size_t out_size, int ndim, const int32_t* shape,
                                           const int32_t* strides, size_t offset, float divisor);
DFB_API dfb_status dfb_compact_scale(const float* a, float* out, size_t out_size, int ndim, const int32_t* shape,
                                     const int32_t* strides, size_t offset, float scale);
DFB_API dfb_status dfb_reduce_max(const float* a, float* out, size_t out_size, size_t reduce_size);

/* ---------------------------------------------------------------------------------------------
 * L1: fused entry points behind nn/ and optim/
 * ------------------------------------------------------------------------------------------- */
/* General row-major GEMM on tcgen05:  C[M,N] (+)= op(A)[M,K] . op(B)[K,N] (+ bias[N]).
 *   trans_a = 0: A stored [M,K] (lda >= K);  trans_a = 1: A stored [K,M] (lda >= M)
 *   trans_b = 0: B stored [K,N] (ldb >= N);  trans_b = 1: B stored [N,K] (ldb >= K)
 *   accumulate != 0: C += result.  bias may be NULL.
 * Replaces BackendTensor.__matmul__ + the compact()ed transposes of matmul.grad_fn
 * (DeepFlows/backend/backend_tensor.py:612-622, DeepFlows/tensor.py:699-716). */
DFB_API dfb_status dfb_gemm(const float* A, const float* B, float* C, int M, int N, int K,
                            int trans_a, int trans_b, int lda, int ldb, int ldc, int accumulate,
                            const float* bias, int mode);

/* Convolution (square kernel R, symmetric zero padding, scalar stride, no dilation/groups),
 * replacing F.conv2d = __pad2d + __im2col2d + permute/compact + matmul
 * (DeepFlows/nn/functional.py:249-344).
 *   x_layout / y layouts: DFB_LAYOUT_NCHW (compact NCHW) or DFB_LAYOUT_NHWC (channels-last).
 *   w is (K, C, R, R) compact, exactly the reference's Conv2d.weight (nn/modules/conv.py:85-88).
 *   y, dy, dx are always channels-last (N, OH, OW, K) / (N, H, W, C) physical order — the same
 *   physical order the reference's conv output has before its transpose(0,3,1,2) view
 *   (functional.py:343-344).
 *   workspace: device scratch of at least dfb_conv2d_workspace_floats(...) floats. */
enum { DFB_LAYOUT_NCHW = 0, DFB_LAYOUT_NHWC = 1 };
/* weight (and weight-gradient) storage: (K,C,R,R) compact like the reference's Conv2d.weight, or
 * channels-last (K,R,R,C) - the same logical tensor viewed through strides, which the tensor-core kernels
 * consume in place (no per-step repacking) */
enum { DFB_WLAYOUT_KCRS = 0, DFB_WLAYOUT_KRSC = 1 };
enum {
  DFB_DGRAD_REFERENCE = 0, /* last-writer-wins scatter of functional.py:285-294 (SURVEY Q1) */
  DFB_DGRAD_EXACT = 1      /* true transposed convolution (sum over taps)                   */
};
DFB_API dfb_status dfb_conv2d_workspace_floats(int N, int C, int H, int W, int K, int R, int pad,
                                               int stride, size_t* n_floats);
DFB_API dfb_status dfb_conv2d_fprop(const float* x, int x_layout, const float* w, int w_layout,
                                    float* y, int N, int C, int H, int W, int K, int R, int pad,
                                    int stride, int mode, float* workspace, size_t workspace_floats);
/* dfb_conv2d_dgrad with DFB_DGRAD_EXACT is also the forward pass of the transposed convolution (ConvTranspose2d) whose
 * weight is w: its input is dy [N,OH,OW,K], its output dx [N,H,W,C], its (in, out, k, k) weight is w's (K, C, R, R). */
DFB_API dfb_status dfb_conv2d_dgrad(const float* dy, const float* w, int w_layout, float* dx, int N,
                                    int C, int H, int W, int K, int R, int pad, int stride, int mode,
                                    int dgrad_mode, float* workspace, size_t workspace_floats);
DFB_API dfb_status dfb_conv2d_wgrad(const float* x, int x_layout, const float* dy, float* dw,
                                    int w_layout, int N, int C, int H, int W, int K, int R, int pad,
                                    int stride, int mode, float* workspace, size_t workspace_floats);

/* Convolutions with fused epilogue work (new; the reference has no equivalent - its BatchNorm is 16 tensor ops of
 * its own, DeepFlows/nn/modules/batchnorm.py:30-55, and residual gradients are summed by Tensor.backward,
 * DeepFlows/tensor.py:484-494). The tensor-core kernels do the extra work while the output tile leaves the SM; every
 * other path runs it as separate passes with the same results.
 *   dfb_conv2d_fprop_stats : y = conv(x, w) and mean_var[2][K] = per-channel mean / biased variance of y, what the
 *                            BatchNorm that follows needs (dfb_bn_fwd_apply), without a statistics pass over y.
 *   dfb_conv2d_dgrad_fused : dx = dgrad(dy, w) [+ addend], and for n_bn (0, 1, 2) BatchNorms whose OUTPUT gradient dx
 *                            is: sums[0][C] = sum(dx), sums[1+i][C] = sum(dx * x_hat_i), x_hat_i = (bn_x_i - mean_i) *
 *                            invstd_i - the two reductions of BatchNorm backward (dfb_bn_bwd_apply does the rest).
 *                            relu != 0: dx is the gradient of relu(bn_0(x_0) [+ bn_1(x_1)] [+ relu_res]) - the output of
 *                            dfb_bn_fwd_apply(.., relu = 1): the ReLU's backward (pre-activation recomputed, >= 0 passes,
 *                            tensor.py:872-877) is applied before dx is written and summed. */
DFB_API dfb_status dfb_conv2d_fprop_stats(const float* x, int x_layout, const float* w, int w_layout, float* y, int N,
                                          int C, int H, int W, int K, int R, int pad, int stride, int mode,
                                          float* mean_var);
DFB_API dfb_status dfb_conv2d_dgrad_fused(const float* dy, const float* w, int w_layout, float* dx, int N, int C, int H,
                                          int W, int K, int R, int pad, int stride, int mode, int dgrad_mode,
                                          const float* addend, int n_bn, const float* bn_x0, const float* bn_mean0,
                                          const float* bn_invstd0, const float* bn_x1, const float* bn_mean1,
                                          const float* bn_invstd1, float* sums, int relu, const float* gamma0,
                                          const float* beta0, const float* gamma1, const float* beta1,
                                          const float* relu_res);
/* The same two calls for a caller that hands the statistics ONLY to the BatchNorm kernels: mean_var is then consumed by
 * exactly one dfb_bn_fwd_apply (as its mean_var or mean_var2), `sums` by n_bn calls of dfb_bn_bwd_apply (dbeta = sums,
 * dgamma = sums + (1 + i) * C). The convolution's CTAs then leave their per-channel sums in a device-side accumulator
 * (fp64 atomics) that the BatchNorm kernel reads in its prologue - no reduction kernel between the two launches - and
 * mean_var / sums hold their float values only after that consumer has run (it writes them). Falls back to the eager
 * behaviour whenever no accumulator is free or the tensor-core path does not take the problem; DFB_STAT_SLOTS=0 always. */
DFB_API dfb_status dfb_conv2d_fprop_stats_lazy(const float* x, int x_layout, const float* w, int w_layout, float* y, int N,
                                               int C, int H, int W, int K, int R, int pad, int stride, int mode,
                                               float* mean_var);
DFB_API dfb_status dfb_conv2d_dgrad_fused_lazy(const float* dy, const float* w, int w_layout, float* dx, int N, int C, int H,
                                               int W, int K, int R, int pad, int stride, int mode, int dgrad_mode,
                                               const float* addend, int n_bn, const float* bn_x0, const float* bn_mean0,
                                               const float* bn_invstd0, const float* bn_x1, const float* bn_mean1,
                                               const float* bn_invstd1, float* sums, int relu, const float* gamma0,
                                               const float* beta0, const float* gamma1, const float* beta1,
                                               const float* relu_res);

/* First layer (image input, C*R*R <= 32) through its column matrix, kept between forward and backward:
 *   dfb_stem_cols         : col[pixel][32] = the receptive field of every output pixel (zero padded to 32 columns, in the
 *                           weight's own memory order) - the reference's im2col (functional.py:249-283) for this layer only;
 *   dfb_stem_pad_weights  : wp[K][32] = the weights with every row padded to 32;
 *   forward               = dfb_conv2d_fprop_stats(col as an (N,OH,OW,32) channels-last tensor, wp as (K,1,1,32), R = 1);
 *   dfb_conv2d_wgrad_cols : dW[K][cols] = sum_pixels dy[pixel][K] * col[pixel][cols]  (the layer's weight gradient). */
DFB_API dfb_status dfb_stem_cols(const float* x, int x_layout, float* col, int N, int C, int H, int W, int R, int pad,
                                 int stride, int w_layout);
DFB_API dfb_status dfb_stem_pad_weights(const float* w, float* wp, int K, int cols);
DFB_API dfb_status dfb_conv2d_wgrad_cols(const float* col, const float* dy, float* dw, int w_layout, int N, int OH, int OW,
                                         int K, int cols, int mode);

/* y[r, c] = x[r, c] + v[c]   (conv bias (1,K,1,1) on channels-last, Linear bias (1,out);
 * replaces broadcast_to + compact + ewise_add, backend_tensor.py:533-542) */
DFB_API dfb_status dfb_add_rowvec(const float* x, const float* v, float* y, size_t rows, int cols);
/* out[c] = sum_r x[r, c]  (broadcast-gradient reduction done on the host by the reference,
 * DeepFlows/tensor.py:462-483) */
DFB_API dfb_status dfb_colsum(const float* x, float* out, size_t rows, int cols);
/* out[r] = sum_c x[r,c] is dfb_reduce_sum. */

/* BatchNorm2d on channels-last data viewed as x[rows = N*H*W, C]
 * (DeepFlows/nn/modules/batchnorm.py:30-55): batch mean, biased variance,
 * x_hat = (x-mean)/(var+eps)**0.5, y = x_hat*gamma + beta; running stats updated in place with
 * the biased variance: run = run*(1-momentum) + batch*momentum (batchnorm.py:44-46).
 * save_mean / save_invstd (C floats each) are written for the backward pass.
 * gamma/beta may be NULL (affine=False); running_* may be NULL (track_running_stats=False). */
DFB_API dfb_status dfb_bn_fwd_train(const float* x, const float* gamma, const float* beta, float* y,
                                    float* save_mean, float* save_invstd, float* running_mean,
                                    float* running_var, float momentum, float eps, size_t rows,
                                    int C);
DFB_API dfb_status dfb_bn_fwd_eval(const float* x, const float* gamma, const float* beta,
                                   const float* running_mean, const float* running_var, float* y,
                                   float eps, size_t rows, int C);
/* dx, dgamma, dbeta of the composed reference graph (equals the textbook BN backward). dx,
 * dgamma, dbeta may each be NULL when not needed. */
DFB_API dfb_status dfb_bn_bwd(const float* x, const float* dy, const float* gamma,
                              const float* save_mean, const float* save_invstd, float* dx,
                              float* dgamma, float* dbeta, size_t rows, int C);

/* BatchNorm in explicit halves, for callers that already hold the reductions (the convolution epilogues above):
 *   dfb_colstats_mean_var : mean_var[2][C] = per-channel mean / biased variance of x[rows, C] (one pass)
 *   dfb_bn_fwd_apply      : y = [relu]( bn(x) [+ bn2(x2)] [+ residual] ) from given statistics, ONE pass; publishes
 *                           save_mean / save_invstd and updates the running statistics of each BatchNorm like
 *                           dfb_bn_fwd_train. x2 == NULL: no second BatchNorm (the 1x1-conv shortcut of a residual block).
 *                           Replaces batchnorm.py:30-55 + the block's `out + identity` (+ F.relu) as one kernel.
 *   dfb_relu_bwd_bn       : dx = z >= 0 ? dy : 0 with z = bn(x) [+ bn2(x2)] [+ residual] recomputed exactly as
 *                           dfb_bn_fwd_apply computed it (the fused forward never stores z)
 *   dfb_bn_bwd_sums / dfb_bn_bwd_apply : the reduction half and the elementwise half of dfb_bn_bwd */
DFB_API dfb_status dfb_colstats_mean_var(const float* x, size_t rows, int C, float* mean_var);
DFB_API dfb_status dfb_bn_fwd_apply(const float* x, const float* mean_var, const float* gamma, const float* beta,
                                    float* save_mean, float* save_invstd, float* running_mean, float* running_var,
                                    float momentum, float eps, const float* x2, const float* mean_var2,
                                    const float* gamma2, const float* beta2, float* save_mean2, float* save_invstd2,
                                    float* running_mean2, float* running_var2, float momentum2, float eps2,
                                    const float* residual, float* y, size_t rows, int C, int relu);
DFB_API dfb_status dfb_relu_bwd_bn(const float* x, const float* mean, const float* invstd, const float* gamma,
                                   const float* beta, const float* x2, const float* mean2, const float* invstd2,
                                   const float* gamma2, const float* beta2, const float* residual, const float* dy,
                                   float* dx, size_t rows, int C);
DFB_API dfb_status dfb_bn_bwd_sums(const float* x, const float* dy, const float* save_mean, const float* save_invstd,
                                   float* dbeta, float* dgamma, size_t rows, int C);
/* Backward of conv -> BatchNorm -> ReLU -> MaxPool(k, stride k) from the pool's gradient down to the BatchNorm's two
 * reductions, in ONE pass over the BatchNorm's input x [N,H,W,C] (replaces dfb_maxpool2d_bwd + dfb_relu_bwd_bn +
 * dfb_bn_bwd_sums: three passes over the largest activation of the net): dy[n,h,w,c] = pool_dy of the window if
 * relu(bn(x)) equals the window's maximum pool_y (ties included, like dfb_maxpool2d_bwd) and bn(x) >= 0, else 0;
 * sums[0][C] = sum(dy), sums[1][C] = sum(dy * x_hat). dfb_bn_bwd_apply(x, dy, .., sums, sums + C, ..) finishes. */
DFB_API dfb_status dfb_maxpool_relu_bn_bwd(const float* x, const float* save_mean, const float* save_invstd,
                                           const float* gamma, const float* beta, const float* pool_y,
                                           const float* pool_dy, float* dy, float* sums, int N, int H, int W, int C,
                                           int k);
DFB_API dfb_status dfb_bn_bwd_apply(const float* x, const float* dy, const float* gamma, const float* save_mean,
                                    const float* save_invstd, float* dbeta, float* dgamma, float* dx,
                                    size_t rows, int C);   /* (dbeta / dgamma are WRITTEN when they come from
                                                              dfb_conv2d_dgrad_fused_lazy: see there) */

/* ReLU (F.relu = maximum(x, 0), functional.py:15-16). Backward follows maximum.grad_fn
 * (tensor.py:872-877): dx = (y == x) * dy, i.e. the gradient passes where x >= 0. */
DFB_API dfb_status dfb_relu_fwd(const float* x, float* y, size_t n);
DFB_API dfb_status dfb_relu_bwd(const float* x, const float* dy, float* dx, size_t n);

/* 2-D max pooling on channels-last data, window k, stride s == k (non-overlapping), no padding
 * — the only shape the configs use (functional.py:347-374). idx (optional, may be NULL) receives
 * the first arg-max position inside the window (r*k + s) as int32, bit-exact with numpy argmax.
 * Backward, reference semantics (tensor.py:779-791): every tied maximum receives the gradient. */
DFB_API dfb_status dfb_maxpool2d_fwd(const float* x, float* y, int32_t* idx, int N, int H, int W,
                                     int C, int k);
DFB_API dfb_status dfb_maxpool2d_bwd(const float* x, const float* y, const float* dy, float* dx,
                                     int N, int H, int W, int C, int k);
/* arg-max routed backward (single winner, torch semantics) */
DFB_API dfb_status dfb_maxpool2d_bwd_idx(const int32_t* idx, const float* dy, float* dx, int N,
                                         int H, int W, int C, int k);
/* average pooling, same geometry (the reference's avg_pool2d raises, SURVEY Q4) */
DFB_API dfb_status dfb_avgpool2d_fwd(const float* x, float* y, int N, int H, int W, int C, int k);
DFB_API dfb_status dfb_avgpool2d_bwd(const float* dy, float* dx, int N, int H, int W, int C, int k);

/* 2-D upsampling by an integer factor 1 <= scale <= 8 on channels-last data (F.interpolate / nn.Upsample):
 * x [N,H,W,C] -> y [N,H*scale,W*scale,C]; the backward maps dy of y's shape to dx of x's shape.
 *   DFB_UPSAMPLE_NEAREST  : y[oh,ow] = x[oh/scale, ow/scale] (a copy, bit-exact); dx sums its scale x scale block.
 *   DFB_UPSAMPLE_BILINEAR : align_corners=False, PyTorch's source rule src = max(0, (o + 0.5)/scale - 0.5), the last
 *                           row / column clamped. The backward gathers: every dx element sums, in a fixed order, the
 *                           output gradients that read it (no atomics; results do not depend on scheduling). */
enum { DFB_UPSAMPLE_NEAREST = 0, DFB_UPSAMPLE_BILINEAR = 1 };
DFB_API dfb_status dfb_upsample2d_fwd(const float* x, float* y, int N, int H, int W, int C, int scale, int mode);
DFB_API dfb_status dfb_upsample2d_bwd(const float* dy, float* dx, int N, int H, int W, int C, int scale, int mode);

/* Channel concatenation of channels-last tensors (torch.cat(dim=1) on NHWC, the U-Net skip connection): source i is a
 * [rows, widths[i]] matrix (rows = N*H*W) and occupies columns off_i .. off_i + widths[i] of y [rows, C], where
 * off_i = widths[0] + ... + widths[i-1] and C = the sum of the widths (< 2^31). 1 <= count <= DFB_CONCAT_MAX_SOURCES:
 * the pointer table travels as a kernel parameter, so a captured graph gets no copy node for it.
 *   fwd: y[:, off_i : off_i + widths[i]] = srcs[i]
 *   bwd: dsrcs[i] = dy[:, off_i : off_i + widths[i]]; a null dsrcs[i] (an input that needs no gradient) is skipped.
 * One launch each way; the kernels copy, so results are bit-exact. The pointer tables are HOST arrays. */
#define DFB_CONCAT_MAX_SOURCES 8
DFB_API dfb_status dfb_concat_channels_fwd(const float* const* srcs, const int* widths, int count, float* y, long long rows);
DFB_API dfb_status dfb_concat_channels_bwd(const float* dy, float* const* dsrcs, const int* widths, int count,
                                           long long rows);

/* Linear layers with at most 16 outputs (the classifier) in one launch each way (F.linear, functional.py:8-12; W is
 * (in, out) = K x N row-major like the reference's Linear.weight, x is M x K, bias N floats or NULL):
 *   fwd: y = x . W + bias          bwd: dx = dy . W^T, dw = x^T . dy, db = column sums of dy (each may be NULL) */
DFB_API dfb_status dfb_linear_small_fwd(const float* x, const float* w, const float* bias, float* y, int M, int K, int N);
DFB_API dfb_status dfb_linear_small_bwd(const float* x, const float* w, const float* dy, float* dx, float* dw, float* db,
                                        int M, int K, int N);

/* Fused softmax cross-entropy with dense targets (F.cross_entropy, functional.py:104-115):
 *   loss = scale * sum_i sum_j -(x_ij - max_i - log sum_j exp(x_ij - max_i)) * t_ij
 * with scale = 1/rows for reduction='mean', 1 for 'sum'. loss is one float.
 * dlogits_ij = scale * upstream[0] * (softmax_ij * sum_j t_ij - t_ij). */
DFB_API dfb_status dfb_softmax_ce_fwd(const float* logits, const float* target, float* loss,
                                      size_t rows, int cols, float scale);
DFB_API dfb_status dfb_softmax_ce_bwd(const float* logits, const float* target,
                                      const float* upstream, float* dlogits, size_t rows, int cols,
                                      float scale);

/* Multi-tensor optimizer steps: ONE launch updates every parameter.
 * The pointer tables are HOST arrays of device pointers, `count` entries each.
 * Adam follows DeepFlows/optim/adam.py:28-63 exactly (L2 decay folded into the gradient,
 * bias correction with t starting at 1, eps outside the sqrt). grad_scale multiplies every
 * gradient first (1/world_size for data parallel).
 * SGD follows DeepFlows/optim/sgd.py:16-24 (velocity v = v*momentum + g, optional nesterov).
 * Hyper-parameters are doubles because the reference derives its float32 scalars from Python
 * doubles (e.g. float32(1 - beta1**t)); velocity may be NULL when momentum == 0. */
DFB_API dfb_status dfb_multi_adam_step(float* const* params, const float* const* grads,
                                       float* const* exp_avg, float* const* exp_avg_sq,
                                       const size_t* sizes, int count, double lr, double beta1,
                                       double beta2, double eps, double weight_decay, int step_t,
                                       double grad_scale);
DFB_API dfb_status dfb_multi_sgd_step(float* const* params, const float* const* grads,
                                      float* const* velocity, const size_t* sizes, int count,
                                      double lr, double momentum, double weight_decay,
                                      int nesterov, double grad_scale);

/* `count` flat device-to-device copies dsts[i][0:sizes[i]] = srcs[i][0:sizes[i]] in ONE launch (packing the
 * gradients of a bucket before its all-reduce). The pointer tables are HOST arrays of device pointers. */
DFB_API dfb_status dfb_multi_copy(const float* const* srcs, float* const* dsts, const size_t* sizes, int count);

/* ---------------------------------------------------------------------------------------------
 * Data parallel (new; the reference has no dist/): one process per GPU, NCCL over NVLink
 * ------------------------------------------------------------------------------------------- */
/* 128-byte ncclUniqueId created on rank 0 and shipped to the other ranks by the host layer. */
DFB_API dfb_status dfb_comm_unique_id(unsigned char* id128);
DFB_API dfb_status dfb_comm_init(const unsigned char* id128, int rank, int world_size);
DFB_API dfb_status dfb_comm_destroy(void);
DFB_API dfb_status dfb_comm_rank(int* rank, int* world_size);
/* In-place sum all-reduce of a gradient bucket on the communication stream. The comm stream
 * first waits for everything enqueued on the compute stream so far. */
DFB_API dfb_status dfb_comm_allreduce_async(float* buf, size_t n);
/* broadcast from rank `root` (initial weights) on the comm stream */
DFB_API dfb_status dfb_comm_broadcast_async(float* buf, size_t n, int root);
/* make the compute stream wait for all communication enqueued so far */
DFB_API dfb_status dfb_comm_wait(void);

/* ---------------------------------------------------------------------------------------------
 * Gradient exchange through NVLink / NVSwitch peer memory (new, csrc/peer.cu): the all-reduce of a bucket
 * as one kernel on the stream that packed it, its completion awaited inside the fused optimizer kernel.
 * ncclAllReduce (above) stays as the fallback; dfb_peer_init decides for all ranks together.
 * ------------------------------------------------------------------------------------------- */
/* Collective over the communicator of dfb_comm_init (2..8 ranks of one box). Allocates this rank's arena of
 * `arena_floats` floats (zero-filled; the gradient buckets live in it), maps every other rank's arena through CUDA
 * IPC and runs a self-test. Fails on EVERY rank (DFB_ERR_RUNTIME, nothing left allocated) if any rank could not map
 * a peer or the self-test did not reproduce the expected sums. `*arena` is owned by the library. */
DFB_API dfb_status dfb_peer_init(size_t arena_floats, float** arena);
/* In-place sum over all ranks of arena[offset, offset + n) (multiples of 4 floats), enqueued on the current compute
 * (or side) stream behind whatever filled the range. `slot` in [0, 63) identifies the bucket: every rank must issue
 * the same sequence of (offset, n, slot). Returns without waiting for the other ranks' slices: dfb_multi_adam_step /
 * dfb_multi_sgd_step wait for all outstanding slots inside their kernel, dfb_peer_wait for everything else.
 * `exposed` != 0 (the bucket nothing overlaps: the last one of a step, at most 256 KB, one per step) selects the
 * one-shot form: one kernel that stores this rank's copy to every peer, waits for theirs and sums all copies. */
DFB_API dfb_status dfb_peer_allreduce_async(size_t offset, size_t n, int slot, int exposed);
/* the compute stream waits (in a one-CTA kernel) until every outstanding slot is complete on this rank */
DFB_API dfb_status dfb_peer_wait(void);
/* sticky error word: non-zero after a peer did not answer within 20 s (the kernels then fall through) */
DFB_API dfb_status dfb_peer_status(unsigned* error_word);
DFB_API dfb_status dfb_peer_destroy(void);

#ifdef __cplusplus
}
#endif
#endif /* DFB200_H_ */
