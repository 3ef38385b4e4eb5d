// Internal helpers shared by every translation unit of libdfb200.so.
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <atomic>

#include "../../include/dfb200.h"

namespace dfb {

// ---- error reporting ------------------------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;
extern std::atomic<uint64_t> g_tc_launches;

// Lazily creates the context/streams. Returns DFB_OK or an error status (message set).
dfb_status ensure_init();
cudaStream_t compute_stream();
cudaStream_t comm_stream();
int sm_count();
// persistent zero-initialised device words for last-CTA-arrives reductions, one per kernel family (runtime.cu)
constexpr int kTicketWords = 8192;  // slots 0..63: one per kernel family; 64..: per-tile counters of the wgrad kernel
unsigned* ticket_counter(int slot);
// CUDA-graph capture support (runtime.cu)
bool graph_capturing();
dfb_status graph_staging(size_t bytes, int kind, void** host, void** dev);
dfb_status graph_early_h2d(void* dev, const void* host, size_t bytes, void* ack_host = nullptr, size_t ack_offset = 0);
void* graph_last_hyper_ack();                      // the echo word of the optimizer block graph_staging handed out last
constexpr size_t kGraphHyperSeqOffset = 252;       // last word of the 256-byte hyper-parameter block: its sequence number
dfb_status graph_hyper_slot(void* graph_exec, int index, int kind, void** host);

#define DFB_FAIL(code, ...)         \
  do {                              \
    ::dfb::set_error(__VA_ARGS__);  \
    return (code);                  \
  } while (0)

#define DFB_REQUIRE(cond, code, ...) \
  do {                               \
    if (!(cond)) DFB_FAIL(code, __VA_ARGS__); \
  } while (0)

#define DFB_CUDA(expr)                                                                   \
  do {                                                                                   \
    cudaError_t _e = (expr);                                                             \
    if (_e != cudaSuccess)                                                               \
      DFB_FAIL(DFB_ERR_RUNTIME, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),  \
               __FILE__, __LINE__);                                                      \
  } while (0)

#define DFB_INIT()                         \
  do {                                     \
    dfb_status _s = ::dfb::ensure_init();  \
    if (_s != DFB_OK) return _s;           \
  } while (0)

// Checks the launch like the reference does after every kernel (cudaGetLastError,
// ndarray_backend_cuda.cu:140) and counts it.
#define DFB_LAUNCH_CHECK(name)                                                            \
  do {                                                                                    \
    ::dfb::g_launches.fetch_add(1, std::memory_order_relaxed);                            \
    cudaError_t _e = cudaGetLastError();                                                  \
    if (_e != cudaSuccess)                                                                \
      DFB_FAIL(DFB_ERR_RUNTIME, "%s kernel launch failed: %s", name, cudaGetErrorString(_e)); \
  } while (0)

static inline unsigned cdiv(size_t a, size_t b) { return (unsigned)((a + b - 1) / b); }

// Grid size for grid-stride bandwidth kernels: enough CTAs to fill 148 SMs a few times over,
// never more than the work.
static inline unsigned bw_grid(size_t work_items, unsigned threads, unsigned ctas_per_sm = 8) {
  size_t need = (work_items + threads - 1) / threads;
  size_t cap = (size_t)sm_count() * ctas_per_sm;
  if (need < 1) need = 1;
  return (unsigned)(need < cap ? need : cap);
}

// ---- kernel launch with programmatic dependent launch (PDL) ------------------------------------------
// Every kernel of the library starts with pdl_sync() (griddepcontrol.wait + launch_dependents) and is launched
// through launch_k() with the programmatic-stream-serialization attribute: the next kernel in the stream is
// scheduled while this one is still running, does its launch / prologue work, and blocks in pdl_sync() until
// this one has completed and its memory is visible. Inside a captured graph the edges become programmatic
// dependencies. This hides most of the per-kernel launch latency that dominates a step made of ~190 kernels of
// a few microseconds each. DFB_PDL=0 disables the attribute (pdl_sync() is then a no-op).
bool pdl_enabled();
// ---- step timeline (dfb_trace_begin / dfb_trace_end, scripts/step_timeline.py) -------------------------------------------
// While a trace is armed, thread 0 of CTA (0,0,0) of every kernel appends (%globaltimer, grid / block fingerprint) to a
// device buffer right after pdl_sync() - the moment its real work starts, also inside a replayed CUDA graph, where no
// host-side tool of this image sees individual kernels - and the host notes (name, fingerprint, stream) of every launch it
// makes (during a graph's capture: the same sequence the replay runs). Unarmed, the cost is one predicated load per kernel.
void trace_host_launch(const void* func, dim3 grid, dim3 block, cudaStream_t stream);
bool trace_host_armed();
void trace_register_symbol(void (*setter)(unsigned long long*));
#ifdef __CUDACC__
static __device__ unsigned long long* d_trace_buf = nullptr;   // one copy per translation unit, all set by dfb_trace_begin
namespace {
struct TraceSymbolInit {
  TraceSymbolInit() {
    trace_register_symbol(+[](unsigned long long* p) { cudaMemcpyToSymbol(d_trace_buf, &p, sizeof(p)); });
  }
};
static TraceSymbolInit trace_symbol_init_;
}  // namespace
template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  if (trace_host_armed()) trace_host_launch(reinterpret_cast<const void*>(kernel), grid, block, stream);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);  // errors are picked up by DFB_LAUNCH_CHECK
}
// (triggering before the wait, which lets the kernel after next launch too, measured no faster on the training step)
__device__ __forceinline__ void pdl_sync() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (threadIdx.x == 0 && (blockIdx.x | blockIdx.y | blockIdx.z) == 0) {
    unsigned long long* tb = d_trace_buf;   // [0] = records so far, [1] = capacity, then (time, fingerprint) pairs
    if (tb) {
      const unsigned long long i = atomicAdd(tb, 1ull);
      if (i < tb[1]) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        tb[2 + 2 * i] = now;
        tb[3 + 2 * i] = (unsigned long long)gridDim.x | ((unsigned long long)gridDim.y << 24) | ((unsigned long long)gridDim.z << 40) |
                        ((unsigned long long)blockDim.x << 52);
      }
    }
  }
}
#endif

// ---- device helpers ---------------------------------------------------------------------------
#ifdef __CUDACC__
// ---- thread-block cluster helpers (reductions through distributed shared memory) --------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t dsmem_addr(uint32_t local_addr, uint32_t rank) {
  uint32_t remote;
  // volatile: stays behind the preceding cluster barrier, and the dependent loads with it
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(local_addr), "r"(rank));
  return remote;
}
// not volatile / no memory clobber: the loads of one reduction step are independent and must pipeline
// (ordering against the cluster barriers comes from the barriers' own memory clobbers)
__device__ __forceinline__ float4 ld_dsmem_f4(uint32_t remote) {
  float4 v;
  asm("ld.shared::cluster.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(remote));
  return v;
}

// a kernel launch in thread-block clusters of shape `cluster` (and the programmatic-dependent-launch attribute); returns
// what cudaLaunchKernelEx returned
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k_cluster(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, dim3 cluster,
                                    Args&&... args) {
  if (trace_host_armed()) trace_host_launch(reinterpret_cast<const void*>(kernel), grid, block, stream);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cluster.x;
  attr[0].val.clusterDim.y = cluster.y;
  attr[0].val.clusterDim.z = cluster.z;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = pdl_enabled() ? 1 : 0;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
__device__ __forceinline__ uint32_t smem_addr_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float ld_dsmem_f32(uint32_t remote) {
  float v;
  asm("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(remote));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// streaming 128-bit accesses (read-once / write-once data; keeps L1 for the reused operands)
__device__ __forceinline__ float4 ld_stream(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w));
}
#endif

}  // namespace dfb
