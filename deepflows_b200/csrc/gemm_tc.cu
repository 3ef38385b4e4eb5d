// Tensor-core path: TMA-fed tcgen05 / TMEM kernels for GEMM and implicit-GEMM convolution (sm_100a).
//
// One warp-specialised kernel skeleton (tc_kernel<Problem>) serves three problem families:
//   GemmProblem   C[M,N] (+)= op(A)[M,K] . op(B)[K,N]     Linear forward / backward, L0 matmul
//   ConvProblem   y[pix, Kout] = sum_taps x[pix + tap, :] . Wt[Kout, tap, :]    conv fprop, and dgrad
//                 for stride 1 (the same contraction over dy with the taps mirrored)
//   WgradProblem  dWt[Kout, tap, C] = sum_pix dy[pix, Kout] * x[pix + tap, C]   (split over pixel ranges;
//                 WgradClusterProblem: the ranges of one group are summed by a cluster through DSMEM)
// plus the first-layer weight gradient as a column matrix + 1x1 WgradProblem (tc_stem_wgrad),
// replacing the reference's pad + k*k strided setitems + permute/compact + one-thread-per-output matmul
// (DeepFlows/nn/functional.py:249-344, ndarray_backend_cuda.cu:443-466). Nothing is materialised: the
// im2col gather is expressed as TMA box coordinates on a 4-d (C,W,H,N) view of the channels-last
// activations, with the zero padding supplied by TMA's out-of-bounds fill. Stride-2 convolutions read a
// 5-d parity view (2C, W/2, 2, H/2, N) of the same buffer, so every tap is again a dense box.
//
// Pipeline (192 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + tcgen05.mma issuer (both run their
// loops warp-convergently and issue through elect.sync), warps 2-5 = epilogue (tcgen05.ld -> registers ->
// global). Operands are fp32 in HBM and are consumed as TF32 (kind::tf32, 128-byte swizzled tiles, BLOCK_K = 32
// elements per stage, 4 MMAs of K=8 per stage); accumulation is fp32 in TMEM (128 lanes x BLOCK_N columns).
// Tiles are 128 x {32, 64, 128, 256}; up to 128 wide two CTAs share an SM (~100 KB of stage ring each).
//
// What the step's small layers need is short latency chains, not math: split-K over a thread-block cluster
// with the partial tiles summed through distributed shared memory (layers with 8-32 tiles), an incremental
// k-block iterator in the producer, the "row halo" variants (ConvProblem / WgradProblem with ROWS) that bring
// a tile's pixels once per filter column and address the three taps of the column by descriptor offsets, and
// programmatic dependent launch (the prologue below runs while the previous kernel drains).
//
// Operand "major-ness": a tile whose reduction index is contiguous in memory is K-major (one TMA box of
// [rows, 32 k]); a tile whose row/column index is contiguous is MN-major ([32 k, 32 mn] boxes, one per
// 32-wide chunk). Both land in shared memory as rows of 128 bytes with the 128B swizzle, only the UMMA
// shared-memory descriptor differs (SBO = 1024 B; MN-major additionally LBO = bytes per 32-wide chunk).
#include "kernels.cuh"

#include <cuda.h>

#include <algorithm>
#include <type_traits>

namespace dfb {
namespace tc {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 32;               // fp32/tf32 elements per stage = one 128-byte swizzle row
constexpr int UMMA_K = 8;                 // tf32
constexpr int kThreads = 192;
constexpr int MAJOR_K = 0, MAJOR_MN = 1;
constexpr uint32_t kChunkBytes = BLOCK_K * 128;  // one [32 k-rows x 128 B] MN-major chunk

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  uint32_t spins = 0;
  while (true) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) break;
    if (++spins > (1u << 24)) {  // a lost TMA / MMA completion must not hang the GPU
      printf("libdfb200: mbarrier wait timed out (block %d,%d,%d thread %d)\n", blockIdx.x, blockIdx.y, blockIdx.z,
             threadIdx.x);
      __trap();
    }
  }
}
// one lane of a converged warp (the same one every time while all 32 lanes are active)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(dst),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(dst),
      "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(COLS));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(COLS));
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// 32 lanes x 32 consecutive fp32 columns: thread t of the warp receives row (lane base + t)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// UMMA shared-memory descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout type [61,64): SWIZZLE_128B = 2, SWIZZLE_128B_BASE32B = 1
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout) {
  return (uint64_t)((addr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) |
         (1ull << 46) | ((uint64_t)layout << 61);
}
// k-step j (8 tf32 = 32 bytes of K) of an operand tile starting at `base`.
//   K-major : rows of 128 B (32 k), 128B swizzle (16-byte atoms), 8-row groups 1024 B apart.
//   MN-major: rows of 128 B (32 consecutive m/n) per k; 32-bit operands that the tensor core has to
//             transpose need the 128B swizzle with 32-BYTE atoms (cute: SWIZZLE_128B_BASE32B,
//             TMA: CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B), whose pattern repeats every 4 k-rows:
//             SBO = 512 B between 4-row groups, LBO = bytes between 32-wide m/n chunks.
// MN-major operand whose 32-wide chunks are `lbo` bytes apart (run-time: the wgrad row-halo kernel addresses the three
// row-shifted views of one x halo tile as the three chunks of ONE N = 96 operand)
__device__ __forceinline__ uint64_t operand_desc_mn(uint32_t base, int j, uint32_t lbo) {
  return smem_desc(base + j * (UMMA_K * 128), lbo, 512, 1);
}
template <int MAJOR, uint32_t CHUNK_BYTES = kChunkBytes>
__device__ __forceinline__ uint64_t operand_desc(uint32_t base, int j) {
  if (MAJOR == MAJOR_K) return smem_desc(base + j * (UMMA_K * 4), 0, 1024, 2);
  return smem_desc(base + j * (UMMA_K * 128), CHUNK_BYTES, 512, 1);
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D=f32, A=B=tf32, majors, N>>3, M>>4
template <int A_MAJOR, int B_MAJOR, int N>
__host__ __device__ constexpr uint32_t instr_desc_tf32() {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)A_MAJOR << 15) | ((uint32_t)B_MAJOR << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(BLOCK_M >> 4) << 24);
}

// ---- optional in-kernel timeline (build with -DDFB_TC_TIMING: scripts/tc_timing_probe.cu) -------------------------
// The first and the last CTA of a launch record clock64() at the hand-over points of the pipeline; off in the shipped
// library (the macro expands to nothing).
#ifdef DFB_TC_TIMING
__device__ unsigned long long g_tc_stamp[2][16];
#define TC_STAMP(i)                                                                                         \
  do {                                                                                                      \
    if (stamp_slot >= 0 && (threadIdx.x & 31) == 0) g_tc_stamp[stamp_slot][i] = (unsigned long long)clock64(); \
  } while (0)
#else
#define TC_STAMP(i)
#endif


// shared-space accesses by 32-bit shared address (generic-pointer LD/ST to shared memory cost more per access)
__device__ __forceinline__ void sts_f4(uint32_t addr, const float4& v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ float* lds_ptr(uint32_t addr) {
  unsigned long long v;
  asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(addr));
  return reinterpret_cast<float*>(v);
}

// ---- fused epilogue of the row-major problems (conv fprop / dgrad) ------------------------------------------------------
// The accumulator tile leaves TMEM through shared memory (the pipeline stages are idle by then) and is written out
// with whole rows per warp instruction - 128-bit stores, lanes along the channel dimension - instead of one row per
// thread. On the way out the same pass can
//   * add a tensor of the output's shape (`addend`: the identity branch's gradient in a residual block's backward),
//   * produce per-channel statistics of what it writes, so that the BatchNorm that follows needs no pass of its own:
//       EPI_STATS  mean / biased variance of the output (forward: conv -> BatchNorm)
//       EPI_BNBWD  sum(d) and sum(d * x_hat) for up to two BatchNorms whose output gradient d is being written
//                  (backward: dgrad -> BatchNorm backward; two when a residual block's shortcut has its own BatchNorm)
// Every lane owns fixed columns, so the sums accumulate in registers; lanes, warps and CTAs are merged in a fixed order
// (deterministic), one partial per CTA goes to global memory, and the last CTA of the launch (ticket) reduces the
// partials. Variance uses shifted sums (shift = the first value a lane sees, re-based at every merge): no cancellation
// when |mean| >> std, no divisions in the loops.
enum { EPI_NONE = 0, EPI_STATS = 1, EPI_BNBWD = 2 };
// compile-time selection of the epilogue work (template parameter EPI of ConvProblem): the write-out loop is
// instruction-bound, a run-time switch per float4 costs more than the work itself
// EF_RELU (with EF_BNBWD): the gradient being written belongs to relu(bn_0(x_0) [+ bn_1(x_1)] [+ residual]); the ReLU's
// backward is applied first (the pre-activation is recomputed exactly as dfb_bn_fwd_apply computed it), the sums are
// taken of the masked gradient
enum { EF_NONE = 0, EF_STATS = 1, EF_ADDEND = 2, EF_BNBWD = 4, EF_RELU = 8 };
struct EpiArgs {
  const float* addend;       // same shape / layout as the output, or null
  int stat_kind;             // EPI_*
  int n_sets;                // EPI_BNBWD: 1 or 2 BatchNorms
  float* stat_part;          // [partials][3][n_out]
  float* stat_cnt;           // [partials] rows behind each partial (EPI_STATS)
  float* stat_out;           // [3][n_out]: EPI_STATS mean, var, -; EPI_BNBWD sum d, sum d*x_hat(set 0), sum d*x_hat(set 1)
  unsigned* stat_ticket;
  const float* bn_x[2];      // EPI_BNBWD: inputs of the BatchNorms (shape of the output)
  const float* bn_mean[2];
  const float* bn_invstd[2];
  const float* bn_gamma[2];  // EF_RELU: affine parameters (null: 1 / 0) and the residual term of the pre-activation
  const float* bn_beta[2];
  const float* relu_res;
  int relu;
  // statistic slot (kernels.cuh): when set, every CTA adds its sums to stat_acc[3][kStatSlotChannels] with fp64 atomics
  // (EPI_STATS: the unshifted sum and sum of squares) instead of writing a partial, and no reduction kernel follows
  double* stat_acc;
  int lazy;                  // host only: the caller allows the slot
};
// (shift, sum of (v - shift), sum of (v - shift)^2, count) of one column over some rows
struct Moments {
  float s, m1, m2, n;
  __device__ __forceinline__ void merge(const Moments& o) {
    if (o.n > 0.f) {
      if (n > 0.f) {
        const float d = o.s - s;
        m2 += o.m2 + 2.f * d * o.m1 + o.n * d * d;
        m1 += o.m1 + o.n * d;
        n += o.n;
      } else {
        *this = o;
      }
    }
  }
};
template <int BN>
struct RowEpi {
  static constexpr int LPR = (BN / 4 < 32) ? BN / 4 : 32;    // lanes per output row
  static constexpr int RPI = 32 / LPR;                        // rows per warp instruction
  static constexpr int NCG = (BN / 4 <= 32) ? 1 : BN / 128;   // float4 column groups per lane
  float a[NCG][4], b[NCG][4], c[NCG][4];                      // EPI_STATS: shift, m1, m2; EPI_BNBWD: sum d, sum d*xh0, sum d*xh1
  float n;
  // per-channel constants of the lane's own columns (EF_BNBWD / EF_RELU), loaded once per CTA: mean, invstd,
  // invstd * gamma, beta of up to two BatchNorms
  float4 k_mu[2][NCG], k_is[2][NCG], k_sc[2][NCG], k_be[2][NCG];
  template <int EF>
  __device__ __forceinline__ void load_consts(const EpiArgs& e, int col_of_group0, int n_out) {
    if constexpr ((EF & EF_BNBWD) != 0) {
#pragma unroll
      for (int s2 = 0; s2 < 2; ++s2) {
        if (s2 >= e.n_sets) break;
#pragma unroll
        for (int g = 0; g < NCG; ++g) {
          const int col = col_of_group0 + g * 128;
          const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f), one = make_float4(1.f, 1.f, 1.f, 1.f);
          const bool ok = col + 4 <= n_out;
          k_mu[s2][g] = ok ? __ldg(reinterpret_cast<const float4*>(e.bn_mean[s2] + col)) : zero;
          k_is[s2][g] = ok ? __ldg(reinterpret_cast<const float4*>(e.bn_invstd[s2] + col)) : zero;
          if constexpr ((EF & EF_RELU) != 0) {
            const float4 gm = (ok && e.bn_gamma[s2]) ? __ldg(reinterpret_cast<const float4*>(e.bn_gamma[s2] + col)) : one;
            k_be[s2][g] = (ok && e.bn_beta[s2]) ? __ldg(reinterpret_cast<const float4*>(e.bn_beta[s2] + col)) : zero;
            k_sc[s2][g] = make_float4(k_is[s2][g].x * gm.x, k_is[s2][g].y * gm.y, k_is[s2][g].z * gm.z, k_is[s2][g].w * gm.w);
          }
        }
      }
    }
  }
  __device__ __forceinline__ void init() {
#pragma unroll
    for (int g = 0; g < NCG; ++g)
#pragma unroll
      for (int q = 0; q < 4; ++q) { a[g][q] = 0.f; b[g][q] = 0.f; c[g][q] = 0.f; }
    n = 0.f;
  }
  // What one float4 of the output needs from global memory besides the accumulator: loaded ahead of the stores of a
  // batch of rows, so that the loads of the whole batch are in flight together.
  struct Extras { float4 add, x0, x1, res; };
  template <int EF>
  __device__ __forceinline__ static Extras load_extras(const EpiArgs& e, const float* out, const float* row_out, int col, int n_out) {
    Extras x{};
    if constexpr (EF == EF_NONE || EF == EF_STATS) return x;
    if (row_out == nullptr || col + 4 > n_out) return x;
    const size_t off = (size_t)(row_out - out) + col;
    if constexpr ((EF & EF_ADDEND) != 0) x.add = __ldg(reinterpret_cast<const float4*>(e.addend + off));
    if constexpr ((EF & EF_BNBWD) != 0) {
      x.x0 = __ldg(reinterpret_cast<const float4*>(e.bn_x[0] + off));
      if (e.n_sets > 1) x.x1 = __ldg(reinterpret_cast<const float4*>(e.bn_x[1] + off));
    }
    if constexpr ((EF & EF_RELU) != 0) {
      x.res = make_float4(0.f, 0.f, 0.f, 0.f);
      if (e.relu_res) x.res = __ldg(reinterpret_cast<const float4*>(e.relu_res + off));
    }
    return x;
  }
  // one float4 of the output: row base pointer `row_out` (inside e's output tensor), absolute column `col`.
  // The caller adds 1 to `n` after the last column group of a row.
  template <int EF>
  __device__ __forceinline__ void emit(const EpiArgs& e, float* row_out, int col, int g, float4 v, const Extras& x, int n_out) {
    if (col + 4 > n_out) return;
    if constexpr ((EF & EF_ADDEND) != 0) { v.x += x.add.x; v.y += x.add.y; v.z += x.add.z; v.w += x.add.w; }
    if constexpr ((EF & EF_RELU) != 0) {
      // z = fmaf(x - mean, invstd * gamma, beta) [+ the same of the second BatchNorm] [+ residual]: dfb_bn_fwd_apply's
      // operations in its order, so the mask is the one the forward pass applied; the gradient passes where z >= 0
      const float xa[4] = {x.x0.x, x.x0.y, x.x0.z, x.x0.w}, xb[4] = {x.x1.x, x.x1.y, x.x1.z, x.x1.w}, rr[4] = {x.res.x, x.res.y, x.res.z, x.res.w};
      const float m0[4] = {k_mu[0][g].x, k_mu[0][g].y, k_mu[0][g].z, k_mu[0][g].w}, s0[4] = {k_sc[0][g].x, k_sc[0][g].y, k_sc[0][g].z, k_sc[0][g].w},
                  b0[4] = {k_be[0][g].x, k_be[0][g].y, k_be[0][g].z, k_be[0][g].w};
      const float m1[4] = {k_mu[1][g].x, k_mu[1][g].y, k_mu[1][g].z, k_mu[1][g].w}, s1[4] = {k_sc[1][g].x, k_sc[1][g].y, k_sc[1][g].z, k_sc[1][g].w},
                  b1[4] = {k_be[1][g].x, k_be[1][g].y, k_be[1][g].z, k_be[1][g].w};
      float d[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float z = fmaf(xa[q] - m0[q], s0[q], b0[q]);
        if (e.n_sets > 1) z = z + fmaf(xb[q] - m1[q], s1[q], b1[q]);
        if (e.relu_res) z = z + rr[q];
        d[q] = z >= 0.f ? d[q] : 0.f;
      }
      v = make_float4(d[0], d[1], d[2], d[3]);
    }
    const float vv[4] = {v.x, v.y, v.z, v.w};
    if constexpr ((EF & EF_STATS) != 0) {
      if (n == 0.f) {
#pragma unroll
        for (int q = 0; q < 4; ++q) a[g][q] = vv[q];
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) { const float d = vv[q] - a[g][q]; b[g][q] += d; c[g][q] = fmaf(d, d, c[g][q]); }
    } else if constexpr ((EF & EF_BNBWD) != 0) {
      const float4 mu0 = k_mu[0][g], is0 = k_is[0][g];
      const float xh0[4] = {(x.x0.x - mu0.x) * is0.x, (x.x0.y - mu0.y) * is0.y, (x.x0.z - mu0.z) * is0.z, (x.x0.w - mu0.w) * is0.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) { a[g][q] += vv[q]; b[g][q] = fmaf(vv[q], xh0[q], b[g][q]); }
      if (e.n_sets > 1) {
        const float4 mu1 = k_mu[1][g], is1 = k_is[1][g];
        const float xh1[4] = {(x.x1.x - mu1.x) * is1.x, (x.x1.y - mu1.y) * is1.y, (x.x1.z - mu1.z) * is1.z, (x.x1.w - mu1.w) * is1.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) c[g][q] = fmaf(vv[q], xh1[q], c[g][q]);
      }
    }
    *reinterpret_cast<float4*>(row_out + col) = v;
  }
  // Merge lanes -> warps -> CTA, write this CTA's partial, and let the last CTA of the launch reduce all partials.
  // Called by the 128 epilogue threads (t = 0..127, warp ew = t / 32); `wstat` is the CTA's [4][4][BN] scratch.
  // `scratch`: 8 KB of shared memory nobody else touches any more (the idle pipeline stages).
  __device__ void finish(const EpiArgs& e, float* wstat, float* scratch, int t, int col0, int n_out, int pidx, int n_partials, unsigned total_ctas) {
    if (e.stat_kind == EPI_NONE) return;
    const int lane = t & 31, ew = t >> 5;
    const bool stats = e.stat_kind == EPI_STATS;
    // lanes that share columns (different rows of one warp instruction)
#pragma unroll
    for (int off = LPR; off < 32; off <<= 1) {
      const float on = __shfl_xor_sync(0xffffffffu, n, off);
#pragma unroll
      for (int g = 0; g < NCG; ++g)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float oa = __shfl_xor_sync(0xffffffffu, a[g][q], off), ob = __shfl_xor_sync(0xffffffffu, b[g][q], off),
                      oc = __shfl_xor_sync(0xffffffffu, c[g][q], off);
          if (stats) {
            Moments m{a[g][q], b[g][q], c[g][q], n};
            // both partners must end with the same bits: merge in lane order (lower lane first)
            Moments o{oa, ob, oc, on};
            if (lane & off) { o.merge(m); m = o; } else { m.merge(o); }
            a[g][q] = m.s; b[g][q] = m.m1; c[g][q] = m.m2;
          } else {
            a[g][q] += oa; b[g][q] += ob; c[g][q] += oc;
          }
        }
      n += on;
    }
    if (lane < LPR) {
#pragma unroll
      for (int g = 0; g < NCG; ++g)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int cl = (g * 32 + lane) * 4 + q;
          wstat[(ew * 4 + 0) * BN + cl] = a[g][q];
          wstat[(ew * 4 + 1) * BN + cl] = b[g][q];
          wstat[(ew * 4 + 2) * BN + cl] = c[g][q];
          wstat[(ew * 4 + 3) * BN + cl] = n;
        }
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    for (int cl = t; cl < BN; cl += 128) {
      const int col = col0 + cl;
      if (col >= n_out) continue;
      float r0, r1, r2, rn;
      if (stats) {
        Moments m{0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int w = 0; w < 4; ++w) m.merge(Moments{wstat[(w * 4 + 0) * BN + cl], wstat[(w * 4 + 1) * BN + cl], wstat[(w * 4 + 2) * BN + cl], wstat[(w * 4 + 3) * BN + cl]});
        r0 = m.s; r1 = m.m1; r2 = m.m2; rn = m.n;
      } else {
        r0 = r1 = r2 = 0.f; rn = 0.f;
#pragma unroll
        for (int w = 0; w < 4; ++w) { r0 += wstat[(w * 4 + 0) * BN + cl]; r1 += wstat[(w * 4 + 1) * BN + cl]; r2 += wstat[(w * 4 + 2) * BN + cl]; }
      }
      if (e.stat_acc) {
        double* acc = e.stat_acc + col;
        if (stats) {
          if (rn > 0.f) {   // sums of (v - s), (v - s)^2 over rn rows -> sums of v, v^2
            const double s = (double)r0, m1 = (double)r1, m2 = (double)r2, n_ = (double)rn;
            atomicAdd(acc, m1 + n_ * s);
            atomicAdd(acc + kStatSlotChannels, m2 + 2.0 * s * m1 + n_ * s * s);
          }
        } else {
          atomicAdd(acc, (double)r0);
          atomicAdd(acc + kStatSlotChannels, (double)r1);
          if (e.n_sets > 1) atomicAdd(acc + 2 * kStatSlotChannels, (double)r2);
        }
        continue;
      }
      float* dst = e.stat_part + (size_t)pidx * 3 * n_out + col;
      dst[0] = r0; dst[n_out] = r1; dst[2 * n_out] = r2;
      if (stats && cl == 0 && col0 == 0) e.stat_cnt[pidx] = rn;
    }
  }
};

// The partials of one launch -> per-channel results, one CTA per float4 column group: 128 threads walk the partials
// (four 128-bit loads per array in flight), a fixed-order shuffle / shared-memory tree adds them. A separate, tiny,
// fully parallel kernel behind the convolution: letting the convolution's last CTA do this (ticket + __threadfence)
// put a serial chain of L2 round trips at the end of every fused launch (+8 us per convolution, measured).
__global__ void __launch_bounds__(128) epi_finalize_kernel(const float* __restrict__ part, const float* __restrict__ cnt, int n_partials,
                                                          int n_out, int stats, float* __restrict__ out) {
  pdl_sync();
  const int ncol4 = n_out >> 2, c4 = blockIdx.x, t = threadIdx.x;
  const float4* part4 = reinterpret_cast<const float4*>(part);
  float4 t0 = make_float4(0.f, 0.f, 0.f, 0.f), t1 = t0, t2 = t0, sref = t0;
  float tn = 0.f;
  if (stats) sref = __ldcg(part4 + c4);   // partial 0 always holds rows (pixel 0 is in it)
  for (int p0 = t; p0 < n_partials; p0 += 4 * 128) {
    float4 pa[4], pb[4], pc[4];
    float pn[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int pp = p0 + u * 128;
      const bool ok = pp < n_partials;
      const float4* src = part4 + (size_t)(ok ? pp : 0) * 3 * ncol4 + c4;
      pa[u] = __ldcg(src);
      pb[u] = __ldcg(src + ncol4);
      pc[u] = __ldcg(src + 2 * ncol4);
      pn[u] = stats ? __ldcg(cnt + (ok ? pp : 0)) : 0.f;
      if (!ok) { pa[u] = sref; pb[u] = pc[u] = make_float4(0.f, 0.f, 0.f, 0.f); pn[u] = 0.f; }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (stats) {
        const float n_ = pn[u];
        float d;
        d = pa[u].x - sref.x; t1.x += pb[u].x + n_ * d; t2.x += pc[u].x + 2.f * d * pb[u].x + n_ * d * d;
        d = pa[u].y - sref.y; t1.y += pb[u].y + n_ * d; t2.y += pc[u].y + 2.f * d * pb[u].y + n_ * d * d;
        d = pa[u].z - sref.z; t1.z += pb[u].z + n_ * d; t2.z += pc[u].z + 2.f * d * pb[u].z + n_ * d * d;
        d = pa[u].w - sref.w; t1.w += pb[u].w + n_ * d; t2.w += pc[u].w + 2.f * d * pb[u].w + n_ * d * d;
        tn += n_;
      } else {
        t0.x += pa[u].x; t0.y += pa[u].y; t0.z += pa[u].z; t0.w += pa[u].w;
        t1.x += pb[u].x; t1.y += pb[u].y; t1.z += pb[u].z; t1.w += pb[u].w;
        t2.x += pc[u].x; t2.y += pc[u].y; t2.z += pc[u].z; t2.w += pc[u].w;
      }
    }
  }
  float v[13] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w, t2.x, t2.y, t2.z, t2.w, tn};
#pragma unroll
  for (int off = 16; off > 0; off >>= 1)
#pragma unroll
    for (int i = 0; i < 13; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], off);
  __shared__ float red[4][13];
  if ((t & 31) == 0) {
#pragma unroll
    for (int i = 0; i < 13; ++i) red[t >> 5][i] = v[i];
  }
  __syncthreads();
  if (t == 0) {
    float r[13];
#pragma unroll
    for (int i = 0; i < 13; ++i) r[i] = ((red[0][i] + red[1][i]) + red[2][i]) + red[3][i];
    float4* out4 = reinterpret_cast<float4*>(out);
    if (stats) {
      const float inv = 1.f / r[12];
      const float4 dm = make_float4(r[4] * inv, r[5] * inv, r[6] * inv, r[7] * inv);
      out4[c4] = make_float4(sref.x + dm.x, sref.y + dm.y, sref.z + dm.z, sref.w + dm.w);   // mean
      out4[ncol4 + c4] = make_float4(fmaxf(r[8] * inv - dm.x * dm.x, 0.f), fmaxf(r[9] * inv - dm.y * dm.y, 0.f),
                                     fmaxf(r[10] * inv - dm.z * dm.z, 0.f), fmaxf(r[11] * inv - dm.w * dm.w, 0.f));  // biased variance (batchnorm.py:38-42)
    } else {
      out4[c4] = make_float4(r[0], r[1], r[2], r[3]);
      out4[ncol4 + c4] = make_float4(r[4], r[5], r[6], r[7]);
      out4[2 * ncol4 + c4] = make_float4(r[8], r[9], r[10], r[11]);
    }
  }
}

// ---- kernel skeleton ----------------------------------------------------------------------------------
// KR: reduction rows per stage (MN-major operands only: 32 or 128). BSUB: B tiles per stage (the row-halo conv
// kernel keeps the three taps of one filter column in a stage, with AROWS = 192 halo rows of A)
// BKR: rows of one B chunk when they differ from KR (wgrad row-halo: 128-pixel A chunks, 192-row B halo chunks).
// OUT: a dedicated output staging tile behind the ring (the persistent kernel's epilogue overlaps the next tile's loads,
// so it cannot borrow the pipeline stages)
// XMUL = 2 (the fp32-accurate "3xTF32" kernels): every stage is followed by a second copy of itself that holds the
// low-order parts of the operands (same relative layout, so the same descriptors + kStageBytes address them)
template <int BN, int AROWS = BLOCK_M, int KR = BLOCK_K, int BSUB = 1, int BKR = KR, bool OUT = false, int XMUL = 1>
struct SmemLayout {
  // What one SM can pull through TMA is bounded by the bytes it keeps in flight (loads take microseconds to
  // return under load), and a CTA's prologue / epilogue / split-K reduction are pure latency: TWO CTAs per SM
  // with ~100 KB of ring each beat one CTA with 192 KB on every layer measured (layer-4 conv 19 -> 14 us,
  // VGG c2_2 wgrad 504 -> 363 us), so that is the budget up to BN = 128; the 128 x 256 kernels keep one CTA per
  // SM (208 KB). AROWS < 128 (wgrad with few output channels) shrinks the A tile to the rows that are really
  // loaded, which buys more stages.
  static constexpr uint32_t kChunk = KR * 128;                 // one [KR k-rows x 128 B] chunk (32 m/n wide)
  static constexpr uint32_t kABytes = (AROWS / 32) * kChunk;
  static constexpr uint32_t kBChunk = BKR * 128;
  static constexpr uint32_t kBTile = (BN / 32) * kBChunk;
  static constexpr uint32_t kBBytes = BSUB * kBTile;
  static constexpr uint32_t kStageBytes = kABytes + kBBytes;            // what TMA fills (and the split warps transform)
  static constexpr uint32_t kStageStride = XMUL * kStageBytes;          // distance between stages
  static constexpr uint32_t kOutBytes = OUT ? ((BLOCK_M * (BN + 4) * 4 + 1023) & ~1023u) : 0;
  // (XMUL = 2: two CTAs per SM while two double stages fit 100 KB, else one CTA with ~200 KB)
  static constexpr uint32_t kBudget = XMUL > 1 ? (2 * kStageStride <= (100u << 10) ? (100u << 10) : (200u << 10))
                                               : (BSUB > 1 ? (BN >= 128 ? (216u << 10) : (108u << 10))
                                                           : (BN >= 256 ? (192u << 10) : (100u << 10))) - kOutBytes;  // (128 x 256 at two CTAs per SM with two stages: measured 7% slower)
  static constexpr int kStagesFit = (int)(kBudget / kStageStride);
  static constexpr int kMinStages = (BSUB > 1 || BKR != KR || XMUL > 1) ? 2 : 3;   // halo variants: two CTAs per SM with two stages each
  static constexpr int kStages = kStagesFit > 12 ? 12 : (kStagesFit < kMinStages ? kMinStages : kStagesFit);
  static constexpr uint32_t kBarOffset = kStages * kStageStride;
  static constexpr int kNumBars = (XMUL > 1 ? 3 : 2) * kStages + 1;     // full, empty, accumulator-complete [, split done]
  // the M = 128 MMA always addresses four 32-row chunks of A: with AROWS < 128 it reads past the A tile (into the
  // B tile / the next stage: rows that are never stored), so the last stage needs that much slack behind it
  // (AROWS == 32: the A descriptor's chunk stride is 0, all four chunks alias the one that is loaded - no over-read)
  static constexpr uint32_t kOverRead = (AROWS == 32 || AROWS >= BLOCK_M) ? 0 : ((BLOCK_M - AROWS) / 32) * kChunk;
  // fused-epilogue scratch behind the barriers (row-major problems): 128 row pointers + per-warp column statistics
  // [4 warps][4 values][BN columns]
  static constexpr uint32_t kEpiOffset = kBarOffset + kOverRead + kNumBars * 8 + 16;
  static constexpr uint32_t kEpiBytes = 1024 + 64 * BN;
  // the persistent kernel's accumulator barriers: full[2], empty[2] (32 bytes of the 48 reserved)
  static constexpr uint32_t kAccBarOffset = (kEpiOffset + 16 + kEpiBytes + 15) & ~15u;
  static constexpr uint32_t kOutOffset = kAccBarOffset + 48;
  static constexpr uint32_t kTotal = kOutOffset + kOutBytes + 1024;  // +1024 for manual alignment
  // split-K partial tile staged in the (idle) pipeline stages: 128 rows, padded pitch against bank conflicts
  static constexpr uint32_t kRedPitch = BN + 4;
  // (the 128 x 256 kernels never split K: they are only chosen for problems with hundreds of tiles)
  static_assert(AROWS < BLOCK_M || BLOCK_M * kRedPitch * 4 <= kBarOffset, "output tile does not fit the pipeline stages");
  static constexpr bool kFits = kTotal <= 227u * 1024u;
  static_assert(XMUL > 1 || kFits, "more shared memory than a CTA can have");
};
// the layout of tc_kernel<P, X3> (OUT = false) and tc_persistent_kernel<P, X3> (OUT = true)
template <class P, bool OUT, bool X3>
using TcLayout = SmemLayout<P::BN, P::AROWS, P::KR, P::kBSub, P::BKR, OUT, X3 ? 2 : 1>;

// X3 = true: fp32-accurate contraction on the tensor pipe ("3xTF32", the package's default fp32 mode). TMA delivers fp32
// operands; warps that are idle during the main loop split every stage in shared memory into a TF32-exact high part
// (written back in place: hi = rna_tf32(v)) and a low part (lo = rna_tf32(v - hi), the second half of the stage), and the
// MMA warp issues hi*hi into the accumulator and lo*hi + hi*lo into a second, small-term accumulator (see tc_kernel) that
// the epilogue adds. What is dropped is lo*lo and the rounding of lo: <= 2^-21 per product relative to |a||b| - the size
// of fp32's own accumulation error (measured against the fp64 contraction in tests/test_gpu_l1.py), and independent of how
// the hardware rounds fp32 operands to TF32. Replaces the FFMA kernels of gemm_simt.cu as what an unchanged script runs
// (reference kernel being replaced: ndarray_backend_cuda.cu:443-466).
__device__ __forceinline__ float rna_tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <class P, bool X3 = false>
__global__ void __launch_bounds__(kThreads) tc_kernel(const __grid_constant__ CUtensorMap map_a,
                                                      const __grid_constant__ CUtensorMap map_b,
                                                      const typename P::Params prm) {
  constexpr int BN = P::BN;
  using L = TcLayout<P, false, X3>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset + L::kOverRead);
  constexpr int kStages = L::kStages;
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full_bar = empty_bar + kStages;
  uint64_t* split_bar = tmem_full_bar + 1;   // [kStages] (X3 only): the stage's hi / lo parts are in place
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(split_bar + (X3 ? kStages : 0));
  (void)split_bar;
  // X3: a second accumulator (columns + kTmemCols) takes the two small terms lo*hi + hi*lo. The tensor core's fp32
  // accumulation is not round-to-nearest (measured: the error against float64 grows linearly with the number of MMAs
  // accumulated into a tile, ~1.2e-8 per MMA relative to the accumulator), so the large term hi*hi gets one accumulation
  // per k-step instead of three, and the small terms, whose own rounding is 2^-11 further down, are added once at the end.
  constexpr int kTmemAlloc = X3 ? 2 * P::kTmemCols : P::kTmemCols;
  static_assert(kTmemAlloc <= 512, "TMEM columns");
  // fused-epilogue scratch: output row pointers of the tile, per-warp column statistics
  float** row_tab = reinterpret_cast<float**>(smem + ((L::kEpiOffset + 15) & ~15u));
  float* wstat = reinterpret_cast<float*>(row_tab + BLOCK_M);
  (void)row_tab; (void)wstat;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#ifdef DFB_TC_TIMING
  const bool first_cta = blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0;
  const bool last_cta = blockIdx.x == gridDim.x - 1 && blockIdx.y == gridDim.y - 1 && blockIdx.z == gridDim.z - 1;
  const int stamp_slot = first_cta ? 0 : (last_cta ? 1 : -1);
  if (warp == 0) TC_STAMP(0);
#endif
  typename P::Tile tile = P::tile(prm);
  // Split-K: the CTAs of a cluster (cluster dims (1,1,S), P::kClusterSplit) share one output tile; CTA `rank`
  // takes the rank-th slice of the k-blocks, accumulates it in its own TMEM, and the S partial tiles are
  // summed through distributed shared memory, each CTA finishing 128/S rows of the tile.
  const int nsplit = P::kClusterSplit ? (int)cluster_nctarank() : 1;
  const int rank = P::kClusterSplit ? (int)cluster_ctarank() : 0;
  int kb_begin = tile.kb_begin, kb_end = tile.kb_end;
  if (nsplit > 1) {
    const int per = (kb_end - kb_begin + nsplit - 1) / nsplit;
    kb_begin = min(kb_end, kb_begin + rank * per);
    kb_end = min(kb_end, kb_begin + per);
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, 1);
      if constexpr (X3) mbar_init(split_bar + s, 4);   // one arrival per split (epilogue) warp
    }
    mbar_init(tmem_full_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<kTmemAlloc>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (warp == 0) TC_STAMP(1);
  // everything above (barrier init, descriptor prefetch, TMEM allocation) overlapped the previous kernel's tail;
  // global memory is touched only from here on
  pdl_sync();
  if (warp == 0) TC_STAMP(2);

  if (warp == 0) {
    // ===== TMA producer =====
    // The whole warp runs the loop convergently (waits, address arithmetic and the k-block iterator then live
    // on the uniform datapath) and one elected lane issues the copies. Issuing from inside `if (lane == 0)`
    // instead makes the compiler wrap every UTMALDG in a uniformisation loop, and the single producer
    // thread's instruction stream is what bounds the pipeline of these short k-blocks. The k-block ->
    // (tap, channel block / pixel block) decomposition is an iterator advanced with adds and compares (the
    // integer divisions happen once, in iter_init).
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t tx = P::tx_bytes(prm, tile);
    typename P::Iter it = P::iter_init(prm, tile, kb_begin);
    for (int kb = kb_begin; kb < kb_end; ++kb) {
      mbar_wait(empty_bar + stage, phase ^ 1);
      const uint32_t a_dst = smem_u32(smem + stage * L::kStageStride);
      const uint32_t b_dst = a_dst + L::kABytes;
      if (elect_one()) {
        mbar_expect_tx(full_bar + stage, tx);
        P::load_a(prm, tile, it, &map_a, full_bar + stage, a_dst);
        P::load_b(prm, tile, it, &map_b, full_bar + stage, b_dst);
      }
      __syncwarp();
      if (kb == kb_begin) TC_STAMP(3);
      P::iter_next(prm, tile, it);
      if (++stage == kStages) { stage = 0; phase ^= 1; }
    }
    TC_STAMP(4);
  } else if (warp == 1) {
    // ===== MMA issuer: the warp waits convergently, one elected lane (always the same one: tcgen05.commit tracks
    // the MMAs of the thread that executes it) issues =====
    constexpr uint32_t idesc = instr_desc_tf32<P::A_MAJOR, P::B_MAJOR, P::kMmaN>();
    int stage = 0;
    uint32_t phase = 0;
    for (int kb = kb_begin; kb < kb_end; ++kb) {
      mbar_wait((X3 ? split_bar : full_bar) + stage, phase);   // X3: the split warps waited for the TMA bytes
      tc_fence_after();
      if (kb == kb_begin) TC_STAMP(5);
      const uint32_t a_base = smem_u32(smem + stage * L::kStageStride);
      const uint32_t b_base = a_base + L::kABytes;
      if (elect_one()) {
        // sub-tiles (taps that share a halo tile of this stage) are the INNER loop: with separate accumulators
        // (wgrad) consecutive MMAs are then independent and pipeline, instead of each waiting for the previous
        // one's accumulation into the same TMEM tile
#pragma unroll
        for (int j = 0; j < P::KR / UMMA_K; ++j) {
#pragma unroll
          for (int t = 0; t < P::kSubTiles; ++t) {
            const uint32_t a_sub = a_base + P::a_sub_offset(prm, t), b_sub = b_base + P::b_sub_offset(prm, t, L::kBTile);
            const uint32_t d_tmem = tmem_base;
            const uint32_t first = (kb > kb_begin || t > 0 || j > 0) ? 1u : 0u;
#pragma unroll
            for (int term = 0; term < (X3 ? 3 : 1); ++term) {   // hi*hi, lo*hi, hi*lo (the low parts: + kStageBytes)
              const uint32_t a_op = a_sub + (term == 1 ? L::kStageBytes : 0u), b_op = b_sub + (term == 2 ? L::kStageBytes : 0u);
              const uint64_t b_desc = P::kRuntimeLbo ? operand_desc_mn(b_op, j, P::b_lbo(prm)) : operand_desc<P::B_MAJOR, L::kBChunk>(b_op, j);
              umma_tf32(d_tmem + (term > 0 ? (uint32_t)P::kTmemCols : 0u), operand_desc<P::A_MAJOR, (P::AROWS == 32 ? 0u : L::kChunk)>(a_op, j), b_desc, idesc,
                        term == 2 ? 1u : first);
            }
          }
        }
        umma_commit(empty_bar + stage);  // frees the smem slot when these MMAs have read it
      }
      __syncwarp();
      if (++stage == kStages) { stage = 0; phase ^= 1; }
    }
    if (elect_one()) umma_commit(tmem_full_bar);  // accumulator complete
    __syncwarp();
    TC_STAMP(6);
  } else {
    // ===== epilogue: warps 2..5 own TMEM lane quarters (warp % 4) =====
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    if constexpr (X3) {
      // ----- split warps: hi in place, lo behind the stage -----
      const int t = (warp - 2) * 32 + lane;
      int stage = 0;
      uint32_t phase = 0;
      for (int kb = kb_begin; kb < kb_end; ++kb) {
        mbar_wait(full_bar + stage, phase);
        const uint32_t base = smem_u32(smem + stage * L::kStageStride) + (uint32_t)t * 16u;
        constexpr int kVecs = (int)(L::kStageBytes / 16 / 128);   // 16-byte vectors per thread (stages are multiples of 4 KB)
        static_assert(L::kStageBytes % 2048 == 0, "stage size");
#pragma unroll 4
        for (int i = 0; i < kVecs; ++i) {
          const uint32_t addr = base + (uint32_t)i * 2048u;
          const float4 v = lds_f4(addr);
          float4 hi, lo;
          hi.x = rna_tf32(v.x); hi.y = rna_tf32(v.y); hi.z = rna_tf32(v.z); hi.w = rna_tf32(v.w);
          lo.x = rna_tf32(v.x - hi.x); lo.y = rna_tf32(v.y - hi.y); lo.z = rna_tf32(v.z - hi.z); lo.w = rna_tf32(v.w - hi.w);
          sts_f4(addr, hi);
          sts_f4(addr + L::kStageBytes, lo);
        }
        fence_proxy_async_smem();   // generic-proxy writes -> visible to the tensor core's (async proxy) operand reads
        __syncwarp();
        if (elect_one()) mbar_arrive(split_bar + stage);
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
    if (kb_end > kb_begin) {
      mbar_wait(tmem_full_bar, 0);
      tc_fence_after();
    }
    if (warp == 2) TC_STAMP(7);
    const uint32_t stage_u32 = smem_u32(smem);  // the pipeline stages are idle once the accumulator is complete
    const uint32_t rowtab_u32 = smem_u32(row_tab);
    constexpr uint32_t kPitch = P::kAccTiles * BN + 4;  // == L::kRedPitch with one accumulator tile
    // row-major problems leave through shared memory (coalesced write-out); the weight-gradient tiles of an unsplit
    // launch go from registers to their partial slab as 128-byte runs per thread
    constexpr bool kStaged = P::kRowMajor;
    if constexpr (P::kRowMajor) row_tab[row] = P::row_ptr(prm, tile, row);
#pragma unroll 1
    for (int cc = 0; cc < P::kAccTiles * BN; cc += 32) {
      const int acc = cc / BN, c0 = cc - acc * BN;  // accumulator tile (wgrad row-halo: one per tap), column inside it
      float v[32];
      if (kb_end > kb_begin) {
        tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)cc, v);
        if constexpr (X3) {   // + the accumulator of the small terms
          float v2[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(P::kTmemCols + cc), v2);
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] += v2[i];
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = 0.f;
      }
      if constexpr (!kStaged) {
        if (nsplit == 1) {
          P::store(prm, tile, row, c0, v, acc);
          continue;
        }
      }
      {
        const uint32_t dst = stage_u32 + (uint32_t)(row * kPitch + cc) * 4u;  // cc == c0 with one accumulator tile
#pragma unroll
        for (int i = 0; i < 32; i += 4) sts_f4(dst + i * 4, make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
      }
    }
    tc_fence_before();
    if (warp == 2) TC_STAMP(8);
    if constexpr (P::kRowMajor) {
      if (nsplit == 1) {
        // each warp writes out the 32 rows it staged itself: no cross-warp synchronisation. Rows go in batches: all
        // shared-memory and global loads of a batch are issued before its first store (a store to a generic pointer
        // would otherwise fence the loads of the next row behind it: measured 3.6 us for a 64 KB tile)
        __syncwarp();
        RowEpi<BN> epi;
        epi.init();
        constexpr int LPR = RowEpi<BN>::LPR, RPI = RowEpi<BN>::RPI, NCG = RowEpi<BN>::NCG;
        constexpr int U = NCG == 1 ? 4 : 2;   // rows in flight per lane
        const int lr = lane / LPR, lc = lane % LPR;
        P::epi_consts(prm, tile, epi, lc * 4);
#pragma unroll 1
        for (int rr = 0; rr < 32; rr += RPI * U) {
          float* rp[U];
          float4 val[U][NCG];
          typename P::Extras ex[U][NCG];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int r = quarter * 32 + rr + u * RPI + lr;
            rp[u] = lds_ptr(rowtab_u32 + r * 8);
#pragma unroll
            for (int g = 0; g < NCG; ++g) val[u][g] = lds_f4(stage_u32 + (uint32_t)(r * kPitch + (g * 32 + lc) * 4) * 4u);
          }
#pragma unroll
          for (int u = 0; u < U; ++u)
#pragma unroll
            for (int g = 0; g < NCG; ++g) ex[u][g] = P::load_extras(prm, tile, rp[u], (g * 32 + lc) * 4);
#pragma unroll
          for (int u = 0; u < U; ++u) {
            if (rp[u]) {
#pragma unroll
              for (int g = 0; g < NCG; ++g) P::emit4(prm, tile, epi, rp[u], (g * 32 + lc) * 4, g, val[u][g], ex[u][g]);
              epi.n += 1.f;
            }
          }
        }
        P::epi_finish(prm, tile, epi, wstat, reinterpret_cast<float*>(smem), (warp - 2) * 32 + lane);
      }
    }
    if (nsplit == 1) P::finish(prm, tile, (warp - 2) * 32 + lane);  // the 128 epilogue threads (wgrad: last CTA of a tile sums the splits)
    if (warp == 2) TC_STAMP(9);
  }
  if (P::kClusterSplit && nsplit > 1) {
    cluster_arrive();
    cluster_wait();  // every partial tile is in its CTA's shared memory
    if (warp == 2) TC_STAMP(10);
    RowEpi<BN> epi;
    epi.init();
    if (warp >= 2) {
      // kDynRedRows (wgrad): only the rows that hold output channels are reduced, spread over all CTAs of the cluster
      const int red_rows = P::kDynRedRows ? P::red_rows(prm, tile) : BLOCK_M;
      const int rows_per = P::kDynRedRows ? (red_rows + nsplit - 1) / nsplit : BLOCK_M / nsplit;
      const int t = (warp - 2) * 32 + lane;   // 0..127
      constexpr int kVecPerRow = P::kAccTiles * BN / 4;
      constexpr uint32_t kRedPitch = P::kAccTiles * BN + 4;
      const uint32_t red_base = smem_u32(smem);
      if constexpr (P::kRowMajor) P::epi_consts(prm, tile, epi, (t % kVecPerRow) * 4);   // this lane's columns never change
      // Two items per pass: every load of a pass (remote shared memory, the epilogue's global operands) is issued before
      // its first global store - a store to a generic pointer orders the next item's loads behind it, and this loop is
      // nothing but load latency (measured 2.2 - 4 us per kernel with one item per pass).
      const int total = rows_per * kVecPerRow;
      for (int idx0 = t; idx0 < total; idx0 += 256) {
        int rr[2], cc[2];
        bool ok[2];
        float* row_out[2] = {nullptr, nullptr};
        typename P::Extras ex[2] = {};
        float4 pv[2][8];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int idx = idx0 + u * 128;
          rr[u] = rank * rows_per + idx / kVecPerRow;
          cc[u] = (idx % kVecPerRow) * 4;
          ok[u] = idx < total && !(P::kDynRedRows && rr[u] >= red_rows);
          if (ok[u]) {
            const uint32_t addr = red_base + (uint32_t)(rr[u] * kRedPitch + cc[u]) * 4u;
            if constexpr (P::kRowMajor) {
              row_out[u] = lds_ptr(smem_u32(row_tab) + rr[u] * 8);
              ex[u] = P::load_extras(prm, tile, row_out[u], cc[u]);   // in flight together with the remote loads below
            }
#pragma unroll
            for (int s2 = 0; s2 < 8; ++s2)
              if (s2 < nsplit) pv[u][s2] = ld_dsmem_f4(dsmem_addr(addr, (uint32_t)s2));
          }
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (!ok[u]) continue;
          float4 acc = pv[u][0];
#pragma unroll
          for (int s2 = 1; s2 < 8; ++s2)  // fixed order: deterministic
            if (s2 < nsplit) { acc.x += pv[u][s2].x; acc.y += pv[u][s2].y; acc.z += pv[u][s2].z; acc.w += pv[u][s2].w; }
          if constexpr (P::kRowMajor) {
            // (a split launch has at most 128 columns: one float4 column group per lane, every row seen once per lane)
            if (row_out[u]) {
              P::emit4(prm, tile, epi, row_out[u], cc[u], 0, acc, ex[u]);
              epi.n += 1.f;
            }
          } else {
            P::store4(prm, tile, rr[u], cc[u], acc);
          }
        }
      }
    }
    // nobody leaves while its shared memory may still be read: arrive once this CTA's remote reads have
    // landed in registers (the global stores above only consume registers), wait just before the exit
    if (warp == 2) TC_STAMP(11);
    cluster_arrive();
    // two-level split (wgrad): the last cluster that finishes a tile adds the clusters' partial tiles
    if (P::kClusterFinish && warp >= 2) P::finish_cluster(prm, tile, (warp - 2) * 32 + lane, rank, nsplit);
    cluster_wait();
    // column statistics: after the wait nobody reads this CTA's staging tile any more (the last CTA's reduction uses it as scratch)
    if constexpr (P::kRowMajor) {
      if (warp >= 2) P::epi_finish(prm, tile, epi, wstat, reinterpret_cast<float*>(smem), (warp - 2) * 32 + lane);
    }
  } else {
    __syncthreads();
  }
  if (warp == 2) TC_STAMP(12);
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<kTmemAlloc>(tmem_base);
    TC_STAMP(13);
  }
}

// ---- persistent variant: many small tiles ------------------------------------------------------------------------------
// A convolution whose output has many more 128-pixel tiles than the GPU has CTA slots (first layer: 2048 tiles, layer 1
// of the ResNet: 512) and few channels pays the per-CTA prologue (barrier init, TMEM allocation, descriptor fetch, the
// first L2/HBM round trip) and a serial load -> MMA -> write-out chain once per TILE, in ~1.7 waves. Here a CTA lives
// for the whole launch and walks tiles blockIdx.x, + gridDim.x, ...: the producer warp keeps the TMA ring full across
// tile boundaries, the MMA warp alternates between two TMEM accumulators, and the epilogue warps drain accumulator i
// (TMEM -> dedicated staging tile -> coalesced stores, statistics in registers across ALL tiles of the CTA: one partial
// per CTA) while the MMAs of tile i + 1 run. Row-major problems without split-K only.
// X3 (fp32-accurate form, see tc_kernel): four more warps (6-9) split every stage into its TF32 high / low parts - the
// epilogue warps are busy with the previous tile here - and each of the two accumulators has a second one for the small terms.
template <class P, bool X3 = false>
__global__ void __launch_bounds__(X3 ? kThreads + 128 : kThreads) tc_persistent_kernel(const __grid_constant__ CUtensorMap map_a,
                                                                                       const __grid_constant__ CUtensorMap map_b,
                                                                                       const typename P::Params prm, const int n_tiles) {
  constexpr int BN = P::BN;
  static_assert(P::kRowMajor && P::kAccTiles == 1 && P::kMmaN == BN && P::kTmemCols == BN,
                "persistent kernel: row-major, one accumulator tile of BN columns (the two accumulators are kAccW apart)");
  static_assert(!P::kRuntimeLbo, "persistent kernel: compile-time operand descriptors");
  using L = TcLayout<P, true, X3>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::kBarOffset + L::kOverRead);
  constexpr int kStages = L::kStages;
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* split_bar = empty_bar + kStages + 1;   // [kStages], X3 only
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(split_bar + (X3 ? kStages : 0));
  (void)split_bar;
  float** row_tab = reinterpret_cast<float**>(smem + ((L::kEpiOffset + 15) & ~15u));
  float* wstat = reinterpret_cast<float*>(row_tab + BLOCK_M);
  uint64_t* tmem_full_bar = reinterpret_cast<uint64_t*>(smem + L::kAccBarOffset);   // [2] full, [2] empty
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;
  constexpr int kAccW = X3 ? 2 * BN : BN;               // columns of one accumulator (X3: + the small-term accumulator)
  constexpr int kAccCols = 2 * kAccW < 32 ? 32 : 2 * kAccW;   // two accumulators (BN is a power of two >= 32)

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, 1);
      if constexpr (X3) mbar_init(split_bar + s, 4);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tmem_full_bar + a, 1);
      mbar_init(tmem_empty_bar + a, 4);   // one arrival per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<kAccCols>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_sync();

  if (warp == 0) {
    // ===== TMA producer: the ring runs across tile boundaries =====
    int stage = 0;
    uint32_t phase = 0;
    for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
      const typename P::Tile tile = P::tile_at(prm, ti);
      const uint32_t tx = P::tx_bytes(prm, tile);
      typename P::Iter it = P::iter_init(prm, tile, tile.kb_begin);
      for (int kb = tile.kb_begin; kb < tile.kb_end; ++kb) {
        mbar_wait(empty_bar + stage, phase ^ 1);
        const uint32_t a_dst = smem_u32(smem + stage * L::kStageStride);
        const uint32_t b_dst = a_dst + L::kABytes;
        if (elect_one()) {
          mbar_expect_tx(full_bar + stage, tx);
          P::load_a(prm, tile, it, &map_a, full_bar + stage, a_dst);
          P::load_b(prm, tile, it, &map_b, full_bar + stage, b_dst);
        }
        __syncwarp();
        P::iter_next(prm, tile, it);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: accumulator lt & 1 for the lt-th tile of this CTA =====
    constexpr uint32_t idesc = instr_desc_tf32<P::A_MAJOR, P::B_MAJOR, P::kMmaN>();
    int stage = 0;
    uint32_t phase = 0;
    int lt = 0;
    for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x, ++lt) {
      const typename P::Tile tile = P::tile_at(prm, ti);
      const int acc = lt & 1;
      if (lt >= 2) {   // the epilogue must have drained this accumulator's previous tile
        mbar_wait(tmem_empty_bar + acc, (uint32_t)(((lt >> 1) - 1) & 1));
        tc_fence_after();
      }
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * kAccW);
      for (int kb = tile.kb_begin; kb < tile.kb_end; ++kb) {
        mbar_wait((X3 ? split_bar : full_bar) + stage, phase);
        tc_fence_after();
        const uint32_t a_base = smem_u32(smem + stage * L::kStageStride);
        const uint32_t b_base = a_base + L::kABytes;
        if (elect_one()) {
#pragma unroll
          for (int j = 0; j < P::KR / UMMA_K; ++j) {
#pragma unroll
            for (int t = 0; t < P::kSubTiles; ++t) {
              const uint32_t a_sub = a_base + P::a_sub_offset(prm, t), b_sub = b_base + P::b_sub_offset(prm, t, L::kBTile);
              const uint32_t first = (kb > tile.kb_begin || t > 0 || j > 0) ? 1u : 0u;
#pragma unroll
              for (int term = 0; term < (X3 ? 3 : 1); ++term) {   // hi*hi | lo*hi, hi*lo into the small-term accumulator
                const uint32_t a_op = a_sub + (term == 1 ? L::kStageBytes : 0u), b_op = b_sub + (term == 2 ? L::kStageBytes : 0u);
                umma_tf32(d_tmem + (term > 0 ? (uint32_t)BN : 0u), operand_desc<P::A_MAJOR, (P::AROWS == 32 ? 0u : L::kChunk)>(a_op, j),
                          operand_desc<P::B_MAJOR, L::kBChunk>(b_op, j), idesc, term == 2 ? 1u : first);
              }
            }
          }
          umma_commit(empty_bar + stage);
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) umma_commit(tmem_full_bar + acc);
      __syncwarp();
    }
  } else if (warp >= 6) {
    // ===== split warps (X3): hi in place, lo behind the stage =====
    if constexpr (X3) {
      const int t = (warp - 6) * 32 + lane;
      int stage = 0;
      uint32_t phase = 0;
      for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
        const typename P::Tile tile = P::tile_at(prm, ti);
        for (int kb = tile.kb_begin; kb < tile.kb_end; ++kb) {
          mbar_wait(full_bar + stage, phase);
          const uint32_t base = smem_u32(smem + stage * L::kStageStride) + (uint32_t)t * 16u;
          constexpr int kVecs = (int)(L::kStageBytes / 16 / 128);
#pragma unroll 4
          for (int i = 0; i < kVecs; ++i) {
            const uint32_t addr = base + (uint32_t)i * 2048u;
            const float4 v = lds_f4(addr);
            float4 hi, lo;
            hi.x = rna_tf32(v.x); hi.y = rna_tf32(v.y); hi.z = rna_tf32(v.z); hi.w = rna_tf32(v.w);
            lo.x = rna_tf32(v.x - hi.x); lo.y = rna_tf32(v.y - hi.y); lo.z = rna_tf32(v.z - hi.z); lo.w = rna_tf32(v.w - hi.w);
            sts_f4(addr, hi);
            sts_f4(addr + L::kStageBytes, lo);
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (elect_one()) mbar_arrive(split_bar + stage);
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else {
    // ===== epilogue warps: drain accumulator lt & 1 while the next tile's MMAs run =====
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t stage_u32 = smem_u32(smem + L::kOutOffset);
    const uint32_t rowtab_u32 = smem_u32(row_tab);
    constexpr uint32_t kPitch = BN + 4;
    constexpr int LPR = RowEpi<BN>::LPR, RPI = RowEpi<BN>::RPI, NCG = RowEpi<BN>::NCG;
    constexpr int U = NCG == 1 ? 4 : 2;
    const int lr = lane / LPR, lc = lane % LPR;
    RowEpi<BN> epi;
    epi.init();
    typename P::Tile tile = P::tile_at(prm, blockIdx.x < (unsigned)n_tiles ? (int)blockIdx.x : 0);
    P::epi_consts(prm, tile, epi, lc * 4);
    int lt = 0;
    for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x, ++lt) {
      tile = P::tile_at(prm, ti);
      const int acc = lt & 1;
      mbar_wait(tmem_full_bar + acc, (uint32_t)((lt >> 1) & 1));
      tc_fence_after();
      row_tab[row] = P::row_ptr(prm, tile, row);   // (this warp finished reading the previous tile's entries)
#pragma unroll 1
      for (int cc = 0; cc < BN; cc += 32) {
        float v[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * kAccW + cc), v);
        if constexpr (X3) {
          float v2[32];
          tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * kAccW + BN + cc), v2);
#pragma unroll
          for (int i = 0; i < 32; ++i) v[i] += v2[i];
        }
        const uint32_t dst = stage_u32 + (uint32_t)(row * kPitch + cc) * 4u;
#pragma unroll
        for (int i = 0; i < 32; i += 4) sts_f4(dst + i * 4, make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
      }
      tc_fence_before();
      __syncwarp();
      if (elect_one()) mbar_arrive(tmem_empty_bar + acc);   // the accumulator is free for the tile after next
      __syncwarp();
#pragma unroll 1
      for (int rr = 0; rr < 32; rr += RPI * U) {
        float* rp[U];
        float4 val[U][NCG];
        typename P::Extras ex[U][NCG];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int r = quarter * 32 + rr + u * RPI + lr;
          rp[u] = lds_ptr(rowtab_u32 + r * 8);
#pragma unroll
          for (int g = 0; g < NCG; ++g) val[u][g] = lds_f4(stage_u32 + (uint32_t)(r * kPitch + (g * 32 + lc) * 4) * 4u);
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
          for (int g = 0; g < NCG; ++g) ex[u][g] = P::load_extras(prm, tile, rp[u], (g * 32 + lc) * 4);
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (rp[u]) {
#pragma unroll
            for (int g = 0; g < NCG; ++g) P::emit4(prm, tile, epi, rp[u], (g * 32 + lc) * 4, g, val[u][g], ex[u][g]);
            epi.n += 1.f;
          }
        }
      }
      __syncwarp();   // the staging rows and row pointers of this warp are free for the next tile
    }
    // one statistics partial per CTA, over all its tiles (a CTA without tiles contributes an empty one)
    P::epi_finish(prm, tile, epi, wstat, nullptr, (warp - 2) * 32 + lane);
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<kAccCols>(tmem_base);
  }
}

// ---- persistent variant for the BIG layers: 128 x 256 tiles, two 256-column accumulators ---------------------------------
// The 128 x 256 kernels above run one tile per CTA at one CTA per SM (208 KB of ring): nothing overlaps a tile's epilogue,
// and the fused epilogues of the training step are not small - a dgrad tile that applies the ReLU mask and takes the
// BatchNorm-backward sums re-reads 128 KB of the BatchNorm's input and costs ~26 us next to a ~30 us main loop
// (VGG / ResNet-34 at 224 x 224, batch 128: conv 256 -> 256 at 56 x 56 fprop 804 us, the same contraction as fused dgrad
// 1186 us). Here a CTA lives for the whole launch, the MMA warp alternates between the two halves of TMEM (512 columns =
// 2 x 256), and the epilogue warps drain tile i while the MMAs of tile i + 1 run.
// There is no room for a 133 KB staging tile beside the ring, and none is needed: every epilogue warp passes its
// 32 rows through its own 32-column staging chunk (4.6 KB), eight chunks per tile, and writes 128-byte row segments -
// whole cache lines. Per-channel statistics: lanes that share columns are merged by shuffles, every warp keeps running
// sums of all channels over all its tiles in shared memory, and the CTA adds them to the statistic slot (fp64 atomics,
// kernels.cuh) once, at the end - so the launch needs the slot (the host falls back to the one-tile-per-CTA kernel
// without it) and at most 512 output channels. Three ring stages (144 KB) leave room for that.
// Tile order: column tile fastest, so the CTAs running at any moment share their activation tiles in L2.
template <class P>
struct WideLayout {
  using LS = SmemLayout<P::BN, P::AROWS, P::KR, P::kBSub, P::BKR>;
  static constexpr int kStages = 3;
  static constexpr uint32_t kStageBytes = LS::kStageBytes;
  static constexpr uint32_t kBarOffset = kStages * kStageBytes;
  static constexpr uint32_t kRowTabOffset = kBarOffset + 128;                    // 2 * kStages + 4 barriers, the TMEM slot
  static constexpr uint32_t kChunkPitch = 36;                                    // floats: 32 columns + 4 (bank spread)
  static constexpr uint32_t kChunkOffset = kRowTabOffset + BLOCK_M * 8;
  static constexpr uint32_t kChunkBytes = 32 * kChunkPitch * 4;                  // per epilogue warp
  // per-warp running statistics of every output channel over ALL tiles of the CTA: [4 warps][kMaxChannels][4 floats]
  static constexpr int kMaxChannels = 512;
  static constexpr uint32_t kAccOffset = kChunkOffset + 4 * kChunkBytes;
  static constexpr uint32_t kAccBytes = 4 * kMaxChannels * 16;
  static constexpr uint32_t kTotal = kAccOffset + kAccBytes + 1024;              // + manual alignment
  static_assert(kTotal <= 227u * 1024u, "shared memory");
  static_assert(2 * kStages + 4 <= 15, "barrier block");
};
// Lanes of a warp that hold the same columns (different rows of one warp instruction) are merged, and the lanes of row
// slot 0 fold the chunk's sums into the WARP's running statistics of those columns in shared memory (RowEpi<32>: 8 lanes
// per row, 4 row slots). Global atomics per warp and chunk were the first version: 2048 fp64 atomics per tile on a few
// hundred addresses serialise in L2 - the 256-channel fprop took 1033 us against 804 us for the one-tile-per-CTA kernel.
// `acc4`: this warp's [channels][4] block: EF_STATS (shift, m1, m2, n), EF_BNBWD (sum d, sum d*xh0, sum d*xh1, -).
template <int EF>
__device__ __forceinline__ void wide_fold_stats(RowEpi<32>& epi, float4* acc4, int lane, int col, int n_out) {
  if constexpr ((EF & (EF_STATS | EF_BNBWD)) == 0) return;
  constexpr bool stats = (EF & EF_STATS) != 0;
#pragma unroll
  for (int off = RowEpi<32>::LPR; off < 32; off <<= 1) {
    const float on = __shfl_xor_sync(0xffffffffu, epi.n, off);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float oa = __shfl_xor_sync(0xffffffffu, epi.a[0][q], off), ob = __shfl_xor_sync(0xffffffffu, epi.b[0][q], off),
                  oc = __shfl_xor_sync(0xffffffffu, epi.c[0][q], off);
      if (stats) {
        Moments m{epi.a[0][q], epi.b[0][q], epi.c[0][q], epi.n};
        Moments o{oa, ob, oc, on};
        if (lane & off) { o.merge(m); m = o; } else { m.merge(o); }
        epi.a[0][q] = m.s; epi.b[0][q] = m.m1; epi.c[0][q] = m.m2;
      } else {
        epi.a[0][q] += oa; epi.b[0][q] += ob; epi.c[0][q] += oc;
      }
    }
    epi.n += on;
  }
  if (lane < RowEpi<32>::LPR && col + 4 <= n_out) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float4 t = acc4[col + q];
      if (stats) {
        Moments m{t.x, t.y, t.z, t.w};
        m.merge(Moments{epi.a[0][q], epi.b[0][q], epi.c[0][q], epi.n});
        t = make_float4(m.s, m.m1, m.m2, m.n);
      } else {
        t.x += epi.a[0][q]; t.y += epi.b[0][q]; t.z += epi.c[0][q];
      }
      acc4[col + q] = t;
    }
  }
}
// end of the launch, the 128 epilogue threads (t): the four warps' statistics of a column are merged in warp order and
// added to the statistic slot - one fp64 atomic per sum, column and CTA
template <int EF>
__device__ __forceinline__ void wide_flush_stats(const EpiArgs& e, const float4* acc4_all, int max_channels, int t, int n_out) {
  if constexpr ((EF & (EF_STATS | EF_BNBWD)) == 0) return;
  constexpr bool stats = (EF & EF_STATS) != 0;
  for (int col = t; col < n_out; col += 128) {
    double* acc = e.stat_acc + col;
    if (stats) {
      Moments m{0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        const float4 v = acc4_all[w * max_channels + col];
        m.merge(Moments{v.x, v.y, v.z, v.w});
      }
      if (m.n > 0.f) {   // sums of (v - s), (v - s)^2 over n rows -> sums of v, v^2
        const double s_ = (double)m.s, m1 = (double)m.m1, m2 = (double)m.m2, n_ = (double)m.n;
        atomicAdd(acc, m1 + n_ * s_);
        atomicAdd(acc + kStatSlotChannels, m2 + 2.0 * s_ * m1 + n_ * s_ * s_);
      }
    } else {
      float r0 = 0.f, r1 = 0.f, r2 = 0.f;
#pragma unroll
      for (int w = 0; w < 4; ++w) {
        const float4 v = acc4_all[w * max_channels + col];
        r0 += v.x; r1 += v.y; r2 += v.z;
      }
      atomicAdd(acc, (double)r0);
      atomicAdd(acc + kStatSlotChannels, (double)r1);
      if (e.n_sets > 1) atomicAdd(acc + 2 * kStatSlotChannels, (double)r2);
    }
  }
}

template <class P, int EF>
__global__ void __launch_bounds__(kThreads) tc_wide_kernel(const __grid_constant__ CUtensorMap map_a,
                                                           const __grid_constant__ CUtensorMap map_b,
                                                           const typename P::Params prm, const int n_tiles, const int col_tiles) {
  constexpr int BN = P::BN;
  static_assert(BN == 256 && P::kRowMajor && P::kSubTiles == 1 && P::kAccTiles == 1, "wide kernel: 128 x 256 row-major tiles");
  using W = WideLayout<P>;
  using LS = typename W::LS;
  constexpr int kStages = W::kStages;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + W::kBarOffset);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tmem_full_bar = empty_bar + kStages;     // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;      // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
  float** row_tab = reinterpret_cast<float**>(smem + W::kRowTabOffset);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < kStages; ++s) {
      mbar_init(full_bar + s, 1);
      mbar_init(empty_bar + s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tmem_full_bar + a, 1);
      mbar_init(tmem_empty_bar + a, 4);   // one arrival per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_sync();

  // tile ti -> (pixel tile ti / col_tiles, column tile ti % col_tiles)
  auto tile_of = [&](int ti) {
    typename P::Tile t = P::tile_at(prm, ti / col_tiles);
    t.col0 = (ti % col_tiles) * BN;
    return t;
  };

  if (warp == 0) {
    // ===== TMA producer: the ring runs across tile boundaries =====
    int stage = 0;
    uint32_t phase = 0;
    for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x) {
      const typename P::Tile tile = tile_of(ti);
      const uint32_t tx = P::tx_bytes(prm, tile);
      typename P::Iter it = P::iter_init(prm, tile, tile.kb_begin);
      for (int kb = tile.kb_begin; kb < tile.kb_end; ++kb) {
        mbar_wait(empty_bar + stage, phase ^ 1);
        const uint32_t a_dst = smem_u32(smem + stage * W::kStageBytes);
        const uint32_t b_dst = a_dst + LS::kABytes;
        if (elect_one()) {
          mbar_expect_tx(full_bar + stage, tx);
          P::load_a(prm, tile, it, &map_a, full_bar + stage, a_dst);
          P::load_b(prm, tile, it, &map_b, full_bar + stage, b_dst);
        }
        __syncwarp();
        P::iter_next(prm, tile, it);
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: accumulator lt & 1 (TMEM columns 0..255 / 256..511) for the lt-th tile of this CTA =====
    constexpr uint32_t idesc = instr_desc_tf32<P::A_MAJOR, P::B_MAJOR, BN>();
    int stage = 0;
    uint32_t phase = 0;
    int lt = 0;
    for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x, ++lt) {
      const typename P::Tile tile = tile_of(ti);
      const int acc = lt & 1;
      if (lt >= 2) {   // the epilogue must have drained this accumulator's previous tile
        mbar_wait(tmem_empty_bar + acc, (uint32_t)(((lt >> 1) - 1) & 1));
        tc_fence_after();
      }
      const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
      for (int kb = tile.kb_begin; kb < tile.kb_end; ++kb) {
        mbar_wait(full_bar + stage, phase);
        tc_fence_after();
        const uint32_t a_base = smem_u32(smem + stage * W::kStageBytes);
        const uint32_t b_base = a_base + LS::kABytes;
        if (elect_one()) {
#pragma unroll
          for (int j = 0; j < P::KR / UMMA_K; ++j)
            umma_tf32(d_tmem, operand_desc<P::A_MAJOR, LS::kChunk>(a_base, j), operand_desc<P::B_MAJOR, LS::kBChunk>(b_base, j), idesc,
                      (kb > tile.kb_begin || j > 0) ? 1u : 0u);
          umma_commit(empty_bar + stage);
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) umma_commit(tmem_full_bar + acc);
      __syncwarp();
    }
  } else {
    // ===== epilogue warps: TMEM lane quarter (warp & 3); each warp stages and writes its own 32 rows, chunk by chunk =====
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const uint32_t chunk_u32 = smem_u32(smem + W::kChunkOffset + quarter * W::kChunkBytes);
    const uint32_t rowtab_u32 = smem_u32(row_tab);
    constexpr int LPR = RowEpi<32>::LPR, RPI = RowEpi<32>::RPI, U = 4;
    const int lr = lane / LPR, lc = lane % LPR;
    float4* acc4_all = reinterpret_cast<float4*>(smem + W::kAccOffset);
    float4* acc4 = acc4_all + quarter * W::kMaxChannels;        // this warp's running statistics
    if constexpr ((EF & (EF_STATS | EF_BNBWD)) != 0) {
      for (int i = lane; i < prm.n_out; i += 32) acc4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      __syncwarp();
    }
    int lt = 0;
    for (int ti = blockIdx.x; ti < n_tiles; ti += gridDim.x, ++lt) {
      const typename P::Tile tile = tile_of(ti);
      const int acc = lt & 1;
      row_tab[row] = P::row_ptr(prm, tile, row);   // (this warp's entries only; its previous tile is written out)
      mbar_wait(tmem_full_bar + acc, (uint32_t)((lt >> 1) & 1));
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < BN; cc += 32) {
        float v[32];
        tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BN + cc), v);
        if (cc + 32 == BN) {   // the last read of this accumulator: free it for the tile after next
          tc_fence_before();
          __syncwarp();
          if (elect_one()) mbar_arrive(tmem_empty_bar + acc);
        }
        __syncwarp();          // the previous chunk's rows have been read by every lane
        const uint32_t dst = chunk_u32 + (uint32_t)(lane * W::kChunkPitch) * 4u;
#pragma unroll
        for (int i = 0; i < 32; i += 4) sts_f4(dst + i * 4, make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]));
        __syncwarp();
        const int col = tile.col0 + cc + lc * 4;     // this lane's four columns of the chunk
        RowEpi<32> epi;
        epi.init();
        epi.template load_consts<EF>(prm.epi, col, prm.n_out);
#pragma unroll 1
        for (int rr = 0; rr < 32; rr += RPI * U) {
          float* rp[U];
          float4 val[U];
          typename RowEpi<32>::Extras ex[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int r = rr + u * RPI + lr;
            rp[u] = lds_ptr(rowtab_u32 + (quarter * 32 + r) * 8);
            val[u] = lds_f4(chunk_u32 + (uint32_t)(r * W::kChunkPitch + lc * 4) * 4u);
          }
#pragma unroll
          for (int u = 0; u < U; ++u) ex[u] = RowEpi<32>::template load_extras<EF>(prm.epi, prm.out, rp[u], col, prm.n_out);
#pragma unroll
          for (int u = 0; u < U; ++u) {
            if (rp[u]) {
              epi.template emit<EF>(prm.epi, rp[u], col, 0, val[u], ex[u], prm.n_out);
              epi.n += 1.f;
            }
          }
        }
        wide_fold_stats<EF>(epi, acc4, lane, col, prm.n_out);
      }
      __syncwarp();   // row pointers are free for the next tile
    }
    if constexpr ((EF & (EF_STATS | EF_BNBWD)) != 0) {
      asm volatile("bar.sync 1, 128;" ::: "memory");   // the four epilogue warps
      wide_flush_stats<EF>(prm.epi, acc4_all, W::kMaxChannels, (warp - 2) * 32 + lane, prm.n_out);
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc<512>(tmem_base);
  }
}

// ---- host: tensor maps ---------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

// dims[0] is the contiguous dimension; strides_elems[i] is the element stride of dims[i] (strides_elems[0] == 1)
static bool make_map(CUtensorMap* map, const float* base, int rank, const uint64_t* dims, const uint64_t* strides_elems,
                     const uint32_t* box, int major) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  if (reinterpret_cast<uintptr_t>(base) & 15) return false;
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bdim[5], estr[5];
  for (int i = 0; i < rank; ++i) {
    gdim[i] = dims[i];
    bdim[i] = box[i];
    estr[i] = 1;
    if (box[i] == 0 || box[i] > 256) return false;
    if (i > 0) {
      gstr[i - 1] = strides_elems[i] * sizeof(float);
      if (gstr[i - 1] % 16 != 0 || gstr[i - 1] >= (1ull << 40)) return false;
    }
  }
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, (cuuint32_t)rank, (void*)base, gdim, gstr, bdim, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE,
                  major == MAJOR_K ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

// fp32-accurate mode of the current call (set by the tc_* entry points): launch() then picks tc_kernel<P, true>
static thread_local bool g_x3 = false;
template <class P>
static constexpr bool x3_fits() { return TcLayout<P, false, true>::kFits; }

// Launches a tcgen05 kernel on the compute stream: sets its dynamic shared-memory size on the first call, launches
// (split_k_cluster: the `splits` CTAs that share a tile form one cluster along z; grid.z already counts them), checks and
// counts the launch.
template <auto Kernel, typename... Args>
static dfb_status launch_tc(const char* name, dim3 grid, unsigned threads, uint32_t smem, bool split_k_cluster, int splits,
                            const Args&... args) {
  static bool configured = false;
  if (!configured) {
    DFB_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = true;
  }
  if (split_k_cluster) {
    const cudaError_t e = launch_k_cluster(Kernel, grid, threads, smem, compute_stream(), dim3(1, 1, (unsigned)splits), args...);
    if (e != cudaSuccess) {
      cudaGetLastError();
      DFB_FAIL(DFB_ERR_RUNTIME, "%s cluster launch (splits %d) failed: %s", name, splits, cudaGetErrorString(e));
    }
  } else {
    launch_k(Kernel, grid, threads, smem, compute_stream(), args...);
  }
  DFB_LAUNCH_CHECK(name);
  g_tc_launches.fetch_add(1, std::memory_order_relaxed);
  return DFB_OK;
}
// one tile per CTA; grid.z already counts the splits
template <class P>
static dfb_status launch(const char* name, const CUtensorMap& ma, const CUtensorMap& mb, const typename P::Params& prm,
                         dim3 grid, int splits = 1) {
  if (g_x3) {
    if constexpr (x3_fits<P>()) {
      return launch_tc<tc_kernel<P, true>>(name, grid, kThreads, TcLayout<P, false, true>::kTotal, P::kClusterSplit, splits, ma, mb, prm);
    } else {
      DFB_FAIL(DFB_ERR_RUNTIME, "%s: this tile variant has no fp32-accurate form (host selection error)", name);
    }
  }
  return launch_tc<tc_kernel<P, false>>(name, grid, kThreads, TcLayout<P, false, false>::kTotal, P::kClusterSplit, splits, ma, mb, prm);
}

// fp32-accurate form only where two CTAs still share an SM (the grid is sized for that): the kernels without row halo
template <class P>
static constexpr bool x3_persistent_ok() {
  return P::kSubTiles == 1 && TcLayout<P, true, true>::kTotal <= 113u * 1024u;
}
template <class P>
static dfb_status launch_persistent(const char* name, const CUtensorMap& ma, const CUtensorMap& mb, const typename P::Params& prm,
                                    int n_tiles, unsigned ctas) {
  if (g_x3) {
    if constexpr (x3_persistent_ok<P>()) {
      return launch_tc<tc_persistent_kernel<P, true>>(name, dim3(ctas, 1, 1), kThreads + 128, TcLayout<P, true, true>::kTotal, false, 1, ma, mb,
                                                      prm, n_tiles);
    } else {
      DFB_FAIL(DFB_ERR_RUNTIME, "%s: no fp32-accurate persistent form of this variant (host selection error)", name);
    }
  }
  return launch_tc<tc_persistent_kernel<P, false>>(name, dim3(ctas, 1, 1), kThreads, TcLayout<P, true, false>::kTotal, false, 1, ma, mb, prm,
                                                   n_tiles);
}
// DFB_CONV_PERSISTENT=0 switches the persistent variant off (every tile its own CTA again)
static bool persistent_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("DFB_CONV_PERSISTENT");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

// DFB_CONV_WIDE=0 switches the persistent 128 x 256 kernel off (one tile per CTA again)
static bool wide_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("DFB_CONV_WIDE");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}
template <class P, int EF>
static dfb_status launch_wide(const char* name, const CUtensorMap& ma, const CUtensorMap& mb, const typename P::Params& prm, int n_tiles,
                              int col_tiles) {
  // whole waves: every CTA walks the same number of tiles (+-1)
  const int sms = sm_count();
  const int waves = (n_tiles + sms - 1) / sms;
  const unsigned ctas = (unsigned)((n_tiles + waves - 1) / waves);
  return launch_tc<tc_wide_kernel<P, EF>>(name, dim3(ctas, 1, 1), kThreads, WideLayout<P>::kTotal, false, 1, ma, mb, prm, n_tiles, col_tiles);
}

// Split-K factor (cluster size along z, a power of two <= 8): enough CTAs to occupy the machine, at least
// four k-blocks per CTA.
static int pick_splits(size_t base_ctas, int k_blocks) {
  int s = 1;
  while (s < 8 && base_ctas * (size_t)(s * 2) <= (size_t)sm_count() * 3 / 2 && k_blocks / (s * 2) >= 4) s *= 2;
  return s;
}

// =====================================================================================================
// Plain GEMM
// =====================================================================================================
struct GemmParams {
  float* C;
  const float* bias;
  int M, N, K, ldc, accumulate;
  int vec_ok;   // C and ldc allow 128-bit accesses
};
struct GemmTile {
  int m0, n0, kb_begin, kb_end;
};
template <int A_MAJ, int B_MAJ, int BN_>
struct GemmProblem {
  static constexpr int BN = BN_, A_MAJOR = A_MAJ, B_MAJOR = B_MAJ;
  static constexpr bool kClusterSplit = true;
  static constexpr int AROWS = BLOCK_M, KR = BLOCK_K, BKR = BLOCK_K, kSubTiles = 1, kBSub = 1, kAccTiles = 1, kTmemCols = BN_;
  __device__ static uint32_t a_sub_offset(const GemmParams&, int) { return 0; }
  __device__ static uint32_t b_sub_offset(const GemmParams&, int, uint32_t) { return 0; }
  static constexpr int kMmaN = BN_;
  static constexpr bool kRuntimeLbo = false;
  __device__ static uint32_t b_lbo(const GemmParams&) { return 0; }
  __device__ static uint32_t tx_bytes(const GemmParams&, const GemmTile&) { return SmemLayout<BN_>::kStageBytes; }
  __device__ static void finish(const GemmParams&, const GemmTile&, int) {}
  static constexpr bool kDynRedRows = false, kClusterFinish = false;
  __device__ static int red_rows(const GemmParams&, const GemmTile&) { return BLOCK_M; }
  __device__ static void finish_cluster(const GemmParams&, const GemmTile&, int, int, int) {}
  using Params = GemmParams;
  using Tile = GemmTile;
  static constexpr bool kRowMajor = true;
  __device__ static float* row_ptr(const Params& p, const Tile& t, int row) {
    const int m = t.m0 + row;
    return m < p.M ? p.C + (size_t)m * p.ldc : nullptr;
  }
  struct Extras { float4 old; };   // C's previous values when accumulating
  __device__ static Extras load_extras(const Params& p, const Tile& t, const float* row_out, int c) {
    Extras x;
    x.old = make_float4(0.f, 0.f, 0.f, 0.f);
    const int n = t.n0 + c;
    if (row_out && p.accumulate && p.vec_ok && n + 4 <= p.N) x.old = *reinterpret_cast<const float4*>(row_out + n);
    return x;
  }
  // four consecutive columns starting at tile column c of the row that starts at row_out
  __device__ static void emit4(const Params& p, const Tile& t, RowEpi<BN_>&, float* row_out, int c, int, float4 q, const Extras& x) {
    const int n = t.n0 + c;
    if (n >= p.N) return;
    float* dst = row_out + n;
    if (p.vec_ok && n + 4 <= p.N) {
      if (p.bias) { const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n)); q.x += b.x; q.y += b.y; q.z += b.z; q.w += b.w; }
      if (p.accumulate) { q.x += x.old.x; q.y += x.old.y; q.z += x.old.z; q.w += x.old.w; }
      *reinterpret_cast<float4*>(dst) = q;
      return;
    }
    const float v[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (n + i < p.N) {
        float x = v[i];
        if (p.bias) x += __ldg(p.bias + n + i);
        dst[i] = p.accumulate ? dst[i] + x : x;
      }
    }
  }
  __device__ static void epi_finish(const Params&, const Tile&, RowEpi<BN_>&, float*, float*, int) {}
  __device__ static void epi_consts(const Params&, const Tile&, RowEpi<BN_>&, int) {}
  __device__ static Tile tile(const Params& p) {
    return {(int)blockIdx.x * BLOCK_M, (int)blockIdx.y * BN, 0, (p.K + BLOCK_K - 1) / BLOCK_K};
  }
  struct Iter { int kb; };
  __device__ static Iter iter_init(const Params&, const Tile&, int kb) { return {kb}; }
  __device__ static void iter_next(const Params&, const Tile&, Iter& it) { ++it.kb; }
  __device__ static void load_a(const Params&, const Tile& t, const Iter& it, const CUtensorMap* m, uint64_t* bar, uint32_t dst) {
    const int kb = it.kb;
    if (A_MAJ == MAJOR_K) {
      tma_load_2d(dst, m, bar, kb * BLOCK_K, t.m0);
    } else {
#pragma unroll
      for (int j = 0; j < BLOCK_M / 32; ++j) tma_load_2d(dst + j * kChunkBytes, m, bar, t.m0 + j * 32, kb * BLOCK_K);
    }
  }
  __device__ static void load_b(const Params&, const Tile& t, const Iter& it, const CUtensorMap* m, uint64_t* bar, uint32_t dst) {
    const int kb = it.kb;
    if (B_MAJ == MAJOR_K) {
      tma_load_2d(dst, m, bar, kb * BLOCK_K, t.n0);
    } else {
#pragma unroll
      for (int j = 0; j < BN / 32; ++j) tma_load_2d(dst + j * kChunkBytes, m, bar, t.n0 + j * 32, kb * BLOCK_K);
    }
  }
};

template <int A_MAJ, int B_MAJ, int BN>
static dfb_status run_gemm(const float* A, const float* B, const GemmParams& prm, int lda, int ldb, bool* handled) {
  CUtensorMap ma, mb;
  bool ok;
  if (A_MAJ == MAJOR_K) {
    uint64_t d[2] = {(uint64_t)prm.K, (uint64_t)prm.M}, s[2] = {1, (uint64_t)lda};
    uint32_t b[2] = {BLOCK_K, BLOCK_M};
    ok = make_map(&ma, A, 2, d, s, b, A_MAJ);
  } else {
    uint64_t d[2] = {(uint64_t)prm.M, (uint64_t)prm.K}, s[2] = {1, (uint64_t)lda};
    uint32_t b[2] = {32, BLOCK_K};
    ok = make_map(&ma, A, 2, d, s, b, A_MAJ);
  }
  if (B_MAJ == MAJOR_K) {
    uint64_t d[2] = {(uint64_t)prm.K, (uint64_t)prm.N}, s[2] = {1, (uint64_t)ldb};
    uint32_t b[2] = {BLOCK_K, (uint32_t)BN};
    ok = ok && make_map(&mb, B, 2, d, s, b, B_MAJ);
  } else {
    uint64_t d[2] = {(uint64_t)prm.N, (uint64_t)prm.K}, s[2] = {1, (uint64_t)ldb};
    uint32_t b[2] = {32, BLOCK_K};
    ok = ok && make_map(&mb, B, 2, d, s, b, B_MAJ);
  }
  if (!ok) return DFB_OK;  // not representable as a tensor map -> FFMA path
  *handled = true;
  dim3 grid(cdiv(prm.M, BLOCK_M), cdiv(prm.N, BN), 1);
  const int k_blocks = (prm.K + BLOCK_K - 1) / BLOCK_K;
  int splits = BN >= 256 ? 1 : pick_splits((size_t)grid.x * grid.y, k_blocks);
  if (BN < 256 && g_x3)   // fp32-accurate mode: at most 128 k-blocks per TMEM accumulator (the partial tiles are added in true fp32)
    while (splits < 8 && k_blocks / splits > 128) splits *= 2;
  grid.z = (unsigned)splits;
  return launch<GemmProblem<A_MAJ, B_MAJ, BN>>("tc_gemm", ma, mb, prm, grid, splits);
}

template <int A_MAJ, int B_MAJ>
static dfb_status run_gemm_bn(const float* A, const float* B, const GemmParams& prm, int lda, int ldb, bool* handled) {
  if (prm.N <= 32) return run_gemm<A_MAJ, B_MAJ, 32>(A, B, prm, lda, ldb, handled);
  if (prm.N <= 64) return run_gemm<A_MAJ, B_MAJ, 64>(A, B, prm, lda, ldb, handled);
  // 128 x 256 tiles move a third fewer operand bytes per FLOP through L2 -> SM, which is what bounds the big
  // problems; only when they still fill the machine twice over
  if (prm.N > 128 && (size_t)cdiv(prm.M, BLOCK_M) * cdiv(prm.N, 256) >= (size_t)sm_count() * 2 && !(g_x3 && prm.K > 128 * BLOCK_K))
    return run_gemm<A_MAJ, B_MAJ, 256>(A, B, prm, lda, ldb, handled);
  return run_gemm<A_MAJ, B_MAJ, 128>(A, B, prm, lda, ldb, handled);
}


// =====================================================================================================
// Implicit-GEMM convolution: fprop, and dgrad for stride 1 (same contraction over dy, taps mirrored)
// =====================================================================================================
struct ConvParams {
  float* out;          // [pixels, n_out] channels-last
  int n_img, OH, OW;   // output pixel grid of one class (the whole output, or one parity class of it)
  int n_out;           // output channels of this contraction (Kout for fprop, C for dgrad)
  int R, cblks;        // taps per side; 32-channel blocks of the reduction channels (padded count / 32)
  int dh0, dw0, sgn;   // input row = oh * stride + dh0 + sgn * r   (stride 2: parity view)
  int stride, c_red;   // 1 or 2; reduction channel count (parity view offset)
  int ow_t, oh_t, n_t, tiles_w, tiles_h;
  // stride-2 dgrad: blockIdx.z = output parity class (ph, pw) of dx. Class (ph, pw) is a stride-1 contraction
  // over dy with the taps r = r0 + 2i, r0 = (ph + pad) & 1:  dx[2a+ph] += dy[a + d0 - i] * w[r0 + 2i],
  // d0 = (ph + pad - r0) / 2. par_pad >= 0 selects this mode; the output is then written at (2a+ph, 2b+pw)
  // of an image with 2*OH x 2*OW pixels.
  int par_pad;
  int splits;          // split-K cluster size along z
  EpiArgs epi;         // fused epilogue: addend, per-channel statistics (see RowEpi)
};
struct ConvTile {
  int n0, oh0, ow0, col0, kb_begin, kb_end;
  int ns, d0h, d0w, r0h, r0w, ph, pw;  // parity mode only
};
// WMODE selects where the weight operand comes from:
//   W_PACKED    : a packed copy Wt[n_out][tap][cp] made by weight_transform_kernel (weights stored (K,C,R,R))
//   W_KRSC_FPROP: the weights themselves, stored channels-last (K,R,R,C): K-major rows Wt[k][tap][c]
//   W_KRSC_DGRAD: the same buffer read as the MN-major operand Wd[(tap,k)][c] - no copy in either direction
enum { W_PACKED = 0, W_KRSC_FPROP = 1, W_KRSC_DGRAD = 2 };
// ROWS: "row halo" variant for 3x3 stride-1 convolutions whose 128-pixel tile is ow_t x oh_t pixels of ONE image
// (ow_t a multiple of 8). A k-block is (filter column s, 32-channel block): ONE TMA box brings the tile's pixels
// shifted by s with one halo row above and below ((oh_t + 2) * ow_t rows of 128 bytes), and the three taps
// (r, s), r = 0..2, are MMAs whose A descriptors start r * ow_t rows into that box - whole multiples of the 1024-byte
// swizzle atom, so the 128B swizzle stays consistent. The activations cross L2 -> SM 3.75-4.5 times per tile
// instead of 9 times; these layers (few channels, many pixels) are bound by exactly that traffic.
template <int BN_, int WMODE, bool ROWS = false, int EF = EF_NONE>
struct ConvProblem {
  static constexpr int BN = BN_, A_MAJOR = MAJOR_K, B_MAJOR = (WMODE == W_KRSC_DGRAD ? MAJOR_MN : MAJOR_K);
  static constexpr bool kClusterSplit = true;
  static constexpr int AROWS = ROWS ? 192 : BLOCK_M, KR = BLOCK_K, BKR = BLOCK_K, kSubTiles = ROWS ? 3 : 1, kBSub = kSubTiles;
  static constexpr int kAccTiles = 1, kTmemCols = BN_;
  using LayoutT = SmemLayout<BN_, AROWS, KR, kBSub, BKR>;
  __device__ static uint32_t b_sub_offset(const ConvParams&, int t, uint32_t b_tile) { return t * b_tile; }
  static constexpr int kMmaN = BN_;
  static constexpr bool kRuntimeLbo = false;
  __device__ static uint32_t b_lbo(const ConvParams&) { return 0; }
  __device__ static uint32_t a_sub_offset(const ConvParams& p, int t) {
    // tap r = t reads input row oh + dh0 + sgn * r; the box starts at the smallest of those rows
    return ROWS ? (uint32_t)((p.sgn > 0 ? t : 2 - t) * p.ow_t * 128) : 0u;
  }
  __device__ static uint32_t tx_bytes(const ConvParams& p, const ConvTile&) {
    return ROWS ? (uint32_t)((p.oh_t + 2) * p.ow_t * 128) + LayoutT::kBBytes : LayoutT::kStageBytes;
  }
  __device__ static void finish(const ConvParams&, const ConvTile&, int) {}
  static constexpr bool kDynRedRows = false, kClusterFinish = false;
  __device__ static int red_rows(const ConvParams&, const ConvTile&) { return BLOCK_M; }
  __device__ static void finish_cluster(const ConvParams&, const ConvTile&, int, int, int) {}
  using Params = ConvParams;
  using Tile = ConvTile;
  __device__ static Tile tile(const Params& p) { return tile_at(p, (int)blockIdx.x); }
  static constexpr bool kPersistentOk = BN_ == 32;   // (the staging tile of wider outputs does not fit beside the ring at two CTAs per SM)
  __device__ static Tile tile_at(const Params& p, int t) {
    int tw = t % p.tiles_w;
    t /= p.tiles_w;
    int th = t % p.tiles_h;
    int tn = t / p.tiles_h;
    Tile o{tn * p.n_t, th * p.oh_t, tw * p.ow_t, (int)blockIdx.y * BN, 0, (ROWS ? p.R : p.R * p.R) * p.cblks, 0, 0, 0, 0, 0, 0, 0};
    if (p.par_pad >= 0) {
      const int cls = (int)blockIdx.z / p.splits;  // blockIdx.z = class * splits + split
      o.ph = cls >> 1;
      o.pw = cls & 1;
      o.r0h = (o.ph + p.par_pad) & 1;
      o.r0w = (o.pw + p.par_pad) & 1;
      const int nr = o.r0h < p.R ? (p.R - o.r0h + 1) / 2 : 0;
      o.ns = o.r0w < p.R ? (p.R - o.r0w + 1) / 2 : 0;
      o.d0h = (o.ph + p.par_pad - o.r0h) / 2;
      o.d0w = (o.pw + p.par_pad - o.r0w) / 2;
      o.kb_end = nr * o.ns * p.cblks;
    }
    return o;
  }
  // k-block = (tap, 32-channel block); tap = (i, j): (r, s) of the filter, or the (i, j)-th tap of a parity class.
  // ROWS: k-block = (filter column j, 32-channel block), i unused.
  struct Iter { int i, j, cb, nj; };
  __device__ static Iter iter_init(const Params& p, const Tile& t, int kb) {
    const int tap = kb / p.cblks;
    if (ROWS) return {0, tap, kb - tap * p.cblks, p.R};
    const int nj = p.par_pad >= 0 ? max(t.ns, 1) : p.R;
    return {tap / nj, tap % nj, kb - tap * p.cblks, nj};
  }
  __device__ static void iter_next(const Params& p, const Tile&, Iter& it) {
    if (++it.cb == p.cblks) {
      it.cb = 0;
      if (++it.j == it.nj) { it.j = 0; ++it.i; }
    }
  }
  __device__ static void load_a(const Params& p, const Tile& t, const Iter& it, const CUtensorMap* m, uint64_t* bar, uint32_t dst) {
    if (ROWS) {
      const int row0 = p.sgn > 0 ? p.dh0 : p.dh0 - 2;  // smallest input-row offset among the three taps
      tma_load_4d(dst, m, bar, it.cb * 32, t.ow0 + p.dw0 + p.sgn * it.j, t.oh0 + row0, t.n0);
      return;
    }
    if (p.par_pad >= 0) {
      tma_load_4d(dst, m, bar, it.cb * 32, t.ow0 + t.d0w - it.j, t.oh0 + t.d0h - it.i, t.n0);
      return;
    }
    const int dh = p.dh0 + p.sgn * it.i, dw = p.dw0 + p.sgn * it.j;
    if (p.stride == 1) {
      tma_load_4d(dst, m, bar, it.cb * 32, t.ow0 + dw, t.oh0 + dh, t.n0);
    } else {
      // parity view (2C, W/2, 2, H/2, N): input row 2*oh + dh = 2*(oh + (dh >> 1)) + (dh & 1)
      tma_load_5d(dst, m, bar, (dw & 1) * p.c_red + it.cb * 32, t.ow0 + (dw >> 1), dh & 1, t.oh0 + (dh >> 1), t.n0);
    }
  }
  __device__ static void load_b_tap(const Params& p, const Tile& t, int tap, int cb, const CUtensorMap* m, uint64_t* bar, uint32_t dst) {
    if (WMODE == W_PACKED) {
      tma_load_2d(dst, m, bar, (tap * p.cblks + cb) * BLOCK_K, t.col0);
    } else if (WMODE == W_KRSC_FPROP) {
      tma_load_3d(dst, m, bar, cb * 32, tap, t.col0);           // rows = output channels, 32 input channels each
    } else {
#pragma unroll
      for (int j = 0; j < BN / 32; ++j)                          // rows = 32 k (output channels of the conv), 32 c each
        tma_load_3d(dst + j * kChunkBytes, m, bar, t.col0 + j * 32, tap, cb * 32);
    }
  }
  __device__ static void load_b(const Params& p, const Tile& t, const Iter& it, const CUtensorMap* m, uint64_t* bar, uint32_t dst) {
    if (ROWS) {
#pragma unroll
      for (int r = 0; r < 3; ++r) load_b_tap(p, t, r * p.R + it.j, it.cb, m, bar, dst + r * LayoutT::kBTile);
      return;
    }
    const int tap = p.par_pad >= 0 ? (t.r0h + 2 * it.i) * p.R + t.r0w + 2 * it.j : it.i * p.R + it.j;
    load_b_tap(p, t, tap, it.cb, m, bar, dst);
  }
  __device__ static float* row_ptr(const Params& p, const Tile& t, int row) {
    const int owi = row % p.ow_t;
    const int rest = row / p.ow_t;
    const int ohi = rest % p.oh_t, ni = rest / p.oh_t;
    const int n = t.n0 + ni;
    int oh = t.oh0 + ohi, ow = t.ow0 + owi;
    if (n >= p.n_img || oh >= p.OH || ow >= p.OW) return nullptr;
    int OHf = p.OH, OWf = p.OW;
    if (p.par_pad >= 0) {
      oh = 2 * oh + t.ph; ow = 2 * ow + t.pw;
      OHf *= 2; OWf *= 2;
    }
    return p.out + (((size_t)n * OHf + oh) * OWf + ow) * p.n_out;
  }
  static constexpr bool kRowMajor = true;
  using Extras = typename RowEpi<BN_>::Extras;
  __device__ static Extras load_extras(const Params& p, const Tile& t, const float* row_out, int c) {
    return RowEpi<BN_>::template load_extras<EF>(p.epi, p.out, row_out, t.col0 + c, p.n_out);
  }
  __device__ static void emit4(const Params& p, const Tile& t, RowEpi<BN_>& epi, float* row_out, int c, int g, const float4& q, const Extras& x) {
    epi.template emit<EF>(p.epi, row_out, t.col0 + c, g, q, x, p.n_out);
  }
  // c = the lane's first column inside the tile (column group 0)
  __device__ static void epi_consts(const Params& p, const Tile& t, RowEpi<BN_>& epi, int c) {
    epi.template load_consts<EF>(p.epi, t.col0 + c, p.n_out);
  }
  __device__ static void epi_finish(const Params& p, const Tile& t, RowEpi<BN_>& epi, float* wstat, float* scratch, int tid) {
    if constexpr ((EF & (EF_STATS | EF_BNBWD)) != 0)
      epi.finish(p.epi, wstat, scratch, tid, t.col0, p.n_out, (int)(blockIdx.x * gridDim.z + blockIdx.z), (int)(gridDim.x * gridDim.z),
                 gridDim.x * gridDim.y * gridDim.z);
  }
};

// =====================================================================================================
// wgrad: dWt[kout][tap][c] = sum over pixels of dy[pix][kout] * x[pix + tap][c]; both operands MN-major
// =====================================================================================================
struct WgradParams {
  float* partial;      // [splits][Kout][taps][Cp]
  float* dw;           // final gradient, (K,C,R,R) or (K,R,R,C); written by the last CTA of each tile when tickets != 0
  unsigned* tickets;   // one self-resetting arrival counter per output tile (null: separate reduction kernel)
  int krsc;
  int kr;              // output pixels per pipeline stage (32 or 128)
  int rows;            // row-halo variant: a CTA per filter column, three taps per stage
  int Kout, C, Cp, R, pad, stride;
  int n_img, OH, OW;
  int ow_t, oh_t, n_t, tiles_w, tiles_h, pix_blocks, blocks_per_split, ctiles;
  int csize, groups;   // WgradClusterProblem: CTAs per cluster (split of one group's pixels), groups of pixels (global partials)
};
struct WgradTile {
  int m0, tap, c0, kb_begin, kb_end;
  int a_chunks;  // 32-row chunks of the dy tile that hold real output channels (the rest is never loaded)
};
// AROWS_: rows of the dy tile that are loaded (32 / 64 / 128 >= output channels of the tile). KR_: output pixels per
// pipeline stage: 32, or 128 for the small-channel layers, whose 8 KB stages are otherwise all barrier hand-offs
// ROWS_ (row-halo variant; 3x3, stride 1, KR_ = 128 pixels = ow_t x oh_t of one image, ow_t a multiple of 8): a CTA
// owns a filter COLUMN s instead of a tap. Per stage ONE TMA box brings the x pixels of the block shifted by s with
// a halo row above and below, the dy chunk is loaded once, and the three taps (r, s) are MMAs into three
// accumulators (TMEM columns r * BN) whose B descriptors start r * ow_t rows into the box (multiples of 1024 bytes,
// a whole number of swizzle periods). Both operands cross L2 -> SM ~2.7 times less often than with a CTA per tap.
template <int BN_, int AROWS_, int KR_, bool ROWS_ = false>
struct WgradProblem {
  static constexpr int BN = BN_, A_MAJOR = MAJOR_MN, B_MAJOR = MAJOR_MN, AROWS = AROWS_, KR = KR_;
  static constexpr int BKR = ROWS_ ? 192 : KR_;       // rows of the x chunk: (oh_t + 2) * ow_t <= 192 with the halo
  static constexpr uint32_t kChunkW = KR_ * 128;
  static constexpr uint32_t kChunkB = BKR * 128;
  // row-halo: the three taps are the three 32-wide chunks of ONE N = 3 * BN operand (chunk stride = ow_t rows), so
  // a k-step is one MMA, not three (with N = 32 the MMA issue latency, not the math, is what a k-step costs)
  static constexpr int kSubTiles = 1, kBSub = 1;
  static constexpr int kAccTiles = ROWS_ ? 3 : 1, kMmaN = ROWS_ ? 3 * BN_ : BN_;
  static constexpr int kTmemCols = ROWS_ ? (BN_ * 3 <= 128 ? 128 : (BN_ * 3 <= 256 ? 256 : 512)) : BN_;
  static constexpr bool kRuntimeLbo = ROWS_;
  static_assert(!ROWS_ || BN_ == 32, "the row-halo wgrad addresses taps as operand chunks: one 32-wide chunk per tap");
  using LayoutT = SmemLayout<BN_, AROWS_, KR_, kBSub, BKR>;
  __device__ static uint32_t a_sub_offset(const WgradParams&, int) { return 0; }
  __device__ static uint32_t b_sub_offset(const WgradParams&, int, uint32_t) { return 0; }
  __device__ static uint32_t b_lbo(const WgradParams& p) { return (uint32_t)(p.ow_t * 128); }
  static constexpr bool kClusterSplit = false, kDynRedRows = false, kClusterFinish = false, kRowMajor = false;
  __device__ static void store4(const WgradParams&, const WgradTile&, int, int, const float4&) {}
  __device__ static float* row_ptr(const WgradParams&, const WgradTile&, int) { return nullptr; }
  struct Extras {};
  __device__ static Extras load_extras(const WgradParams&, const WgradTile&, const float*, int) { return Extras{}; }
  __device__ static void emit4(const WgradParams&, const WgradTile&, RowEpi<BN_>&, float*, int, int, const float4&, const Extras&) {}
  __device__ static void epi_finish(const WgradParams&, const WgradTile&, RowEpi<BN_>&, float*, float*, int) {}
  __device__ static void epi_consts(const WgradParams&, const WgradTile&, RowEpi<BN_>&, int) {}
  __device__ static int red_rows(const WgradParams&, const WgradTile&) { return BLOCK_M; }
  __device__ static void finish_cluster(const WgradParams&, const WgradTile&, int, int, int) {}
  using Params = WgradParams;
  using Tile = WgradTile;
  __device__ static Tile tile(const Params& p) {
    const int tap = blockIdx.y / p.ctiles, ct = blockIdx.y - tap * p.ctiles;
    const int b0 = blockIdx.z * p.blocks_per_split;
    const int m0 = (int)blockIdx.x * BLOCK_M;
    return {m0, tap, ct * BN, b0, min(p.pix_blocks, b0 + p.blocks_per_split), min(AROWS / 32, (p.Kout - m0 + 31) / 32)};
  }
  // rows of the accumulator beyond Kout multiply whatever the idle part of the stage holds; they are never stored
  __device__ static uint32_t tx_bytes(const Params& p, const Tile& t) {
    return t.a_chunks * kChunkW + (ROWS_ ? (uint32_t)((BN / 32) * (p.oh_t + 2) * p.ow_t * 128) : LayoutT::kBBytes);
  }
  // k-block = a block of 32 output pixels (tw, th, tn); the tap offset is fixed per CTA
  struct Iter { int tw, th, tn, dh, dw; };
  __device__ static Iter iter_init(const Params& p, const Tile& t, int kb) {
    const int tw = kb % p.tiles_w;
    kb /= p.tiles_w;
    const int r = t.tap / p.R, s = t.tap - r * p.R;
    if (ROWS_) return {tw, kb % p.tiles_h, kb / p.tiles_h, -p.pad, t.tap - p.pad};  // t.tap is the filter column here
    return {tw, kb % p.tiles_h, kb / p.tiles_h, r - p.pad, s - p.pad};
  }
  __device__ static void iter_next(const Params& p, const Tile&, Iter& it) {
    if (++it.tw == p.tiles_w) {
      it.tw = 0;
      if (++it.th == p.tiles_h) { it.th = 0; ++it.tn; }
    }
  }
  __device__ static void load_a(const Params& p, const Tile& t, const Iter& it, const CUtensorMap* m, uint64_t* bar, uint32_t dst) {
    const int n0 = it.tn * p.n_t, oh0 = it.th * p.oh_t, ow0 = it.tw * p.ow_t;
#pragma unroll
    for (int j = 0; j < AROWS / 32; ++j)
      if (j < t.a_chunks) tma_load_4d(dst + j * kChunkW, m, bar, t.m0 + j * 32, ow0, oh0, n0);
  }
  __device__ static void load_b(const Params& p, const Tile& t, const Iter& it, const CUtensorMap* m, uint64_t* bar, uint32_t dst) {
    const int n0 = it.tn * p.n_t, oh0 = it.th * p.oh_t, ow0 = it.tw * p.ow_t;
    const int dh = it.dh, dw = it.dw;
#pragma unroll
    for (int j = 0; j < BN / 32; ++j) {
      if (p.stride == 1)
        tma_load_4d(dst + j * kChunkB, m, bar, t.c0 + j * 32, ow0 + dw, oh0 + dh, n0);
      else
        tma_load_5d(dst + j * kChunkB, m, bar, (dw & 1) * p.C + t.c0 + j * 32, ow0 + (dw >> 1), dh & 1, oh0 + (dh >> 1), n0);
    }
  }
  // filter tap an accumulator tile belongs to: the CTA's tap, or (r = acc, s = CTA's column) in the row-halo variant
  __device__ static int tap_of(const Params& p, const Tile& t, int acc) { return ROWS_ ? acc * p.R + t.tap : t.tap; }
  __device__ static void store(const Params& p, const Tile& t, int row, int c0, const float (&v)[32], int acc) {
    const int k = t.m0 + row;
    if (k >= p.Kout) return;
    const int taps = p.R * p.R;
    float* dst = p.partial + (((size_t)blockIdx.z * p.Kout + k) * taps + tap_of(p, t, acc)) * p.Cp + t.c0 + c0;
#pragma unroll
    for (int i = 0; i < 32; i += 4) *reinterpret_cast<float4*>(dst + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
  }
  // The last of the gridDim.z CTAs that share this output tile adds their partial tiles in split order
  // (deterministic) and writes the gradient in the weight's layout. Called by the 128 epilogue threads.
  __device__ static void finish(const Params& p, const Tile& t, int tid) {
    if (!p.tickets) return;
    __shared__ int s_last;
    __threadfence();
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (tid == 0) {
      unsigned* ticket = p.tickets + blockIdx.x + gridDim.x * blockIdx.y;
      const unsigned arrived = atomicAdd(ticket, 1u);
      s_last = arrived == gridDim.z - 1;
      if (s_last) *ticket = 0;
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (!s_last) return;
    __threadfence();
    const int taps = p.R * p.R;
    const int rows = min(BLOCK_M, p.Kout - t.m0);
    constexpr int kVec = BN / 4;
    const size_t slab = (size_t)p.Kout * taps * p.Cp;
    const int splits = gridDim.z;
    for (int idx = tid; idx < kAccTiles * rows * kVec; idx += 128) {
      const int acc_tile = idx / (rows * kVec), rem = idx - acc_tile * rows * kVec;
      const int tap = tap_of(p, t, acc_tile);
      const int k = t.m0 + rem / kVec;
      const int c = t.c0 + (rem % kVec) * 4;
      if (c >= p.C) continue;  // channel padding
      const float4* src = reinterpret_cast<const float4*>(p.partial + ((size_t)k * taps + tap) * p.Cp + c);
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      int z = 0;
      for (; z + 4 <= splits; z += 4) {
        float4 q[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) q[u] = __ldcg(src + (size_t)(z + u) * (slab / 4));
#pragma unroll
        for (int u = 0; u < 4; ++u) { acc.x += q[u].x; acc.y += q[u].y; acc.z += q[u].z; acc.w += q[u].w; }
      }
      for (; z < splits; ++z) {
        const float4 q = __ldcg(src + (size_t)z * (slab / 4));
        acc.x += q.x; acc.y += q.y; acc.z += q.z; acc.w += q.w;
      }
      if (p.krsc) {
        *reinterpret_cast<float4*>(p.dw + ((size_t)k * taps + tap) * p.C + c) = acc;
      } else {
        float* o = p.dw + ((size_t)k * p.C + c) * taps + tap;
        o[0] = acc.x; o[taps] = acc.y; o[2 * taps] = acc.z; o[3 * taps] = acc.w;
      }
    }
  }
};

// Two-level pixel split for wgrad. The pixel blocks are cut into `groups` ranges and each range is shared by the
// `csize` (2..8) CTAs of a thread-block cluster along z: the cluster sums its CTAs' accumulators through distributed
// shared memory (the kernel's split-K path) and only ONE partial tile per group reaches global memory - none at all
// with a single group, where the cluster writes dW directly. With several groups the last cluster to finish a tile adds
// the groups' partial tiles in group order, each of its CTAs for its own rows (one arrival counter per tile and rank).
// Against one partial per CTA plus a separate reduction kernel this is `csize` times fewer partial bytes and one
// launch less on the critical path of the backward pass (the wgrad chain on the side stream).
template <int BN_, int AROWS_, int KR_, bool ROWS_ = false>
struct WgradClusterProblem : WgradProblem<BN_, AROWS_, KR_, ROWS_> {
  using Base = WgradProblem<BN_, AROWS_, KR_, ROWS_>;
  using Params = WgradParams;
  using Tile = WgradTile;
  static constexpr bool kClusterSplit = true, kDynRedRows = true, kClusterFinish = true;
  static constexpr int kCols = Base::kAccTiles * BN_;
  static_assert(BN_ < 256, "the 128 x 256 wgrad tiles keep one partial per CTA");
  static_assert((uint32_t)BLOCK_M * (kCols + 4) * 4 <= Base::LayoutT::kBarOffset, "partial tile does not fit the pipeline stages");
  __device__ static Tile tile(const Params& p) {
    const int tap = blockIdx.y / p.ctiles, ct = blockIdx.y - tap * p.ctiles;
    const int b0 = ((int)blockIdx.z / p.csize) * p.blocks_per_split;  // the kernel cuts [b0, b1) by cluster rank
    const int m0 = (int)blockIdx.x * BLOCK_M;
    return {m0, tap, ct * BN_, b0, min(p.pix_blocks, b0 + p.blocks_per_split), min(AROWS_ / 32, (p.Kout - m0 + 31) / 32)};
  }
  __device__ static int red_rows(const Params& p, const Tile& t) { return min(BLOCK_M, p.Kout - t.m0); }
  __device__ static void finish(const Params&, const Tile&, int) {}
  __device__ static void write_dw(const Params& p, int k, int tap, int c, const float4& q) {
    const int taps = p.R * p.R;
    if (p.krsc) {
      *reinterpret_cast<float4*>(p.dw + ((size_t)k * taps + tap) * p.C + c) = q;
    } else {
      float* o = p.dw + ((size_t)k * p.C + c) * taps + tap;
      o[0] = q.x; o[taps] = q.y; o[2 * taps] = q.z; o[3 * taps] = q.w;
    }
  }
  // `col` counts over the accumulator tiles of the CTA (row-halo: three taps of BN channels each)
  __device__ static void store4(const Params& p, const Tile& t, int row, int col, const float4& q) {
    const int acc = col / BN_, c = t.c0 + col - acc * BN_;
    if (c >= p.C) return;  // channel padding
    const int k = t.m0 + row, tap = Base::tap_of(p, t, acc);
    if (p.groups == 1) {
      write_dw(p, k, tap, c, q);
    } else {
      const int g = (int)blockIdx.z / p.csize;
      *reinterpret_cast<float4*>(p.partial + (((size_t)g * p.Kout + k) * (p.R * p.R) + tap) * p.Cp + c) = q;
    }
  }
  __device__ static void finish_cluster(const Params& p, const Tile& t, int tid, int rank, int nsplit) {
    if (p.groups == 1) return;
    __shared__ int s_last_group;
    __threadfence();
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (tid == 0) {
      unsigned* ticket = p.tickets + (blockIdx.x + gridDim.x * blockIdx.y) * 8 + rank;
      const unsigned arrived = atomicAdd(ticket, 1u);
      s_last_group = arrived == (unsigned)p.groups - 1;
      if (s_last_group) *ticket = 0;
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (!s_last_group) return;
    __threadfence();
    const int taps = p.R * p.R;
    const int rows = red_rows(p, t), rows_per = (rows + nsplit - 1) / nsplit;
    const int r0 = rank * rows_per, nrows = min(rows, r0 + rows_per) - r0;
    constexpr int kVec = kCols / 4;
    const size_t slab4 = (size_t)p.Kout * taps * p.Cp / 4;
    for (int idx = tid; idx < nrows * kVec; idx += 128) {
      const int col = (idx % kVec) * 4, acc = col / BN_, c = t.c0 + col - acc * BN_;
      if (c >= p.C) continue;
      const int k = t.m0 + r0 + idx / kVec, tap = Base::tap_of(p, t, acc);
      const float4* src = reinterpret_cast<const float4*>(p.partial + ((size_t)k * taps + tap) * p.Cp + c);
      float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
      int g = 0;
      for (; g + 4 <= p.groups; g += 4) {
        float4 q[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) q[u] = __ldcg(src + (size_t)(g + u) * slab4);
#pragma unroll
        for (int u = 0; u < 4; ++u) { sum.x += q[u].x; sum.y += q[u].y; sum.z += q[u].z; sum.w += q[u].w; }
      }
      for (; g < p.groups; ++g) {
        const float4 q = __ldcg(src + (size_t)g * slab4);
        sum.x += q.x; sum.y += q.y; sum.z += q.z; sum.w += q.w;
      }
      write_dw(p, k, tap, c, sum);
    }
  }
};

// ---- small helper kernels -----------------------------------------------------------------------------
// Wt[k][tap][cp] = w[k][c][tap] (DGRAD = false)   or   Wd[c][tap][kp] = w[k][c][tap] (DGRAD = true); zero padding
template <bool DGRAD>
__global__ void __launch_bounds__(256) weight_transform_kernel(const float* __restrict__ w, float* __restrict__ out, int K, int C,
                                                              int taps, int inner_pad) {
  pdl_sync();
  const int rows = DGRAD ? C : K;
  size_t total = (size_t)rows * taps * inner_pad;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int in = (int)(i % inner_pad);
    size_t t = i / inner_pad;
    int tap = (int)(t % taps);
    int row = (int)(t / taps);
    int k = DGRAD ? in : row, c = DGRAD ? row : in;
    out[i] = (k < K && c < C) ? __ldg(w + ((size_t)k * C + c) * taps + tap) : 0.f;
  }
}
// dW[k][c][tap] (KCRS) or dW[k][tap][c] (KRSC) = sum_z partial[z][k][tap][c]. LPO lanes share one output: lane l adds the
// splits l, l + LPO, ... and a shuffle tree (fixed order) adds the lanes - with one thread per output the first layer's
// 864 outputs x 128 splits were a 34 us chain of dependent loads at the very end of the backward pass.
template <int LPO>
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw, int splits,
                                                          int K, int C, int Cp, int taps, int krsc) {
  pdl_sync();
  const size_t total = (size_t)K * C * taps;
  const size_t slab = (size_t)K * taps * Cp;
  const size_t stride = (size_t)gridDim.x * blockDim.x / LPO;
  const int l = threadIdx.x % LPO;
  // (every lane of a group runs the same trip count: the shuffles below are warp-convergent)
  for (size_t i0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / LPO; i0 < (total + stride - 1) / stride * stride; i0 += stride) {
    const bool ok = i0 < total;
    const size_t i = ok ? i0 : 0;
    int tap, c, k;
    if (krsc) {
      c = (int)(i % C);
      size_t t = i / C;
      tap = (int)(t % taps);
      k = (int)(t / taps);
    } else {
      tap = (int)(i % taps);
      size_t t = i / taps;
      c = (int)(t % C);
      k = (int)(t / C);
    }
    const float* src = partial + ((size_t)k * taps + tap) * Cp + c;
    float acc = 0.f;
    if (ok) {
      int z = l;
      for (; z + 3 * LPO < splits; z += 4 * LPO) {
        const float q0 = __ldcg(src + (size_t)z * slab), q1 = __ldcg(src + (size_t)(z + LPO) * slab),
                    q2 = __ldcg(src + (size_t)(z + 2 * LPO) * slab), q3 = __ldcg(src + (size_t)(z + 3 * LPO) * slab);
        acc += q0; acc += q1; acc += q2; acc += q3;
      }
      for (; z < splits; z += LPO) acc += __ldcg(src + (size_t)z * slab);
    }
#pragma unroll
    for (int off = LPO / 2; off > 0; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    if (ok && l == 0) dw[i] = acc;
  }
}

static int pow2_ceil(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}
static void pixel_tile(int pixels_per_tile, int OH, int OW, int* ow_t, int* oh_t, int* n_t) {
  *ow_t = std::min(pixels_per_tile, pow2_ceil(OW));
  *oh_t = std::min(pixels_per_tile / *ow_t, pow2_ceil(OH));
  *n_t = pixels_per_tile / (*ow_t * *oh_t);
}

// activation map for a tile of `pix` pixels: stride 1 -> 4-d (C, W, H, N); stride 2 -> 5-d parity view
static bool make_act_map(CUtensorMap* map, const float* base, int N, int H, int W, int C, int stride, int ow_t, int oh_t,
                         int n_t, int major) {
  if (stride == 1) {
    uint64_t d[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    uint64_t s[4] = {1, (uint64_t)C, (uint64_t)W * C, (uint64_t)H * W * C};
    uint32_t b[4] = {32, (uint32_t)ow_t, (uint32_t)oh_t, (uint32_t)n_t};
    return make_map(map, base, 4, d, s, b, major);
  }
  uint64_t d[5] = {(uint64_t)2 * C, (uint64_t)W / 2, 2, (uint64_t)H / 2, (uint64_t)N};
  uint64_t s[5] = {1, (uint64_t)2 * C, (uint64_t)W * C, (uint64_t)2 * W * C, (uint64_t)H * W * C};
  uint32_t b[5] = {32, (uint32_t)ow_t, 1, (uint32_t)oh_t, (uint32_t)n_t};
  return make_map(map, base, 5, d, s, b, major);
}

// The epilogue work of a convolution (EF_* flags) -> the EF template argument, for every kernel family. Only the
// combinations the host asks for are instantiated: fprop + statistics, dgrad + addend / BatchNorm-backward sums (with or
// without the ReLU mask) / both, with channels-last weights. conv_like refuses the others (fprop with an addend or
// BatchNorm-backward sums, dgrad with statistics, any fused epilogue with packed weights); should one arrive anyway, the
// flags a pass has no variant for are dropped: fprop keeps only EF_STATS, dgrad ignores EF_STATS, packed weights get
// EF_NONE.
template <int WMODE, class F>
static dfb_status with_conv_epilogue(int ef, F&& launch_ef) {
  using std::integral_constant;
  if constexpr (WMODE == W_KRSC_FPROP) {
    if (ef & EF_STATS) return launch_ef(integral_constant<int, EF_STATS>());
  } else if constexpr (WMODE == W_KRSC_DGRAD) {
    switch (ef & ~EF_STATS) {
      case EF_BNBWD | EF_RELU | EF_ADDEND: return launch_ef(integral_constant<int, EF_BNBWD | EF_RELU | EF_ADDEND>());
      case EF_BNBWD | EF_RELU: return launch_ef(integral_constant<int, EF_BNBWD | EF_RELU>());
      case EF_BNBWD | EF_ADDEND: return launch_ef(integral_constant<int, EF_BNBWD | EF_ADDEND>());
      case EF_BNBWD: return launch_ef(integral_constant<int, EF_BNBWD>());
      case EF_ADDEND: return launch_ef(integral_constant<int, EF_ADDEND>());
      default: break;
    }
  }
  return launch_ef(integral_constant<int, EF_NONE>());
}

template <int BN, int WMODE, bool ROWS = false>
static dfb_status run_conv(const char* name, const CUtensorMap& ma, const float* wt, int n_out, int taps, int cp, int K, int C,
                           ConvParams prm, bool* handled) {
  CUtensorMap mb;
  bool ok;
  if (WMODE == W_PACKED) {
    uint64_t d[2] = {(uint64_t)taps * cp, (uint64_t)n_out}, s[2] = {1, (uint64_t)taps * cp};
    uint32_t b[2] = {BLOCK_K, (uint32_t)BN};
    ok = make_map(&mb, wt, 2, d, s, b, MAJOR_K);
  } else {
    uint64_t d[3] = {(uint64_t)C, (uint64_t)taps, (uint64_t)K}, s[3] = {1, (uint64_t)C, (uint64_t)taps * C};
    uint32_t b[3] = {32, 1, (uint32_t)(WMODE == W_KRSC_FPROP ? BN : 32)};
    ok = make_map(&mb, wt, 3, d, s, b, WMODE == W_KRSC_FPROP ? MAJOR_K : MAJOR_MN);
  }
  if (!ok) return DFB_OK;
  *handled = true;
  int tiles_n = cdiv(prm.n_img, prm.n_t);
  const int classes = prm.par_pad >= 0 ? 4 : 1;
  dim3 grid((unsigned)(prm.tiles_w * prm.tiles_h * tiles_n), cdiv(n_out, BN), 1);
  // stride-2 dgrad classes hold about a quarter of the taps each
  const int kblocks = ROWS ? prm.R * prm.cblks : prm.R * prm.R * prm.cblks / (classes == 4 ? 4 : 1);
  prm.splits = BN >= 256 ? 1 : pick_splits((size_t)grid.x * grid.y * classes, kblocks > 0 ? kblocks : 1);
  if (BN < 256 && g_x3)
    while (prm.splits < 8 && kblocks * (ROWS ? 3 : 1) / prm.splits > 128) prm.splits *= 2;
  grid.z = (unsigned)(classes * prm.splits);
  float* part = nullptr;
  prm.epi.stat_acc = nullptr;
  if (prm.epi.stat_kind != EPI_NONE && prm.epi.lazy)   // the consumer kernel takes the sums from a statistic slot: no partials, no reduction kernel
    prm.epi.stat_acc = stat_slot_acquire(prm.epi.stat_out, prm.epi.stat_kind == EPI_BNBWD ? prm.epi.n_sets : 1, n_out);
  if (prm.epi.stat_kind != EPI_NONE && !prm.epi.stat_acc) {  // one partial per (pixel tile, class / split rank) + its row count
    const size_t partials = (size_t)grid.x * grid.z;
    dfb_status st = dfb_malloc(partials * 3 * n_out + partials, &part);
    if (st != DFB_OK) return st;
    prm.epi.stat_part = part;
    prm.epi.stat_cnt = part + partials * 3 * n_out;
  }
  const bool add = prm.epi.addend != nullptr;
  const int ef = (prm.epi.stat_kind == EPI_STATS ? EF_STATS : 0) | (add ? EF_ADDEND : 0) |
                 (prm.epi.stat_kind == EPI_BNBWD ? EF_BNBWD | (prm.epi.relu ? EF_RELU : 0) : 0);
  dfb_status st = DFB_OK;
  bool launched = false;
  // Many more tiles than CTA slots, one column tile, no split: CTAs that live for the whole launch (tc_persistent_kernel),
  // as many as balance the tiles over whole waves (512 tiles on 296 slots -> 256 CTAs with two tiles each)
  if constexpr (BN == 32 && WMODE != W_PACKED) {
    const size_t slots = (size_t)sm_count() * 2;
    if (persistent_enabled() && (!g_x3 || !ROWS) && classes == 1 && prm.splits == 1 && grid.y == 1 && (size_t)grid.x > slots) {
      const int n_tiles = (int)grid.x;
      const int waves = (int)((grid.x + slots - 1) / slots);
      const unsigned ctas = (unsigned)((n_tiles + waves - 1) / waves);
      if (part) {   // one partial per CTA instead of one per tile
        prm.epi.stat_cnt = part + (size_t)ctas * 3 * n_out;
      }
      grid = dim3(ctas, 1, 1);
      st = with_conv_epilogue<WMODE>(ef, [&](auto e) {
        return launch_persistent<ConvProblem<BN, WMODE, ROWS, decltype(e)::value>>(name, ma, mb, prm, n_tiles, ctas);
      });
      launched = true;
    }
  }
  // Big layers (128 x 256 tiles, hundreds of them): CTAs that live for the whole launch and overlap a tile's epilogue
  // with the next tile's MMAs (tc_wide_kernel). Statistics go to the statistic slot, so the call needs one.
  if constexpr (BN == 256 && !ROWS) {
    const int n_tiles = (int)(grid.x * grid.y), col_tiles = (int)grid.y;
    const bool slot_ok = prm.epi.stat_kind == EPI_NONE || prm.epi.stat_acc != nullptr;
    if (wide_enabled() && !g_x3 && classes == 1 && prm.splits == 1 && slot_ok && n_out <= 512 && (size_t)n_tiles >= (size_t)sm_count() * 2) {
      st = with_conv_epilogue<WMODE>(ef, [&](auto e) {
        return launch_wide<ConvProblem<BN, WMODE, ROWS, decltype(e)::value>, decltype(e)::value>(name, ma, mb, prm, n_tiles, col_tiles);
      });
      launched = true;
    }
  }
  if (!launched)
    st = with_conv_epilogue<WMODE>(ef, [&](auto e) { return launch<ConvProblem<BN, WMODE, ROWS, decltype(e)::value>>(name, ma, mb, prm, grid, prm.splits); });
  if (st == DFB_OK && part) {
    launch_k(epi_finalize_kernel, (unsigned)(n_out / 4), 128, 0, compute_stream(), (const float*)prm.epi.stat_part, (const float*)prm.epi.stat_cnt,
             (int)(grid.x * grid.z), n_out, prm.epi.stat_kind == EPI_STATS ? 1 : 0, prm.epi.stat_out);
    cudaError_t e = cudaGetLastError();
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (e != cudaSuccess) {
      dfb_free(part);
      DFB_FAIL(DFB_ERR_RUNTIME, "epi_finalize launch failed: %s", cudaGetErrorString(e));
    }
  }
  if (part) dfb_free(part);  // stream-ordered
  return st;
}
// row-halo variant (ConvProblem<.., ROWS = true>): n_out <= 128
template <int WMODE>
static dfb_status run_conv_rows(const char* name, const CUtensorMap& ma, const float* wt, int n_out, int taps, int cp, int K, int C,
                                const ConvParams& prm, bool* handled) {
  if (n_out <= 32) return run_conv<32, WMODE, true>(name, ma, wt, n_out, taps, cp, K, C, prm, handled);
  if (n_out <= 64) return run_conv<64, WMODE, true>(name, ma, wt, n_out, taps, cp, K, C, prm, handled);
  return run_conv<128, WMODE, true>(name, ma, wt, n_out, taps, cp, K, C, prm, handled);
}
static bool conv_rows_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("DFB_CONV_ROWS");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}
template <int WMODE>
static dfb_status run_conv_bn(const char* name, const CUtensorMap& ma, const float* wt, int n_out, int taps, int cp, int K, int C,
                              const ConvParams& prm, bool* handled) {
  if (n_out <= 32) return run_conv<32, WMODE>(name, ma, wt, n_out, taps, cp, K, C, prm, handled);
  if (n_out <= 64) return run_conv<64, WMODE>(name, ma, wt, n_out, taps, cp, K, C, prm, handled);
  const size_t m_tiles = (size_t)prm.tiles_w * prm.tiles_h * cdiv(prm.n_img, prm.n_t) * (prm.par_pad >= 0 ? 4 : 1);
  if (n_out > 128 && m_tiles * cdiv(n_out, 256) >= (size_t)sm_count() * 2)  // big layers: 128 x 256 tiles (see run_gemm_bn)
    return run_conv<256, WMODE>(name, ma, wt, n_out, taps, cp, K, C, prm, handled);
  return run_conv<128, WMODE>(name, ma, wt, n_out, taps, cp, K, C, prm, handled);
}

// y[pix, n_out] = sum_{taps, c} act[pix*stride + off(tap), c] * Wt[n_out][tap][c]
static dfb_status conv_like(const char* name, const float* act, const float* w, int w_layout, float* out, bool dgrad, int N,
                            int actC, int actH, int actW, int n_out, int R, int OH, int OW, int stride, int dh0, int sgn, int K,
                            int C, bool* handled, int par_pad = -1, const ConvFuse* fuse = nullptr) {
  const int taps = R * R;
  const int cp = (actC + 31) / 32 * 32;
  ConvParams prm;
  prm.epi = EpiArgs{};
  if (fuse && (fuse->addend || fuse->kind != FUSE_NONE)) {
    // fused epilogues exist for channels-last weights: statistics on fprop, addend / BatchNorm sums on dgrad
    if (w_layout != DFB_WLAYOUT_KRSC || (dgrad && fuse->kind == FUSE_STATS) || (!dgrad && (fuse->addend || fuse->kind == FUSE_BNBWD)))
      return DFB_OK;  // not handled: the dispatcher runs the work as separate kernels
  }
  if (fuse) {  // the partial buffers depend on the grid: run_conv fills them in
    prm.epi.addend = fuse->addend;
    prm.epi.stat_kind = fuse->kind;
    prm.epi.n_sets = fuse->n_sets;
    prm.epi.stat_out = fuse->stats_out;
    for (int i = 0; i < 2; ++i) {
      prm.epi.bn_x[i] = fuse->bn_x[i]; prm.epi.bn_mean[i] = fuse->bn_mean[i]; prm.epi.bn_invstd[i] = fuse->bn_invstd[i];
      prm.epi.bn_gamma[i] = fuse->bn_gamma[i]; prm.epi.bn_beta[i] = fuse->bn_beta[i];
    }
    prm.epi.relu = fuse->relu;
    prm.epi.relu_res = fuse->relu_res;
    prm.epi.lazy = fuse->lazy;
  }
  prm.out = out; prm.n_img = N; prm.OH = OH; prm.OW = OW; prm.n_out = n_out; prm.R = R; prm.cblks = cp / 32;
  prm.dh0 = dh0; prm.dw0 = dh0; prm.sgn = sgn; prm.stride = stride; prm.c_red = actC; prm.par_pad = par_pad;
  pixel_tile(BLOCK_M, OH, OW, &prm.ow_t, &prm.oh_t, &prm.n_t);
  // Row-halo kernel: 3x3, stride 1, at most 128 output channels (beyond that the weights dominate the traffic),
  // and a 128-pixel tile of ow_t x oh_t pixels inside one image with ow_t in {8, 16, 32}.
  bool rows = false;
  if (conv_rows_enabled() && stride == 1 && par_pad < 0 && R == 3 && n_out <= (g_x3 ? 64 : 128)) {   // (fp32-accurate mode: two double stages of the 128-wide halo variant do not fit)
    const int ow_r = std::min(32, pow2_ceil(OW)), oh_r = BLOCK_M / ow_r;
    if (ow_r >= 8 && pow2_ceil(OH) >= oh_r) {
      rows = true;
      prm.ow_t = ow_r; prm.oh_t = oh_r; prm.n_t = 1;
    }
  }
  prm.tiles_w = cdiv(OW, prm.ow_t);
  prm.tiles_h = cdiv(OH, prm.oh_t);
  CUtensorMap ma;
  if (!make_act_map(&ma, act, N, actH, actW, actC, stride, prm.ow_t, rows ? prm.oh_t + 2 : prm.oh_t, prm.n_t, MAJOR_K)) return DFB_OK;
  if (w_layout == DFB_WLAYOUT_KRSC) {  // channels-last weights are consumed in place
    if (rows) {
      if (dgrad) return run_conv_rows<W_KRSC_DGRAD>(name, ma, w, n_out, taps, cp, K, C, prm, handled);
      return run_conv_rows<W_KRSC_FPROP>(name, ma, w, n_out, taps, cp, K, C, prm, handled);
    }
    if (dgrad) return run_conv_bn<W_KRSC_DGRAD>(name, ma, w, n_out, taps, cp, K, C, prm, handled);
    return run_conv_bn<W_KRSC_FPROP>(name, ma, w, n_out, taps, cp, K, C, prm, handled);
  }
  float* wt = nullptr;
  size_t wt_n = (size_t)n_out * taps * cp;
  dfb_status st = dfb_malloc(wt_n, &wt);
  if (st != DFB_OK) return st;
  if (dgrad) launch_k(weight_transform_kernel<true>, bw_grid(wt_n, 256), 256, 0, compute_stream(), w, wt, K, C, taps, cp);
  else launch_k(weight_transform_kernel<false>, bw_grid(wt_n, 256), 256, 0, compute_stream(), w, wt, K, C, taps, cp);
  DFB_LAUNCH_CHECK("weight_transform");
  st = rows ? run_conv_rows<W_PACKED>(name, ma, wt, n_out, taps, cp, K, C, prm, handled)
            : run_conv_bn<W_PACKED>(name, ma, wt, n_out, taps, cp, K, C, prm, handled);
  dfb_free(wt);
  return st;
}

// cluster variant (WgradClusterProblem): grid.z = groups * csize, clusters of csize CTAs along z
template <int BN>
static dfb_status run_wgrad_cluster(const CUtensorMap& ma, const CUtensorMap& mb, const WgradParams& prm) {
  dim3 grid(cdiv(prm.Kout, BLOCK_M), (unsigned)(prm.R * prm.R * prm.ctiles), (unsigned)(prm.groups * prm.csize));
  if (prm.rows) {
    grid.y = (unsigned)(prm.R * prm.ctiles);
    return launch<WgradClusterProblem<32, 32, 128, true>>("tc_conv_wgrad_rows_cl", ma, mb, prm, grid, prm.csize);
  }
  if (prm.kr == 128) return launch<WgradClusterProblem<32, 32, 128>>("tc_conv_wgrad_cl", ma, mb, prm, grid, prm.csize);
  if (prm.Kout <= 32) return launch<WgradClusterProblem<BN, 32, 32>>("tc_conv_wgrad_cl", ma, mb, prm, grid, prm.csize);
  if (prm.Kout <= 64) return launch<WgradClusterProblem<BN, 64, 32>>("tc_conv_wgrad_cl", ma, mb, prm, grid, prm.csize);
  return launch<WgradClusterProblem<BN, 128, 32>>("tc_conv_wgrad_cl", ma, mb, prm, grid, prm.csize);
}
// DFB_WGRAD_CLUSTER = largest cluster size (2, 4 or 8; default 8); 0: one partial per CTA and the separate reduction.
// Measured on the ResNet-18 step (batch 256): 1.368 ms without, 1.353 ms with clusters of 4, 1.351 ms with clusters of 8.
static int wgrad_cluster_max() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("DFB_WGRAD_CLUSTER");
    const int want = e ? atoi(e) : 8;
    v = want >= 8 ? 8 : (want >= 4 ? 4 : (want >= 2 ? 2 : 0));
  }
  return v;
}

template <int BN>
static dfb_status run_wgrad(const CUtensorMap& ma, const CUtensorMap& mb, WgradParams prm, int splits) {
  dim3 grid(cdiv(prm.Kout, BLOCK_M), (unsigned)(prm.R * prm.R * prm.ctiles), (unsigned)splits);
  if (prm.rows) {  // a CTA per filter column (BN == 32, Kout <= 32: host)
    grid.y = (unsigned)(prm.R * prm.ctiles);
    return launch<WgradProblem<32, 32, 128, true>>("tc_conv_wgrad_rows", ma, mb, prm, grid);
  }
  if (prm.kr == 128) return launch<WgradProblem<32, 32, 128>>("tc_conv_wgrad", ma, mb, prm, grid);  // BN == 32 (host)
  if (prm.Kout <= 32) return launch<WgradProblem<BN, 32, 32>>("tc_conv_wgrad", ma, mb, prm, grid);
  if (prm.Kout <= 64) return launch<WgradProblem<BN, 64, 32>>("tc_conv_wgrad", ma, mb, prm, grid);
  return launch<WgradProblem<BN, 128, 32>>("tc_conv_wgrad", ma, mb, prm, grid);
}
// which kernel family serves `mode`: TF32 -> one MMA per k-step; FP32 -> the fp32-accurate three-term kernels (X3), unless
// DFB_FP32_TC=0 keeps the fp32 mode on the FFMA kernels of gemm_simt.cu; BF16 / SIMT -> not here
static bool select_mode(int mode) {
  static int fp32_tc = -1;
  if (fp32_tc < 0) {
    const char* e = getenv("DFB_FP32_TC");
    fp32_tc = (e && e[0] == '0') ? 0 : 1;
  }
  if (mode == DFB_MODE_TF32) { g_x3 = false; return true; }
  if (mode == DFB_MODE_FP32 && fp32_tc) { g_x3 = true; return true; }
  return false;
}
// The first layer (through its column matrix) is fp32-accurate in TF32 mode as well: its weight gradient is a sum over
// every pixel of the batch of terms that the BatchNorm behind it has made cancel (measured with TF32 operands: 4e-2 of its
// own size at batch 256), and three MMAs instead of one cost an HBM-bound layer nothing.
static int stem_mode(int mode) { return (mode == DFB_MODE_TF32 && select_mode(DFB_MODE_FP32)) ? DFB_MODE_FP32 : mode; }
}  // namespace tc

static bool tc_disabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("DFB_TC_DISABLE");
    v = (e && e[0] == '1') ? 1 : 0;
  }
  return v == 1;
}

dfb_status tc_gemm(const float* A, const float* B, float* C, int M, int N, int K, int trans_a, int trans_b, int lda, int ldb,
                   int ldc, int accumulate, const float* bias, int mode, bool* handled) {
  using namespace tc;
  *handled = false;
  if (tc_disabled() || !select_mode(mode)) return DFB_OK;
  if (K <= 0 || (lda & 3) || (ldb & 3)) return DFB_OK;
  if ((size_t)M * N < 4096 || K < 16) return DFB_OK;  // launch-latency territory: FFMA kernel is as fast
  const int vec_ok = ((ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(C) & 15) == 0 && (!bias || (reinterpret_cast<uintptr_t>(bias) & 15) == 0)) ? 1 : 0;
  GemmParams prm{C, bias, M, N, K, ldc, accumulate, vec_ok};
  if (!trans_a && !trans_b) return run_gemm_bn<MAJOR_K, MAJOR_MN>(A, B, prm, lda, ldb, handled);
  if (!trans_a && trans_b) return run_gemm_bn<MAJOR_K, MAJOR_K>(A, B, prm, lda, ldb, handled);
  if (trans_a && !trans_b) return run_gemm_bn<MAJOR_MN, MAJOR_MN>(A, B, prm, lda, ldb, handled);
  return run_gemm_bn<MAJOR_MN, MAJOR_K>(A, B, prm, lda, ldb, handled);
}

static bool conv_tc_ok(int N, int C, int H, int W, int K, int R, int pad, int stride, int mode) {
  if (tc_disabled() || !tc::select_mode(mode)) return false;
  if ((C & 3) || (K & 3) || R > 11 || stride < 1 || stride > 2) return false;
  if (stride == 2 && ((H & 1) || (W & 1))) return false;
  if (H + 2 * pad < R || W + 2 * pad < R) return false;
  return true;
}

dfb_status tc_conv_fprop(const float* x, const float* w, int w_layout, float* y, int N, int C, int H, int W, int K, int R, int pad,
                         int stride, int mode, float*, size_t, bool* handled, const ConvFuse* fuse) {
  *handled = false;
  if (!conv_tc_ok(N, C, H, W, K, R, pad, stride, mode)) return DFB_OK;
  const int OH = (H + 2 * pad - R) / stride + 1, OW = (W + 2 * pad - R) / stride + 1;
  return tc::conv_like("tc_conv_fprop", x, w, w_layout, y, false, N, C, H, W, K, R, OH, OW, stride, -pad, +1, K, C, handled, -1, fuse);
}

dfb_status tc_conv_dgrad(const float* dy, const float* w, int w_layout, float* dx, int N, int C, int H, int W, int K, int R, int pad,
                         int stride, int mode, float*, size_t, bool* handled, const ConvFuse* fuse) {
  *handled = false;
  if (!conv_tc_ok(N, C, H, W, K, R, pad, stride, mode)) return DFB_OK;
  const int OH = (H + 2 * pad - R) / stride + 1, OW = (W + 2 * pad - R) / stride + 1;
  if (stride == 1) {
    // dx[n,h,w,c] = sum_{r,s,k} dy[n, h + pad - r, w + pad - s, k] * w[k][c][r][s]
    return tc::conv_like("tc_conv_dgrad", dy, w, w_layout, dx, true, N, K, OH, OW, C, R, H, W, 1, pad, -1, K, C, handled, -1, fuse);
  }
  // stride 2: four output-parity classes of dx, each a stride-1 contraction over dy with every other tap
  // (ConvParams::par_pad); one launch, blockIdx.z = class. H and W are even (conv_tc_ok).
  return tc::conv_like("tc_conv_dgrad_s2", dy, w, w_layout, dx, true, N, K, OH, OW, C, R, H / 2, W / 2, 1, 0, 0, K, C, handled, pad, fuse);
}

// c_valid <= C: channels of x that belong to the gradient (the first-layer path pads its column matrix to 32 channels);
// dW then has c_valid channels. The in-kernel reductions store float4s, so they need c_valid % 4 == 0.
static dfb_status wgrad_impl(const float* x, const float* dy, float* dw, int w_layout, int N, int C, int H, int W, int K, int R, int pad,
                             int stride, int mode, int c_valid, bool* handled) {
  using namespace tc;
  *handled = false;
  if (!conv_tc_ok(N, C, H, W, K, R, pad, stride, mode)) return DFB_OK;
  const int OH = (H + 2 * pad - R) / stride + 1, OW = (W + 2 * pad - R) / stride + 1;
  const bool vec_ok = (c_valid & 3) == 0;
  WgradParams prm;
  prm.Kout = K; prm.C = c_valid; prm.Cp = (C + 31) / 32 * 32; prm.R = R; prm.pad = pad; prm.stride = stride;
  prm.n_img = N; prm.OH = OH; prm.OW = OW;
  int bn = prm.Cp % 128 == 0 ? 128 : (prm.Cp % 64 == 0 ? 64 : 32);
  if (prm.Cp % 256 == 0 && (size_t)N * OH * OW >= 16384) bn = 256;  // big layers: 128 x 256 tiles (see run_gemm_bn)
  // few channels on both sides and many pixels: 128-pixel stages (32 KB) instead of 32-pixel ones (8 KB)
  prm.kr = (K <= 32 && bn == 32 && (size_t)N * OH * OW >= 16384) ? 128 : BLOCK_K;
  pixel_tile(prm.kr, OH, OW, &prm.ow_t, &prm.oh_t, &prm.n_t);
  prm.rows = 0;
  // Row-halo wgrad (WgradProblem<.., ROWS_ = true>): 2.7x fewer operand bytes per tile. It needs two CTAs per SM (two
  // 40 KB stages each): with one CTA per SM and three stages it was SLOWER than the CTA-per-tap kernel (40 us vs 26 us
  // on 256x32x16x16 -> 32), with two it takes 18 us.
  if (conv_rows_enabled() && prm.kr == 128 && stride == 1 && R == 3) {
    const int ow_r = std::min(32, pow2_ceil(OW)), oh_r = 128 / ow_r;
    if (ow_r >= 8 && pow2_ceil(OH) >= oh_r) {
      prm.rows = 1;
      prm.ow_t = ow_r; prm.oh_t = oh_r; prm.n_t = 1;
    }
  }
  prm.tiles_w = cdiv(OW, prm.ow_t);
  prm.tiles_h = cdiv(OH, prm.oh_t);
  prm.pix_blocks = prm.tiles_w * prm.tiles_h * (int)cdiv(N, prm.n_t);
  prm.ctiles = prm.Cp / bn;
  CUtensorMap ma, mb;
  {
    uint64_t d[4] = {(uint64_t)K, (uint64_t)OW, (uint64_t)OH, (uint64_t)N};
    uint64_t s[4] = {1, (uint64_t)K, (uint64_t)OW * K, (uint64_t)OH * OW * K};
    uint32_t b[4] = {32, (uint32_t)prm.ow_t, (uint32_t)prm.oh_t, (uint32_t)prm.n_t};
    if (!make_map(&ma, dy, 4, d, s, b, MAJOR_MN)) return DFB_OK;
  }
  if (!make_act_map(&mb, x, N, H, W, C, stride, prm.ow_t, prm.rows ? prm.oh_t + 2 : prm.oh_t, prm.n_t, MAJOR_MN)) return DFB_OK;
  const int taps = R * R;
  size_t base_ctas = (size_t)cdiv(K, BLOCK_M) * (prm.rows ? R : taps) * prm.ctiles;
  int splits = (int)std::max<size_t>(1, ((size_t)sm_count() * 2 + base_ctas - 1) / base_ctas);  // two CTAs per SM
  splits = std::min(splits, std::max(1, prm.pix_blocks / 8));
  splits = std::min(splits, 128);
  // fp32-accurate mode: at most 512 k-steps accumulate into one TMEM tile (see tc_kernel: the tensor core's accumulation
  // error grows with their number); the partial tiles are then added in true fp32
  const int x3_need = g_x3 ? std::min(512, (int)cdiv(prm.pix_blocks, 4096 / prm.kr)) : 1;
  splits = std::max(splits, x3_need);
  prm.csize = 1; prm.groups = 1;
  prm.krsc = w_layout == DFB_WLAYOUT_KRSC ? 1 : 0;
  prm.dw = dw;
  // Two-level split (WgradClusterProblem): clusters of up to 8 CTAs reduce through distributed
  // shared memory; one partial per cluster, summed by the last cluster of each tile - no separate reduction kernel.
  if (wgrad_cluster_max() >= 2 && vec_ok && bn < 256 && splits >= 2 && base_ctas * 8 <= (size_t)kTicketWords - 128) {
    int cs = 2;
    while (cs * 2 <= std::min(splits, wgrad_cluster_max())) cs *= 2;
    // a cluster lives inside one GPC (18-20 SMs, two CTAs each): 4 clusters of 8 or 9 of 4 per GPC are co-resident,
    // and a second wave would double the kernel's time
    const size_t slots = cs == 8 ? 256 : (cs == 4 ? 288 : (size_t)sm_count() * 2);
    int groups = (int)std::max<size_t>(1, std::min<size_t>((size_t)(splits / cs), slots / (base_ctas * cs)));
    groups = std::max(groups, (int)cdiv(x3_need, cs));
    prm.blocks_per_split = (prm.pix_blocks + groups - 1) / groups;  // per group; the kernel cuts it by cluster rank
    groups = (prm.pix_blocks + prm.blocks_per_split - 1) / prm.blocks_per_split;
    prm.csize = cs; prm.groups = groups;
    float* partial = nullptr;
    if (groups > 1) {
      dfb_status st = dfb_malloc((size_t)groups * K * taps * prm.Cp, &partial);
      if (st != DFB_OK) return st;
    }
    prm.partial = partial;
    prm.tickets = groups > 1 ? ticket_counter(64) : nullptr;
    *handled = true;
    dfb_status st = bn == 128 ? run_wgrad_cluster<128>(ma, mb, prm) : (bn == 64 ? run_wgrad_cluster<64>(ma, mb, prm) : run_wgrad_cluster<32>(ma, mb, prm));
    if (partial) dfb_free(partial);
    return st;
  }
  prm.blocks_per_split = (prm.pix_blocks + splits - 1) / splits;
  splits = (prm.pix_blocks + prm.blocks_per_split - 1) / prm.blocks_per_split;
  float* partial = nullptr;
  dfb_status st = dfb_malloc((size_t)splits * K * taps * prm.Cp, &partial);
  if (st != DFB_OK) return st;
  prm.partial = partial;
  prm.dw = dw;
  prm.krsc = w_layout == DFB_WLAYOUT_KRSC ? 1 : 0;
  // one arrival counter per output tile; (K * taps * Cp) % 4 == 0 keeps the float4 walk of the slabs aligned
  // The in-kernel reduction is done by ONE CTA per tile: worth it (one launch less) while a tile's partials are
  // small; beyond that the separate reduction kernel, which spreads over the machine, is faster.
  const size_t tile_partial_bytes = (size_t)splits * std::min(K, BLOCK_M) * bn * sizeof(float);
  prm.tickets = (vec_ok && base_ctas <= (size_t)kTicketWords - 64 && tile_partial_bytes <= (192u << 10)) ? ticket_counter(64) : nullptr;
  *handled = true;
  if (bn == 256) st = run_wgrad<256>(ma, mb, prm, splits);
  else if (bn == 128) st = run_wgrad<128>(ma, mb, prm, splits);
  else if (bn == 64) st = run_wgrad<64>(ma, mb, prm, splits);
  else st = run_wgrad<32>(ma, mb, prm, splits);
  if (st == DFB_OK && !prm.tickets) {
    const size_t outs = (size_t)K * c_valid * taps;
    const int krsc = w_layout == DFB_WLAYOUT_KRSC ? 1 : 0;
    if (splits > 16) launch_k(wgrad_reduce_kernel<32>, bw_grid(outs * 32, 256), 256, 0, compute_stream(), partial, dw, splits, K, c_valid, prm.Cp, taps, krsc);
    else if (splits > 4) launch_k(wgrad_reduce_kernel<4>, bw_grid(outs * 4, 256), 256, 0, compute_stream(), partial, dw, splits, K, c_valid, prm.Cp, taps, krsc);
    else launch_k(wgrad_reduce_kernel<1>, bw_grid(outs, 256), 256, 0, compute_stream(), partial, dw, splits, K, c_valid, prm.Cp, taps, krsc);
    cudaError_t e = cudaGetLastError();
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (e != cudaSuccess) {
      dfb_free(partial);
      DFB_FAIL(DFB_ERR_RUNTIME, "wgrad_reduce launch failed: %s", cudaGetErrorString(e));
    }
  }
  dfb_free(partial);
  return st;
}

dfb_status tc_conv_wgrad(const float* x, const float* dy, float* dw, int w_layout, int N, int C, int H, int W, int K, int R, int pad,
                         int stride, int mode, float*, size_t, bool* handled) {
  return wgrad_impl(x, dy, dw, w_layout, N, C, H, W, K, R, pad, stride, mode, C, handled);
}

// ---- first layer (image input, C <= 4) on the tensor pipe ------------------------------------------------------
// The weight gradient of the first layer is a [K x C*R*R] = [32 x 27] matrix summed over a quarter of a million
// pixels: as a gather kernel on the FFMA pipe it is latency bound (74 us for the ResNet stem at batch 256, 8 % of the
// HBM roofline). Here the receptive fields are first written out as a [pixels x 32] column matrix (C*R*R <= 32 columns,
// zero padded; one coalesced 128-byte row per pixel, the 3 MB image stays in L1/L2), and the gradient becomes the
// weight gradient of a 1x1 convolution over 32 "channels": the tcgen05 wgrad kernel with 128-pixel stages. The column
// order is the gradient's own memory order (tap-major for channels-last weights, channel-major for (K,C,R,R)), so a
// row of the GEMM result is a row of dW.
__global__ void __launch_bounds__(256) stem_cols_kernel(const float* __restrict__ x, int nchw, float* __restrict__ col, int N, int C,
                                                        int H, int W, int R, int pad, int stride, int OH, int OW, int krsc) {
  pdl_sync();
  const int taps = R * R, cols = C * taps;
  // eight threads per pixel, a float4 (four columns) each. Which four columns is fixed per thread (the grid step is a
  // multiple of 8): their (channel, row offset, column offset) are decoded once, outside the pixel loop.
  const int q = (int)(threadIdx.x & 7);
  int dh[4], dw[4];
  size_t coff[4];
  bool live[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int j = q * 4 + u;
    live[u] = j < cols;
    const int tap = live[u] ? (krsc ? j / C : j % taps) : 0, c = live[u] ? (krsc ? j % C : j / taps) : 0;
    dh[u] = tap / R - pad;
    dw[u] = tap % R - pad;
    coff[u] = nchw ? (size_t)c * H * W : (size_t)c;
  }
  const size_t pixels = (size_t)N * OH * OW;
  const size_t step = ((size_t)gridDim.x * blockDim.x) >> 3;
  const int pix_stride = nchw ? 1 : C;
  for (size_t pix = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 3; pix < pixels; pix += step) {
    const int ow = (int)(pix % OW);
    const size_t t = pix / OW;
    const int oh = (int)(t % OH), n = (int)(t / OH);
    const float* xn = x + (size_t)n * C * H * W;
    const int ih0 = oh * stride, iw0 = ow * stride;
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int ih = ih0 + dh[u], iw = iw0 + dw[u];
      v[u] = 0.f;
      if (live[u] && (unsigned)ih < (unsigned)H && (unsigned)iw < (unsigned)W)
        v[u] = __ldg(xn + coff[u] + ((size_t)ih * W + iw) * pix_stride);
    }
    reinterpret_cast<float4*>(col)[pix * 8 + q] = make_float4(v[0], v[1], v[2], v[3]);
  }
}
// Wp[k][32] = the first-layer weights in the column order of stem_cols_kernel (dW's own memory order), zero padded
__global__ void __launch_bounds__(256) stem_pad_weights_kernel(const float* __restrict__ w, float* __restrict__ wp, int K, int cols) {
  pdl_sync();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < K * 32) {
    const int k = i >> 5, j = i & 31;
    wp[i] = j < cols ? __ldg(w + (size_t)k * cols + j) : 0.f;
  }
}
// on by default (DFB_STEM_TC=0: the gather kernel in every mode). ResNet stem at batch 256: 74 us -> the column pass plus
// the tensor-core kernel; the training step 1.349 -> 1.308 ms.
static bool stem_tc_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("DFB_STEM_TC");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}
dfb_status tc_stem_wgrad(const float* x, int x_layout, const float* dy, float* dw, int w_layout, int N, int C, int H, int W, int K, int R,
                         int pad, int stride, int mode, bool* handled) {
  *handled = false;
  if (!stem_tc_enabled() || tc_disabled() || mode != DFB_MODE_TF32) return DFB_OK;   // (fp32 mode: the exact FFMA gather kernel)
  const int cols = C * R * R;
  if (C > 4 || cols > 32 || (K & 3) || stride < 1 || H + 2 * pad < R || W + 2 * pad < R) return DFB_OK;
  const int OH = (H + 2 * pad - R) / stride + 1, OW = (W + 2 * pad - R) / stride + 1;
  const size_t pixels = (size_t)N * OH * OW;
  if (pixels < 16384) return DFB_OK;  // small batches: the gather kernel is a single short launch
  float* col = nullptr;
  dfb_status st = dfb_malloc(pixels * 32, &col);
  if (st != DFB_OK) return st;
  launch_k(stem_cols_kernel, bw_grid(pixels * 8, 256), 256, 0, compute_stream(), x, x_layout == DFB_LAYOUT_NCHW ? 1 : 0, col, N, C, H, W, R,
           pad, stride, OH, OW, w_layout == DFB_WLAYOUT_KRSC ? 1 : 0);
  cudaError_t e = cudaGetLastError();
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (e != cudaSuccess) {
    dfb_free(col);
    DFB_FAIL(DFB_ERR_RUNTIME, "stem_cols launch failed: %s", cudaGetErrorString(e));
  }
  // the column matrix is an (N, OH, OW, 32) channels-last activation; its 1x1 wgrad has cols valid channels
  st = wgrad_impl(col, dy, dw, w_layout, N, 32, OH, OW, K, 1, 0, 1, tc::stem_mode(mode), cols, handled);
  dfb_free(col);
  return st;
}

size_t tc_conv_workspace_floats(int, int, int, int, int, int, int, int) { return 0; }

// ---- first layer through its column matrix, for callers that keep the matrix between forward and backward --------------
// (DeepFlows/nn/functional.py:_conv2d): col = receptive fields [pixels x 32]; the forward convolution is then a 1x1
// convolution of `col` with the padded weights (dfb_conv2d_fprop_stats on the tensor pipe, statistics included), and the
// weight gradient the 1x1 wgrad of `col` - the 33 us gather kernel of the forward pass and the second column pass of the
// backward pass disappear.
dfb_status tc_stem_cols(const float* x, int x_layout, float* col, int N, int C, int H, int W, int R, int pad, int stride, int w_layout) {
  const int OH = (H + 2 * pad - R) / stride + 1, OW = (W + 2 * pad - R) / stride + 1;
  const size_t pixels = (size_t)N * OH * OW;
  launch_k(stem_cols_kernel, bw_grid(pixels * 8, 256), 256, 0, compute_stream(), x, x_layout == DFB_LAYOUT_NCHW ? 1 : 0, col, N, C, H, W, R,
           pad, stride, OH, OW, w_layout == DFB_WLAYOUT_KRSC ? 1 : 0);
  DFB_LAUNCH_CHECK("stem_cols");
  return DFB_OK;
}
dfb_status tc_stem_pad_weights(const float* w, float* wp, int K, int cols) {
  launch_k(stem_pad_weights_kernel, cdiv((size_t)K * 32, 256), 256, 0, compute_stream(), w, wp, K, cols);
  DFB_LAUNCH_CHECK("stem_pad_weights");
  return DFB_OK;
}
dfb_status tc_wgrad_cols(const float* col, const float* dy, float* dw, int w_layout, int N, int OH, int OW, int K, int cols, int mode,
                         bool* handled) {
  return wgrad_impl(col, dy, dw, w_layout, N, 32, OH, OW, K, 1, 0, 1, tc::stem_mode(mode), cols, handled);
}

#ifdef DFB_TC_TIMING
extern "C" __attribute__((visibility("default"))) int dfb_debug_tc_stamps(unsigned long long* out32) {
  return (int)cudaMemcpyFromSymbol(out32, tc::g_tc_stamp, sizeof(unsigned long long) * 32);
}
#endif

}  // namespace dfb
