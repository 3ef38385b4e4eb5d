// Bandwidth-bound L1 kernels on channels-last data: BatchNorm forward/backward, ReLU, row-vector
// add, column sums, max/avg pooling, fused softmax cross-entropy.
//
// The reference composes each of these from dozens of out-of-place L0 kernels with the
// broadcast operands materialised and the broadcast gradients reduced on the host
// (DeepFlows/nn/modules/batchnorm.py:30-55, DeepFlows/nn/functional.py:104-115,347-374,
// DeepFlows/tensor.py:462-483). Here each op is one or two passes over HBM with 128-bit accesses.
//
// Data layout: activations are (rows = N*H*W, C) row-major, i.e. NHWC. A "column group" is 4
// adjacent channels (one float4) when C % 4 == 0, otherwise one channel.
#include "kernels.cuh"

#include <algorithm>
#include <cmath>

namespace dfb {

constexpr int kT = 256;

// -------------------------------------------------------------------------------------------------
// Column statistics. A CTA owns a contiguous chunk of rows; thread t handles column group
// (t % G) on row lanes (t / G), so a warp reads whole 128-byte lines.
// -------------------------------------------------------------------------------------------------
template <int V>
struct Vec;
template <>
struct Vec<4> {
  using T = float4;
  static __device__ __forceinline__ void get(const float* p, float (&v)[4]) {
    float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  // streaming load as volatile asm: a run of these is issued back to back (the compiler otherwise pairs each
  // load with its consumer and keeps only two in flight), which is what a bandwidth-bound loop needs
  static __device__ __forceinline__ void get_stream(const float* p, float (&v)[4]) {
    float4 t = ld_stream(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void put(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <>
struct Vec<1> {
  static __device__ __forceinline__ void get(const float* p, float (&v)[1]) { v[0] = *p; }
  static __device__ __forceinline__ void get_stream(const float* p, float (&v)[1]) { v[0] = *p; }
  static __device__ __forceinline__ void put(float* p, const float (&v)[1]) { *p = v[0]; }
};

struct ColPlan {
  int V;            // 4 or 1
  int G;            // column groups = C / V
  int lanes;        // row lanes per CTA = max(1, kT / G)
  int gpass;        // column-group passes per CTA = ceil(G / kT)
  unsigned ctas;    // CTAs (row chunks) = partial results per channel
  size_t rows_per_cta;
};
// Row chunking for the column reductions. Every thread should see only a handful of rows (the loop is a
// chain of dependent-latency loads otherwise), but the number of CTAs is also the number of partials the last
// CTA has to merge, so it is capped at two CTAs per SM.
static ColPlan plan_cols(size_t rows, int C, const void* p0, const void* p1 = nullptr) {
  ColPlan p;
  bool al = ((reinterpret_cast<uintptr_t>(p0) | reinterpret_cast<uintptr_t>(p1)) & 15) == 0;
  p.V = (C % 4 == 0 && al) ? 4 : 1;
  p.G = C / p.V;
  p.lanes = std::max(1, kT / p.G);
  p.gpass = (p.G + kT - 1) / kT;
  size_t want = (rows + (size_t)p.lanes * 4 - 1) / ((size_t)p.lanes * 4);  // ~4 rows per thread
  // big inputs are bandwidth problems (more CTAs = more loads in flight), small ones latency problems (fewer
  // partials for the last CTA to merge)
  size_t cap = (size_t)sm_count() * (rows * (size_t)C >= ((size_t)4 << 20) ? 4 : 2);
  p.ctas = (unsigned)std::max<size_t>(1, std::min(want, cap));
  p.rows_per_cta = (rows + p.ctas - 1) / p.ctas;
  p.ctas = (unsigned)((rows + p.rows_per_cta - 1) / p.rows_per_cta);
  return p;
}

// Ticket counters for "the last CTA to finish merges the partials" (threadfence-reduction pattern): one
// persistent zero-initialised word per kernel family, reset by the last CTA. All users run on the single
// compute stream, so two kernels never share a counter concurrently.
// returns true in every thread of the last CTA to arrive; all global writes made by the CTA's threads before
// the call are visible to the last CTA afterwards (read them with __ldcg).
__device__ __forceinline__ bool last_cta_arrives(unsigned* ticket) {
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned t = atomicAdd(ticket, 1u);
    s_last = (t == gridDim.x - 1);
    if (s_last) *ticket = 0;  // ready for the next launch
  }
  __syncthreads();
  if (s_last) __threadfence();
  return s_last;
}

// Two sums per channel over all rows, in one launch: sum f0(row), sum f1(row), where (f0, f1) is
//   STATS : (x - shift, (x - shift)^2)  with shift = x[row 0] (keeps the variance well conditioned when
//           |mean| >> std without Welford's divisions; partials merge by plain addition in a fixed order)
//   BNBWD : (dy, dy * x_hat)
//   COLSUM: (x, -)
// Thread t owns column group (t % G) on row lane (t / G); a warp reads whole 128-byte lines. Each CTA writes
// its partial sums, the last CTA to finish adds the partials (fixed order => deterministic) and hands the
// totals to `Fin`.
//   POOLBN: BNBWD of a gradient that is computed on the way: dy = max-pool backward (tie-faithful) of the pooled gradient,
//           masked by the ReLU between the BatchNorm and the pool - the backward of conv -> BatchNorm -> ReLU -> MaxPool
//           up to the BatchNorm's reductions in ONE pass over the BatchNorm's input (dy is also written out)
enum { SUMS_STATS = 0, SUMS_BNBWD = 1, SUMS_COLSUM = 2, SUMS_POOLBN = 3 };
struct SumsArgs {
  const float* x;
  const float* dy;       // BNBWD
  const float* mean;     // BNBWD
  const float* invstd;   // BNBWD
  float* part;           // [ctas][2][C]
  unsigned* ticket;
  // finalisation
  float* out0;           // STATS: save_mean   BNBWD: dbeta   COLSUM: out
  float* out1;           // STATS: save_invstd BNBWD: dgamma
  float* running_mean;   // STATS
  float* running_var;    // STATS
  float eps, momentum;
  int raw_var;           // STATS: out1 = biased variance instead of 1/sqrt(var + eps); running statistics untouched
  // POOLBN: dy = gradient of the POOLED tensor; rows are the pixels (n, h, w) of the BatchNorm's input x
  const float* gamma;    // affine parameters of the BatchNorm (null: 1 / 0)
  const float* beta;
  const float* pool_y;   // the pool's output [N, OH, OW, C]
  float* dy_out;         // [rows, C]: the gradient that reaches the BatchNorm's output
  int H, W, OH, OW, pool_k;
};

// Pairwise (tree) sum over the row lanes of a CTA through shared memory; the result lands in lane 0. A tree
// keeps the rounding error at O(log lanes) like numpy's pairwise summation (the oracle), and the order is
// fixed, so results are reproducible. Must be called by all threads of the CTA.
template <int V, bool TWO>
__device__ __forceinline__ void lane_tree_sum(float* sm, float (&s0)[V], float (&s1)[V], int lane, int lanes, int g, int C,
                                              bool active) {
  int top = 1;
  while (top < lanes) top <<= 1;
  __syncthreads();  // shared memory may still be read by a previous user
  if (active) {
    Vec<V>::put(sm + (size_t)(lane * 2 + 0) * C + g * V, s0);
    if (TWO) Vec<V>::put(sm + (size_t)(lane * 2 + 1) * C + g * V, s1);
  }
  for (int off = top >> 1; off > 0; off >>= 1) {
    __syncthreads();
    const bool take = active && lane < off && lane + off < lanes;
    if (take) {
      float t0[V], t1[V];
      Vec<V>::get(sm + (size_t)((lane + off) * 2 + 0) * C + g * V, t0);
      if (TWO) Vec<V>::get(sm + (size_t)((lane + off) * 2 + 1) * C + g * V, t1);
#pragma unroll
      for (int v = 0; v < V; ++v) { s0[v] += t0[v]; if (TWO) s1[v] += t1[v]; }
    }
    __syncthreads();
    if (take && off > 1) {
      Vec<V>::put(sm + (size_t)(lane * 2 + 0) * C + g * V, s0);
      if (TWO) Vec<V>::put(sm + (size_t)(lane * 2 + 1) * C + g * V, s1);
    }
  }
}

// POOLBN helpers. Row r = pixel (n, h, w) of the pool's input; its window is row (n, h / k, w / k) of the pooled tensors
// (pixels beyond OH * k / OW * k belong to no window: no gradient).
__device__ __forceinline__ size_t pooled_row(const SumsArgs& a, size_t r, bool* inside) {
  const unsigned r32 = (unsigned)r;   // (rows < 2^31, checked on the host: 32-bit divisions, a tenth of the 64-bit ones' cost)
  const unsigned t = r32 / (unsigned)a.W, w = r32 - t * (unsigned)a.W;
  const unsigned n = t / (unsigned)a.H, h = t - n * (unsigned)a.H;
  const unsigned oh = h / (unsigned)a.pool_k, ow = w / (unsigned)a.pool_k;
  *inside = oh < (unsigned)a.OH && ow < (unsigned)a.OW;
  return *inside ? ((size_t)n * a.OH + oh) * a.OW + ow : 0;
}
// z = the BatchNorm's output (pre-activation), act = relu(z) = what the pool saw; every maximum of the window (ties
// included, SURVEY Q2: maxpool2d_bwd) takes the pooled gradient, and the ReLU passes it where z >= 0 (tensor.py:872-877)
__device__ __forceinline__ float pool_relu_grad(float x, float mean, float scale, float shift, float pooled, float g, bool inside) {
  const float z = fmaf(x - mean, scale, shift);
  const float act = fmaxf(z, 0.f);
  return (inside && act == pooled && z >= 0.f) ? g : 0.f;
}

template <int V, int KIND>
__global__ void __launch_bounds__(kT, 2)
col_sums_kernel(SumsArgs a, size_t rows, int C, ColPlan p) {
  pdl_sync();
  extern __shared__ float sm[];  // [lanes][2][C] when lanes > 1
  const int G = p.G;
  const size_t r0 = (size_t)blockIdx.x * p.rows_per_cta;
  const size_t r1 = r0 + p.rows_per_cta < rows ? r0 + p.rows_per_cta : rows;
  const int gsel = threadIdx.x % (G < kT ? G : kT);
  const int lane = G < kT ? threadIdx.x / G : 0;
  for (int gp = 0; gp < p.gpass; ++gp) {
    const int g = gp * kT + gsel;
    const bool active = g < G && lane < p.lanes;
    constexpr bool kBwd = KIND == SUMS_BNBWD || KIND == SUMS_POOLBN;
    float s0[V], s1[V], c0[V], c1[V], c2[V], c3[V];
#pragma unroll
    for (int v = 0; v < V; ++v) { s0[v] = 0.f; s1[v] = 0.f; c0[v] = 0.f; c1[v] = 0.f; c2[v] = 0.f; c3[v] = 0.f; }
    if (active) {
      if (KIND == SUMS_STATS) Vec<V>::get(a.x + (size_t)g * V, c0);  // shift = row 0
      if (kBwd) {
#pragma unroll
        for (int v = 0; v < V; ++v) { c0[v] = a.mean[g * V + v]; c1[v] = a.invstd[g * V + v]; }
      }
      if (KIND == SUMS_POOLBN) {   // the pre-activation exactly as bn_apply_fused_kernel computed it: fmaf(x - mean, invstd * gamma, beta)
#pragma unroll
        for (int v = 0; v < V; ++v) { c2[v] = c1[v] * (a.gamma ? a.gamma[g * V + v] : 1.0f); c3[v] = a.beta ? a.beta[g * V + v] : 0.0f; }
      }
      const size_t step = p.lanes;
      size_t r = r0 + lane;
      // kU independent rows in flight per thread: ~64-128 bytes per thread, enough outstanding loads across the
      // grid to cover HBM latency at full bandwidth
      constexpr int kU = kBwd ? 4 : 8;
      for (; r + (kU - 1) * step < r1; r += kU * step) {
        float xv[kU][V], dv[kBwd ? kU : 1][V], yv[KIND == SUMS_POOLBN ? kU : 1][V];
        bool in_pool[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          Vec<V>::get_stream(a.x + (r + u * step) * C + (size_t)g * V, xv[u]);
          if (KIND == SUMS_BNBWD) Vec<V>::get_stream(a.dy + (r + u * step) * C + (size_t)g * V, dv[u]);
          if (KIND == SUMS_POOLBN) {
            const size_t pr = pooled_row(a, r + u * step, &in_pool[u]);
            Vec<V>::get(a.dy + pr * C + (size_t)g * V, dv[u]);       // (re-read by the k*k pixels of the window: cached)
            Vec<V>::get(a.pool_y + pr * C + (size_t)g * V, yv[u]);
          }
        }
        // compiler fence on the loaded values: keeps the arithmetic below behind ALL the loads above, so the
        // loads are issued back to back instead of being paired with their consumers
#pragma unroll
        for (int u = 0; u < kU; ++u)
#pragma unroll
          for (int v = 0; v < V; ++v) {
            asm volatile("" : "+f"(xv[u][v]));
            if (kBwd) asm volatile("" : "+f"(dv[u][v]));
          }
        if (KIND == SUMS_POOLBN) {
#pragma unroll
          for (int u = 0; u < kU; ++u) {
#pragma unroll
            for (int v = 0; v < V; ++v) dv[u][v] = pool_relu_grad(xv[u][v], c0[v], c2[v], c3[v], yv[u][v], dv[u][v], in_pool[u]);
            Vec<V>::put(a.dy_out + (r + u * step) * C + (size_t)g * V, dv[u]);
          }
        }
#pragma unroll
        for (int u = 0; u < kU; ++u)
#pragma unroll
          for (int v = 0; v < V; ++v) {
            if (KIND == SUMS_STATS) { float d = xv[u][v] - c0[v]; s0[v] += d; s1[v] = fmaf(d, d, s1[v]); }
            if (kBwd) { s0[v] += dv[u][v]; s1[v] = fmaf(dv[u][v], (xv[u][v] - c0[v]) * c1[v], s1[v]); }
            if (KIND == SUMS_COLSUM) s0[v] += xv[u][v];
          }
      }
      for (; r < r1; r += step) {
        float xv[V], dv[V];
        Vec<V>::get(a.x + r * C + (size_t)g * V, xv);
        if (KIND == SUMS_BNBWD) Vec<V>::get(a.dy + r * C + (size_t)g * V, dv);
        if (KIND == SUMS_POOLBN) {
          bool inside;
          const size_t pr = pooled_row(a, r, &inside);
          float yv[V];
          Vec<V>::get(a.dy + pr * C + (size_t)g * V, dv);
          Vec<V>::get(a.pool_y + pr * C + (size_t)g * V, yv);
#pragma unroll
          for (int v = 0; v < V; ++v) dv[v] = pool_relu_grad(xv[v], c0[v], c2[v], c3[v], yv[v], dv[v], inside);
          Vec<V>::put(a.dy_out + r * C + (size_t)g * V, dv);
        }
#pragma unroll
        for (int v = 0; v < V; ++v) {
          if (KIND == SUMS_STATS) { float d = xv[v] - c0[v]; s0[v] += d; s1[v] = fmaf(d, d, s1[v]); }
          if (kBwd) { s0[v] += dv[v]; s1[v] = fmaf(dv[v], (xv[v] - c0[v]) * c1[v], s1[v]); }
          if (KIND == SUMS_COLSUM) s0[v] += xv[v];
        }
      }
    }
    if (p.lanes > 1) lane_tree_sum<V, KIND != SUMS_COLSUM>(sm, s0, s1, lane, p.lanes, g, C, active);
    if (active && lane == 0) {
      Vec<V>::put(a.part + ((size_t)blockIdx.x * 2 + 0) * C + g * V, s0);
      if (KIND != SUMS_COLSUM) Vec<V>::put(a.part + ((size_t)blockIdx.x * 2 + 1) * C + g * V, s1);
    }
  }
  if (!last_cta_arrives(a.ticket)) return;

  // ---- last CTA: totals over the partials. Same thread mapping: lane l adds partials l, l+lanes, ... -----
  const int parts = gridDim.x;
  for (int gp = 0; gp < p.gpass; ++gp) {
    const int g = gp * kT + gsel;
    const bool active = g < G && lane < p.lanes;
    float s0[V], s1[V];
#pragma unroll
    for (int v = 0; v < V; ++v) { s0[v] = 0.f; s1[v] = 0.f; }
    if (active) {
      int q = lane;
      for (; q + 3 * p.lanes < parts; q += 4 * p.lanes) {
        float t0[4][V], t1[4][V];
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < V; ++v) {
            t0[u][v] = __ldcg(a.part + ((size_t)(q + u * p.lanes) * 2 + 0) * C + g * V + v);
            t1[u][v] = KIND != SUMS_COLSUM ? __ldcg(a.part + ((size_t)(q + u * p.lanes) * 2 + 1) * C + g * V + v) : 0.f;
          }
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < V; ++v) { s0[v] += t0[u][v]; s1[v] += t1[u][v]; }
      }
      for (; q < parts; q += p.lanes)
#pragma unroll
        for (int v = 0; v < V; ++v) {
          s0[v] += __ldcg(a.part + ((size_t)q * 2 + 0) * C + g * V + v);
          if (KIND != SUMS_COLSUM) s1[v] += __ldcg(a.part + ((size_t)q * 2 + 1) * C + g * V + v);
        }
    }
    if (p.lanes > 1) lane_tree_sum<V, true>(sm, s0, s1, lane, p.lanes, g, C, active);
    if (active && lane == 0) {
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const int c = g * V + v;
        if (KIND == SUMS_STATS) {
          // mean = shift + s0/n ; biased var = s1/n - (s0/n)^2 ; running stats use the biased variance
          // like batchnorm.py:44-46
          const float n = (float)rows;
          const float dm = s0[v] / n;
          const float mean = a.x[c] + dm;
          const float var = fmaxf(s1[v] / n - dm * dm, 0.f);
          a.out0[c] = mean;
          a.out1[c] = a.raw_var ? var : 1.0f / sqrtf(var + a.eps);
          if (a.running_mean) a.running_mean[c] = a.running_mean[c] * (1.0f - a.momentum) + mean * a.momentum;
          if (a.running_var) a.running_var[c] = a.running_var[c] * (1.0f - a.momentum) + var * a.momentum;
        } else {
          if (a.out0) a.out0[c] = s0[v];
          if ((KIND == SUMS_BNBWD || KIND == SUMS_POOLBN) && a.out1) a.out1[c] = s1[v];
        }
      }
    }
  }
}

// SUMS_POOLBN for the geometry every script uses (2x2 windows, stride 2, even H and W, channels a multiple of 4): one
// work item = one WINDOW x four channels. The pooled gradient and the pooled value are loaded once per window instead of
// once per pixel, the four pixels of U windows are in flight together (8 x 128-bit loads + 4 per thread), there is no
// per-pixel index arithmetic and no remainder loop. The general kernel above needed 38 us for the stem of the ResNet
// (33.5 MB in, 33.5 MB out: a dependent-latency chain of ~5 round trips per thread at 25 % occupancy).
template <int U>
__global__ void __launch_bounds__(kT, 2)
pool2_relu_bn_bwd_kernel(SumsArgs a, unsigned prows, int C, unsigned rows_per_cta, int lanes) {
  pdl_sync();
  extern __shared__ float sm[];  // [lanes][2][C]
  const int G = C >> 2;
  const int g = threadIdx.x % G, lane = threadIdx.x / G;
  const bool active = lane < lanes;
  float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
  if (active) {
    float mu[4], is[4], sc[4], sh[4];
    Vec<4>::get(a.mean + g * 4, mu);
    Vec<4>::get(a.invstd + g * 4, is);
#pragma unroll
    for (int v = 0; v < 4; ++v) { sc[v] = is[v] * (a.gamma ? a.gamma[g * 4 + v] : 1.0f); sh[v] = a.beta ? a.beta[g * 4 + v] : 0.0f; }
    const unsigned r0 = blockIdx.x * rows_per_cta;
    const unsigned r1 = min(prows, r0 + rows_per_cta);
    const unsigned OW = (unsigned)a.OW, OH = (unsigned)a.OH, W = (unsigned)a.W;
    for (unsigned r = r0 + lane; r < r1; r += U * lanes) {
      float xv[U][4][4], gv[U][4], yv[U][4];
      size_t px[U];
      bool ok[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const unsigned pr = r + u * lanes;
        ok[u] = pr < r1;
        const unsigned q = ok[u] ? pr : r;
        const unsigned t = q / OW, ow = q - t * OW;
        const unsigned n = t / OH, oh = t - n * OH;
        px[u] = ((size_t)(n * 2 * OH + 2 * oh) * W + 2 * ow) * C + (size_t)g * 4;   // (H == 2 * OH)
        Vec<4>::get_stream(a.dy + (size_t)q * C + g * 4, gv[u]);
        Vec<4>::get_stream(a.pool_y + (size_t)q * C + g * 4, yv[u]);
#pragma unroll
        for (int i = 0; i < 2; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j) Vec<4>::get_stream(a.x + px[u] + ((size_t)i * W + j) * C, xv[u][i * 2 + j]);
      }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v) {
          asm volatile("" : "+f"(gv[u][v]), "+f"(yv[u][v]));
#pragma unroll
          for (int w = 0; w < 4; ++w) asm volatile("" : "+f"(xv[u][w][v]));
        }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (!ok[u]) continue;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          float d[4];
#pragma unroll
          for (int v = 0; v < 4; ++v) {
            d[v] = pool_relu_grad(xv[u][w][v], mu[v], sc[v], sh[v], yv[u][v], gv[u][v], true);
            s0[v] += d[v];
            s1[v] = fmaf(d[v], (xv[u][w][v] - mu[v]) * is[v], s1[v]);
          }
          Vec<4>::put(a.dy_out + px[u] + ((size_t)(w >> 1) * W + (w & 1)) * C, d);
        }
      }
    }
  }
  if (lanes > 1) lane_tree_sum<4, true>(sm, s0, s1, lane, lanes, g, C, active);
  if (active && lane == 0) {
    Vec<4>::put(a.part + ((size_t)blockIdx.x * 2 + 0) * C + g * 4, s0);
    Vec<4>::put(a.part + ((size_t)blockIdx.x * 2 + 1) * C + g * 4, s1);
  }
  if (!last_cta_arrives(a.ticket)) return;
  // last CTA: lane l adds partials l, l + lanes, ... (fixed order), then the lane tree
  const int parts = gridDim.x;
#pragma unroll
  for (int v = 0; v < 4; ++v) { s0[v] = 0.f; s1[v] = 0.f; }
  if (active) {
    for (int q = lane; q < parts; q += lanes) {
      float t0[4], t1[4];
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        t0[v] = __ldcg(a.part + ((size_t)q * 2 + 0) * C + g * 4 + v);
        t1[v] = __ldcg(a.part + ((size_t)q * 2 + 1) * C + g * 4 + v);
      }
#pragma unroll
      for (int v = 0; v < 4; ++v) { s0[v] += t0[v]; s1[v] += t1[v]; }
    }
  }
  if (lanes > 1) lane_tree_sum<4, true>(sm, s0, s1, lane, lanes, g, C, active);
  if (active && lane == 0) {
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      if (a.out0) a.out0[g * 4 + v] = s0[v];
      if (a.out1) a.out1[g * 4 + v] = s1[v];
    }
  }
}
static bool pool2_fast_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("DFB_POOL2_FAST");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}
// returns false when the geometry is not the fast kernel's
static bool launch_pool2_bwd(SumsArgs a, int N, int C, dfb_status* st) {
  constexpr int U = 2;
  const int G = C / 4;
  if (!pool2_fast_enabled() || a.pool_k != 2 || (a.H & 1) || (a.W & 1) || (C & 3) || G > kT || kT % G != 0) return false;
  if ((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.dy) | reinterpret_cast<uintptr_t>(a.pool_y) |
       reinterpret_cast<uintptr_t>(a.dy_out) | reinterpret_cast<uintptr_t>(a.mean) | reinterpret_cast<uintptr_t>(a.invstd)) & 15)
    return false;
  const size_t prows = (size_t)N * a.OH * a.OW;
  const int lanes = kT / G;
  const size_t smem = (size_t)lanes * 2 * C * sizeof(float);
  if (prows >= (1ull << 31) || smem > 48 * 1024) return false;
  const size_t unit = (size_t)lanes * U;                       // windows one pass of a CTA covers
  const size_t units = (prows + unit - 1) / unit;
  const size_t cap = (size_t)sm_count() * 2;                   // one wave at two CTAs per SM
  const size_t per_cta = (units + cap - 1) / cap;
  const unsigned ctas = (unsigned)((units + per_cta - 1) / per_cta);
  a.ticket = ticket_counter(SUMS_POOLBN);
  float* part = nullptr;
  *st = dfb_malloc((size_t)ctas * 2 * C, &part);
  if (*st != DFB_OK) return true;
  a.part = part;
  launch_k(pool2_relu_bn_bwd_kernel<U>, ctas, kT, smem, compute_stream(), a, (unsigned)prows, C, (unsigned)(per_cta * unit), lanes);
  dfb_free(part);  // stream-ordered
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("maxpool_relu_bn_bwd kernel launch failed: %s", cudaGetErrorString(e));
    *st = DFB_ERR_RUNTIME;
  }
  return true;
}

template <int KIND>
static dfb_status launch_col_sums(const char* name, SumsArgs a, size_t rows, int C, const void* p0, const void* p1 = nullptr) {
  ColPlan p = plan_cols(rows, C, p0, p1);
  size_t smem = p.lanes > 1 ? (size_t)p.lanes * 2 * C * sizeof(float) : 0;
  DFB_REQUIRE(smem <= 48 * 1024, DFB_ERR_INVALID, "%s: %d channels need %zu B of shared memory", name, C, smem);
  a.ticket = ticket_counter(KIND);
  DFB_REQUIRE(a.ticket != nullptr, DFB_ERR_NOMEM, "%s: cannot allocate the ticket counters", name);
  float* part = nullptr;
  dfb_status st = dfb_malloc((size_t)p.ctas * 2 * C, &part);
  if (st != DFB_OK) return st;
  a.part = part;
  cudaStream_t s = compute_stream();
  if (p.V == 4) launch_k(col_sums_kernel<4, KIND>, p.ctas, kT, smem, s, a, rows, C, p);
  else launch_k(col_sums_kernel<1, KIND>, p.ctas, kT, smem, s, a, rows, C, p);
  dfb_free(part);  // stream-ordered: the next user of the block runs after this kernel
  DFB_LAUNCH_CHECK(name);
  return DFB_OK;
}

// -------------------------------------------------------------------------------------------------
// BatchNorm for small activations (a few MB: the deep layers of a CIFAR-size net): ONE kernel per
// direction. A CTA of 1024 threads owns a block of CB channels for ALL rows, so the statistics need no
// cross-CTA step: pass 1 accumulates the two sums per channel (thread = (float4 channel group, row lane),
// four rows in flight), a fixed-order shuffle + shared-memory tree adds the lanes, pass 2 re-reads the rows
// (L2 hits) and writes the result. Versus the two-kernel path this saves a launch and a dependent
// global-memory round trip per BatchNorm, which is what these launch-latency-bound layers cost.
// -------------------------------------------------------------------------------------------------
constexpr int kSmallT = 1024;
// sums s0, s1 (float4 each) over all row lanes of the CTA; result valid in lane 0 of each group (tid < GPB)
template <int GPB>
__device__ __forceinline__ void block_lane_sum(float (&s0)[4], float (&s1)[4], float* sm /* [32 warps][GPB][8] */) {
  // threads are (lane * GPB + g): xor offsets >= GPB stay inside a channel group
#pragma unroll
  for (int off = 16; off >= GPB; off >>= 1)
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      s0[v] += __shfl_xor_sync(0xffffffffu, s0[v], off);
      s1[v] += __shfl_xor_sync(0xffffffffu, s1[v], off);
    }
  const int warp = threadIdx.x >> 5, lane_in_warp = threadIdx.x & 31;
  __syncthreads();
  if (lane_in_warp < GPB) {
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      sm[(warp * GPB + lane_in_warp) * 8 + v] = s0[v];
      sm[(warp * GPB + lane_in_warp) * 8 + 4 + v] = s1[v];
    }
  }
  __syncthreads();
  if (threadIdx.x < GPB) {
#pragma unroll
    for (int v = 0; v < 4; ++v) { s0[v] = 0.f; s1[v] = 0.f; }
    for (int w = 0; w < kSmallT / 32; ++w)
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        s0[v] += sm[(w * GPB + threadIdx.x) * 8 + v];
        s1[v] += sm[(w * GPB + threadIdx.x) * 8 + 4 + v];
      }
  }
  // The CTAs of a cluster own the same channels and different rows: publish this CTA's totals, then add all
  // ranks' totals in rank order (every CTA gets the same bits) through distributed shared memory.
  const int nrank = (int)cluster_nctarank();
  if (nrank > 1) {
    float* pub = sm + (kSmallT / 32) * GPB * 8;  // [GPB][8]
    if (threadIdx.x < GPB) {
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        pub[threadIdx.x * 8 + v] = s0[v];
        pub[threadIdx.x * 8 + 4 + v] = s1[v];
      }
    }
    cluster_arrive();
    cluster_wait();
    if (threadIdx.x < GPB) {
      const uint32_t mine = smem_addr_u32(pub + threadIdx.x * 8);
      float t[8][8];
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < nrank) {
          const uint32_t remote = dsmem_addr(mine, (uint32_t)r);
#pragma unroll
          for (int v = 0; v < 8; ++v) t[r][v] = ld_dsmem_f32(remote + 4u * v);
        }
#pragma unroll
      for (int v = 0; v < 4; ++v) { s0[v] = 0.f; s1[v] = 0.f; }
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if (r < nrank) {
#pragma unroll
          for (int v = 0; v < 4; ++v) { s0[v] += t[r][v]; s1[v] += t[r][4 + v]; }
        }
    }
    cluster_arrive();  // peers may leave only after everybody has read their totals; waited for at kernel end
  }
}
// pairs with the trailing cluster_arrive() of block_lane_sum
__device__ __forceinline__ void block_lane_sum_finish() {
  if (cluster_nctarank() > 1) cluster_wait();
}

template <int GPB>  // float4 channel groups per CTA (CB = 4 * GPB channels)
__global__ void __launch_bounds__(kSmallT)
bn_small_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                    float* __restrict__ y, float* __restrict__ save_mean, float* __restrict__ save_invstd,
                    float* __restrict__ running_mean, float* __restrict__ running_var, float momentum, float eps, int rows,
                    int C) {
  pdl_sync();
  __shared__ float sm[(kSmallT / 32) * GPB * 8 + GPB * 8];
  __shared__ float s_scale[GPB * 4], s_shift[GPB * 4], s_mean[GPB * 4];
  const int g = threadIdx.x % GPB, lane = threadIdx.x / GPB;
  constexpr int kLanes = kSmallT / GPB;
  // cluster of S CTAs along x: same channel block, rows split S ways
  const int nrank = (int)cluster_nctarank(), rank = (int)cluster_ctarank();
  const int c0 = (((int)blockIdx.x / nrank) * GPB + g) * 4;
  const int rows_per = (rows + nrank - 1) / nrank;
  const int r_lo = rank * rows_per, r_hi = min(rows, r_lo + rows_per);
  const float* xc = x + c0;
  float shift[4], s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
  Vec<4>::get(xc, shift);  // row 0 (the same shift in every CTA)
  int r = r_lo + lane;
  for (; r + 3 * kLanes < r_hi; r += 4 * kLanes) {
    float v[4][4];
#pragma unroll
    for (int u = 0; u < 4; ++u) Vec<4>::get(xc + (size_t)(r + u * kLanes) * C, v[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int q = 0; q < 4; ++q) { float d = v[u][q] - shift[q]; s0[q] += d; s1[q] = fmaf(d, d, s1[q]); }
  }
  for (; r < r_hi; r += kLanes) {
    float v[4];
    Vec<4>::get(xc + (size_t)r * C, v);
#pragma unroll
    for (int q = 0; q < 4; ++q) { float d = v[q] - shift[q]; s0[q] += d; s1[q] = fmaf(d, d, s1[q]); }
  }
  block_lane_sum<GPB>(s0, s1, sm);
  if (threadIdx.x < GPB) {
    const float n = (float)rows;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int c = c0 + q;
      const float dm = s0[q] / n;
      const float mean = shift[q] + dm;
      const float var = fmaxf(s1[q] / n - dm * dm, 0.f);   // biased, like batchnorm.py:38-42
      const float invstd = 1.0f / sqrtf(var + eps);
      if (rank == 0) {  // every rank holds the same values; one of them publishes
        save_mean[c] = mean;
        save_invstd[c] = invstd;
        if (running_mean) running_mean[c] = running_mean[c] * (1.0f - momentum) + mean * momentum;
        if (running_var) running_var[c] = running_var[c] * (1.0f - momentum) + var * momentum;
      }
      s_scale[g * 4 + q] = invstd * (gamma ? gamma[c] : 1.0f);
      s_shift[g * 4 + q] = beta ? beta[c] : 0.0f;
      s_mean[g * 4 + q] = mean;
    }
  }
  __syncthreads();
  float sc[4], sh[4], mu[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) { sc[q] = s_scale[g * 4 + q]; sh[q] = s_shift[g * 4 + q]; mu[q] = s_mean[g * 4 + q]; }
  // y = (x - mean) * (invstd * gamma) + beta; subtracting the mean first keeps the result accurate when |mean| >> std
  for (r = r_lo + lane; r < r_hi; r += kLanes) {
    float v[4], o[4];
    Vec<4>::get(xc + (size_t)r * C, v);
#pragma unroll
    for (int q = 0; q < 4; ++q) o[q] = fmaf(v[q] - mu[q], sc[q], sh[q]);
    Vec<4>::put(y + c0 + (size_t)r * C, o);
  }
  block_lane_sum_finish();
}

template <int GPB>
__global__ void __launch_bounds__(kSmallT)
bn_small_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, const float* __restrict__ gamma,
                    const float* __restrict__ mean, const float* __restrict__ invstd, float* __restrict__ dx,
                    float* __restrict__ dgamma, float* __restrict__ dbeta, int rows, int C) {
  pdl_sync();
  __shared__ float sm[(kSmallT / 32) * GPB * 8 + GPB * 8];
  __shared__ float s_mb[GPB * 4], s_mg[GPB * 4];
  const int g = threadIdx.x % GPB, lane = threadIdx.x / GPB;
  constexpr int kLanes = kSmallT / GPB;
  const int nrank = (int)cluster_nctarank(), rank = (int)cluster_ctarank();
  const int c0 = (((int)blockIdx.x / nrank) * GPB + g) * 4;
  const int rows_per = (rows + nrank - 1) / nrank;
  const int r_lo = rank * rows_per, r_hi = min(rows, r_lo + rows_per);
  const float* xc = x + c0;
  const float* dc = dy + c0;
  float mu[4], is[4], s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
  Vec<4>::get(mean + c0, mu);
  Vec<4>::get(invstd + c0, is);
  int r = r_lo + lane;
  for (; r + 1 * kLanes < r_hi; r += 2 * kLanes) {
    float xv[2][4], dv[2][4];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      Vec<4>::get(xc + (size_t)(r + u * kLanes) * C, xv[u]);
      Vec<4>::get(dc + (size_t)(r + u * kLanes) * C, dv[u]);
    }
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int q = 0; q < 4; ++q) { s0[q] += dv[u][q]; s1[q] = fmaf(dv[u][q], (xv[u][q] - mu[q]) * is[q], s1[q]); }
  }
  for (; r < r_hi; r += kLanes) {
    float xv[4], dv[4];
    Vec<4>::get(xc + (size_t)r * C, xv);
    Vec<4>::get(dc + (size_t)r * C, dv);
#pragma unroll
    for (int q = 0; q < 4; ++q) { s0[q] += dv[q]; s1[q] = fmaf(dv[q], (xv[q] - mu[q]) * is[q], s1[q]); }
  }
  block_lane_sum<GPB>(s0, s1, sm);
  if (threadIdx.x < GPB) {
    const float inv_n = 1.0f / (float)rows;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (dbeta && rank == 0) dbeta[c0 + q] = s0[q];
      if (dgamma && rank == 0) dgamma[c0 + q] = s1[q];
      s_mb[g * 4 + q] = s0[q] * inv_n;
      s_mg[g * 4 + q] = s1[q] * inv_n;
    }
  }
  __syncthreads();
  if (!dx) {
    block_lane_sum_finish();
    return;
  }
  float k1[4], mb[4], mg[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    k1[q] = is[q] * (gamma ? gamma[c0 + q] : 1.0f);
    mb[q] = s_mb[g * 4 + q];
    mg[q] = s_mg[g * 4 + q];
  }
  for (r = r_lo + lane; r < r_hi; r += kLanes) {
    float xv[4], dv[4], o[4];
    Vec<4>::get(xc + (size_t)r * C, xv);
    Vec<4>::get(dc + (size_t)r * C, dv);
#pragma unroll
    for (int q = 0; q < 4; ++q) o[q] = k1[q] * (dv[q] - mb[q] - (xv[q] - mu[q]) * is[q] * mg[q]);
    Vec<4>::put(dx + c0 + (size_t)r * C, o);
  }
  block_lane_sum_finish();
}

// Plan of the single-kernel path: channel groups per CTA (0 = use the two-kernel path) and cluster size S (CTAs
// that split the rows of one channel block).
struct SmallBnPlan { int gpb, cluster; };
static SmallBnPlan bn_small_plan(bool fwd, size_t rows, int C, const void* a, const void* b = nullptr, const void* c = nullptr) {
  // Only while a thread sees at most four rows per pass (one batch of loads in flight): with more, the CTAs of
  // this path become chains of dependent-latency loads and the two-kernel path (hundreds of CTAs) wins.
  if (C % 16 != 0 || rows < 64) return {0, 1};
  if (((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c)) & 15) != 0) return {0, 1};
  const int groups = C / 4;
  if (rows <= 1024) {
    const int gpb = rows > 512 ? 4 : (rows > 256 ? 2 : 1);   // 256 / 512 / 1024 row lanes per CTA
    return {groups % gpb == 0 ? gpb : 0, 1};
  }
  // larger: a cluster of 8 CTAs per channel block, about two rows per thread and pass
  // (16-byte row segments - one channel group per CTA - measured slower than the two-kernel path)
  // forward reads one tensor, backward two: the forward pass still wins with four rows per thread and pass
  // (16384 x 64: 10.7 us vs 12.3 us for the two-kernel path; backward 12.6 us vs 11.0 us)
  const size_t limit = fwd ? 32768 : 16384;
  for (int gpb = 4; gpb >= 2; gpb >>= 1)
    if (rows * gpb <= limit && groups % gpb == 0) return {gpb, 8};
  return {0, 1};
}

// y = (x - mean) * (invstd * gamma) + beta, optionally followed by max(.,0)
template <int V, bool RELU>
__global__ void __launch_bounds__(kT)
bn_apply_kernel(const float* __restrict__ x, float* __restrict__ y, size_t rows, int C,
                const float* __restrict__ mean, const float* __restrict__ invstd,
                const float* __restrict__ gamma, const float* __restrict__ beta) {
  pdl_sync();
  extern __shared__ float sm[];  // mean[C], scale[C], shift[C]
  float* s_mean = sm;
  float* s_scale = sm + C;
  float* s_shift = sm + 2 * C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    s_mean[c] = mean[c];
    s_scale[c] = invstd[c] * (gamma ? gamma[c] : 1.0f);
    s_shift[c] = beta ? beta[c] : 0.0f;
  }
  __syncthreads();
  const int G = C / V;
  size_t total = rows * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    float xv[V], yv[V];
    Vec<V>::get(x + i * V, xv);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      int c = g * V + v;
      float t = fmaf(xv[v] - s_mean[c], s_scale[c], s_shift[c]);
      yv[v] = RELU ? fmaxf(t, 0.f) : t;
    }
    Vec<V>::put(y + i * V, yv);
  }
}

// Statistic slot as the source of a BatchNorm kernel's per-channel sums (kernels.cuh): `row` = which of the slot's rows
// holds the second sum, `clear` = this launch is the slot's last consumer.
struct StatSrc {
  double* acc;
  int row, clear;
};
// Called by every thread of every CTA after the CTA has read what it needs from the slot (and synchronised): the last CTA
// to arrive clears the slot for its next user.
__device__ __forceinline__ void stat_slot_release(double* acc, int C) {
  __shared__ int s_last;
  unsigned* counter = stat_slot_counter(acc);
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = atomicAdd(counter, 1u) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last) {
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      acc[c] = 0.0;
      acc[kStatSlotChannels + c] = 0.0;
      acc[2 * kStatSlotChannels + c] = 0.0;
    }
    if (threadIdx.x == 0) *counter = 0u;
  }
}

// pass 2: dx = gamma * invstd * (dy - dbeta/n - x_hat * dgamma/n)
template <int V>
__global__ void __launch_bounds__(kT)
bn_bwd_apply_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx,
                    size_t rows, int C, const float* __restrict__ mean, const float* __restrict__ invstd,
                    const float* __restrict__ gamma, float* dbeta, float* dgamma, StatSrc src) {
  pdl_sync();
  extern __shared__ float sm[];  // mean, invstd, k1 = gamma*invstd, mb = dbeta/n, mg = dgamma/n
  float* s_mean = sm;
  float* s_is = sm + C;
  float* s_k1 = sm + 2 * C;
  float* s_mb = sm + 3 * C;
  float* s_mg = sm + 4 * C;
  float inv_n = 1.0f / (float)rows;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float db, dg;
    if (src.acc) {   // the sums are still in the statistic slot the dgrad epilogue added them to (kernels.cuh)
      db = (float)__ldcg(src.acc + c);
      dg = (float)__ldcg(src.acc + src.row * kStatSlotChannels + c);
      if (blockIdx.x == 0) { dbeta[c] = db; dgamma[c] = dg; }   // the parameter gradients themselves
    } else {
      db = dbeta[c];
      dg = dgamma[c];
    }
    s_mean[c] = mean[c];
    s_is[c] = invstd[c];
    s_k1[c] = invstd[c] * (gamma ? gamma[c] : 1.0f);
    s_mb[c] = db * inv_n;
    s_mg[c] = dg * inv_n;
  }
  __syncthreads();
  if (src.acc && src.clear) stat_slot_release(src.acc, C);
  const int G = C / V;
  size_t total = rows * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    float xv[V], dv[V], ov[V];
    Vec<V>::get(x + i * V, xv);
    Vec<V>::get(dy + i * V, dv);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      int c = g * V + v;
      float xh = (xv[v] - s_mean[c]) * s_is[c];
      ov[v] = s_k1[c] * (dv[v] - s_mb[c] - xh * s_mg[c]);
    }
    Vec<V>::put(dx + i * V, ov);
  }
}

// -------------------------------------------------------------------------------------------------
// elementwise
// -------------------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(kT)
add_rowvec_kernel(const float* __restrict__ x, const float* __restrict__ vec, float* __restrict__ y,
                  size_t rows, int C) {
  pdl_sync();
  const int G = C / V;
  size_t total = rows * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    float xv[V], bv[V];
    Vec<V>::get(x + i * V, xv);
    Vec<V>::get(vec + (size_t)g * V, bv);
#pragma unroll
    for (int v = 0; v < V; ++v) xv[v] += bv[v];
    Vec<V>::put(y + i * V, xv);
  }
}

__global__ void __launch_bounds__(kT)
relu_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx, size_t n) {
  pdl_sync();
  size_t stride = (size_t)gridDim.x * blockDim.x;
  size_t n4 = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy) |
                reinterpret_cast<uintptr_t>(dx)) & 15) == 0 ? n / 4 : 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
    float4 a = ld_stream(reinterpret_cast<const float4*>(x) + i);
    float4 d = ld_stream(reinterpret_cast<const float4*>(dy) + i);
    float4 o;
    // maximum.grad_fn: (max(x,0) == x) * dy  <=>  x >= 0 ? dy : 0   (tensor.py:872-877)
    o.x = a.x >= 0.f ? d.x : 0.f; o.y = a.y >= 0.f ? d.y : 0.f;
    o.z = a.z >= 0.f ? d.z : 0.f; o.w = a.w >= 0.f ? d.w : 0.f;
    st_stream(reinterpret_cast<float4*>(dx) + i, o);
  }
  for (size_t i = n4 * 4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    dx[i] = x[i] >= 0.f ? dy[i] : 0.f;
}

// -------------------------------------------------------------------------------------------------
// pooling (window k, stride k, no padding) on NHWC
// -------------------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(kT)
maxpool_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int32_t* __restrict__ idx, int N,
                   int H, int W, int C, int k, int OH, int OW) {
  pdl_sync();
  const int G = C / V;
  size_t total = (size_t)N * OH * OW * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    size_t t = i / G;
    int ow = (int)(t % OW);
    t /= OW;
    int oh = (int)(t % OH);
    int n = (int)(t / OH);
    float best[V];
    int bi[V];
#pragma unroll
    for (int v = 0; v < V; ++v) { best[v] = -INFINITY; bi[v] = 0; }
    for (int r = 0; r < k; ++r)
      for (int s = 0; s < k; ++s) {
        float xv[V];
        Vec<V>::get(x + (((size_t)n * H + oh * k + r) * W + ow * k + s) * C + (size_t)g * V, xv);
#pragma unroll
        for (int v = 0; v < V; ++v)
          if (xv[v] > best[v] || (r == 0 && s == 0)) { best[v] = xv[v]; bi[v] = r * k + s; }
      }
    Vec<V>::put(y + i * V, best);
    if (idx) {
#pragma unroll
      for (int v = 0; v < V; ++v) idx[i * V + v] = bi[v];
    }
  }
}

// MODE 0: every tied maximum receives dy (reference, tensor.py:779-791); MODE 1: arg-max routed
template <int V, int MODE>
__global__ void __launch_bounds__(kT)
maxpool_bwd_kernel(const float* __restrict__ x, const float* __restrict__ y, const int32_t* __restrict__ idx,
                   const float* __restrict__ dy, float* __restrict__ dx, int N, int H, int W, int C, int k,
                   int OH, int OW) {
  pdl_sync();
  const int G = C / V;
  size_t total = (size_t)N * H * W * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    size_t t = i / G;
    int w = (int)(t % W);
    t /= W;
    int h = (int)(t % H);
    int n = (int)(t / H);
    int oh = h / k, ow = w / k;
    float o[V];
#pragma unroll
    for (int v = 0; v < V; ++v) o[v] = 0.f;
    if (oh < OH && ow < OW) {
      size_t oo = (((size_t)n * OH + oh) * OW + ow) * C + (size_t)g * V;
      float dv[V];
      Vec<V>::get(dy + oo, dv);
      if (MODE == 0) {
        float xv[V], yv[V];
        Vec<V>::get(x + i * V, xv);
        Vec<V>::get(y + oo, yv);
#pragma unroll
        for (int v = 0; v < V; ++v) o[v] = xv[v] == yv[v] ? dv[v] : 0.f;
      } else {
        int pos = (h - oh * k) * k + (w - ow * k);
#pragma unroll
        for (int v = 0; v < V; ++v) o[v] = idx[oo + v] == pos ? dv[v] : 0.f;
      }
    }
    Vec<V>::put(dx + i * V, o);
  }
}

template <int V>
__global__ void __launch_bounds__(kT)
avgpool_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int H, int W, int C, int k,
                   int OH, int OW) {
  pdl_sync();
  const int G = C / V;
  size_t total = (size_t)N * OH * OW * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  float inv = 1.0f / (float)(k * k);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    size_t t = i / G;
    int ow = (int)(t % OW);
    t /= OW;
    int oh = (int)(t % OH);
    int n = (int)(t / OH);
    float acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = 0.f;
    for (int r = 0; r < k; ++r)
      for (int s = 0; s < k; ++s) {
        float xv[V];
        Vec<V>::get(x + (((size_t)n * H + oh * k + r) * W + ow * k + s) * C + (size_t)g * V, xv);
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v] += xv[v];
      }
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] *= inv;
    Vec<V>::put(y + i * V, acc);
  }
}
template <int V>
__global__ void __launch_bounds__(kT)
avgpool_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, int N, int H, int W, int C, int k,
                   int OH, int OW) {
  pdl_sync();
  const int G = C / V;
  size_t total = (size_t)N * H * W * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  float inv = 1.0f / (float)(k * k);
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    size_t t = i / G;
    int w = (int)(t % W);
    t /= W;
    int h = (int)(t % H);
    int n = (int)(t / H);
    int oh = h / k, ow = w / k;
    float o[V];
#pragma unroll
    for (int v = 0; v < V; ++v) o[v] = 0.f;
    if (oh < OH && ow < OW) {
      Vec<V>::get(dy + (((size_t)n * OH + oh) * OW + ow) * C + (size_t)g * V, o);
#pragma unroll
      for (int v = 0; v < V; ++v) o[v] *= inv;
    }
    Vec<V>::put(dx + i * V, o);
  }
}

// -------------------------------------------------------------------------------------------------
// upsampling by an integer factor s on NHWC: x [N,H,W,C] -> y [N,H*s,W*s,C]. Both backward kernels gather (one thread per
// input pixel sums, in a fixed order, every output gradient that read it): no atomics, so results do not depend on scheduling.
// -------------------------------------------------------------------------------------------------
template <int V>
__global__ void __launch_bounds__(kT)
upsample_nearest_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int H, int W, int C, int s) {
  pdl_sync();
  const int G = C / V, OH = H * s, OW = W * s;
  size_t total = (size_t)N * OH * OW * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    size_t t = i / G;
    int ow = (int)(t % OW);
    t /= OW;
    int oh = (int)(t % OH);
    int n = (int)(t / OH);
    float v[V];
    Vec<V>::get(x + (((size_t)n * H + oh / s) * W + ow / s) * C + (size_t)g * V, v);
    Vec<V>::put(y + i * V, v);
  }
}

template <int V>
__global__ void __launch_bounds__(kT)
upsample_nearest_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, int N, int H, int W, int C, int s) {
  pdl_sync();
  const int G = C / V, OH = H * s, OW = W * s;
  size_t total = (size_t)N * H * W * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    size_t t = i / G;
    int w = (int)(t % W);
    t /= W;
    int h = (int)(t % H);
    int n = (int)(t / H);
    float acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = 0.f;
    for (int a = 0; a < s; ++a)
      for (int b = 0; b < s; ++b) {
        float d[V];
        Vec<V>::get(dy + (((size_t)n * OH + h * s + a) * OW + w * s + b) * C + (size_t)g * V, d);
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v] += d[v];
      }
    Vec<V>::put(dx + i * V, acc);
  }
}

// Bilinear, align_corners=False (PyTorch's rule for an integer scale): output index o reads input indices i0 and i1
// (i1 == i0 on the last row / column) with weights l0 and l1. Forward and backward use this one function, so the
// backward finds exactly the taps the forward pass used.
struct UpLerp {
  int i0, i1;
  float l0, l1;
};
__device__ __forceinline__ UpLerp up_lerp(int o, int s, int n) {
  const float src = fmaxf(0.f, ((float)o + 0.5f) / (float)s - 0.5f);
  UpLerp r;
  r.i0 = (int)src;
  r.i1 = r.i0 + (r.i0 < n - 1 ? 1 : 0);
  r.l1 = src - (float)r.i0;
  r.l0 = 1.f - r.l1;
  return r;
}

template <int V>
__global__ void __launch_bounds__(kT)
upsample_bilinear_fwd_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int H, int W, int C, int s) {
  pdl_sync();
  const int G = C / V, OH = H * s, OW = W * s;
  size_t total = (size_t)N * OH * OW * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    size_t t = i / G;
    int ow = (int)(t % OW);
    t /= OW;
    int oh = (int)(t % OH);
    int n = (int)(t / OH);
    const UpLerp r = up_lerp(oh, s, H), c = up_lerp(ow, s, W);
    const float* base = x + (size_t)n * H * W * C + (size_t)g * V;
    float x00[V], x01[V], x10[V], x11[V], o[V];
    Vec<V>::get(base + ((size_t)r.i0 * W + c.i0) * C, x00);
    Vec<V>::get(base + ((size_t)r.i0 * W + c.i1) * C, x01);
    Vec<V>::get(base + ((size_t)r.i1 * W + c.i0) * C, x10);
    Vec<V>::get(base + ((size_t)r.i1 * W + c.i1) * C, x11);
#pragma unroll
    for (int v = 0; v < V; ++v)
      o[v] = r.l0 * (c.l0 * x00[v] + c.l1 * x01[v]) + r.l1 * (c.l0 * x10[v] + c.l1 * x11[v]);
    Vec<V>::put(y + i * V, o);
  }
}

template <int V>
__global__ void __launch_bounds__(kT)
upsample_bilinear_bwd_kernel(const float* __restrict__ dy, float* __restrict__ dx, int N, int H, int W, int C, int s) {
  pdl_sync();
  const int G = C / V, OH = H * s, OW = W * s;
  size_t total = (size_t)N * H * W * G;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    int g = (int)(i % G);
    size_t t = i / G;
    int w = (int)(t % W);
    t /= W;
    int h = (int)(t % H);
    int n = (int)(t / H);
    float acc[V];
#pragma unroll
    for (int v = 0; v < V; ++v) acc[v] = 0.f;
    // an output index o has i0 = floor(max(0, (o + 0.5) / s - 0.5)): it reads input h (as i0 or i1) only when
    // i0 is h - 1 or h, which needs s * (h - 1) <= o < s * (h + 2)
    const int oh0 = max(0, s * (h - 1)), oh1 = min(OH, s * (h + 2));
    const int ow0 = max(0, s * (w - 1)), ow1 = min(OW, s * (w + 2));
    for (int oh = oh0; oh < oh1; ++oh) {
      const UpLerp r = up_lerp(oh, s, H);
      if (r.i0 != h && r.i1 != h) continue;
      const float wr = (r.i0 == h ? r.l0 : 0.f) + (r.i1 == h ? r.l1 : 0.f);
      for (int ow = ow0; ow < ow1; ++ow) {
        const UpLerp c = up_lerp(ow, s, W);
        if (c.i0 != w && c.i1 != w) continue;
        const float wt = wr * ((c.i0 == w ? c.l0 : 0.f) + (c.i1 == w ? c.l1 : 0.f));
        float d[V];
        Vec<V>::get(dy + (((size_t)n * OH + oh) * OW + ow) * C + (size_t)g * V, d);
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v] += wt * d[v];
      }
    }
    Vec<V>::put(dx + i * V, acc);
  }
}

// -------------------------------------------------------------------------------------------------
// channel concatenation on NHWC: slice s is a [rows, width[s]] matrix and occupies columns off[s] .. off[s] + width[s]
// of y [rows, C]. The slice table is a kernel parameter, so a captured graph keeps it in the kernel node (no device
// table, no upload). blockIdx.y picks the slice; its CTAs walk it with a grid-stride loop, kConcatUnroll vectors per
// thread loaded before any is stored: the slice side is read / written contiguously, the y side in row segments.
// -------------------------------------------------------------------------------------------------
constexpr int kConcatUnroll = 4;
struct ConcatSlices {
  float* p[DFB_CONCAT_MAX_SOURCES];   // the source (forward) or its gradient (backward)
  int off[DFB_CONCAT_MAX_SOURCES];
  int width[DFB_CONCAT_MAX_SOURCES];
};

template <int V, bool BWD>
__global__ void __launch_bounds__(kT)
concat_channels_kernel(const __grid_constant__ ConcatSlices t, float* __restrict__ y, int C, long long rows) {
  pdl_sync();
  const int s = blockIdx.y;
  float* __restrict__ part = t.p[s];
  float* __restrict__ ys = y + t.off[s];
  const int G = t.width[s] / V;
  const size_t total = (size_t)rows * G;
  const size_t stride = (size_t)gridDim.x * blockDim.x * kConcatUnroll;
  for (size_t base = (size_t)blockIdx.x * blockDim.x * kConcatUnroll + threadIdx.x; base < total; base += stride) {
    float v[kConcatUnroll][V];
#pragma unroll
    for (int u = 0; u < kConcatUnroll; ++u) {
      const size_t i = base + (size_t)u * blockDim.x;
      if (i >= total) break;
      const size_t r = i / G;
      Vec<V>::get(BWD ? ys + r * C + (i - r * G) * V : part + i * V, v[u]);
    }
#pragma unroll
    for (int u = 0; u < kConcatUnroll; ++u) {
      const size_t i = base + (size_t)u * blockDim.x;
      if (i >= total) break;
      const size_t r = i / G;
      Vec<V>::put(BWD ? part + i * V : ys + r * C + (i - r * G) * V, v[u]);
    }
  }
}

// -------------------------------------------------------------------------------------------------
// softmax cross-entropy with dense targets. One CTA: the batch dimension of every config is
// <= a few thousand rows, and a single CTA keeps the sum order fixed.
// -------------------------------------------------------------------------------------------------
constexpr int kCeThreads = 1024;
__global__ void __launch_bounds__(kCeThreads)
softmax_ce_fwd_kernel(const float* __restrict__ logits, const float* __restrict__ target,
                      float* __restrict__ loss, size_t rows, int cols, float scale) {
  pdl_sync();
  __shared__ float warp_part[kCeThreads / 32];
  float acc = 0.f;
  for (size_t r = threadIdx.x; r < rows; r += blockDim.x) {
    const float* xr = logits + r * cols;
    const float* tr = target + r * cols;
    float m = -INFINITY;
    for (int j = 0; j < cols; ++j) m = fmaxf(m, xr[j]);
    float se = 0.f;
    for (int j = 0; j < cols; ++j) se += expf(xr[j] - m);
    float lse = logf(se);
    float row = 0.f;
    for (int j = 0; j < cols; ++j) row += -((xr[j] - m) - lse) * tr[j];
    acc += row;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) warp_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < kCeThreads / 32 ? warp_part[threadIdx.x] : 0.f;
    v = warp_sum(v);
    if (threadIdx.x == 0) loss[0] = v * scale;
  }
}
__global__ void __launch_bounds__(kT)
softmax_ce_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ target,
                      const float* __restrict__ upstream, float* __restrict__ dlogits, size_t rows,
                      int cols, float scale) {
  pdl_sync();
  float k = scale * (upstream ? upstream[0] : 1.0f);
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += stride) {
    const float* xr = logits + r * cols;
    const float* tr = target + r * cols;
    float m = -INFINITY, ts = 0.f;
    for (int j = 0; j < cols; ++j) { m = fmaxf(m, xr[j]); ts += tr[j]; }
    float se = 0.f;
    for (int j = 0; j < cols; ++j) se += expf(xr[j] - m);
    float inv = 1.0f / se;
    for (int j = 0; j < cols; ++j)
      dlogits[r * cols + j] = k * (expf(xr[j] - m) * inv * ts - tr[j]);
  }
}


// -------------------------------------------------------------------------------------------------
// BatchNorm forward from statistics that already exist (the producing convolution's epilogue, or
// dfb_colstats_mean_var): ONE pass that normalises, and - when the host saw them coming - also adds the
// other branch of a residual block (a plain tensor, or a second BatchNorm applied on the fly: the shortcut's
// conv + BatchNorm) and applies ReLU. Replaces bn_stats + bn_apply (+ binary add) (+ scalar_maximum).
// CTA 0 additionally publishes mean / invstd for the backward pass and updates the running statistics.
// -------------------------------------------------------------------------------------------------
struct BnSide {
  const float* x;
  const float* mean_var;   // [2][C]: batch mean, biased batch variance
  const float* gamma;
  const float* beta;
  float* save_mean;
  float* save_invstd;
  float* running_mean;
  float* running_var;
  float momentum, eps;
  double* acc;             // statistic slot with sum / sum of squares (lazy producer), or null: mean_var holds the floats
  float* mean_var_out;     // where CTA 0 publishes mean / variance taken from the slot
  float inv_rows;
};
__device__ __forceinline__ void bn_side_prologue(const BnSide& s, int C, float* s_mean, float* s_scale, float* s_shift) {
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float mean, var;
    if (s.acc) {
      const double m = __ldcg(s.acc + c) * (double)s.inv_rows;
      const double v = __ldcg(s.acc + kStatSlotChannels + c) * (double)s.inv_rows - m * m;   // biased variance (batchnorm.py:38-42)
      mean = (float)m;
      var = fmaxf((float)v, 0.0f);
      if (blockIdx.x == 0) { s.mean_var_out[c] = mean; s.mean_var_out[C + c] = var; }
    } else {
      mean = s.mean_var[c];
      var = s.mean_var[C + c];
    }
    const float invstd = 1.0f / sqrtf(var + s.eps);
    s_mean[c] = mean;
    s_scale[c] = invstd * (s.gamma ? s.gamma[c] : 1.0f);
    s_shift[c] = s.beta ? s.beta[c] : 0.0f;
    if (blockIdx.x == 0) {
      s.save_mean[c] = mean;
      s.save_invstd[c] = invstd;
      if (s.running_mean) s.running_mean[c] = s.running_mean[c] * (1.0f - s.momentum) + mean * s.momentum;
      if (s.running_var) s.running_var[c] = s.running_var[c] * (1.0f - s.momentum) + var * s.momentum;
    }
  }
}
template <int V, bool RELU, bool DUAL, bool RES>
__global__ void __launch_bounds__(kT)
bn_apply_fused_kernel(BnSide a, BnSide b, const float* __restrict__ res, float* __restrict__ y, size_t rows, int C) {
  pdl_sync();
  extern __shared__ float sm[];  // mean, scale, shift per side
  float* am = sm; float* as = sm + C; float* ah = sm + 2 * C;
  float* bm = sm + 3 * C; float* bs = sm + 4 * C; float* bh = sm + 5 * C;
  bn_side_prologue(a, C, am, as, ah);
  if (DUAL) bn_side_prologue(b, C, bm, bs, bh);
  __syncthreads();
  if (a.acc) stat_slot_release(a.acc, C);
  if (DUAL && b.acc) stat_slot_release(b.acc, C);
  const int G = C / V;
  const size_t total = rows * G;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int g = (int)(i % G);
    float xv[V], x2[V], rv[V], o[V];
    Vec<V>::get(a.x + i * V, xv);
    if (DUAL) Vec<V>::get(b.x + i * V, x2);
    if (RES) Vec<V>::get(res + i * V, rv);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const int c = g * V + v;
      float t = fmaf(xv[v] - am[c], as[c], ah[c]);
      if (DUAL) t = t + fmaf(x2[v] - bm[c], bs[c], bh[c]);
      if (RES) t = t + rv[v];
      o[v] = RELU ? fmaxf(t, 0.f) : t;
    }
    Vec<V>::put(y + i * V, o);
  }
}

// ReLU backward through a fused BatchNorm(+residual)+ReLU: the pre-activation z is recomputed exactly as the forward
// kernel computed it (same operations, same operands), dx = z >= 0 ? dy : 0 (maximum.grad_fn, tensor.py:872-877)
template <int V, bool DUAL, bool RES>
__global__ void __launch_bounds__(kT)
relu_bwd_bn_kernel(const float* __restrict__ xa, const float* __restrict__ mean_a, const float* __restrict__ invstd_a,
                   const float* __restrict__ gamma_a, const float* __restrict__ beta_a, const float* __restrict__ xb,
                   const float* __restrict__ mean_b, const float* __restrict__ invstd_b, const float* __restrict__ gamma_b,
                   const float* __restrict__ beta_b, const float* __restrict__ res, const float* __restrict__ dy,
                   float* __restrict__ dx, size_t rows, int C) {
  pdl_sync();
  extern __shared__ float sm[];
  float* am = sm; float* as = sm + C; float* ah = sm + 2 * C;
  float* bm = sm + 3 * C; float* bs = sm + 4 * C; float* bh = sm + 5 * C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    am[c] = mean_a[c]; as[c] = invstd_a[c] * (gamma_a ? gamma_a[c] : 1.0f); ah[c] = beta_a ? beta_a[c] : 0.0f;
    if (DUAL) { bm[c] = mean_b[c]; bs[c] = invstd_b[c] * (gamma_b ? gamma_b[c] : 1.0f); bh[c] = beta_b ? beta_b[c] : 0.0f; }
  }
  __syncthreads();
  const int G = C / V;
  const size_t total = rows * G;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int g = (int)(i % G);
    float xv[V], x2[V], rv[V], dv[V], o[V];
    Vec<V>::get(xa + i * V, xv);
    if (DUAL) Vec<V>::get(xb + i * V, x2);
    if (RES) Vec<V>::get(res + i * V, rv);
    Vec<V>::get(dy + i * V, dv);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      const int c = g * V + v;
      float t = fmaf(xv[v] - am[c], as[c], ah[c]);
      if (DUAL) t = t + fmaf(x2[v] - bm[c], bs[c], bh[c]);
      if (RES) t = t + rv[v];
      o[v] = t >= 0.f ? dv[v] : 0.f;
    }
    Vec<V>::put(dx + i * V, o);
  }
}

static unsigned ew_grid(size_t items) { return bw_grid(items, kT, 8); }

}  // namespace dfb

namespace dfb {
// -------------------------------------------------------------------------------------------------
// Linear layers with few outputs (the classifier at the end of every network: N <= 16) in ONE launch each way.
// Through the general path x @ W + b is an FFMA GEMM with split-K, its reduction and a row-vector add (three launches,
// 10 us inside the captured ResNet step for 0.66 MFLOP), and the backward a column-sum kernel, two GEMMs and another
// split-K reduction (16 us): all launch floor. F.linear, functional.py:8-12; W is (in, out) like the reference's.
// -------------------------------------------------------------------------------------------------
constexpr int kLinN = 16;
// y[m, :] = x[m, :] . W + b: one warp per row, lanes over k (coalesced x), N running sums per lane, shuffle tree
__global__ void __launch_bounds__(256) linear_small_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                               const float* __restrict__ bias, float* __restrict__ y, int M, int K, int N) {
  pdl_sync();
  const int lane = threadIdx.x & 31, m = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (m >= M) return;
  float acc[kLinN];
#pragma unroll
  for (int n = 0; n < kLinN; ++n) acc[n] = 0.f;
  for (int k0 = lane; k0 < K; k0 += 128) {   // four k per pass: independent loads in flight together
    float xv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) xv[u] = k0 + u * 32 < K ? x[(size_t)m * K + k0 + u * 32] : 0.f;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int k = k0 + u * 32;
      if (k < K) {
        const float* wr = w + (size_t)k * N;
#pragma unroll
        for (int n = 0; n < kLinN; ++n)
          if (n < N) acc[n] = fmaf(xv[u], wr[n], acc[n]);
      }
    }
  }
#pragma unroll
  for (int n = 0; n < kLinN; ++n)
    if (n < N) acc[n] = warp_sum(acc[n]);
  if (lane == 0) {
#pragma unroll
    for (int n = 0; n < kLinN; ++n)
      if (n < N) y[(size_t)m * N + n] = acc[n] + (bias ? bias[n] : 0.f);
  }
}
// One launch, three kinds of CTA (blockIdx ranges), 1024 threads each:
//   dx[m, k] = sum_n dy[m, n] W[k, n]                     one thread per element
//   dW[k, n] = sum_m x[m, k] dy[m, n]                     a CTA per 32 columns k: 32 warps over rows (coalesced x: 256 rows per
//                                                         pass, eight independent loads per lane), lanes own a k; the warps'
//                                                         sums merged through shared memory in warp order, eight warps a round
//   db[n]    = sum_m dy[m, n]                             the last CTA
// (with 8 warps per CTA the weight-gradient CTAs walked the rows in four dependent passes: 13.5 us in the step)
constexpr int kLinT = 1024;
__global__ void __launch_bounds__(kLinT) linear_small_bwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                                 const float* __restrict__ dy, float* __restrict__ dx, float* __restrict__ dw,
                                                                 float* __restrict__ db, int M, int K, int N, int dx_blocks, int dw_blocks) {
  pdl_sync();
  __shared__ float red[8][32][kLinN + 1];
  const int b = blockIdx.x;
  if (b < dx_blocks) {
    const size_t i = (size_t)b * kLinT + threadIdx.x;
    if (i < (size_t)M * K) {
      const int m = (int)(i / K), k = (int)(i - (size_t)m * K);
      const float* g = dy + (size_t)m * N;
      const float* wr = w + (size_t)k * N;
      float acc = 0.f;
#pragma unroll
      for (int n = 0; n < kLinN; ++n)
        if (n < N) acc = fmaf(g[n], wr[n], acc);
      dx[i] = acc;
    }
    return;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;   // 32 warps
  if (b < dx_blocks + dw_blocks) {
    const int k = (b - dx_blocks) * 32 + lane;
    float acc[kLinN];
#pragma unroll
    for (int n = 0; n < kLinN; ++n) acc[n] = 0.f;
    // eight rows per warp and pass: their loads are independent and in flight together (the loop is nothing but load latency)
    for (int m0 = warp; m0 < M; m0 += 256) {
      float xv[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int m = m0 + u * 32;
        xv[u] = (k < K && m < M) ? x[(size_t)m * K + k] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int m = m0 + u * 32;
        if (m < M) {
          const float* g = dy + (size_t)m * N;
#pragma unroll
          for (int n = 0; n < kLinN; ++n)
            if (n < N) acc[n] = fmaf(xv[u], g[n], acc[n]);
        }
      }
    }
    // merge the 32 warps, eight at a time (warp order: deterministic); thread o < 32 * N owns output (k = o / N, n = o % N)
    const int o = threadIdx.x, kl = o / N, n_o = o - kl * N;
    float total = 0.f;
    for (int round = 0; round < 4; ++round) {
      __syncthreads();   // the previous round's sums have been read
      if ((warp >> 3) == round) {
#pragma unroll
        for (int n = 0; n < kLinN; ++n) red[warp & 7][lane][n] = acc[n];
      }
      __syncthreads();
      if (o < 32 * N) {
#pragma unroll
        for (int q = 0; q < 8; ++q) total += red[q][kl][n_o];
      }
    }
    if (o < 32 * N) {
      const int kk = (b - dx_blocks) * 32 + kl;
      if (kk < K) dw[(size_t)kk * N + n_o] = total;
    }
    return;
  }
  // db: thread (row lane r = t / 16 of 64, n = t % 16)
  {
    float* red2 = &red[0][0][0];   // 64 x 16 floats fit the slab (8 x 32 x 17)
    const int n = threadIdx.x & 15, r = threadIdx.x >> 4;
    float acc = 0.f;
    if (n < N) {
#pragma unroll 4
      for (int m = r; m < M; m += 64) acc += dy[(size_t)m * N + n];
    }
    red2[r * 16 + n] = acc;
    __syncthreads();
    if (threadIdx.x < N) {
      float s2 = 0.f;
#pragma unroll 8
      for (int q = 0; q < 64; ++q) s2 += red2[q * 16 + threadIdx.x];
      db[threadIdx.x] = s2;
    }
  }
}

}  // namespace dfb

using namespace dfb;

extern "C" {

dfb_status dfb_add_rowvec(const float* x, const float* v, float* y, size_t rows, int cols) {
  DFB_INIT();
  DFB_REQUIRE(x && v && y, DFB_ERR_INVALID, "add_rowvec: null pointer");
  DFB_REQUIRE(cols > 0, DFB_ERR_INVALID, "add_rowvec: cols must be positive");
  if (rows == 0) return DFB_OK;
  bool al = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(v) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
  if (cols % 4 == 0 && al)
    launch_k(add_rowvec_kernel<4>, ew_grid(rows * (cols / 4)), kT, 0, compute_stream(), x, v, y, rows, cols);
  else
    launch_k(add_rowvec_kernel<1>, ew_grid(rows * cols), kT, 0, compute_stream(), x, v, y, rows, cols);
  DFB_LAUNCH_CHECK("add_rowvec");
  return DFB_OK;
}

dfb_status dfb_colsum(const float* x, float* out, size_t rows, int cols) {
  DFB_INIT();
  DFB_REQUIRE(x && out, DFB_ERR_INVALID, "colsum: null pointer");
  DFB_REQUIRE(cols > 0, DFB_ERR_INVALID, "colsum: cols must be positive");
  if (rows == 0) return dfb_fill(out, 0.f, cols);
  SumsArgs a{};
  a.x = x;
  a.out0 = out;
  return launch_col_sums<SUMS_COLSUM>("colsum", a, rows, cols, x);
}

static dfb_status bn_stats(const float* x, size_t rows, int C, float eps, float momentum, float* save_mean,
                           float* save_invstd, float* running_mean, float* running_var) {
  SumsArgs a{};
  a.x = x;
  a.out0 = save_mean;
  a.out1 = save_invstd;
  a.running_mean = running_mean;
  a.running_var = running_var;
  a.eps = eps;
  a.momentum = momentum;
  return launch_col_sums<SUMS_STATS>("bn_stats", a, rows, C, x);
}

static dfb_status bn_apply(const float* x, float* y, size_t rows, int C, const float* mean, const float* invstd,
                           const float* gamma, const float* beta, bool relu) {
  bool al = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
  size_t smem = (size_t)3 * C * sizeof(float);
  DFB_REQUIRE(smem <= 48 * 1024, DFB_ERR_INVALID, "batchnorm: too many channels (%d)", C);
  cudaStream_t s = compute_stream();
  if (C % 4 == 0 && al) {
    unsigned grid = ew_grid(rows * (C / 4));
    if (relu) launch_k(bn_apply_kernel<4, true>, grid, kT, smem, s, x, y, rows, C, mean, invstd, gamma, beta);
    else launch_k(bn_apply_kernel<4, false>, grid, kT, smem, s, x, y, rows, C, mean, invstd, gamma, beta);
  } else {
    unsigned grid = ew_grid(rows * C);
    if (relu) launch_k(bn_apply_kernel<1, true>, grid, kT, smem, s, x, y, rows, C, mean, invstd, gamma, beta);
    else launch_k(bn_apply_kernel<1, false>, grid, kT, smem, s, x, y, rows, C, mean, invstd, gamma, beta);
  }
  DFB_LAUNCH_CHECK("bn_apply");
  return DFB_OK;
}

dfb_status dfb_bn_fwd_train(const float* x, const float* gamma, const float* beta, float* y, float* save_mean,
                            float* save_invstd, float* running_mean, float* running_var, float momentum,
                            float eps, size_t rows, int C) {
  DFB_INIT();
  DFB_REQUIRE(x && y && save_mean && save_invstd, DFB_ERR_INVALID, "bn_fwd_train: null pointer");
  DFB_REQUIRE(rows > 0 && C > 0, DFB_ERR_INVALID, "bn_fwd_train: empty input");
  const SmallBnPlan sp = bn_small_plan(true, rows, C, x, y);
  if (const int gpb = sp.gpb) {
    const unsigned grid = (unsigned)(C / 4 / gpb) * sp.cluster;
    cudaStream_t s = compute_stream();
#define DFB_BN_SMALL_FWD(G) launch_k_cluster(bn_small_fwd_kernel<G>, grid, kSmallT, 0, s, dim3(sp.cluster, 1, 1), x, gamma, beta, y, save_mean, \
                                             save_invstd, running_mean, running_var, momentum, eps, (int)rows, C)
    if (gpb == 1) DFB_BN_SMALL_FWD(1);
    else if (gpb == 2) DFB_BN_SMALL_FWD(2);
    else DFB_BN_SMALL_FWD(4);
#undef DFB_BN_SMALL_FWD
    DFB_LAUNCH_CHECK("bn_fwd_train(small)");
    return DFB_OK;
  }
  dfb_status st = bn_stats(x, rows, C, eps, momentum, save_mean, save_invstd, running_mean, running_var);
  if (st != DFB_OK) return st;
  return bn_apply(x, y, rows, C, save_mean, save_invstd, gamma, beta, false);
}

// eval: x_hat = (x - running_mean) / (running_var + eps)**0.5 (batchnorm.py:49-50)
__global__ void bn_eval_prep_kernel(const float* __restrict__ rv, float eps, int C, float* __restrict__ invstd) {
  pdl_sync();
  int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) invstd[c] = 1.0f / sqrtf(rv[c] + eps);
}
dfb_status dfb_bn_fwd_eval(const float* x, const float* gamma, const float* beta, const float* running_mean,
                           const float* running_var, float* y, float eps, size_t rows, int C) {
  DFB_INIT();
  DFB_REQUIRE(x && y && running_mean && running_var, DFB_ERR_INVALID, "bn_fwd_eval: null pointer");
  if (rows == 0) return DFB_OK;
  float* invstd = nullptr;
  dfb_status st = dfb_malloc(C, &invstd);
  if (st != DFB_OK) return st;
  launch_k(bn_eval_prep_kernel, cdiv(C, kT), kT, 0, compute_stream(), running_var, eps, C, invstd);
  DFB_LAUNCH_CHECK("bn_eval_prep");
  st = bn_apply(x, y, rows, C, running_mean, invstd, gamma, beta, false);
  dfb_free(invstd);
  return st;
}

dfb_status dfb_bn_bwd(const float* x, const float* dy, const float* gamma, const float* save_mean,
                      const float* save_invstd, float* dx, float* dgamma, float* dbeta, size_t rows, int C) {
  DFB_INIT();
  DFB_REQUIRE(x && dy && save_mean && save_invstd, DFB_ERR_INVALID, "bn_bwd: null pointer");
  DFB_REQUIRE(rows > 0 && C > 0, DFB_ERR_INVALID, "bn_bwd: empty input");
  const SmallBnPlan sp = bn_small_plan(false, rows, C, x, dy, dx);
  if (const int gpb = sp.gpb) {
    const unsigned grid = (unsigned)(C / 4 / gpb) * sp.cluster;
    cudaStream_t s = compute_stream();
#define DFB_BN_SMALL_BWD(G) launch_k_cluster(bn_small_bwd_kernel<G>, grid, kSmallT, 0, s, dim3(sp.cluster, 1, 1), x, dy, gamma, save_mean, \
                                             save_invstd, dx, dgamma, dbeta, (int)rows, C)
    if (gpb == 1) DFB_BN_SMALL_BWD(1);
    else if (gpb == 2) DFB_BN_SMALL_BWD(2);
    else DFB_BN_SMALL_BWD(4);
#undef DFB_BN_SMALL_BWD
    DFB_LAUNCH_CHECK("bn_bwd(small)");
    return DFB_OK;
  }
  float* scratch = nullptr;
  dfb_status st = dfb_malloc(2 * (size_t)C, &scratch);
  if (st != DFB_OK) return st;
  float* db = dbeta ? dbeta : scratch;
  float* dg = dgamma ? dgamma : scratch + C;
  SumsArgs a{};
  a.x = x;
  a.dy = dy;
  a.mean = save_mean;
  a.invstd = save_invstd;
  a.out0 = db;
  a.out1 = dg;
  st = launch_col_sums<SUMS_BNBWD>("bn_bwd_reduce", a, rows, C, x, dy);
  if (st != DFB_OK) {
    dfb_free(scratch);
    return st;
  }
  cudaStream_t s = compute_stream();
  if (dx) {
    bool al = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(dx)) & 15) == 0;
    size_t sm2 = (size_t)5 * C * sizeof(float);
    if (C % 4 == 0 && al)
      launch_k(bn_bwd_apply_kernel<4>, ew_grid(rows * (C / 4)), kT, sm2, s, x, dy, dx, rows, C, save_mean, save_invstd, gamma, db, dg, StatSrc{nullptr, 0, 0});
    else
      launch_k(bn_bwd_apply_kernel<1>, ew_grid(rows * C), kT, sm2, s, x, dy, dx, rows, C, save_mean, save_invstd, gamma, db, dg, StatSrc{nullptr, 0, 0});
    DFB_LAUNCH_CHECK("bn_bwd_apply");
  }
  dfb_free(scratch);
  return DFB_OK;
}

dfb_status dfb_colstats_mean_var(const float* x, size_t rows, int C, float* mean_var) {
  DFB_INIT();
  DFB_REQUIRE(x && mean_var, DFB_ERR_INVALID, "colstats_mean_var: null pointer");
  DFB_REQUIRE(rows > 0 && C > 0, DFB_ERR_INVALID, "colstats_mean_var: empty input");
  stat_slot_drop(mean_var);
  SumsArgs a{};
  a.x = x;
  a.out0 = mean_var;
  a.out1 = mean_var + C;
  a.raw_var = 1;
  return launch_col_sums<SUMS_STATS>("colstats_mean_var", a, rows, C, x);
}

dfb_status dfb_bn_fwd_apply(const float* x, const float* mean_var, const float* gamma, const float* beta, float* save_mean,
                            float* save_invstd, float* running_mean, float* running_var, float momentum, float eps,
                            const float* x2, const float* mean_var2, const float* gamma2, const float* beta2, float* save_mean2,
                            float* save_invstd2, float* running_mean2, float* running_var2, float momentum2, float eps2,
                            const float* residual, float* y, size_t rows, int C, int relu) {
  DFB_INIT();
  DFB_REQUIRE(x && mean_var && save_mean && save_invstd && y, DFB_ERR_INVALID, "bn_fwd_apply: null pointer");
  DFB_REQUIRE(!x2 || (mean_var2 && save_mean2 && save_invstd2), DFB_ERR_INVALID, "bn_fwd_apply: second BatchNorm incomplete");
  DFB_REQUIRE(rows > 0 && C > 0, DFB_ERR_INVALID, "bn_fwd_apply: empty input");
  const size_t smem = (size_t)(x2 ? 6 : 3) * C * sizeof(float);
  DFB_REQUIRE(smem <= 48 * 1024, DFB_ERR_INVALID, "bn_fwd_apply: too many channels (%d)", C);
  // lazy statistics (dfb_conv2d_fprop_stats_lazy): still in their statistic slots
  int last_a = 0, last_b = 0;
  double* acc_a = stat_slot_take(mean_var, &last_a);
  double* acc_b = x2 ? stat_slot_take(mean_var2, &last_b) : nullptr;
  const float inv_rows = 1.0f / (float)rows;
  BnSide a{x, mean_var, gamma, beta, save_mean, save_invstd, running_mean, running_var, momentum, eps, acc_a, const_cast<float*>(mean_var), inv_rows};
  BnSide b{x2, mean_var2, gamma2, beta2, save_mean2, save_invstd2, running_mean2, running_var2, momentum2, eps2, acc_b, const_cast<float*>(mean_var2), inv_rows};
  const bool vec = C % 4 == 0 && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(x2) | reinterpret_cast<uintptr_t>(residual) |
                                   reinterpret_cast<uintptr_t>(y)) & 15) == 0;
  cudaStream_t s = compute_stream();
  const unsigned grid = vec ? ew_grid(rows * (C / 4)) : ew_grid(rows * C);
  const int sel = (relu ? 4 : 0) | (x2 ? 2 : 0) | (residual ? 1 : 0);
#define DFB_BN_APPLY(R, D, S)                                                                                         \
  do {                                                                                                                \
    if (vec) launch_k(bn_apply_fused_kernel<4, R, D, S>, grid, kT, smem, s, a, b, residual, y, rows, C);              \
    else launch_k(bn_apply_fused_kernel<1, R, D, S>, grid, kT, smem, s, a, b, residual, y, rows, C);                  \
  } while (0)
  switch (sel) {
    case 0: DFB_BN_APPLY(false, false, false); break;
    case 1: DFB_BN_APPLY(false, false, true); break;
    case 2: DFB_BN_APPLY(false, true, false); break;
    case 3: DFB_BN_APPLY(false, true, true); break;
    case 4: DFB_BN_APPLY(true, false, false); break;
    case 5: DFB_BN_APPLY(true, false, true); break;
    case 6: DFB_BN_APPLY(true, true, false); break;
    default: DFB_BN_APPLY(true, true, true); break;
  }
#undef DFB_BN_APPLY
  DFB_LAUNCH_CHECK("bn_fwd_apply");
  return DFB_OK;
}

dfb_status dfb_relu_bwd_bn(const float* x, const float* mean, const float* invstd, const float* gamma, const float* beta,
                           const float* x2, const float* mean2, const float* invstd2, const float* gamma2, const float* beta2,
                           const float* residual, const float* dy, float* dx, size_t rows, int C) {
  DFB_INIT();
  DFB_REQUIRE(x && mean && invstd && dy && dx, DFB_ERR_INVALID, "relu_bwd_bn: null pointer");
  DFB_REQUIRE(!x2 || (mean2 && invstd2), DFB_ERR_INVALID, "relu_bwd_bn: second BatchNorm incomplete");
  if (rows == 0) return DFB_OK;
  const size_t smem = (size_t)(x2 ? 6 : 3) * C * sizeof(float);
  DFB_REQUIRE(smem <= 48 * 1024, DFB_ERR_INVALID, "relu_bwd_bn: too many channels (%d)", C);
  const bool vec = C % 4 == 0 && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(x2) | reinterpret_cast<uintptr_t>(residual) |
                                   reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(dx)) & 15) == 0;
  cudaStream_t s = compute_stream();
  const unsigned grid = vec ? ew_grid(rows * (C / 4)) : ew_grid(rows * C);
#define DFB_RELU_BN(D, S)                                                                                                          \
  do {                                                                                                                             \
    if (vec) launch_k(relu_bwd_bn_kernel<4, D, S>, grid, kT, smem, s, x, mean, invstd, gamma, beta, x2, mean2, invstd2, gamma2, beta2, \
                      residual, dy, dx, rows, C);                                                                                  \
    else launch_k(relu_bwd_bn_kernel<1, D, S>, grid, kT, smem, s, x, mean, invstd, gamma, beta, x2, mean2, invstd2, gamma2, beta2,  \
                  residual, dy, dx, rows, C);                                                                                      \
  } while (0)
  if (x2 && residual) DFB_RELU_BN(true, true);
  else if (x2) DFB_RELU_BN(true, false);
  else if (residual) DFB_RELU_BN(false, true);
  else DFB_RELU_BN(false, false);
#undef DFB_RELU_BN
  DFB_LAUNCH_CHECK("relu_bwd_bn");
  return DFB_OK;
}

// BatchNorm backward in two explicit halves, for callers whose sums come from somewhere else (the dgrad epilogue)
dfb_status dfb_bn_bwd_sums(const float* x, const float* dy, const float* save_mean, const float* save_invstd, float* dbeta,
                           float* dgamma, size_t rows, int C) {
  DFB_INIT();
  DFB_REQUIRE(x && dy && save_mean && save_invstd && dbeta && dgamma, DFB_ERR_INVALID, "bn_bwd_sums: null pointer");
  DFB_REQUIRE(rows > 0 && C > 0, DFB_ERR_INVALID, "bn_bwd_sums: empty input");
  stat_slot_drop(dbeta);
  SumsArgs a{};
  a.x = x;
  a.dy = dy;
  a.mean = save_mean;
  a.invstd = save_invstd;
  a.out0 = dbeta;
  a.out1 = dgamma;
  return launch_col_sums<SUMS_BNBWD>("bn_bwd_sums", a, rows, C, x, dy);
}
dfb_status dfb_maxpool_relu_bn_bwd(const float* x, const float* save_mean, const float* save_invstd, const float* gamma,
                                   const float* beta, const float* pool_y, const float* pool_dy, float* dy, float* sums, int N, int H,
                                   int W, int C, int k) {
  DFB_INIT();
  DFB_REQUIRE(x && save_mean && save_invstd && pool_y && pool_dy && dy && sums, DFB_ERR_INVALID, "maxpool_relu_bn_bwd: null pointer");
  DFB_REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && k >= 1 && H >= k && W >= k, DFB_ERR_INVALID, "maxpool_relu_bn_bwd: bad geometry");
  DFB_REQUIRE((size_t)N * H * W < (1ull << 31), DFB_ERR_INVALID, "maxpool_relu_bn_bwd: more than 2^31 pixels");
  stat_slot_drop(sums);
  SumsArgs a{};
  a.x = x;
  a.dy = pool_dy;
  a.mean = save_mean;
  a.invstd = save_invstd;
  a.gamma = gamma;
  a.beta = beta;
  a.pool_y = pool_y;
  a.dy_out = dy;
  a.out0 = sums;
  a.out1 = sums + C;
  a.H = H; a.W = W; a.OH = (H - k) / k + 1; a.OW = (W - k) / k + 1; a.pool_k = k;
  dfb_status st = DFB_OK;
  if (launch_pool2_bwd(a, N, C, &st)) return st;
  return launch_col_sums<SUMS_POOLBN>("maxpool_relu_bn_bwd", a, (size_t)N * H * W, C, x, dy);
}
dfb_status dfb_bn_bwd_apply(const float* x, const float* dy, const float* gamma, const float* save_mean, const float* save_invstd,
                            float* dbeta, float* dgamma, float* dx, size_t rows, int C) {
  DFB_INIT();
  DFB_REQUIRE(x && dy && save_mean && save_invstd && dbeta && dgamma && dx, DFB_ERR_INVALID, "bn_bwd_apply: null pointer");
  DFB_REQUIRE(rows > 0 && C > 0, DFB_ERR_INVALID, "bn_bwd_apply: empty input");
  const bool al = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(dy) | reinterpret_cast<uintptr_t>(dx)) & 15) == 0;
  const size_t sm2 = (size_t)5 * C * sizeof(float);
  DFB_REQUIRE(sm2 <= 48 * 1024, DFB_ERR_INVALID, "bn_bwd_apply: too many channels (%d)", C);
  cudaStream_t s = compute_stream();
  // lazy sums (dfb_conv2d_dgrad_fused_lazy): still in their statistic slot, keyed by the base of the sums buffer = dbeta
  StatSrc src{nullptr, 0, 0};
  int last = 0;
  if (dgamma > dbeta && (size_t)(dgamma - dbeta) % (size_t)C == 0 && (dgamma - dbeta) / C <= 2) {
    src.acc = stat_slot_take(dbeta, &last);
    src.row = (int)((dgamma - dbeta) / C);
    src.clear = last;
  }
  if (C % 4 == 0 && al)
    launch_k(bn_bwd_apply_kernel<4>, ew_grid(rows * (C / 4)), kT, sm2, s, x, dy, dx, rows, C, save_mean, save_invstd, gamma, dbeta, dgamma, src);
  else
    launch_k(bn_bwd_apply_kernel<1>, ew_grid(rows * C), kT, sm2, s, x, dy, dx, rows, C, save_mean, save_invstd, gamma, dbeta, dgamma, src);
  DFB_LAUNCH_CHECK("bn_bwd_apply");
  return DFB_OK;
}

dfb_status dfb_relu_fwd(const float* x, float* y, size_t n) { return dfb_scalar_maximum(x, 0.0f, y, n); }

dfb_status dfb_relu_bwd(const float* x, const float* dy, float* dx, size_t n) {
  DFB_INIT();
  DFB_REQUIRE(x && dy && dx, DFB_ERR_INVALID, "relu_bwd: null pointer");
  if (n == 0) return DFB_OK;
  launch_k(relu_bwd_kernel, ew_grid(n / 4 + 1), kT, 0, compute_stream(), x, dy, dx, n);
  DFB_LAUNCH_CHECK("relu_bwd");
  return DFB_OK;
}

static dfb_status pool_geom(const char* name, int N, int H, int W, int C, int k, int* OH, int* OW) {
  DFB_REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && k > 0 && H >= k && W >= k, DFB_ERR_INVALID,
              "%s: bad geometry N=%d H=%d W=%d C=%d k=%d", name, N, H, W, C, k);
  *OH = (H - k) / k + 1;
  *OW = (W - k) / k + 1;
  return DFB_OK;
}
#define POOL_DISPATCH(KERNEL, items_scalar, ...)                                               \
  do {                                                                                         \
    if (vec) launch_k(KERNEL<4>, ew_grid((items_scalar) / 4), kT, 0, compute_stream(), __VA_ARGS__); \
    else launch_k(KERNEL<1>, ew_grid(items_scalar), kT, 0, compute_stream(), __VA_ARGS__);           \
  } while (0)

static bool all_aligned(const void* a, const void* b = nullptr, const void* c = nullptr, const void* d = nullptr) {
  return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c) |
           reinterpret_cast<uintptr_t>(d)) & 15) == 0;
}

dfb_status dfb_maxpool2d_fwd(const float* x, float* y, int32_t* idx, int N, int H, int W, int C, int k) {
  DFB_INIT();
  DFB_REQUIRE(x && y, DFB_ERR_INVALID, "maxpool2d_fwd: null pointer");
  int OH, OW;
  dfb_status st = pool_geom("maxpool2d_fwd", N, H, W, C, k, &OH, &OW);
  if (st != DFB_OK) return st;
  bool vec = C % 4 == 0 && all_aligned(x, y, idx);
  POOL_DISPATCH(maxpool_fwd_kernel, (size_t)N * OH * OW * C, x, y, idx, N, H, W, C, k, OH, OW);
  DFB_LAUNCH_CHECK("maxpool2d_fwd");
  return DFB_OK;
}
dfb_status dfb_maxpool2d_bwd(const float* x, const float* y, const float* dy, float* dx, int N, int H, int W,
                             int C, int k) {
  DFB_INIT();
  DFB_REQUIRE(x && y && dy && dx, DFB_ERR_INVALID, "maxpool2d_bwd: null pointer");
  int OH, OW;
  dfb_status st = pool_geom("maxpool2d_bwd", N, H, W, C, k, &OH, &OW);
  if (st != DFB_OK) return st;
  bool vec = C % 4 == 0 && all_aligned(x, y, dy, dx);
  size_t items = (size_t)N * H * W * C;
  if (vec) launch_k(maxpool_bwd_kernel<4, 0>, ew_grid(items / 4), kT, 0, compute_stream(), x, y, nullptr, dy, dx, N, H, W, C, k, OH, OW);
  else launch_k(maxpool_bwd_kernel<1, 0>, ew_grid(items), kT, 0, compute_stream(), x, y, nullptr, dy, dx, N, H, W, C, k, OH, OW);
  DFB_LAUNCH_CHECK("maxpool2d_bwd");
  return DFB_OK;
}
dfb_status dfb_maxpool2d_bwd_idx(const int32_t* idx, const float* dy, float* dx, int N, int H, int W, int C, int k) {
  DFB_INIT();
  DFB_REQUIRE(idx && dy && dx, DFB_ERR_INVALID, "maxpool2d_bwd_idx: null pointer");
  int OH, OW;
  dfb_status st = pool_geom("maxpool2d_bwd_idx", N, H, W, C, k, &OH, &OW);
  if (st != DFB_OK) return st;
  bool vec = C % 4 == 0 && all_aligned(idx, dy, dx);
  size_t items = (size_t)N * H * W * C;
  if (vec) launch_k(maxpool_bwd_kernel<4, 1>, ew_grid(items / 4), kT, 0, compute_stream(), nullptr, nullptr, idx, dy, dx, N, H, W, C, k, OH, OW);
  else launch_k(maxpool_bwd_kernel<1, 1>, ew_grid(items), kT, 0, compute_stream(), nullptr, nullptr, idx, dy, dx, N, H, W, C, k, OH, OW);
  DFB_LAUNCH_CHECK("maxpool2d_bwd_idx");
  return DFB_OK;
}
dfb_status dfb_avgpool2d_fwd(const float* x, float* y, int N, int H, int W, int C, int k) {
  DFB_INIT();
  DFB_REQUIRE(x && y, DFB_ERR_INVALID, "avgpool2d_fwd: null pointer");
  int OH, OW;
  dfb_status st = pool_geom("avgpool2d_fwd", N, H, W, C, k, &OH, &OW);
  if (st != DFB_OK) return st;
  bool vec = C % 4 == 0 && all_aligned(x, y);
  POOL_DISPATCH(avgpool_fwd_kernel, (size_t)N * OH * OW * C, x, y, N, H, W, C, k, OH, OW);
  DFB_LAUNCH_CHECK("avgpool2d_fwd");
  return DFB_OK;
}
dfb_status dfb_avgpool2d_bwd(const float* dy, float* dx, int N, int H, int W, int C, int k) {
  DFB_INIT();
  DFB_REQUIRE(dy && dx, DFB_ERR_INVALID, "avgpool2d_bwd: null pointer");
  int OH, OW;
  dfb_status st = pool_geom("avgpool2d_bwd", N, H, W, C, k, &OH, &OW);
  if (st != DFB_OK) return st;
  bool vec = C % 4 == 0 && all_aligned(dy, dx);
  POOL_DISPATCH(avgpool_bwd_kernel, (size_t)N * H * W * C, dy, dx, N, H, W, C, k, OH, OW);
  DFB_LAUNCH_CHECK("avgpool2d_bwd");
  return DFB_OK;
}

static dfb_status upsample_geom(const char* name, int N, int H, int W, int C, int scale, int mode) {
  DFB_REQUIRE(N > 0 && H > 0 && W > 0 && C > 0 && scale >= 1 && scale <= 8, DFB_ERR_INVALID,
              "%s: bad geometry N=%d H=%d W=%d C=%d scale=%d (1 <= scale <= 8)", name, N, H, W, C, scale);
  DFB_REQUIRE((long long)H * scale < (1ll << 31) && (long long)W * scale < (1ll << 31), DFB_ERR_INVALID, "%s: output too large",
              name);
  DFB_REQUIRE(mode == DFB_UPSAMPLE_NEAREST || mode == DFB_UPSAMPLE_BILINEAR, DFB_ERR_INVALID, "%s: bad mode %d", name, mode);
  return DFB_OK;
}
dfb_status dfb_upsample2d_fwd(const float* x, float* y, int N, int H, int W, int C, int scale, int mode) {
  DFB_INIT();
  DFB_REQUIRE(x && y, DFB_ERR_INVALID, "upsample2d_fwd: null pointer");
  dfb_status st = upsample_geom("upsample2d_fwd", N, H, W, C, scale, mode);
  if (st != DFB_OK) return st;
  bool vec = C % 4 == 0 && all_aligned(x, y);
  size_t items = (size_t)N * H * scale * W * scale * C;
  if (mode == DFB_UPSAMPLE_NEAREST) POOL_DISPATCH(upsample_nearest_fwd_kernel, items, x, y, N, H, W, C, scale);
  else POOL_DISPATCH(upsample_bilinear_fwd_kernel, items, x, y, N, H, W, C, scale);
  DFB_LAUNCH_CHECK("upsample2d_fwd");
  return DFB_OK;
}
dfb_status dfb_upsample2d_bwd(const float* dy, float* dx, int N, int H, int W, int C, int scale, int mode) {
  DFB_INIT();
  DFB_REQUIRE(dy && dx, DFB_ERR_INVALID, "upsample2d_bwd: null pointer");
  dfb_status st = upsample_geom("upsample2d_bwd", N, H, W, C, scale, mode);
  if (st != DFB_OK) return st;
  bool vec = C % 4 == 0 && all_aligned(dy, dx);
  size_t items = (size_t)N * H * W * C;
  if (mode == DFB_UPSAMPLE_NEAREST) POOL_DISPATCH(upsample_nearest_bwd_kernel, items, dy, dx, N, H, W, C, scale);
  else POOL_DISPATCH(upsample_bilinear_bwd_kernel, items, dy, dx, N, H, W, C, scale);
  DFB_LAUNCH_CHECK("upsample2d_bwd");
  return DFB_OK;
}

// One launch for the slices whose pointer is not null (the backward skips inputs that need no gradient); y is the
// concatenated matrix, read by the backward and written by the forward.
static dfb_status concat_channels(const char* name, float* const* parts, const int* widths, int count, float* y,
                                  long long rows, bool bwd) {
  DFB_REQUIRE(count >= 1 && count <= DFB_CONCAT_MAX_SOURCES, DFB_ERR_INVALID, "%s: %d sources (1 to %d)", name, count,
              DFB_CONCAT_MAX_SOURCES);
  DFB_REQUIRE(parts && widths && y, DFB_ERR_INVALID, "%s: null pointer", name);
  DFB_REQUIRE(rows > 0, DFB_ERR_INVALID, "%s: rows must be positive, got %lld", name, rows);
  ConcatSlices t = {};
  int n = 0, widest = 0;
  long long C = 0;
  bool vec = all_aligned(y);
  for (int i = 0; i < count; ++i) {
    DFB_REQUIRE(widths[i] > 0, DFB_ERR_INVALID, "%s: width %d of source %d must be positive", name, widths[i], i);
    vec = vec && widths[i] % 4 == 0 && all_aligned(parts[i]);
    if (parts[i]) {
      t.p[n] = parts[i];
      t.off[n] = (int)C;
      t.width[n] = widths[i];
      widest = std::max(widest, widths[i]);
      ++n;
    }
    C += widths[i];
    DFB_REQUIRE(C < (1ll << 31), DFB_ERR_INVALID, "%s: %lld channels or more (limit 2^31 - 1)", name, C);
  }
  if (n == 0) return DFB_OK;
  const int V = vec ? 4 : 1;
  const unsigned per_slice = std::max(1u, (unsigned)(sm_count() * 8 / n));
  const size_t vectors = ((size_t)rows * (widest / V) + kConcatUnroll - 1) / kConcatUnroll;
  const dim3 grid(std::min(bw_grid(vectors, kT), per_slice), n);
  if (bwd) {
    if (vec) launch_k(concat_channels_kernel<4, true>, grid, kT, 0, compute_stream(), t, y, (int)C, rows);
    else launch_k(concat_channels_kernel<1, true>, grid, kT, 0, compute_stream(), t, y, (int)C, rows);
  } else {
    if (vec) launch_k(concat_channels_kernel<4, false>, grid, kT, 0, compute_stream(), t, y, (int)C, rows);
    else launch_k(concat_channels_kernel<1, false>, grid, kT, 0, compute_stream(), t, y, (int)C, rows);
  }
  DFB_LAUNCH_CHECK(name);
  return DFB_OK;
}
dfb_status dfb_concat_channels_fwd(const float* const* srcs, const int* widths, int count, float* y, long long rows) {
  DFB_INIT();
  for (int i = 0; srcs && i < count && i < DFB_CONCAT_MAX_SOURCES; ++i)
    DFB_REQUIRE(srcs[i], DFB_ERR_INVALID, "concat_channels_fwd: source %d is null", i);
  return concat_channels("concat_channels_fwd", const_cast<float* const*>(srcs), widths, count, y, rows, false);
}
dfb_status dfb_concat_channels_bwd(const float* dy, float* const* dsrcs, const int* widths, int count, long long rows) {
  DFB_INIT();
  return concat_channels("concat_channels_bwd", dsrcs, widths, count, const_cast<float*>(dy), rows, true);
}

dfb_status dfb_linear_small_fwd(const float* x, const float* w, const float* bias, float* y, int M, int K, int N) {
  DFB_INIT();
  DFB_REQUIRE(x && w && y, DFB_ERR_INVALID, "linear_small_fwd: null pointer");
  DFB_REQUIRE(M > 0 && K > 0 && N > 0 && N <= kLinN, DFB_ERR_INVALID, "linear_small_fwd: M = %d, K = %d, N = %d (1 <= N <= %d)", M, K, N, kLinN);
  launch_k(linear_small_fwd_kernel, (unsigned)((M + 7) / 8), 256, 0, compute_stream(), x, w, bias, y, M, K, N);
  DFB_LAUNCH_CHECK("linear_small_fwd");
  return DFB_OK;
}
dfb_status dfb_linear_small_bwd(const float* x, const float* w, const float* dy, float* dx, float* dw, float* db, int M, int K, int N) {
  DFB_INIT();
  DFB_REQUIRE(dy != nullptr, DFB_ERR_INVALID, "linear_small_bwd: null gradient");
  DFB_REQUIRE(M > 0 && K > 0 && N > 0 && N <= kLinN, DFB_ERR_INVALID, "linear_small_bwd: M = %d, K = %d, N = %d (1 <= N <= %d)", M, K, N, kLinN);
  DFB_REQUIRE((!dx || w) && (!dw || x), DFB_ERR_INVALID, "linear_small_bwd: dx needs w, dw needs x");
  DFB_REQUIRE((size_t)M * K < ((size_t)1 << 38), DFB_ERR_INVALID, "linear_small_bwd: input too large");
  const int dx_blocks = dx ? (int)(((size_t)M * K + kLinT - 1) / kLinT) : 0, dw_blocks = dw ? (K + 31) / 32 : 0, db_blocks = db ? 1 : 0;
  if (dx_blocks + dw_blocks + db_blocks == 0) return DFB_OK;
  launch_k(linear_small_bwd_kernel, (unsigned)(dx_blocks + dw_blocks + db_blocks), kLinT, 0, compute_stream(), x, w, dy, dx, dw, db, M, K,
           N, dx_blocks, dw_blocks);
  DFB_LAUNCH_CHECK("linear_small_bwd");
  return DFB_OK;
}

dfb_status dfb_softmax_ce_fwd(const float* logits, const float* target, float* loss, size_t rows, int cols,
                              float scale) {
  DFB_INIT();
  DFB_REQUIRE(logits && target && loss, DFB_ERR_INVALID, "softmax_ce_fwd: null pointer");
  DFB_REQUIRE(cols > 0, DFB_ERR_INVALID, "softmax_ce_fwd: cols must be positive");
  launch_k(softmax_ce_fwd_kernel, 1, kCeThreads, 0, compute_stream(), logits, target, loss, rows, cols, scale);
  DFB_LAUNCH_CHECK("softmax_ce_fwd");
  return DFB_OK;
}
dfb_status dfb_softmax_ce_bwd(const float* logits, const float* target, const float* upstream, float* dlogits,
                              size_t rows, int cols, float scale) {
  DFB_INIT();
  DFB_REQUIRE(logits && target && dlogits, DFB_ERR_INVALID, "softmax_ce_bwd: null pointer");
  if (rows == 0) return DFB_OK;
  launch_k(softmax_ce_bwd_kernel, bw_grid(rows, kT), kT, 0, compute_stream(), logits, target, upstream, dlogits, rows, cols, scale);
  DFB_LAUNCH_CHECK("softmax_ce_bwd");
  return DFB_OK;
}

}  // extern "C"
