// Joint two-phase metering of the ISP (reference: camera_isp.py:102-175) as two deterministic
// reductions: per-thread sequential accumulate -> warp shuffle tree -> block tree -> per-block
// partial in the workspace -> the last block to finish (ticket counter) folds the partials in fixed
// order and applies the moving-average blend on the device.  No host synchronisation, and the
// result is bit-reproducible run to run (the reference's float atomics are not).
//
//   phase 1: (mn, mx) over all sampled values; b = lerp(alpha, (mn,mx), prev.bounds)      :149-157
//   phase 2: per sample  scaled = (rgb - b.min) / (b.max - b.min + 1e-6)                  :119
//            gray = rgb_gray(scaled); lg = log(max(gray, 1e-4)); min/max lg, sums         :120-128
//            normalise by n; metrics = lerp(alpha, [b, lmin, lmax, lmean, mean, rgb], prev) :131-134, :164-166
// `alpha` is the weight of the PREVIOUS value: lerp(t,a,b) = a + t*(b-a) (util.py:82-84).
#pragma once
#include "common.cuh"
#include "exchange.cuh"
#include <stdlib.h>

namespace isp {

// Sampler concept:  __device__ void sample(long long idx, float (&rgb)[3]) const;   idx in [0, n)
//                   rgb as stored by the ISP (already rounded through the ISP dtype).

// ---------------------------------------------------------------- sample iteration
// for_each_sample(smp, n, f): calls f(idx, rgb) for this thread's share of the n samples.  Samplers that define
// kRowStructured iterate themselves (Packed12FastSampler: a warp walks sample rows, no index division per
// sample); the others take a flat grid-stride loop unrolled by 4 so that several samples' loads are in flight.
constexpr int kMeterUnroll = 4;

template <class Sampler, class = void> struct is_row_structured { static constexpr bool value = false; };
template <class Sampler> struct is_row_structured<Sampler, std::enable_if_t<Sampler::kRowStructured>> { static constexpr bool value = true; };

template <class Sampler, class F>
__device__ __forceinline__ void for_each_sample(const Sampler& smp, long long n, F&& f) {
  if constexpr (is_row_structured<Sampler>::value) {
    smp.for_each(n, f);
  } else {
    // n < 2^31 / 3 always (<= 64 frames of <= 2^24 samples): 32-bit index arithmetic
    const unsigned T = gridDim.x * blockDim.x, n32 = (unsigned)n;
    for (unsigned i0 = blockIdx.x * blockDim.x + threadIdx.x; i0 < n32; i0 += T * kMeterUnroll) {
      float rgb[kMeterUnroll][3];
#pragma unroll
      for (int u = 0; u < kMeterUnroll; ++u) smp.sample((long long)min(i0 + u * T, n32 - 1), rgb[u]);   // clamped: branch-free loads
#pragma unroll
      for (int u = 0; u < kMeterUnroll; ++u)
        if (i0 + u * T < n32) f((long long)(i0 + u * T), rgb[u]);
    }
  }
}

template <int NV>
__device__ __forceinline__ void block_fold(float (&v)[NV], const int (&op)[NV], float* smem /* [8][NV] */) {
  // op: 0 = min, 1 = max, 2 = sum
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NV; ++k) v[k] = op[k] == 0 ? warp_min(v[k]) : (op[k] == 1 ? warp_max(v[k]) : warp_sum(v[k]));
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < NV; ++k) smem[warp * NV + k] = v[k];
  }
  __syncthreads();
  if (warp == 0) {
    const int nw = blockDim.x >> 5;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      float x = lane < nw ? smem[lane * NV + k] : (op[k] == 0 ? INFINITY : (op[k] == 1 ? -INFINITY : 0.f));
      v[k] = op[k] == 0 ? warp_min(x) : (op[k] == 1 ? warp_max(x) : warp_sum(x));
    }
  }
  __syncthreads();
}

// Returns true in ALL threads of the last block to arrive; partials of every block are then visible.
__device__ __forceinline__ bool last_block_ticket(unsigned int* counter) {
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(counter, 1u);
    s_last = (t == gridDim.x - 1);
    if (s_last) *counter = 0u;   // leave the workspace zeroed for the next launch
  }
  __syncthreads();
  if (s_last) __threadfence();
  return s_last;
}

template <class Sampler>
__global__ void __launch_bounds__(256) meter_phase1_kernel(const Sampler smp, long long n, float alpha,
                                                           const float* __restrict__ prev, Workspace* ws,
                                                           float* __restrict__ cache /* n*3 floats or null */,
                                                           float* __restrict__ rec_out = nullptr /* shared exposure: raw {min,max} */) {
  __shared__ float smem[8 * 2];
  float v[2] = {INFINITY, -INFINITY};
  for_each_sample(smp, n, [&](long long i, const float (&rgb)[3]) {
    if (cache) { const unsigned o = 3u * (unsigned)i; cache[o] = rgb[0]; cache[o + 1] = rgb[1]; cache[o + 2] = rgb[2]; }
    v[0] = fminf(v[0], fminf(rgb[0], fminf(rgb[1], rgb[2])));
    v[1] = fmaxf(v[1], fmaxf(rgb[0], fmaxf(rgb[1], rgb[2])));
  });
  const int op[2] = {0, 1};
  block_fold<2>(v, op, smem);
  if (threadIdx.x == 0) {
    ws->partials[blockIdx.x * kPartialStride + 0] = v[0];
    ws->partials[blockIdx.x * kPartialStride + 1] = v[1];
  }
  if (last_block_ticket(&ws->counter[0])) {
    float f[2] = {INFINITY, -INFINITY};
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
      f[0] = fminf(f[0], __ldcg(&ws->partials[b * kPartialStride + 0]));
      f[1] = fmaxf(f[1], __ldcg(&ws->partials[b * kPartialStride + 1]));
    }
    block_fold<2>(f, op, smem);
    if (threadIdx.x == 0) {
      if (rec_out) {                       // multi-GPU: the ranks' records are folded after the exchange
        rec_out[0] = f[0]; rec_out[1] = f[1];
      } else {
        // b = lerp(alpha, new, prev) = new + alpha * (prev - new)          camera_isp.py:156
        ws->bounds[0] = __fadd_rn(f[0], __fmul_rn(alpha, __fsub_rn(prev[0], f[0])));
        ws->bounds[1] = __fadd_rn(f[1], __fmul_rn(alpha, __fsub_rn(prev[1], f[1])));
      }
    }
  }
}

// camera_isp.py:119-128 for one sample.  The reference divides by (max - min + 1e-6); here the reciprocal is
// taken once (IEEE) and multiplied, and the logarithm is the hardware lg2 -- both far inside what the
// reference's own unordered float atomics and fast-math build leave defined (SURVEY H7, ~1e-6 relative).
__device__ __forceinline__ void meter_accum(const float (&rgb)[3], float bmin, float inv_den, float (&v)[7]) {
  const float r = __fmul_rn(__fsub_rn(rgb[0], bmin), inv_den);
  const float g = __fmul_rn(__fsub_rn(rgb[1], bmin), inv_den);
  const float b = __fmul_rn(__fsub_rn(rgb[2], bmin), inv_den);
  const float gray = rgb_gray(r, g, b);
  const float lg = __logf(fmaxf(gray, 1e-4f));
  v[0] = fminf(v[0], lg);
  v[1] = fmaxf(v[1], lg);
  v[2] += lg; v[3] += gray; v[4] += r; v[5] += g; v[6] += b;
}

template <class Sampler>
__global__ void __launch_bounds__(256) meter_phase2_kernel(const Sampler smp, long long n, float alpha,
                                                           const float* prev, float* metrics /* out; may alias prev */, Workspace* ws,
                                                           float* __restrict__ rec_out = nullptr /* shared exposure: raw record 2 */) {
  __shared__ float smem[8 * 7];
  const float bmin = __ldcg(&ws->bounds[0]), bmax = __ldcg(&ws->bounds[1]);
  const float inv_den = __fdiv_rn(1.0f, __fadd_rn(__fsub_rn(bmax, bmin), 1e-6f));
  float v[7] = {INFINITY, -INFINITY, 0.f, 0.f, 0.f, 0.f, 0.f};
  for_each_sample(smp, n, [&](long long, const float (&rgb)[3]) { meter_accum(rgb, bmin, inv_den, v); });
  const int op[7] = {0, 1, 2, 2, 2, 2, 2};
  block_fold<7>(v, op, smem);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < 7; ++k) ws->partials[blockIdx.x * kPartialStride + k] = v[k];
  }
  if (last_block_ticket(&ws->counter[0])) {
    float f[7] = {INFINITY, -INFINITY, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
      f[0] = fminf(f[0], __ldcg(&ws->partials[b * kPartialStride + 0]));
      f[1] = fmaxf(f[1], __ldcg(&ws->partials[b * kPartialStride + 1]));
#pragma unroll
      for (int k = 2; k < 7; ++k) f[k] += __ldcg(&ws->partials[b * kPartialStride + k]);
    }
    block_fold<7>(f, op, smem);
    if (threadIdx.x == 0 && rec_out) {
#pragma unroll
      for (int k = 0; k < 7; ++k) rec_out[k] = f[k];
      rec_out[7] = (float)n;
    } else if (threadIdx.x == 0) {
      const float fn = (float)n;                                          // camera_isp.py:131-134
      const float stats[9] = {bmin, bmax, f[0], f[1], __fdiv_rn(f[2], fn), __fdiv_rn(f[3], fn),
                              __fdiv_rn(f[4], fn), __fdiv_rn(f[5], fn), __fdiv_rn(f[6], fn)};
#pragma unroll
      for (int k = 0; k < 9; ++k) {                                       // camera_isp.py:165-166
        const float p = prev[k];
        metrics[k] = __fadd_rn(stats[k], __fmul_rn(alpha, __fsub_rn(p, stats[k])));
      }
    }
  }
}

// ---------------------------------------------------------------- multi-GPU shared exposure (SURVEY 8e)
// gathered1: [world][2] = every rank's {min, max}; gathered2: [world][8] = {log_min, log_max, sum_log, sum_gray,
// sum_r, sum_g, sum_b, n}.  Folded in rank order -> every rank computes bit-identical metrics.
__device__ __forceinline__ void fold_bounds(const float* __restrict__ g1, int world, float alpha, const float* __restrict__ prev,
                                            float& bmin, float& bmax) {
  float mn = INFINITY, mx = -INFINITY;
  for (int r = 0; r < world; ++r) { mn = fminf(mn, g1[2 * r]); mx = fmaxf(mx, g1[2 * r + 1]); }
  bmin = __fadd_rn(mn, __fmul_rn(alpha, __fsub_rn(prev[0], mn)));          // camera_isp.py:156
  bmax = __fadd_rn(mx, __fmul_rn(alpha, __fsub_rn(prev[1], mx)));
}

// The fold kernels of the shared exposure and phase 2 over the cached samples, defined in fused_api.cu so that each is compiled
// once.
int launch_meter_fold_bounds(const float* g1, int world, float alpha, const float* prev, Workspace* ws, cudaStream_t s);
int launch_meter_finalize(const float* g1, const float* g2, int world, float alpha, const float* prev, float* metrics, cudaStream_t s);
struct CachedSampler;
int launch_meter_phase2_cached(int grid, const CachedSampler& smp, long long n, float alpha, const float* prev, float* metrics, Workspace* ws,
                               cudaStream_t s, float* rec_out);

// ---------------------------------------------------------------- shared exposure with the exchange INSIDE the kernels
// Same two reductions, but the last block to finish a phase also runs that phase's cross-rank exchange (one warp:
// post the record into every rank's mailbox over NVLink, spin until every rank's record has arrived; exchange.cuh)
// and the fold that follows it.  A joint metering update is then 2 launches instead of 8 (phase 1, post, wait, bounds
// fold, phase 2, post, wait, finalize), with no launch gap between a reduction and its exchange.
template <class Sampler>
__global__ void __launch_bounds__(256) meter_phase1x_kernel(const Sampler smp, long long n, float alpha, const float* __restrict__ prev,
                                                            Workspace* ws, float* __restrict__ cache, const PeerXchg xc) {
  __shared__ float smem[8 * 2];
  __shared__ float s_rec[2];
  __shared__ float s_g[kXchgRanks * 2];
  float v[2] = {INFINITY, -INFINITY};
  for_each_sample(smp, n, [&](long long i, const float (&rgb)[3]) {
    if (cache) { const unsigned o = 3u * (unsigned)i; cache[o] = rgb[0]; cache[o + 1] = rgb[1]; cache[o + 2] = rgb[2]; }
    v[0] = fminf(v[0], fminf(rgb[0], fminf(rgb[1], rgb[2])));
    v[1] = fmaxf(v[1], fmaxf(rgb[0], fmaxf(rgb[1], rgb[2])));
  });
  const int op[2] = {0, 1};
  block_fold<2>(v, op, smem);
  if (threadIdx.x == 0) {
    ws->partials[blockIdx.x * kPartialStride + 0] = v[0];
    ws->partials[blockIdx.x * kPartialStride + 1] = v[1];
  }
  if (last_block_ticket(&ws->counter[0])) {
    float f[2] = {INFINITY, -INFINITY};
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
      f[0] = fminf(f[0], __ldcg(&ws->partials[b * kPartialStride + 0]));
      f[1] = fmaxf(f[1], __ldcg(&ws->partials[b * kPartialStride + 1]));
    }
    block_fold<2>(f, op, smem);
    if (threadIdx.x == 0) { s_rec[0] = f[0]; s_rec[1] = f[1]; }
    __syncthreads();
    if (threadIdx.x < 32) {
      const uint32_t seq = mailbox_post_warp(xc.p, xc.world, xc.rank, 0, s_rec, B200ISP_REC1);
      mailbox_wait_warp(xc.p[xc.rank], xc.world, 0, seq, s_g, B200ISP_REC1);
      if (threadIdx.x == 0) fold_bounds(s_g, xc.world, alpha, prev, ws->bounds[0], ws->bounds[1]);     // identical on every rank
    }
  }
}

template <class Sampler>
__global__ void __launch_bounds__(256) meter_phase2x_kernel(const Sampler smp, long long n, float alpha, const float* prev,
                                                            float* metrics /* out; may alias prev */, Workspace* ws, const PeerXchg xc) {
  __shared__ float smem[8 * 7];
  __shared__ float s_rec[8];
  __shared__ float s_g[kXchgRanks * 8];
  const float bmin = __ldcg(&ws->bounds[0]), bmax = __ldcg(&ws->bounds[1]);
  const float inv_den = __fdiv_rn(1.0f, __fadd_rn(__fsub_rn(bmax, bmin), 1e-6f));
  float v[7] = {INFINITY, -INFINITY, 0.f, 0.f, 0.f, 0.f, 0.f};
  for_each_sample(smp, n, [&](long long, const float (&rgb)[3]) { meter_accum(rgb, bmin, inv_den, v); });
  const int op[7] = {0, 1, 2, 2, 2, 2, 2};
  block_fold<7>(v, op, smem);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < 7; ++k) ws->partials[blockIdx.x * kPartialStride + k] = v[k];
  }
  if (last_block_ticket(&ws->counter[0])) {
    float f[7] = {INFINITY, -INFINITY, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
      f[0] = fminf(f[0], __ldcg(&ws->partials[b * kPartialStride + 0]));
      f[1] = fmaxf(f[1], __ldcg(&ws->partials[b * kPartialStride + 1]));
#pragma unroll
      for (int k = 2; k < 7; ++k) f[k] += __ldcg(&ws->partials[b * kPartialStride + k]);
    }
    block_fold<7>(f, op, smem);
    if (threadIdx.x == 0) {
#pragma unroll
      for (int k = 0; k < 7; ++k) s_rec[k] = f[k];
      s_rec[7] = (float)n;
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      const uint32_t seq = mailbox_post_warp(xc.p, xc.world, xc.rank, 1, s_rec, B200ISP_REC2);
      mailbox_wait_warp(xc.p[xc.rank], xc.world, 1, seq, s_g, B200ISP_REC2);
      if (threadIdx.x == 0) {                                             // meter_finalize_kernel with the blended bounds at hand
        float g[8] = {INFINITY, -INFINITY, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int r = 0; r < xc.world; ++r) {
          g[0] = fminf(g[0], s_g[8 * r]);
          g[1] = fmaxf(g[1], s_g[8 * r + 1]);
          for (int k = 2; k < 8; ++k) g[k] += s_g[8 * r + k];
        }
        const float fn = g[7];                                            // camera_isp.py:131-134 with n = all ranks' samples
        const float stats[9] = {bmin, bmax, g[0], g[1], __fdiv_rn(g[2], fn), __fdiv_rn(g[3], fn),
                                __fdiv_rn(g[4], fn), __fdiv_rn(g[5], fn), __fdiv_rn(g[6], fn)};
        for (int k = 0; k < 9; ++k) {                                     // camera_isp.py:165-166
          const float p = prev[k];
          metrics[k] = __fadd_rn(stats[k], __fmul_rn(alpha, __fsub_rn(p, stats[k])));
        }
      }
    }
  }
}

// samples cached by phase 1 (3 floats each), read back coalesced by phase 2
struct CachedSampler {
  const float* cache;
  __device__ __forceinline__ void sample(long long idx, float (&rgb)[3]) const {
    const unsigned o = 3u * (unsigned)idx;
    rgb[0] = __ldcg(cache + o); rgb[1] = __ldcg(cache + o + 1); rgb[2] = __ldcg(cache + o + 2);
  }
};

// ---------------------------------------------------------------- both phases in ONE cooperative launch
// The grid is launched with cudaLaunchCooperativeKernel (all CTAs co-resident), so the dependency between the
// phases -- every sample's min / max before any sample's log-luminance -- is a grid barrier instead of a
// kernel boundary: one launch, one tail, and phase 2 re-reads the samples phase 1 just wrote while they are
// still in L2 (22 MB at cfg2).  Sample loops are unrolled by 4 so that the nine loads of several samples are
// in flight together.  Phase-2 partials use the upper half of the partial table: a fast CTA may already be
// writing them while a slow one still folds the phase-1 entries.
__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void grid_barrier(unsigned int* counter) {     // cooperative launch only
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(counter, 1u);
    while (ld_acquire_gpu(counter) < gridDim.x) __nanosleep(32);
    __threadfence();
  }
  __syncthreads();
}

template <class Sampler>
__global__ void __launch_bounds__(256) meter_fused_kernel(const Sampler smp, long long n, float alpha, const float* prev,
                                                          float* metrics /* out; may alias prev */, Workspace* ws,
                                                          float* __restrict__ cache /* n*3 floats or null */) {
  __shared__ float smem[8 * 7];
  __shared__ float s_bounds[2];
  float* part2 = ws->partials + (kMaxPartialBlocks / 2) * kPartialStride;

  // ---- phase 1: min / max of every sampled value
  float v2[2] = {INFINITY, -INFINITY};
  for_each_sample(smp, n, [&](long long i, const float (&rgb)[3]) {
    if (cache) { const unsigned o = 3u * (unsigned)i; cache[o] = rgb[0]; cache[o + 1] = rgb[1]; cache[o + 2] = rgb[2]; }
    v2[0] = fminf(v2[0], fminf(rgb[0], fminf(rgb[1], rgb[2])));
    v2[1] = fmaxf(v2[1], fmaxf(rgb[0], fmaxf(rgb[1], rgb[2])));
  });
  const int op2[2] = {0, 1};
  block_fold<2>(v2, op2, smem);
  if (threadIdx.x == 0) {
    ws->partials[blockIdx.x * kPartialStride + 0] = v2[0];
    ws->partials[blockIdx.x * kPartialStride + 1] = v2[1];
  }
  grid_barrier(&ws->counter[1]);

  // ---- every CTA folds the partials in the same order -> identical blended bounds everywhere
  {
    float f[2] = {INFINITY, -INFINITY};
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
      f[0] = fminf(f[0], __ldcg(&ws->partials[b * kPartialStride + 0]));
      f[1] = fmaxf(f[1], __ldcg(&ws->partials[b * kPartialStride + 1]));
    }
    block_fold<2>(f, op2, smem);
    if (threadIdx.x == 0) {                                               // camera_isp.py:156
      s_bounds[0] = __fadd_rn(f[0], __fmul_rn(alpha, __fsub_rn(prev[0], f[0])));
      s_bounds[1] = __fadd_rn(f[1], __fmul_rn(alpha, __fsub_rn(prev[1], f[1])));
    }
    __syncthreads();
  }
  const float bmin = s_bounds[0], bmax = s_bounds[1];
  const float inv_den = __fdiv_rn(1.0f, __fadd_rn(__fsub_rn(bmax, bmin), 1e-6f));

  // ---- phase 2: statistics w.r.t. the blended bounds (samples from the L2-resident cache, else recomputed)
  float v[7] = {INFINITY, -INFINITY, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (cache) for_each_sample(CachedSampler{cache}, n, [&](long long, const float (&rgb)[3]) { meter_accum(rgb, bmin, inv_den, v); });
  else for_each_sample(smp, n, [&](long long, const float (&rgb)[3]) { meter_accum(rgb, bmin, inv_den, v); });
  const int op[7] = {0, 1, 2, 2, 2, 2, 2};
  block_fold<7>(v, op, smem);
  if (threadIdx.x == 0) {
#pragma unroll
    for (int k = 0; k < 7; ++k) part2[blockIdx.x * kPartialStride + k] = v[k];
  }
  if (last_block_ticket(&ws->counter[0])) {
    float f[7] = {INFINITY, -INFINITY, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int b = threadIdx.x; b < (int)gridDim.x; b += blockDim.x) {
      f[0] = fminf(f[0], __ldcg(&part2[b * kPartialStride + 0]));
      f[1] = fmaxf(f[1], __ldcg(&part2[b * kPartialStride + 1]));
#pragma unroll
      for (int k = 2; k < 7; ++k) f[k] += __ldcg(&part2[b * kPartialStride + k]);
    }
    block_fold<7>(f, op, smem);
    if (threadIdx.x == 0) {
      ws->counter[1] = 0u;                                                // barrier counter back to zero for the next launch
      ws->bounds[0] = bmin; ws->bounds[1] = bmax;
      const float fn = (float)n;                                          // camera_isp.py:131-134
      const float stats[9] = {bmin, bmax, f[0], f[1], __fdiv_rn(f[2], fn), __fdiv_rn(f[3], fn),
                              __fdiv_rn(f[4], fn), __fdiv_rn(f[5], fn), __fdiv_rn(f[6], fn)};
#pragma unroll
      for (int k = 0; k < 9; ++k) {                                       // camera_isp.py:165-166
        const float p = prev[k];
        metrics[k] = __fadd_rn(stats[k], __fmul_rn(alpha, __fsub_rn(p, stats[k])));
      }
    }
  }
}

inline int meter_grid(long long n) {
  long long b = (n + 256 * 4 - 1) / (256 * 4);
  if (b < 1) b = 1;
  if (b > 4 * kNumSMs) b = 4 * kNumSMs;
  return (int)b;
}

// Grid of the two-launch (look-ahead / shared) form, which runs on a high-priority side stream UNDER the previous batch's
// sweep: its CTAs take SM slots away from the sweep for as long as they live, so a latency-bound sampler should not
// flood the GPU.  Samplers may define kSideGridCap (CTAs).
template <class Sampler, class = void> struct side_grid_cap { static constexpr int value = 4 * kNumSMs; };
template <class Sampler> struct side_grid_cap<Sampler, std::enable_if_t<(Sampler::kSideGridCap > 0)>> { static constexpr int value = Sampler::kSideGridCap; };
template <class Sampler>
inline int meter_side_grid(long long n) {
  const int cap = side_grid_cap<Sampler>::value;
  const int g = meter_grid(n);
  return g < cap ? g : cap;
}

// cache: optional device scratch of n*3 floats -- phase 2 then re-reads the phase-1 samples instead of
// recomputing them (the samples are identical either way).
// prev: metrics before this update (read), metrics: updated metrics (written; may be the same buffer).
// cooperative = false forces the two-launch form, whose CTAs can interleave with another kernel's CTAs on a
// busy GPU (a cooperative grid must wait until all of its CTAs fit at once): used by the look-ahead metering
// that runs on a side stream under the previous batch's sweep.
template <class Sampler>
inline int launch_metering(const Sampler& smp, long long n, float alpha, const float* prev, float* metrics, Workspace* ws,
                           cudaStream_t s, float* cache = nullptr, bool cooperative = true) {
  int dev = 0, sms = 0, per_sm = 0, coop = 0;
  if (cooperative && cudaGetDevice(&dev) == cudaSuccess &&
      cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev) == cudaSuccess && coop &&
      cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess &&
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, meter_fused_kernel<Sampler>, 256, 0) == cudaSuccess && per_sm > 0) {
    long long want = (n + 256 * kMeterUnroll - 1) / (256 * kMeterUnroll);
    long long cap = (long long)per_sm * sms;
    if (cap > kMaxPartialBlocks / 2) cap = kMaxPartialBlocks / 2;
    int grid = (int)(want < 1 ? 1 : (want > cap ? cap : want));
    void* args[] = {(void*)&smp, (void*)&n, (void*)&alpha, (void*)&prev, (void*)&metrics, (void*)&ws, (void*)&cache};
    const cudaError_t e = cudaLaunchCooperativeKernel((const void*)meter_fused_kernel<Sampler>, dim3(grid), dim3(256), args, 0, s);
    if (e == cudaSuccess) return B200ISP_OK;
    (void)cudaGetLastError();         // fall through to the two-launch form
  }
  const int grid = cooperative ? meter_grid(n) : meter_side_grid<Sampler>(n);
  meter_phase1_kernel<Sampler><<<grid, 256, 0, s>>>(smp, n, alpha, prev, ws, cache);
  int st = cuda_status(cudaPeekAtLastError(), "meter_phase1_kernel");
  if (st) return st;
  if (cache) return launch_meter_phase2_cached(grid, CachedSampler{cache}, n, alpha, prev, metrics, ws, s, nullptr);
  meter_phase2_kernel<Sampler><<<grid, 256, 0, s>>>(smp, n, alpha, prev, metrics, ws);
  return cuda_status(cudaPeekAtLastError(), "meter_phase2_kernel");
}

// the two halves of launch_metering for the shared-exposure exchange
template <class Sampler>
inline int launch_metering_phase1(const Sampler& smp, long long n, Workspace* ws, cudaStream_t s, float* cache, float* rec1) {
  meter_phase1_kernel<Sampler><<<meter_grid(n), 256, 0, s>>>(smp, n, 0.f, nullptr, ws, cache, rec1);
  return cuda_status(cudaPeekAtLastError(), "meter_phase1_kernel");
}
template <class Sampler>
inline int launch_metering_phase2(const Sampler& smp, long long n, const float* g1, int world, float alpha, const float* prev,
                                  Workspace* ws, cudaStream_t s, const float* cache, float* rec2) {
  const int st = launch_meter_fold_bounds(g1, world, alpha, prev, ws, s);
  if (st) return st;
  const int grid = meter_grid(n);
  if (cache) return launch_meter_phase2_cached(grid, CachedSampler{cache}, n, alpha, nullptr, nullptr, ws, s, rec2);
  meter_phase2_kernel<Sampler><<<grid, 256, 0, s>>>(smp, n, alpha, nullptr, nullptr, ws, rec2);
  return cuda_status(cudaPeekAtLastError(), "meter_phase2_kernel");
}

// joint metering update of all ranks in two launches (the exchange runs inside the kernels' last block)
template <class Sampler>
inline int launch_metering_shared(const Sampler& smp, long long n, float alpha, const float* prev, float* metrics, Workspace* ws,
                                  cudaStream_t s, float* cache, const PeerXchg& xc) {
  const int grid = meter_side_grid<Sampler>(n);
  meter_phase1x_kernel<Sampler><<<grid, 256, 0, s>>>(smp, n, alpha, prev, ws, cache, xc);
  int st = cuda_status(cudaPeekAtLastError(), "meter_phase1x_kernel");
  if (st) return st;
  if (cache) meter_phase2x_kernel<CachedSampler><<<grid, 256, 0, s>>>(CachedSampler{cache}, n, alpha, prev, metrics, ws, xc);
  else meter_phase2x_kernel<Sampler><<<grid, 256, 0, s>>>(smp, n, alpha, prev, metrics, ws, xc);
  return cuda_status(cudaPeekAtLastError(), "meter_phase2x_kernel");
}

// Sampler over materialised (H, W, 3) images of the ISP dtype (camera_isp.py:168-170)
template <typename T>
struct ImageSampler {
  const T* img[B200ISP_MAX_FRAMES];
  int W, stride, hs, ws_;     // hs = ceil(H/stride), ws_ = ceil(W/stride)
  __device__ __forceinline__ void sample(long long idx, float (&rgb)[3]) const {
    const int j = (int)(idx % ws_);
    const long long q = idx / ws_;
    const int i = (int)(q % hs);
    const int f = (int)(q / hs);
    const T* p = img[f] + ((size_t)i * stride * W + (size_t)j * stride) * 3;
    rgb[0] = to_f32(p[0]); rgb[1] = to_f32(p[1]); rgb[2] = to_f32(p[2]);
  }
};

}  // namespace isp
