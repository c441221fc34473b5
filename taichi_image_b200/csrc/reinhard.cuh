// Reinhard photoreceptor tone map of the ISP (reference: camera_isp.py:177-218; the same per-pixel
// map as tonemap.py:107-131): the parameter block and the MUFU-based (lg2/ex2/rcp) evaluation every Reinhard kernel uses;
// relative error ~1e-6, far inside the <= 1 LSB contract of the quantised outputs.
#pragma once
#include "common.cuh"

namespace isp {

struct ReinhardParams {
  float bmin, range;       // metrics[0], metrics[1]-metrics[0]
  float inv_range;         // 1 / range
  float map_key;           // 0.3 + 0.7 * key^1.4                        camera_isp.py:192-193
  float ki;                // exp(-intensity)                            camera_isp.py:208
  float mean[3];           // lerp(ca, stats.mean, stats.rgb_mean)       camera_isp.py:195
  float la, ca;
};

__device__ __forceinline__ ReinhardParams reinhard_params(const float* __restrict__ m, float intensity,
                                                          float light_adapt, float color_adapt) {
  ReinhardParams p;
  const float bmin = m[0], bmax = m[1], lmin = m[2], lmax = m[3], lmean = m[4], mean = m[5];
  p.bmin = bmin;
  p.range = __fsub_rn(bmax, bmin);
  p.inv_range = __frcp_rn(p.range);
  const float key = __fdiv_rn(__fsub_rn(lmax, lmean), __fsub_rn(lmax, lmin));
  p.map_key = __fadd_rn(0.3f, __fmul_rn(0.7f, powf(key, 1.4f)));
  p.ki = expf(-intensity);
  p.la = light_adapt; p.ca = color_adapt;
#pragma unroll
  for (int k = 0; k < 3; ++k) p.mean[k] = __fadd_rn(mean, __fmul_rn(color_adapt, __fsub_rn(m[6 + k], mean)));
  return p;
}

// x^y through the two MUFU ops only (lg2.approx / ex2.approx, no range fix-ups: arguments are O(1) here; x <= 0
// gives NaN / 0 like powf's domain error, which the callers saturate)
__device__ __forceinline__ float fast_pow(float x, float y) {
  float l, r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l) : "f"(x));
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(y * l));
  return r;
}
__device__ __forceinline__ float fast_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }

// s = scaled RGB (already (x - bmin) * inv_range).  CA0: color_adapt == 0 -> one shared adaptation level.
template <bool CA0>
__device__ __forceinline__ void reinhard_map_fast(const ReinhardParams& p, const float (&s)[3], float (&out)[3]) {
  const float gray = fmaf(s[2], 0.114f, fmaf(s[1], 0.587f, s[0] * 0.299f));
  if constexpr (CA0) {
    const float am = fmaf(p.la, gray - p.mean[0], p.mean[0]);
    const float adapt = fast_pow(p.ki * am, p.map_key);
#pragma unroll
    for (int k = 0; k < 3; ++k) out[k] = s[k] * fast_rcp(adapt + s[k]);
  } else {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float ac = fmaf(p.ca, s[k] - gray, gray);
      const float am = fmaf(p.la, ac - p.mean[k], p.mean[k]);
      const float adapt = fast_pow(p.ki * am, p.map_key);
      out[k] = s[k] * fast_rcp(adapt + s[k]);
    }
  }
}

}  // namespace isp
