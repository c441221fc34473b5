// Stand-alone CFA mosaic / Malvar-He-Cutler demosaic on typed planes
// (reference: bayer.py:101-112 rgb_to_bayer_kernel, bayer.py:114-190 bayer_to_rgb_kernel).
#include "stream_engine.cuh"
#include "pixel_ops.cuh"

namespace isp {

// same-dtype, aligned planes: the pair-engine sweep of plane_sweep.cuh (instantiated per dtype in demosaic_inst.cu)
template <typename T>
int run_demosaic_sweep(const void* bayer, void* rgb, int H, int W, int pattern, const float* ccm, bool bilinear, cudaStream_t s);

// ---------------------------------------------------------------- per-pixel kernel
// Literal bayer.py:137-155 (see pixel_ops.cuh): whole image (mixed dtypes, widths that are not a
// multiple of 8, unaligned views).
template <typename T> struct PlaneSrc {
  const T* base; int W;
  __device__ __forceinline__ float at(int, int r, int c) const { return to_f32(base[(size_t)r * W + c]); }
};

template <typename InT, typename OutT>
__global__ void __launch_bounds__(256) demosaic_pixel_kernel(const InT* __restrict__ bayer, OutT* __restrict__ out,
                                                             int H, int W, int pattern, int ccm, const float9 m, long long count) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= count) return;
  const int row = (int)(idx / W), col = (int)(idx % W);
  const PlaneSrc<InT> src{bayer, W};
  float c[3], t[3];
  malvar_pixel(src, 0, pattern, row, col, H, W, c, t);
  constexpr float is = DT<InT>::scale, os = DT<OutT>::scale;
  float cr = __fdiv_rn(c[0], __fmul_rn(is, t[0])), cg = __fdiv_rn(c[1], __fmul_rn(is, t[1])), cb = __fdiv_rn(c[2], __fmul_rn(is, t[2]));
  if (ccm) ccm_apply(m.v, cr, cg, cb);
  OutT* o = out + ((size_t)row * W + col) * 3;
  o[0] = cast_from_f32<OutT>(__fmul_rn(clamp01(cr), os));
  o[1] = cast_from_f32<OutT>(__fmul_rn(clamp01(cg), os));
  o[2] = cast_from_f32<OutT>(__fmul_rn(clamp01(cb), os));
}

template <typename InT, typename OutT>
static int run_demosaic_pixel(const void* bayer, void* rgb, int H, int W, int pattern, const float* ccm, cudaStream_t s) {
  float9 m;
  for (int i = 0; i < 9; ++i) m.v[i] = ccm ? ccm[i] : 0.f;
  const long long count = (long long)H * W;
  demosaic_pixel_kernel<InT, OutT><<<(unsigned)((count + 255) / 256), 256, 0, s>>>(
      (const InT*)bayer, (OutT*)rgb, H, W, pattern, ccm != nullptr, m, count);
  return cuda_status(cudaPeekAtLastError(), "demosaic_pixel_kernel");
}

// ---------------------------------------------------------------- bilinear demosaic (EXTENSION)
// north_star names "Malvar-He-Cutler / bilinear demosaic"; the reference has only Malvar (SURVEY 2.4).  Defined as the
// classic 3x3 bilinear CFA interpolation evaluated with the SAME rule as bayer.py:137-155: per channel
// c = sum of in-bounds (v * w), t = sum of in-bounds w, c / (in_scale * t), [CCM], clamp, cast(c * out_scale) --
// i.e. the mean of the in-bounds neighbours of that colour.  Site kernels (x4; taps in row-major 3x3 order):
//   K0 R site: R = centre, G = N,S,E,W, B = 4 diagonals       K3 B site: K0 with R <-> B
//   K1 G site with R above/below: R = N,S, B = E,W            K2 G site with R left/right: R = E,W, B = N,S
// accumulate tap i (weight W) into channel CH exactly like the generic loop: c += v * w (separately rounded), t += w
#define ISP_BL_TAP(CH, I, Wt) { c[CH] = __fadd_rn(c[CH], __fmul_rn(v[I], Wt)); t[CH] += m[I] * Wt; }

template <typename InT, typename OutT>
__global__ void __launch_bounds__(256) demosaic_bilinear_kernel(const InT* __restrict__ bayer, OutT* __restrict__ out,
                                                                int H, int W, int pattern, int ccm, const float9 m9) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  const int row = blockIdx.y;
  if (col >= W || row >= H) return;
  const int K = site_kernel(pattern, row, col);
  // 3x3 neighbourhood, 0 outside the image (m = in-bounds indicator); taps in row-major order
  float v[9], m[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    const int rr = row + i / 3 - 1, cc = col + i % 3 - 1;
    const bool in = rr >= 0 && rr < H && cc >= 0 && cc < W;
    v[i] = in ? to_f32(bayer[(size_t)rr * W + cc]) : 0.f;
    m[i] = in ? 1.f : 0.f;
  }
  float c[3] = {0.f, 0.f, 0.f}, t[3] = {0.f, 0.f, 0.f};
  // c_bilinear[K] with compile-time weights (zero-weight taps add exactly 0 and are skipped); same tap order
  if (K == 0) {              // R site: R centre, G cross, B diagonals
    ISP_BL_TAP(2, 0, 1.f) ISP_BL_TAP(1, 1, 1.f) ISP_BL_TAP(2, 2, 1.f) ISP_BL_TAP(1, 3, 1.f) ISP_BL_TAP(0, 4, 4.f)
    ISP_BL_TAP(1, 5, 1.f) ISP_BL_TAP(2, 6, 1.f) ISP_BL_TAP(1, 7, 1.f) ISP_BL_TAP(2, 8, 1.f)
  } else if (K == 3) {       // B site: the same with R <-> B
    ISP_BL_TAP(0, 0, 1.f) ISP_BL_TAP(1, 1, 1.f) ISP_BL_TAP(0, 2, 1.f) ISP_BL_TAP(1, 3, 1.f) ISP_BL_TAP(2, 4, 4.f)
    ISP_BL_TAP(1, 5, 1.f) ISP_BL_TAP(0, 6, 1.f) ISP_BL_TAP(1, 7, 1.f) ISP_BL_TAP(0, 8, 1.f)
  } else if (K == 1) {       // G site, R above / below, B left / right
    ISP_BL_TAP(0, 1, 2.f) ISP_BL_TAP(2, 3, 2.f) ISP_BL_TAP(1, 4, 4.f) ISP_BL_TAP(2, 5, 2.f) ISP_BL_TAP(0, 7, 2.f)
  } else {                   // G site, R left / right, B above / below
    ISP_BL_TAP(2, 1, 2.f) ISP_BL_TAP(0, 3, 2.f) ISP_BL_TAP(1, 4, 4.f) ISP_BL_TAP(0, 5, 2.f) ISP_BL_TAP(2, 7, 2.f)
  }
  constexpr float is = DT<InT>::scale, os = DT<OutT>::scale;
  // a 2-pixel-wide image can leave a colour without any in-bounds neighbour (t = 0): define it as 0
  float cr = t[0] > 0.f ? __fdiv_rn(c[0], __fmul_rn(is, t[0])) : 0.f;
  float cg = t[1] > 0.f ? __fdiv_rn(c[1], __fmul_rn(is, t[1])) : 0.f;
  float cb = t[2] > 0.f ? __fdiv_rn(c[2], __fmul_rn(is, t[2])) : 0.f;
  if (ccm) ccm_apply(m9.v, cr, cg, cb);
  OutT* o = out + ((size_t)row * W + col) * 3;
  o[0] = cast_from_f32<OutT>(__fmul_rn(clamp01(cr), os));
  o[1] = cast_from_f32<OutT>(__fmul_rn(clamp01(cg), os));
  o[2] = cast_from_f32<OutT>(__fmul_rn(clamp01(cb), os));
}
#undef ISP_BL_TAP

// ---------------------------------------------------------------- rgb_to_bayer (bayer.py:101-112)
// pixel_orders (bayer.py:85-90): channel at ((r0,c0),(r0,c1),(r1,c0),(r1,c1)), 2 bits each
template <typename T>
__global__ void __launch_bounds__(256) rgb_to_bayer_kernel(const T* __restrict__ rgb, T* __restrict__ bayer,
                                                           int H, int W, unsigned order) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  if (c >= (W & ~1) || r >= (H & ~1)) return;
  const int ch = (order >> (2 * ((r & 1) * 2 + (c & 1)))) & 3;
  bayer[(size_t)r * W + c] = rgb[((size_t)r * W + c) * 3 + ch];
}

// eight pixels per thread with 8 / 16-byte accesses (W % 8 == 0, 16-byte aligned bases)
template <typename T>
__global__ void __launch_bounds__(128) rgb_to_bayer_vec_kernel(const T* __restrict__ rgb, T* __restrict__ bayer,
                                                               int H, int W, unsigned order) {
  const int gx = blockIdx.x * blockDim.x + threadIdx.x;
  const int r = blockIdx.y;
  if (gx >= W / 8) return;
  alignas(16) T px[24];
  alignas(16) T out[8];
  ld_bytes<24 * sizeof(T)>(rgb + ((size_t)r * W + 8 * gx) * 3, px);
  const int ch0 = (order >> (2 * ((r & 1) * 2))) & 3, ch1 = (order >> (2 * ((r & 1) * 2 + 1))) & 3;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const int ch = (c & 1) ? ch1 : ch0;
    out[c] = ch == 0 ? px[3 * c] : (ch == 1 ? px[3 * c + 1] : px[3 * c + 2]);
  }
  st_bytes<8 * sizeof(T)>(bayer + (size_t)r * W + 8 * gx, out);
}

}  // namespace isp

using namespace isp;

extern "C" int b200isp_rgb_to_bayer(const void* rgb, void* bayer, int dtype, int height, int width,
                                    int pattern, b200isp_stream stream) {
  ISP_REQUIRE(height >= 0 && width >= 0, B200ISP_E_SHAPE, "rgb_to_bayer: negative size");
  ISP_REQUIRE(pattern >= 0 && pattern <= 3, B200ISP_E_ARG, "rgb_to_bayer: unknown pattern %d", pattern);
  if (height < 2 || width < 2) return B200ISP_OK;
  ISP_REQUIRE(rgb && bayer, B200ISP_E_ARG, "rgb_to_bayer: null pointer");
  // RGGB (0,1,1,2) GRBG (1,0,2,1) GBRG (1,2,0,1) BGGR (2,1,1,0)
  const unsigned orders[4] = {0u | (1u << 2) | (1u << 4) | (2u << 6), 1u | (0u << 2) | (2u << 4) | (1u << 6),
                              1u | (2u << 2) | (0u << 4) | (1u << 6), 2u | (1u << 2) | (1u << 4) | (0u << 6)};
  cudaStream_t s = (cudaStream_t)stream;
  if (width % 8 == 0 && height % 2 == 0 && ((reinterpret_cast<uintptr_t>(rgb) | reinterpret_cast<uintptr_t>(bayer)) & 15u) == 0) {
    const dim3 grid((width / 8 + 127) / 128, height);
    ISP_DISPATCH_DTYPE(dtype, T, (rgb_to_bayer_vec_kernel<T><<<grid, 128, 0, s>>>((const T*)rgb, (T*)bayer, height, width, orders[pattern])));
  } else {
    const dim3 grid((width + 255) / 256, height);
    ISP_DISPATCH_DTYPE(dtype, T, (rgb_to_bayer_kernel<T><<<grid, 256, 0, s>>>((const T*)rgb, (T*)bayer, height, width, orders[pattern])));
  }
  ISP_LAUNCH_CHECK("rgb_to_bayer_kernel");
  return B200ISP_OK;
}

extern "C" int b200isp_bayer_to_rgb(const void* bayer, int in_dtype, void* rgb, int out_dtype,
                                    int height, int width, int pattern, const float* ccm9_host,
                                    b200isp_stream stream) {
  ISP_REQUIRE(height >= 0 && width >= 0 && height % 2 == 0 && width % 2 == 0, B200ISP_E_SHAPE,
              "bayer_to_rgb: image must be even size, got %dx%d", height, width);
  ISP_REQUIRE(pattern >= 0 && pattern <= 3, B200ISP_E_ARG, "bayer_to_rgb: unknown pattern %d", pattern);
  ISP_REQUIRE(valid_dtype(in_dtype) && valid_dtype(out_dtype), B200ISP_E_DTYPE, "bayer_to_rgb: bad dtype");
  if (height == 0 || width == 0) return B200ISP_OK;
  ISP_REQUIRE(bayer && rgb, B200ISP_E_ARG, "bayer_to_rgb: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  const bool aligned = (width % 8 == 0) && ((reinterpret_cast<uintptr_t>(bayer) | reinterpret_cast<uintptr_t>(rgb)) & 15u) == 0;
  if (aligned && in_dtype == out_dtype && height >= 4 && width >= 8) {
    ISP_DISPATCH_DTYPE(in_dtype, T, return (run_demosaic_sweep<T>(bayer, rgb, height, width, pattern, ccm9_host, false, s)));
  }
  ISP_DISPATCH_DTYPE(in_dtype, InT, {
    ISP_DISPATCH_DTYPE(out_dtype, OutT, return (run_demosaic_pixel<InT, OutT>(bayer, rgb, height, width, pattern, ccm9_host, s)));
  });
  return B200ISP_OK;
}

extern "C" int b200isp_bayer_to_rgb_bilinear(const void* bayer, int in_dtype, void* rgb, int out_dtype,
                                             int height, int width, int pattern, const float* ccm9_host,
                                             b200isp_stream stream) {
  ISP_REQUIRE(height >= 0 && width >= 0 && height % 2 == 0 && width % 2 == 0, B200ISP_E_SHAPE,
              "bayer_to_rgb_bilinear: image must be even size, got %dx%d", height, width);
  ISP_REQUIRE(pattern >= 0 && pattern <= 3, B200ISP_E_ARG, "bayer_to_rgb_bilinear: unknown pattern %d", pattern);
  ISP_REQUIRE(valid_dtype(in_dtype) && valid_dtype(out_dtype), B200ISP_E_DTYPE, "bayer_to_rgb_bilinear: bad dtype");
  if (height == 0 || width == 0) return B200ISP_OK;
  ISP_REQUIRE(bayer && rgb, B200ISP_E_ARG, "bayer_to_rgb_bilinear: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  const bool aligned = (width % 8 == 0) && ((reinterpret_cast<uintptr_t>(bayer) | reinterpret_cast<uintptr_t>(rgb)) & 15u) == 0;
  if (aligned && in_dtype == out_dtype && height >= 4 && width >= 8) {      // the same sweep with the bilinear row formulas
    ISP_DISPATCH_DTYPE(in_dtype, T, return (run_demosaic_sweep<T>(bayer, rgb, height, width, pattern, ccm9_host, true, s)));
  }
  float9 m;
  for (int i = 0; i < 9; ++i) m.v[i] = ccm9_host ? ccm9_host[i] : 0.f;
  const dim3 grid((width + 255) / 256, height);
  ISP_DISPATCH_DTYPE(in_dtype, InT, {
    ISP_DISPATCH_DTYPE(out_dtype, OutT, (demosaic_bilinear_kernel<InT, OutT><<<grid, 256, 0, s>>>(
        (const InT*)bayer, (OutT*)rgb, height, width, pattern, ccm9_host != nullptr, m)));
  });
  ISP_LAUNCH_CHECK("demosaic_bilinear_kernel");
  return B200ISP_OK;
}
