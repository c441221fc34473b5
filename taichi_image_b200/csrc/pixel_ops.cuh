// Per-pixel (gather) form of the Malvar demosaic, literal to bayer.py:137-155: 13 bounds-checked taps
// accumulated in table order, products and sums rounded separately, normaliser t = in-bounds weights.
// Used by the sparse metering samplers, the resizing ISP's gather and the ragged / mixed-dtype stand-alone demosaic.
#pragma once
#include "common.cuh"

namespace isp {

// bayer.py:30-55 expanded (SURVEY Appendix A): [site kernel][tap][channel]; entries 4..7: the bilinear demosaic
// (extension) in the same layout, weights x4 (c / t is unchanged bit for bit by the power of two)
static __constant__ signed char c_taps[8][13][3] = {
  {{0,-2,-3},{0,0,4},{0,4,0},{0,0,4},{0,-2,-3},{0,4,0},{16,8,12},{0,4,0},{0,-2,-3},{0,0,4},{0,4,0},{0,0,4},{0,-2,-3}},
  {{-2,0,1},{-2,0,-2},{8,0,0},{-2,0,-2},{1,0,-2},{0,0,8},{10,16,10},{0,0,8},{1,0,-2},{-2,0,-2},{8,0,0},{-2,0,-2},{-2,0,1}},
  {{1,0,-2},{-2,0,-2},{0,0,8},{-2,0,-2},{-2,0,1},{8,0,0},{10,16,10},{8,0,0},{-2,0,1},{-2,0,-2},{0,0,8},{-2,0,-2},{1,0,-2}},
  {{-3,-2,0},{4,0,0},{0,4,0},{4,0,0},{-3,-2,0},{0,4,0},{12,8,16},{0,4,0},{-3,-2,0},{4,0,0},{0,4,0},{4,0,0},{-3,-2,0}},
  {{0,0,0},{0,0,4},{0,4,0},{0,0,4},{0,0,0},{0,4,0},{16,0,0},{0,4,0},{0,0,0},{0,0,4},{0,4,0},{0,0,4},{0,0,0}},
  {{0,0,0},{0,0,0},{8,0,0},{0,0,0},{0,0,0},{0,0,8},{0,16,0},{0,0,8},{0,0,0},{0,0,0},{8,0,0},{0,0,0},{0,0,0}},
  {{0,0,0},{0,0,0},{0,0,8},{0,0,0},{0,0,0},{8,0,0},{0,16,0},{8,0,0},{0,0,0},{0,0,0},{0,0,8},{0,0,0},{0,0,0}},
  {{0,0,0},{4,0,0},{0,4,0},{4,0,0},{0,0,0},{0,4,0},{0,0,16},{0,4,0},{0,0,0},{4,0,0},{0,4,0},{4,0,0},{0,0,0}}};
static __constant__ signed char c_d0[13] = {-2, -1, -1, -1, 0, 0, 0, 0, 0, 1, 1, 1, 2};
static __constant__ signed char c_d1[13] = {0, -1, 0, 1, -2, -1, 0, 1, 2, -1, 0, 1, 0};

// kernel_patterns of bayer.py:92-97: site kernel at slot k = (row&1) + 2*(col&1)
__device__ __forceinline__ int site_kernel(int pattern, int row, int col) {
  // 2 bits per slot: RGGB (0,1,2,3) GRBG (2,3,0,1) GBRG (1,0,3,2) BGGR (3,2,1,0)
  const unsigned table = pattern == 0 ? 0xE4u : (pattern == 1 ? 0x4Eu : (pattern == 2 ? 0xB1u : 0x1Bu));
  const int slot = (row & 1) + 2 * (col & 1);
  return (table >> (2 * slot)) & 3;
}

// Src concept: float at(int frame, int row, int col) const   -- CFA sample as f32 (in-bounds only)
// returns c = sum(w*v) and t = sum(w) over the in-bounds taps.
template <class Src>
__device__ __forceinline__ void malvar_pixel(const Src& src, int frame, int pattern, int row, int col,
                                             int H, int W, float (&c)[3], float (&t)[3], int kbase = 0) {
  const int K = site_kernel(pattern, row, col) + kbase;
  c[0] = c[1] = c[2] = 0.f;
  t[0] = t[1] = t[2] = 0.f;
#pragma unroll
  for (int i = 0; i < 13; ++i) {
    const int rr = row + c_d0[i], cc = col + c_d1[i];
    if (rr >= 0 && rr < H && cc >= 0 && cc < W) {
      const float v = src.at(frame, rr, cc);
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        const float w = (float)c_taps[K][i][k];
        c[k] = __fadd_rn(c[k], __fmul_rn(v, w));
        t[k] += w;
      }
    }
  }
}

// mat3 @ vec3 with separately rounded products / sums (bayer.py:152-153)
__device__ __forceinline__ void ccm_apply(const float* m, float& r, float& g, float& b) {
  const float x = __fadd_rn(__fadd_rn(__fmul_rn(r, m[0]), __fmul_rn(g, m[1])), __fmul_rn(b, m[2]));
  const float y = __fadd_rn(__fadd_rn(__fmul_rn(r, m[3]), __fmul_rn(g, m[4])), __fmul_rn(b, m[5]));
  const float z = __fadd_rn(__fadd_rn(__fmul_rn(r, m[6]), __fmul_rn(g, m[7])), __fmul_rn(b, m[8]));
  r = x; g = y; b = z;
}

}  // namespace isp
