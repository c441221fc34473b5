// In-sweep renormalisation of the 2-pixel image frame (reference: bayer.py:145-151).
//
// The streaming engines feed "zero samples" for taps outside the image and divide every filter sum by 16.
// The reference divides by t = the sum of the IN-BOUNDS weights of that channel instead.  Because the zero
// samples contribute nothing to the value part of the sum, the exact result is obtained by scaling the
// value part with 16 / t:
//     Camera16 (unbiased samples):  S' = S * 16 / t
//     Camera32 (samples biased by 1.0, all 13 taps always contribute their bias):  S' = (S - 16) * 16 / t + 16
// in units of the x16 filter sum.  t depends only on the site kernel K (bayer.py:92-97), the row class and the
// column class of the pixel (0: first, 1: second, 2: interior, 3: second to last, 4: last), so it is a
// 4 x 5 x 5 x 3 table, built at compile time from the tap table of bayer.py:30-55 (SURVEY Appendix A;
// min |t| = 10, never 0).
// Entries K = 4..7 are the same table for the BILINEAR demosaic (north_star extension; 3 x 3 taps written in
// the 13-tap layout with weights x4, so they also sum to 16 and every formula above holds; min t = 4).
#pragma once
#include "common.cuh"

namespace isp {

constexpr int kBilinearBase = 4;     // site kernel K + kBilinearBase = the bilinear kernel of the same site
struct BorderTable {
  float t[8][5][5][3];   // t = sum of the in-bounds weights (bayer.py:147-149)
  float f[8][5][5][3];   // 16 / t
};

namespace border_detail {
constexpr signed char kTaps[8][13][3] = {
  {{0,-2,-3},{0,0,4},{0,4,0},{0,0,4},{0,-2,-3},{0,4,0},{16,8,12},{0,4,0},{0,-2,-3},{0,0,4},{0,4,0},{0,0,4},{0,-2,-3}},
  {{-2,0,1},{-2,0,-2},{8,0,0},{-2,0,-2},{1,0,-2},{0,0,8},{10,16,10},{0,0,8},{1,0,-2},{-2,0,-2},{8,0,0},{-2,0,-2},{-2,0,1}},
  {{1,0,-2},{-2,0,-2},{0,0,8},{-2,0,-2},{-2,0,1},{8,0,0},{10,16,10},{8,0,0},{-2,0,1},{-2,0,-2},{0,0,8},{-2,0,-2},{1,0,-2}},
  {{-3,-2,0},{4,0,0},{0,4,0},{4,0,0},{-3,-2,0},{0,4,0},{12,8,16},{0,4,0},{-3,-2,0},{4,0,0},{0,4,0},{4,0,0},{-3,-2,0}},
  // bilinear x4: R site (own centre, G cross, B diagonals); G site, R above / below; G site, R left / right; B site
  {{0,0,0},{0,0,4},{0,4,0},{0,0,4},{0,0,0},{0,4,0},{16,0,0},{0,4,0},{0,0,0},{0,0,4},{0,4,0},{0,0,4},{0,0,0}},
  {{0,0,0},{0,0,0},{8,0,0},{0,0,0},{0,0,0},{0,0,8},{0,16,0},{0,0,8},{0,0,0},{0,0,0},{8,0,0},{0,0,0},{0,0,0}},
  {{0,0,0},{0,0,0},{0,0,8},{0,0,0},{0,0,0},{8,0,0},{0,16,0},{8,0,0},{0,0,0},{0,0,0},{0,0,8},{0,0,0},{0,0,0}},
  {{0,0,0},{4,0,0},{0,4,0},{4,0,0},{0,0,0},{0,4,0},{0,0,16},{0,4,0},{0,0,0},{4,0,0},{0,4,0},{4,0,0},{0,0,0}}};
constexpr int kD0[13] = {-2, -1, -1, -1, 0, 0, 0, 0, 0, 1, 1, 1, 2};
constexpr int kD1[13] = {0, -1, 0, 1, -2, -1, 0, 1, 2, -1, 0, 1, 0};
constexpr bool in_bounds(int cls, int d) {
  return cls == 0 ? d >= 0 : cls == 1 ? d >= -1 : cls == 2 ? true : cls == 3 ? d <= 1 : d <= 0;
}
constexpr BorderTable make_table() {
  BorderTable t{};
  for (int K = 0; K < 8; ++K)
    for (int rc = 0; rc < 5; ++rc)
      for (int cc = 0; cc < 5; ++cc)
        for (int ch = 0; ch < 3; ++ch) {
          int s = 0;
          for (int i = 0; i < 13; ++i)
            if (in_bounds(rc, kD0[i]) && in_bounds(cc, kD1[i])) s += kTaps[K][i][ch];
          t.t[K][rc][cc][ch] = (float)s;
          t.f[K][rc][cc][ch] = 16.0f / (float)s;
        }
  return t;
}
}  // namespace border_detail

static __constant__ BorderTable c_border = border_detail::make_table();

__device__ __forceinline__ int edge_class(int x, int n) { return x < 2 ? x : (x >= n - 2 ? x - n + 5 : 2); }

// x = the demosaiced value of one channel normalised by 16 (what the sweep computes everywhere); returns the
// value normalised by the in-bounds weight sum t instead.  x * 16 is exact, the IEEE division keeps the
// Camera16 result correctly rounded (quotients of f16-valued sums by small integers hit f16 rounding ties
// often; a reciprocal multiply breaks them).
__device__ __forceinline__ float frame_exact(float x, float t) { return __fdiv_rn(__fmul_rn(x, 16.f), t); }

// site kernel from the row type and the site type (see fused_isp.cuh): R row -> K0 at R sites, K2 at G sites;
// B row -> K3 at B sites, K1 at G sites
__host__ __device__ constexpr int site_kernel_of(bool brow, bool gsite) { return gsite ? (brow ? 1 : 2) : (brow ? 3 : 0); }

// column class of pixel q (0..7) of a thread: edge bit 0 = first thread column, bit 1 = last
__host__ __device__ constexpr int col_class(int q, int edge) {
  return q < 2 ? ((edge & 1) ? q : 2) : (q >= 6 ? ((edge & 2) ? q - 3 : 2) : 2);
}

struct Vals24 { float v[24]; };    // 8 pixels x RGB, pixel-major

}  // namespace isp
