// Gather kernels: bilinear resize, area resize (extension) and the 8 rotate/flip transforms
// (reference: interpolate.py:19-66 bilinear, :36-56 / :93-108 transform).
#include <cstdlib>
#include "common.cuh"

namespace isp {

__device__ __forceinline__ float mixf(float a, float b, float t) {   // GLSL mix: a*(1-t) + b*t, rounded per op
  return __fadd_rn(__fmul_rn(a, __fsub_rn(1.0f, t)), __fmul_rn(b, t));
}

// interpolate.py:59-66: p = I / scale (no half-pixel offset), p1 = trunc(p), clamp-to-edge taps,
// mix along dim 0 first (frac.x), then dim 1; cast(out * intensity_scale) truncating.
template <typename InT, typename OutT>
__global__ void __launch_bounds__(256) bilinear_kernel(const InT* __restrict__ src, int hs, int ws,
                                                       OutT* __restrict__ dst, int hd, int wd,
                                                       float scale_r, float scale_c, float intensity) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  const int row = blockIdx.y;
  if (col >= wd) return;
  const float pr = __fdiv_rn((float)row, scale_r), pc = __fdiv_rn((float)col, scale_c);
  const int r1 = (int)pr, c1 = (int)pc;
  const float fr = __fsub_rn(pr, (float)r1), fc = __fsub_rn(pc, (float)c1);
  const int ra = min(max(r1, 0), hs - 1), rb = min(max(r1 + 1, 0), hs - 1);
  const int ca = min(max(c1, 0), ws - 1), cb = min(max(c1 + 1, 0), ws - 1);
  const InT* s00 = src + ((size_t)ra * ws + ca) * 3;
  const InT* s10 = src + ((size_t)rb * ws + ca) * 3;
  const InT* s01 = src + ((size_t)ra * ws + cb) * 3;
  const InT* s11 = src + ((size_t)rb * ws + cb) * 3;
  OutT* o = dst + ((size_t)row * wd + col) * 3;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float y1 = mixf(to_f32(s00[k]), to_f32(s10[k]), fr);
    const float y2 = mixf(to_f32(s01[k]), to_f32(s11[k]), fr);
    o[k] = cast_from_f32<OutT>(__fmul_rn(mixf(y1, y2, fc), intensity));
  }
}

// EXTENSION (no reference kernel): exact box filter.  Output pixel (i, j) averages the source over
// [i*hs/hd, (i+1)*hs/hd) x [j*ws/wd, (j+1)*ws/wd) with fractional coverage weights.
template <typename InT, typename OutT>
__global__ void __launch_bounds__(256) area_kernel(const InT* __restrict__ src, int hs, int ws,
                                                   OutT* __restrict__ dst, int hd, int wd, float intensity) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  const int row = blockIdx.y;
  if (col >= wd) return;
  const float fr = (float)hs / (float)hd, fc = (float)ws / (float)wd;
  const float r0 = row * fr, r1 = fminf((row + 1) * fr, (float)hs);
  const float c0 = col * fc, c1 = fminf((col + 1) * fc, (float)ws);
  float acc[3] = {0.f, 0.f, 0.f}, wsum = 0.f;
  for (int r = (int)r0; r < hs && (float)r < r1; ++r) {
    const float wr = fminf(r1, (float)(r + 1)) - fmaxf(r0, (float)r);
    if (wr <= 0.f) continue;
    for (int c = (int)c0; c < ws && (float)c < c1; ++c) {
      const float wc = fminf(c1, (float)(c + 1)) - fmaxf(c0, (float)c);
      if (wc <= 0.f) continue;
      const float w = wr * wc;
      const InT* p = src + ((size_t)r * ws + c) * 3;
      acc[0] = fmaf(w, to_f32(p[0]), acc[0]);
      acc[1] = fmaf(w, to_f32(p[1]), acc[1]);
      acc[2] = fmaf(w, to_f32(p[2]), acc[2]);
      wsum += w;
    }
  }
  OutT* o = dst + ((size_t)row * wd + col) * 3;
  const float inv = wsum > 0.f ? intensity / wsum : 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k) o[k] = cast_from_f32<OutT>(acc[k] * inv);
}

// interpolate.py:36-56: source index for destination (r, c); (H, W) = SOURCE shape.
// rotate_90 is clockwise (SURVEY Q11); transverse is the corrected anti-transpose (SURVEY Q10).
__device__ __forceinline__ void transformed(int t, int r, int c, int H, int W, int& sr, int& sc) {
  switch (t) {
    case B200ISP_T_ROT90:      sr = H - 1 - c; sc = r;         break;
    case B200ISP_T_ROT180:     sr = H - 1 - r; sc = W - 1 - c; break;
    case B200ISP_T_ROT270:     sr = c;         sc = W - 1 - r; break;
    case B200ISP_T_TRANSPOSE:  sr = c;         sc = r;         break;
    case B200ISP_T_FLIP_VERT:  sr = H - 1 - r; sc = c;         break;
    case B200ISP_T_FLIP_HORIZ: sr = r;         sc = W - 1 - c; break;
    case B200ISP_T_TRANSVERSE: sr = H - 1 - c; sc = W - 1 - r; break;
    default:                   sr = r;         sc = c;         break;
  }
}

// 32x32-pixel tiles staged through shared memory so that both the read and the write side stay
// row-contiguous for the transposing transforms.
template <typename T>
__global__ void __launch_bounds__(256) transform_kernel(const T* __restrict__ src, T* __restrict__ dst,
                                                        int H, int W, int hd, int wd, int t) {
  __shared__ T tile[32][32 * 3 + 1];
  const bool swaps = (t == B200ISP_T_ROT90 || t == B200ISP_T_ROT270 || t == B200ISP_T_TRANSPOSE || t == B200ISP_T_TRANSVERSE);
  const int dr0 = blockIdx.y * 32, dc0 = blockIdx.x * 32;      // destination tile origin
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8 threads
  if (!swaps) {
    // row-preserving: each destination row maps to one source row, columns possibly reversed
    for (int y = ty; y < 32; y += 8) {
      const int r = dr0 + y;
      if (r >= hd) continue;
      for (int e = tx; e < 96; e += 32) {
        const int c = dc0 + e / 3, k = e % 3;
        if (c >= wd) continue;
        int sr, sc;
        transformed(t, r, c, H, W, sr, sc);
        dst[((size_t)r * wd + c) * 3 + k] = src[((size_t)sr * W + sc) * 3 + k];
      }
    }
    return;
  }
  // transposing: load the source tile row-wise (source rows <-> destination columns)
  for (int y = ty; y < 32; y += 8) {
    // source pixel for destination (dr0 + x, dc0 + y): walk x fastest on the destination ROW index so
    // that consecutive threads read consecutive source columns.
    for (int e = tx; e < 96; e += 32) {
      const int x = e / 3, k = e % 3;
      const int r = dr0 + x, c = dc0 + y;
      if (r < hd && c < wd) {
        int sr, sc;
        transformed(t, r, c, H, W, sr, sc);
        tile[x][y * 3 + k] = src[((size_t)sr * W + sc) * 3 + k];
      }
    }
  }
  __syncthreads();
  for (int y = ty; y < 32; y += 8) {
    const int r = dr0 + y;
    if (r >= hd) continue;
    for (int e = tx; e < 96; e += 32) {
      const int c = dc0 + e / 3;
      if (c < wd) dst[((size_t)r * wd + c) * 3 + e % 3] = tile[y][e];
    }
  }
}

// ---------------------------------------------------------------- word-granular transform (the fast path)
// Same tiling idea, but the global accesses are 4-byte words on both sides and the tile is addressed as raw bytes:
// a pixel is PB = 3 * sizeof(T) bytes, moved in granules of G = gcd(PB, 4) bytes (1 for u8, 2 for u16 / f16, 4 for
// f32).  Phase 1 copies the source tile row segments (word-aligned start rounded down, `boff` = the bytes skipped)
// into shared memory; phase 2 assembles every destination word from its 4 / G granules through the affine map
// destination (y, x) -> source (sy, sx) of the transform (tile-local).  Needs 4-byte aligned bases and row pitches
// (W * PB and wd * PB multiples of 4); everything else takes transform_kernel above.  The padded row pitch is an
// odd number of words, so the column-wise reads of the transposing transforms are bank-conflict free.
template <int PB, int TILE>
__global__ void __launch_bounds__(256) transform_words_kernel(const uint32_t* __restrict__ src, uint32_t* __restrict__ dst,
                                                              int H, int W, int hd, int wd, int t) {
  constexpr int G = (PB % 4 == 0) ? 4 : ((PB % 2 == 0) ? 2 : 1);
  constexpr int ROW_WORDS = TILE * PB / 4 + 1;                       // + 1 word for a misaligned start; odd pitch
  static_assert(ROW_WORDS % 2 == 1, "odd smem pitch");
  __shared__ uint32_t tile[TILE][ROW_WORDS];
  const int dr0 = blockIdx.y * TILE, dc0 = blockIdx.x * TILE;
  const int nr = min(TILE, hd - dr0), nc = min(TILE, wd - dc0);     // destination tile extent
  // affine map in global coordinates: corners -> source tile origin and extent
  int sra, sca, srb, scb;
  transformed(t, dr0, dc0, H, W, sra, sca);
  transformed(t, dr0 + nr - 1, dc0 + nc - 1, H, W, srb, scb);
  const int sr0 = min(sra, srb), sc0 = min(sca, scb);
  const int snr = abs(srb - sra) + 1, snc = abs(scb - sca) + 1;      // source tile extent
  // phase 1: source rows sr0 .. sr0+snr-1, bytes [sc0 * PB, (sc0 + snc) * PB) of each, as aligned words
  const int src_pitch_w = W * PB / 4;
  const int b0 = sc0 * PB, w0 = b0 >> 2, boff = b0 & 3;
  const int nwords = ((b0 + snc * PB + 3) >> 2) - w0;
  for (int i = threadIdx.x; i < snr * nwords; i += 256) {
    const int y = i / nwords, w = i - y * nwords;
    tile[y][w] = __ldg(src + (size_t)(sr0 + y) * src_pitch_w + w0 + w);
  }
  __syncthreads();
  // tile-local affine map: (sy, sx) = (oy + ayy * y + ayx * x, ox + axy * y + axx * x)
  int s00r, s00c, s10r, s10c, s01r, s01c;
  transformed(t, dr0, dc0, H, W, s00r, s00c);
  transformed(t, dr0 + 1, dc0, H, W, s10r, s10c);
  transformed(t, dr0, dc0 + 1, H, W, s01r, s01c);
  const int oy = s00r - sr0, ox = s00c - sc0;
  const int ayy = s10r - s00r, axy = s10c - s00c, ayx = s01r - s00r, axx = s01c - s00c;
  const unsigned char* tb = reinterpret_cast<const unsigned char*>(&tile[0][0]);
  const int dst_pitch_w = wd * PB / 4;
  // phase 2: 12-byte groups (4 / 2 / 1 pixels = 3 words): one affine map per pixel, compile-time byte positions.
  // The destination tile starts word-aligned (TILE * PB % 4 == 0); nc * PB is a multiple of 4 because the row pitch
  // is, and for PB = 3 / 6 / 12 that makes it a multiple of 12 as well (nc % 4 == 0 / nc % 2 == 0 / any nc).
  constexpr int PPG = 12 / PB;
  const int dw0 = dc0 * PB / 4;
  const int groups = nc / PPG;
  for (int i = threadIdx.x; i < nr * groups; i += 256) {
    const int y = i / groups, gi = i - y * groups;
    uint32_t o[3] = {0u, 0u, 0u};
#pragma unroll
    for (int j = 0; j < PPG; ++j) {
      const int x = gi * PPG + j;
      const int sy = oy + ayy * y + ayx * x, sx = ox + axy * y + axx * x;
      const unsigned char* q = tb + (size_t)sy * (ROW_WORDS * 4) + boff + sx * PB;
#pragma unroll
      for (int g = 0; g < PB / G; ++g) {
        uint32_t v;
        if constexpr (G == 4) v = *reinterpret_cast<const uint32_t*>(q + 4 * g);
        else if constexpr (G == 2) v = *reinterpret_cast<const unsigned short*>(q + 2 * g);
        else v = q[g];
        const int bpos = j * PB + g * G;                             // byte within the 12-byte group (compile time)
        o[bpos >> 2] |= v << (8 * (bpos & 3));
      }
    }
    uint32_t* d = dst + (size_t)(dr0 + y) * dst_pitch_w + dw0 + 3 * gi;
    d[0] = o[0]; d[1] = o[1]; d[2] = o[2];
  }
}

// ---------------------------------------------------------------- transposing transforms of u8 / 16-bit RGB, the turned path
// rotate_90 / rotate_270 / transpose / transverse of images whose height and width are multiples of 8 (every frame the fused
// sweep accepts with H % 8 == 0): destination (i, j) = source (r, c), r = j or H-1-j (MR), c = i or W-1-i (MC).
// CTA = 128 destination columns (source rows) x 32 destination rows (source columns).  A pixel travels through shared memory
// as whole 32-bit words -- one word for 3-byte pixels (R | G << 8 | B << 16), two words in two planes for 6-byte pixels
// (c0 | c1 << 16, c2) -- instead of byte granules: per pixel 1 / 2 STS + 1 / 2 LDS and two or three PRMT on each side.
// Load phase: thread = 8 consecutive source pixels (24 / 48 bytes, 8- / 16-byte vectors), a warp covers 8 source rows x 32
// columns; store phase: thread = 8 consecutive destination pixels, a half warp writes 384 / 768 contiguous bytes of one
// destination row.  Layout [dest row li][lr + (lr >> 3)] with row pitch 144 words and 8 extra words per 8 rows: both the
// stores of the load phase and the loads of the store phase are bank-conflict free.  blockIdx.x runs along the destination
// row, so the partial sectors at the ends of a piece meet their neighbours' in L2 (default write policy).
constexpr int kTurnRows = 128, kTurnCols = 32, kTurnPitch = 144, kTurnPlane = kTurnCols * kTurnPitch + 8 * (kTurnCols / 8 - 1);
template <int PB>
__global__ void __launch_bounds__(256) transform_turn_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int H, int W,
                                                             int mirror_r, int mirror_c) {
  static_assert(PB == 3 || PB == 6, "u8 or 16-bit RGB");
  constexpr int NP = PB / 3;                       // planes of words per pixel
  constexpr int NW = 2 * PB;                       // 32-bit words of 8 pixels
  __shared__ uint32_t tile[NP][kTurnPlane];
  const int j0 = blockIdx.x * kTurnRows, i0 = blockIdx.y * kTurnCols;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int id = threadIdx.x + 256 * it;
    const int cg = id & 3, lr = id >> 2;
    const int j = j0 + lr, ig = i0 + 8 * cg;       // first destination row of the group
    if (j < H && ig < W) {
      const int r = mirror_r ? H - 1 - j : j;
      const int cs = mirror_c ? W - 8 - ig : ig;   // first SOURCE column of the eight
      const uint8_t* sp = src + ((size_t)r * W + cs) * PB;
      uint32_t w[NW];
      if constexpr (PB == 3) {
#pragma unroll
        for (int v = 0; v < 3; ++v) { const uint2 x = __ldg(reinterpret_cast<const uint2*>(sp) + v); w[2 * v] = x.x; w[2 * v + 1] = x.y; }
      } else {
#pragma unroll
        for (int v = 0; v < 3; ++v) { const uint4 x = __ldg(reinterpret_cast<const uint4*>(sp) + v); w[4 * v] = x.x; w[4 * v + 1] = x.y; w[4 * v + 2] = x.z; w[4 * v + 3] = x.w; }
      }
      uint32_t pa[8], pb[8];
      if constexpr (PB == 3) {
#pragma unroll
        for (int g = 0; g < 2; ++g) {              // 4 pixels = 3 words; the top byte of a pixel word is never read
          pa[4 * g] = w[3 * g];
          pa[4 * g + 1] = __byte_perm(w[3 * g], w[3 * g + 1], 0x0543);
          pa[4 * g + 2] = __byte_perm(w[3 * g + 1], w[3 * g + 2], 0x0432);
          pa[4 * g + 3] = w[3 * g + 2] >> 8;
        }
      } else {
#pragma unroll
        for (int g = 0; g < 4; ++g) {              // 2 pixels = 3 words; the top half of a plane-1 word is never read
          pa[2 * g] = w[3 * g];
          pb[2 * g] = w[3 * g + 1];
          pa[2 * g + 1] = __byte_perm(w[3 * g + 1], w[3 * g + 2], 0x5432);
          pb[2 * g + 1] = w[3 * g + 2] >> 16;
        }
      }
      const int pos = lr + (lr >> 3);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const int li = 8 * cg + (mirror_c ? 7 - q : q);
        const int at = li * kTurnPitch + 8 * cg + pos;
        tile[0][at] = pa[q];
        if constexpr (NP == 2) tile[1][at] = pb[q];
      }
    }
  }
  __syncthreads();
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int id = threadIdx.x + 256 * it;
    const int rg = id & 15, li = id >> 4;
    const int i = i0 + li, j = j0 + 8 * rg;
    if (i < W && j < H) {
      const int at = li * kTurnPitch + 8 * (li >> 3) + 9 * rg;
      uint32_t pa[8], pb[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        pa[q] = tile[0][at + q];
        if constexpr (NP == 2) pb[q] = tile[1][at + q];
      }
      uint8_t* dp = dst + ((size_t)i * H + j) * PB;
      if constexpr (PB == 3) {
        uint2* d = reinterpret_cast<uint2*>(dp);
        d[0] = make_uint2(__byte_perm(pa[0], pa[1], 0x4210), __byte_perm(pa[1], pa[2], 0x5421));
        d[1] = make_uint2(__byte_perm(pa[2], pa[3], 0x6542), __byte_perm(pa[4], pa[5], 0x4210));
        d[2] = make_uint2(__byte_perm(pa[5], pa[6], 0x5421), __byte_perm(pa[6], pa[7], 0x6542));
      } else {
        uint32_t o[12];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          o[3 * g] = pa[2 * g];
          o[3 * g + 1] = __byte_perm(pb[2 * g], pa[2 * g + 1], 0x5410);
          o[3 * g + 2] = __byte_perm(pa[2 * g + 1], pb[2 * g + 1], 0x5432);
        }
        uint4* d = reinterpret_cast<uint4*>(dp);
#pragma unroll
        for (int v = 0; v < 3; ++v) d[v] = make_uint4(o[4 * v], o[4 * v + 1], o[4 * v + 2], o[4 * v + 3]);
      }
    }
  }
}

}  // namespace isp

using namespace isp;

extern "C" int b200isp_resize_bilinear(const void* src, int in_dtype, int src_h, int src_w, void* dst, int out_dtype,
                                       int dst_h, int dst_w, float scale_row, float scale_col, b200isp_stream stream) {
  ISP_REQUIRE(src_h > 0 && src_w > 0 && dst_h >= 0 && dst_w >= 0, B200ISP_E_SHAPE, "resize_bilinear: bad shape");
  ISP_REQUIRE(scale_row > 0.f && scale_col > 0.f, B200ISP_E_ARG, "resize_bilinear: scale must be positive");
  if (dst_h == 0 || dst_w == 0) return B200ISP_OK;
  ISP_REQUIRE(src && dst, B200ISP_E_ARG, "resize_bilinear: null pointer");
  const dim3 grid((dst_w + 255) / 256, dst_h);
  cudaStream_t s = (cudaStream_t)stream;
  ISP_DISPATCH_DTYPE(in_dtype, InT, {
    ISP_DISPATCH_DTYPE(out_dtype, OutT, {
      const float intensity = (float)((double)DT<OutT>::scale / (double)DT<InT>::scale);   // interpolate.py:78
      bilinear_kernel<InT, OutT><<<grid, 256, 0, s>>>((const InT*)src, src_h, src_w, (OutT*)dst, dst_h, dst_w,
                                                      scale_row, scale_col, intensity);
    });
  });
  ISP_LAUNCH_CHECK("bilinear_kernel");
  return B200ISP_OK;
}

extern "C" int b200isp_resize_area(const void* src, int in_dtype, int src_h, int src_w, void* dst, int out_dtype,
                                   int dst_h, int dst_w, b200isp_stream stream) {
  ISP_REQUIRE(src_h > 0 && src_w > 0 && dst_h >= 0 && dst_w >= 0, B200ISP_E_SHAPE, "resize_area: bad shape");
  if (dst_h == 0 || dst_w == 0) return B200ISP_OK;
  ISP_REQUIRE(src && dst, B200ISP_E_ARG, "resize_area: null pointer");
  const dim3 grid((dst_w + 255) / 256, dst_h);
  cudaStream_t s = (cudaStream_t)stream;
  ISP_DISPATCH_DTYPE(in_dtype, InT, {
    ISP_DISPATCH_DTYPE(out_dtype, OutT, {
      const float intensity = (float)((double)DT<OutT>::scale / (double)DT<InT>::scale);
      area_kernel<InT, OutT><<<grid, 256, 0, s>>>((const InT*)src, src_h, src_w, (OutT*)dst, dst_h, dst_w, intensity);
    });
  });
  ISP_LAUNCH_CHECK("area_kernel");
  return B200ISP_OK;
}

extern "C" int b200isp_transform(const void* src, void* dst, int dtype, int src_h, int src_w, int transform,
                                 b200isp_stream stream) {
  ISP_REQUIRE(src_h >= 0 && src_w >= 0, B200ISP_E_SHAPE, "transform: bad shape");
  ISP_REQUIRE(transform >= B200ISP_T_NONE && transform <= B200ISP_T_TRANSVERSE, B200ISP_E_ARG, "transform: unknown transform %d", transform);
  if (src_h == 0 || src_w == 0) return B200ISP_OK;
  ISP_REQUIRE(src && dst, B200ISP_E_ARG, "transform: null pointer");
  const bool swaps = (transform == B200ISP_T_ROT90 || transform == B200ISP_T_ROT270 ||
                      transform == B200ISP_T_TRANSPOSE || transform == B200ISP_T_TRANSVERSE);
  const int hd = swaps ? src_w : src_h, wd = swaps ? src_h : src_w;
  cudaStream_t s = (cudaStream_t)stream;
  const int esz = dtype == B200ISP_U8 ? 1 : (dtype == B200ISP_F32 ? 4 : 2), pb = 3 * esz;
  const bool words = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 3u) == 0 &&
                     ((size_t)src_w * pb) % 4 == 0 && ((size_t)wd * pb) % 4 == 0;
  // 3- / 6-byte pixels, both extents multiples of 8, vector-aligned bases: whole-word pixel tiles (transform_turn_kernel)
  if (swaps && (pb == 3 || pb == 6) && src_h % 8 == 0 && src_w % 8 == 0 &&
      ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & (pb == 3 ? 7u : 15u)) == 0) {
    const int mr = (transform == B200ISP_T_ROT90 || transform == B200ISP_T_TRANSVERSE) ? 1 : 0;
    const int mc = (transform == B200ISP_T_ROT270 || transform == B200ISP_T_TRANSVERSE) ? 1 : 0;
    const dim3 grid((src_h + kTurnRows - 1) / kTurnRows, (src_w + kTurnCols - 1) / kTurnCols);
    if (pb == 3) transform_turn_kernel<3><<<grid, 256, 0, s>>>((const uint8_t*)src, (uint8_t*)dst, src_h, src_w, mr, mc);
    else transform_turn_kernel<6><<<grid, 256, 0, s>>>((const uint8_t*)src, (uint8_t*)dst, src_h, src_w, mr, mc);
    ISP_LAUNCH_CHECK("transform_turn_kernel");
    return B200ISP_OK;
  }
  if (words) {
    const uint32_t* sw = (const uint32_t*)src;
    uint32_t* dw = (uint32_t*)dst;
    if (pb == 3) {
      const dim3 grid((wd + 63) / 64, (hd + 63) / 64);
      transform_words_kernel<3, 64><<<grid, 256, 0, s>>>(sw, dw, src_h, src_w, hd, wd, transform);
    } else if (pb == 6) {
      const dim3 grid((wd + 63) / 64, (hd + 63) / 64);
      transform_words_kernel<6, 64><<<grid, 256, 0, s>>>(sw, dw, src_h, src_w, hd, wd, transform);
    } else {
      const dim3 grid((wd + 31) / 32, (hd + 31) / 32);
      transform_words_kernel<12, 32><<<grid, 256, 0, s>>>(sw, dw, src_h, src_w, hd, wd, transform);
    }
    ISP_LAUNCH_CHECK("transform_words_kernel");
    return B200ISP_OK;
  }
  const dim3 grid((wd + 31) / 32, (hd + 31) / 32);
  ISP_DISPATCH_DTYPE(dtype, T, (transform_kernel<T><<<grid, 256, 0, s>>>((const T*)src, (T*)dst, src_h, src_w, hd, wd, transform)));
  ISP_LAUNCH_CHECK("transform_kernel");
  return B200ISP_OK;
}
