// Fused camera-ISP sweep: packed12 Bayer -> [metering] -> demosaic -> WB/CCM -> tone map -> RGB8/16/f16
// without materialising the CFA or the float RGB image.
//
// Reference path replaced (camera_isp.py): load_packed12 :333-340 (decode12 packed.py:91-131 +
// bayer_to_rgb bayer.py:114-177), update_metering :376-385 (metering_kernel :142-166),
// tonemap_linear :405-413 (tonemap.py:11-17), tonemap_reinhard :394-403 (reinhard_kernel :177-218).
// Rounding points of the ISP dtype (SURVEY Appendix C) are reproduced: Camera16 rounds the CFA,
// the demosaiced RGB and the Reinhard intermediate through f16; Camera32 keeps f32.
//
// Launch plan per call (all on one stream, no host sync; the 2-pixel image frame is renormalised INSIDE the sweep,
// border_fix.cuh -- there is no border kernel):
//   [metering]  meter_fused_kernel (one cooperative launch) or meter_phase1 -> meter_phase2; sampler straight from the packed bytes
//   linear      stream2<EpiLinear2>                          one sweep
//   reinhard    Camera32: stream2<EpiReinhardMax2> (frame-global max of the mapped values) -> stream2<EpiReinhard2>
//                         (the write sweep recomputes the map), one pair of launches for all frames of the call
//               Camera32 -> u8 (color_adapt 0, gamma 0.3 .. 1): stream2<EpiReinhardMax2, STORE> (u16 fixed-point map)
//                         -> reinhard_map16_out_kernel (normalise / gamma / quantise) -> the two gated exact sweeps
//                         (they leave at once unless the map declined a frame)
//               Camera16: stream2<EpiReinhardMax2, STORE> (writes the f16 map the reference stores back anyway)
//                         -> reinhard_scratch_out_kernel (element-wise normalise / gamma / quantise)
//               either one-sweep form -> u8 with a transposing ISP transform: the pass is reinhard_out_transposed_kernel
//                         (same arithmetic, the image turned through a shared-memory tile; Camera32: after the gated sweeps)
//   none        stream2<EpiRgb2>                             load_packed12 only: float RGB out
//   resizing ISP: csrc/resize_sweep.cuh (stream2_resize_kernel + orphan columns [+ normalise pass])
#pragma once
#include <algorithm>
#include "stream2.cuh"
#include "border_fix.cuh"
#include "pixel_ops.cuh"
#include "metering.cuh"
#include "reinhard.cuh"

namespace isp {

constexpr float kInv4095 = (float)(1.0 / 4095.0);      // packed.py:99 with scale 1.0

struct FramePtrs {
  const uint8_t* in[B200ISP_MAX_FRAMES];
  void* out[B200ISP_MAX_FRAMES];
};

// ---------------------------------------------------------------- packed12 row loader (standard layout)
// Thread column tcol owns pixels 8*tcol..8*tcol+7 = bytes 12*tcol..12*tcol+11 = words 3*tcol..3*tcol+2;
// the halo pixels live in the top 3 bytes of word 3*tcol-1 and the low 3 bytes of word 3*tcol+3.
// Camera32: samples are decoded as b = 1 + v/4096 (12 bits dropped into the mantissa of 1.0f: one
// shift + one LOP3 per pixel, no int->float conversion).  All filter weights sum to 16, so the sums
// come out as 16 + S/4096 exactly and the bias folds into the epilogue's FMA.
// Camera16: the reference stores cfa = f16(v * f32(1/4095)); the same value is produced with one FMA
// (exact product, single rounding) and a packed f32->f16->f32 round trip.
// (biased_from_shifted: common.cuh)

// ---------------------------------------------------------------- packed12 row loader of the pair engine (stream2.cuh)
// Same words and the same one-LOP3 decode as Packed12Loader, but: the decode mask is a register (0 for rows
// outside the image and for the halo columns of the first / last thread column -> "zero sample"), the halo
// loads are predicated on per-thread constants instead of being zero-filled, and the row is delivered as the
// eight pairs (v[k], v[k+4]).
// IDS layout (packed.py:36-44): a pixel pair is the bytes (b0, b1, b2) with p0 = b0 << 4 | (b2 & 0xF), p1 = b1 << 4 | b2 >> 4,
// so a sample's twelve bits are a byte plus a nibble from another byte.  Given the two shifted copies of the word(s) that
// bring the byte to mantissa bits 15..22 (a) and the nibble to bits 11..14 (b), the biased sample 1 + v/4096 is two LOP3:
// a bit select and the usual mask-or -- 4 instead of 2 instructions per sample, still no conversion and no re-pack pass.
__device__ __forceinline__ float ids_sample(uint32_t a, uint32_t b) {
  uint32_t t;
  asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(t) : "r"(a), "r"(b), "r"(0x007F8000u));      // (a & m) | (b & ~m)
  return biased_from_shifted(t, 0x007FF800u, 0x3F800000u);
}

// EXT: the "extended" instantiation that also decodes the IDS layout (run-time flag `ids`).  The lean instantiation carries
// none of that code: the sweep is so sensitive to the size of its hot loop that the run-time branch alone cost the cfg2
// kernel 5 % (160.7 -> 168.8 us) -- measured, profiles/r02_ids_flip.txt.
template <bool CAM16, bool EXT = false>
struct Packed12Loader2 {
  FramePtrs fp;
  int pitch_words;       // W * 3 / 8
  int ids;               // 0: standard layout (packed.py:23-31), 1: IDS layout (packed.py:36-44), kernel-uniform
  static constexpr uint32_t kRowMask = 0x007FF800u;
  struct Raw { uint32_t w[5]; };
  struct Cursor { const uint32_t* p; uint32_t mL, mR; bool left, right, pf; };

  __device__ __forceinline__ ptrdiff_t pitch() const { return pitch_words; }

  template <int KIND>
  __device__ __forceinline__ void open(Cursor& c, int frame, int tcol, const StreamGeom& g) const {
    c.p = reinterpret_cast<const uint32_t*>(fp.in[frame]) + 3 * tcol;
    c.left = KIND == K_CORE || tcol > 0;
    c.right = KIND == K_CORE || tcol < g.ntcols - 1;
    c.mL = c.left ? 0xFFFFFFFFu : 0u;
    c.mR = c.right ? 0xFFFFFFFFu : 0u;
    const int lane = threadIdx.x & 31;
    c.pf = (lane & 7) == 0 || lane == 31;      // 12-byte segments 96 bytes apart touch every 128-byte line of the strip
  }

  template <int KIND>
  __device__ __forceinline__ void fetch(const Cursor& c, const uint32_t* p, Raw& raw) const {
    if (KIND == K_CORE || c.left) raw.w[0] = __ldg(p - 1);       // not loaded -> stale register, masked by mL in decode
    raw.w[1] = __ldg(p);
    raw.w[2] = __ldg(p + 1);
    raw.w[3] = __ldg(p + 2);
    if (KIND == K_CORE || c.right) raw.w[4] = __ldg(p + 3);
  }

  __device__ __forceinline__ void prefetch(const Cursor& c, const uint32_t* p) const {
    if (c.pf) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
  }

  template <int KIND>
  __device__ __forceinline__ void decode(const Cursor& c, const Raw& raw, uint32_t m, f2 (&P)[8]) const {
    const uint32_t w0 = raw.w[0], w1 = raw.w[1], w2 = raw.w[2], w3 = raw.w[3], w4 = raw.w[4];
    const uint32_t one = 0x3F800000u;
    if (KIND != K_GENERAL) m = kRowMask;                     // immediates: one LOP3 per pixel
    const uint32_t mL = KIND == K_CORE ? kRowMask : (m & c.mL), mR = KIND == K_CORE ? kRowMask : (m & c.mR);
    float v[12];
    if (EXT && ids) {
      // pairs = byte triples: (-2,-1) = bytes 1..3 of w0; (0,1) = bytes 0..2 of w1; (2,3) = byte 3 of w1 + bytes 0..1 of w2;
      // (4,5) = bytes 2..3 of w2 + byte 0 of w3; (6,7) = bytes 1..3 of w3; (8,9) = bytes 0..2 of w4
      v[0] = ids_sample(w0 << 7, w0 >> 13);
      v[1] = ids_sample(w0 >> 1, w0 >> 17);
      v[2] = ids_sample(w1 << 15, w1 >> 5);
      v[3] = ids_sample(w1 << 7, w1 >> 9);
      v[4] = ids_sample(__funnelshift_r(w1, w2, 9), __funnelshift_r(w1, w2, 29));
      v[5] = ids_sample(__funnelshift_r(w1, w2, 17), w2 >> 1);
      v[6] = ids_sample(w2 >> 1, __funnelshift_r(w2, w3, 21));
      v[7] = ids_sample(__funnelshift_r(w2, w3, 9), __funnelshift_r(w2, w3, 25));
      v[8] = ids_sample(w3 << 7, w3 >> 13);
      v[9] = ids_sample(w3 >> 1, w3 >> 17);
      v[10] = ids_sample(w4 << 15, w4 >> 5);
      v[11] = ids_sample(w4 << 7, w4 >> 9);
      if (KIND != K_CORE) {                  // zero samples: rows outside the image, halo columns of the first / last thread column
        const float z = __uint_as_float(one);
        if (mL == 0u) { v[0] = z; v[1] = z; }
        if (mR == 0u) { v[10] = z; v[11] = z; }
        if (m == 0u) {
#pragma unroll
          for (int j = 2; j < 10; ++j) v[j] = z;
        }
      }
    } else {
    v[0] = biased_from_shifted(w0 << 3, mL, one);                      // pixel -2: bits 8..19 of w0
    v[1] = biased_from_shifted(w0 >> 9, mL, one);                      // pixel -1: bits 20..31 of w0
    v[2] = biased_from_shifted(w1 << 11, m, one);                      // pixel 0 : bits 0..11 of w1
    v[3] = biased_from_shifted(w1 >> 1, m, one);                       // pixel 1 : bits 12..23
    v[4] = biased_from_shifted(__funnelshift_r(w1, w2, 13), m, one);   // pixel 2 : bits 24..35 of (w2:w1)
    v[5] = biased_from_shifted(w2 << 7, m, one);                       // pixel 3 : bits 4..15 of w2
    v[6] = biased_from_shifted(w2 >> 5, m, one);                       // pixel 4 : bits 16..27 of w2
    v[7] = biased_from_shifted(__funnelshift_r(w2, w3, 17), m, one);   // pixel 5 : bits 28..39 of (w3:w2)
    v[8] = biased_from_shifted(w3 << 3, m, one);                       // pixel 6 : bits 8..19 of w3
    v[9] = biased_from_shifted(w3 >> 9, m, one);                       // pixel 7 : bits 20..31 of w3
    v[10] = biased_from_shifted(w4 << 11, mR, one);                    // pixel 8
    v[11] = biased_from_shifted(w4 >> 1, mR, one);                     // pixel 9
    }
    if constexpr (CAM16) {
      constexpr float k = 4096.f * kInv4095;         // (b - 1) * 4096 * f32(1/4095), one rounding, then through f16
#pragma unroll
      for (int j = 0; j < 12; j += 2) {
        const __half2 h = __floats2half2_rn(fmaf(v[j], k, -k), fmaf(v[j + 1], k, -k));
        v[j] = __low2float(h);
        v[j + 1] = __high2float(h);
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) P[i] = pk(v[i], v[i + 4]);
  }
};

// per-pixel CFA sample, literal packed.py:23-31 + :98-100 (used by the samplers and border kernels)
template <bool CAM16>
struct Packed12Src {
  FramePtrs fp;
  int pitch;             // bytes per packed row
  int ids = 0;           // 1: IDS layout (packed.py:36-44)
  __device__ __forceinline__ float at(int frame, int r, int c) const {
    const uint8_t* p = fp.in[frame] + (size_t)r * pitch + 3 * (c >> 1);
    const uint32_t b1 = p[1];
    uint32_t v = (c & 1) ? ((uint32_t)p[2] << 4) | (b1 >> 4) : ((b1 & 0xFu) << 8) | p[0];
    if (ids) v = (c & 1) ? (b1 << 4) | ((uint32_t)p[2] >> 4) : ((uint32_t)p[0] << 4) | ((uint32_t)p[2] & 0xFu);
    return round_isp<CAM16>(__fmul_rn((float)v, kInv4095));
  }
};

// ---------------------------------------------------------------- shared front end: sums -> ISP RGB
struct IspConsts {
  int H, W, pattern;
  int ccm;
  float m[9];
  // tone map
  float gamma, intensity, la, ca;
  const float* metrics;      // device, 9 floats
  Workspace* ws;
  int kbase;                 // 0: Malvar-He-Cutler, kBilinearBase: bilinear demosaic (offset into c_taps / c_border)
  int ids;                   // packed layout of the input frames: 0 standard, 1 IDS
  int flip;                  // transform applied inside the call: bit 0 horizontal, bit 1 vertical (rotate_180 = 3) by the store;
                             //    bit 2 transposed, by reinhard_out_transposed_kernel only (the sweep never sees it)
  int orow;                  // elements per OUTPUT row: 3 W for dense frames, more when the frames are tiles of a grid image
  int gate;                  // 1: the sweep runs only on the frames the one-sweep u16 Reinhard map declined (reinhard_map16_declined),
                             //    their max goes to / comes from ws->frame_max2; 0 everywhere else
};

// literal front end for one pixel (bayer.py:137-155 + ISP dtype rounding), used off the hot path
template <bool CAM16>
__device__ __forceinline__ void isp_rgb_pixel(const Packed12Src<CAM16>& src, const IspConsts& k, int frame, int row, int col,
                                              float (&rgb)[3]) {
  float c[3], t[3];
  malvar_pixel(src, frame, k.pattern, row, col, k.H, k.W, c, t, k.kbase);
  float r = __fdiv_rn(c[0], t[0]), g = __fdiv_rn(c[1], t[1]), b = __fdiv_rn(c[2], t[2]);   // in_scale = 1.0
  if (k.ccm) ccm_apply(k.m, r, g, b);
  rgb[0] = round_isp<CAM16>(clamp01(r));
  rgb[1] = round_isp<CAM16>(clamp01(g));
  rgb[2] = round_isp<CAM16>(clamp01(b));
}

// hot-path front end: scaled filter sums (value * scale = x16 sum; biased by 16 for Camera32) -> ISP RGB in [0,1]
// cr/cg/cb are the compile-time SiteScale factors of this pixel; they fold into the constants.
template <bool CAM16, bool CCM>
__device__ __forceinline__ void isp_rgb_fast(const IspConsts& k, float sr, float sg, float sb, float cr, float cg, float cb,
                                             float (&rgb)[3]) {
  float r, g, b;
  if constexpr (CAM16) {
    r = sr * (cr * 0.0625f); g = sg * (cg * 0.0625f); b = sb * (cb * 0.0625f);
  } else {
    constexpr float kn = 256.f * kInv4095;           // 4096 * f32(1/4095) / 16
    r = fmaf(sr, cr * kn, -16.f * kn); g = fmaf(sg, cg * kn, -16.f * kn); b = fmaf(sb, cb * kn, -16.f * kn);
  }
  if constexpr (CCM) {
    const float x = fmaf(b, k.m[2], fmaf(g, k.m[1], r * k.m[0]));
    const float y = fmaf(b, k.m[5], fmaf(g, k.m[4], r * k.m[3]));
    const float z = fmaf(b, k.m[8], fmaf(g, k.m[7], r * k.m[6]));
    r = x; g = y; b = z;
  }
  r = clamp01(r); g = clamp01(g); b = clamp01(b);
  if constexpr (CAM16) {
    const __half2 h = __floats2half2_rn(r, g);
    rgb[0] = __low2float(h); rgb[1] = __high2float(h); rgb[2] = __half2float(__float2half_rn(b));
  } else {
    rgb[0] = r; rgb[1] = g; rgb[2] = b;
  }
}

// ---------------------------------------------------------------- quantisers
// trunc(y * scale) for y in [0, ~1]: one FMA in round-toward-zero mode against 2^23 leaves the integer
// in the low mantissa bits (no F2I); differs from trunc(rn(y*scale)) only when y*scale rounds up to an
// integer within half an ulp, i.e. by at most 1 LSB in ~1e-7 of the cases.
template <typename OutT> struct Quant;
template <> struct Quant<uint8_t> {
  static constexpr int kWords = 6;     // 24 bytes per 8 pixels
  static __device__ __forceinline__ uint32_t q(float y) { return __float_as_uint(__fmaf_rz(y, 255.f, 8388608.f)); }
  static __device__ __forceinline__ void pack(const uint32_t (&v)[24], uint32_t (&w)[6]) {
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const uint32_t lo = __byte_perm(v[4 * i], v[4 * i + 1], 0x0040);
      const uint32_t hi = __byte_perm(v[4 * i + 2], v[4 * i + 3], 0x0040);
      w[i] = __byte_perm(lo, hi, 0x5410);
    }
  }
};
template <> struct Quant<uint16_t> {
  static constexpr int kWords = 12;
  static __device__ __forceinline__ uint32_t q(float y) { return __float_as_uint(__fmaf_rz(y, 65535.f, 8388608.f)); }
  static __device__ __forceinline__ void pack(const uint32_t (&v)[24], uint32_t (&w)[12]) {
#pragma unroll
    for (int i = 0; i < 12; ++i) w[i] = __byte_perm(v[2 * i], v[2 * i + 1], 0x5410);
  }
};
template <> struct Quant<__half> {
  static constexpr int kWords = 12;
  static __device__ __forceinline__ uint32_t q(float y) { return __float_as_uint(y); }
  static __device__ __forceinline__ void pack(const uint32_t (&v)[24], uint32_t (&w)[12]) {
#pragma unroll
    for (int i = 0; i < 12; ++i) {
      const __half2 h = __floats2half2_rn(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
      w[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
  }
};
template <> struct Quant<float> {
  static constexpr int kWords = 24;
  static __device__ __forceinline__ uint32_t q(float y) { return __float_as_uint(y); }
  static __device__ __forceinline__ void pack(const uint32_t (&v)[24], uint32_t (&w)[24]) {
#pragma unroll
    for (int i = 0; i < 24; ++i) w[i] = v[i];
  }
};

// quantised row of 8 pixels -> packed words -> warp-cooperative contiguous store (stream_engine.cuh)
template <typename OutT, bool FULL = false>
__device__ __forceinline__ void store_row8(const WarpCtx& wc, OutT* warp_out /* frame + 24 * tcol0 */, int orow /* elements per output row */,
                                           int row, const uint32_t (&v)[24]) {
  constexpr int NW = Quant<OutT>::kWords;
  uint32_t w[NW];
  Quant<OutT>::pack(v, w);
  warp_store_row<NW, FULL>(wc, warp_out + (size_t)((unsigned)row * (unsigned)orow), w);
}

// The same with the ISP's flip transforms applied in the store (interpolate.py:36-56: flip_vert = row H-1-r, flip_horiz =
// column W-1-c, rotate_180 = both): a flipped row is the row's pixels in reverse order, so the warp's strip lands mirrored
// (lane order reversed in the stage, the lane's eight pixels reversed before packing) -- no extra pass over the image.
// k.flip: bit 0 = horizontal, bit 1 = vertical; kernel-uniform, 0 on the hot path.
// EXT: only the extended instantiations carry the flip code (see Packed12Loader2).
template <typename OutT, bool FULL = false, bool EXT = false>
__device__ __forceinline__ void store_out(const WarpCtx& wc, OutT* warp_out /* frame + 24 * tcol0 */, const IspConsts& k, int row,
                                          const uint32_t (&v)[24]) {
  if (!EXT || k.flip == 0) {
    store_row8<OutT, FULL>(wc, warp_out, k.orow, row, v);
    return;
  }
  const int orow_idx = (k.flip & 2) ? k.H - 1 - row : row;
  if (!(k.flip & 1)) {
    store_row8<OutT, false>(wc, warp_out, k.orow, orow_idx, v);
    return;
  }
  uint32_t r[24];
#pragma unroll
  for (int q = 0; q < 8; ++q) { r[3 * q] = v[3 * (7 - q)]; r[3 * q + 1] = v[3 * (7 - q) + 1]; r[3 * q + 2] = v[3 * (7 - q) + 2]; }
  constexpr int NW = Quant<OutT>::kWords;
  uint32_t w[NW];
  Quant<OutT>::pack(r, w);
  OutT* base = warp_out - 24 * wc.tcol0 + 3 * (k.W - 8 * (wc.tcol0 + wc.nvalid));        // mirrored strip start
  warp_store_row<NW, false>(wc, base + (size_t)((unsigned)orow_idx * (unsigned)k.orow), w, wc.lane < wc.nvalid ? wc.nvalid - 1 - wc.lane : wc.lane);
}

template <typename OutT> __device__ __forceinline__ void store_px(void* frame_out, int W, int row, int col, const float (&y)[3]) {
  OutT* dst = reinterpret_cast<OutT*>(frame_out) + ((size_t)row * W + col) * 3;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    if constexpr (DT<OutT>::is_int) dst[k] = (OutT)(Quant<OutT>::q(y[k]) & (uint32_t)DT<OutT>::scale);
    else dst[k] = cast_from_f32<OutT>(y[k]);
  }
}

// ---------------------------------------------------------------- tone-map stages (per pixel, shared by hot + border)
struct LinearConsts { float a, bmin, inv_gamma; int has_gamma; };

__device__ __forceinline__ LinearConsts linear_consts(const float* __restrict__ metrics, float gamma) {
  LinearConsts c;
  const float bmin = metrics[0], bmax = metrics[1];
  c.a = __fdiv_rn(1.0f, __fsub_rn(bmax, bmin));        // tonemap.py:12
  c.bmin = bmin;
  c.inv_gamma = __fdiv_rn(1.0f, gamma);
  c.has_gamma = gamma != 1.0f;
  return c;
}

// tonemap.py:15-16: clamp(((x - min) * inv_range)^(1/gamma), 0, 1).  The subtraction and the product
// are rounded separately, exactly like the reference expression: saturated pixels (x == max) then hit
// the same side of the truncating quantiser as the reference (an FMA would not).
template <bool GAMMA>
__device__ __forceinline__ void linear_px(const LinearConsts& c, const float (&rgb)[3], float (&y)[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float v = __saturatef(__fmul_rn(__fsub_rn(rgb[k], c.bmin), c.a));
    if constexpr (GAMMA) v = __saturatef(fast_pow(v, c.inv_gamma));
    y[k] = v;
  }
}

struct ReinhardConsts { ReinhardParams p; float b; float out_scale_inv_max; float max_out; float inv_gamma; int has_gamma; int ca0;
                        float kla, kml; /* ki * la, ki * mean * (1 - la): ki * adapt_mean = gray * kla + kml (color_adapt == 0) */ };

template <bool CAM16, bool CA0>
__device__ __forceinline__ void reinhard_p(const ReinhardConsts& c, const float (&rgb)[3], float (&p)[3]) {
  float s[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) s[k] = fmaf(rgb[k], c.p.inv_range, c.b);
  reinhard_map_fast<CA0>(c.p, s, p);
}

// run-time colour-adapt switch (kernel-uniform) for the pair-engine epilogues
template <bool CAM16>
__device__ __forceinline__ void reinhard_p_rt(const ReinhardConsts& c, const float (&rgb)[3], float (&p)[3]) {
  if (c.ca0) reinhard_p<CAM16, true>(c, rgb, p);
  else reinhard_p<CAM16, false>(c, rgb, p);
}

// camera_isp.py:211-218: stored = cast_T(p); out = trunc(scale * (stored / max_out)^(1/gamma))
template <bool CAM16, bool GAMMA>
__device__ __forceinline__ void reinhard_out(const ReinhardConsts& c, const float (&p)[3], float (&y)[3]) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    // the reference does not clamp (q <= 1 + one f16 ulp); saturate for the RZ-FMA quantiser: one FMUL.SAT (NaN -> 0)
    float q = __saturatef(round_isp<CAM16>(p[k]) * c.out_scale_inv_max);
    if constexpr (GAMMA) q = __saturatef(fast_pow(q, c.inv_gamma));
    y[k] = q;
  }
}

// One-sweep Camera32 Reinhard -> u8 (EpiReinhardMax2<false, CA0, STORE>): the map p = s / (adapt + s) is stored as
// trunc(sat(p) * 65535) in a u16 scratch.  That is lossless enough for a u8 result only while every p lies in [0, 1) and the
// frame maximum is not tiny: p >= 1 or inf (a channel far below the metered minimum makes its denominator <= 0; the
// reference takes such a quotient into max_out, camera_isp.py:213) saturates to exactly 1.0, so a stored maximum of 1.0
// means "something may have been clipped"; a maximum below 1/64 would magnify the 2^-17 quantisation step past 1/4 LSB of
// u8 for the gammas the path accepts.  Such frames are declined: the normalise pass skips them and the gated max + write
// sweeps (IspConsts::gate) redo them exactly.  Decided from ws->frame_max alone, so every kernel agrees without a flag.
__device__ __forceinline__ bool reinhard_map16_declined(float mx) { return !(mx < 1.0f && mx >= 0.015625f); }
constexpr float kMap16Scale = 65535.0f;

__device__ __forceinline__ ReinhardConsts reinhard_consts(const IspConsts& k, int frame, bool with_max) {
  ReinhardConsts c;
  c.p = reinhard_params(k.metrics, k.intensity, k.la, k.ca);
  c.b = -c.p.bmin * c.p.inv_range;
  c.ca0 = k.ca == 0.f;
  c.kla = c.p.ki * c.p.la;
  c.kml = c.p.ki * c.p.mean[0] * (1.0f - c.p.la);
  c.inv_gamma = (float)(1.0 / (double)k.gamma);
  c.has_gamma = k.gamma != 1.0f;
  c.out_scale_inv_max = 0.f;
  c.max_out = 1.0f;
  if (with_max) {
    c.max_out = fmaxf(1e-6f, __ldcg(k.gate ? &k.ws->frame_max2[frame] : &k.ws->frame_max[frame]));      // camera_isp.py:190, :213
    c.out_scale_inv_max = __fdiv_rn(1.0f, c.max_out);
  }
  return c;
}

// ================================================================ pair-engine epilogues (stream2.cuh)
// Conventions: pixel q (0..7) of a thread = pair q & 3, lane q >> 2.  "raw" = demosaiced value normalised by 16,
// unclamped, before CCM.  The 2-pixel image frame is renormalised on the raw values (border_fix.cuh):
// whole border rows through the out-of-line frame_patch_nl, the frame COLUMNS of interior rows (pixels 0,1 of
// the first thread column, 6,7 of the last) in line.
__device__ __forceinline__ int edge_bits(int tcol, int W) { return (tcol == 0 ? 1 : 0) | (tcol == (W >> 3) - 1 ? 2 : 0); }

template <bool CAM16, bool BROW, bool GFIRST>
__device__ __forceinline__ void pairs_to_raw(const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4], Vals24& x) {
  using SS = SiteScale2<BROW, GFIRST>;
  constexpr float kn = 256.f * kInv4095;           // 4096 * f32(1/4095) / 16
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float s[3][2];
    upk(R[j], s[0][0], s[0][1]); upk(G[j], s[1][0], s[1][1]); upk(B[j], s[2][0], s[2][1]);
    const float sc[3] = {SS::r(j), SS::g(j), SS::b(j)};
#pragma unroll
    for (int ch = 0; ch < 3; ++ch)
#pragma unroll
      for (int l = 0; l < 2; ++l)
        x.v[3 * (j + 4 * l) + ch] = CAM16 ? s[ch][l] * (sc[ch] * 0.0625f) : fmaf(s[ch][l], sc[ch] * kn, -16.f * kn);
  }
}

// Renormalisation of the frame columns of an interior row on the raw values, exact (division) form: pixels
// 0,1 of the first thread column / 6,7 of the last (edge != 0 only there).
template <bool BROW, bool GFIRST>
__device__ __forceinline__ void patch_cols(Vals24& x, int edge, int kbase) {
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    if (q >= 2 && q < 6) continue;
    if ((q < 2 && (edge & 1)) || (q >= 6 && (edge & 2))) {
      const int K = site_kernel_of(BROW, SiteScale2<BROW, GFIRST>::gsite(q & 3)) + kbase;
      const float* t = c_border.t[K][2][q < 2 ? q : q - 3];
      x.v[3 * q] = frame_exact(x.v[3 * q], t[0]);
      x.v[3 * q + 1] = frame_exact(x.v[3 * q + 1], t[1]);
      x.v[3 * q + 2] = frame_exact(x.v[3 * q + 2], t[2]);
    }
  }
}

// K_GENERAL front end, out of line and rolled (cold code: border tasks): pair sums -> raw values, every pixel
// renormalised by the in-bounds weight sum of its own (row class, column class) -- t = 16, an exact no-op, for
// pixels that are not on the image frame.  brow / gfirst = row type at run time.
struct Pairs12 { f2 R[4], G[4], B[4]; };
template <bool CAM16>
static __device__ __noinline__ Vals24 general_raw(Pairs12 s, int rc, int edge, int brow, int gfirst, int kbase) {
  Vals24 x;
  constexpr float kn = 256.f * kInv4095;
#pragma unroll 1
  for (int j = 0; j < 4; ++j) {
    const bool gsite = ((j & 1) == 0) == (gfirst != 0);
    const float sc[3] = {gsite ? -2.f : (brow ? 4.f : 16.f), gsite ? 16.f : -2.f, gsite ? -2.f : (brow ? 16.f : 4.f)};
    float v[3][2];
    upk(s.R[j], v[0][0], v[0][1]); upk(s.G[j], v[1][0], v[1][1]); upk(s.B[j], v[2][0], v[2][1]);
    const int K = site_kernel_of(brow != 0, gsite) + kbase;
#pragma unroll 1
    for (int l = 0; l < 2; ++l) {
      const int q = j + 4 * l;
      const float* t = c_border.t[K][rc][col_class(q, edge)];
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) {
        const float raw = CAM16 ? v[ch][l] * (sc[ch] * 0.0625f) : fmaf(v[ch][l], sc[ch] * kn, -16.f * kn);
        x.v[3 * q + ch] = frame_exact(raw, t[ch]);
      }
    }
  }
  return x;
}

template <bool CAM16, bool BROW, bool GFIRST, int KIND>
__device__ __forceinline__ void raw_with_frame(const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4], int row, int H, int edge,
                                               int kbase, Vals24& x) {
  if constexpr (KIND == K_GENERAL) {
    Pairs12 s;
#pragma unroll
    for (int j = 0; j < 4; ++j) { s.R[j] = R[j]; s.G[j] = G[j]; s.B[j] = B[j]; }
    x = general_raw<CAM16>(s, edge_class(row, H), edge, BROW, GFIRST, kbase);
  } else {
    pairs_to_raw<CAM16, BROW, GFIRST>(R, G, B, x);
    if (KIND == K_EDGE && edge) patch_cols<BROW, GFIRST>(x, edge, kbase);
  }
}

// raw -> ISP RGB in [0,1]: CCM, clamp (bayer.py:152-155), rounding through the ISP dtype
template <bool CAM16>
__device__ __forceinline__ void raw_to_rgb(const IspConsts& k, const float* x, float (&rgb)[3]) {
  // The matrix is applied unconditionally: without colour correction the host passes the identity, for which
  // fma(b, 0, fma(g, 0, r * 1)) == r exactly -- one code copy, no branch.
  const float u = fmaf(x[2], k.m[2], fmaf(x[1], k.m[1], x[0] * k.m[0]));
  const float v = fmaf(x[2], k.m[5], fmaf(x[1], k.m[4], x[0] * k.m[3]));
  const float w = fmaf(x[2], k.m[8], fmaf(x[1], k.m[7], x[0] * k.m[6]));
  float r = u, g = v, b = w;
  r = clamp01(r); g = clamp01(g); b = clamp01(b);
  if constexpr (CAM16) {
    const __half2 h = __floats2half2_rn(r, g);
    rgb[0] = __low2float(h); rgb[1] = __high2float(h); rgb[2] = __half2float(__float2half_rn(b));
  } else {
    rgb[0] = r; rgb[1] = g; rgb[2] = b;
  }
}

// ---------------------------------------------------------------- packed (pair) form of the generic stages
// raw pairs: demosaiced value normalised by 16 (unclamped, before CCM) of pixel pair j (pixels j, j+4), channel c
template <bool CAM16, bool BROW, bool GFIRST>
__device__ __forceinline__ void pairs_to_raw2(const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4], f2 (&X)[4][3]) {
  using SS = SiteScale2<BROW, GFIRST>;
  constexpr float kn = 256.f * kInv4095;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if constexpr (CAM16) {
      X[j][0] = mul2(R[j], bc(SS::r(j) * 0.0625f)); X[j][1] = mul2(G[j], bc(SS::g(j) * 0.0625f)); X[j][2] = mul2(B[j], bc(SS::b(j) * 0.0625f));
    } else {
      X[j][0] = fma2k(SS::r(j) * kn, R[j], bc(-16.f * kn)); X[j][1] = fma2k(SS::g(j) * kn, G[j], bc(-16.f * kn));
      X[j][2] = fma2k(SS::b(j) * kn, B[j], bc(-16.f * kn));
    }
  }
}

// Camera32 without colour matrix, no frame column in this lane: demosaiced value and the clamp of bayer.py:152-155 as ONE
// saturating scalar FMA per value (same product, same addend, same single rounding as the packed FMA of pairs_to_raw2, then
// the clamp) -- two issue slots per value pair instead of three (packed FMA + two saturating moves)
template <bool BROW, bool GFIRST>
__device__ __forceinline__ void pairs_to_rgb2_sat(const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4], f2 (&rgb)[4][3]) {
  using SS = SiteScale2<BROW, GFIRST>;
  constexpr float kn = 256.f * kInv4095;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const f2 in[3] = {R[j], G[j], B[j]};
    const float sc[3] = {SS::r(j) * kn, SS::g(j) * kn, SS::b(j) * kn};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float lo, hi;
      upk(in[c], lo, hi);
      rgb[j][c] = pk(__saturatef(__fmaf_rn(sc[c], lo, -16.f * kn)), __saturatef(__fmaf_rn(sc[c], hi, -16.f * kn)));
    }
  }
}

// frame columns of an interior row on the raw pairs, exact (division) form; edge != 0 only in the first / last thread column
template <bool BROW, bool GFIRST>
__device__ __forceinline__ void patch_cols_pairs(f2 (&X)[4][3], int edge, int kbase) {
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    if (q >= 2 && q < 6) continue;
    if ((q < 2 && (edge & 1)) || (q >= 6 && (edge & 2))) {
      const int K = site_kernel_of(BROW, SiteScale2<BROW, GFIRST>::gsite(q & 3)) + kbase;
      const float* t = c_border.t[K][2][q < 2 ? q : q - 3];
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) {
        float lo, hi;
        upk(X[q & 3][ch], lo, hi);
        if (q < 4) lo = frame_exact(lo, t[ch]); else hi = frame_exact(hi, t[ch]);
        X[q & 3][ch] = pk(lo, hi);
      }
    }
  }
}

// raw pair -> ISP RGB pair in [0,1]: CCM (kernel-uniform run-time flag), clamp (bayer.py:152-155), ISP dtype rounding
// colour matrix on the four pixel pairs of a row under ONE kernel-uniform branch (inside raw2_to_rgb2 it is taken once per
// pair: 0.5 BRA per pixel in the Reinhard sweeps); callers then use raw2_to_rgb2<CAM16, false>
__device__ __forceinline__ void ccm2_row(const IspConsts& k, f2 (&X)[4][3]) {
  if (k.ccm) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const f2 x0 = X[j][0], x1 = X[j][1], x2 = X[j][2];
#pragma unroll
      for (int c = 0; c < 3; ++c)
        X[j][c] = fma2(x2, bc(k.m[3 * c + 2]), fma2(x1, bc(k.m[3 * c + 1]), mul2(x0, bc(k.m[3 * c]))));
    }
  }
}

template <bool CAM16, bool DO_CCM = true>
__device__ __forceinline__ void raw2_to_rgb2(const IspConsts& k, const f2 (&x)[3], f2 (&rgb)[3]) {
  f2 y[3] = {x[0], x[1], x[2]};
  if (DO_CCM && k.ccm) {
#pragma unroll
    for (int c = 0; c < 3; ++c)
      y[c] = fma2(x[2], bc(k.m[3 * c + 2]), fma2(x[1], bc(k.m[3 * c + 1]), mul2(x[0], bc(k.m[3 * c]))));
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float lo, hi;
    upk(y[c], lo, hi);
    lo = clamp01(lo); hi = clamp01(hi);
    if constexpr (CAM16) {
      const __half2 h = __floats2half2_rn(lo, hi);
      lo = __low2float(h); hi = __high2float(h);
    }
    rgb[c] = pk(lo, hi);
  }
}

// ISP RGB pairs of a row for the packed Reinhard epilogues: the lean form (pairs_to_rgb2_sat) where it applies, else raw
// pairs -> frame columns -> colour matrix -> clamp / ISP rounding
template <bool CAM16, bool BROW, bool GFIRST, int KIND>
__device__ __forceinline__ void row_rgb2(const IspConsts& k, int edge, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4], f2 (&rgb)[4][3]) {
  bool lean = false;
  if constexpr (!CAM16) lean = !k.ccm && !(KIND == K_EDGE && edge);
  if (lean) {
    if constexpr (!CAM16) pairs_to_rgb2_sat<BROW, GFIRST>(R, G, B, rgb);
  } else {
    f2 X[4][3];
    pairs_to_raw2<CAM16, BROW, GFIRST>(R, G, B, X);
    if (KIND == K_EDGE && edge) patch_cols_pairs<BROW, GFIRST>(X, edge, k.kbase);
    ccm2_row(k, X);
#pragma unroll
    for (int j = 0; j < 4; ++j) raw2_to_rgb2<CAM16, false>(k, X[j], rgb[j]);
  }
}

// camera_isp.py:200-210 for a pixel pair, color_adapt == 0 (one adaptation level per pixel): p = s / (adapt + s).
// MUFU diet (profiles/r01_reinhard_sweep_ncu.txt: the sweep was MUFU-bound at 11 MUFU per pixel):
//  * s = (x - min) * (1 / range) with the subtraction rounded on its own (exact near x == min, where a folded
//    FMA loses all relative accuracy and gamma > 1 amplifies it: r02_error_histogram, 16 LSB of u16 before);
//  * ONE reciprocal per pixel instead of three: with d_c = adapt + s_c,  p_c = s_c * (d_x * d_y) / (d_r * d_g * d_b),
//    five packed multiplies more, two MUFU less; `post` scales the denominator (the write sweep passes max_out, so
//    the normalisation p / max_out costs no instruction of its own).
__device__ __forceinline__ void reinhard_s2(const ReinhardConsts& c, const f2 (&rgb)[3], f2 (&s)[3]) {
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) s[ch] = mul2(add2(rgb[ch], bc(-c.p.bmin)), bc(c.p.inv_range));
}

__device__ __forceinline__ f2 reinhard_adapt2(const ReinhardConsts& c, const f2 (&s)[3]) {
  const f2 gray = fma2(s[2], bc(0.114f), fma2(s[1], bc(0.587f), mul2(s[0], bc(0.299f))));
  float tl, th;
  upk(fma2(gray, bc(c.kla), bc(c.kml)), tl, th);                  // ki * lerp(la, mean, gray)
  return pk(fast_pow(tl, c.p.map_key), fast_pow(th, c.p.map_key));
}

// numerators n_c and the shared reciprocal r:  p_c / post = n_c * r
__device__ __forceinline__ void reinhard_nr2(const ReinhardConsts& c, const f2 (&rgb)[3], f2 post, f2 (&n)[3], f2& r) {
  f2 s[3];
  reinhard_s2(c, rgb, s);
  const f2 adapt = reinhard_adapt2(c, s);
  const f2 dr = add2(adapt, s[0]), dg = add2(adapt, s[1]), db = add2(adapt, s[2]);
  const f2 gb = mul2(dg, db);
  n[0] = mul2(s[0], gb);
  n[1] = mul2(s[1], mul2(dr, db));
  n[2] = mul2(s[2], mul2(dr, dg));
  float pl, ph;
  upk(mul2(mul2(dr, post), gb), pl, ph);
  r = pk(fast_rcp(pl), fast_rcp(ph));
}

template <bool CAM16>
__device__ __forceinline__ void reinhard_p2(const ReinhardConsts& c, const f2 (&rgb)[3], f2 (&p)[3]) {
  f2 n[3], r;
  reinhard_nr2(c, rgb, bc(1.0f), n, r);
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) p[ch] = mul2(n[ch], r);
}

// max over the three channels of p for a pixel pair: p = s / (adapt + s) is increasing in s_c as long as every
// denominator is positive, so the largest channel carries it -- one reciprocal and no per-channel quotient (the max
// sweep only needs the frame maximum).  A channel far BELOW the metered minimum (s_c < -adapt; possible because the
// bounds come from the strided samples only) makes its denominator negative and its quotient large and positive --
// the reference takes that value into max_out too (camera_isp.py:213).  dmin tracks the smallest denominator; the
// caller re-evaluates the row exactly when it ever is negative (cold path).
__device__ __forceinline__ f2 reinhard_pmax2(const ReinhardConsts& c, const f2 (&rgb)[3], float& dmin) {
  f2 s[3];
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) s[ch] = fma2(rgb[ch], bc(c.p.inv_range), bc(c.b));
  const f2 adapt = reinhard_adapt2(c, s);
  float l[3], h[3];
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) upk(s[ch], l[ch], h[ch]);
  const f2 sm = pk(fmaxf(l[0], fmaxf(l[1], l[2])), fmaxf(h[0], fmaxf(h[1], h[2])));
  const f2 sn = pk(fminf(l[0], fminf(l[1], l[2])), fminf(h[0], fminf(h[1], h[2])));
  float dl, dh, el, eh;
  upk(add2(adapt, sm), dl, dh);
  upk(add2(adapt, sn), el, eh);
  dmin = fminf(dmin, fminf(el, eh));
  return mul2(sm, pk(fast_rcp(dl), fast_rcp(dh)));
}

template <bool CAM16, typename OutT, bool EXT = false>
struct EpiRgb2 {      // load_packed12: ISP-dtype float RGB out
  FramePtrs fp;
  IspConsts k;
  static constexpr int kStageWords = 32 * Quant<OutT>::kWords;
  struct State { OutT* out; WarpCtx wc; int edge; };
  __device__ __forceinline__ void init(State& st, int frame, int tcol, const WarpCtx& wc) const {
    st.out = reinterpret_cast<OutT*>(fp.out[frame]) + 24 * wc.tcol0;
    st.wc = wc;
    st.edge = edge_bits(tcol, k.W);
  }
  __device__ __forceinline__ void finish(State&, int, int, bool) const {}
  static constexpr bool kSplitEdge = false;
  static constexpr bool kCompactLoop = false;
  __device__ __forceinline__ bool fast_kinds_ok(const State&) const { return true; }
  template <bool BROW, bool GFIRST, int KIND>
  __device__ __forceinline__ void emit(State& st, int row, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4]) const {
    Vals24 x;
    raw_with_frame<CAM16, BROW, GFIRST, KIND>(R, G, B, row, k.H, st.edge, k.kbase, x);
    uint32_t v[24];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float rgb[3];
      raw_to_rgb<CAM16>(k, &x.v[3 * q], rgb);
      v[3 * q] = __float_as_uint(rgb[0]); v[3 * q + 1] = __float_as_uint(rgb[1]); v[3 * q + 2] = __float_as_uint(rgb[2]);
    }
    store_out<OutT, false, EXT>(st.wc, st.out, k, row, v);
  }
};

// FAST: Camera32, no CCM, gamma 1 -- the configuration the roofline is quoted on; everything stays in pairs.
template <bool CAM16, typename OutT, bool FAST, bool EXT = false>
struct EpiLinear2 {
  static_assert(!(FAST && CAM16), "the packed fast path is Camera32 only");
  FramePtrs fp;
  IspConsts k;
  static constexpr int kStageWords = 32 * Quant<OutT>::kWords;
  struct State { LinearConsts c; OutT* out; WarpCtx wc; int edge; bool inside; };
  __device__ __forceinline__ void init(State& st, int frame, int tcol, const WarpCtx& wc) const {
    st.c = linear_consts(k.metrics, k.gamma);
    st.out = reinterpret_cast<OutT*>(fp.out[frame]) + 24 * wc.tcol0;
    st.wc = wc;
    st.edge = edge_bits(tcol, k.W);
    // With bounds inside [0,1] (always true for metered bounds: the metered images are clamped to [0,1],
    // bayer.py:155)  clamp((clamp(c,0,1) - min) * inv, 0, 1) == clamp((c - min) * inv, 0, 1), so the demosaic
    // clamp needs no instruction of its own.  Other bounds take the generic row routine.
    st.inside = st.c.bmin >= 0.f && k.metrics[1] <= 1.0f;
  }
  __device__ __forceinline__ void finish(State&, int, int, bool) const {}

  static constexpr bool kSplitEdge = FAST;
  // single-step loop (stream2_rows), measured on cfg2 against the 3x unrolled one: kernel alone 169 vs 171 us, step
  // (sweep || metering) 197 vs 204 us
  static constexpr bool kCompactLoop = true;
  template <bool GAMMA>
  __device__ __forceinline__ void emit_t(const State& st, int row, const Vals24& x) const {
    uint32_t v[24];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float rgb[3], y[3];
      raw_to_rgb<CAM16>(k, &x.v[3 * q], rgb);
      linear_px<GAMMA>(st.c, rgb, y);
      v[3 * q] = Quant<OutT>::q(y[0]); v[3 * q + 1] = Quant<OutT>::q(y[1]); v[3 * q + 2] = Quant<OutT>::q(y[2]);
    }
    store_out<OutT, false, EXT>(st.wc, st.out, k, row, v);
  }
  template <bool BROW, bool GFIRST, int KIND>
  __device__ __forceinline__ void emit_generic(const State& st, int row, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4]) const {
    Vals24 x;
    raw_with_frame<CAM16, BROW, GFIRST, KIND>(R, G, B, row, k.H, st.edge, k.kbase, x);
    if (st.c.has_gamma) emit_t<true>(st, row, x);
    else emit_t<false>(st, row, x);
  }

  // the packed kinds need bounds inside [0,1]; otherwise every task takes K_GENERAL (generic arithmetic)
  __device__ __forceinline__ bool fast_kinds_ok(const State& st) const { return !FAST || st.inside; }

  template <bool BROW, bool GFIRST, int KIND>
  __device__ __forceinline__ void emit(State& st, int row, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4]) const {
    if constexpr (!FAST || KIND == K_GENERAL) {
      emit_generic<BROW, GFIRST, KIND>(st, row, R, G, B);
    } else {
      using SS = SiteScale2<BROW, GFIRST>;
      constexpr float kn = 256.f * kInv4095;             // 4096 * f32(1/4095) / 16
      f2 X[4][3];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        X[j][0] = fma2k(SS::r(j) * kn, R[j], bc(-16.f * kn));      // demosaiced value (unclamped)
        X[j][1] = fma2k(SS::g(j) * kn, G[j], bc(-16.f * kn));
        X[j][2] = fma2k(SS::b(j) * kn, B[j], bc(-16.f * kn));
      }
      if (KIND == K_EDGE && st.edge) {       // frame columns: only the lanes of the first / last thread column
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          if (q >= 2 && q < 6) continue;
          if ((q < 2 && (st.edge & 1)) || (q >= 6 && (st.edge & 2))) {
            const int K = site_kernel_of(BROW, SS::gsite(q & 3)) + k.kbase;
            const float* f = c_border.f[K][2][q < 2 ? q : q - 3];
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
              float lo, hi;
              upk(X[q & 3][ch], lo, hi);
              if (q < 4) lo *= f[ch]; else hi *= f[ch];
              X[q & 3][ch] = pk(lo, hi);
            }
          }
        }
      }
      const f2 nbmin = bc(-st.c.bmin);
      const float a = st.c.a;
      uint32_t v[24];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          float lo, hi;
          upk(add2(X[j][ch], nbmin), lo, hi);                       // tonemap.py:15  (x - min) ...
          lo = __saturatef(__fmul_rn(lo, a));                       //                ... * inv, clamp
          hi = __saturatef(__fmul_rn(hi, a));
          if constexpr (DT<OutT>::is_int) {
            float qlo, qhi;
            upk(fma2_rz(pk(lo, hi), bc(DT<OutT>::scale), bc(8388608.f)), qlo, qhi);
            v[3 * j + ch] = __float_as_uint(qlo);
            v[3 * (j + 4) + ch] = __float_as_uint(qhi);
          } else {
            v[3 * j + ch] = __float_as_uint(lo);
            v[3 * (j + 4) + ch] = __float_as_uint(hi);
          }
        }
      }
      store_out<OutT, KIND == K_CORE, EXT>(st.wc, st.out, k, row, v);
    }
  }
};

// CA0 (color_adapt == 0) and GAMMA (gamma != 1) are host-known: separate instantiations keep each kernel's code small
// (the sweep is instruction-cache sensitive, see stream2.cuh)
// STORE (Camera16 only): also write the un-normalised map p, rounded through f16 exactly like the reference's in-place
// write-back (camera_isp.py:211), to a scratch image -- the second pass then only normalises and quantises that
// scratch (reinhard_scratch_out_kernel) instead of sweeping the packed frames again.
template <bool CAM16, bool CA0, bool STORE = false, bool GATED = false>
struct EpiReinhardMax2 {      // pass 1: frame-global max of the mapped values (+ the map itself when STORE)
  FramePtrs fp;               // .out = scratch images (STORE only)
  IspConsts k;
  // STORE: Camera16 writes the f16 map the reference stores back (exact); Camera32 writes a u16 fixed-point map that is
  // accurate enough for u8 outputs only (reinhard_map16_declined)
  using ScratchT = std::conditional_t<CAM16, __half, uint16_t>;
  static_assert(!(STORE && GATED), "the gated instantiation is the plain max sweep of the fallback");
  static constexpr bool kGated = GATED;
  static constexpr int kStageWords = STORE ? 32 * Quant<ScratchT>::kWords : 0;
  struct State { ReinhardConsts c; float mx; int edge; ScratchT* out; WarpCtx wc; };
  __device__ __forceinline__ bool enabled(int frame) const { return reinhard_map16_declined(__ldcg(&k.ws->frame_max[frame])); }
  __device__ __forceinline__ void init(State& st, int frame, int tcol, const WarpCtx& wc) const {
    st.c = reinhard_consts(k, frame, false);
    st.mx = 0.f;
    st.edge = edge_bits(tcol, k.W);
    st.wc = wc;
    st.out = STORE ? reinterpret_cast<ScratchT*>(fp.out[frame]) + 24 * wc.tcol0 : nullptr;
  }
  static constexpr bool kSplitEdge = false;     // measured: a separate K_CORE copy costs more (instruction cache) than its leaner code saves
  static constexpr bool kCompactLoop = true;
  __device__ __forceinline__ bool fast_kinds_ok(const State&) const { return true; }
  __device__ __forceinline__ void emit_t(State& st, int row, const Vals24& x) const {
    float mx = st.mx;
    uint32_t v[24];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float rgb[3], p[3];
      raw_to_rgb<CAM16>(k, &x.v[3 * q], rgb);
      reinhard_p<CAM16, CA0>(st.c, rgb, p);
      if constexpr (STORE && !CAM16) {
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          p[ch] = __saturatef(p[ch]);                   // NaN / negative -> 0, >= 1 -> 1.0 (declines the frame)
          v[3 * q + ch] = __float_as_uint(__fmaf_rz(p[ch], kMap16Scale, 8388608.f));
        }
        mx = fmaxf(mx, fmaxf(p[0], fmaxf(p[1], p[2])));
      } else {
        mx = fmaxf(mx, fmaxf(p[0], fmaxf(p[1], p[2])));
        v[3 * q] = __float_as_uint(p[0]); v[3 * q + 1] = __float_as_uint(p[1]); v[3 * q + 2] = __float_as_uint(p[2]);
      }
    }
    st.mx = mx;
    if constexpr (STORE) store_row8<ScratchT>(st.wc, st.out, k.W * 3, row, v);
  }
  template <bool BROW, bool GFIRST, int KIND>
  __device__ __forceinline__ void emit(State& st, int row, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4]) const {
    if constexpr (KIND != K_GENERAL && CA0) {        // packed path
      f2 P[4][3];
      row_rgb2<CAM16, BROW, GFIRST, KIND>(k, st.edge, R, G, B, P);
      float mx = st.mx;
      if constexpr (STORE && CAM16) {
        uint32_t v[24];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          f2 p[3];
          reinhard_p2<CAM16>(st.c, P[j], p);
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) {
            float lo, hi;
            upk(p[ch], lo, hi);
            mx = fmaxf(mx, fmaxf(lo, hi));
            v[3 * j + ch] = __float_as_uint(lo);
            v[3 * (j + 4) + ch] = __float_as_uint(hi);
          }
        }
        store_row8<__half>(st.wc, st.out, k.W * 3, row, v);
      } else if constexpr (STORE) {
        // Camera32: u16 fixed point.  The saturating product is the quotient itself (p = n * r), one FMUL.SAT per value;
        // the quantiser is the packed RZ-FMA against 2^23 of the integer outputs.
        uint32_t v[24];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          f2 n[3], r;
          reinhard_nr2(st.c, P[j], bc(1.0f), n, r);
          float rl, rh;
          upk(r, rl, rh);
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) {
            float lo, hi, ql, qh;
            upk(n[ch], lo, hi);
            lo = __saturatef(lo * rl);
            hi = __saturatef(hi * rh);
            mx = fmaxf(mx, fmaxf(lo, hi));
            upk(fma2_rz(pk(lo, hi), bc(kMap16Scale), bc(8388608.f)), ql, qh);
            v[3 * j + ch] = __float_as_uint(ql);
            v[3 * (j + 4) + ch] = __float_as_uint(qh);
          }
        }
        store_row8<uint16_t, KIND == K_CORE>(st.wc, st.out, k.W * 3, row, v);
      } else {
        float dmin = 0.f;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float lo, hi;
          upk(reinhard_pmax2(st.c, P[j], dmin), lo, hi);
          mx = fmaxf(mx, fmaxf(lo, hi));
        }
        if (dmin < 0.f) {                      // some channel's denominator is negative: all three quotients, exactly
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            f2 p[3];
            reinhard_p2<CAM16>(st.c, P[j], p);
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) mx = fmaxf(mx, fmaxf(lo_of(p[ch]), hi_of(p[ch])));
          }
        }
      }
      st.mx = mx;
    } else {
      Vals24 x;
      raw_with_frame<CAM16, BROW, GFIRST, KIND>(R, G, B, row, k.H, st.edge, k.kbase, x);
      emit_t(st, row, x);
    }
  }
  __device__ __forceinline__ void finish(State& st, int frame, int lane, bool task_ok) const {
    const float m = warp_max(st.mx);
    if (lane == 0 && task_ok && m > 0.f)
      atomicMax(reinterpret_cast<unsigned int*>(GATED ? &k.ws->frame_max2[frame] : &k.ws->frame_max[frame]),
                __float_as_uint(m));
  }
};

template <bool CAM16, typename OutT, bool CA0, bool GAMMA, bool EXT = false, bool GATED = false>
struct EpiReinhard2 {         // pass 2 recomputed from the packed frame: map, normalise by the max, gamma, quantise
  FramePtrs fp;
  IspConsts k;                // GATED (k.gate == 1): only the frames the one-sweep u16 map declined, max from ws->frame_max2
  static constexpr bool kGated = GATED;
  __device__ __forceinline__ bool enabled(int frame) const { return reinhard_map16_declined(__ldcg(&k.ws->frame_max[frame])); }
  static constexpr int kStageWords = 32 * Quant<OutT>::kWords;
  struct State { ReinhardConsts c; OutT* out; WarpCtx wc; int edge; };
  __device__ __forceinline__ void init(State& st, int frame, int tcol, const WarpCtx& wc) const {
    st.c = reinhard_consts(k, frame, true);
    st.out = reinterpret_cast<OutT*>(fp.out[frame]) + 24 * wc.tcol0;
    st.wc = wc;
    st.edge = edge_bits(tcol, k.W);
  }
  __device__ __forceinline__ void finish(State&, int, int, bool) const {}
  static constexpr bool kSplitEdge = false;     // measured: a separate K_CORE copy costs more (instruction cache) than its leaner code saves
  static constexpr bool kCompactLoop = true;
  __device__ __forceinline__ void emit_t(const State& st, int row, const Vals24& x) const {
    uint32_t v[24];
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      float rgb[3], p[3], y[3];
      raw_to_rgb<CAM16>(k, &x.v[3 * q], rgb);
      reinhard_p<CAM16, CA0>(st.c, rgb, p);
      reinhard_out<CAM16, GAMMA>(st.c, p, y);
      v[3 * q] = Quant<OutT>::q(y[0]); v[3 * q + 1] = Quant<OutT>::q(y[1]); v[3 * q + 2] = Quant<OutT>::q(y[2]);
    }
    store_out<OutT, false, EXT>(st.wc, st.out, k, row, v);
  }
  __device__ __forceinline__ bool fast_kinds_ok(const State&) const { return true; }
  // packed path: color_adapt == 0, any gamma (kernel-uniform)
  template <bool BROW, bool GFIRST, int KIND>
  __device__ __forceinline__ void emit_pairs(const State& st, int row, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4]) const {
    f2 P[4][3];
    row_rgb2<CAM16, BROW, GFIRST, KIND>(k, st.edge, R, G, B, P);
    uint32_t v[24];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      f2 n[3], r;
      // Camera32: q = p / max_out straight from the shared reciprocal; Camera16: p is rounded through f16 first
      reinhard_nr2(st.c, P[j], bc(CAM16 ? 1.0f : st.c.max_out), n, r);
      float rl, rh;
      upk(r, rl, rh);
#pragma unroll
      for (int ch = 0; ch < 3; ++ch) {                 // camera_isp.py:211-218
        float lo, hi;
        upk(n[ch], lo, hi);
        if constexpr (CAM16) {
          const __half2 h = __floats2half2_rn(lo * rl, hi * rh);
          lo = __saturatef(__low2float(h) * st.c.out_scale_inv_max);
          hi = __saturatef(__high2float(h) * st.c.out_scale_inv_max);
        } else {
          lo = __saturatef(lo * rl);                   // the reference does not clamp; NaN / negative -> 0 (SURVEY H8)
          hi = __saturatef(hi * rh);
        }
        if constexpr (GAMMA) { lo = fast_pow(lo, st.c.inv_gamma); hi = fast_pow(hi, st.c.inv_gamma); }
        if constexpr (DT<OutT>::is_int) {
          float ql, qh;
          upk(fma2_rz(pk(lo, hi), bc(DT<OutT>::scale), bc(8388608.f)), ql, qh);
          v[3 * j + ch] = __float_as_uint(ql);
          v[3 * (j + 4) + ch] = __float_as_uint(qh);
        } else {
          v[3 * j + ch] = __float_as_uint(lo);
          v[3 * (j + 4) + ch] = __float_as_uint(hi);
        }
      }
    }
    store_out<OutT, KIND == K_CORE, EXT>(st.wc, st.out, k, row, v);
  }

  template <bool BROW, bool GFIRST, int KIND>
  __device__ __forceinline__ void emit(State& st, int row, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4]) const {
    if constexpr (KIND != K_GENERAL && CA0) {
      emit_pairs<BROW, GFIRST, KIND>(st, row, R, G, B);
    } else {
      Vals24 x;
      raw_with_frame<CAM16, BROW, GFIRST, KIND>(R, G, B, row, k.H, st.edge, k.kbase, x);
      emit_t(st, row, x);
    }
  }
};

enum { MODE_RGB = 0, MODE_LINEAR = 1, MODE_RMAX = 2, MODE_REINHARD = 3 };

// ---------------------------------------------------------------- metering samplers straight from packed12
// generic: any stride, literal per-pixel demosaic
template <bool CAM16>
struct Packed12Sampler {
  Packed12Src<CAM16> src;
  IspConsts k;
  int stride, hs, ws_;
  __device__ __forceinline__ void sample(long long idx, float (&rgb)[3]) const {
    const int j = (int)(idx % ws_);
    const long long q = idx / ws_;
    const int i = (int)(q % hs);
    const int f = (int)(q / hs);
    isp_rgb_pixel<CAM16>(src, k, f, i * stride, j * stride, rgb);
  }
};

// stride % 8 == 0 (the default 8): a sample is pixel 0 of thread column col/8 of the streaming kernel.
// It reads nine 32-bit words (1/2/3/2/1 over the five rows; consecutive samples of a row are 12 bytes
// apart, so a warp's loads are contiguous) and evaluates exactly the partial-sum formulas of the sweep,
// i.e. the very value the sweep will produce for that pixel -- including the samples on the 2-pixel image
// frame (row 0 / column 0), which use the same zero-sample + renormalisation scheme (border_fix.cuh).
template <bool CAM16>
struct Packed12FastSampler {
  Packed12Src<CAM16> src;
  IspConsts k;
  int stride, hs, ws_;
  int pitch_words;

  static constexpr bool kRowStructured = true;

  static __device__ __forceinline__ float dec(uint32_t shifted) {
    const float b = biased_from_shifted(shifted, 0x007FF800u, 0x3F800000u);       // 1 + v/4096, one LOP3
    if constexpr (CAM16) {
      constexpr float kk = 4096.f * kInv4095;
      return __half2float(__float2half_rn(fmaf(b, kk, -kk)));
    } else {
      return b;
    }
  }

  static __device__ __forceinline__ float idec(uint32_t a, uint32_t b) {      // IDS layout, see ids_sample
    const float v = ids_sample(a, b);
    if constexpr (CAM16) {
      constexpr float kk = 4096.f * kInv4095;
      return __half2float(__float2half_rn(fmaf(v, kk, -kk)));
    } else {
      return v;
    }
  }

  // the nine words of a sample -> scaled filter sums S (S * sc = x16 sum) of the three channels
  __device__ __forceinline__ void sums_from_words(uint32_t a0, uint32_t bm, uint32_t b0, uint32_t cm, uint32_t c0, uint32_t c1,
                                                  uint32_t dm, uint32_t d0, uint32_t e0, int row, float (&S)[3], float (&sc)[3],
                                                  bool& brow, bool& gsite) const {
    // pixel col-2 = bits 8..19 of word -1, col-1 = bits 20..31; col = bits 0..11 of word 0, col+1 = bits 12..23,
    // col+2 = bits 24..35 of (word 1 : word 0)
    float C, EW, EEWW, NS, D, NNSS;
    if (src.ids) {
      // IDS layout: pixel col = first sample of the triple in bytes 0..2 of the word, col+1 its second; col-2 / col-1 = the
      // triple in bytes 1..3 of the previous word; col+2 = first sample of the triple that starts in byte 3
      C = idec(c0 << 15, c0 >> 5);
      EW = idec(cm >> 1, cm >> 17) + idec(c0 << 7, c0 >> 9);
      EEWW = idec(cm << 7, cm >> 13) + idec(__funnelshift_r(c0, c1, 9), __funnelshift_r(c0, c1, 29));
      NS = idec(b0 << 15, b0 >> 5) + idec(d0 << 15, d0 >> 5);
      D = (idec(bm >> 1, bm >> 17) + idec(dm >> 1, dm >> 17)) + (idec(b0 << 7, b0 >> 9) + idec(d0 << 7, d0 >> 9));
      NNSS = idec(a0 << 15, a0 >> 5) + idec(e0 << 15, e0 >> 5);
    } else {
      C = dec(c0 << 11);
      EW = dec(cm >> 9) + dec(c0 >> 1);
      EEWW = dec(cm << 3) + dec(__funnelshift_r(c0, c1, 13));
      NS = dec(b0 << 11) + dec(d0 << 11);
      D = (dec(bm >> 9) + dec(dm >> 9)) + (dec(b0 >> 1) + dec(d0 >> 1));
      NNSS = dec(a0 << 11) + dec(e0 << 11);
    }
    const bool brow0 = (k.pattern == B200ISP_GBRG || k.pattern == B200ISP_BGGR);
    const bool gfirst0 = (k.pattern == B200ISP_GRBG || k.pattern == B200ISP_GBRG);
    brow = brow0 != ((row & 1) != 0);
    gsite = gfirst0 != ((row & 1) != 0);
    if (!gsite) {
      float g2, opp4;
      if (k.kbase) { g2 = 2.f * (NS + EW); opp4 = D; }              // bilinear (kernel-uniform): same scales, see bilinear_row2
      else malvar_csite(C, NS, EW, NNSS, EEWW, D, g2, opp4);
      S[1] = g2; sc[1] = 2.f;
      S[0] = brow ? opp4 : C; sc[0] = brow ? 4.f : 16.f;
      S[2] = brow ? C : opp4; sc[2] = brow ? 16.f : 4.f;
    } else {
      float h2, v2;
      if (k.kbase) { h2 = 4.f * EW; v2 = 4.f * NS; }
      else malvar_gsite(C, NS, EW, NNSS, EEWW, D, h2, v2);
      S[1] = C; sc[1] = 16.f;
      S[0] = brow ? v2 : h2; sc[0] = 2.f;
      S[2] = brow ? h2 : v2; sc[2] = 2.f;
    }
  }

  // interior sample: p = word of pixel (row, col) (col % 8 == 0)
  __device__ __forceinline__ void sample_fast(const uint32_t* p, int row, float (&rgb)[3]) const {
    const uint32_t a0 = __ldg(p - 2 * pitch_words);                                   // row-2: col
    const uint32_t bm = __ldg(p - pitch_words - 1), b0 = __ldg(p - pitch_words);      // row-1: col-1..col+1
    const uint32_t cm = __ldg(p - 1), c0 = __ldg(p), c1 = __ldg(p + 1);               // row  : col-2..col+2
    const uint32_t dm = __ldg(p + pitch_words - 1), d0 = __ldg(p + pitch_words);      // row+1
    const uint32_t e0 = __ldg(p + 2 * pitch_words);                                   // row+2
    float S[3], sc[3];
    bool brow, gsite;
    sums_from_words(a0, bm, b0, cm, c0, c1, dm, d0, e0, row, S, sc, brow, gsite);
    if (k.ccm) isp_rgb_fast<CAM16, true>(k, S[0], S[1], S[2], sc[0], sc[1], sc[2], rgb);
    else isp_rgb_fast<CAM16, false>(k, S[0], S[1], S[2], sc[0], sc[1], sc[2], rgb);
  }

  // sample on the image frame: the words outside the image are replaced by 0 (-> zero samples) and the raw
  // values are renormalised by the in-bounds weight sum of the pixel's (row class, column class)
  __device__ __forceinline__ void sample_frame(int f, int row, int col, float (&rgb)[3]) const {
    const uint32_t* p = reinterpret_cast<const uint32_t*>(src.fp.in[f]) + (size_t)row * pitch_words + 3 * (col >> 3);
    const bool m2 = row >= 2, m1 = row >= 1, p1 = row + 1 < k.H, p2 = row + 2 < k.H, cl = col >= 2;
    const uint32_t a0 = m2 ? __ldg(p - 2 * pitch_words) : 0u;
    const uint32_t bm = (m1 && cl) ? __ldg(p - pitch_words - 1) : 0u, b0 = m1 ? __ldg(p - pitch_words) : 0u;
    const uint32_t cm = cl ? __ldg(p - 1) : 0u, c0 = __ldg(p), c1 = __ldg(p + 1);
    const uint32_t dm = (p1 && cl) ? __ldg(p + pitch_words - 1) : 0u, d0 = p1 ? __ldg(p + pitch_words) : 0u;
    const uint32_t e0 = p2 ? __ldg(p + 2 * pitch_words) : 0u;
    float S[3], sc[3];
    bool brow, gsite;
    sums_from_words(a0, bm, b0, cm, c0, c1, dm, d0, e0, row, S, sc, brow, gsite);
    const float* t = c_border.t[site_kernel_of(brow, gsite) + k.kbase][edge_class(row, k.H)][edge_class(col, k.W)];
    constexpr float kn = 256.f * kInv4095;
    float x[3];
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) x[ch] = frame_exact(CAM16 ? S[ch] * (sc[ch] * 0.0625f) : fmaf(S[ch], sc[ch] * kn, -16.f * kn), t[ch]);
    raw_to_rgb<CAM16>(k, x, rgb);       // the sweep's own CCM (FMA chain; identity without CCM), clamp and rounding
  }

  __device__ __forceinline__ bool on_frame(int row, int col) const { return row < 2 || row >= k.H - 2 || col < 2 || col >= k.W - 2; }

  __device__ __forceinline__ void sample(long long idx, float (&rgb)[3]) const {
    const int j = (int)(idx % ws_);
    const long long q = idx / ws_;
    const int i = (int)(q % hs);
    const int f = (int)(q / hs);
    const int row = i * stride, col = j * stride;
    if (on_frame(row, col)) sample_frame(f, row, col, rgb);
    else sample_fast(reinterpret_cast<const uint32_t*>(src.fp.in[f]) + (size_t)row * pitch_words + 3 * (col >> 3), row, rgb);
  }

  // Pass A -- interior samples.  A warp task = 128 consecutive samples of one interior sample row: lanes take
  // consecutive samples (12 bytes apart, so the warp's loads are contiguous), four per lane.  The loop body is
  // branch-free (a lane without a sample of its own -- past the row end, or the frame column j = 0 -- reloads a
  // valid neighbour and drops the result), so all 36 loads of a lane are in flight together.
  // Pass B -- the samples on the image frame (sample row 0 and sample column 0; a few thousand): one per thread.
  template <class F>
  __device__ __forceinline__ void for_each(long long n, F&& f) const {
    const int nrows = (int)(n / ws_), nframes = nrows / hs;
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    const int wstep = stride >> 3;                       // thread columns (3 words) between samples
    // interior sample rows: i in [i_lo, i_hi); interior sample columns: j in [j_lo, j_hi)
    const int i_lo = (2 + stride - 1) / stride, i_hi = min(hs, (k.H - 3) / stride + 1);
    const int j_lo = (2 + stride - 1) / stride, j_hi = min(ws_, (k.W - 3) / stride + 1);
    const int rows_in = max(i_hi - i_lo, 0), cols_in = max(j_hi - j_lo, 0);
    const int nseg = (cols_in + 32 * kMeterUnroll - 1) / (32 * kMeterUnroll);
    const int ntasks = nframes * rows_in * nseg;
    for (int task = blockIdx.x * wpb + (threadIdx.x >> 5); task < ntasks; task += gridDim.x * wpb) {
      const int rt = task / nseg, seg = task - rt * nseg;
      const int fr = rt / rows_in, i = i_lo + (rt - fr * rows_in);
      const int row = i * stride;
      const unsigned base = (unsigned)((fr * hs + i) * ws_);
      const uint32_t* prow = reinterpret_cast<const uint32_t*>(src.fp.in[fr]) + (size_t)row * pitch_words;
      const int j0 = j_lo + seg * 32 * kMeterUnroll + lane;
      float rgb[kMeterUnroll][3];
#pragma unroll
      for (int u = 0; u < kMeterUnroll; ++u) sample_fast(prow + 3 * wstep * min(j0 + 32 * u, j_hi - 1), row, rgb[u]);
#pragma unroll
      for (int u = 0; u < kMeterUnroll; ++u)
        if (j0 + 32 * u < j_hi) f((long long)(base + (unsigned)(j0 + 32 * u)), rgb[u]);
    }
    // frame samples: per frame, (hs - rows_in) whole sample rows + (ws_ - cols_in) columns of the interior rows
    const int frame_rows = hs - rows_in, frame_cols = ws_ - cols_in;
    const int per_frame = frame_rows * ws_ + rows_in * frame_cols;
    const int total = nframes * per_frame;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < total; t += gridDim.x * blockDim.x) {
      const int fr = t / per_frame;
      int r = t - fr * per_frame, i, j;
      if (r < frame_rows * ws_) {
        const int ri = r / ws_;
        j = r - ri * ws_;
        i = ri < i_lo ? ri : i_hi + (ri - i_lo);                  // sample rows before / after the interior band
      } else {
        r -= frame_rows * ws_;
        const int ii = r / frame_cols, cj = r - ii * frame_cols;
        i = i_lo + ii;
        j = cj < j_lo ? cj : j_hi + (cj - j_lo);
      }
      float rgb[3];
      sample_frame(fr, i * stride, j * stride, rgb);
      f((long long)((fr * hs + i) * ws_ + j), rgb);
    }
  }
};

// ---------------------------------------------------------------- host orchestration
// profile hooks: inside a stream capture the record must be an "external" event node to stay queryable
static inline void record_profile_event(void* ev, cudaStream_t s) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive)
    cudaEventRecordWithFlags((cudaEvent_t)ev, s, cudaEventRecordExternal);
  else
    cudaEventRecord((cudaEvent_t)ev, s);
}

// host dispatch of the Reinhard write sweep on (color_adapt == 0, gamma != 1)
template <int P, bool CAM16, typename OutT, bool EXT>
static int launch_reinhard(const Packed12Loader2<CAM16, EXT>& ld, const FramePtrs& fp, const IspConsts& k, const Stream2Geom& g, cudaStream_t s) {
  const bool ca0 = k.ca == 0.f, gam = k.gamma != 1.0f, bl = !EXT && k.kbase != 0;
  if (ca0 && gam) { EpiReinhard2<CAM16, OutT, true, true, EXT> e{fp, k}; return launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard>", bl); }
  if (ca0) { EpiReinhard2<CAM16, OutT, true, false, EXT> e{fp, k}; return launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard>", bl); }
  if (gam) { EpiReinhard2<CAM16, OutT, false, true, EXT> e{fp, k}; return launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard>", bl); }
  EpiReinhard2<CAM16, OutT, false, false, EXT> e{fp, k};
  return launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard>", bl);
}

// EXT: the extended kernels (IDS layout in the row loader, flips in the store); Malvar only -- the host mirror routes
// bilinear + IDS / flip through the re-pack pass / the transform kernel.
template <bool CAM16, int MODE, typename OutT, bool EXT>
static int run_pass_ext(const FramePtrs& fp, IspConsts k, int nframes, int rows_per_task, cudaStream_t s, void* ev_start, void* ev_stop) {
  const Stream2Geom g = make_geom2(k.H, k.W, nframes, rows_per_task);
  const bool bl = !EXT && k.kbase != 0;
  if (EXT && k.kbase != 0) { set_error("process_packed12: the IDS layout / flips are fused for the Malvar demosaic only"); return B200ISP_E_ARG; }
  Packed12Loader2<CAM16, EXT> ld;
  ld.fp = fp; ld.pitch_words = k.W * 3 / 8; ld.ids = k.ids;
  int st = B200ISP_OK;
  auto record = [&](void* ev) { record_profile_event(ev, s); };
  if (ev_start) record(ev_start);
  ISP_DISPATCH_PATTERN(k.pattern, P, {
    if constexpr (MODE == MODE_RGB) { EpiRgb2<CAM16, OutT, EXT> e{fp, k}; st = launch_stream2<P>(ld, e, g, s, "isp_stream<rgb>", bl); }
    else if constexpr (MODE == MODE_LINEAR) {
      bool fast = false;
      if constexpr (!CAM16) fast = !k.ccm && k.gamma == 1.0f;
      if constexpr (!CAM16) { if (fast) { EpiLinear2<false, OutT, true, EXT> e{fp, k}; st = launch_stream2<P>(ld, e, g, s, "isp_stream<linear,fast>", bl); } }
      if (!fast) { EpiLinear2<CAM16, OutT, false, EXT> e{fp, k}; st = launch_stream2<P>(ld, e, g, s, "isp_stream<linear>", bl); }
    }
    else if constexpr (MODE == MODE_RMAX) {
      if (k.ca == 0.f) { EpiReinhardMax2<CAM16, true> e{fp, k}; st = launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard_max>", bl); }
      else { EpiReinhardMax2<CAM16, false> e{fp, k}; st = launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard_max>", bl); }
    } else {
      st = launch_reinhard<P, CAM16, OutT, EXT>(ld, fp, k, g, s);
    }
  });
  if (ev_stop) record(ev_stop);
  return st;     // the 2-pixel image frame is renormalised inside the sweep (border_fix.cuh): no border kernel
}

template <bool CAM16, int MODE, typename OutT>
static int run_pass(const FramePtrs& fp, IspConsts k, int nframes, int rows_per_task, cudaStream_t s,
                    void* ev_start = nullptr, void* ev_stop = nullptr) {
  // the max sweep stores nothing: it only needs the extended loader for IDS frames
  const bool ext = k.ids != 0 || (MODE != MODE_RMAX && k.flip != 0);
  if (ext) return run_pass_ext<CAM16, MODE, OutT, true>(fp, k, nframes, rows_per_task, s, ev_start, ev_stop);
  return run_pass_ext<CAM16, MODE, OutT, false>(fp, k, nframes, rows_per_task, s, ev_start, ev_stop);
}

// ---------------------------------------------------------------- Camera16 Reinhard in ONE sweep + a light second pass
// pass A: the max sweep with STORE over all frames (scratch = f16 map); pass B: out = quantise((p / max)^(1/gamma))
// element-wise on the scratch, all frames in one launch (blockIdx.y = frame).
template <typename OutT>
__global__ void __launch_bounds__(256) reinhard_scratch_out_kernel(const FramePtrs scratch /* .out = f16 maps */, const FramePtrs fp,
                                                                   long long n_elems /* per frame, % 8 == 0 */, float gamma, const Workspace* ws) {
  const int frame = gridDim.y - 1 - blockIdx.y;       // last frame first: the sweep wrote it last, part of its map is still in L2
  const __half* src = reinterpret_cast<const __half*>(scratch.out[frame]);
  OutT* dst = reinterpret_cast<OutT*>(fp.out[frame]);
  const float inv_max = __fdiv_rn(1.0f, fmaxf(1e-6f, __ldcg(&ws->frame_max[frame])));
  const float inv_gamma = (float)(1.0 / (double)gamma);
  const bool has_gamma = gamma != 1.0f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_elems / 8; i += (long long)gridDim.x * blockDim.x) {
    const uint4 w = __ldcs(reinterpret_cast<const uint4*>(src) + i);
    const __half* t = reinterpret_cast<const __half*>(&w);
    uint32_t v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float q = __saturatef(__half2float(t[j]) * inv_max);
      if (has_gamma) q = fast_pow(q, inv_gamma);
      v[j] = Quant<OutT>::q(q);
    }
    if constexpr (std::is_same<OutT, uint8_t>::value) {
      uint2 o;
      o.x = __byte_perm(__byte_perm(v[0], v[1], 0x0040), __byte_perm(v[2], v[3], 0x0040), 0x5410);
      o.y = __byte_perm(__byte_perm(v[4], v[5], 0x0040), __byte_perm(v[6], v[7], 0x0040), 0x5410);
      __stcs(reinterpret_cast<uint2*>(dst) + i, o);
    } else if constexpr (std::is_same<OutT, uint16_t>::value) {
      uint4 o = make_uint4(__byte_perm(v[0], v[1], 0x5410), __byte_perm(v[2], v[3], 0x5410), __byte_perm(v[4], v[5], 0x5410),
                           __byte_perm(v[6], v[7], 0x5410));
      __stcs(reinterpret_cast<uint4*>(dst) + i, o);
    } else {
      alignas(16) __half o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = __float2half_rn(__uint_as_float(v[j]));
      __stcs(reinterpret_cast<uint4*>(dst) + i, *reinterpret_cast<const uint4*>(o));
    }
  }
}

// pass B of the one-sweep Camera32 Reinhard -> u8 path: out = trunc(255 * ((v + 0.5) / 65535 / max)^(1/gamma)) for the u16
// map v of EpiReinhardMax2<false, CA0, STORE>; frames the map declined are skipped (the gated sweeps write them).
// u16 -> f32 by dropping the halves into the mantissa of 2^23 (PRMT) and one exact packed subtraction -- no conversion
// instruction, packed arithmetic throughout.  Dense outputs: 16 values per thread and iteration (two 16-byte loads, one
// 16-byte store); PITCHED (the outputs are tiles of a grid image, orow > 3 W): 8 values, row / column from the chunk index.
__device__ __forceinline__ void map16_pair(uint32_t w, f2 a2, f2 h2, f2 ig2, bool gamma, uint32_t& v0, uint32_t& v1) {
  const f2 t = add2(pk(__uint_as_float(__byte_perm(w, 0x4B000000u, 0x7610)), __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7632))),
                    bc(-8388608.f));
  f2 q = fma2(t, a2, h2);
  if (gamma) {
    float lo, hi, l0, l1;
    upk(q, lo, hi);
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l0) : "f"(lo));
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l1) : "f"(hi));
    upk(mul2(pk(l0, l1), ig2), lo, hi);
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(l0) : "f"(lo));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(l1) : "f"(hi));
    q = pk(l0, l1);
  }
  float ql, qh;
  upk(fma2_rz(q, bc(255.f), bc(8388608.f)), ql, qh);
  v0 = __float_as_uint(ql);
  v1 = __float_as_uint(qh);
}
__device__ __forceinline__ uint32_t pack4_u8(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  return __byte_perm(__byte_perm(a, b, 0x0040), __byte_perm(c, d, 0x0040), 0x5410);
}

template <bool GAMMA, bool PITCHED>
__global__ void __launch_bounds__(256) reinhard_map16_out_kernel(const FramePtrs scratch /* .out = u16 maps */, const FramePtrs fp,
                                                                 int H, int W, int orow, float gamma, const Workspace* ws) {
  const int frame = gridDim.y - 1 - blockIdx.y;       // last frame first: the sweep wrote it last, part of its map is still in L2
  const float mx = __ldcg(&ws->frame_max[frame]);
  if (reinhard_map16_declined(mx)) return;
  const uint4* src = reinterpret_cast<const uint4*>(scratch.out[frame]);
  const float a = __fdiv_rn(__fdiv_rn(1.0f, mx), kMap16Scale);
  const f2 a2 = bc(a), h2 = bc(0.5f * a), ig2 = bc((float)(1.0 / (double)gamma));
  const long long stride = (long long)gridDim.x * blockDim.x;
  if constexpr (!PITCHED) {
    // two 16-value chunks per iteration, the four 16-byte loads issued before the first use.  Measured on cfg3 (gamma 0.9):
    // 8 CTAs per SM 131 us, 4: 155 us, 2: slower still -- unlike a plain copy this pass wants every thread slot
    // (profiles/r02_reinhard_map16.txt)
    uint4* dst = reinterpret_cast<uint4*>(fp.out[frame]);
    const long long n16 = (long long)H * W * 3 / 16;                   // H even, W % 8 == 0
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += 2 * stride) {
      const long long i2 = i + stride;
      const bool two = i2 < n16;
      const uint4 w0 = __ldcs(src + 2 * i), w1 = __ldcs(src + 2 * i + 1);
      uint4 w2 = w0, w3 = w1;
      if (two) { w2 = __ldcs(src + 2 * i2); w3 = __ldcs(src + 2 * i2 + 1); }
      {
        const uint32_t w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
        uint32_t v[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) map16_pair(w[j], a2, h2, ig2, GAMMA, v[2 * j], v[2 * j + 1]);
        __stcs(dst + i, make_uint4(pack4_u8(v[0], v[1], v[2], v[3]), pack4_u8(v[4], v[5], v[6], v[7]), pack4_u8(v[8], v[9], v[10], v[11]),
                                   pack4_u8(v[12], v[13], v[14], v[15])));
      }
      if (two) {
        const uint32_t w[8] = {w2.x, w2.y, w2.z, w2.w, w3.x, w3.y, w3.z, w3.w};
        uint32_t v[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) map16_pair(w[j], a2, h2, ig2, GAMMA, v[2 * j], v[2 * j + 1]);
        __stcs(dst + i2, make_uint4(pack4_u8(v[0], v[1], v[2], v[3]), pack4_u8(v[4], v[5], v[6], v[7]), pack4_u8(v[8], v[9], v[10], v[11]),
                                    pack4_u8(v[12], v[13], v[14], v[15])));
      }
    }
  } else {
    uint8_t* dst = reinterpret_cast<uint8_t*>(fp.out[frame]);
    const int cpr = W * 3 / 8;                                         // 8-value chunks per row
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)H * cpr; i += stride) {
      const int row = (int)(i / cpr), c = (int)(i - (long long)row * cpr);
      const uint4 w0 = __ldcs(src + i);
      const uint32_t w[4] = {w0.x, w0.y, w0.z, w0.w};
      uint32_t v[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) map16_pair(w[j], a2, h2, ig2, GAMMA, v[2 * j], v[2 * j + 1]);
      __stcs(reinterpret_cast<uint2*>(dst + (size_t)row * orow + 8 * c), make_uint2(pack4_u8(v[0], v[1], v[2], v[3]), pack4_u8(v[4], v[5], v[6], v[7])));
    }
  }
}

// pass B through a table (Camera16, gamma != 1, dense u8 outputs): the f16 map has only 65 536 patterns, and the output is a
// pure function of the pattern and the frame maximum.  reinhard_lut_build_kernel evaluates that function once per pattern and
// frame with exactly the arithmetic of reinhard_scratch_out_kernel (so the result is bit-identical to it); reinhard_lut_out_kernel
// keeps the frame's 64 KB table in shared memory and turns every value into one LDS.U8: no MUFU (the arithmetic pass needs 6 per
// pixel and sits at 74 % of the MUFU pipe), 10 instead of 21 instructions per pixel -- the pass becomes a plain HBM stream.
// Camera32 has no table form: its pass (reinhard_map16_out_kernel) is bound by its 2 : 1 read / write DRAM stream (4.75 TB/s),
// not by the MUFU pipe, and the table form measured 134.9 vs 131.5 us on cfg3.
constexpr int kLutBytes = 65536;
// the table form of pass B (defined in fused_api.cu); lut = n_frames x 64 KB behind the maps in the caller's scratch
int run_lut_pass(const FramePtrs& sc, const FramePtrs& fp, int n_frames, long long n_elems, uint8_t* lut, float gamma, const Workspace* ws,
                 cudaStream_t s);

// pass B with planar YUV 4:2:0 output (SURVEY 8f-2, for video encoders): the u8 RGB of reinhard_scratch_out_kernel
// is formed in registers and converted with the arithmetic of color/yuv_420.py:47-64 (csrc/yuv420.cu: x / 255, the
// BT.601 matrix applied to the BGR-swizzled pixel, chroma = mean of the 2x2 quad, one-sided clamp) -- bit-identical
// to rgb_yuv420_image(process_packed12(...)) without writing or re-reading the RGB image: 1.5 B/px out instead of 3.
// Thread = 8 pixel columns x 2 rows (four quads); out = (3H/2, W) u8: H rows of Y, then chroma plane 0 (third
// matrix row) and plane 1 (second matrix row).
static __global__ void __launch_bounds__(128) reinhard_scratch_yuv_kernel(const FramePtrs scratch, const FramePtrs fp, int H, int W, float gamma,
                                                                   const Workspace* ws) {
  // x / 255 (correctly rounded, yuv_420.py:50) for the 256 possible inputs: a table instead of three IEEE divisions per pixel
  __shared__ float unit[256];
  for (int i = threadIdx.x; i < 256; i += blockDim.x) unit[i] = __fdiv_rn((float)i, 255.0f);
  __syncthreads();
  const int gx = blockIdx.x * blockDim.x + threadIdx.x, qy = blockIdx.y, frame = blockIdx.z;
  if (gx >= W / 8) return;
  const __half* src = reinterpret_cast<const __half*>(scratch.out[frame]);
  uint8_t* yuv = reinterpret_cast<uint8_t*>(fp.out[frame]);
  const float inv_max = __fdiv_rn(1.0f, fmaxf(1e-6f, __ldcg(&ws->frame_max[frame])));
  const float inv_gamma = (float)(1.0 / (double)gamma);
  const bool has_gamma = gamma != 1.0f;
  constexpr float M[9] = {0.299f, 0.587f, 0.114f, -0.168736f, -0.331264f, 0.5f, 0.5f, -0.418688f, -0.081312f};   // yuv_420.py:12-16
  float rgb[2][24];
#pragma unroll
  for (int dy = 0; dy < 2; ++dy) {
    alignas(16) __half h[24];
    ld_bytes<48>(src + ((size_t)(2 * qy + dy) * W + 8 * gx) * 3, h);
#pragma unroll
    for (int e = 0; e < 24; ++e) {
      float q = __saturatef(__half2float(h[e]) * inv_max);
      if (has_gamma) q = fast_pow(q, inv_gamma);
      rgb[dy][e] = unit[Quant<uint8_t>::q(q) & 0xFFu];                          // the u8 value the RGB path stores, / in_scale
    }
  }
  alignas(8) uint8_t yrow[2][8];
  alignas(4) uint8_t cu4[4], cv4[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float u = 0.f, v = 0.f;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const float* p = &rgb[dy][3 * (2 * q + dx)];
        float o[3];
#pragma unroll
        for (int r = 0; r < 3; ++r)      // M @ (B, G, R), products and sums rounded separately, left to right
          o[r] = __fadd_rn(__fadd_rn(__fmul_rn(M[3 * r], p[2]), __fmul_rn(M[3 * r + 1], p[1])), __fmul_rn(M[3 * r + 2], p[0]));
        const float cu = __fadd_rn(o[1], 0.5f), cv = __fadd_rn(o[2], 0.5f);
        yrow[dy][2 * q + dx] = cast_from_f32<uint8_t>(__fmul_rn(fminf(1.0f, o[0]), 255.0f));
        if (dy == 0 && dx == 0) { u = cu; v = cv; } else { u = __fadd_rn(u, cu); v = __fadd_rn(v, cv); }
      }
    // u / 4.0 (yuv_420.py:62-63): a power-of-two divisor, the product with 0.25 is the same correctly rounded value
    cu4[q] = cast_from_f32<uint8_t>(__fmul_rn(fminf(1.0f, __fmul_rn(u, 0.25f)), 255.0f));
    cv4[q] = cast_from_f32<uint8_t>(__fmul_rn(fminf(1.0f, __fmul_rn(v, 0.25f)), 255.0f));
  }
#pragma unroll
  for (int dy = 0; dy < 2; ++dy) st_bytes<8>(yuv + (size_t)(2 * qy + dy) * W + 8 * gx, yrow[dy]);
  uint8_t* planes = yuv + (size_t)H * W;
  const size_t plane = (size_t)(H / 2) * (W / 2), idx = (size_t)qy * (W / 2) + 4 * gx;
  st_bytes<4>(planes + plane + idx, cu4);
  st_bytes<4>(planes + idx, cv4);
}

// pass B with a TRANSPOSING transform (k.flip bit 2: transpose / rotate_90 / rotate_270 / transverse, interpolate.py:36-56 --
// rotate_90 is the rig script's default, scripts/tonemap_scan.py) for both one-sweep Reinhard -> u8 forms: the element-wise
// pass is the cheap place to turn the image, the sweep keeps its plain row stores and the separate transform kernel
// (3 + 3 B/px) disappears.  Output (i, j) = source (r, c), i = c or W-1-c (bit 0), j = r or H-1-r (bit 1), shape (W, H).
// CTA = a tile of 128 output columns (source rows) x 16 source columns.  Load phase: thread = 8 pixels of one source row
// (3 x 16 bytes of the map; the tile's 96-byte row segments are whole sectors), normalise / gamma / quantise exactly like
// the dense pass, one RGBx word per pixel into shared memory at [column][j + (j >> 3)] (row pitch 144 words).  Store phase:
// thread = 8 consecutive pixels of one OUTPUT row (24 bytes, three 8-byte stores): a half warp writes 384 contiguous
// bytes, and with that layout the 32 lanes of every LDS hit 32 different banks.  Default write policy: the two partial
// sectors at the ends of a 384-byte piece meet their neighbours' (blockIdx.x runs along the output row) in L2.
// Camera32: frames the u16 map declined were written as plain (H, W, 3) u8 into the frame's scratch by the gated write sweep
// BEFORE this pass, which then only turns them.
#ifndef ISP_TURNED_MINBLOCKS
#define ISP_TURNED_MINBLOCKS 6     // measured: 8 CTAs per SM (32 registers, no spills) gain 2 % on eager Camera32 calls but lose 1 % on
                                   // Camera16 and 2 % on the graphed look-ahead step (cfg3_rot90 214 -> 207 Gpixel/s)
#endif
constexpr int kTpRows = 128, kTpCols = 16, kTpPitch = 144;
template <bool CAM16, bool GAMMA>
__global__ void __launch_bounds__(256, ISP_TURNED_MINBLOCKS) reinhard_out_transposed_kernel(const FramePtrs scratch, const FramePtrs fp, int H, int W, int orow, int flip,
                                                                      float gamma, const Workspace* ws) {
  __shared__ uint32_t tile[kTpCols * kTpPitch];
  const int frame = gridDim.z - 1 - blockIdx.z;        // last frame first, like the dense pass
  const int j0 = blockIdx.x * kTpRows, c0 = blockIdx.y * kTpCols;
  const float mx = __ldcg(&ws->frame_max[frame]);
  {
    const int cg = threadIdx.x & 1, lr = threadIdx.x >> 1;
    const int j = j0 + lr, c = c0 + 8 * cg;
    if (j < H && c < W) {
      const int r = (flip & 2) ? H - 1 - j : j;
      const size_t px = (size_t)r * W + c;
      uint32_t v[24];
      if constexpr (CAM16) {
        const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(scratch.out[frame]) + px * 3);
        const uint4 w3[3] = {__ldcs(src), __ldcs(src + 1), __ldcs(src + 2)};
        const __half* t = reinterpret_cast<const __half*>(w3);
        const float inv_max = __fdiv_rn(1.0f, fmaxf(1e-6f, mx));
        const float inv_gamma = (float)(1.0 / (double)gamma);
#pragma unroll
        for (int e = 0; e < 24; ++e) {
          float q = __saturatef(__half2float(t[e]) * inv_max);
          if (GAMMA) q = fast_pow(q, inv_gamma);
          v[e] = Quant<uint8_t>::q(q);
        }
      } else if (reinhard_map16_declined(mx)) {
        const uint2* src = reinterpret_cast<const uint2*>(reinterpret_cast<const uint8_t*>(scratch.out[frame]) + px * 3);
        const uint2 b3[3] = {__ldcs(src), __ldcs(src + 1), __ldcs(src + 2)};
        const uint8_t* t = reinterpret_cast<const uint8_t*>(b3);
#pragma unroll
        for (int e = 0; e < 24; ++e) v[e] = t[e];
      } else {
        const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const uint16_t*>(scratch.out[frame]) + px * 3);
        const uint4 w3[3] = {__ldcs(src), __ldcs(src + 1), __ldcs(src + 2)};
        const uint32_t* w = reinterpret_cast<const uint32_t*>(w3);
        const float a = __fdiv_rn(__fdiv_rn(1.0f, mx), kMap16Scale);
        const f2 a2 = bc(a), h2 = bc(0.5f * a), ig2 = bc((float)(1.0 / (double)gamma));
#pragma unroll
        for (int e = 0; e < 12; ++e) map16_pair(w[e], a2, h2, ig2, GAMMA, v[2 * e], v[2 * e + 1]);
      }
      uint32_t* col = tile + (8 * cg) * kTpPitch + lr + (lr >> 3);
#pragma unroll
      for (int q = 0; q < 8; ++q)      // the values' low bytes -> R | G << 8 | B << 16 (the top byte is never read)
        col[q * kTpPitch] = __byte_perm(__byte_perm(v[3 * q], v[3 * q + 1], 0x0040), v[3 * q + 2], 0x0410);
    }
  }
  __syncthreads();
  {
    const int rg = threadIdx.x & 15, lc = threadIdx.x >> 4;
    const int j = j0 + 8 * rg, c = c0 + lc;
    if (j < H && c < W) {                               // H % 8 == 0: the group is inside the row or entirely outside
      const uint32_t* sp = tile + lc * kTpPitch + 9 * rg;
      uint32_t p[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) p[q] = sp[q];
      const int i = (flip & 1) ? W - 1 - c : c;
      uint2* d = reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(fp.out[frame]) + (size_t)i * orow + 3 * j);
      d[0] = make_uint2(__byte_perm(p[0], p[1], 0x4210), __byte_perm(p[1], p[2], 0x5421));
      d[1] = make_uint2(__byte_perm(p[2], p[3], 0x6542), __byte_perm(p[4], p[5], 0x4210));
      d[2] = make_uint2(__byte_perm(p[5], p[6], 0x5421), __byte_perm(p[6], p[7], 0x6542));
    }
  }
}
template <bool CAM16>
static int run_out_transposed(const FramePtrs& sc, const FramePtrs& fp, int n_frames, const IspConsts& k, cudaStream_t s) {
  const dim3 grid((unsigned)((k.H + kTpRows - 1) / kTpRows), (unsigned)((k.W + kTpCols - 1) / kTpCols), (unsigned)n_frames);
  if (k.gamma != 1.0f) reinhard_out_transposed_kernel<CAM16, true><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.flip, k.gamma, k.ws);
  else reinhard_out_transposed_kernel<CAM16, false><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.flip, k.gamma, k.ws);
  return cuda_status(cudaPeekAtLastError(), "reinhard_out_transposed_kernel");
}

// pass A for frames [0, nframes): instantiated once per ISP dtype (fused_inst.cu with ISP_INST_RMAX); Camera16 stores the f16
// map (any color_adapt), Camera32 the u16 fixed-point map (color_adapt == 0 only: the caller checks)
template <bool CAM16>
int run_rstore(const FramePtrs& fp_scratch, IspConsts k, int nframes, int rows_per_task, cudaStream_t s, void* ev_start, void* ev_stop) {
  const Stream2Geom g = make_geom2(k.H, k.W, nframes, rows_per_task);
  int st = B200ISP_OK;
  if (ev_start) record_profile_event(ev_start, s);
  auto launch = [&](auto ld, bool bl) -> int {
    ld.fp = fp_scratch; ld.pitch_words = k.W * 3 / 8; ld.ids = k.ids;
    ISP_DISPATCH_PATTERN(k.pattern, P, {
      if (k.ca == 0.f) { EpiReinhardMax2<CAM16, true, true> e{fp_scratch, k}; st = launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard_store>", bl); }
      else if constexpr (CAM16) { EpiReinhardMax2<true, false, true> e{fp_scratch, k}; st = launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard_store>", bl); }
      else { set_error("process_packed12: the one-sweep Camera32 Reinhard map needs color_adapt == 0"); return B200ISP_E_ARG; }
    });
    return st;
  };
  if (k.ids) {
    if (k.kbase != 0) { set_error("process_packed12: the IDS layout is fused for the Malvar demosaic only"); return B200ISP_E_ARG; }
    st = launch(Packed12Loader2<CAM16, true>{}, false);
  } else {
    st = launch(Packed12Loader2<CAM16, false>{}, k.kbase != 0);
  }
  if (ev_stop) record_profile_event(ev_stop, s);
  return st;
}

// The gated exact fallback of the one-sweep Camera32 path (color_adapt == 0, standard layout): max sweep into ws->frame_max2
// + write sweep, both over all frames, every warp leaving at once unless its frame was declined -- in the usual case two
// launches of CTAs that exit immediately.
int run_rmax_gated(const FramePtrs& fp, IspConsts k, int nframes, int rows_per_task, cudaStream_t s);

// frame-global Reinhard max: independent of the output dtype, instantiated once per ISP dtype (fused_inst.cu with ISP_INST_RMAX)
template <bool CAM16>
int run_rmax(const FramePtrs& fp, IspConsts k, int nframes, int rows_per_task, cudaStream_t s) {
  return run_pass<CAM16, MODE_RMAX, uint8_t>(fp, k, nframes, rows_per_task, s);
}

int run_write_gated(const FramePtrs& fp, IspConsts k, int nframes, int rows_per_task, cudaStream_t s);

// How b200isp_process_packed12 runs the Reinhard tone map of a parameter block that passed its checks, and the bytes of
// reinhard_scratch that form uses: the maps of all frames, plus the per-frame tables of kF16Table.  reinhard_plan
// (fused_api.cu) is the only place that decides this; run_fused, run_resize_t and b200isp_reinhard_scratch_bytes ask it.
// A scratch smaller than map_bytes means the exact form (YUV 4:2:0 and resizing ISPs: refused); one that holds the maps
// but not the tables means kF16Arith, whose result is bit-identical to kF16Table's.
enum class ReinhardForm {
  kNone,          // no Reinhard tone map (linear, TM_NONE): one sweep
  kExact,         // max sweep + write sweep (run_rmax, MODE_REINHARD)
  kResizeMap,     // resizing ISP: the map at output resolution in the ISP dtype + a normalise pass (fused_resize.cu)
  kF16Turned,     // Camera16 f16 map + reinhard_out_transposed_kernel (transposing transforms)
  kF16Yuv,        // Camera16 f16 map + reinhard_scratch_yuv_kernel
  kF16Table,      // Camera16 f16 map + run_lut_pass (u8, gamma != 1: a 64 KB table per frame behind the maps)
  kF16Arith,      // Camera16 f16 map + reinhard_scratch_out_kernel
  kU16Map,        // Camera32 u16 fixed-point map + reinhard_map16_out_kernel + the gated exact sweeps
  kU16Turned,     // Camera32 u16 fixed-point map + the gated exact sweeps + reinhard_out_transposed_kernel
};
struct ReinhardPlan {
  ReinhardForm form;
  size_t map_bytes, bytes;    // 0 for kNone and kExact
};
ReinhardPlan reinhard_plan(const b200isp_fused_params& p, const IspConsts& k, int n_frames);

template <bool CAM16, typename OutT>
int run_fused(const FramePtrs& fp, int n_frames, const b200isp_fused_params& p, IspConsts k, cudaStream_t s) {
  const int rpt = p.rows_per_task;
  ReinhardPlan plan = reinhard_plan(p, k, n_frames);
  if (plan.map_bytes && (!p.reinhard_scratch || p.reinhard_scratch_bytes < plan.map_bytes)) plan.form = ReinhardForm::kExact;
  else if (plan.form == ReinhardForm::kF16Table && p.reinhard_scratch_bytes < plan.bytes) plan.form = ReinhardForm::kF16Arith;
  if (p.out_yuv420 && plan.form == ReinhardForm::kExact) {
    set_error("process_packed12: YUV 4:2:0 output needs Camera16 (f16), Reinhard, u8 and the reinhard_scratch buffer");
    return B200ISP_E_ARG;
  }
  if ((k.flip & 4) && plan.form == ReinhardForm::kExact) {
    set_error("process_packed12: the transposing transforms need the reinhard_scratch buffer (b200isp_reinhard_scratch_bytes)");
    return B200ISP_E_ARG;
  }
  constexpr bool kIspOut = (CAM16 && std::is_same<OutT, __half>::value) || (!CAM16 && std::is_same<OutT, float>::value);
  if (p.tonemap == B200ISP_TM_NONE) {
    if constexpr (kIspOut) return run_pass<CAM16, MODE_RGB, OutT>(fp, k, n_frames, rpt, s, p.profile_start, p.profile_stop);
    else { set_error("process_packed12: TM_NONE writes the ISP dtype"); return B200ISP_E_DTYPE; }
  }
  if constexpr (std::is_same<OutT, float>::value) {
    set_error("process_packed12: tone-mapped output must be u8, u16 or f16");
    return B200ISP_E_DTYPE;
  } else {
    if (p.tonemap == B200ISP_TM_LINEAR) return run_pass<CAM16, MODE_LINEAR, OutT>(fp, k, n_frames, rpt, s, p.profile_start, p.profile_stop);
    // frame_max and frame_max2 are adjacent in the workspace: one memset node
    static_assert(offsetof(Workspace, frame_max2) == offsetof(Workspace, frame_max) + sizeof(float) * B200ISP_MAX_FRAMES, "adjacent");
    int st = cuda_status(cudaMemsetAsync(k.ws->frame_max, 0, sizeof(float) * 2 * B200ISP_MAX_FRAMES, s), "memset frame_max");
    if (st) return st;
    if constexpr (CAM16) {
      // Camera16: the reference stores the map as f16 anyway -> one sweep writes it to the caller's scratch, a light
      // element-wise pass normalises it (no second sweep, no L2 grouping)
      if (plan.form != ReinhardForm::kExact) {
        FramePtrs sc = fp;
        for (int f = 0; f < n_frames; ++f) sc.out[f] = (char*)p.reinhard_scratch + (size_t)f * k.H * k.W * 3 * sizeof(__half);
        IspConsts kp = k;            // the map is a plain dense (H, W, 3) image whatever the output looks like
        kp.flip = 0;
        kp.orow = 3 * k.W;
        st = run_rstore<true>(sc, kp, n_frames, rpt, s, p.profile_start, p.profile_stop);
        if (st) return st;
        if (plan.form == ReinhardForm::kF16Turned) return run_out_transposed<true>(sc, fp, n_frames, k, s);     // the normalise pass turns the image
        if (plan.form == ReinhardForm::kF16Yuv) {
          const dim3 grid((unsigned)((k.W / 8 + 127) / 128), (unsigned)(k.H / 2), (unsigned)n_frames);
          reinhard_scratch_yuv_kernel<<<grid, 128, 0, s>>>(sc, fp, k.H, k.W, k.gamma, k.ws);
          return cuda_status(cudaPeekAtLastError(), "reinhard_scratch_yuv_kernel");
        }
        const long long n_elems = (long long)k.H * k.W * 3;
        if constexpr (std::is_same<OutT, uint8_t>::value) {
          if (plan.form == ReinhardForm::kF16Table)
            return run_lut_pass(sc, fp, n_frames, n_elems, (uint8_t*)p.reinhard_scratch + plan.map_bytes, k.gamma, k.ws, s);
        }
        const dim3 grid((unsigned)std::min<long long>((n_elems / 8 + 255) / 256, 4 * kNumSMs), (unsigned)n_frames);
        reinhard_scratch_out_kernel<OutT><<<grid, 256, 0, s>>>(sc, fp, n_elems, k.gamma, k.ws);
        return cuda_status(cudaPeekAtLastError(), "reinhard_scratch_out_kernel");
      }
    }
    if constexpr (!CAM16 && std::is_same<OutT, uint8_t>::value) {
      // Camera32 -> u8, color_adapt == 0, gamma in [0.3, 1]: ONE sweep that also stores the map as u16 fixed point
      // (6 B/px scratch) + an element-wise normalise / gamma / quantise pass.  The second demosaic of the two-sweep form
      // (66 of its 106 instructions per pixel) disappears; the u8 result is within 1 LSB of the two-sweep result
      // (measured: profiles/r02_reinhard_map16.txt).  Frames whose map does not fit [0, 1) (reinhard_map16_declined) are
      // redone exactly by the gated sweeps.
      if (plan.form != ReinhardForm::kExact) {
        FramePtrs sc = fp;
        for (int f = 0; f < n_frames; ++f) sc.out[f] = (char*)p.reinhard_scratch + (size_t)f * k.H * k.W * 3 * sizeof(uint16_t);
        if (plan.form == ReinhardForm::kU16Turned) {
          // transposing transform: map sweep (plain row stores), then the gated exact sweeps leave the frames the map declined
          // as plain (H, W, 3) u8 images in their scratch, then ONE pass normalises / turns every frame into the output
          IspConsts kp = k;
          kp.flip = 0;
          kp.orow = 3 * k.W;
          st = run_rstore<false>(sc, kp, n_frames, rpt, s, p.profile_start, p.profile_stop);
          if (st) return st;
          kp.gate = 1;
          st = run_rmax_gated(sc, kp, n_frames, rpt, s);
          if (st) return st;
          st = run_write_gated(sc, kp, n_frames, rpt, s);
          if (st) return st;
          return run_out_transposed<false>(sc, fp, n_frames, k, s);
        }
        // the normalise pass runs after the sweep with 8 CTAs per SM; running it under the sweep on a side stream measured
        // 212-186 vs 215 Gpixel/s on cfg3 (profiles/r02_reinhard_map16.txt)
        st = run_rstore<false>(sc, k, n_frames, rpt, s, p.profile_start, p.profile_stop);
        if (st) return st;
        const long long n_elems = (long long)k.H * k.W * 3;
        const bool gam = k.gamma != 1.0f, pitched = k.orow != 3 * k.W;
        const dim3 grid((unsigned)std::min<long long>((n_elems / 16 + 255) / 256, (8 * kNumSMs + n_frames - 1) / n_frames), (unsigned)n_frames);
        if (gam && pitched) reinhard_map16_out_kernel<true, true><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.gamma, k.ws);
        else if (gam) reinhard_map16_out_kernel<true, false><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.gamma, k.ws);
        else if (pitched) reinhard_map16_out_kernel<false, true><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.gamma, k.ws);
        else reinhard_map16_out_kernel<false, false><<<grid, 256, 0, s>>>(sc, fp, k.H, k.W, k.orow, k.gamma, k.ws);
        if ((st = cuda_status(cudaPeekAtLastError(), "reinhard_map16_out_kernel"))) return st;
        IspConsts kg = k;
        kg.gate = 1;
        st = run_rmax_gated(fp, kg, n_frames, rpt, s);
        if (st) return st;
        return run_write_gated(fp, kg, n_frames, rpt, s);
      }
    }
    // Camera32 (or no scratch): max sweep, then the write sweep recomputes the map.  Both sweeps are bound by
    // instruction issue, not by DRAM, so the second read of the packed frames (1.5 B/px) is cheaper than cutting the
    // call into L2-sized groups whose short launches end in idle tails (measured, profiles/r02_reinhard_diet.txt).
    st = run_rmax<CAM16>(fp, k, n_frames, rpt, s);
    if (st) return st;
    return run_pass<CAM16, MODE_REINHARD, OutT>(fp, k, n_frames, rpt, s, p.profile_start, p.profile_stop);
  }
}

extern template int run_rstore<true>(const FramePtrs&, IspConsts, int, int, cudaStream_t, void*, void*);
extern template int run_rstore<false>(const FramePtrs&, IspConsts, int, int, cudaStream_t, void*, void*);
extern template int run_rmax<true>(const FramePtrs&, IspConsts, int, int, cudaStream_t);
extern template int run_rmax<false>(const FramePtrs&, IspConsts, int, int, cudaStream_t);

}  // namespace isp
