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
// border_fix.cuh -- there is no border kernel).  run_fused (fused_api.cu) issues it, one case per ReinhardForm (below); the
// sweeps are launched by fused_inst.cu, the normalise passes live in normalise.cu:
//   [metering]  meter_fused_kernel (one cooperative launch) or meter_phase1 -> meter_phase2; sampler straight from the packed bytes
//   linear      stream2<EpiLinear2>                          one sweep
//   reinhard    kExact: stream2<EpiReinhardMax2> (frame-global max of the mapped values) -> stream2<EpiReinhard2>
//                         (the write sweep recomputes the map), one pair of launches for all frames of the call
//               kU16Map (Camera32 -> u8, color_adapt 0, gamma 0.3 .. 1): stream2<EpiReinhardMax2, STORE> (u16 fixed-point
//                         map) -> reinhard_map16_out_kernel (normalise / gamma / quantise) -> the two gated exact sweeps
//                         (they leave at once unless the map declined a frame)
//               kF16*: stream2<EpiReinhardMax2, STORE> (writes the f16 map the reference stores back anyway)
//                         -> reinhard_scratch_out_kernel (element-wise normalise / gamma / quantise), the table pass (u8,
//                         gamma != 1) or reinhard_scratch_yuv_kernel (YUV 4:2:0)
//               kF16Turned / kU16Turned (either one-sweep form -> u8 with a transposing ISP transform): the pass is
//                         reinhard_out_transposed_kernel (same arithmetic, the image turned through a shared-memory tile;
//                         Camera32: after the gated sweeps)
//   none        stream2<EpiRgb2>                             load_packed12 only: float RGB out
//   resizing ISP: fused_resize.cu (stream2_resize_kernel + orphan columns [-> resize_normalise_kernel or
//                         reinhard_scratch_out_kernel: kResizeMap])
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

// ---------------------------------------------------------------- packed12 row loader of the pair engine (stream2.cuh)
// Thread column tcol owns pixels 8*tcol..8*tcol+7 = bytes 12*tcol..12*tcol+11 = words 3*tcol..3*tcol+2; the halo pixels
// live in the top 3 bytes of word 3*tcol-1 and the low 3 bytes of word 3*tcol+3.  The decode mask is a register (0 for rows
// outside the image and for the halo columns of the first / last thread column -> "zero sample"), the halo loads are
// predicated on per-thread constants, and the row is delivered as the eight pairs (v[k], v[k+4]).
// Camera32: samples are decoded as b = 1 + v/4096 (12 bits dropped into the mantissa of 1.0f: one shift + one LOP3 per
// pixel, no int->float conversion).  All filter weights sum to 16, so the sums come out as 16 + S/4096 exactly and the bias
// folds into the epilogue's FMA.
// Camera16: the reference stores cfa = f16(v * f32(1/4095)); the same value is produced with one FMA (exact product,
// single rounding) and a packed f32->f16->f32 round trip.
// (biased_from_shifted: common.cuh)
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

// ---------------------------------------------------------------- what b200isp_process_packed12 launches (run_fused, fused_api.cu)
// How a call runs the Reinhard tone map of a parameter block that passed its checks, and the bytes of reinhard_scratch that
// form uses: the maps of all frames, plus the per-frame tables of kF16Table.  reinhard_plan (fused_api.cu) is the only place
// that decides this; run_fused and b200isp_reinhard_scratch_bytes ask it.  A scratch smaller than map_bytes means the exact
// form (YUV 4:2:0, transposing transforms and resizing ISPs: refused); one that holds the maps but not the tables means
// kF16Arith, whose result is bit-identical to kF16Table's.
enum class ReinhardForm {
  kNone,          // no Reinhard tone map (linear, TM_NONE): one sweep
  kExact,         // Sweep::kMax + Sweep::kReinhard
  kResizeMap,     // resizing ISP: the map at output resolution in the ISP dtype (run_resize) + a normalise pass
  kF16Turned,     // Camera16 f16 map (Sweep::kStore) + run_out_transposed (transposing transforms)
  kF16Yuv,        // Camera16 f16 map + run_scratch_yuv
  kF16Table,      // Camera16 f16 map + run_lut_pass (u8, gamma != 1: a 64 KB table per frame behind the maps)
  kF16Arith,      // Camera16 f16 map + run_scratch_out
  kU16Map,        // Camera32 u16 fixed-point map (Sweep::kStore) + run_map16_out + the gated exact sweeps
  kU16Turned,     // Camera32 u16 fixed-point map + the gated exact sweeps + run_out_transposed
};
struct ReinhardPlan {
  ReinhardForm form;
  size_t map_bytes, bytes;    // 0 for kNone and kExact
};
ReinhardPlan reinhard_plan(const b200isp_fused_params& p, const IspConsts& k, int n_frames);

// The sweeps over the packed frames fp.in (fused_inst.cu, one translation unit per group so that the kernel variants compile
// in parallel).  rows_per_task <= 0: auto_rows_per_task2.
enum class Sweep {
  kRgb,           // EpiRgb2: the ISP dtype's float RGB (TM_NONE)
  kLinear,        // EpiLinear2
  kReinhard,      // EpiReinhard2: the write sweep of the exact form, max from ws->frame_max
  kMax,           // EpiReinhardMax2: the max sweep of the exact form
  kStore,         // EpiReinhardMax2<STORE>: the max sweep that also writes the map to fp.out (Camera32: color_adapt == 0)
  kMaxGated,      // the exact max sweep (into ws->frame_max2) and write sweep of the frames the u16 map declined
  kReinhardGated, //   (Camera32 -> u8, color_adapt == 0, standard layout; k.gate == 1): CTAs that exit at once otherwise
};
template <bool CAM16, typename OutT>     // kRgb, kLinear, kReinhard writing OutT
int run_out_sweep(Sweep sw, const FramePtrs& fp, const IspConsts& k, int nframes, int rows_per_task, cudaStream_t s);
template <bool CAM16>                    // kMax, kStore
int run_max_sweep(Sweep sw, const FramePtrs& fp, const IspConsts& k, int nframes, int rows_per_task, cudaStream_t s);
int run_gated_sweep(Sweep sw, const FramePtrs& fp, const IspConsts& k, int nframes, int rows_per_task, cudaStream_t s);

// The normalise passes of the one-sweep forms (normalise.cu): the maps sc.out -> the outputs fp.out, frame maxima from k.ws.
constexpr int kLutBytes = 65536;         // kF16Table: one u8 per f16 pattern and frame
// kF16Arith, and kResizeMap on Camera16: n_elems values per frame, % 8 == 0; at most max_ctas CTAs per frame
int run_scratch_out(const FramePtrs& sc, const FramePtrs& fp, int n_frames, long long n_elems, int out_dtype, float gamma,
                    const Workspace* ws, int max_ctas, cudaStream_t s);
int run_lut_pass(const FramePtrs& sc, const FramePtrs& fp, int n_frames, long long n_elems, uint8_t* lut, float gamma, const Workspace* ws,
                 cudaStream_t s);                                       // kF16Table; lut = n_frames x kLutBytes behind the maps
int run_scratch_yuv(const FramePtrs& sc, const FramePtrs& fp, int n_frames, const IspConsts& k, cudaStream_t s);        // kF16Yuv
int run_map16_out(const FramePtrs& sc, const FramePtrs& fp, int n_frames, const IspConsts& k, cudaStream_t s);          // kU16Map
int run_out_transposed(bool cam16, const FramePtrs& sc, const FramePtrs& fp, int n_frames, const IspConsts& k, cudaStream_t s);
int run_resize_normalise(const FramePtrs& sc, const FramePtrs& fp, int n_frames, long long n_elems, bool cam16, int out_dtype,
                         float gamma, const Workspace* ws, cudaStream_t s);     // kResizeMap: any n_elems, the ISP dtype's map

}  // namespace isp
