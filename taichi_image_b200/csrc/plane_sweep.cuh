// Stand-alone bayer_to_rgb (reference: bayer.py:114-190) on the pair engine of stream2.cuh: typed CFA planes in,
// interleaved RGB of the same dtype out -- BASELINE configs[3] (round-trip sweep at 8K).  Replaces the first,
// scalar streaming engine + its border kernel (r01: u8 31.5 %, u16 60.7 %, f32 54.8 % of the measured HBM peak at 8K,
// issue-bound at 41 instructions per pixel).
//
// Loaders (Loader2 concept of stream2.cuh).  Integer samples are decoded WITHOUT an int->float conversion by dropping
// their bits into the mantissa of a power of two (u8: one PRMT -> 2^15 + v; u16 / i16: shift + LOP3 -> 2^16 + v,
// i16 offset by 2^15 first); every filter sums to 16, so the x16 sums come out as 16 * bias + S exactly (all partial
// sums stay below 2^24) and the bias folds into the epilogue's constant.  The "zero sample" of rows / columns outside
// the image is the bias itself.
//
// Epilogue.  The reference computes  c = S / (in_scale * t);  [c = M c];  clamp(c, 0, 1);  trunc(c * out_scale)  with
// t = the in-bounds weight sum (16 in the interior).  Integer planes without CCM take the proven integer identity
// clamp(floor(S / t), 0, scale) (tests/test_host_cpu.py::test_integer_demosaic_equals_floor_division): one FFMA2.RZ
// against 2^23 (floor, bias removal and the /16 in one instruction) + an integer clamp on the float's bits.  Everything
// else (float planes, CCM, the pixels of the 2-pixel image frame) runs the literal chain with IEEE division.
#pragma once
#include "stream2.cuh"
#include "border_fix.cuh"
#include "pixel_ops.cuh"
#include <stdlib.h>

namespace isp {

__device__ __forceinline__ int plane_edge_bits(int tcol, int ntcols) { return (tcol == 0 ? 1 : 0) | (tcol == ntcols - 1 ? 2 : 0); }

template <typename T> struct PlaneLoader2;

// ---------------------------------------------------------------- u8: 8 pixels = 2 words, halo = upper / lower half of the neighbours
template <> struct PlaneLoader2<uint8_t> {
  const uint8_t* base;
  int pitch_words;                              // W / 4
  static constexpr uint32_t kRowMask = 1u;
  static constexpr float kBias = 32768.f;       // a sample is decoded as 2^15 + v
  struct Raw { uint32_t w[4]; };
  struct Cursor { const uint32_t* p; bool left, right, pf; };
  __device__ __forceinline__ ptrdiff_t pitch() const { return pitch_words; }
  template <int KIND> __device__ __forceinline__ void open(Cursor& c, int, int tcol, const StreamGeom& g) const {
    c.p = reinterpret_cast<const uint32_t*>(base) + 2 * tcol;
    c.left = KIND == K_CORE || tcol > 0;
    c.right = KIND == K_CORE || tcol < g.ntcols - 1;
    c.pf = (threadIdx.x & 15) == 0;              // 8 bytes per lane: lanes 0 and 16 touch the two 128-byte lines of the strip
  }
  template <int KIND> __device__ __forceinline__ void fetch(const Cursor& c, const uint32_t* p, Raw& raw) const {
    if (KIND == K_CORE || c.left) raw.w[0] = __ldg(p - 1);
    raw.w[1] = __ldg(p);
    raw.w[2] = __ldg(p + 1);
    if (KIND == K_CORE || c.right) raw.w[3] = __ldg(p + 2);
  }
  __device__ __forceinline__ void prefetch(const Cursor& c, const uint32_t* p) const {
    if (c.pf) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
  }
  template <int B> static __device__ __forceinline__ float dec(uint32_t w) {      // byte B of w -> 2^15 + v: bytes [0, v, 0, 0x47]
    return __uint_as_float(__byte_perm(w, 0x47000000u, 0x7604u | (B << 4)));
  }
  template <int KIND> __device__ __forceinline__ void decode(const Cursor& c, const Raw& raw, uint32_t m, f2 (&P)[8]) const {
    float v[12];
    v[0] = dec<2>(raw.w[0]); v[1] = dec<3>(raw.w[0]);
    v[2] = dec<0>(raw.w[1]); v[3] = dec<1>(raw.w[1]); v[4] = dec<2>(raw.w[1]); v[5] = dec<3>(raw.w[1]);
    v[6] = dec<0>(raw.w[2]); v[7] = dec<1>(raw.w[2]); v[8] = dec<2>(raw.w[2]); v[9] = dec<3>(raw.w[2]);
    v[10] = dec<0>(raw.w[3]); v[11] = dec<1>(raw.w[3]);
    if constexpr (KIND != K_CORE) {
      const bool row_ok = KIND != K_GENERAL || m != 0;
      if (!(row_ok && c.left)) { v[0] = kBias; v[1] = kBias; }
      if (!(row_ok && c.right)) { v[10] = kBias; v[11] = kBias; }
      if (!row_ok) {
#pragma unroll
        for (int j = 2; j < 10; ++j) v[j] = kBias;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) P[i] = pk(v[i], v[i + 4]);
  }
};

// ---------------------------------------------------------------- u16 / i16 / f16: 8 pixels = one 16-byte vector, halo = one word per side
template <typename T> struct PlaneLoader16x {
  const T* base;
  int pitch_words;                              // W / 2
  static constexpr uint32_t kRowMask = 1u;
  static constexpr bool kInt = DT<T>::is_int;
  static constexpr bool kSigned = std::is_same<T, int16_t>::value;
  static constexpr float kBias = kInt ? (kSigned ? 98304.f : 65536.f) : 0.f;      // 2^16 + v (i16: v offset by 2^15 first)
  struct Raw { uint32_t w[6]; };
  struct Cursor { const uint32_t* p; bool left, right, pf; };
  __device__ __forceinline__ ptrdiff_t pitch() const { return pitch_words; }
  template <int KIND> __device__ __forceinline__ void open(Cursor& c, int, int tcol, const StreamGeom& g) const {
    c.p = reinterpret_cast<const uint32_t*>(base) + 4 * tcol;
    c.left = KIND == K_CORE || tcol > 0;
    c.right = KIND == K_CORE || tcol < g.ntcols - 1;
    c.pf = (threadIdx.x & 7) == 0;               // 16 bytes per lane: every 8th lane starts a 128-byte line
  }
  template <int KIND> __device__ __forceinline__ void fetch(const Cursor& c, const uint32_t* p, Raw& raw) const {
    if (KIND == K_CORE || c.left) raw.w[0] = __ldg(p - 1);
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(p));
    raw.w[1] = q.x; raw.w[2] = q.y; raw.w[3] = q.z; raw.w[4] = q.w;
    if (KIND == K_CORE || c.right) raw.w[5] = __ldg(p + 4);
  }
  __device__ __forceinline__ void prefetch(const Cursor& c, const uint32_t* p) const {
    if (c.pf) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
  }
  template <int KIND> __device__ __forceinline__ void decode(const Cursor& c, const Raw& raw, uint32_t m, f2 (&P)[8]) const {
    float v[12];
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      uint32_t w = raw.w[i];
      if constexpr (kInt) {
        if constexpr (kSigned) w ^= 0x80008000u;
        v[2 * i] = biased_from_shifted(w << 7, 0x007FFF80u, 0x47800000u);          // low half -> 2^16 + v
        v[2 * i + 1] = biased_from_shifted(w >> 9, 0x007FFF80u, 0x47800000u);      // high half
      } else {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w));
        v[2 * i] = f.x; v[2 * i + 1] = f.y;
      }
    }
    if constexpr (KIND != K_CORE) {
      const bool row_ok = KIND != K_GENERAL || m != 0;
      if (!(row_ok && c.left)) { v[0] = kBias; v[1] = kBias; }
      if (!(row_ok && c.right)) { v[10] = kBias; v[11] = kBias; }
      if (!row_ok) {
#pragma unroll
        for (int j = 2; j < 10; ++j) v[j] = kBias;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) P[i] = pk(v[i], v[i + 4]);
  }
};
template <> struct PlaneLoader2<uint16_t> : PlaneLoader16x<uint16_t> {};
template <> struct PlaneLoader2<int16_t> : PlaneLoader16x<int16_t> {};
template <> struct PlaneLoader2<__half> : PlaneLoader16x<__half> {};

// ---------------------------------------------------------------- f32
template <> struct PlaneLoader2<float> {
  const float* base;
  int pitch_words;                              // W
  static constexpr uint32_t kRowMask = 1u;
  static constexpr float kBias = 0.f;
  struct Raw { float v[12]; };
  struct Cursor { const float* p; bool left, right, pf; };
  __device__ __forceinline__ ptrdiff_t pitch() const { return pitch_words; }
  template <int KIND> __device__ __forceinline__ void open(Cursor& c, int, int tcol, const StreamGeom& g) const {
    c.p = base + 8 * tcol;
    c.left = KIND == K_CORE || tcol > 0;
    c.right = KIND == K_CORE || tcol < g.ntcols - 1;
    c.pf = (threadIdx.x & 3) == 0;               // 32 bytes per lane: every 4th lane starts a 128-byte line
  }
  template <int KIND> __device__ __forceinline__ void fetch(const Cursor& c, const float* p, Raw& raw) const {
    if (KIND == K_CORE || c.left) { const float2 l = __ldg(reinterpret_cast<const float2*>(p - 2)); raw.v[0] = l.x; raw.v[1] = l.y; }
    const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p + 4));
    raw.v[2] = a.x; raw.v[3] = a.y; raw.v[4] = a.z; raw.v[5] = a.w;
    raw.v[6] = b.x; raw.v[7] = b.y; raw.v[8] = b.z; raw.v[9] = b.w;
    if (KIND == K_CORE || c.right) { const float2 r = __ldg(reinterpret_cast<const float2*>(p + 8)); raw.v[10] = r.x; raw.v[11] = r.y; }
  }
  __device__ __forceinline__ void prefetch(const Cursor& c, const float* p) const {
    if (c.pf) asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
  }
  template <int KIND> __device__ __forceinline__ void decode(const Cursor& c, const Raw& raw, uint32_t m, f2 (&P)[8]) const {
    float v[12];
#pragma unroll
    for (int j = 0; j < 12; ++j) v[j] = raw.v[j];
    if constexpr (KIND != K_CORE) {
      const bool row_ok = KIND != K_GENERAL || m != 0;
      if (!(row_ok && c.left)) { v[0] = 0.f; v[1] = 0.f; }
      if (!(row_ok && c.right)) { v[10] = 0.f; v[11] = 0.f; }
      if (!row_ok) {
#pragma unroll
        for (int j = 2; j < 10; ++j) v[j] = 0.f;
      }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) P[i] = pk(v[i], v[i + 4]);
  }
};

// ---------------------------------------------------------------- epilogue
template <typename T>
struct EpiDemosaic2 {
  T* out;
  int H, W;
  int ccm;                  // runtime (kernel-uniform) flag
  int kbase;                // 0: Malvar-He-Cutler, kBilinearBase: bilinear
  float m[9];
  static constexpr float kBias = PlaneLoader2<T>::kBias;
  static constexpr int kRowWords = 24 * (int)sizeof(T) / 4;
  static constexpr int kStageWords = 32 * kRowWords;
  static constexpr bool kSplitEdge = true;
  static constexpr bool kCompactLoop = true;
  struct State { T* out; WarpCtx wc; int edge; };
  __device__ __forceinline__ void init(State& st, int, int tcol, const WarpCtx& wc) const {
    st.out = out + 24 * wc.tcol0;
    st.wc = wc;
    st.edge = plane_edge_bits(tcol, (W + 7) / 8);
  }
  __device__ __forceinline__ void finish(State&, int, int, bool) const {}
  __device__ __forceinline__ bool fast_kinds_ok(const State&) const { return true; }

  // bit pattern of one output element in the low bits of a word (the row is packed from 24 such words)
  static __device__ __forceinline__ uint32_t bits_of(float x) {
    if constexpr (std::is_same<T, float>::value) return __float_as_uint(x);
    else if constexpr (std::is_same<T, __half>::value) return (uint32_t)__half_as_ushort(__float2half_rn(x));
    else return (uint32_t)(uint16_t)cast_from_f32<T>(x);
  }
  static __device__ __forceinline__ void pack_row(const uint32_t (&v)[24], uint32_t (&w)[24 * (int)sizeof(T) / 4]) {
    if constexpr (sizeof(T) == 1) {
#pragma unroll
      for (int i = 0; i < 6; ++i)
        w[i] = __byte_perm(__byte_perm(v[4 * i], v[4 * i + 1], 0x0040), __byte_perm(v[4 * i + 2], v[4 * i + 3], 0x0040), 0x5410);
    } else if constexpr (sizeof(T) == 2) {
#pragma unroll
      for (int i = 0; i < 12; ++i) w[i] = __byte_perm(v[2 * i], v[2 * i + 1], 0x5410);
    } else {
#pragma unroll
      for (int i = 0; i < 24; ++i) w[i] = v[i];
    }
  }

  // literal chain for one pixel: S = exact x16 sums (bias removed), t = in-bounds weight sums      bayer.py:150-155, :132-134
  __device__ __forceinline__ void literal_px(const float (&S)[3], const float* t, uint32_t* o) const {
    constexpr float is = DT<T>::scale, os = DT<T>::scale;
    float c0 = __fdiv_rn(S[0], __fmul_rn(is, t[0])), c1 = __fdiv_rn(S[1], __fmul_rn(is, t[1])), c2 = __fdiv_rn(S[2], __fmul_rn(is, t[2]));
    if (ccm) ccm_apply(m, c0, c1, c2);
    o[0] = bits_of(__fmul_rn(clamp01(c0), os));
    o[1] = bits_of(__fmul_rn(clamp01(c1), os));
    o[2] = bits_of(__fmul_rn(clamp01(c2), os));
  }

  // frame columns of an interior row (pixels 0, 1 of the first / 6, 7 of the last thread column): literal chain with the
  // in-bounds weight sums of their column class; o = the row's 24 element values
  template <bool BROW, bool GFIRST>
  __device__ __forceinline__ void patch_edge(int edge, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4], uint32_t (&o)[24]) const {
    using SS = SiteScale2<BROW, GFIRST>;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      if (q >= 2 && q < 6) continue;
      if ((q < 2 && (edge & 1)) || (q >= 6 && (edge & 2))) {
        const int j = q & 3;
        const float S[3] = {fmaf(q < 4 ? lo_of(R[j]) : hi_of(R[j]), SS::r(j), -16.f * kBias),
                            fmaf(q < 4 ? lo_of(G[j]) : hi_of(G[j]), SS::g(j), -16.f * kBias),
                            fmaf(q < 4 ? lo_of(B[j]) : hi_of(B[j]), SS::b(j), -16.f * kBias)};
        literal_px(S, c_border.t[site_kernel_of(BROW, SS::gsite(j)) + kbase][2][q < 2 ? q : q - 3], &o[3 * q]);
      }
    }
  }

  template <bool BROW, bool GFIRST, int KIND>
  __device__ __forceinline__ void emit(State& st, int row, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4]) const {
    using SS = SiteScale2<BROW, GFIRST>;
    uint32_t o[24];
    if constexpr (KIND == K_GENERAL) {
      // border rows (cold): every pixel through the literal chain with its own in-bounds weight sums
      const int rc = edge_class(row, H);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float s[3][2];
        upk(R[j], s[0][0], s[0][1]); upk(G[j], s[1][0], s[1][1]); upk(B[j], s[2][0], s[2][1]);
        const float sc[3] = {SS::r(j), SS::g(j), SS::b(j)};
        const int K = site_kernel_of(BROW, SS::gsite(j)) + kbase;
#pragma unroll
        for (int l = 0; l < 2; ++l) {
          const int q = j + 4 * l;
          const float S[3] = {fmaf(s[0][l], sc[0], -16.f * kBias), fmaf(s[1][l], sc[1], -16.f * kBias), fmaf(s[2][l], sc[2], -16.f * kBias)};
          literal_px(S, c_border.t[K][rc][col_class(q, st.edge)], o + 3 * q);
        }
      }
    } else {
      if (DT<T>::is_int && !ccm) {
        // clamp(floor(S / 16), 0, scale): floor, /16 and the bias removal in one RZ FMA against 1.5 * 2^23 (the sum stays
        // positive, so round-toward-zero IS floor, also for negative values); the integer is the float's bits minus the
        // magic's.  u8 / u16: the clamp rides on the saturating pack (cvt.pack.sat: two values per instruction) -- the
        // integer pipe, not instruction issue, bounded the first version (profiles/r02_plane_sweep_ncu.txt: 6.1 VIMNMX +
        // 4.1 PRMT of 30.9 instructions per pixel at half rate).
        constexpr float magic = 12582912.f - kBias;
        constexpr int kMagicBits = 0x4B400000;
        uint32_t n[24];             // signed values in two's complement
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const f2 q[3] = {fma2_rz(R[j], bc(SS::r(j) * 0.0625f), bc(magic)), fma2_rz(G[j], bc(SS::g(j) * 0.0625f), bc(magic)),
                           fma2_rz(B[j], bc(SS::b(j) * 0.0625f), bc(magic))};
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) {
            float a, b;
            upk(q[ch], a, b);
            n[3 * j + ch] = (uint32_t)(__float_as_int(a) - kMagicBits);
            n[3 * (j + 4) + ch] = (uint32_t)(__float_as_int(b) - kMagicBits);
          }
        }
        if (KIND == K_EDGE && st.edge) patch_edge<BROW, GFIRST>(st.edge, R, G, B, n);     // in-range values pass the saturation unchanged
        if constexpr (std::is_same<T, uint8_t>::value) {
          uint32_t w[6];
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            uint32_t lo2, w4;
            asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(lo2) : "r"(n[4 * i + 1]), "r"(n[4 * i]), "r"(0));
            asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(w4) : "r"(n[4 * i + 3]), "r"(n[4 * i + 2]), "r"(0));
            w[i] = __byte_perm(lo2, w4, 0x5410);
          }
          warp_store_row<kRowWords, KIND == K_CORE>(st.wc, st.out + (size_t)((unsigned)row * (unsigned)W) * 3, w);
          return;
        } else if constexpr (std::is_same<T, uint16_t>::value) {
          uint32_t w[12];
#pragma unroll
          for (int i = 0; i < 12; ++i) asm("cvt.pack.sat.u16.s32 %0, %1, %2;" : "=r"(w[i]) : "r"(n[2 * i + 1]), "r"(n[2 * i]));
          warp_store_row<kRowWords, KIND == K_CORE>(st.wc, st.out + (size_t)((unsigned)row * (unsigned)W) * 3, w);
          return;
        } else {
#pragma unroll
          for (int i = 0; i < 24; ++i) o[i] = (uint32_t)max(0, min((int)n[i], (int)DT<T>::scale));
          uint32_t w[kRowWords];
          pack_row(o, w);
          warp_store_row<kRowWords, KIND == K_CORE>(st.wc, st.out + (size_t)((unsigned)row * (unsigned)W) * 3, w);
          return;
        }
      } else {
        constexpr float is = DT<T>::scale;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float s[3][2];
          upk(R[j], s[0][0], s[0][1]); upk(G[j], s[1][0], s[1][1]); upk(B[j], s[2][0], s[2][1]);
          const float sc[3] = {SS::r(j), SS::g(j), SS::b(j)};
#pragma unroll
          for (int l = 0; l < 2; ++l) {
            float c[3];
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
              // S / (in_scale * 16): a power of two for the float planes (exact product), an IEEE division otherwise
              if constexpr (!DT<T>::is_int) c[ch] = s[ch][l] * (sc[ch] * 0.0625f);
              else c[ch] = __fdiv_rn(fmaf(s[ch][l], sc[ch], -16.f * kBias), is * 16.f);
            }
            if (ccm) ccm_apply(m, c[0], c[1], c[2]);
            uint32_t* p = o + 3 * (j + 4 * l);
            p[0] = bits_of(__fmul_rn(clamp01(c[0]), is));
            p[1] = bits_of(__fmul_rn(clamp01(c[1]), is));
            p[2] = bits_of(__fmul_rn(clamp01(c[2]), is));
          }
        }
      }
      if (KIND == K_EDGE && st.edge) patch_edge<BROW, GFIRST>(st.edge, R, G, B, o);
    }
    uint32_t w[kRowWords];
    pack_row(o, w);
    warp_store_row<kRowWords, KIND == K_CORE>(st.wc, st.out + (size_t)((unsigned)row * (unsigned)W) * 3, w);
  }
};

// host: one sweep over an (H, W) plane -> (H, W, 3); H even >= 4, W % 8 == 0, 16-byte aligned bases
template <typename T>
int run_demosaic_sweep(const void* bayer, void* rgb, int H, int W, int pattern, const float* ccm, bool bilinear, cudaStream_t s);

template <typename T>
int run_demosaic_sweep_impl(const void* bayer, void* rgb, int H, int W, int pattern, const float* ccm, bool bilinear, cudaStream_t s) {
  PlaneLoader2<T> ld;
  ld.base = (const T*)bayer;
  ld.pitch_words = W * (int)sizeof(T) / 4;
  EpiDemosaic2<T> epi;
  epi.out = (T*)rgb; epi.H = H; epi.W = W; epi.ccm = ccm != nullptr; epi.kbase = bilinear ? kBilinearBase : 0;
  for (int i = 0; i < 9; ++i) epi.m[i] = ccm ? ccm[i] : 0.f;
  // one frame per call: 16-row chunks (measured at 8K, profiles/r02_plane_sweep.txt: 12-16 rows best for u8 / u16 / f32,
  // 24+ rows lose 5-10 % to the tail of the last wave)
  const Stream2Geom g = make_geom2(H, W, 1, 16);
  int st = B200ISP_OK;
  ISP_DISPATCH_PATTERN(pattern, P, { st = launch_stream2<P>(ld, epi, g, s, "bayer_to_rgb", bilinear); });
  return st;
}

}  // namespace isp
