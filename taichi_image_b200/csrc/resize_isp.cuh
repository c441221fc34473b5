// Fused packed12 -> demosaic -> bilinear resize -> [tone map] gather for an ISP that resizes (BASELINE configs[4]).
//
// Reference order (camera_isp.py:371-373, :302-315; SURVEY Appendix C): demosaic the FULL frame, round it through
// the ISP dtype, resize it bilinearly (interpolate.py:19-34, :59-66: p = I / scale, p1 = trunc(p), clamp-to-edge
// taps, mix along dim 0 first, cast to the ISP dtype), THEN meter and tone-map the resized image.  The staged path
// materialises the full-resolution RGB (6 / 12 B per input pixel written and read back).  Here a thread owns one
// OUTPUT pixel: it decodes the 6 x 6 CFA window around its 2 x 2 bilinear taps straight from the packed rows
// (word loads + funnel shifts), demosaics exactly those four pixels (one of each CFA site; the two diagonals are
// evaluated as f32x2 pairs), applies CCM / clamp / ISP-dtype rounding, mixes with the reference's per-op rounding and
// tone-maps -- 1.5 B in + out bytes * (Wo Ho / W H) per input pixel, nothing else touches HBM.
// Taps on the 2-pixel image frame (or clamped beyond it) take the literal per-pixel path (pixel_ops.cuh).
//
//   TM_NONE   -> resized ISP-dtype RGB (= ISP.load_packed12 of a resizing ISP)
//   linear    -> quantised output in the same pass
//   Reinhard  -> pass A writes the un-normalised map p as the ISP dtype (the value the reference stores back,
//                camera_isp.py:211: exact for Camera16 AND Camera32) into an output-resolution scratch + frame max;
//                pass B normalises / gamma / quantises the scratch element-wise.
#pragma once
#include "fused_isp.cuh"

namespace isp {

template <bool CAM16>
struct ResizeSrc {
  FramePtrs fp;
  IspConsts k;
  int pitch_words;          // W * 3 / 8
  int Ho, Wo;
  float scale_r, scale_c;

  static __device__ __forceinline__ float dec(uint32_t shifted) {
    const float b = biased_from_shifted(shifted, 0x007FF800u, 0x3F800000u);       // 1 + v/4096, one LOP3
    if constexpr (CAM16) {
      constexpr float kk = 4096.f * kInv4095;
      return __half2float(__float2half_rn(fmaf(b, kk, -kk)));
    } else {
      return b;
    }
  }

  // six consecutive samples of one packed row from column cs (0 <= cs, cs + 6 <= W - 2): 72 bits from bit 12 cs
  __device__ __forceinline__ void row6(const uint32_t* __restrict__ row, int cs, float (&v)[6]) const {
    const int bit = 12 * cs;
    const uint32_t* p = row + (bit >> 5);
    const int sh = bit & 31;
    const uint32_t w0 = __ldg(p), w1 = __ldg(p + 1), w2 = __ldg(p + 2), w3 = __ldg(p + 3);
    const uint32_t a0 = __funnelshift_r(w0, w1, sh), a1 = __funnelshift_r(w1, w2, sh), a2 = __funnelshift_r(w2, w3, sh);
    v[0] = dec(a0 << 11);
    v[1] = dec(a0 >> 1);
    v[2] = dec(__funnelshift_r(a0, a1, 13));
    v[3] = dec(a1 << 7);
    v[4] = dec(a1 >> 5);
    v[5] = dec(__funnelshift_r(a1, a2, 17));
  }

  // scaled filter sums of one pair of same-class pixels -> ISP RGB pair.  sr / sb: per-lane scale of the R / B sums
  __device__ __forceinline__ void pair_rgb(f2 R, f2 G, f2 B, f2 sr, float sg, f2 sb, f2 (&rgb)[3]) const {
    constexpr float kn = 256.f * kInv4095;           // 4096 * f32(1/4095) / 16
    f2 x[3];
    if constexpr (CAM16) {
      x[0] = mul2(R, mul2(sr, bc(0.0625f))); x[1] = mul2(G, bc(sg * 0.0625f)); x[2] = mul2(B, mul2(sb, bc(0.0625f)));
    } else {
      x[0] = fma2(R, mul2(sr, bc(kn)), bc(-16.f * kn)); x[1] = fma2(G, bc(sg * kn), bc(-16.f * kn));
      x[2] = fma2(B, mul2(sb, bc(kn)), bc(-16.f * kn));
    }
    raw2_to_rgb2<CAM16>(k, x, rgb);
  }

  // ISP RGB of the 2 x 2 block with top-left pixel (r1, c1), all four pixels and their windows inside the image
  // interior (2 <= r1, r1 + 1 <= H - 3, likewise for the columns): S[i][j][ch]
  __device__ __forceinline__ void block_fast(int frame, int r1, int c1, float (&S)[2][2][3]) const {
    const uint32_t* base = reinterpret_cast<const uint32_t*>(fp.in[frame]) + (size_t)(r1 - 2) * pitch_words;
    float v[6][6];
#pragma unroll
    for (int a = 0; a < 6; ++a) row6(base + (size_t)a * pitch_words, c1 - 2, v[a]);
    // pair P = pixels (0,0) | (1,1), pair Q = pixels (0,1) | (1,0): the two pixels of a pair are the same site class
    f2 C[2], NS[2], EW[2], NNSS[2], EEWW[2], D[2];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const int i0 = 0, j0 = q, i1 = 1, j1 = 1 - q;           // lo pixel (i0, j0), hi pixel (i1, j1)
      C[q] = pk(v[2 + i0][2 + j0], v[2 + i1][2 + j1]);
      NS[q] = pk(v[1 + i0][2 + j0] + v[3 + i0][2 + j0], v[1 + i1][2 + j1] + v[3 + i1][2 + j1]);
      EW[q] = pk(v[2 + i0][1 + j0] + v[2 + i0][3 + j0], v[2 + i1][1 + j1] + v[2 + i1][3 + j1]);
      NNSS[q] = pk(v[i0][2 + j0] + v[4 + i0][2 + j0], v[i1][2 + j1] + v[4 + i1][2 + j1]);
      EEWW[q] = pk(v[2 + i0][j0] + v[2 + i0][4 + j0], v[2 + i1][j1] + v[2 + i1][4 + j1]);
      D[q] = pk((v[1 + i0][1 + j0] + v[3 + i0][1 + j0]) + (v[1 + i0][3 + j0] + v[3 + i0][3 + j0]),
                (v[1 + i1][1 + j1] + v[3 + i1][1 + j1]) + (v[1 + i1][3 + j1] + v[3 + i1][3 + j1]));
    }
    const bool brow0 = (k.pattern == B200ISP_GBRG || k.pattern == B200ISP_BGGR);
    const bool gfirst0 = (k.pattern == B200ISP_GRBG || k.pattern == B200ISP_GBRG);
    const bool brow_t = brow0 != ((r1 & 1) != 0);                          // row r1 carries B (not R)
    const bool gA = gfirst0 != (((r1 ^ c1) & 1) != 0);                     // pixel (0,0) is a G site -> so is (1,1)
    const bool bilinear = k.kbase != 0;                                    // kernel-uniform
    // lane scales of the colour sums: lo lane = row r1, hi lane = row r1 + 1
    const f2 sOwnOpp_R = pk(brow_t ? 4.f : 16.f, brow_t ? 16.f : 4.f), sOwnOpp_B = pk(brow_t ? 16.f : 4.f, brow_t ? 4.f : 16.f);
    f2 rgbP[3], rgbQ[3];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const bool gsite = (q == 0) == gA;
      // both site formulas in packed form (stream_engine.cuh malvar_csite / malvar_gsite; bilinear: stream2.cuh
      // bilinear_row2 in the x2 / x4 convention), the site class selects -- no divergent branch
      const f2 A = add2(NS[q], EW[q]), Bq = add2(NNSS[q], EEWW[q]);
      f2 g2, opp4, h2, v2;
      if (bilinear) {
        g2 = mul2(bc(2.f), A); opp4 = D[q];
        h2 = mul2(bc(4.f), EW[q]); v2 = mul2(bc(4.f), NS[q]);
      } else {
        g2 = fma2k(4.f, C[q], fma2k(2.f, A, mul2(bc(-1.f), Bq)));
        opp4 = fma2k(-0.75f, Bq, fma2k(3.f, C[q], D[q]));
        const f2 T = fma2k(5.f, C[q], mul2(bc(-1.f), D[q]));
        h2 = fma2k(0.5f, NNSS[q], add2(fma2k(4.f, EW[q], T), mul2(bc(-1.f), EEWW[q])));
        v2 = fma2k(0.5f, EEWW[q], add2(fma2k(4.f, NS[q], T), mul2(bc(-1.f), NNSS[q])));
      }
      // C site: R = brow ? opp4 : C, B = brow ? C : opp4 (x16 / x4), G = g2 (x2)
      // G site: R = brow ? v2 : h2, B = brow ? h2 : v2 (x2), G = C (x16);  brow = brow_t in the lo lane, !brow_t in the hi lane
      float cl, ch_, ol, oh, hl, hh, vl, vh;
      upk(C[q], cl, ch_); upk(opp4, ol, oh); upk(h2, hl, hh); upk(v2, vl, vh);
      const f2 Rc = pk(brow_t ? ol : cl, brow_t ? ch_ : oh), Bc = pk(brow_t ? cl : ol, brow_t ? oh : ch_);
      const f2 Rg = pk(brow_t ? vl : hl, brow_t ? hh : vh), Bg = pk(brow_t ? hl : vl, brow_t ? vh : hh);
      const f2 R = gsite ? Rg : Rc, B = gsite ? Bg : Bc, G = gsite ? C[q] : g2;
      const f2 sr = gsite ? bc(2.f) : sOwnOpp_R, sb = gsite ? bc(2.f) : sOwnOpp_B;
      pair_rgb(R, G, B, sr, gsite ? 16.f : 2.f, sb, q == 0 ? rgbP : rgbQ);
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      upk(rgbP[c], S[0][0][c], S[1][1][c]);
      upk(rgbQ[c], S[0][1][c], S[1][0][c]);
    }
  }

  // resized ISP-dtype RGB of output pixel (ro, co): interpolate.py:59-66 on the demosaiced image
  __device__ __forceinline__ void pixel(int frame, int ro, int co, float (&rgb)[3]) const {
    const float pr = __fdiv_rn((float)ro, scale_r), pc = __fdiv_rn((float)co, scale_c);
    const int r1 = (int)pr, c1 = (int)pc;
    const float fr = __fsub_rn(pr, (float)r1), fc = __fsub_rn(pc, (float)c1);
    float S[2][2][3];
    if (r1 >= 2 && r1 + 1 <= k.H - 3 && c1 >= 2 && c1 + 1 <= k.W - 3) {
      block_fast(frame, r1, c1, S);
    } else {
      const Packed12Src<CAM16> lit{fp, k.W * 3 / 2};
      const int ra = min(max(r1, 0), k.H - 1), rb = min(max(r1 + 1, 0), k.H - 1);
      const int ca = min(max(c1, 0), k.W - 1), cb = min(max(c1 + 1, 0), k.W - 1);
      isp_rgb_pixel<CAM16>(lit, k, frame, ra, ca, S[0][0]);
      isp_rgb_pixel<CAM16>(lit, k, frame, ra, cb, S[0][1]);
      isp_rgb_pixel<CAM16>(lit, k, frame, rb, ca, S[1][0]);
      isp_rgb_pixel<CAM16>(lit, k, frame, rb, cb, S[1][1]);
    }
    const float gr = __fsub_rn(1.0f, fr), gc = __fsub_rn(1.0f, fc);
#pragma unroll
    for (int c = 0; c < 3; ++c) {         // mix(a, b, t) = a * (1 - t) + b * t, every operation rounded (resize.cu mixf)
      const float y1 = __fadd_rn(__fmul_rn(S[0][0][c], gr), __fmul_rn(S[1][0][c], fr));
      const float y2 = __fadd_rn(__fmul_rn(S[0][1][c], gr), __fmul_rn(S[1][1][c], fr));
      rgb[c] = round_isp<CAM16>(__fadd_rn(__fmul_rn(y1, gc), __fmul_rn(y2, fc)));     // cast to the ISP dtype (scale ratio 1)
    }
  }
};

// metering sampler over the RESIZED image (camera_isp.py:168-170 on what _process_image returns)
template <bool CAM16>
struct ResizedSampler {
  ResizeSrc<CAM16> src;
  int stride, hs, ws_;
  // look-ahead / shared form under the previous sweep: this sampler is latency-bound (a 6 x 6 window per sample); 592 CTAs of
  // it displace the sweep for their whole 79 us, 296 CTAs cost 6.6 % less per step on cfg5 (profiles/r02_meter_grid_cap.txt)
  static constexpr int kSideGridCap = 2 * kNumSMs;
  __device__ __forceinline__ void sample(long long idx, float (&rgb)[3]) const {
    const int j = (int)(idx % ws_);
    const long long q = idx / ws_;
    const int i = (int)(q % hs);
    const int f = (int)(q / hs);
    src.pixel(f, i * stride, j * stride, rgb);
  }
};

inline bool resizes(const b200isp_fused_params& p) { return p.out_height > 0 && p.out_width > 0; }

template <bool CAM16>
inline ResizeSrc<CAM16> make_resize_src(const FramePtrs& fp, const IspConsts& k, const b200isp_fused_params& p) {
  return ResizeSrc<CAM16>{fp, k, p.width * 3 / 8, p.out_height, p.out_width, p.scale_r, p.scale_c};
}

// The resizing pass of p.tonemap into io.out (fused_resize.cu): the output images, or with Reinhard the output-resolution
// maps in the ISP dtype (ReinhardForm::kResizeMap) and the frame maxima in ws->frame_max.
int run_resize(const FramePtrs& io, int n_frames, const b200isp_fused_params& p, const IspConsts& k, cudaStream_t s);

}  // namespace isp
