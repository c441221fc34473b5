// Bilinear down-scaling fused into the pair-engine sweep (stream2.cuh): BASELINE configs[4], "full ISP + resize".
//
// At scales around 1/2 almost every demosaiced pixel is a bilinear tap of some output pixel, so the cheapest
// way to produce the taps is the sweep itself (22 instructions per input pixel for decode + Malvar, everything
// shared between neighbours) -- the per-output-pixel gather of resize_isp.cuh costs ~700 instructions per OUTPUT
// pixel = 150 per input pixel (profiles/r02_resize_gather_ncu.txt) because nothing is shared.  Here
//   * a task = (frame, chunk of OUTPUT rows, 256-pixel strip); its source rows run from the first tap row of its
//     first output row to the second tap row of its last one, so a task never needs a row of another task;
//   * emit(row) converts the row to ISP RGB (CCM, clamp, ISP-dtype rounding: what the reference resizes,
//     camera_isp.py:371-373) and parks it in a per-warp ring of two rows in shared memory;
//   * when the parked row is the lower tap row of the pending output row, the warp produces that output row: every
//     lane takes output columns co0 + lane, + 32, ..., reads its 2 x 2 taps from the ring, mixes vertically then
//     horizontally with the reference's per-operation rounding (interpolate.py:59-66, resize.cu mixf), rounds to the
//     ISP dtype, tone-maps and stores -- consecutive lanes write consecutive output pixels;
//   * index arithmetic is bit-identical to interpolate.py:60-61 (f32 division, truncation, clamp to the edge).
// A strip owns the output columns whose left tap AND right tap lie inside it; the one output column per strip
// boundary whose taps straddle two strips ("orphan") is produced afterwards by the gather front end
// (resize_isp.cuh), which is also the metering sampler and the path for up-scaling.
#pragma once
#include "resize_isp.cuh"

namespace isp {

enum { RZ_RGB = 0, RZ_LINEAR = 1, RZ_RSTORE = 2 };

template <typename T> __device__ __forceinline__ void store3(T* dst, const float (&y)[3]) {
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    if constexpr (DT<T>::is_int) dst[c] = (T)(Quant<T>::q(y[c]) & (uint32_t)DT<T>::scale);
    else dst[c] = cast_from_f32<T>(y[c]);
  }
}

// interpolate.py:60-61 for one axis
__device__ __host__ __forceinline__ int tap_of(int o, float scale) { return (int)((float)o / scale); }

// smallest output index whose left tap is >= x (scale <= 1: tap_of is strictly increasing)
__device__ __host__ inline int first_out_with_tap_ge(int x, float scale, int n_out) {
  int g = (int)((float)x * scale);
  if (g < 0) g = 0;
  if (g > n_out) g = n_out;
  while (g > 0 && tap_of(g - 1, scale) >= x) --g;
  while (g < n_out && tap_of(g, scale) < x) ++g;
  return g;
}

// tone-map stage of one resized pixel, shared by the sweep epilogue and the gather kernel (orphans, up-scaling)
template <bool CAM16, int MODE, typename OutT>
struct ResizeTone {
  LinearConsts lc;
  ReinhardConsts rc;
  __device__ __forceinline__ void init(const IspConsts& k, int frame) {
    if constexpr (MODE == RZ_LINEAR) lc = linear_consts(k.metrics, k.gamma);
    if constexpr (MODE == RZ_RSTORE) rc = reinhard_consts(k, frame, false);
  }
  // returns max(p) for RZ_RSTORE (f32 p before the dtype rounding, camera_isp.py:213), 0 otherwise
  __device__ __forceinline__ float apply(const float (&rgb)[3], OutT* dst) const {
    if constexpr (MODE == RZ_RGB) {
      store3<OutT>(dst, rgb);
      return 0.f;
    } else if constexpr (MODE == RZ_LINEAR) {
      float y[3];
      if (lc.has_gamma) linear_px<true>(lc, rgb, y); else linear_px<false>(lc, rgb, y);
      store3<OutT>(dst, y);
      return 0.f;
    } else {
      float sc[3], p[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) sc[c] = __fmul_rn(__fsub_rn(rgb[c], rc.p.bmin), rc.p.inv_range);     // exact near x == min
      if (rc.ca0) reinhard_map_fast<true>(rc.p, sc, p); else reinhard_map_fast<false>(rc.p, sc, p);
      store3<OutT>(dst, p);                                   // stored as the ISP dtype (camera_isp.py:211)
      return fmaxf(p[0], fmaxf(p[1], p[2]));
    }
  }
};

// two resized pixels at once (f32x2 lanes = output columns co and co + 32 of one lane): the Reinhard map of the common
// case (color_adapt == 0) stays packed; `b_ok` = the second pixel exists
template <bool CAM16, int MODE, typename OutT>
__device__ __forceinline__ float resize_tone2(const ResizeTone<CAM16, MODE, OutT>& t, const f2 (&rgb)[3], OutT* dst_a, OutT* dst_b, bool b_ok) {
  if constexpr (MODE == RZ_RSTORE) {
    if (t.rc.ca0) {
      f2 n[3], r;
      reinhard_nr2(t.rc, rgb, bc(1.0f), n, r);
      float pa[3], pb[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) upk(mul2(n[c], r), pa[c], pb[c]);
      store3<OutT>(dst_a, pa);
      float m = fmaxf(pa[0], fmaxf(pa[1], pa[2]));
      if (b_ok) { store3<OutT>(dst_b, pb); m = fmaxf(m, fmaxf(pb[0], fmaxf(pb[1], pb[2]))); }
      return m;
    }
  }
  float a[3], b[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) upk(rgb[c], a[c], b[c]);
  float m = t.apply(a, dst_a);
  if (b_ok) m = fmaxf(m, t.apply(b, dst_b));
  return m;
}

template <bool CAM16, int MODE, typename OutT>
struct EpiResize2 {
  FramePtrs fp;              // .out = output (RZ_RSTORE: scratch) frames, (Ho, Wo, 3) OutT
  IspConsts k;
  int Ho, Wo;
  float scale_r, scale_c;
  static constexpr int kRowWords = 32 * 24;              // 256 pixels x RGB as f32
  static constexpr int kMaxCols = 264;                   // output columns of one strip (scale <= 1: at most 257)
  static constexpr int kStageWords = 2 * kRowWords + 2 * kMaxCols;   // ring of two rows + the column table, per warp
  static constexpr bool kSplitEdge = false;
  static constexpr bool kCompactLoop = true;

  struct State {
    ResizeTone<CAM16, MODE, OutT> tone;
    OutT* out;
    float* ring;
    int lane, edge, col0;
    int ro, ro_end, rb;      // pending output row, end of the task's output rows, lower tap row of the pending row
    int co0, co1;            // output columns owned by this strip
    float mx;
  };

  __device__ __forceinline__ int lower_tap(int ro) const { return min(tap_of(ro, scale_r) + 1, k.H - 1); }

  __device__ __forceinline__ void init(State& st, int frame, int tcol, const WarpCtx& wc, int ro0, int ro1, bool last_strip) const {
    st.tone.init(k, frame);
    st.out = reinterpret_cast<OutT*>(fp.out[frame]);
    st.ring = reinterpret_cast<float*>(wc.stage);
    st.lane = wc.lane;
    st.edge = edge_bits(tcol, k.W);
    st.col0 = wc.tcol0 * 8;
    st.ro = ro0; st.ro_end = ro1;
    st.rb = lower_tap(ro0);
    st.co0 = first_out_with_tap_ge(st.col0, scale_c, Wo);
    st.co1 = last_strip ? Wo : first_out_with_tap_ge(st.col0 + 255, scale_c, Wo);      // tap col0 + 255 straddles: orphan
    st.co1 = min(st.co1, st.co0 + kMaxCols);
    st.mx = 0.f;
    // column table of the strip (the same for every output row of the task): left tap offset and fraction
    // (interpolate.py:60-61 in f32), so that the per-pixel loop carries no division
    int* tab = reinterpret_cast<int*>(st.ring + 2 * kRowWords);
    for (int co = st.co0 + st.lane; co < st.co1; co += 32) {
      const float pc = __fdiv_rn((float)co, scale_c);
      const int c1 = (int)pc;
      tab[2 * (co - st.co0)] = 3 * (c1 - st.col0) | ((c1 + 1 <= k.W - 1 ? 3 : 0) << 16);      // tap offset | right-tap step
      tab[2 * (co - st.co0) + 1] = __float_as_int(__fsub_rn(pc, (float)c1));
    }
    __syncwarp();
  }
  __device__ __forceinline__ bool fast_kinds_ok(const State&) const { return true; }

  // one output row from the two parked rows
  __device__ __forceinline__ void produce(State& st, int ro) const {
    const float pr = __fdiv_rn((float)ro, scale_r);
    const int r1 = (int)pr;
    const float fr = __fsub_rn(pr, (float)r1), gr = __fsub_rn(1.0f, fr);
    const float* A = st.ring + (min(r1, k.H - 1) & 1) * kRowWords;
    const float* B = st.ring + (min(r1 + 1, k.H - 1) & 1) * kRowWords;
    OutT* orow = st.out + (size_t)ro * Wo * 3;
    float mx = st.mx;
    const int2* tab = reinterpret_cast<const int2*>(st.ring + 2 * kRowWords);
    // two output pixels per iteration (columns co and co + 32): the mixes stay SCALAR __fmul_rn / __fadd_rn -- ptxas contracts
    // mul.rn.f32x2 + add.rn.f32x2 into FFMA2 (the rounding modifier is mandatory on the packed forms, so it does not protect
    // them), which breaks the reference's per-operation rounding (interpolate.py:62-66; caught by the bit-exactness test) --
    // and the tone map that follows runs packed on the pair
    for (int co = st.co0 + st.lane; co < st.co1; co += 64) {
      const bool b_ok = co + 32 < st.co1;
      const int2 e2[2] = {tab[co - st.co0], tab[(b_ok ? co + 32 : co) - st.co0]};
      float px[2][3];
#pragma unroll
      for (int l = 0; l < 2; ++l) {
        const float fc = __int_as_float(e2[l].y), gc = __fsub_rn(1.0f, fc);
        const int ia = e2[l].x & 0xFFFF, ib = ia + (e2[l].x >> 16);
#pragma unroll
        for (int c = 0; c < 3; ++c) {     // mix along dim 0 first, then dim 1; every operation rounded
          const float y1 = __fadd_rn(__fmul_rn(A[ia + c], gr), __fmul_rn(B[ia + c], fr));
          const float y2 = __fadd_rn(__fmul_rn(A[ib + c], gr), __fmul_rn(B[ib + c], fr));
          px[l][c] = __fadd_rn(__fmul_rn(y1, gc), __fmul_rn(y2, fc));
        }
      }
      f2 rgb[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {       // cast to the ISP dtype
        if constexpr (CAM16) {
          const __half2 h = __floats2half2_rn(px[0][c], px[1][c]);
          rgb[c] = pk(__low2float(h), __high2float(h));
        } else {
          rgb[c] = pk(px[0][c], px[1][c]);
        }
      }
      mx = fmaxf(mx, resize_tone2<CAM16, MODE, OutT>(st.tone, rgb, orow + (size_t)co * 3, orow + (size_t)(co + 32) * 3, b_ok));
    }
    st.mx = mx;
  }

  template <bool BROW, bool GFIRST, int KIND>
  __device__ __forceinline__ void emit(State& st, int row, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4]) const {
    float rgb[8][3];
    if constexpr (KIND == K_GENERAL) {
      Vals24 x;
      raw_with_frame<CAM16, BROW, GFIRST, KIND>(R, G, B, row, k.H, st.edge, k.kbase, x);
#pragma unroll
      for (int q = 0; q < 8; ++q) raw_to_rgb<CAM16>(k, &x.v[3 * q], rgb[q]);
    } else {
      f2 X[4][3];
      pairs_to_raw2<CAM16, BROW, GFIRST>(R, G, B, X);
      if (KIND == K_EDGE && st.edge) patch_cols_pairs<BROW, GFIRST>(X, st.edge, k.kbase);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        f2 c2[3];
        raw2_to_rgb2<CAM16>(k, X[j], c2);
#pragma unroll
        for (int c = 0; c < 3; ++c) upk(c2[c], rgb[j][c], rgb[j + 4][c]);
      }
    }
    __syncwarp();                                   // the previous output row has been read out of this slot
    float4* slot = reinterpret_cast<float4*>(st.ring + (row & 1) * kRowWords + 24 * st.lane);
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      const float* f = &rgb[0][0] + 4 * i;
      slot[i] = make_float4(f[0], f[1], f[2], f[3]);
    }
    __syncwarp();
    while (st.ro < st.ro_end && st.rb == row) {     // warp-uniform
      produce(st, st.ro);
      ++st.ro;
      st.rb = lower_tap(st.ro);
    }
  }

  __device__ __forceinline__ void finish(State& st, int frame, int lane, bool task_ok) const {
    if constexpr (MODE == RZ_RSTORE) {
      const float m = warp_max(st.mx);
      if (lane == 0 && task_ok && m > 0.f)
        atomicMax(reinterpret_cast<unsigned int*>(&k.ws->frame_max[frame]), __float_as_uint(m));
    }
  }
};

// task table of the resizing sweep: interior chunks of OUTPUT rows + one top and one bottom border task per strip
struct ResizeTasks {
  StreamGeom g;
  int out_rows_per_task, nchunks;
  int ro_top;          // output rows [0, ro_top) touch source rows 0 / 1 (K_GENERAL)
  int ro_bot;          // output rows [ro_bot, Ho) touch source rows H-2 / H-1 (K_GENERAL)
  int Ho;
  float scale_r;
  long long interior_tasks, total_tasks;
};

inline ResizeTasks make_resize_tasks(int H, int W, int nframes, int Ho, float scale_r, int out_rows_per_task) {
  ResizeTasks t;
  t.g = make_geom(H, W, nframes, 24);
  t.Ho = Ho; t.scale_r = scale_r;
  t.ro_top = first_out_with_tap_ge(2, scale_r, Ho);
  t.ro_bot = first_out_with_tap_ge(H - 3, scale_r, Ho);          // lower tap = tap + 1 >= H - 2
  if (t.ro_bot < t.ro_top) t.ro_bot = t.ro_top;
  if (out_rows_per_task <= 0) out_rows_per_task = 12;
  t.out_rows_per_task = out_rows_per_task;
  const int interior = t.ro_bot - t.ro_top;
  t.nchunks = (interior + out_rows_per_task - 1) / out_rows_per_task;
  t.interior_tasks = (long long)nframes * t.nchunks * t.g.warps_per_row;
  t.total_tasks = t.interior_tasks + (long long)nframes * 2 * t.g.warps_per_row;
  return t;
}

template <int PATTERN, bool BL, class Loader, class Epi>
__global__ void __launch_bounds__(ISP_S2_THREADS, ISP_S2_MINBLOCKS) stream2_resize_kernel(const Loader ld, const Epi epi, const ResizeTasks rt) {
  constexpr bool BROW0 = (PATTERN == B200ISP_GBRG || PATTERN == B200ISP_BGGR);
  constexpr bool GFIRST0 = (PATTERN == B200ISP_GRBG || PATTERN == B200ISP_GBRG);
  const StreamGeom& g = rt.g;
  const int lane = threadIdx.x & 31;
  long long task = (long long)blockIdx.x * kS2Warps + (threadIdx.x >> 5);
  bool task_ok = task < rt.total_tasks;
  if (!task_ok) task = 0;
  const bool border = task >= rt.interior_tasks;
  int strip, frame, ro0, ro1;
  if (!border) {
    strip = (int)(task % g.warps_per_row);
    const long long t2 = task / g.warps_per_row;
    const int chunk = (int)(t2 % rt.nchunks);
    frame = (int)(t2 / rt.nchunks);
    ro0 = rt.ro_top + chunk * rt.out_rows_per_task;
    ro1 = min(ro0 + rt.out_rows_per_task, rt.ro_bot);
  } else {
    const long long t = task - rt.interior_tasks;
    strip = (int)(t % g.warps_per_row);
    const long long t2 = t / g.warps_per_row;
    frame = (int)(t2 >> 1);
    ro0 = (t2 & 1) ? rt.ro_bot : 0;
    ro1 = (t2 & 1) ? rt.Ho : rt.ro_top;
  }
  if (ro0 >= ro1) task_ok = false;                           // empty border task
  const int tcol = min(strip * 32 + lane, g.ntcols - 1);

  __shared__ __align__(16) uint32_t stage[kS2Warps][Epi::kStageWords];
  WarpCtx wc;
  wc.lane = lane;
  wc.tcol0 = strip * 32;
  wc.nvalid = min(32, g.ntcols - strip * 32);
  wc.stage = stage[threadIdx.x >> 5];

  typename Epi::State st;
  epi.init(st, frame, tcol, wc, ro0, max(ro1, ro0), strip == g.warps_per_row - 1);
  if (task_ok) {
    // source rows: first tap row of the first output row (rounded down to even) .. lower tap row of the last one
    const int rs = min(tap_of(ro0, rt.scale_r), g.H - 1) & ~1;
    const int re = min((min(tap_of(ro1 - 1, rt.scale_r) + 1, g.H - 1) + 2) & ~1, g.H);
    if (border) stream2_rows<BROW0, GFIRST0, K_GENERAL, BL>(ld, epi, st, g, frame, tcol, rs, re);
    else stream2_rows<BROW0, GFIRST0, K_EDGE, BL>(ld, epi, st, g, frame, tcol, rs, re);
  }
  epi.finish(st, frame, lane, task_ok);
}

// the orphan columns (one per inner strip boundary and output row) through the gather front end
template <bool CAM16, int MODE, typename OutT>
__global__ void __launch_bounds__(128) resize_orphans_kernel(const ResizeSrc<CAM16> src, const FramePtrs outs, int nbound) {
  const int ro = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y, frame = blockIdx.z;
  const IspConsts& k = src.k;
  float mx = 0.f;
  if (ro < src.Ho && b < nbound) {
    const int x = 256 * b + 255;                               // last column of strip b; the right tap is in strip b + 1
    const int co = first_out_with_tap_ge(x, src.scale_c, src.Wo);
    if (co < src.Wo && tap_of(co, src.scale_c) == x) {
      ResizeTone<CAM16, MODE, OutT> tone;
      tone.init(k, frame);
      float rgb[3];
      src.pixel(frame, ro, co, rgb);
      mx = tone.apply(rgb, reinterpret_cast<OutT*>(outs.out[frame]) + ((size_t)ro * src.Wo + co) * 3);
    }
  }
  if constexpr (MODE == RZ_RSTORE) {
    mx = warp_max(mx);
    if ((threadIdx.x & 31) == 0 && mx > 0.f) atomicMax(reinterpret_cast<unsigned int*>(&k.ws->frame_max[frame]), __float_as_uint(mx));
  }
}

}  // namespace isp
