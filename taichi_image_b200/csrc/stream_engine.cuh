// Shared pieces of the streaming sweeps (stream2.cuh): task geometry, the scalar per-site Malvar-He-Cutler formulas
// (used by the metering samplers), the warp-cooperative row store and the pattern dispatch.
//
// History: this file used to hold the first, scalar register-window engine (41 instructions per pixel, r01); every
// sweep now runs on the packed-f32x2 pair engine of stream2.cuh, the scalar kernel is gone.
//
// Partial sums of the 13-tap filters (SURVEY 7.3 H1, tables of bayer.py:30-55 x16):
//   NS(c) = v[r-1][c]+v[r+1][c]   EW = v[r][c-1]+v[r][c+1]   NNSS = v[r-2][c]+v[r+2][c]
//   EEWW = v[r][c-2]+v[r][c+2]    D = NS(c-1)+NS(c+1)
//   R/B site:  own = 16C   G = 8C+4(NS+EW)-2(NNSS+EEWW)   opposite = 12C+4D-3(NNSS+EEWW)
//   G site:    G = 16C     colour with horizontal neighbours = 10C+8EW-2D-2EEWW+NNSS
//                          colour with vertical neighbours   = 10C+8NS-2D-2NNSS+EEWW
// The sums are exact for integer-valued inputs (|sum| < 2^24), so the evaluation order does not matter there.
#pragma once
#include "common.cuh"


namespace isp {

struct StreamGeom {
  int H, W;
  int ntcols;          // ceil(W / 8): thread columns per row
  int warps_per_row;   // ceil(ntcols / 32)
  int rows_per_task;   // even
  int nchunks;         // ceil(H / rows_per_task)
  int nframes;
  long long total_tasks;   // nframes * nchunks * warps_per_row (warp tasks)
};

inline StreamGeom make_geom(int H, int W, int nframes, int rows_per_task) {
  StreamGeom g;
  g.H = H; g.W = W;
  g.ntcols = (W + 7) / 8;
  g.warps_per_row = (g.ntcols + 31) / 32;
  if (rows_per_task <= 0) {
    // aim at >= ~6 waves of 16 warps on 148 SMs, keep the 4 halo rows <= ~12 % of the loads
    rows_per_task = 48;
    while (rows_per_task > 12 &&
           (long long)nframes * ((H + rows_per_task - 1) / rows_per_task) * g.warps_per_row < 6LL * 16 * kNumSMs)
      rows_per_task -= 12;
  }
  rows_per_task += rows_per_task & 1;
  g.rows_per_task = rows_per_task;
  g.nchunks = (H + rows_per_task - 1) / rows_per_task;
  g.nframes = nframes;
  g.total_tasks = (long long)nframes * g.nchunks * g.warps_per_row;
  return g;
}

// ---------------------------------------------------------------- per-site filter formulas (scaled)
// R/B site: own colour = C (x16), G = 4C + 2(NS+EW) - (NNSS+EEWW) (x2), opposite = 3C + D - 0.75(NNSS+EEWW) (x4)
__device__ __forceinline__ void malvar_csite(float C, float NS, float EW, float NNSS, float EEWW, float D,
                                             float& g2, float& opp4) {
  const float A = NS + EW, Bq = NNSS + EEWW;
  g2 = fmaf(4.f, C, fmaf(2.f, A, -Bq));
  opp4 = fmaf(-0.75f, Bq, fmaf(3.f, C, D));
}
// G site: G = C (x16), horizontal-neighbour colour = 5C - D + 4EW - EEWW + 0.5NNSS (x2), vertical likewise
__device__ __forceinline__ void malvar_gsite(float C, float NS, float EW, float NNSS, float EEWW, float D,
                                             float& h2, float& v2) {
  const float T = fmaf(5.f, C, -D);
  h2 = fmaf(0.5f, NNSS, fmaf(4.f, EW, T) - EEWW);
  v2 = fmaf(0.5f, EEWW, fmaf(4.f, NS, T) - NNSS);
}

// ---------------------------------------------------------------- warp-cooperative row store
// A lane owns 8 pixels x 3 channels = NW 32-bit words of an output row, i.e. a 4*NW-byte segment with a
// 4*NW-byte lane stride: stored straight from registers, every STG.128 would touch 32 scattered 16-byte
// pieces (half sectors) of twelve 128-byte lines.  Measured on B200 with the sweep's 1.5 B : 6 B traffic
// mix (profiles/r01_membench.txt) that shape tops out at ~3.9 TB/s, the same bytes written as whole
// contiguous 512-byte runs reach ~5.8 TB/s.  So each warp transposes the row through a private
// shared-memory stage (conflict-free for NW = 6 and 12) and writes it as consecutive 16-byte (8-byte when
// the row pitch is only 8-byte aligned: RGB8) chunks; only __syncwarp, no block barrier.
struct WarpCtx {
  int lane;
  int tcol0;            // first thread column of the warp's strip
  int nvalid;           // lanes of the strip that map to real thread columns (the others compute a clamped copy)
  uint32_t* stage;      // this warp's staging buffer, Epi::kStageWords words
};

// Output rows are written once and never re-read by the ISP: store them with the evict-first policy so that
// they do not push the packed input rows (which the metering pass has just pulled into the 126 MB L2 and the
// sweep is about to read) out of L2.
__device__ __forceinline__ void st_out(uint4* p, const uint4& v) { __stcs(p, v); }
__device__ __forceinline__ void st_out(uint2* p, const uint2& v) { __stcs(p, v); }
// the same store executed only where idx < n, as ONE predicated instruction: written in C (`if (idx < n) st_out(...)`) the
// compiler sinks the shared-memory load and the address arithmetic into the condition and branches over them -- BSSY + BRA +
// BSYNC per store, 9 instructions per row in every sweep without a K_CORE copy (ncu source view of the Reinhard map sweep)
__device__ __forceinline__ void st_out_lt(uint4* p, const uint4& v, int idx, int n) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.lt.s32 q, %5, %6;\n\t@q st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};\n\t}"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(idx), "r"(n) : "memory");
}
__device__ __forceinline__ void st_out_lt(uint2* p, const uint2& v, int idx, int n) {
  asm volatile("{\n\t.reg .pred q;\n\tsetp.lt.s32 q, %3, %4;\n\t@q st.global.cs.v2.u32 [%0], {%1, %2};\n\t}"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(idx), "r"(n) : "memory");
}

template <int NW, bool FULL = false>       // FULL: all 32 lanes map to real thread columns (no store predicates)
__device__ __forceinline__ void warp_store_row(const WarpCtx& wc, void* row_dst /* warp's first byte of the row */,
                                               const uint32_t (&w)[NW], int slot = -1 /* staging slot; default: the lane */) {
  constexpr int CW = (NW % 4 == 0) ? 4 : 2;     // words per chunk
  constexpr int PER_LANE = NW / CW;
  const int nchunks = wc.nvalid * PER_LANE;
  if (slot < 0) slot = wc.lane;
  __syncwarp();
  if constexpr (CW == 4) {
    uint4* s = reinterpret_cast<uint4*>(wc.stage);
#pragma unroll
    for (int i = 0; i < PER_LANE; ++i) s[PER_LANE * slot + i] = make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]);
    __syncwarp();
    uint4* d = reinterpret_cast<uint4*>(row_dst);
#pragma unroll
    for (int i = 0; i < PER_LANE; ++i) {
      const int idx = i * 32 + wc.lane;
      if constexpr (FULL) st_out(d + idx, s[idx]);
      else st_out_lt(d + idx, s[idx], idx, nchunks);        // s[idx] is always inside the stage
    }
  } else {
    uint2* s = reinterpret_cast<uint2*>(wc.stage);
#pragma unroll
    for (int i = 0; i < PER_LANE; ++i) s[PER_LANE * slot + i] = make_uint2(w[2 * i], w[2 * i + 1]);
    __syncwarp();
    uint2* d = reinterpret_cast<uint2*>(row_dst);
#pragma unroll
    for (int i = 0; i < PER_LANE; ++i) {
      const int idx = i * 32 + wc.lane;
      if constexpr (FULL) st_out(d + idx, s[idx]);
      else st_out_lt(d + idx, s[idx], idx, nchunks);
    }
  }
}

#define ISP_DISPATCH_PATTERN(p, P, ...)                                        \
  switch (p) {                                                                 \
    case B200ISP_RGGB: { constexpr int P = B200ISP_RGGB; __VA_ARGS__; break; } \
    case B200ISP_GRBG: { constexpr int P = B200ISP_GRBG; __VA_ARGS__; break; } \
    case B200ISP_GBRG: { constexpr int P = B200ISP_GBRG; __VA_ARGS__; break; } \
    case B200ISP_BGGR: { constexpr int P = B200ISP_BGGR; __VA_ARGS__; break; } \
    default: isp::set_error("unknown bayer pattern %d", (int)(p)); return B200ISP_E_ARG; \
  }

}  // namespace isp
