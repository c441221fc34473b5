// Second-generation streaming engine: the Malvar-He-Cutler sweep of stream_engine.cuh evaluated with
// Blackwell's packed FP32 instructions (FFMA2 / FADD2 / FMUL2: two f32 lanes per issue slot).
//
// Why: the first engine is instruction-issue bound, not DRAM bound (profiles/r01_stream_kernel_ncu.txt:
// 41 warp-instructions per 32 pixels, 70 % issue-active, DRAM at 51 %); 24.5 of those 41 are scalar FP32.
// B200 keeps the FP32 lane rate for the packed forms (profiles/r01_membench.txt: 1.98 FFMA2 vs 3.86 FFMA
// warp-instructions / clk / SM) but each one takes a single issue slot, so the same math costs half the
// slots.  Operands that are equal in both lanes are free: ptxas encodes them as an immediate or as a
// broadcast 32-bit register (`FFMA2 R14, R8.F32x2.HI_LO, 3, R6.F32x2.HI_LO`).
//
// Mapping (as before): a thread owns 8 consecutive pixel columns and walks down the image, a warp owns a
// 256-pixel strip, a task is (frame, row chunk, strip).  New: the 12-column window row is held as eight
// register PAIRS  P[k] = (v[k], v[k+4]),  k = 0..7  (column c0-2+k in the low lane, c0+2+k in the high
// lane).  Pixel j (0..3) and pixel j+4 are the same CFA site type, so every partial sum and every filter
// formula of a row is evaluated once per pair:  48 packed instructions per 8 pixels instead of 94 scalar.
// Only columns 4..7 are needed in both lanes (4 extra decode LOP3 per row).
//
// The filters use the partial sums of stream_engine.cuh (NS, EW, NNSS, EEWW, D).  Signs are folded so no
// negation is ever needed; the epilogue multiplies by the (signed) SiteScale2 factor anyway:
//   R/B site:  own = C (x16)   G' = (NNSS+EEWW) - 2(NS+EW) - 4C (x -2)   opposite = 3C + D - 0.75(NNSS+EEWW) (x4)
//   G site:    G = C (x16)     H' = (D - 5C) - 4EW + EEWW - 0.5NNSS (x -2)   V' likewise with NS / NNSS <-> EW / EEWW
//
// Rows are addressed through incrementally advanced pointers; rows outside the image are never zero-filled by
// predicated loads: the load is clamped to a valid row and the DECODE mask of that row is 0, which yields
// the "zero sample" (biased 1.0f for Camera32, 0 for Camera16) the border arithmetic needs.  The same trick
// masks the halo columns of the first / last thread column.  Six full pair rows form the window.  The shipped
// loop is ONE copy of the two-row step that slides the window with register moves (+4 MOV per pixel): rotating the
// rows by unrolling the step three times needs no moves but triples the hot code, and the sweep is instruction-cache
// bound before it is move bound (DESIGN 6c: 3x unrolled 171 us vs single step 162 us on cfg2).  Epilogues with
// Epi::kCompactLoop == false (the small RGB epilogue of TM_NONE) keep the three-copy form outside K_GENERAL.
#pragma once
#include "stream_engine.cuh"

namespace isp {

// ---------------------------------------------------------------- packed f32x2 helpers (sm_100a)
typedef unsigned long long f2;
__device__ __forceinline__ f2 pk(float lo, float hi) { f2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ f2 bc(float x) { return pk(x, x); }
__device__ __forceinline__ void upk(f2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ float lo_of(f2 v) { float a, b; upk(v, a, b); return a; }
__device__ __forceinline__ float hi_of(f2 v) { float a, b; upk(v, a, b); return b; }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { f2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { f2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { f2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f2 fma2_rz(f2 a, f2 b, f2 c) { f2 r; asm("fma.rz.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f2 fma2k(float k, f2 b, f2 c) { return fma2(bc(k), b, c); }   // k equal in both lanes: immediate / broadcast

// (value * scale) = x16 filter sum, per output pair j (pixels j and j+4 of the thread's 8)
template <bool BROW, bool GFIRST>
struct SiteScale2 {
  static __host__ __device__ constexpr bool gsite(int j) { return ((j & 1) == 0) == GFIRST; }
  static __host__ __device__ constexpr float r(int j) { return gsite(j) ? -2.f : (BROW ? 4.f : 16.f); }
  static __host__ __device__ constexpr float g(int j) { return gsite(j) ? 16.f : -2.f; }
  static __host__ __device__ constexpr float b(int j) { return gsite(j) ? -2.f : (BROW ? 16.f : 4.f); }
};

// One output row.  All rows are full pair rows (index k = pair (column k, column k+4)); of the row two above
// only pairs 2..5 are read, of the row above and below pairs 1..6, of the row two below pairs 2..5.
template <bool BROW, bool GFIRST>
__device__ __forceinline__ void malvar_row2(const f2 (&m2)[8], const f2 (&m1)[8], const f2 (&z)[8], const f2 (&p1)[8],
                                            const f2 (&p2)[8], f2 (&R)[4], f2 (&G)[4], f2 (&B)[4]) {
  f2 ns[8];
#pragma unroll
  for (int i = 1; i <= 6; ++i) ns[i] = add2(m1[i], p1[i]);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const f2 C = z[j + 2];
    const f2 EW = add2(z[j + 1], z[j + 3]);
    const f2 EEWW = add2(z[j], z[j + 4]);
    const f2 NS = ns[j + 2];
    const f2 D = add2(ns[j + 1], ns[j + 3]);
    const f2 NNSS = add2(m2[j + 2], p2[j + 2]);
    if (!SiteScale2<BROW, GFIRST>::gsite(j)) {
      const f2 A = add2(NS, EW), Bq = add2(NNSS, EEWW);
      const f2 gn = fma2k(-4.f, C, fma2k(-2.f, A, Bq));
      const f2 opp = fma2k(-0.75f, Bq, fma2k(3.f, C, D));
      G[j] = gn;
      R[j] = BROW ? opp : C;
      B[j] = BROW ? C : opp;
    } else {
      const f2 Tn = fma2k(-5.f, C, D);
      const f2 hn = fma2k(-0.5f, NNSS, add2(fma2k(-4.f, EW, Tn), EEWW));
      const f2 vn = fma2k(-0.5f, EEWW, add2(fma2k(-4.f, NS, Tn), NNSS));
      G[j] = C;
      R[j] = BROW ? vn : hn;
      B[j] = BROW ? hn : vn;
    }
  }
}

// Bilinear demosaic (north_star extension) in the same output convention, so every epilogue is shared: with the
// 3 x 3 weights scaled by 4 the channel sums are again x16 sums whose weights total 16 (bias and frame
// renormalisation as for Malvar, border_fix.cuh K = 4..7):
//   R/B site:  own = C (x16)   G' = -2 (NS + EW) (x -2)   opposite = D (x4)
//   G site:    G = C (x16)     H' = -4 EW (x -2)          V' = -4 NS (x -2)
template <bool BROW, bool GFIRST>
__device__ __forceinline__ void bilinear_row2(const f2 (&m1)[8], const f2 (&z)[8], const f2 (&p1)[8], f2 (&R)[4], f2 (&G)[4],
                                              f2 (&B)[4]) {
  f2 ns[8];
#pragma unroll
  for (int i = 1; i <= 6; ++i) ns[i] = add2(m1[i], p1[i]);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const f2 C = z[j + 2];
    const f2 EW = add2(z[j + 1], z[j + 3]);
    if (!SiteScale2<BROW, GFIRST>::gsite(j)) {
      const f2 opp = add2(ns[j + 1], ns[j + 3]);
      G[j] = mul2(bc(-2.f), add2(ns[j + 2], EW));
      R[j] = BROW ? opp : C;
      B[j] = BROW ? C : opp;
    } else {
      const f2 hn = mul2(bc(-4.f), EW), vn = mul2(bc(-4.f), ns[j + 2]);
      G[j] = C;
      R[j] = BROW ? vn : hn;
      B[j] = BROW ? hn : vn;
    }
  }
}

// Task kinds.  The image rows 2 .. H-3 are cut into chunks of rows_per_task rows ("interior tasks": no row of
// their window is ever outside the image); the four border rows of every frame form two extra 2-row tasks per
// strip.  One warp per task; interior tasks first.  Each kind is its own instantiation of the row loop, chosen
// by a warp-uniform branch at task start, so the hot loop carries nothing it does not need:
//   K_CORE     interior rows, strips 1 .. last-1: no frame pixel, no masks, no predicated loads or stores
//   K_EDGE     interior rows, first / last strip: the first / last thread column owns frame columns and reads
//              no halo beyond the image; the last strip may be partial
//   K_GENERAL  any rows (the border tasks; every task when the epilogue declines the fast kinds): rows outside
//              the image are masked, every pixel is renormalised by its own in-bounds weight sum
enum { K_CORE = 0, K_EDGE = 1, K_GENERAL = 2 };

// Loader2 concept:
//   static constexpr uint32_t kRowMask                              decode mask of a row inside the image
//   struct Raw;  struct Cursor;
//   template <int KIND> void open(Cursor&, int frame, int tcol, const StreamGeom&)   per-task pointer of row 0 (+ edge masks)
//   template <int KIND> void fetch(const Cursor&, const P* row_ptr, Raw&)            loads of one (valid) row
//   void prefetch(const Cursor&, const P* row_ptr)                                   optional L2 prefetch
//   template <int KIND> void decode(const Cursor&, const Raw&, uint32_t row_mask, f2 (&P)[8])
//                                                                   row_mask (K_GENERAL only) = 0 -> zero samples
//   ptrdiff_t pitch() const                                         row pitch in elements of the cursor pointer
// Epi2 concept:
//   static constexpr int kStageWords
//   struct State;  void init(State&, int frame, int tcol, const WarpCtx&);  void finish(State&, int frame, int lane, bool task_ok)
//   static constexpr bool kSplitEdge                                false: no K_CORE instantiation, interior tasks run K_EDGE
//   static constexpr bool kCompactLoop                              true: single-step loop body (register moves) for every kind
//   bool fast_kinds_ok(const State&)                                false -> every task runs K_GENERAL
//   template <bool BROW, bool GFIRST, int KIND> void emit(State&, int row, const f2 (&R)[4], const f2 (&G)[4], const f2 (&B)[4])
//       scaled filter sums (SiteScale2); out-of-image taps contributed the zero sample; the epilogue renormalises
//       the frame pixels its KIND can contain (border_fix.cuh).

constexpr int kBorderRows = 2;   // rows of the top / bottom border tasks (K_GENERAL)

struct Stream2Geom {
  StreamGeom g;             // rows_per_task / nchunks describe the INTERIOR rows 2 .. H-3
  long long interior_tasks; // nframes * nchunks * warps_per_row
  long long total_tasks;    // + nframes * 2 * warps_per_row
};

// rows_per_task <= 0: 24 rows per task (4 halo rows = 17 % extra loads, all L2 hits), shrunk for small jobs until
// the tasks fill one wave of 148 SMs x 16 resident warps.  Measured (scripts/rpt_sweep.py, profiles/r02_rpt_sweep.txt):
// the sweep time is flat within 3 % between 16 and 32 rows for 1 x 4096x3000, 6 x 4096x3000 and 6 x 5472x3648; chunks
// of 48+ rows lose 10-50 % (the tail of the last wave is one whole task long), a wave-count model predicts nothing
// finer than that.
inline int auto_rows_per_task2(int H, int W, int nframes) {
  const int interior = H - 4;
  if (interior <= 0) return 2;
  const long long wpr = ((W + 7) / 8 + 31) / 32;
  int rpt = 24;
  while (rpt > 8 && (long long)nframes * wpr * ((interior + rpt - 1) / rpt + 2) < (long long)(0.9 * 16 * kNumSMs)) rpt -= 2;
  return rpt;
}

inline Stream2Geom make_geom2(int H, int W, int nframes, int rows_per_task) {
  Stream2Geom s;
  if (rows_per_task <= 0) rows_per_task = auto_rows_per_task2(H, W, nframes);
  const int interior = H - 2 * kBorderRows;
  s.g = make_geom(interior > 0 ? interior : 0, W, nframes, rows_per_task);      // chunking of the interior rows
  s.g.H = H;
  s.interior_tasks = (interior > 0) ? s.g.total_tasks : 0;
  s.total_tasks = s.interior_tasks + (long long)nframes * 2 * s.g.warps_per_row;
  return s;
}

#ifndef ISP_S2_PF_ROWS
#define ISP_S2_PF_ROWS 6        // L2 prefetch distance beyond the register fetch (rows row+4+PF, row+5+PF); 2 / 6 / 12 measured: 173.6 / 171.4 / 172.4 us
#endif
#ifndef ISP_S2_THREADS
#define ISP_S2_THREADS 128      // 4 warps per CTA
#endif
#ifndef ISP_S2_MINBLOCKS
#define ISP_S2_MINBLOCKS 4      // 16 warps / SM at 128 registers (measured: 175 us vs 182 us with 3 blocks / 168 registers on cfg2)
#endif
constexpr int kS2Warps = ISP_S2_THREADS / 32;

// rows [r0, rend) of one strip of one frame; r0 even, rend - r0 even
template <bool BROW0, bool GFIRST0, int KIND, bool BL, class Loader, class Epi>
__device__ __forceinline__ void stream2_rows(const Loader& ld, const Epi& epi, typename Epi::State& st, const StreamGeom& g,
                                             int frame, int tcol, int r0, int rend) {
  constexpr uint32_t kMask = Loader::kRowMask;
  constexpr bool MASKED = KIND == K_GENERAL;
  typename Loader::Cursor cur;
  ld.template open<KIND>(cur, frame, tcol, g);
  const ptrdiff_t pitch = ld.pitch();

  // six full pair rows, rotating: step U reads W[(2U+k) % 6], k = 0..5 = rows row-2 .. row+3
  f2 W[6][8];
  typename Loader::Raw raw0{}, raw1{};

  // Row pairs (rr, rr+1), rr even, are inside the image together or outside together (H is even); an outside
  // pair is fetched from the nearest valid pair and (K_GENERAL; the other kinds never use one) decoded with mask 0.
  auto clamped = [&](int rr) { return min(max(rr, 0), g.H - 2); };
  auto row_mask = [&](int rr) -> uint32_t { return (!MASKED || (unsigned)rr < (unsigned)g.H) ? kMask : 0u; };
  {
    const auto* p = cur.p + (ptrdiff_t)clamped(r0 - 2) * pitch;
    const uint32_t m = row_mask(r0 - 2);
    ld.template fetch<KIND>(cur, p, raw0);
    ld.template fetch<KIND>(cur, p + pitch, raw1);
    ld.template decode<KIND>(cur, raw0, m, W[0]);
    ld.template decode<KIND>(cur, raw1, m, W[1]);
  }
  {
    const auto* p = cur.p + (ptrdiff_t)r0 * pitch;
    ld.template fetch<KIND>(cur, p, raw0);
    ld.template fetch<KIND>(cur, p + pitch, raw1);
    ld.template decode<KIND>(cur, raw0, kMask, W[2]);
    ld.template decode<KIND>(cur, raw1, kMask, W[3]);
  }
  // pn / mask describe the pair waiting in raw0 / raw1 (rows row+2, row+3 of the step about to run)
  const auto* pn = cur.p + (ptrdiff_t)clamped(r0 + 2) * pitch;
  uint32_t mask = row_mask(r0 + 2);
  ld.template fetch<KIND>(cur, pn, raw0);
  ld.template fetch<KIND>(cur, pn + pitch, raw1);
#pragma unroll
  for (int d = 4; d < 4 + ISP_S2_PF_ROWS; d += 2) {
    ld.prefetch(cur, cur.p + (ptrdiff_t)clamped(r0 + d) * pitch);
    ld.prefetch(cur, cur.p + (ptrdiff_t)clamped(r0 + d) * pitch + pitch);
  }

#define ISP_STEP(U, ROW)                                                                                        \
  {                                                                                                             \
    const int row_ = (ROW);                                                                                     \
    const uint32_t m_ = mask;                                                                                   \
    ld.template decode<KIND>(cur, raw0, m_, W[(2 * (U) + 4) % 6]);                                              \
    /* next pair: rows row+4, row+5 (clamped to the last pair when past the image) */                         \
    const bool in_ = row_ + 4 < g.H;                                                                            \
    pn += in_ ? 2 * pitch : 0;                                                                                  \
    if (MASKED) mask = in_ ? kMask : 0u;                                                                        \
    ld.template fetch<KIND>(cur, pn, raw0);                                                                     \
    if (row_ + 4 + ISP_S2_PF_ROWS < g.H) ld.prefetch(cur, pn + ISP_S2_PF_ROWS * pitch);                                                     \
    f2 R_[4], G_[4], B_[4];                                                                                     \
    if constexpr (BL) bilinear_row2<BROW0, GFIRST0>(W[(2 * (U) + 1) % 6], W[(2 * (U) + 2) % 6], W[(2 * (U) + 3) % 6], R_, G_, B_); \
    else malvar_row2<BROW0, GFIRST0>(W[(2 * (U)) % 6], W[(2 * (U) + 1) % 6], W[(2 * (U) + 2) % 6],              \
                                     W[(2 * (U) + 3) % 6], W[(2 * (U) + 4) % 6], R_, G_, B_);                   \
    epi.template emit<BROW0, GFIRST0, KIND>(st, row_, R_, G_, B_);                                              \
    ld.template decode<KIND>(cur, raw1, m_, W[(2 * (U) + 5) % 6]);                                              \
    ld.template fetch<KIND>(cur, pn + pitch, raw1);                                                             \
    if (row_ + 4 + ISP_S2_PF_ROWS < g.H) ld.prefetch(cur, pn + (ISP_S2_PF_ROWS + 1) * pitch);                                                     \
    if constexpr (BL) bilinear_row2<!BROW0, !GFIRST0>(W[(2 * (U) + 2) % 6], W[(2 * (U) + 3) % 6], W[(2 * (U) + 4) % 6], R_, G_, B_); \
    else malvar_row2<!BROW0, !GFIRST0>(W[(2 * (U) + 1) % 6], W[(2 * (U) + 2) % 6], W[(2 * (U) + 3) % 6],        \
                                       W[(2 * (U) + 4) % 6], W[(2 * (U) + 5) % 6], R_, G_, B_);                 \
    epi.template emit<!BROW0, !GFIRST0, KIND>(st, row_ + 1, R_, G_, B_);                                        \
  }

  if constexpr (KIND == K_GENERAL || BL || Epi::kCompactLoop) {
    // cold kind, or an epilogue so large that three copies of the step overflow the instruction cache (Reinhard:
    // 51 KB hot, no_instruction 3.1 cycles per issue): one copy of the step, the window slides by register moves
    // (measured: 1 step 607 / 147 Gpx/s (cfg2 / cfg3), 2 steps 585 / 120 -- code size beats moves).
    // The slide as packed additions of -0.0 (exact identity for every float): one FADD2 moves a register PAIR, and because
    // the result is a fresh value ptxas gives it the loop-carried register directly -- a plain copy costs two MOVs per pair
    // (64 per step = 4 per pixel).  ptxas does not fold the addition away.
#pragma unroll 1
    for (int row = r0; row < rend; row += 2) {
      ISP_STEP(0, row);
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int i = 0; i < 8; ++i) W[k][i] = add2(W[k + 2][i], bc(-0.0f));
    }
  } else {
#pragma unroll 1
    for (int row = r0; row < rend; row += 6) {
      ISP_STEP(0, row);
      if (row + 2 >= rend) break;
      ISP_STEP(1, row + 2);
      if (row + 4 >= rend) break;
      ISP_STEP(2, row + 4);
    }
  }
#undef ISP_STEP
}

// Epi::kGated: the epilogue can decline whole frames at run time (enabled(frame), warp-uniform) -- the gated fallback sweeps
// of the one-sweep Reinhard path (fused_isp.cuh); every other epilogue has no such member and no such code.
template <class Epi, class = void> struct has_gate { static constexpr bool value = false; };
template <class Epi> struct has_gate<Epi, std::enable_if_t<Epi::kGated>> { static constexpr bool value = true; };

// BL: bilinear demosaic instead of Malvar-He-Cutler.  The bilinear kernels have no K_CORE copy of the loop and use
// the single-step body (their binary stays small; the arithmetic saved is hidden behind the same DRAM traffic).
template <int PATTERN, bool BL, class Loader, class Epi>
__device__ __forceinline__ void stream2_task(const Loader& ld, const Epi& epi, const Stream2Geom& sg, long long task, uint32_t* stage_warp) {
  constexpr bool BROW0 = (PATTERN == B200ISP_GBRG || PATTERN == B200ISP_BGGR);
  constexpr bool GFIRST0 = (PATTERN == B200ISP_GRBG || PATTERN == B200ISP_GBRG);
  const StreamGeom& g = sg.g;
  const int lane = threadIdx.x & 31;
  const bool task_ok = task < sg.total_tasks;
  if (!task_ok) task = 0;
  const bool border = task >= sg.interior_tasks;
  int strip, frame, r0, rend;
  if (!border) {
    strip = (int)(task % g.warps_per_row);
    const long long t2 = task / g.warps_per_row;
    const int chunk = (int)(t2 % g.nchunks);
    frame = (int)(t2 / g.nchunks);
    r0 = kBorderRows + chunk * g.rows_per_task;
    rend = min(r0 + g.rows_per_task, g.H - kBorderRows);
  } else {
    const long long t = task - sg.interior_tasks;
    strip = (int)(t % g.warps_per_row);
    const long long t2 = t / g.warps_per_row;
    frame = (int)(t2 >> 1);
    r0 = (t2 & 1) ? g.H - kBorderRows : 0;
    rend = r0 + kBorderRows;
  }
  const int tcol = min(strip * 32 + lane, g.ntcols - 1);   // lanes past the last column recompute it (never stored)
  if constexpr (has_gate<Epi>::value) {
    if (!epi.enabled(frame)) return;                       // the whole warp works on one frame: uniform exit
  }

  WarpCtx wc;
  wc.lane = lane;
  wc.tcol0 = strip * 32;
  wc.nvalid = min(32, g.ntcols - strip * 32);
  wc.stage = stage_warp;

  constexpr bool kSplit = Epi::kSplitEdge && !BL;

  typename Epi::State st;
  epi.init(st, frame, tcol, wc);
  if (task_ok) {
    // Epi::kSplitEdge = false: the epilogue does not want a separate K_CORE copy of the loop (K_EDGE covers it)
    const int kind = (border || !epi.fast_kinds_ok(st)) ? K_GENERAL
                     : ((!kSplit || strip == 0 || strip == g.warps_per_row - 1) ? K_EDGE : K_CORE);
    if constexpr (kSplit) {
      if (kind == K_CORE) stream2_rows<BROW0, GFIRST0, K_CORE, BL>(ld, epi, st, g, frame, tcol, r0, rend);
    }
    if (kind == K_EDGE) stream2_rows<BROW0, GFIRST0, K_EDGE, BL>(ld, epi, st, g, frame, tcol, r0, rend);
    else if (kind == K_GENERAL) stream2_rows<BROW0, GFIRST0, K_GENERAL, BL>(ld, epi, st, g, frame, tcol, r0, rend);
  }
  epi.finish(st, frame, lane, task_ok);
}


// One warp per task, one launch of ceil(tasks / 4) CTAs.  Gated epilogues (has_gate: the exact fallback of the one-sweep
// Reinhard path, which in the usual case has nothing to do) run a small persistent grid that strides over the tasks instead:
// launching and retiring thousands of CTAs that exit at once costs 6.5 us per kernel, a few hundred cost 2.
template <int PATTERN, bool BL, class Loader, class Epi>
__global__ void __launch_bounds__(ISP_S2_THREADS, ISP_S2_MINBLOCKS) stream2_kernel(const Loader ld, const Epi epi, const Stream2Geom sg) {
  __shared__ __align__(16) uint32_t stage[kS2Warps][Epi::kStageWords > 0 ? Epi::kStageWords : 1];
  uint32_t* stage_warp = stage[threadIdx.x >> 5];
  if constexpr (has_gate<Epi>::value) {
    // the usual case -- no frame declined -- ends here after one look at the per-frame flags (a lane per frame) instead of
    // one task decode (three 64-bit divisions) + flag load per task of the stride loop
    bool any = false;
    for (int f = threadIdx.x & 31; f < sg.g.nframes; f += 32) any |= epi.enabled(f);
    if (!__any_sync(0xffffffffu, any)) return;
    for (long long task = (long long)blockIdx.x * kS2Warps + (threadIdx.x >> 5); task < sg.total_tasks; task += (long long)gridDim.x * kS2Warps)
      stream2_task<PATTERN, BL>(ld, epi, sg, task, stage_warp);
  } else {
    stream2_task<PATTERN, BL>(ld, epi, sg, (long long)blockIdx.x * kS2Warps + (threadIdx.x >> 5), stage_warp);
  }
}

template <int PATTERN, class Loader, class Epi>
inline int launch_stream2(const Loader& ld, const Epi& epi, const Stream2Geom& sg, cudaStream_t s, const char* what,
                          bool bilinear = false) {
  if (sg.total_tasks == 0) return B200ISP_OK;
  long long blocks = (sg.total_tasks + kS2Warps - 1) / kS2Warps;
  if (has_gate<Epi>::value && blocks > ISP_S2_MINBLOCKS * kNumSMs) blocks = ISP_S2_MINBLOCKS * kNumSMs;      // persistent (see stream2_kernel)
  if (bilinear) stream2_kernel<PATTERN, true, Loader, Epi><<<(unsigned)blocks, ISP_S2_THREADS, 0, s>>>(ld, epi, sg);
  else stream2_kernel<PATTERN, false, Loader, Epi><<<(unsigned)blocks, ISP_S2_THREADS, 0, s>>>(ld, epi, sg);
  return cuda_status(cudaPeekAtLastError(), what);
}

}  // namespace isp
