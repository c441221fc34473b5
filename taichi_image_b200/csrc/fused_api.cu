// C entry points of the fused packed12 sweep and its sparse metering (see fused_isp.cuh), and run_fused: the launch sequence of
// every ReinhardForm.
#include "fused_isp.cuh"
#include "resize_isp.cuh"

using namespace isp;

// Checks of the parameter block common to the fused entry points, and the constants derived from it, except the two
// pointers k.metrics / k.ws.  Reads no pointer, so b200isp_reinhard_scratch_bytes runs it on a machine without a GPU.
static int fused_consts(const char* what, int n_frames, const b200isp_fused_params& p, IspConsts& k) {
  ISP_REQUIRE(n_frames >= 1 && n_frames <= B200ISP_MAX_FRAMES, B200ISP_E_FRAMES,
              "%s: %d frames (1..%d supported per call)", what, n_frames, B200ISP_MAX_FRAMES);
  ISP_REQUIRE(p.height >= 4 && p.width >= 8 && p.height % 2 == 0 && p.width % 8 == 0, B200ISP_E_SHAPE,
              "%s: fused path needs even height >= 4 and width %% 8 == 0, got %dx%d", what, p.height, p.width);
  ISP_REQUIRE(p.pattern >= 0 && p.pattern <= 3, B200ISP_E_ARG, "%s: unknown pattern %d", what, p.pattern);
  ISP_REQUIRE(p.isp_dtype == B200ISP_F16 || p.isp_dtype == B200ISP_F32, B200ISP_E_DTYPE, "%s: isp_dtype must be f16/f32", what);
  k.H = p.height; k.W = p.width; k.pattern = p.pattern;
  k.ccm = p.has_ccm ? 1 : 0;
  for (int i = 0; i < 9; ++i) k.m[i] = p.has_ccm ? p.ccm[i] : (i % 4 == 0 ? 1.f : 0.f);   // identity: see raw_to_rgb
  k.gamma = p.gamma; k.intensity = p.intensity; k.la = p.light_adapt; k.ca = p.color_adapt;
  ISP_REQUIRE(p.demosaic == B200ISP_DEMOSAIC_MALVAR || p.demosaic == B200ISP_DEMOSAIC_BILINEAR, B200ISP_E_ARG,
              "%s: unknown demosaic %d", what, p.demosaic);
  k.kbase = p.demosaic == B200ISP_DEMOSAIC_BILINEAR ? kBilinearBase : 0;
  k.flip = p.flip & 7;
  k.gate = 0;
  ISP_REQUIRE(!(k.flip && (resizes(p) || p.out_yuv420)), B200ISP_E_ARG, "%s: flips in the store need the plain RGB sweep (no resize, no YUV)", what);
  ISP_REQUIRE(!(k.flip & 4) || (p.height % 8 == 0 && p.height >= 16), B200ISP_E_SHAPE,
              "%s: the transposing transforms need height %% 8 == 0 and height >= 16, got %dx%d", what, p.height, p.width);
  k.ids = p.ids_layout ? 1 : 0;
  ISP_REQUIRE(!(k.ids && resizes(p)), B200ISP_E_ARG, "%s: the IDS layout is not available with the fused resize (re-pack first)", what);
  const int out_cols = (k.flip & 4) ? p.height : p.width;        // the transposing transforms write (W, H) images
  k.orow = p.out_pitch > 0 ? p.out_pitch : 3 * out_cols;
  ISP_REQUIRE(p.out_pitch <= 0 || (k.orow >= 3 * out_cols && (k.orow * (int)dtype_size(p.out_dtype)) % 16 == 0), B200ISP_E_ALIGN,
              "%s: out_pitch must be >= 3 * (output width) elements and a multiple of 16 bytes", what);
  ISP_REQUIRE(p.out_pitch <= 0 || (!resizes(p) && !p.out_yuv420), B200ISP_E_ARG, "%s: out_pitch needs the plain RGB sweep (no resize, no YUV)", what);
  return B200ISP_OK;
}

// fused_consts + the frame table of the fused entry points.
static int fused_setup(const char* what, const uint8_t* const* packed_host, void* const* out_host, int n_frames,
                       const b200isp_fused_params* params, float* metrics, void* workspace, FramePtrs& fp, IspConsts& k) {
  ISP_REQUIRE(packed_host && params && workspace, B200ISP_E_ARG, "%s: null pointer", what);
  const int st = fused_consts(what, n_frames, *params, k);
  if (st) return st;
  for (int i = 0; i < n_frames; ++i) {
    fp.in[i] = packed_host[i];
    fp.out[i] = out_host ? out_host[i] : nullptr;
    ISP_REQUIRE(fp.in[i] && (fp.out[i] || !out_host), B200ISP_E_ARG, "%s: null frame pointer %d", what, i);
    ISP_REQUIRE(((reinterpret_cast<uintptr_t>(fp.in[i]) & 3u) == 0) && ((reinterpret_cast<uintptr_t>(fp.out[i]) & 15u) == 0),
                B200ISP_E_ALIGN, "%s: frame %d needs 4-byte aligned input and 16-byte aligned output", what, i);
  }
  k.metrics = metrics; k.ws = (Workspace*)workspace;
  return B200ISP_OK;
}

// The further checks of b200isp_process_packed12 that read only the parameter block (k: its fused_consts).
static int process_checks(const b200isp_fused_params& p, const IspConsts& k) {
  ISP_REQUIRE(p.tonemap >= B200ISP_TM_LINEAR && p.tonemap <= B200ISP_TM_NONE, B200ISP_E_ARG, "process_packed12: unknown tonemap %d", p.tonemap);
  ISP_REQUIRE(p.tonemap == B200ISP_TM_NONE || p.gamma > 0.f, B200ISP_E_ARG, "process_packed12: gamma must be positive");
  if (p.tonemap == B200ISP_TM_NONE)
    ISP_REQUIRE(p.out_dtype == p.isp_dtype, B200ISP_E_DTYPE, "process_packed12: TM_NONE writes the ISP dtype");
  else
    ISP_REQUIRE(p.out_dtype == B200ISP_U8 || p.out_dtype == B200ISP_U16 || p.out_dtype == B200ISP_F16, B200ISP_E_DTYPE,
                "process_packed12: tone-mapped output must be u8, u16 or f16");
  if (resizes(p)) {
    ISP_REQUIRE(p.scale_r > 0.f && p.scale_c > 0.f, B200ISP_E_ARG, "process_packed12: resize scales must be positive");
    ISP_REQUIRE(!p.out_yuv420, B200ISP_E_ARG, "process_packed12: YUV 4:2:0 output is not available with resize");
  }
  ISP_REQUIRE(!p.out_yuv420 || (p.isp_dtype == B200ISP_F16 && p.out_dtype == B200ISP_U8 && p.tonemap == B200ISP_TM_REINHARD),
              B200ISP_E_ARG, "process_packed12: YUV 4:2:0 output needs Camera16 (f16), Reinhard, u8 and the reinhard_scratch buffer");
  if (k.flip & 4) {        // only the normalise pass of the one-sweep Reinhard -> u8 forms turns the image
    const ReinhardForm f = reinhard_plan(p, k, 1).form;
    ISP_REQUIRE(f == ReinhardForm::kF16Turned || f == ReinhardForm::kU16Turned, B200ISP_E_ARG,
                "process_packed12: the transposing transforms need a one-sweep Reinhard -> u8 form (b200isp_reinhard_scratch_bytes > 0)");
  }
  return B200ISP_OK;
}

namespace isp {
ReinhardPlan reinhard_plan(const b200isp_fused_params& p, const IspConsts& k, int n_frames) {
  if (p.tonemap != B200ISP_TM_REINHARD) return {ReinhardForm::kNone, 0, 0};
  const bool cam16 = p.isp_dtype == B200ISP_F16;
  if (resizes(p)) {
    const size_t map = (size_t)n_frames * p.out_height * p.out_width * 3 * (cam16 ? sizeof(__half) : sizeof(float));
    return {ReinhardForm::kResizeMap, map, map};
  }
  const size_t map = (size_t)n_frames * k.H * k.W * 3 * (cam16 ? sizeof(__half) : sizeof(uint16_t));
  const bool u8 = p.out_dtype == B200ISP_U8;
  // the normalise pass turns the image (reinhard_out_transposed_kernel); the map itself is a plain (H, W, 3) image
  const bool turned = (k.flip & 4) && u8 && k.orow % 8 == 0 && k.ids == 0;
  if (cam16) {
    if (turned) return {ReinhardForm::kF16Turned, map, map};
    // the other normalise passes index the output flat: dense, unflipped outputs only
    if (k.flip != 0 || k.orow != 3 * k.W) return {ReinhardForm::kExact, 0, 0};
    if (p.out_yuv420) return {ReinhardForm::kF16Yuv, map, map};
    if (u8 && k.gamma != 1.0f) return {ReinhardForm::kF16Table, map, map + (size_t)n_frames * kLutBytes};
    return {ReinhardForm::kF16Arith, map, map};
  }
  if (u8 && p.reinhard_mode == 0 && k.ca == 0.f && k.gamma <= 1.0f && k.gamma >= 0.3f && (k.flip == 0 || turned) && k.ids == 0)
    return {turned ? ReinhardForm::kU16Turned : ReinhardForm::kU16Map, map, map};
  return {ReinhardForm::kExact, 0, 0};
}

}  // namespace isp

extern "C" size_t b200isp_reinhard_scratch_bytes(const b200isp_fused_params* params, int n_frames) {
  IspConsts k;
  if (!params || fused_consts("reinhard_scratch_bytes", n_frames, *params, k) || process_checks(*params, k)) return 0;
  return reinhard_plan(*params, k, n_frames).bytes;
}

namespace isp {
// The metering kernels that do not depend on the sampler (metering.cuh), compiled here only.
__global__ void meter_fold_bounds_kernel(const float* __restrict__ g1, int world, float alpha, const float* __restrict__ prev,
                                         Workspace* ws) {
  if (threadIdx.x == 0 && blockIdx.x == 0) fold_bounds(g1, world, alpha, prev, ws->bounds[0], ws->bounds[1]);
}

__global__ void meter_finalize_kernel(const float* __restrict__ g1, const float* __restrict__ g2, int world, float alpha,
                                      const float* prev, float* metrics /* out; may alias prev */) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  float bmin, bmax;
  fold_bounds(g1, world, alpha, prev, bmin, bmax);
  float f[8] = {INFINITY, -INFINITY, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int r = 0; r < world; ++r) {
    f[0] = fminf(f[0], g2[8 * r]);
    f[1] = fmaxf(f[1], g2[8 * r + 1]);
    for (int k = 2; k < 8; ++k) f[k] += g2[8 * r + k];
  }
  const float fn = f[7];                                                  // camera_isp.py:131-134 with n = all ranks' samples
  const float stats[9] = {bmin, bmax, f[0], f[1], __fdiv_rn(f[2], fn), __fdiv_rn(f[3], fn),
                          __fdiv_rn(f[4], fn), __fdiv_rn(f[5], fn), __fdiv_rn(f[6], fn)};
  for (int k = 0; k < 9; ++k) {                                           // camera_isp.py:165-166
    const float p = prev[k];
    metrics[k] = __fadd_rn(stats[k], __fmul_rn(alpha, __fsub_rn(p, stats[k])));
  }
}

int launch_meter_fold_bounds(const float* g1, int world, float alpha, const float* prev, Workspace* ws, cudaStream_t s) {
  meter_fold_bounds_kernel<<<1, 32, 0, s>>>(g1, world, alpha, prev, ws);
  return cuda_status(cudaPeekAtLastError(), "meter_fold_bounds_kernel");
}

int launch_meter_finalize(const float* g1, const float* g2, int world, float alpha, const float* prev, float* metrics, cudaStream_t s) {
  meter_finalize_kernel<<<1, 32, 0, s>>>(g1, g2, world, alpha, prev, metrics);
  return cuda_status(cudaPeekAtLastError(), "meter_finalize_kernel");
}

int launch_meter_phase2_cached(int grid, const CachedSampler& smp, long long n, float alpha, const float* prev, float* metrics, Workspace* ws,
                               cudaStream_t s, float* rec_out) {
  meter_phase2_kernel<CachedSampler><<<grid, 256, 0, s>>>(smp, n, alpha, prev, metrics, ws, rec_out);
  return cuda_status(cudaPeekAtLastError(), "meter_phase2_kernel");
}

}  // namespace isp

// Builds the metering sampler for the packed frames (stride % 8 == 0: word-aligned fast sampler) and
// hands it to f(sampler, n_samples, cache).
template <class F>
static int with_packed12_sampler(const FramePtrs& fp, const b200isp_fused_params& p, const IspConsts& k, int n_frames, F f) {
  const int stride = p.metering_stride > 0 ? p.metering_stride : 8;
  const bool cam16 = p.isp_dtype == B200ISP_F16;
  if (resizes(p)) {                     // the reference meters what _process_image returns: the RESIZED image
    const int hs = (p.out_height + stride - 1) / stride, wsamp = (p.out_width + stride - 1) / stride;
    const long long n = (long long)n_frames * hs * wsamp;
    float* cache = (p.meter_cache && p.meter_cache_bytes >= (size_t)n * 3 * sizeof(float)) ? (float*)p.meter_cache : nullptr;
    if (cam16) return f(ResizedSampler<true>{make_resize_src<true>(fp, k, p), stride, hs, wsamp}, n, cache);
    return f(ResizedSampler<false>{make_resize_src<false>(fp, k, p), stride, hs, wsamp}, n, cache);
  }
  const int hs = (p.height + stride - 1) / stride, wsamp = (p.width + stride - 1) / stride;
  const long long n = (long long)n_frames * hs * wsamp;
  float* cache = (p.meter_cache && p.meter_cache_bytes >= (size_t)n * 3 * sizeof(float)) ? (float*)p.meter_cache : nullptr;
  if (stride % 8 == 0) {
    if (cam16) return f(Packed12FastSampler<true>{Packed12Src<true>{fp, p.width * 3 / 2, k.ids}, k, stride, hs, wsamp, p.width * 3 / 8}, n, cache);
    return f(Packed12FastSampler<false>{Packed12Src<false>{fp, p.width * 3 / 2, k.ids}, k, stride, hs, wsamp, p.width * 3 / 8}, n, cache);
  }
  if (cam16) return f(Packed12Sampler<true>{Packed12Src<true>{fp, p.width * 3 / 2, k.ids}, k, stride, hs, wsamp}, n, cache);
  return f(Packed12Sampler<false>{Packed12Src<false>{fp, p.width * 3 / 2, k.ids}, k, stride, hs, wsamp}, n, cache);
}

extern "C" int b200isp_meter_packed12_phase1(const uint8_t* const* packed_host, int n_frames, const b200isp_fused_params* params,
                                             float* rec1, void* workspace, b200isp_stream stream) {
  FramePtrs fp; IspConsts k;
  const int st = fused_setup("meter_packed12_phase1", packed_host, nullptr, n_frames, params, nullptr, workspace, fp, k);
  if (st) return st;
  ISP_REQUIRE(rec1, B200ISP_E_ARG, "meter_packed12_phase1: null record");
  cudaStream_t s = (cudaStream_t)stream;
  return with_packed12_sampler(fp, *params, k, n_frames, [&](const auto& smp, long long n, float* cache) {
    return launch_metering_phase1(smp, n, k.ws, s, cache, rec1);
  });
}

extern "C" int b200isp_meter_packed12_phase2(const uint8_t* const* packed_host, int n_frames, const b200isp_fused_params* params,
                                             const float* gathered1, int world, const float* metrics_prev, float* rec2,
                                             void* workspace, b200isp_stream stream) {
  FramePtrs fp; IspConsts k;
  const int st = fused_setup("meter_packed12_phase2", packed_host, nullptr, n_frames, params, nullptr, workspace, fp, k);
  if (st) return st;
  ISP_REQUIRE(gathered1 && metrics_prev && rec2 && world >= 1, B200ISP_E_ARG, "meter_packed12_phase2: bad argument");
  cudaStream_t s = (cudaStream_t)stream;
  const float alpha = params->alpha;
  return with_packed12_sampler(fp, *params, k, n_frames, [&](const auto& smp, long long n, float* cache) {
    return launch_metering_phase2(smp, n, gathered1, world, alpha, metrics_prev, k.ws, s, cache, rec2);
  });
}

extern "C" int b200isp_metering_finalize(const float* gathered1, const float* gathered2, int world, float alpha,
                                         const float* metrics_prev, float* metrics_out, b200isp_stream stream) {
  ISP_REQUIRE(gathered1 && gathered2 && metrics_prev && metrics_out && world >= 1, B200ISP_E_ARG, "metering_finalize: bad argument");
  return launch_meter_finalize(gathered1, gathered2, world, alpha, metrics_prev, metrics_out, (cudaStream_t)stream);
}

extern "C" int b200isp_meter_packed12(const uint8_t* const* packed_host, int n_frames, const b200isp_fused_params* params,
                                      const float* metrics_prev, float* metrics_out, int cooperative, void* workspace,
                                      b200isp_stream stream) {
  FramePtrs fp; IspConsts k;
  const int st = fused_setup("meter_packed12", packed_host, nullptr, n_frames, params, nullptr, workspace, fp, k);
  if (st) return st;
  ISP_REQUIRE(metrics_prev && metrics_out, B200ISP_E_ARG, "meter_packed12: null metrics");
  cudaStream_t s = (cudaStream_t)stream;
  const float alpha = params->alpha;
  return with_packed12_sampler(fp, *params, k, n_frames, [&](const auto& smp, long long n, float* cache) {
    return launch_metering(smp, n, alpha, metrics_prev, metrics_out, k.ws, s, cache, cooperative != 0);
  });
}

// camera_isp.py:376-385 jointly over the frames of ALL ranks (each rank passes its own), with both record exchanges inside
// the two metering kernels (metering.cuh meter_phase1x / meter_phase2x, exchange.cuh): every rank ends with bit-identical
// metrics_out = lerp(alpha, joint statistics, metrics_prev).  peers_host: the world mailbox pointers of
// b200isp_mailbox_create / _open (entry `rank` = this rank's own).
extern "C" int b200isp_meter_packed12_shared(const uint8_t* const* packed_host, int n_frames, const b200isp_fused_params* params,
                                             void* const* peers_host, int world, int rank, const float* metrics_prev,
                                             float* metrics_out, void* workspace, b200isp_stream stream) {
  FramePtrs fp; IspConsts k;
  const int st = fused_setup("meter_packed12_shared", packed_host, nullptr, n_frames, params, nullptr, workspace, fp, k);
  if (st) return st;
  ISP_REQUIRE(metrics_prev && metrics_out && peers_host, B200ISP_E_ARG, "meter_packed12_shared: null pointer");
  ISP_REQUIRE(world >= 1 && world <= kXchgRanks && rank >= 0 && rank < world, B200ISP_E_ARG, "meter_packed12_shared: world %d rank %d", world, rank);
  PeerXchg xc;
  xc.world = world; xc.rank = rank;
  for (int r = 0; r < kXchgRanks; ++r) xc.p[r] = r < world ? (uint32_t*)peers_host[r] : nullptr;
  for (int r = 0; r < world; ++r) ISP_REQUIRE(xc.p[r], B200ISP_E_ARG, "meter_packed12_shared: null mailbox of rank %d", r);
  cudaStream_t s = (cudaStream_t)stream;
  const float alpha = params->alpha;
  return with_packed12_sampler(fp, *params, k, n_frames, [&](const auto& smp, long long n, float* cache) {
    return launch_metering_shared(smp, n, alpha, metrics_prev, metrics_out, k.ws, s, cache, xc);
  });
}

// profile hooks: inside a stream capture the record must be an "external" event node to stay queryable
static void record_profile_event(void* ev, cudaStream_t s) {
  if (!ev) return;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(s, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusActive)
    cudaEventRecordWithFlags((cudaEvent_t)ev, s, cudaEventRecordExternal);
  else
    cudaEventRecord((cudaEvent_t)ev, s);
}

// Sweep sw over fp with k: the instantiation of the call's ISP dtype (and output dtype, for the sweeps that write the output)
static int run_sweep(Sweep sw, const FramePtrs& fp, const IspConsts& k, const b200isp_fused_params& p, int n_frames, cudaStream_t s) {
  const int rpt = p.rows_per_task;
  const bool cam16 = p.isp_dtype == B200ISP_F16;
  if (sw == Sweep::kMax || sw == Sweep::kStore)
    return cam16 ? run_max_sweep<true>(sw, fp, k, n_frames, rpt, s) : run_max_sweep<false>(sw, fp, k, n_frames, rpt, s);
  if (sw == Sweep::kMaxGated || sw == Sweep::kReinhardGated) return run_gated_sweep(sw, fp, k, n_frames, rpt, s);
#define RUN(CAM, T) return run_out_sweep<CAM, T>(sw, fp, k, n_frames, rpt, s)
  if (cam16) {
    switch (p.out_dtype) {
      case B200ISP_U8: RUN(true, uint8_t);
      case B200ISP_U16: RUN(true, uint16_t);
      case B200ISP_F16: RUN(true, __half);
      default: break;
    }
  } else {
    switch (p.out_dtype) {
      case B200ISP_U8: RUN(false, uint8_t);
      case B200ISP_U16: RUN(false, uint16_t);
      case B200ISP_F16: RUN(false, __half);
      case B200ISP_F32: RUN(false, float);
      default: break;
    }
  }
#undef RUN
  isp::set_error("process_packed12: unsupported isp/out dtype combination %d/%d", p.isp_dtype, p.out_dtype);
  return B200ISP_E_DTYPE;
}

// The launches of a b200isp_process_packed12 call after its metering: the Reinhard form's sequence (fused_isp.cuh) or the one
// sweep without Reinhard.  p.profile_start / p.profile_stop bracket the pass that writes the output or the maps (the max sweep
// of kExact and the normalise passes stay outside).
static int run_fused(const FramePtrs& fp, int n_frames, const b200isp_fused_params& p, const IspConsts& k, cudaStream_t s) {
  ReinhardPlan plan = reinhard_plan(p, k, n_frames);
  if (plan.form == ReinhardForm::kResizeMap)
    ISP_REQUIRE(p.reinhard_scratch && p.reinhard_scratch_bytes >= plan.bytes, B200ISP_E_ARG,
                "process_packed12: Reinhard with resize needs reinhard_scratch of n_frames * out_height * out_width * 3 ISP-dtype values");
  else if (plan.map_bytes && (!p.reinhard_scratch || p.reinhard_scratch_bytes < plan.map_bytes)) plan = {ReinhardForm::kExact, 0, 0};
  else if (plan.form == ReinhardForm::kF16Table && p.reinhard_scratch_bytes < plan.bytes) plan.form = ReinhardForm::kF16Arith;
  ISP_REQUIRE(!(p.out_yuv420 && plan.form == ReinhardForm::kExact), B200ISP_E_ARG,
              "process_packed12: YUV 4:2:0 output needs Camera16 (f16), Reinhard, u8 and the reinhard_scratch buffer");
  ISP_REQUIRE(!((k.flip & 4) && plan.form == ReinhardForm::kExact), B200ISP_E_ARG,
              "process_packed12: the transposing transforms need the reinhard_scratch buffer (b200isp_reinhard_scratch_bytes)");
  // The extended sweeps (IDS layout, flips in the store) are Malvar only.  The map sweeps write plain images: only the layout counts.
  const bool one_sweep = plan.form != ReinhardForm::kNone && plan.form != ReinhardForm::kExact;
  ISP_REQUIRE(k.kbase == 0 || !(k.ids || (k.flip && !one_sweep)), B200ISP_E_ARG, "process_packed12: the IDS layout %s fused for the Malvar demosaic only",
              one_sweep ? "is" : "/ flips are");
  if (plan.form != ReinhardForm::kNone) {
    // frame_max and frame_max2 are adjacent in the workspace: one memset node
    static_assert(offsetof(Workspace, frame_max2) == offsetof(Workspace, frame_max) + sizeof(float) * B200ISP_MAX_FRAMES, "adjacent");
    const int st = cuda_status(cudaMemsetAsync(k.ws->frame_max, 0, sizeof(float) * 2 * B200ISP_MAX_FRAMES, s), "memset frame_max");
    if (st) return st;
  }

  const bool cam16 = p.isp_dtype == B200ISP_F16;
  FramePtrs sc = fp;                     // the one-sweep forms: each frame's map in the caller's scratch
  for (int f = 0; f < n_frames; ++f) sc.out[f] = (char*)p.reinhard_scratch + (size_t)f * (plan.map_bytes / n_frames);
  IspConsts km = k;                      // the map is a plain dense (H, W, 3) image whatever the output looks like
  km.flip = 0;
  km.orow = 3 * k.W;
  IspConsts kg = k;                      // the gated exact sweeps of the u16 map forms
  kg.gate = 1;
  const long long n_elems = (long long)k.H * k.W * 3;
  auto timed = [&](auto&& pass) {
    record_profile_event(p.profile_start, s);
    const int st = pass();
    record_profile_event(p.profile_stop, s);
    return st;
  };
  auto store = [&] { return timed([&] { return run_sweep(Sweep::kStore, sc, km, p, n_frames, s); }); };
  int st;
  switch (plan.form) {
    case ReinhardForm::kNone:
      if (resizes(p)) return timed([&] { return run_resize(fp, n_frames, p, k, s); });
      return timed([&] { return run_sweep(p.tonemap == B200ISP_TM_NONE ? Sweep::kRgb : Sweep::kLinear, fp, k, p, n_frames, s); });
    case ReinhardForm::kExact:
      // max sweep, then the write sweep recomputes the map.  Both sweeps are bound by instruction issue, not by DRAM, so the
      // second read of the packed frames (1.5 B/px) is cheaper than cutting the call into L2-sized groups whose short launches
      // end in idle tails (measured, profiles/r02_reinhard_diet.txt).
      if ((st = run_sweep(Sweep::kMax, fp, k, p, n_frames, s))) return st;
      return timed([&] { return run_sweep(Sweep::kReinhard, fp, k, p, n_frames, s); });
    case ReinhardForm::kResizeMap: {
      if ((st = timed([&] { return run_resize(sc, n_frames, p, k, s); }))) return st;
      const long long n_out = (long long)p.out_height * p.out_width * 3;
      if (cam16 && n_out % 8 == 0) return run_scratch_out(sc, fp, n_frames, n_out, p.out_dtype, k.gamma, k.ws, 8 * kNumSMs, s);
      return run_resize_normalise(sc, fp, n_frames, n_out, cam16, p.out_dtype, k.gamma, k.ws, s);
    }
    // Camera16: the reference stores the map as f16 anyway -> one sweep writes it to the caller's scratch, a light element-wise
    // pass normalises it (no second sweep)
    case ReinhardForm::kF16Turned:       // the normalise pass turns the image
      if ((st = store())) return st;
      return run_out_transposed(true, sc, fp, n_frames, k, s);
    case ReinhardForm::kF16Yuv:
      if ((st = store())) return st;
      return run_scratch_yuv(sc, fp, n_frames, k, s);
    case ReinhardForm::kF16Table:
      if ((st = store())) return st;
      return run_lut_pass(sc, fp, n_frames, n_elems, (uint8_t*)p.reinhard_scratch + plan.map_bytes, k.gamma, k.ws, s);
    case ReinhardForm::kF16Arith:
      if ((st = store())) return st;
      return run_scratch_out(sc, fp, n_frames, n_elems, p.out_dtype, k.gamma, k.ws, 4 * kNumSMs, s);
    // Camera32 -> u8, color_adapt == 0, gamma in [0.3, 1]: ONE sweep that also stores the map as u16 fixed point (6 B/px
    // scratch) + an element-wise normalise / gamma / quantise pass.  The second demosaic of the two-sweep form (66 of its 106
    // instructions per pixel) disappears; the u8 result is within 1 LSB of the two-sweep result (measured:
    // profiles/r02_reinhard_map16.txt).  Frames whose map does not fit [0, 1) (reinhard_map16_declined) are redone exactly by
    // the gated sweeps.
    case ReinhardForm::kU16Map:
      // the normalise pass runs after the sweep with 8 CTAs per SM; running it under the sweep on a side stream measured
      // 212-186 vs 215 Gpixel/s on cfg3 (profiles/r02_reinhard_map16.txt)
      if ((st = store())) return st;
      if ((st = run_map16_out(sc, fp, n_frames, k, s))) return st;
      if ((st = run_sweep(Sweep::kMaxGated, fp, kg, p, n_frames, s))) return st;
      return run_sweep(Sweep::kReinhardGated, fp, kg, p, n_frames, s);
    case ReinhardForm::kU16Turned:
      // the gated sweeps leave the frames the map declined as plain (H, W, 3) u8 images in their scratch, then ONE pass
      // normalises / turns every frame into the output
      if ((st = store())) return st;
      km.gate = 1;
      if ((st = run_sweep(Sweep::kMaxGated, sc, km, p, n_frames, s))) return st;
      if ((st = run_sweep(Sweep::kReinhardGated, sc, km, p, n_frames, s))) return st;
      return run_out_transposed(false, sc, fp, n_frames, k, s);
  }
  return B200ISP_E_ARG;
}

extern "C" int b200isp_process_packed12(const uint8_t* const* packed_host, void* const* out_host, int n_frames,
                                        const b200isp_fused_params* params, float* metrics, void* workspace,
                                        b200isp_stream stream) {
  FramePtrs fp; IspConsts k;
  ISP_REQUIRE(out_host, B200ISP_E_ARG, "process_packed12: null output list");
  {
    int st = fused_setup("process_packed12", packed_host, out_host, n_frames, params, metrics, workspace, fp, k);
    if (!st) st = process_checks(*params, k);
    if (st) return st;
  }
  const b200isp_fused_params& p = *params;
  ISP_REQUIRE(p.tonemap == B200ISP_TM_NONE || metrics, B200ISP_E_ARG, "process_packed12: metrics required for tone mapping");
  cudaStream_t s = (cudaStream_t)stream;

  if (p.update_metering && p.tonemap != B200ISP_TM_NONE) {
    const int st = with_packed12_sampler(fp, p, k, n_frames, [&](const auto& smp, long long n, float* cache) {
      return launch_metering(smp, n, p.alpha, metrics, metrics, k.ws, s, cache);
    });
    if (st) return st;
  }

  return run_fused(fp, n_frames, p, k, s);
}
