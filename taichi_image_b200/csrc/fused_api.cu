// C entry point of the fused packed12 sweep + the sparse metering launch (see fused_isp.cuh), and the table form of the
// Camera16 Reinhard normalise pass.
#include "fused_isp.cuh"
#include "resize_isp.cuh"

namespace isp {
extern template int run_fused<true, uint8_t>(const FramePtrs&, int, const b200isp_fused_params&, IspConsts, cudaStream_t);
extern template int run_fused<true, uint16_t>(const FramePtrs&, int, const b200isp_fused_params&, IspConsts, cudaStream_t);
extern template int run_fused<true, __half>(const FramePtrs&, int, const b200isp_fused_params&, IspConsts, cudaStream_t);
extern template int run_fused<false, uint8_t>(const FramePtrs&, int, const b200isp_fused_params&, IspConsts, cudaStream_t);
extern template int run_fused<false, uint16_t>(const FramePtrs&, int, const b200isp_fused_params&, IspConsts, cudaStream_t);
extern template int run_fused<false, __half>(const FramePtrs&, int, const b200isp_fused_params&, IspConsts, cudaStream_t);
extern template int run_fused<false, float>(const FramePtrs&, int, const b200isp_fused_params&, IspConsts, cudaStream_t);
}  // namespace isp

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

// ReinhardForm::kF16Table: the table form of the Camera16 normalise pass (see kLutBytes in fused_isp.cuh)
__global__ void __launch_bounds__(256) reinhard_lut_build_kernel(uint8_t* lut /* n_frames x 65536 */, float gamma, const Workspace* ws) {
  const int frame = blockIdx.y;
  const uint32_t v = blockIdx.x * 256 + threadIdx.x;
  const float inv_max = __fdiv_rn(1.0f, fmaxf(1e-6f, __ldcg(&ws->frame_max[frame])));
  float q = __saturatef(__half2float(__ushort_as_half((unsigned short)v)) * inv_max);
  if (gamma != 1.0f) q = fast_pow(q, (float)(1.0 / (double)gamma));
  lut[(size_t)frame * kLutBytes + v] = (uint8_t)Quant<uint8_t>::q(q);
}

__global__ void __launch_bounds__(512) reinhard_lut_out_kernel(const FramePtrs scratch, const FramePtrs fp, long long n16 /* 16-value chunks per frame */,
                                                               const uint8_t* __restrict__ lut) {
  extern __shared__ __align__(16) uint8_t s_lut[];
  const int frame = gridDim.y - 1 - blockIdx.y;       // last frame first: the sweep wrote it last, part of its map is still in L2
  {
    const uint4* g = reinterpret_cast<const uint4*>(lut + (size_t)frame * kLutBytes);
    uint4* s4 = reinterpret_cast<uint4*>(s_lut);
    for (int i = threadIdx.x; i < kLutBytes / 16; i += blockDim.x) s4[i] = __ldg(g + i);
  }
  __syncthreads();
  const uint4* src = reinterpret_cast<const uint4*>(scratch.out[frame]);
  uint4* dst = reinterpret_cast<uint4*>(fp.out[frame]);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (long long)gridDim.x * blockDim.x) {
    const uint4 w0 = __ldcs(src + 2 * i), w1 = __ldcs(src + 2 * i + 1);
    const uint32_t w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t a = s_lut[w[2 * j] & 0xFFFFu], b = s_lut[w[2 * j] >> 16], c = s_lut[w[2 * j + 1] & 0xFFFFu], d = s_lut[w[2 * j + 1] >> 16];
      o[j] = a | (b << 8) | (c << 16) | (d << 24);
    }
    __stcs(dst + i, make_uint4(o[0], o[1], o[2], o[3]));
  }
}

int run_lut_pass(const FramePtrs& sc, const FramePtrs& fp, int n_frames, long long n_elems, uint8_t* lut, float gamma, const Workspace* ws,
                 cudaStream_t s) {
  reinhard_lut_build_kernel<<<dim3(kLutBytes / 256, (unsigned)n_frames), 256, 0, s>>>(lut, gamma, ws);
  int st = cuda_status(cudaPeekAtLastError(), "reinhard_lut_build_kernel");
  if (st) return st;
  static bool attr_set = false;          // per process; the attribute belongs to the function, not to a device context
  if (!attr_set) {
    st = cuda_status(cudaFuncSetAttribute(reinhard_lut_out_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLutBytes), "lut smem attribute");
    if (st) return st;
    attr_set = true;
  }
  const dim3 grid((unsigned)std::min<long long>((n_elems / 16 + 511) / 512, (3 * kNumSMs + n_frames - 1) / n_frames), (unsigned)n_frames);
  reinhard_lut_out_kernel<<<grid, 512, kLutBytes, s>>>(sc, fp, n_elems / 16, lut);
  return cuda_status(cudaPeekAtLastError(), "reinhard_lut_out_kernel");
}
}  // namespace isp

extern "C" size_t b200isp_reinhard_scratch_bytes(const b200isp_fused_params* params, int n_frames) {
  IspConsts k;
  if (!params || fused_consts("reinhard_scratch_bytes", n_frames, *params, k) || process_checks(*params, k)) return 0;
  return reinhard_plan(*params, k, n_frames).bytes;
}

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
  meter_finalize_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(gathered1, gathered2, world, alpha, metrics_prev, metrics_out);
  ISP_LAUNCH_CHECK("meter_finalize_kernel");
  return B200ISP_OK;
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
  const bool cam16 = p.isp_dtype == B200ISP_F16;

  if (p.update_metering && p.tonemap != B200ISP_TM_NONE) {
    const int st = with_packed12_sampler(fp, p, k, n_frames, [&](const auto& smp, long long n, float* cache) {
      return launch_metering(smp, n, p.alpha, metrics, metrics, k.ws, s, cache);
    });
    if (st) return st;
  }

  if (resizes(p)) return run_resize(fp, n_frames, p, k, s);
#define RUN(CAM, T) return run_fused<CAM, T>(fp, n_frames, p, k, s)
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
