// Kernels and host orchestration of the fused demosaic + resize gather (resize_isp.cuh has the per-pixel front end).
#include "resize_sweep.cuh"

namespace isp {

// per-output-pixel gather (up-scaling, or when the sweep form does not apply): one thread per output pixel
template <bool CAM16, int MODE, typename OutT>
__global__ void __launch_bounds__(256) resize_gather_kernel(const ResizeSrc<CAM16> src, const FramePtrs outs) {
  const int co = blockIdx.x * blockDim.x + threadIdx.x, ro = blockIdx.y, frame = blockIdx.z;
  const IspConsts& k = src.k;
  float mx = 0.f;
  if (co < src.Wo) {
    ResizeTone<CAM16, MODE, OutT> tone;
    tone.init(k, frame);
    float rgb[3];
    src.pixel(frame, ro, co, rgb);
    mx = tone.apply(rgb, reinterpret_cast<OutT*>(outs.out[frame]) + ((size_t)ro * src.Wo + co) * 3);
  }
  if constexpr (MODE == RZ_RSTORE) {
    mx = warp_max(mx);
    if ((threadIdx.x & 31) == 0 && mx > 0.f) atomicMax(reinterpret_cast<unsigned int*>(&k.ws->frame_max[frame]), __float_as_uint(mx));
  }
}

// One pass over the packed frames -> output-resolution images (io.out): the sweep form for down-scaling, the gather
// otherwise.  Instantiated per (ISP dtype, mode) in resize_inst.cu.
template <bool CAM16, int MODE, typename OutT>
int run_resize_pass(const FramePtrs& io, const IspConsts& k, const b200isp_fused_params& p, int n_frames, cudaStream_t s);

template <bool CAM16, int MODE, typename OutT>
int run_resize_pass_impl(const FramePtrs& io, const IspConsts& k0, const b200isp_fused_params& p, int n_frames, cudaStream_t s) {
  IspConsts k = k0;
  const ResizeSrc<CAM16> src = make_resize_src<CAM16>(io, k, p);
  const bool sweep = p.scale_r <= 1.0f && p.scale_c <= 1.0f && p.out_width >= 64 && p.out_height >= 8 && !p.resize_gather;
  if (!sweep) {
    const dim3 grid((unsigned)((p.out_width + 255) / 256), (unsigned)p.out_height, (unsigned)n_frames);
    resize_gather_kernel<CAM16, MODE, OutT><<<grid, 256, 0, s>>>(src, io);
    return cuda_status(cudaPeekAtLastError(), "resize_gather_kernel");
  }
  const ResizeTasks rt = make_resize_tasks(k.H, k.W, n_frames, p.out_height, p.scale_r, p.rows_per_task);
  Packed12Loader2<CAM16> ld;
  ld.fp = io; ld.pitch_words = k.W * 3 / 8; ld.ids = 0;
  const EpiResize2<CAM16, MODE, OutT> epi{io, k, p.out_height, p.out_width, p.scale_r, p.scale_c};
  const long long blocks = (rt.total_tasks + kS2Warps - 1) / kS2Warps;
  ISP_DISPATCH_PATTERN(k.pattern, P, {
    if (k.kbase != 0) stream2_resize_kernel<P, true, Packed12Loader2<CAM16>, EpiResize2<CAM16, MODE, OutT>><<<(unsigned)blocks, ISP_S2_THREADS, 0, s>>>(ld, epi, rt);
    else stream2_resize_kernel<P, false, Packed12Loader2<CAM16>, EpiResize2<CAM16, MODE, OutT>><<<(unsigned)blocks, ISP_S2_THREADS, 0, s>>>(ld, epi, rt);
  });
  int st = cuda_status(cudaPeekAtLastError(), "stream2_resize_kernel");
  if (st) return st;
  const int nbound = rt.g.warps_per_row - 1;                 // inner strip boundaries
  if (nbound > 0) {
    const dim3 grid((unsigned)((p.out_height + 127) / 128), (unsigned)nbound, (unsigned)n_frames);
    resize_orphans_kernel<CAM16, MODE, OutT><<<grid, 128, 0, s>>>(src, io, nbound);
    st = cuda_status(cudaPeekAtLastError(), "resize_orphans_kernel");
  }
  return st;
}

#ifndef ISP_RZ_INST
extern template int run_resize_pass<true, RZ_RGB, __half>(const FramePtrs&, const IspConsts&, const b200isp_fused_params&, int, cudaStream_t);
extern template int run_resize_pass<false, RZ_RGB, float>(const FramePtrs&, const IspConsts&, const b200isp_fused_params&, int, cudaStream_t);
extern template int run_resize_pass<true, RZ_RSTORE, __half>(const FramePtrs&, const IspConsts&, const b200isp_fused_params&, int, cudaStream_t);
extern template int run_resize_pass<false, RZ_RSTORE, float>(const FramePtrs&, const IspConsts&, const b200isp_fused_params&, int, cudaStream_t);
#define ISP_RZ_EXT(CAM, T) extern template int run_resize_pass<CAM, RZ_LINEAR, T>(const FramePtrs&, const IspConsts&, const b200isp_fused_params&, int, cudaStream_t);
ISP_RZ_EXT(true, uint8_t) ISP_RZ_EXT(true, uint16_t) ISP_RZ_EXT(true, __half)
ISP_RZ_EXT(false, uint8_t) ISP_RZ_EXT(false, uint16_t) ISP_RZ_EXT(false, __half)
#undef ISP_RZ_EXT

template <bool CAM16>
static int run_resize_t(const FramePtrs& io, int n_frames, const b200isp_fused_params& p, const IspConsts& k, cudaStream_t s) {
  using IspT = std::conditional_t<CAM16, __half, float>;
  if (p.tonemap == B200ISP_TM_NONE) return run_resize_pass<CAM16, RZ_RGB, IspT>(io, k, p, n_frames, s);
  if (p.tonemap == B200ISP_TM_REINHARD) return run_resize_pass<CAM16, RZ_RSTORE, IspT>(io, k, p, n_frames, s);
  switch (p.out_dtype) {
    case B200ISP_U8: return run_resize_pass<CAM16, RZ_LINEAR, uint8_t>(io, k, p, n_frames, s);
    case B200ISP_U16: return run_resize_pass<CAM16, RZ_LINEAR, uint16_t>(io, k, p, n_frames, s);
    default: return run_resize_pass<CAM16, RZ_LINEAR, __half>(io, k, p, n_frames, s);
  }
}

int run_resize(const FramePtrs& io, int n_frames, const b200isp_fused_params& p, const IspConsts& k, cudaStream_t s) {
  return p.isp_dtype == B200ISP_F16 ? run_resize_t<true>(io, n_frames, p, k, s) : run_resize_t<false>(io, n_frames, p, k, s);
}
#endif

}  // namespace isp
