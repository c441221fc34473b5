// Explicit instantiations of the fused sweep, one translation unit per (ISP dtype, output dtype) so
// the 64 streaming-kernel variants compile in parallel.  Build with
//   -DISP_INST_CAM16=0|1  and either  -DISP_INST_OUT=<type>  or  -DISP_INST_RMAX
#include "fused_isp.cuh"

namespace isp {
#ifdef ISP_INST_RMAX
template int run_rmax<ISP_INST_CAM16 != 0>(const FramePtrs&, IspConsts, int, int, cudaStream_t);
template int run_rstore<ISP_INST_CAM16 != 0>(const FramePtrs&, IspConsts, int, int, cudaStream_t, void*, void*);
#else
template int run_fused<ISP_INST_CAM16 != 0, ISP_INST_OUT>(const FramePtrs&, int, const b200isp_fused_params&, IspConsts, cudaStream_t);
#endif
}  // namespace isp
