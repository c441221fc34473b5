// The gated exact fallback of the one-sweep Camera32 Reinhard -> u8 path (fused_isp.cuh, run_fused): the ordinary max sweep
// and write sweep (color_adapt == 0, standard layout, u8), instantiated with Epi::kGated so that every warp whose frame the
// u16 map accepted leaves at once.  Frames the map declined (reinhard_map16_declined: a quotient >= 1 was clipped, or the
// frame maximum is tiny) are recomputed exactly as the two-sweep form does: camera_isp.py:177-218.
#include "fused_isp.cuh"

namespace isp {

int run_rmax_gated(const FramePtrs& fp, IspConsts k, int nframes, int rows_per_task, cudaStream_t s) {
  const Stream2Geom g = make_geom2(k.H, k.W, nframes, rows_per_task);
  Packed12Loader2<false, false> ld;
  ld.fp = fp; ld.pitch_words = k.W * 3 / 8; ld.ids = 0;
  int st = B200ISP_OK;
  ISP_DISPATCH_PATTERN(k.pattern, P, {
    EpiReinhardMax2<false, true, false, true> e{fp, k};
    st = launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard_max,gated>", k.kbase != 0);
  });
  return st;
}

int run_write_gated(const FramePtrs& fp, IspConsts k, int nframes, int rows_per_task, cudaStream_t s) {
  const Stream2Geom g = make_geom2(k.H, k.W, nframes, rows_per_task);
  Packed12Loader2<false, false> ld;
  ld.fp = fp; ld.pitch_words = k.W * 3 / 8; ld.ids = 0;
  int st = B200ISP_OK;
  ISP_DISPATCH_PATTERN(k.pattern, P, {
    if (k.gamma != 1.0f) { EpiReinhard2<false, uint8_t, true, true, false, true> e{fp, k}; st = launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard,gated>", k.kbase != 0); }
    else { EpiReinhard2<false, uint8_t, true, false, false, true> e{fp, k}; st = launch_stream2<P>(ld, e, g, s, "isp_stream<reinhard,gated>", k.kbase != 0); }
  });
  return st;
}

}  // namespace isp
