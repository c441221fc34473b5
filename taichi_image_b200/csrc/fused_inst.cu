// The sweeps of b200isp_process_packed12 (Sweep, fused_isp.cuh), one translation unit per group so that the 64 streaming-
// kernel variants compile in parallel.  Build with -DISP_INST_CAM16=0|1 and one of
//   -DISP_INST_OUT=<type>   run_out_sweep<CAM16, type>: kRgb / kLinear / kReinhard
//   -DISP_INST_RMAX         run_max_sweep<CAM16>: kMax / kStore (independent of the output dtype)
//   -DISP_INST_GATED        run_gated_sweep: kMaxGated / kReinhardGated (Camera32 -> u8 only)
#include "fused_isp.cuh"

namespace isp {
namespace {

// One sweep of the packed frames fp.in with the epilogue make_epi(std::bool_constant<EXT>{}): fills the row loader, builds
// the geometry and launches the kernel of the Bayer pattern.  EXT is the extended instantiation (IDS layout in the loader,
// flips in the store; see Packed12Loader2), taken where `ext` is set and compiled only where MAY_EXT is.  It is Malvar only:
// run_fused refuses bilinear calls that would need it (the host mirror routes them through the re-pack pass / the
// transform kernel), so its bilinear kernels are never launched.
template <bool CAM16, bool MAY_EXT, class MakeEpi>
int launch_sweep(const FramePtrs& fp, const IspConsts& k, bool ext, int nframes, int rows_per_task, cudaStream_t s,
                 const char* what, MakeEpi make_epi) {
  const Stream2Geom g = make_geom2(k.H, k.W, nframes, rows_per_task);
  auto launch = [&](auto ext_c) -> int {
    constexpr bool EXT = decltype(ext_c)::value;
    Packed12Loader2<CAM16, EXT> ld;
    ld.fp = fp; ld.pitch_words = k.W * 3 / 8; ld.ids = k.ids;
    const auto epi = make_epi(ext_c);
    int st = B200ISP_OK;
    ISP_DISPATCH_PATTERN(k.pattern, P, { st = launch_stream2<P>(ld, epi, g, s, what, !EXT && k.kbase != 0); });
    return st;
  };
  if constexpr (MAY_EXT) {
    if (ext) return launch(std::true_type{});
  }
  return launch(std::false_type{});
}

}  // namespace

template <bool CAM16, typename OutT>
int run_out_sweep(Sweep sw, const FramePtrs& fp, const IspConsts& k, int nframes, int rpt, cudaStream_t s) {
  const bool ext = k.ids != 0 || k.flip != 0;
  auto run = [&](const char* what, auto make_epi) { return launch_sweep<CAM16, true>(fp, k, ext, nframes, rpt, s, what, make_epi); };
  constexpr bool kIspOut = std::is_same<OutT, std::conditional_t<CAM16, __half, float>>::value;
  if constexpr (kIspOut) {
    if (sw == Sweep::kRgb) return run("isp_stream<rgb>", [&](auto x) { return EpiRgb2<CAM16, OutT, decltype(x)::value>{fp, k}; });
  }
  if constexpr (!std::is_same<OutT, float>::value) {
    if (sw == Sweep::kLinear) {
      if constexpr (!CAM16) {
        if (!k.ccm && k.gamma == 1.0f) return run("isp_stream<linear,fast>", [&](auto x) { return EpiLinear2<false, OutT, true, decltype(x)::value>{fp, k}; });
      }
      return run("isp_stream<linear>", [&](auto x) { return EpiLinear2<CAM16, OutT, false, decltype(x)::value>{fp, k}; });
    }
    if (sw == Sweep::kReinhard) {
      // color_adapt == 0 and gamma != 1 are separate instantiations: each kernel's code stays small (instruction cache)
      const bool ca0 = k.ca == 0.f, gam = k.gamma != 1.0f;
      const char* what = "isp_stream<reinhard>";
      if (ca0 && gam) return run(what, [&](auto x) { return EpiReinhard2<CAM16, OutT, true, true, decltype(x)::value>{fp, k}; });
      if (ca0) return run(what, [&](auto x) { return EpiReinhard2<CAM16, OutT, true, false, decltype(x)::value>{fp, k}; });
      if (gam) return run(what, [&](auto x) { return EpiReinhard2<CAM16, OutT, false, true, decltype(x)::value>{fp, k}; });
      return run(what, [&](auto x) { return EpiReinhard2<CAM16, OutT, false, false, decltype(x)::value>{fp, k}; });
    }
  }
  set_error("process_packed12: unsupported isp/out dtype combination %d/%d", CAM16 ? B200ISP_F16 : B200ISP_F32, DT<OutT>::id);
  return B200ISP_E_DTYPE;
}

template <bool CAM16>
int run_max_sweep(Sweep sw, const FramePtrs& fp, const IspConsts& k, int nframes, int rpt, cudaStream_t s) {
  // the max sweeps store nothing through the epilogue's flips: only IDS frames need the extended loader
  auto run = [&](const char* what, auto make_epi) { return launch_sweep<CAM16, true>(fp, k, k.ids != 0, nframes, rpt, s, what, make_epi); };
  const bool ca0 = k.ca == 0.f;
  if (sw == Sweep::kMax) {
    if (ca0) return run("isp_stream<reinhard_max>", [&](auto) { return EpiReinhardMax2<CAM16, true>{fp, k}; });
    return run("isp_stream<reinhard_max>", [&](auto) { return EpiReinhardMax2<CAM16, false>{fp, k}; });
  }
  // Camera16 stores the f16 map (any color_adapt), Camera32 the u16 fixed-point map (color_adapt == 0 only)
  if (ca0) return run("isp_stream<reinhard_store>", [&](auto) { return EpiReinhardMax2<CAM16, true, true>{fp, k}; });
  if constexpr (CAM16) return run("isp_stream<reinhard_store>", [&](auto) { return EpiReinhardMax2<true, false, true>{fp, k}; });
  set_error("process_packed12: the one-sweep Camera32 Reinhard map needs color_adapt == 0");
  return B200ISP_E_ARG;
}

#if defined(ISP_INST_OUT)
template int run_out_sweep<ISP_INST_CAM16 != 0, ISP_INST_OUT>(Sweep, const FramePtrs&, const IspConsts&, int, int, cudaStream_t);
#elif defined(ISP_INST_RMAX)
template int run_max_sweep<ISP_INST_CAM16 != 0>(Sweep, const FramePtrs&, const IspConsts&, int, int, cudaStream_t);
#elif defined(ISP_INST_GATED)
// The gated exact fallback of the one-sweep Camera32 Reinhard -> u8 forms: the ordinary max sweep and write sweep (color_adapt
// == 0, standard layout, u8), instantiated with Epi::kGated so that every warp whose frame the u16 map accepted leaves at once.
// Frames the map declined (reinhard_map16_declined: a quotient >= 1 was clipped, or the frame maximum is tiny) are recomputed
// exactly as the two-sweep form does: camera_isp.py:177-218.
int run_gated_sweep(Sweep sw, const FramePtrs& fp, const IspConsts& k, int nframes, int rpt, cudaStream_t s) {
  auto run = [&](const char* what, auto make_epi) { return launch_sweep<false, false>(fp, k, false, nframes, rpt, s, what, make_epi); };
  if (sw == Sweep::kMaxGated) return run("isp_stream<reinhard_max,gated>", [&](auto) { return EpiReinhardMax2<false, true, false, true>{fp, k}; });
  if (k.gamma != 1.0f) return run("isp_stream<reinhard,gated>", [&](auto) { return EpiReinhard2<false, uint8_t, true, true, false, true>{fp, k}; });
  return run("isp_stream<reinhard,gated>", [&](auto) { return EpiReinhard2<false, uint8_t, true, false, false, true>{fp, k}; });
}
#endif

}  // namespace isp
