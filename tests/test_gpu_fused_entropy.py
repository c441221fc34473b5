"""GPU parity of the fused packed12 path (ISP.process_packed12: csrc/stream2.cuh + csrc/fused_isp.cuh) on FULL-ENTROPY frames.

Smooth test frames hide demosaic mistakes: a tap that reads the wrong same-colour neighbour changes a gradient image by a
few thousandths, which the tone map can round away.  Here every CFA site is an independent uniform 12-bit code:

* ``full``: codes 0..4095 (heavy clipping, full range);
* ``mid``: codes in [1024, 3071]: the demosaiced values clip at 0 or 1 only where the negative taps of the R/B-at-B/R
  filter all meet extreme codes (a few values in 10^5 with the oracle), so nearly every tap shows in the output.

Each frame of a group scales its code range by its own factor (1.0 down to 0.6), so a frame read in place of another
gives a large error, not noise.

A. Sweep geometry x epilogue (``test_sweep_geometry_and_epilogue``): twelve epilogue families, each over every shape of
   ``SHAPES`` (``TURN_SHAPES`` for the transposing normalise pass).  ``axes`` picks the Bayer pattern, ``rows_per_task``,
   ISP dtype, CCM, demosaic and frame kind for each case so that every pair of values of two axes occurs somewhere.
B. Every metering sample (``ISP._meter_cache``, f32 RGB at ``(frame * hs + i) * ws + j``) against the oracle's
   ``load_packed12(f)[::s, ::s]`` for the generic (strides 1..7), fast (8..32) and resized samplers.  The shapes put the
   last sample row / column on ``H-2``, ``H-1``, ``W-2`` or ``W-1``.  The fast sampler's samples also equal the sweep's
   own ``load_packed12`` value at the same pixel bit for bit.  Then the nine metrics over two moving-average steps.
C. Groups of 40 and 64 frames (the C ABI's limit): the per-frame tables past frame 31 and the gated fallback's flag scan of
   frames 32..63; 65 frames are refused.
D. Full size on mid frames against the C oracle: a cfg3 shard and cfg2.
"""
import numpy as np
import pytest
import torch

from oracle import c_oracle
from oracle import isp_oracle as O
from tests.util import rng, to_cuda, to_np, assert_close_int, assert_close_float, assert_u16_from_f16_isp

pytestmark = pytest.mark.gpu

FRAME_MAX_OFS = 10          # Workspace (csrc/common.cuh): counter[8], bounds[2], frame_max[64], frame_max2[64]
SCRIPT_TM = dict(gamma=0.9, intensity=3.0, light_adapt=0.9, color_adapt=0.0)


# ---------------------------------------------------------------- frames
def frame_factor(i):
    """code-range factor of frame i of a group: 1.0 for frame 0, then spread over [0.6, 1.0)"""
    return 1.0 - 0.4 * ((i * 0.6180339887) % 1.0)


def entropy_codes(r, h, w, kind, factor=1.0):
    """(h, w) uint16 12-bit codes, independent per site: ``full`` uniform in [0, 4095 f], ``mid`` in [1024 f, 3071 f]"""
    lo, hi = {"full": (0, 4095), "mid": (1024, 3071)}[kind]
    return r.integers(round(lo * factor), round(hi * factor) + 1, size=(h, w)).astype(np.uint16)


def entropy_frames(r, n, h, w, kind, ids_format=False):
    return [O.encode12(entropy_codes(r, h, w, kind, frame_factor(i)), ids_format=ids_format) for i in range(n)]


# ---------------------------------------------------------------- helpers
def make(dt, pattern="RGGB", **kw):
    from taichi_image_b200 import camera_isp, bayer
    return getattr(camera_isp, "Camera16" if dt == "f16" else "Camera32")(bayer.BayerPattern[pattern], **kw)


def frame_max(n):
    from taichi_image_b200 import _lib
    torch.cuda.synchronize()
    return to_np(_lib.workspace(torch.device("cuda", 0)).view(torch.float32)[FRAME_MAX_OFS:FRAME_MAX_OFS + n])


def declined(mx):
    """csrc/fused_isp.cuh reinhard_map16_declined"""
    return ~((mx < 1.0) & (mx >= 1.0 / 64))


def float_tol(dt):
    return dict(rtol=1e-3, atol=1e-3 if dt == "f16" else 2e-6)


def check_out(got, exp, dt, out, what, gain=1.0):
    """the fused-path tolerances of tests/test_gpu_camera_isp.py: integers within 1 LSB, Camera16 -> u16 one f16 ulp
    through the tone map (tests/util.py), f16 outputs rtol 2e-3 / atol 1e-3.

    A pixel below the metered minimum (the bounds come from every 8th pixel only; full-entropy frames have many) makes the
    linear map's base negative, and the oracle's f16 output of x^(1/gamma) is then NaN, as in the reference.  The ISP
    defines such values as 0 (SURVEY H8; the oracle's integer casts and its Reinhard map do the same), so a NaN of the
    oracle must be exactly 0 in the result."""
    g = to_np(got)
    assert g.shape == exp.shape, f"{what}: shape {g.shape} != {exp.shape}"
    if out == "f16":
        nan = np.isnan(exp)
        assert not np.isnan(g).any(), f"{what}: NaN in the result"
        assert (g[nan] == 0).all(), f"{what}: {int((g[nan] != 0).sum())} values the oracle leaves NaN are not 0"
        assert_close_float(g[~nan], exp[~nan], rtol=2e-3, atol=1e-3, what=what)
    elif out == "u16" and dt == "f16":
        assert_u16_from_f16_isp(g, exp, gain, what)
    else:
        assert_close_int(g, exp, 1, what)


def reinhard_gain(ref, ims, tm):
    """1 / max_out of the oracle's Reinhard map (the slope of the u16 output in the ISP value at gamma 1)"""
    return max(1.0, max(1.0 / float(O.isp_reinhard(im, ref.metrics, tm.get("gamma", 1.0), tm.get("intensity", 1.0),
                                                    tm.get("light_adapt", 1.0), tm.get("color_adapt", 0.0),
                                                    return_intermediate=True)[2]) for im in ims))


def map16_with_covering_bounds(isp, dev, ims, rpt, what, tname="none"):
    """Camera32 one-sweep Reinhard -> u8 (u16 map + normalise pass) with the script's settings under metrics whose bounds
    are [0, 1] and whose statistics are the oracle's for these frames.  With the frames' own metered bounds the u16 map
    declines most full-entropy frames: the bounds come from every 8th pixel, and a pixel far enough below the metered
    minimum gives a map value of 1 or more (csrc/fused_isp.cuh reinhard_map16_declined); the gated exact sweeps then write
    the frame (the exact_u8 family covers that form).  Bounds that hold every pixel keep the map in [0, 1), which is
    asserted from the per-frame maxima.  Returns (results, oracle results)."""
    m = O.metering_update(ims, np.zeros(9, np.float32), 0.0)
    m[0], m[1] = 0.0, 1.0
    isp.metrics = torch.from_numpy(m).cuda()
    got = isp.process_packed12(dev, tonemap="reinhard", update_metering=False, rows_per_task=rpt, **SCRIPT_TM)
    mx = frame_max(len(dev))
    assert not declined(mx).any(), f"{what}: the u16 map declined a frame (maxima {mx}): the fallback got tested"
    tm = (SCRIPT_TM["gamma"], SCRIPT_TM["intensity"], SCRIPT_TM["light_adapt"], SCRIPT_TM["color_adapt"])
    return got, [O.transform(O.isp_reinhard(im, m, *tm, "u8"), tname) for im in ims]


# ---------------------------------------------------------------- A. sweep geometry x epilogue
# W: 8 = one thread column (left and right edge bits both set); 16 = two; 248 = one partial strip of 31 columns; 256 = one
# full strip; 264 = a full strip + a one-column strip; 512 = two strips, no K_CORE; 520 / 776 / 1032 = interior (K_CORE)
# strips and a partial last strip.  H: 4 = border tasks only; 6 = one interior row pair; 10 / 18 / 26 = H == 2 mod 8 (the
# fast sampler's bottom frame rows at stride 8); 16 / 24 = the transposing normalise pass (H % 8 == 0, H >= 16).
SHAPES = [(4, 8), (6, 16), (10, 248), (18, 256), (26, 264), (16, 512), (24, 520), (10, 776), (18, 1032), (4, 1032)]
TURN_SHAPES = [(16, 8), (24, 16), (16, 248), (24, 256), (16, 264), (24, 512), (16, 520), (24, 776), (16, 1032)]
RPTS = (0, 2, 6, 10, 40)            # 0 = auto; 40 > every H here: one task per strip and frame
FAMILIES = ["rgb", "lin_u16", "lin_u8", "lin_f16", "map16", "exact_u8", "rei_u16", "rei_f16", "cam16_u8_yuv", "turn", "ids",
            "resize"]
RESIZES = [dict(resize_width=79), dict(scale=0.469), dict(scale=1.3)]


def axes(fam, i):
    """pattern, rows_per_task, ISP dtype, CCM, demosaic and frame kind of case i of a family: cyclic with distinct strides,
    so that every pair of axis values meets over the whole set; families that own an axis fix it"""
    fi = FAMILIES.index(fam)
    a = dict(pattern=O.PATTERNS[(i + fi) % 4], rpt=RPTS[(2 * i + fi) % 5], dt=("f32", "f16")[(i // 2 + fi) % 2],
             ccm=bool((i + i // 4 + fi) % 2), demosaic=("malvar", "malvar", "bilinear")[(i + 2 * fi) % 3],
             kind=("mid", "mid", "full")[(i + fi) % 3])
    if fam in ("map16", "exact_u8"):
        a["dt"] = "f32"
    if fam == "cam16_u8_yuv":
        a["dt"] = "f16"
    if fam in ("turn", "ids"):
        a["demosaic"] = "malvar"       # the fused transposing pass and the IDS row loader are Malvar-only
    return a


def sweep_cases():
    for fam in FAMILIES:
        for i, shape in enumerate(TURN_SHAPES if fam == "turn" else SHAPES):
            yield pytest.param(fam, i, shape, id=f"{fam}-{shape[0]}x{shape[1]}")


@pytest.mark.parametrize("fam,i,shape", list(sweep_cases()))
def test_sweep_geometry_and_epilogue(cuda, fam, i, shape):
    h, w = shape
    a = axes(fam, i)
    dt, pattern, rpt = a["dt"], a["pattern"], a["rpt"]
    what = f"{fam} {h}x{w} {a}"
    r = rng(1000 + 37 * FAMILIES.index(fam) + i)
    kw = dict(correct_colors=a["ccm"], demosaic=a["demosaic"])
    ref_kw = dict(correct_colors=a["ccm"], demosaic=a["demosaic"])
    if fam == "resize":
        kw.update(RESIZES[(i + 2) % 3])          # every shape resizes to at least one output row
        ref_kw.update(RESIZES[(i + 2) % 3])
    ids = fam == "ids"
    fr = entropy_frames(r, 2, h, w, a["kind"], ids_format=ids)
    dev = [to_cuda(f) for f in fr]

    def ref_isp(**extra):
        return O.ISP(dt, pattern, **ref_kw, **extra)

    def ref_images(ref):
        return [ref.load_packed12(f, ids_format=ids) for f in fr]

    if fam in ("rgb", "resize"):
        # the float RGB epilogue: the direct demosaic probe (a resizing ISP: demosaic + bilinear gather)
        isp = make(dt, pattern, **kw)
        got = isp._run_fused(dev, "none", isp.dtype, None, {}, rows_per_task=rpt)
        for g, e in zip(got, ref_images(ref_isp())):
            assert tuple(g.shape) == e.shape
            assert_close_float(to_np(g), e, **float_tol(dt), what=f"rgb {what}")
    if fam == "resize":
        for tm, out, tkw in (("reinhard", "u8", SCRIPT_TM), ("linear", "u16", dict(gamma=0.8))):
            ref = ref_isp()
            got = make(dt, pattern, **kw).process_packed12(dev, tonemap=tm, dtype=out, rows_per_task=rpt, **tkw)
            ims = ref_images(ref)
            if tm == "reinhard":
                exp = ref.tonemap_reinhard(ims, out_dtype=out, **tkw)
            else:
                exp = ref.tonemap_linear(ims, out_dtype=out, **tkw)
            gain = 1.25 / float(ref.metrics[1] - ref.metrics[0])
            for g, e in zip(got, exp):
                check_out(g, e, dt, out, f"{tm}->{out} {what}", gain)
        return
    if fam == "rgb":
        return

    if fam.startswith("lin_"):
        out, tkw = {"lin_u16": ("u16", dict()), "lin_u8": ("u8", dict(gamma=0.7)), "lin_f16": ("f16", dict(gamma=0.8))}[fam]
        ref = ref_isp()
        got = make(dt, pattern, **kw).process_packed12(dev, tonemap="linear", dtype=out, rows_per_task=rpt, **tkw)
        exp = ref.tonemap_linear(ref_images(ref), out_dtype=out, **tkw)
        gain = max(1.0, 1.0 / tkw.get("gamma", 1.0)) / float(ref.metrics[1] - ref.metrics[0])
        for g, e in zip(got, exp):
            check_out(g, e, dt, out, what, gain)
        return

    if fam == "ids":
        for tm, out, tkw in (("linear", "u16", dict()), ("reinhard", "u8", SCRIPT_TM)):
            ref = ref_isp()
            got = make(dt, pattern, **kw).process_packed12(dev, tonemap=tm, dtype=out, rows_per_task=rpt, ids_format=True, **tkw)
            ims = ref_images(ref)
            exp = ref.tonemap_linear(ims, out_dtype=out) if tm == "linear" else ref.tonemap_reinhard(ims, out_dtype=out, **tkw)
            gain = 1.0 / float(ref.metrics[1] - ref.metrics[0])
            for g, e in zip(got, exp):
                check_out(g, e, dt, out, f"ids {tm}->{out} {what}", gain)
        return

    if fam == "turn":
        # rotate_90 / transpose of the Reinhard -> u8 forms: the element-wise normalise pass turns the image
        # (csrc/normalise.cu reinhard_out_transposed_kernel) -- Camera32 from its u16 map, Camera16 from its f16 map
        from taichi_image_b200.dtypes import u8
        from taichi_image_b200.interpolate import ImageTransform
        tname = ("rotate_90", "transpose")[i % 2]
        ref = ref_isp(transform=tname)
        isp = make(dt, pattern, transform=ImageTransform[tname], **kw)
        assert isp._fused_flip(h, "reinhard", u8, SCRIPT_TM["gamma"], 0.0) & 4, "the call would not take the turning pass"
        if dt == "f32":
            got, exp = map16_with_covering_bounds(isp, dev, ref_images(ref), rpt, what, tname)
        else:
            got = isp.process_packed12(dev, tonemap="reinhard", rows_per_task=rpt, **SCRIPT_TM)
            exp = ref.tonemap_reinhard(ref_images(ref), **SCRIPT_TM)
        for g, e in zip(got, exp):
            assert tuple(g.shape) == (w, h, 3)
            check_out(g, e, dt, "u8", f"{tname} {what}")
        return

    if fam == "cam16_u8_yuv":
        # Camera16 Reinhard -> u8 at gamma != 1: f16 map scratch + table pass; yuv420 from the same map (no RGB image)
        tkw = dict(gamma=0.6, intensity=2.0, light_adapt=0.8)
        ref = ref_isp()
        rgb = make(dt, pattern, **kw).process_packed12(dev, tonemap="reinhard", rows_per_task=rpt, **tkw)
        yuv = make(dt, pattern, **kw).process_packed12(dev, tonemap="reinhard", rows_per_task=rpt, yuv420=True, **tkw)
        exp = ref.tonemap_reinhard(ref_images(ref), **tkw)
        for g, y, e in zip(rgb, yuv, exp):
            check_out(g, e, dt, "u8", f"rgb8 {what}")
            assert np.array_equal(to_np(y), O.rgb_yuv420(to_np(g))), f"yuv420 {what}: not the YUV of the RGB8 result"
        return

    # Reinhard families
    out, tkw, exact = {"map16": ("u8", SCRIPT_TM, False), "exact_u8": ("u8", dict(gamma=0.6), True),
                       "rei_u16": ("u16", dict(intensity=2.0, light_adapt=0.8), False),
                       "rei_f16": ("f16", dict(gamma=0.8), False)}[fam]
    ref = ref_isp()
    if fam == "map16":
        got, exp = map16_with_covering_bounds(make(dt, pattern, **kw), dev, ref_images(ref), rpt, what)
        for g, e in zip(got, exp):
            check_out(g, e, dt, out, what)
        return
    got = make(dt, pattern, reinhard_exact=exact, **kw).process_packed12(dev, tonemap="reinhard", dtype=out, rows_per_task=rpt, **tkw)
    ims = ref_images(ref)
    exp = ref.tonemap_reinhard(ims, out_dtype=out, **tkw)
    gain = reinhard_gain(ref, ims, tkw) if (dt == "f16" and out == "u16") else 1.0
    for g, e in zip(got, exp):
        check_out(g, e, dt, out, what, gain)


# ---------------------------------------------------------------- B. every metering sample
# (stride, (H, W), ISP dtype, pattern, extra ISP arguments); the comment names where the last sample row / column lands
METER_CASES = [
    (1, (10, 16), "f32", "RGGB", dict()),                                   # H-1, W-1
    (2, (18, 24), "f16", "GRBG", dict()),                                   # H-2, W-2
    (3, (10, 56), "f32", "GBRG", dict(correct_colors=True)),                # H-1, W-2
    (3, (26, 64), "f16", "BGGR", dict()),                                   # H-2, W-1
    (4, (18, 40), "f32", "BGGR", dict(demosaic="bilinear")),                # H-2, W-4
    (5, (16, 32), "f32", "RGGB", dict()),                                   # H-1, W-2
    (5, (16, 16), "f16", "GBRG", dict(correct_colors=True)),                # H-1, W-1
    (7, (22, 64), "f32", "GRBG", dict(ids_format=True)),                    # H-1, W-1 (IDS layout)
    (7, (30, 72), "f16", "RGGB", dict(demosaic="bilinear")),                # H-2, W-2
    (7, (6, 16), "f32", "BGGR", dict()),                                    # stride > H: one sample row
    (8, (10, 64), "f32", "RGGB", dict()),                                   # H-2: bottom frame row of the fast sampler
    (8, (18, 1032), "f16", "GRBG", dict(correct_colors=True)),              # H-2
    (8, (10, 520), "f32", "GBRG", dict(ids_format=True)),                   # H-2, IDS layout
    (8, (26, 256), "f32", "BGGR", dict(demosaic="bilinear")),               # H-2, bilinear
    (8, (4, 8), "f16", "RGGB", dict()),                                     # one sample, on the frame
    (16, (18, 64), "f32", "GRBG", dict(correct_colors=True)),               # H-2
    (16, (34, 776), "f16", "BGGR", dict()),                                 # H-2
    (24, (26, 776), "f32", "RGGB", dict(demosaic="bilinear")),              # H-2
    (24, (50, 264), "f16", "GBRG", dict(ids_format=True)),                  # H-2, IDS layout
    (32, (34, 264), "f32", "BGGR", dict()),                                 # H-2
    (32, (10, 256), "f32", "GRBG", dict()),                                 # stride > H
    (8, (40, 96), "f32", "RGGB", dict(resize_width=79)),                    # the resized sampler
    (3, (30, 64), "f16", "GBRG", dict(scale=0.469)),
    (5, (24, 48), "f32", "BGGR", dict(scale=1.3, correct_colors=True)),
]


@pytest.mark.parametrize("stride,shape,dt,pattern,extra", METER_CASES,
                         ids=[f"s{c[0]}-{c[1][0]}x{c[1][1]}-{c[2]}-{c[3]}" + "".join(f"-{k}" for k in c[4]) for c in METER_CASES])
def test_every_metering_sample(cuda, stride, shape, dt, pattern, extra):
    h, w = shape
    kw = dict(extra)
    ids = kw.pop("ids_format", False)
    r = rng(2000 + 7 * stride + h + w)
    isp, ref = make(dt, pattern, metering_stride=stride, **kw), O.ISP(dt, pattern, metering_stride=stride, **kw)
    resizes = any(k in kw for k in ("resize_width", "scale"))
    for step, kind in enumerate(("mid", "full")):
        fr = entropy_frames(r, 3, h, w, kind, ids_format=ids)
        dev = [to_cuda(f) for f in fr]
        isp.process_packed12(dev, tonemap="linear", dtype="u16", ids_format=ids)
        ims = [ref.load_packed12(f, ids_format=ids) for f in fr]
        ho, wo = ims[0].shape[:2]
        hs, ws = -(-ho // stride), -(-wo // stride)
        n = len(fr)
        assert isp._meter_n == n * hs * ws
        samples = to_np(isp._meter_cache[: isp._meter_n * 12].view(torch.float32).reshape(n, hs, ws, 3))
        for f in range(n):
            exp = ims[f][::stride, ::stride].astype(np.float32)
            got = samples[f]
            err = np.abs(got.astype(np.float64) - exp) - (float_tol(dt)["atol"] + float_tol(dt)["rtol"] * np.abs(exp.astype(np.float64)))
            if err.max() > 0:
                bad = np.argwhere(err.max(-1) > 0)
                raise AssertionError(f"step {step} frame {f}: {len(bad)} of {hs * ws} samples off the oracle, first (i, j) "
                                     f"{[tuple(b) for b in bad[:6]]} = pixels {[(int(b[0]) * stride, int(b[1]) * stride) for b in bad[:6]]}")
            if stride % 8 == 0 and not resizes:
                # Packed12FastSampler evaluates the sweep's own formulas (csrc/fused_isp.cuh): the very value of the sweep
                sweep = to_np(isp.load_packed12(dev[f], ids_format=ids).float())[::stride, ::stride]
                same = sweep == got
                assert same.all(), (f"step {step} frame {f}: samples differ from the sweep's value at sample (i, j) "
                                    f"{[tuple(b) for b in np.argwhere(~same.all(-1))[:6]]}")
        ref.update_metering(ims)
        assert_close_float(to_np(isp.metrics), ref.metrics, rtol=1e-4, atol=1e-5, what=f"metrics step {step}")


# ---------------------------------------------------------------- C. large groups
GROUP_H, GROUP_W = 24, 64


@pytest.mark.parametrize("n", [40, 64])
@pytest.mark.parametrize("case", ["cam32_map16_u8", "cam32_linear_u16", "cam16_reinhard_u8"])
def test_large_groups_every_frame(cuda, n, case):
    """n distinct full-entropy frames in one call: per-frame pointers, per-frame maxima and the normalise passes' frame
    index (blockIdx.y) past frame 7 and past frame 31"""
    r = rng(3000 + n)
    kinds = ("mid", "full")
    fr = [O.encode12(entropy_codes(r, GROUP_H, GROUP_W, kinds[i % 2], frame_factor(i))) for i in range(n)]
    dev = [to_cuda(f) for f in fr]
    dt = "f16" if case.startswith("cam16") else "f32"
    ref = O.ISP(dt)
    isp = make(dt)
    ims = [ref.load_packed12(f) for f in fr]
    if case == "cam32_linear_u16":
        got = isp.process_packed12(dev, tonemap="linear", dtype="u16")
        exp = ref.tonemap_linear(ims, out_dtype="u16")
    else:
        tm = SCRIPT_TM if case == "cam32_map16_u8" else dict(gamma=0.6, intensity=2.0, light_adapt=0.8)
        got = isp.process_packed12(dev, tonemap="reinhard", **tm)
        if dt == "f32":
            mx = frame_max(n)
            assert not declined(mx).any(), f"the u16 map declined frames {np.flatnonzero(declined(mx))}"
        exp = ref.tonemap_reinhard(ims, **tm)
    assert_close_float(to_np(isp.metrics), ref.metrics, rtol=1e-4, atol=1e-5, what="metrics")
    for k, (g, e) in enumerate(zip(got, exp)):
        assert_close_int(to_np(g), e, 1, f"{case} frame {k} of {n}")


def _grey_frames(r, n, cyan):
    """frames of a distinct grey level each (0.52 .. 0.70, +-5 % noise); frames in ``cyan`` carry a saturated cyan block,
    whose red channel lies far below the preset metered minimum: the u16 map declines them
    (tests/test_gpu_reinhard_map16.py _cyan_frames)"""
    out = []
    for i in range(n):
        g = 0.52 + 0.18 * ((i * 0.6180339887) % 1.0)
        rgb = np.full((GROUP_H, GROUP_W, 3), g, np.float32) + 0.1 * (r.random((GROUP_H, GROUP_W, 3), dtype=np.float32) - 0.5)
        if i in cyan:
            rgb[8:24, 16:48] = (0.0, 1.0, 1.0)
        out.append(O.encode12(O.rgb_to_bayer(rgb, "RGGB"), scaled=True))
    return out


@pytest.mark.parametrize("n,cyan", [(64, (1, 33, 63)), (40, (1, 33)), (64, (40,)), (40, (33,))])
def test_large_group_declined_frames(cuda, n, cyan):
    """Camera32 one-sweep Reinhard -> u8 with preset metrics: exactly the cyan frames are declined and redone by the gated
    exact sweeps (bit for bit the reinhard_exact=True result); the others keep the map.  Declined frames only past frame 31
    take the second iteration of the gated kernels' per-frame flag scan (stream2_kernel, one lane per frame)."""
    r = rng(3100 + n + sum(cyan))
    fr = _grey_frames(r, n, set(cyan))
    dev = [to_cuda(f) for f in fr]
    m = torch.tensor([0.4, 1.0, -3.0, 0.0, -1.0, 0.4, 0.4, 0.4, 0.4], dtype=torch.float32, device="cuda")
    fast, exact = make("f32"), make("f32", reinhard_exact=True)
    fast.metrics, exact.metrics = m.clone(), m.clone()
    got = fast.process_packed12(dev, tonemap="reinhard", update_metering=False, gamma=0.9)
    mx = frame_max(n)
    assert list(np.flatnonzero(declined(mx))) == list(cyan), f"declined frames {np.flatnonzero(declined(mx))}, maxima {mx}"
    two = exact.process_packed12(dev, tonemap="reinhard", update_metering=False, gamma=0.9)
    ref = O.ISP("f32")
    for k, (g, t, f) in enumerate(zip(got, two, fr)):
        if k in cyan:
            assert torch.equal(g, t), f"declined frame {k}: not the exact form"
        e = O.isp_reinhard(ref.load_packed12(f), to_np(m), 0.9, 1.0, 1.0, 0.0, "u8")
        assert_close_int(to_np(g), e, 1, f"frame {k} of {n}")


def test_65_frames_are_refused(cuda):
    from taichi_image_b200 import _lib
    from taichi_image_b200.dtypes import u16
    r = rng(3200)
    dev = [to_cuda(O.encode12(entropy_codes(r, 8, 16, "mid")))] * 65
    isp = make("f32")
    with pytest.raises(AssertionError):
        isp.process_packed12(dev, tonemap="linear", dtype="u16")
    isp.metrics = torch.zeros(9, dtype=torch.float32, device="cuda")
    with pytest.raises(_lib.B200ISPError, match="too many frames"):
        isp.meter_packed12(dev, 0.0)
    # the C entry point itself refuses before it touches the 64-entry frame tables
    outs = [torch.empty((8, 16, 3), dtype=torch.uint16, device="cuda") for _ in range(65)]
    p = isp._fused_params(dev[:1], "linear", u16, {})
    st = _lib.lib.b200isp_process_packed12(_lib.ptr_array(dev), _lib.ptr_array(outs), 65, p, isp.metrics.data_ptr(),
                                           _lib.workspace(isp.device).data_ptr(), _lib.stream_ptr(isp.device))
    assert st == -6, f"status {st}"


# ---------------------------------------------------------------- D. full size, full entropy
def mid_packed(n, h, w, seed):
    """mid frames (codes in [1024 f, 3071 f], f = frame_factor(i)) generated and packed on the device; + host copies"""
    from tests.test_gpu_fullsize import packed_from_cfa
    g = torch.Generator(device="cuda").manual_seed(seed)
    dev, host = [], []
    for i in range(n):
        f = frame_factor(i)
        cfa = torch.randint(round(1024 * f), round(3071 * f) + 1, (h, w), generator=g, device="cuda", dtype=torch.int32)
        dev.append(packed_from_cfa(cfa))
        host.append(dev[-1].cpu().numpy())
    return dev, host


@pytest.mark.parametrize("name,n,h,w,tonemap,out,tm", [
    ("cfg3_shard", 6, 3000, 4096, "reinhard", "u8", SCRIPT_TM),
    ("cfg2", 2, 3648, 5472, "linear", "u16", dict(gamma=1.0)),
])
def test_full_size_mid_frames_vs_c_oracle(cuda, name, n, h, w, tonemap, out, tm):
    """the real strip counts and the auto rows_per_task on content where every seam shows: one step against the C oracle"""
    from tests.test_gpu_fullsize import compare_with_c_oracle
    dev, host = mid_packed(n, h, w, seed=4000 + n)
    isp = make("f32")
    got = isp.process_packed12(dev, tonemap=tonemap, dtype=out, **tm)
    if tonemap == "reinhard":
        mx = frame_max(n)
        assert not declined(mx).any(), f"the u16 map declined frames {np.flatnonzero(declined(mx))}"
    exp, metrics = c_oracle.process(host, "RGGB", False, out, tonemap, None, tm.get("gamma", 1.0), tm.get("intensity", 1.0),
                                    tm.get("light_adapt", 1.0), tm.get("color_adapt", 0.0), stride=8)
    np.testing.assert_allclose(isp.metrics.cpu().numpy(), metrics, rtol=2e-5, atol=2e-6, err_msg=name)
    compare_with_c_oracle(f"{name} mid", got, exp)
