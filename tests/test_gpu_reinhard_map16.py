"""GPU parity of the one-sweep Camera32 Reinhard -> u8 path (csrc/fused_isp.cuh: EpiReinhardMax2<Camera32, STORE> writes the
map of camera_isp.py:200-211 as u16 fixed point, reinhard_map16_out_kernel normalises / gamma-maps / quantises it):

* against the oracle and against the exact two-sweep form (``ISP(reinhard_exact=True)``): <= 1 LSB of u8, and the fraction of
  values that differ from the exact form at all stays small (the quantisation step is 2^-16 of the map's range);
* frames whose map leaves [0, 1) -- a channel far below the metered minimum makes a denominator negative and its quotient
  large, which the reference takes into max_out (camera_isp.py:213) -- are declined by the map and redone by the gated exact
  sweeps: their result equals the two-sweep form bit for bit;
* outputs the path does not apply to (u16, gamma > 1, color_adapt != 0, pitched tiles) still take the exact form.
"""
import numpy as np
import pytest
import torch

from oracle import isp_oracle as O
from tests.util import rng, packed_frame, to_cuda, to_np, assert_close_int

pytestmark = pytest.mark.gpu

TM = [dict(), dict(gamma=0.6), dict(gamma=0.9, intensity=3.0, light_adapt=0.9, color_adapt=0.0), dict(gamma=0.35, intensity=0.5)]
FRAME_MAX_OFS = 10          # Workspace (csrc/common.cuh): counter[8], bounds[2], frame_max[64], frame_max2[64]


def make(exact, **kw):
    from taichi_image_b200 import camera_isp, bayer
    pattern = kw.pop("bayer_pattern", "RGGB")
    return camera_isp.Camera32(bayer.BayerPattern[pattern], reinhard_exact=exact, **kw)


def frame_max(n):
    from taichi_image_b200 import _lib
    torch.cuda.synchronize()
    return to_np(_lib.workspace(torch.device("cuda", 0)).view(torch.float32)[FRAME_MAX_OFS:FRAME_MAX_OFS + n])


def declined(mx):
    return ~((mx < 1.0) & (mx >= 1.0 / 64))


@pytest.mark.parametrize("pattern", O.PATTERNS)
@pytest.mark.parametrize("tm", TM)
@pytest.mark.parametrize("shape", [(40, 64), (30, 776)])
def test_map16_within_one_lsb_of_oracle_and_exact_form(cuda, pattern, tm, shape):
    r = rng(71)
    fast, exact, ref = make(False, bayer_pattern=pattern), make(True, bayer_pattern=pattern), O.ISP("f32", pattern)
    for step in range(2):
        fr = [packed_frame(r, *shape, pattern) for _ in range(3)]
        dev = [to_cuda(f) for f in fr]
        got = fast.process_packed12(dev, tonemap="reinhard", **tm)
        mx = frame_max(len(fr))
        assert not declined(mx).any(), f"smooth frames must take the map: frame maxima {mx}"
        two = exact.process_packed12(dev, tonemap="reinhard", **tm)
        exp = ref.tonemap_reinhard([ref.load_packed12(f) for f in fr], **tm)
        assert torch.equal(fast.metrics, exact.metrics)
        for g, t, e in zip(got, two, exp):
            assert g.dtype == torch.uint8
            assert_close_int(to_np(g), e, 1, f"oracle {pattern} {tm} step {step}")
            frac = assert_close_int(to_np(g), to_np(t), 1, f"exact form {pattern} {tm} step {step}")
            assert frac < 0.02, f"{frac:.4f} of the values differ from the exact form"


def _cyan_frames(r, h, w):
    """saturated cyan blocks on a mid-grey ground: with a metered minimum well above 0 their red channel lies far below it"""
    out = []
    for i in range(3):
        rgb = np.full((h, w, 3), 0.55, np.float32) + 0.02 * (r.random((h, w, 3), dtype=np.float32) - 0.5)
        if i != 1:                                              # frame 1 stays plain: it must take the map
            rgb[8:24, 16:48] = (0.0, 1.0, 1.0)
        out.append(O.encode12(O.rgb_to_bayer(rgb, "RGGB"), scaled=True))
    return out


def test_map16_declined_frames_equal_the_exact_form(cuda):
    r = rng(72)
    fr = _cyan_frames(r, 40, 64)
    dev = [to_cuda(f) for f in fr]
    fast, exact = make(False), make(True)
    # metrics as a previous, brighter scene would have left them: bounds [0.4, 1.0] (camera_isp.py:102-115 layout)
    m = torch.tensor([0.4, 1.0, -3.0, 0.0, -1.0, 0.4, 0.4, 0.4, 0.4], dtype=torch.float32, device="cuda")
    fast.metrics, exact.metrics = m.clone(), m.clone()
    got = fast.process_packed12(dev, tonemap="reinhard", update_metering=False, gamma=0.9)
    mx = frame_max(3)
    assert declined(mx)[0] and declined(mx)[2] and not declined(mx)[1], f"frame maxima {mx}"
    two = exact.process_packed12(dev, tonemap="reinhard", update_metering=False, gamma=0.9)
    assert torch.equal(got[0], two[0]) and torch.equal(got[2], two[2]), "declined frames are redone by the exact sweeps"
    assert_close_int(to_np(got[1]), to_np(two[1]), 1, "accepted frame")
    ref = O.ISP("f32")
    for g, f in zip(got, fr):
        e = O.isp_reinhard(ref.load_packed12(f), to_np(m), 0.9, 1.0, 1.0, 0.0, "u8")
        assert_close_int(to_np(g), e, 1, "oracle, preset metrics")


def test_map16_random_frames(cuda):
    """pure-random 12-bit frames: heavy clamping, quotients at and beyond 1 -- whichever way each frame goes, <= 1 LSB"""
    r = rng(73)
    fast, exact, ref = make(False), make(True), O.ISP("f32")
    fr = [packed_frame(r, 64, 96, smooth=False) for _ in range(4)]
    dev = [to_cuda(f) for f in fr]
    tm = dict(gamma=0.9, intensity=3.0, light_adapt=0.9)
    got = fast.process_packed12(dev, tonemap="reinhard", **tm)
    two = exact.process_packed12(dev, tonemap="reinhard", **tm)
    exp = ref.tonemap_reinhard([ref.load_packed12(f) for f in fr], **tm)
    for g, t, e in zip(got, two, exp):
        assert_close_int(to_np(g), to_np(t), 1, "exact form")
        assert_close_int(to_np(g), e, 1, "oracle")


@pytest.mark.parametrize("kw,out", [(dict(gamma=1.5), "u8"), (dict(color_adapt=0.3), "u8"), (dict(), "u16")])
def test_outside_the_map16_conditions_the_exact_form_runs(cuda, kw, out):
    r = rng(74)
    from taichi_image_b200 import dtypes
    fast, exact = make(False), make(True)
    dev = [to_cuda(packed_frame(r, 40, 64)) for _ in range(2)]
    a = fast.process_packed12(dev, tonemap="reinhard", dtype=getattr(dtypes, out), **kw)
    b = exact.process_packed12(dev, tonemap="reinhard", dtype=getattr(dtypes, out), **kw)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_map16_bilinear_demosaic_and_full_rows(cuda):
    """the bilinear instantiation of the map sweep, at a width with interior strips and a partial last strip"""
    r = rng(75)
    fast, exact = make(False, demosaic="bilinear"), make(True, demosaic="bilinear")
    dev = [to_cuda(packed_frame(r, 36, 520)) for _ in range(2)]
    a = fast.process_packed12(dev, tonemap="reinhard", gamma=0.8)
    b = exact.process_packed12(dev, tonemap="reinhard", gamma=0.8)
    for x, y in zip(a, b):
        assert_close_int(to_np(x), to_np(y), 1, "bilinear")


@pytest.mark.parametrize("n", [4, 5, 7])
def test_map16_overlapped_groups(cuda, n):
    """>= 4 frames: the frames are cut into groups and the normalise pass of a group runs on a side stream under the next
    group's map sweep (fork / join through events inside the call) -- same results, also back to back and with a declined frame"""
    r = rng(76)
    fast, exact, ref = make(False), make(True), O.ISP("f32")
    tm = dict(gamma=0.9, intensity=3.0, light_adapt=0.9)
    for step in range(3):
        fr = [packed_frame(r, 30, 776) for _ in range(n)]
        if step == 2:
            fr[1] = packed_frame(r, 30, 776, smooth=False)          # pure noise: quotients beyond 1 -> declined -> gated exact sweeps
        dev = [to_cuda(f) for f in fr]
        got = fast.process_packed12(dev, tonemap="reinhard", **tm)
        two = exact.process_packed12(dev, tonemap="reinhard", **tm)
        exp = ref.tonemap_reinhard([ref.load_packed12(f) for f in fr], **tm)
        for i, (g, t, e) in enumerate(zip(got, two, exp)):
            assert_close_int(to_np(g), to_np(t), 1, f"exact form, step {step} frame {i}")
            assert_close_int(to_np(g), e, 1, f"oracle, step {step} frame {i}")


@pytest.mark.parametrize("cam,gamma", [("Camera32", 0.9), ("Camera32", 1.0), ("Camera16", 0.6)])
def test_scratch_and_outputs_stay_inside_their_buffers(cuda, cam, gamma):
    """guard bands (compute-sanitizer is not available on the GPU pool): the map scratch -- exactly the size the host mirror asks
    for -- and the outputs are views into canary-filled buffers; the map sweep, the normalise passes (arithmetic, table, dense)
    and the gated sweeps must leave every canary byte alone"""
    from taichi_image_b200 import camera_isp, bayer
    r = rng(78)
    n, h, w = 5, 30, 776
    isp = getattr(camera_isp, cam)(bayer.BayerPattern.RGGB)
    dev = [to_cuda(packed_frame(r, h, w)) for _ in range(n)]
    dev[3] = to_cuda(packed_frame(r, h, w, smooth=False))                 # a declined frame (Camera32): the gated sweeps run too
    need = n * h * w * 6 + n * 65536
    pad = 1 << 16
    sbuf = torch.full((need + 2 * pad,), 0xA5, dtype=torch.uint8, device="cuda")
    isp._reinhard_scratch = sbuf[pad:pad + need]
    obuf = torch.full((n, h * w * 3 + pad), 0x5A, dtype=torch.uint8, device="cuda")
    outs = [obuf[i, :h * w * 3].view(h, w, 3) for i in range(n)]
    ref = getattr(camera_isp, cam)(bayer.BayerPattern.RGGB).process_packed12(dev, tonemap="reinhard", gamma=gamma)
    got = isp.process_packed12(dev, tonemap="reinhard", gamma=gamma, out=outs)
    torch.cuda.synchronize()
    assert isp._reinhard_scratch.data_ptr() == sbuf[pad:].data_ptr(), "the preset scratch was replaced: its size no longer matches the host mirror"
    assert bool((sbuf[:pad] == 0xA5).all()) and bool((sbuf[pad + need:] == 0xA5).all()), "write outside the map scratch"
    assert bool((obuf[:, h * w * 3:] == 0x5A).all()), "write outside an output image"
    for g, e in zip(got, ref):
        assert torch.equal(g, e)
