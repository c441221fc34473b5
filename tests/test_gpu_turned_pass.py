"""Transposing ISP transforms (interpolate.py:36-56; rotate_90 is the default of scripts/tonemap_scan.py) applied by the
element-wise normalise pass of the one-sweep Reinhard -> u8 forms (csrc/normalise.cu reinhard_out_transposed_kernel):

* the turned result equals ``interpolate.transform`` of the untransformed result of the SAME path bit for bit (the pass runs
  the same arithmetic; only the store differs) -- Camera16 (f16 map, arithmetic and table pass) and Camera32 (u16 map), all
  four transforms, tiles of 128 x 16 that are full, ragged in both directions and single;
* Camera32 frames the u16 map declined are redone by the gated exact sweeps into the scratch and turned by the same pass;
* row-pitched outputs (rig.GridOutput tiles), the CUDA-graph stream and the reference comparison through the oracle.
"""
import numpy as np
import pytest
import torch

from oracle import isp_oracle as O
from tests.util import rng, packed_frame, to_cuda, to_np, assert_close_int

pytestmark = pytest.mark.gpu

TRANSPOSING = ["rotate_90", "rotate_270", "transpose", "transverse"]


def make(dt, **kw):
    from taichi_image_b200 import camera_isp, bayer
    cls = camera_isp.Camera16 if dt == "f16" else camera_isp.Camera32
    return cls(bayer.BayerPattern.RGGB, **kw)


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("tname", TRANSPOSING)
@pytest.mark.parametrize("shape", [(40, 64), (16, 776), (136, 72), (264, 1032), (128, 16)])
def test_turned_pass_equals_transform_of_the_plain_result(cuda, dt, tname, shape):
    from taichi_image_b200.interpolate import ImageTransform, transform
    t = ImageTransform[tname]
    r = rng(311)
    h, w = shape
    cu = [to_cuda(packed_frame(r, h, w)) for _ in range(3)]
    # the last setting keeps Camera16 on the turned pass (any gamma / color_adapt) and sends Camera32 to the exact sweeps +
    # transform kernel: equal to the transform of the plain result either way
    for kw in (dict(gamma=0.9, intensity=2.0), dict(), dict(gamma=0.45, light_adapt=0.8), dict(gamma=1.2, color_adapt=0.5)):
        plain, turned = make(dt), make(dt, transform=t)
        exp = [transform(o, t) for o in plain.process_packed12(cu, tonemap="reinhard", **kw)]
        assert tuple(exp[0].shape) == (w, h, 3)
        bufs = [torch.full_like(e, 77) for e in exp]
        got = turned.process_packed12(cu, tonemap="reinhard", out=bufs, **kw)
        assert got[0].data_ptr() == bufs[0].data_ptr(), "the pass writes the caller's (W, H, 3) buffers itself"
        assert torch.equal(turned.metrics, plain.metrics)
        for g, e in zip(got, exp):
            assert torch.equal(g, e), f"{dt} {tname} {shape} {kw}"


@pytest.mark.parametrize("tname", ["rotate_90", "transverse"])
def test_turned_pass_against_the_oracle(cuda, tname):
    from taichi_image_b200.interpolate import ImageTransform
    r = rng(312)
    fr = [packed_frame(r, 48, 136) for _ in range(2)]
    for dt in ("f16", "f32"):
        isp, ref = make(dt, transform=ImageTransform[tname]), O.ISP(dt, transform=tname)
        got = isp.process_packed12([to_cuda(f) for f in fr], tonemap="reinhard", gamma=0.9)
        exp = ref.tonemap_reinhard([ref.load_packed12(f) for f in fr], gamma=0.9)
        for g, e in zip(got, exp):
            assert tuple(g.shape) == e.shape == (136, 48, 3)
            assert_close_int(to_np(g), e, 1, f"{dt} {tname}")


def test_turned_pass_with_declined_frames(cuda):
    """saturated cyan blocks under preset bounds: frames 0 and 2 leave the u16 map's range -> gated exact sweeps -> turned"""
    from taichi_image_b200.interpolate import ImageTransform, transform
    from tests.test_gpu_reinhard_map16 import _cyan_frames, frame_max, declined
    r = rng(72)
    dev = [to_cuda(f) for f in _cyan_frames(r, 40, 64)]
    m = torch.tensor([0.4, 1.0, -3.0, 0.0, -1.0, 0.4, 0.4, 0.4, 0.4], dtype=torch.float32, device="cuda")
    for tname in TRANSPOSING:
        t = ImageTransform[tname]
        plain, turned = make("f32"), make("f32", transform=t)
        plain.metrics, turned.metrics = m.clone(), m.clone()
        exp = [transform(o, t) for o in plain.process_packed12(dev, tonemap="reinhard", update_metering=False, gamma=0.9)]
        got = turned.process_packed12(dev, tonemap="reinhard", update_metering=False, gamma=0.9)
        mx = frame_max(3)
        assert declined(mx)[0] and declined(mx)[2] and not declined(mx)[1], f"frame maxima {mx}"
        for i, (g, e) in enumerate(zip(got, exp)):
            assert torch.equal(g, e), f"{tname} frame {i}"


@pytest.mark.parametrize("dt", ["f16", "f32"])
def test_turned_pass_into_pitched_grid_tiles(cuda, dt):
    """rotate_90 straight into row-pitched tiles of one grid image (scripts/tonemap_scan.py:91-100 with its default transform)"""
    from taichi_image_b200.interpolate import ImageTransform, transform
    r = rng(313)
    h, w, n = 48, 72, 3
    cu = [to_cuda(packed_frame(r, h, w)) for _ in range(n)]
    plain, turned = make(dt), make(dt, transform=ImageTransform.rotate_90)
    exp = [transform(o, ImageTransform.rotate_90) for o in plain.process_packed12(cu, tonemap="reinhard", gamma=0.9)]
    grid = torch.zeros((w, n * h + 16, 3), dtype=torch.uint8, device="cuda")        # n tiles of (w, h) side by side + padding
    tiles = [grid[:, i * h:(i + 1) * h] for i in range(n)]
    turned.process_packed12(cu, tonemap="reinhard", gamma=0.9, out=tiles)
    for i in range(n):
        assert torch.equal(grid[:, i * h:(i + 1) * h], exp[i]), f"tile {i}"
    assert int(grid[:, n * h:].max()) == 0, "the padding columns stay untouched"


def test_turned_pass_in_the_graphed_stream(cuda):
    from taichi_image_b200.graphed import GraphedStream
    from taichi_image_b200.interpolate import ImageTransform
    r = rng(314)
    h, w, n = 136, 64, 2
    cu = [to_cuda(packed_frame(r, h, w)) for _ in range(n)]
    outs = [torch.empty((w, h, 3), dtype=torch.uint8, device="cuda") for _ in range(n)]
    eager = make("f32", transform=ImageTransform.rotate_90, moving_alpha=0.2)
    gisp = make("f32", transform=ImageTransform.rotate_90, moving_alpha=0.2)
    gs = GraphedStream(gisp, cu, outs, tonemap="reinhard", gamma=0.9)
    for k in range(3):
        exp = eager.process_packed12(cu, tonemap="reinhard", gamma=0.9)
        got = [o.clone() for o in gs.step()]
        torch.cuda.synchronize()
        for x, y in zip(exp, got):
            assert_close_int(to_np(x), to_np(y), 1, f"graphed step {k}")
