"""GPU: pipeline.RigPipeline (SURVEY 8f-1: pinned host buffers -> H2D -> fused ISP -> D2H -> pinned host, three streams,
``depth`` slots) against plain ``process_packed12`` calls: same outputs, same metrics trajectory, slots reused."""
import numpy as np
import pytest
import torch

from tests.test_gpu_camera_isp import frames, make_isp
from tests.util import rng, to_cuda, to_np

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("dt,tm,out", [("f32", "linear", "u16"), ("f32", "reinhard", "u8"), ("f16", "reinhard", "u8")])
def test_rig_pipeline_equals_direct_calls(cuda, dt, tm, out):
    from taichi_image_b200.pipeline import RigPipeline
    r = rng(60)
    n, h, w, steps = 3, 48, 72, 5
    host = [frames(r, n, h, w) for _ in range(steps)]
    direct, piped = make_isp(dt, moving_alpha=0.2), make_isp(dt, moving_alpha=0.2)
    pipe = RigPipeline(piped, n, h, w, tonemap=tm, dtype=out, depth=2, gamma=0.9)
    pinned = [RigPipeline.pin(b) for b in host]
    exp, traj = [], []
    for b in host:
        exp.append([to_np(o) for o in direct.process_packed12([to_cuda(f) for f in b], tonemap=tm, dtype=out, gamma=0.9)])
        traj.append(to_np(direct.metrics).copy())
    # submit two steps ahead of collecting (depth 2): slot 0 is reused by steps 2 and 4, slot 1 by step 3
    tickets, got, slots_used = [], [], []
    for k in range(steps):
        tickets.append(pipe.submit(pinned[k]))
        slots_used.append(tickets[-1])
        if len(tickets) == 2:
            got.append([o.numpy().copy() for o in pipe.result(tickets.pop(0))])
    while tickets:
        got.append([o.numpy().copy() for o in pipe.result(tickets.pop(0))])
    pipe.drain()
    assert slots_used == [0, 1, 0, 1, 0]
    assert len(got) == steps
    for k in range(steps):
        for a, b in zip(got[k], exp[k]):
            assert a.shape == b.shape and a.dtype == b.dtype
            assert np.array_equal(a, b), f"step {k}: pipeline output differs from the direct call"
    np.testing.assert_array_equal(to_np(piped.metrics), traj[-1])
    assert pipe.h2d_bytes_per_step == n * h * w * 3 // 2
    assert pipe.d2h_bytes_per_step == n * h * w * 3 * (2 if out == "u16" else 1)


def test_rig_pipeline_metrics_trajectory(cuda):
    """the moving average advances once per submitted step, in submission order"""
    from taichi_image_b200.pipeline import RigPipeline
    r = rng(61)
    n, h, w = 2, 40, 64
    host = [frames(r, n, h, w) for _ in range(5)]
    direct, piped = make_isp("f32", moving_alpha=0.3), make_isp("f32", moving_alpha=0.3)
    pipe = RigPipeline(piped, n, h, w, tonemap="reinhard", depth=3)
    for b in host:
        direct.process_packed12([to_cuda(f) for f in b], tonemap="reinhard")
        pipe.process(RigPipeline.pin(b))
        np.testing.assert_array_equal(to_np(piped.metrics), to_np(direct.metrics))


@pytest.mark.parametrize("tname", ["rotate_90", "transverse", "flip_vert"])
def test_rig_pipeline_with_a_transforming_isp(cuda, tname):
    """the rig script's default transform (rotate_90, scripts/tonemap_scan.py) through the host-buffer pipeline: the normalise
    pass of the one-sweep Reinhard form (transposing transforms) or the sweep's store (flips) writes the image straight into
    the slot"""
    from taichi_image_b200.interpolate import ImageTransform
    from taichi_image_b200.pipeline import RigPipeline
    r = rng(62)
    n, h, w = 2, 48, 72
    t = ImageTransform[tname]
    direct, piped = make_isp("f32", moving_alpha=0.2, transform=t), make_isp("f32", moving_alpha=0.2, transform=t)
    pipe = RigPipeline(piped, n, h, w, tonemap="reinhard", gamma=0.9)
    for _ in range(3):
        b = frames(r, n, h, w)
        exp = direct.process_packed12([to_cuda(f) for f in b], tonemap="reinhard", gamma=0.9)
        got = pipe.process(RigPipeline.pin(b))
        for g, e in zip(got, exp):
            assert tuple(g.shape) == ((h, w, 3) if tname == "flip_vert" else (w, h, 3))
            assert np.array_equal(g.numpy(), to_np(e))
