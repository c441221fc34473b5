"""GPU parity: camera_isp.py -- eager stage-by-stage API and the fused packed12 sweep against the
oracle ISP (Camera16 / Camera32, metering moving average, Reinhard / linear, u8 / u16 / f16 outputs)."""
import numpy as np
import pytest
import torch

from oracle import isp_oracle as O
from tests.util import rng, packed_frame, smooth_rgb, to_cuda, to_np, assert_close_int, assert_close_float, assert_u16_from_f16_isp

pytestmark = pytest.mark.gpu
CAMS = {"f16": "Camera16", "f32": "Camera32"}


def make_isp(dt, **kw):
    from taichi_image_b200 import camera_isp, bayer
    kw = dict(kw)
    pattern = kw.pop("bayer_pattern", "RGGB")
    return getattr(camera_isp, CAMS[dt])(bayer.BayerPattern[pattern], **kw)


def frames(r, n, h, w, pattern="RGGB"):
    return [packed_frame(r, h, w, pattern) for _ in range(n)]


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("pattern", O.PATTERNS)
@pytest.mark.parametrize("shape", [(32, 48), (30, 36)])     # fused loader / generic (width % 8 != 0)
@pytest.mark.parametrize("ccm", [False, True])
def test_load_packed12(cuda, dt, pattern, shape, ccm):
    pk = packed_frame(rng(30), *shape, pattern)
    isp = make_isp(dt, bayer_pattern=pattern, correct_colors=ccm)
    got = to_np(isp.load_packed12(to_cuda(pk)))
    ref = O.ISP(dt, pattern, correct_colors=ccm).load_packed12(pk)
    assert got.dtype == ref.dtype and got.shape == ref.shape
    assert_close_float(got, ref, rtol=1e-3, atol=1e-3 if dt == "f16" else 2e-6, what=f"{dt} {pattern}")


@pytest.mark.parametrize("dt", ["f16", "f32"])
def test_load_other_formats(cuda, dt):
    r = rng(31)
    raw16 = r.integers(0, 65536, size=(16, 24)).astype(np.uint16)
    isp, ref = make_isp(dt), O.ISP(dt)
    assert_close_float(to_np(isp.load_16u(to_cuda(raw16))), ref.load_16u(raw16), atol=1e-3 if dt == "f16" else 2e-6)
    f = r.random((16, 24), dtype=np.float32)
    assert_close_float(to_np(isp.load_32f(to_cuda(f))), ref.load_32f(f), atol=1e-3 if dt == "f16" else 2e-6)
    b = raw16.view(np.uint8).reshape(16, 48)
    assert_close_float(to_np(isp.load_packed16(to_cuda(b))), ref.load_packed16(b), atol=1e-3 if dt == "f16" else 2e-6)
    pk = O.encode12(r.integers(0, 4096, size=(16, 24)).astype(np.uint16), ids_format=True)
    assert_close_float(to_np(isp.load_packed12(to_cuda(pk), ids_format=True)), ref.load_packed12(pk, ids_format=True),
                       atol=1e-3 if dt == "f16" else 2e-6)


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("stride", [8, 3])
def test_metering_moving_average(cuda, dt, stride):
    r = rng(32)
    isp, ref = make_isp(dt, metering_stride=stride, moving_alpha=0.1), O.ISP(dt, metering_stride=stride, moving_alpha=0.1)
    for step in range(3):
        fr = frames(r, 3, 40, 56)
        ims_ref = [ref.load_packed12(f) for f in fr]
        ims = [to_cuda(i) for i in ims_ref]           # identical inputs: isolates the metering kernels
        isp.update_metering(ims)
        ref.update_metering(ims_ref)
        assert_close_float(to_np(isp.metrics), ref.metrics, rtol=2e-5, atol=2e-6, what=f"step {step}")


TM = [dict(), dict(gamma=0.6), dict(gamma=0.9, intensity=3.0, light_adapt=0.9, color_adapt=0.0),
      dict(gamma=0.8, intensity=2.0, light_adapt=0.7, color_adapt=0.3)]


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("tm", TM)
def test_eager_tonemap_reinhard(cuda, dt, tm):
    r = rng(33)
    isp, ref = make_isp(dt), O.ISP(dt)
    for step in range(2):
        fr = frames(r, 2, 32, 48)
        got = isp.tonemap_reinhard([isp.load_packed12(to_cuda(f)) for f in fr], **tm)
        exp = ref.tonemap_reinhard([ref.load_packed12(f) for f in fr], **tm)
        for g, e in zip(got, exp):
            assert g.dtype == torch.uint8
            assert_close_int(to_np(g), e, 1, f"{dt} {tm} step {step}")
    assert_close_float(to_np(isp.metrics), ref.metrics, rtol=1e-4, atol=1e-5)


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("gamma", [1.0, 0.7])
def test_eager_tonemap_linear(cuda, dt, gamma):
    r = rng(34)
    isp, ref = make_isp(dt), O.ISP(dt)
    fr = frames(r, 2, 32, 48)
    got = isp.tonemap_linear([isp.load_packed12(to_cuda(f)) for f in fr], gamma=gamma)
    exp = ref.tonemap_linear([ref.load_packed12(f) for f in fr], gamma=gamma)
    for g, e in zip(got, exp):
        assert_close_int(to_np(g), e, 1, f"{dt} gamma {gamma}")


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("pattern", O.PATTERNS)
@pytest.mark.parametrize("tm", TM[:3])
def test_fused_reinhard_u8(cuda, dt, pattern, tm):
    r = rng(35)
    isp, ref = make_isp(dt, bayer_pattern=pattern), O.ISP(dt, pattern)
    for step in range(3):
        fr = frames(r, 3, 40, 64, pattern)
        got = isp.process_packed12([to_cuda(f) for f in fr], tonemap="reinhard", **tm)
        exp = ref.tonemap_reinhard([ref.load_packed12(f) for f in fr], **tm)
        for g, e in zip(got, exp):
            assert_close_int(to_np(g), e, 1, f"{dt} {pattern} {tm} step {step}")
        assert_close_float(to_np(isp.metrics), ref.metrics, rtol=1e-4, atol=1e-5, what="metrics")


@pytest.mark.parametrize("dt,out", [("f32", "u8"), ("f32", "u16"), ("f16", "u8"), ("f16", "u16")])
@pytest.mark.parametrize("gamma", [1.0, 0.7])
@pytest.mark.parametrize("ccm", [False, True])
def test_fused_linear(cuda, dt, out, gamma, ccm):
    """u16 from Camera16 is allowed one f16 ulp of the intermediate RGB (values < 1: 2^-11) seen through the
    tone map's gain 1 / (max - min): 32 / (max - min) LSB of u16 (SURVEY H7: trunc / f16 rounding flips)"""
    r = rng(36)
    isp, ref = make_isp(dt, correct_colors=ccm), O.ISP(dt, correct_colors=ccm)
    for step in range(2):
        fr = frames(r, 2, 36, 72)
        got = isp.process_packed12([to_cuda(f) for f in fr], tonemap="linear", gamma=gamma, dtype=out)
        exp = ref.tonemap_linear([ref.load_packed12(f) for f in fr], gamma=gamma, out_dtype=out)
        for g, e in zip(got, exp):
            if dt == "f16" and out == "u16":
                gain = max(1.0, 1.0 / gamma) / float(ref.metrics[1] - ref.metrics[0])      # slope of x^(1/gamma) <= 1/gamma
                assert_u16_from_f16_isp(to_np(g), e, gain, f"{dt}->{out} gamma {gamma}")
            else:
                assert_close_int(to_np(g), e, 1, f"{dt}->{out} gamma {gamma}")


@pytest.mark.parametrize("dt", ["f16", "f32"])
def test_fused_f16_output_and_transform(cuda, dt):
    from taichi_image_b200.interpolate import ImageTransform
    r = rng(37)
    isp, ref = make_isp(dt, transform=ImageTransform.rotate_90), O.ISP(dt, transform="rotate_90")
    fr = frames(r, 2, 32, 40)
    got = isp.process_packed12([to_cuda(f) for f in fr], tonemap="reinhard", gamma=0.8, dtype="f16")
    exp = ref.tonemap_reinhard([ref.load_packed12(f) for f in fr], gamma=0.8, out_dtype="f16")
    for g, e in zip(got, exp):
        assert g.dtype == torch.float16 and tuple(g.shape) == (40, 32, 3)
        assert_close_float(to_np(g), e, rtol=2e-3, atol=1e-3)


@pytest.mark.parametrize("dt", ["f16", "f32"])
def test_fused_with_resize_falls_back_to_staged_kernels(cuda, dt):
    r = rng(38)
    isp, ref = make_isp(dt, resize_width=40), O.ISP(dt, resize_width=40)
    fr = frames(r, 2, 48, 80)
    got = isp.process_packed12([to_cuda(f) for f in fr], tonemap="reinhard", gamma=0.6)
    exp = ref.tonemap_reinhard([ref.load_packed12(f) for f in fr], gamma=0.6)
    for g, e in zip(got, exp):
        assert tuple(g.shape) == e.shape == (24, 40, 3)
        assert_close_int(to_np(g), e, 1, "resize")


def test_fused_random_frames_worst_case(cuda):
    """pure-random 12-bit frames (SURVEY 8d): heavy clamping, full dynamic range"""
    r = rng(39)
    isp, ref = make_isp("f32"), O.ISP("f32")
    fr = [packed_frame(r, 64, 96, smooth=False) for _ in range(2)]
    got = isp.process_packed12([to_cuda(f) for f in fr], tonemap="reinhard", gamma=0.9, intensity=3.0, light_adapt=0.9)
    exp = ref.tonemap_reinhard([ref.load_packed12(f) for f in fr], gamma=0.9, intensity=3.0, light_adapt=0.9)
    for g, e in zip(got, exp):
        assert_close_int(to_np(g), e, 1, "random frames")


def test_isp_api_surface(cuda):
    from taichi_image_b200 import camera_isp, bayer
    isp = camera_isp.Camera32(bayer.BayerPattern.RGGB, moving_alpha=0.2)
    assert camera_isp.Camera16.__qualname__ == "Camera16" and isp.metrics is None
    isp.set(resize_width=100)
    assert isp.resize_width == 100 and isp.scale is None
    isp.set(scale=0.5)
    assert isp.scale == 0.5 and isp.resize_width == 0
    assert isp.color_correct_matrix is None
    isp.set(correct_colors=True)
    assert np.allclose(isp.color_correct_matrix, O.DEFAULT_CC * O.DEFAULT_WB)
    with pytest.raises(Exception):
        camera_isp.Camera32("RGGB")          # beartype: pattern must be a BayerPattern
    with pytest.raises(AssertionError):
        camera_isp.Camera32(bayer.BayerPattern.RGGB, scale=0.5, resize_width=10)


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("tm", ["linear", "reinhard"])
def test_lookahead_metering_is_equivalent(cuda, dt, tm):
    """process_packed12(lookahead=next batch) -- metering of batch k+1 on a side stream under sweep k -- must give
    the same outputs and the same metrics trajectory as strictly serial calls, also when the announcement is
    wrong (the pending update is then discarded)"""
    r = rng(41)
    batches = [[to_cuda(f) for f in frames(r, 3, 40, 64)] for _ in range(5)]
    serial, ahead = make_isp(dt, moving_alpha=0.2), make_isp(dt, moving_alpha=0.2)
    for i, b in enumerate(batches):
        ya = serial.process_packed12(b, tonemap=tm, gamma=0.9)
        nxt = batches[i + 1] if i + 1 < len(batches) else None
        if i == 2:
            nxt = batches[0]                                  # wrong announcement: batch 3 follows, not batch 0
        yb = ahead.process_packed12(b, tonemap=tm, gamma=0.9, lookahead=nxt)
        torch.cuda.synchronize()
        np.testing.assert_allclose(to_np(ahead.metrics), to_np(serial.metrics), rtol=2e-6, atol=1e-7)
        for x, y in zip(ya, yb):
            assert_close_int(to_np(x), to_np(y), 1, f"lookahead {dt} {tm} step {i}")


def test_lookahead_first_call_large_frames(cuda):
    """ADVICE r1 (high): on the FIRST look-ahead call the second metrics buffer used to be zero-filled on the main
    stream behind the sweep, i.e. after the side-stream metering had written it -- visible only when the sweep
    outlasts the metering (frames of real size).  Batch 2 must be tone-mapped with the serial metrics."""
    from tests.test_gpu_fullsize import synth_packed
    b0, _ = synth_packed(2, 3000, 4096, seed=3)
    b1, _ = synth_packed(2, 3000, 4096, seed=5)
    serial, ahead = make_isp("f32", moving_alpha=0.2), make_isp("f32", moving_alpha=0.2)
    serial.process_packed12(b0, tonemap="linear", dtype="u16")
    ys = serial.process_packed12(b1, tonemap="linear", dtype="u16")
    ahead.process_packed12(b0, tonemap="linear", dtype="u16", lookahead=b1)
    ya = ahead.process_packed12(b1, tonemap="linear", dtype="u16")
    torch.cuda.synchronize()
    np.testing.assert_allclose(to_np(ahead.metrics), to_np(serial.metrics), rtol=2e-6, atol=1e-7)
    assert float(ahead.metrics[1]) > float(ahead.metrics[0]) > 0.0
    for x, y in zip(ys, ya):
        assert int((x.int() - y.int()).abs().max()) <= 1


@pytest.mark.parametrize("tm,out", [("linear", "u16"), ("reinhard", "u8")])
def test_graphed_stream_matches_eager(cuda, tm, out):
    """graphed.GraphedStream with double-buffered ingest (CUDA-graph replay of sweep k || metering k+1) == eager
    ``process_packed12`` calls on a CHANGING scene: same outputs (<= 1 LSB) and the same metrics trajectory"""
    from taichi_image_b200.graphed import GraphedStream
    from taichi_image_b200 import as_dtype
    r = rng(43)
    h, w, n, steps = 40, 64, 3, 6
    host = [frames(r, n, h, w) for _ in range(steps + 1)]
    for k in range(steps + 1):                 # a scene whose exposure really changes from batch to batch
        gain = 0.55 + 0.45 * np.cos(0.9 * k)
        host[k] = [O.encode12((O.decode12(f, "u16").astype(np.float32) * gain).astype(np.uint16)) for f in host[k]]
    bufs = [[torch.empty((h, w * 3 // 2), dtype=torch.uint8, device="cuda") for _ in range(n)] for _ in range(2)]
    outs = [torch.empty((h, w, 3), dtype=as_dtype(out).torch, device="cuda") for _ in range(n)]
    eager, gisp = make_isp("f32", moving_alpha=0.2), make_isp("f32", moving_alpha=0.2)

    def fill(p, k):
        for b, f in zip(bufs[p], host[k]):
            b.copy_(to_cuda(f))

    fill(0, 0)
    fill(1, 1)
    gs = GraphedStream(gisp, bufs[0], outs, tonemap=tm, dtype=out, next_frames=bufs[1], gamma=0.9)
    for k in range(steps):
        exp = eager.process_packed12([to_cuda(f) for f in host[k]], tonemap=tm, gamma=0.9, dtype=out)
        assert gs.frames[0].data_ptr() == bufs[k % 2][0].data_ptr()
        got = [o.clone() for o in gs.step()]
        torch.cuda.synchronize()
        for x, y in zip(exp, got):
            assert_close_int(to_np(x), to_np(y), 1, f"graphed {tm} step {k}")
        fill(k % 2, k + 2 if k + 2 <= steps else 0)           # batch k + 2 into the set the sweep has just left
        # isp.metrics already holds the update for batch k + 1
        probe = make_isp("f32", moving_alpha=0.2)
        probe.metrics = eager.metrics.clone()
        probe.process_packed12([to_cuda(f) for f in host[k + 1]], tonemap=tm, gamma=0.9, dtype=out)
        np.testing.assert_allclose(to_np(gisp.metrics), to_np(probe.metrics), rtol=2e-6, atol=1e-7)


def test_graphed_stream_single_buffer_lags_one_step(cuda):
    """single-buffered GraphedStream on a constant scene == eager calls (the documented one-step exposure lag is
    invisible there); first step exact"""
    from taichi_image_b200.graphed import GraphedStream
    r = rng(44)
    h, w, n = 40, 64, 2
    cu = [to_cuda(f) for f in frames(r, n, h, w)]
    outs = [torch.empty((h, w, 3), dtype=torch.uint8, device="cuda") for _ in range(n)]
    eager, gisp = make_isp("f32", moving_alpha=0.2), make_isp("f32", moving_alpha=0.2)
    gs = GraphedStream(gisp, cu, outs, tonemap="reinhard", gamma=0.9)
    assert not gs.double_buffered
    for k in range(4):
        exp = eager.process_packed12(cu, tonemap="reinhard", gamma=0.9)
        got = [o.clone() for o in gs.step()]
        torch.cuda.synchronize()
        for x, y in zip(exp, got):
            assert_close_int(to_np(x), to_np(y), 1, f"graphed single-buffer step {k}")


@pytest.mark.parametrize("dt", ["f16", "f32"])
def test_metering_histogram_and_percentiles(cuda, dt):
    """EXTENSION (no reference counterpart): luminance histogram / percentiles of the metering samples, checked
    against numpy on the oracle's samples; counts may move by one bin where gray * bins lands on an integer"""
    r = rng(45)
    fr = frames(r, 3, 48, 64)
    isp, ref = make_isp(dt), O.ISP(dt)
    isp.process_packed12([to_cuda(f) for f in fr], tonemap="linear")
    hist = to_np(isp.metering_histogram(64))
    samples = np.stack([ref.load_packed12(f)[::8, ::8] for f in fr]).astype(np.float32).reshape(-1, 3)
    gray = O.rgb_gray(samples)
    exp = np.bincount(np.minimum(63, (gray * np.float32(64)).astype(np.int64)), minlength=64)
    assert hist.sum() == exp.sum() == samples.shape[0]
    assert np.abs(np.cumsum(hist) - np.cumsum(exp)).max() <= max(2, samples.shape[0] // 200)
    pct = to_np(isp.metering_percentiles((1.0, 50.0, 99.0), 64))
    cum = np.cumsum(hist)
    for p, v in zip((1.0, 50.0, 99.0), pct):
        b = int(np.searchsorted(cum, p * 0.01 * cum[-1]))
        assert abs(v - (min(b, 63) + 1) / 64.0) < 1e-6
    assert pct[0] <= pct[1] <= pct[2]


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("pattern", O.PATTERNS)
@pytest.mark.parametrize("shape,rpt", [((30, 1288), 0), ((52, 768), 0), ((44, 1032), 6), ((40, 776), 2), ((64, 520), 24)])
def test_fused_wide_frames_all_task_kinds(cuda, dt, pattern, shape, rpt):
    """Frames wide enough for interior strips (K_CORE: W > 512), with exact and partial last strips, several row
    chunks and chunk sizes that are not a multiple of the unrolled step -- every task kind of the pair engine
    (stream2.cuh) against the oracle: load_packed12 (float RGB), linear -> u16 (packed fast path for Camera32) and
    Reinhard -> u8 (packed Reinhard path)."""
    h, w = shape
    r = rng(50 + h)
    fr = frames(r, 2, h, w, pattern)
    cu = [to_cuda(f) for f in fr]
    isp, ref = make_isp(dt, bayer_pattern=pattern), O.ISP(dt, pattern)
    got = to_np(isp.load_packed12(cu[0]))
    exp = ref.load_packed12(fr[0])
    assert_close_float(got, exp, rtol=1e-3, atol=1e-3 if dt == "f16" else 2e-6, what=f"rgb {dt} {pattern} {shape}")
    ims = [ref.load_packed12(f) for f in fr]
    lin = isp.process_packed12(cu, tonemap="linear", dtype="u16", rows_per_task=rpt)
    exp_lin = ref.tonemap_linear([im.copy() for im in ims], out_dtype="u16")
    for g, e in zip(lin, exp_lin):
        if dt == "f32":
            assert_close_int(to_np(g), e, 1, f"linear {dt} {pattern} {shape}")
        else:
            assert_u16_from_f16_isp(to_np(g), e, 1.0 / float(ref.metrics[1] - ref.metrics[0]), f"linear {dt} {pattern} {shape}")
    isp2, ref2 = make_isp(dt, bayer_pattern=pattern), O.ISP(dt, pattern)
    rei = isp2.process_packed12(cu, tonemap="reinhard", gamma=0.9, intensity=2.0, light_adapt=0.8, dtype="u8", rows_per_task=rpt)
    exp_rei = ref2.tonemap_reinhard([ref2.load_packed12(f) for f in fr], gamma=0.9, intensity=2.0, light_adapt=0.8, out_dtype="u8")
    for g, e in zip(rei, exp_rei):
        assert_close_int(to_np(g), e, 1, f"reinhard {dt} {pattern} {shape}")


# ---------------------------------------------------------------- IDS layout through the fused sweep (SURVEY 8f-4)
@pytest.mark.parametrize("n_bytes", [0, 3, 9, 12, 36, 3 * 1001, 48 * 64])
def test_repack12_ids_bit_exact(cuda, n_bytes):
    from taichi_image_b200 import packed
    ids = rng(90).integers(0, 256, size=(n_bytes,)).astype(np.uint8)
    got = to_np(packed.repack12_ids(to_cuda(ids)))
    assert np.array_equal(got, O.repack12_ids(ids))
    if n_bytes:      # the re-packed stream decodes (standard layout) to what the IDS stream decodes to
        assert np.array_equal(O.decode12_raw(got), O.decode12_raw(ids, ids_format=True))
    view = to_cuda(np.concatenate([np.zeros(1, np.uint8), ids]))[1:]           # unaligned base: byte-wise kernel path
    assert np.array_equal(to_np(packed.repack12_ids(view)), O.repack12_ids(ids))


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("tonemap", ["linear", "reinhard"])
def test_fused_ids_format(cuda, dt, tonemap):
    """IDS frames: re-packed on the device, then the fused sweep -- same results as the reference's staged order"""
    r = rng(91)
    isp, ref = make_isp(dt, bayer_pattern="GBRG"), O.ISP(dt, "GBRG")
    for step in range(2):
        fr = [O.encode12(O.rgb_to_bayer(smooth_rgb(r, 36, 72), "GBRG"), scaled=True, ids_format=True) for _ in range(2)]
        got = isp.process_packed12([to_cuda(f) for f in fr], tonemap=tonemap, gamma=0.8, ids_format=True)
        imgs = [ref.load_packed12(f, ids_format=True) for f in fr]
        exp = ref.tonemap_linear(imgs, gamma=0.8) if tonemap == "linear" else ref.tonemap_reinhard(imgs, gamma=0.8)
        for g, e in zip(got, exp):
            assert_close_int(to_np(g), e, 1, f"ids {dt} {tonemap} step {step}")
    one = O.encode12(O.rgb_to_bayer(smooth_rgb(r, 36, 72), "GBRG"), scaled=True, ids_format=True)
    assert_close_float(to_np(isp.load_packed12(to_cuda(one), ids_format=True)), ref.load_packed12(one, ids_format=True),
                       rtol=1e-3, atol=1e-3 if dt == "f16" else 2e-6)


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("pattern", ["RGGB", "GBRG"])
def test_ids_layout_in_the_row_loader_equals_repack(cuda, dt, pattern):
    """IDS frames decoded inside the sweep's row loader and the metering sampler (csrc/fused_isp.cuh ids_sample) give bit for
    bit the outputs and metrics of the same frames re-packed into the standard layout first -- at a width with interior
    strips (K_CORE), a partial last strip and several row chunks"""
    from taichi_image_b200 import packed
    r = rng(96)
    h, w = 44, 1032
    # reinhard_exact: IDS frames always take the exact Reinhard sweeps, the standard layout would take the one-sweep u16 map
    a, b = make_isp(dt, bayer_pattern=pattern, reinhard_exact=True), make_isp(dt, bayer_pattern=pattern, reinhard_exact=True)
    for step in range(2):
        ids = [to_cuda(O.encode12(r.integers(0, 4096, size=(h, w)).astype(np.uint16), ids_format=True)) for _ in range(2)]
        std = [packed.repack12_ids(f) for f in ids]
        for tm, out in (("linear", "u16"), ("reinhard", "u8")):
            ya = a.process_packed12(ids, tonemap=tm, dtype=out, gamma=0.9, ids_format=True, rows_per_task=6)
            yb = b.process_packed12(std, tonemap=tm, dtype=out, gamma=0.9, rows_per_task=6)
            assert torch.equal(a.metrics, b.metrics), f"{tm} step {step}: metrics"
            for x, y in zip(ya, yb):
                assert torch.equal(x, y), f"{tm} step {step}"
    assert torch.equal(a.load_packed12(ids[0], ids_format=True), b.load_packed12(std[0]))


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("tname", ["flip_horiz", "flip_vert", "rotate_180"])
@pytest.mark.parametrize("shape", [(40, 64), (44, 1032), (36, 776)])
def test_flips_in_the_store(cuda, dt, tname, shape):
    """flip_horiz / flip_vert / rotate_180 applied by the sweep's store (interpolate.py:36-56 without the extra pass): bit for
    bit interpolate.transform of the untransformed result, for every epilogue family, with full and partial last strips;
    `out=` then holds the transformed images"""
    from taichi_image_b200.interpolate import ImageTransform, transform
    r = rng(97)
    h, w = shape
    t = ImageTransform[tname]
    cu = [to_cuda(f) for f in frames(r, 2, h, w)]
    for tm, out, kw in (("linear", "u16", dict()), ("linear", "u8", dict(gamma=0.8)), ("reinhard", "u8", dict(gamma=0.9, intensity=2.0)),
                        ("reinhard", "f16", dict())):
        plain, flipped = make_isp(dt, reinhard_exact=True), make_isp(dt, transform=t, reinhard_exact=True)      # like with like: the flips take the exact Reinhard sweeps
        exp = [transform(o, t) for o in plain.process_packed12(cu, tonemap=tm, dtype=out, rows_per_task=6, **kw)]
        bufs = [torch.empty_like(e) for e in exp]
        got = flipped.process_packed12(cu, tonemap=tm, dtype=out, rows_per_task=6, out=bufs, **kw)
        assert got[0].data_ptr() == bufs[0].data_ptr()
        for g, e in zip(got, exp):
            if dt == "f16" and tm == "reinhard":
                # Camera16 Reinhard with a flip takes the two-sweep form instead of the f16-scratch form: max_out comes from a
                # different (equally valid) evaluation order, so the two differ in the last bit of a few values
                assert float((g.float() - e.float()).abs().max()) <= (1.0 if out == "u8" else 2e-3), f"{dt} {tname} {tm}->{out} {shape}"
            elif dt == "f32" and tm == "linear" and not kw:
                # the unflipped reference ran the packed fast epilogue (frame columns renormalised by a reciprocal multiply),
                # the flipped one the generic epilogue (IEEE division): the image-frame pixels may differ in the last bit
                d = (g.int() - e.int()).abs()
                assert int(d.max()) <= 1 and int((d != 0).sum()) <= 8 * (h + w), f"{dt} {tname} {tm}->{out} {shape}"
            else:
                assert torch.equal(g, e), f"{dt} {tname} {tm}->{out} {shape}"


@pytest.mark.parametrize("dt", ["f16", "f32"])
@pytest.mark.parametrize("tname", ["rotate_90", "rotate_270", "transpose", "transverse"])
@pytest.mark.parametrize("shape", [(40, 64), (48, 1032), (16, 776), (64, 264), (44, 72)])
def test_transposing_transforms_after_the_sweep_or_in_the_turned_pass(cuda, dt, tname, shape):
    """rotate_90 (the rig script's default) / rotate_270 / transpose / transverse: the normalise pass of the one-sweep
    Reinhard -> u8 forms turns the image (csrc/normalise.cu reinhard_out_transposed_kernel; here Camera16, whose turned form
    does not depend on reinhard_exact), every other call runs the transform kernel on its results -- bit for bit
    interpolate.transform of the untransformed result for every output dtype, default tasks and tasks of 8 rows"""
    from taichi_image_b200.interpolate import ImageTransform, transform
    r = rng(99)
    h, w = shape
    t = ImageTransform[tname]
    cu = [to_cuda(f) for f in frames(r, 2, h, w)]
    for tm, out, kw in (("linear", "u16", dict()), ("linear", "u8", dict(gamma=0.8)), ("reinhard", "u8", dict(gamma=0.9, intensity=2.0)),
                        ("reinhard", "f16", dict()), ("linear", "f16", dict(gamma=0.7))):
        for rpt in (0, 8):
            plain, turned = make_isp(dt, reinhard_exact=True), make_isp(dt, transform=t, reinhard_exact=True)      # like with like
            exp = [transform(o, t) for o in plain.process_packed12(cu, tonemap=tm, dtype=out, rows_per_task=rpt, **kw)]
            assert tuple(exp[0].shape) == (w, h, 3)
            bufs = [torch.empty_like(e) for e in exp]
            got = turned.process_packed12(cu, tonemap=tm, dtype=out, rows_per_task=rpt, out=bufs, **kw)
            assert got[0].data_ptr() == bufs[0].data_ptr()
            for g, e in zip(got, exp):
                assert torch.equal(g, e), f"{dt} {tname} {tm}->{out} {shape} rpt {rpt}"


@pytest.mark.parametrize("tname", ["rotate_90", "transverse"])
def test_rotated_tiles_of_a_grid_image(cuda, tname):
    """a transposing transform straight into row-pitched tiles of one grid image (scripts/tonemap_scan.py:91-100; rotate_90 is
    its default): Camera32 Reinhard -> u8 turns the image in its normalise pass"""
    from taichi_image_b200.interpolate import ImageTransform, transform
    r = rng(100)
    h, w, n = 48, 72, 3
    t = ImageTransform[tname]
    cu = [to_cuda(f) for f in frames(r, n, h, w)]
    plain, turned = make_isp("f32"), make_isp("f32", transform=t)
    exp = [transform(o, t) for o in plain.process_packed12(cu, tonemap="reinhard", gamma=0.9)]
    grid = torch.zeros((w, n * h + 16, 3), dtype=torch.uint8, device="cuda")        # n tiles of (w, h) side by side + padding
    tiles = [grid[:, i * h:(i + 1) * h] for i in range(n)]
    turned.process_packed12(cu, tonemap="reinhard", gamma=0.9, out=tiles)
    for i in range(n):
        assert torch.equal(grid[:, i * h:(i + 1) * h], exp[i]), f"tile {i}"
    assert int(grid[:, n * h:].max()) == 0


def test_graphed_stream_and_pipeline_with_ids_frames(cuda):
    """IDS frames through the CUDA-graph stream and the host-buffer pipeline == eager calls on the same frames"""
    from taichi_image_b200.graphed import GraphedStream
    from taichi_image_b200.pipeline import RigPipeline
    r = rng(98)
    h, w, n = 40, 64, 2
    ids = [O.encode12(r.integers(0, 4096, size=(h, w)).astype(np.uint16), ids_format=True) for _ in range(n)]
    cu = [to_cuda(f) for f in ids]
    outs = [torch.empty((h, w, 3), dtype=torch.uint8, device="cuda") for _ in range(n)]
    eager, gisp, pisp = make_isp("f32", moving_alpha=0.2), make_isp("f32", moving_alpha=0.2), make_isp("f32", moving_alpha=0.2)
    gs = GraphedStream(gisp, cu, outs, tonemap="reinhard", ids_format=True, gamma=0.9)
    pipe = RigPipeline(pisp, n, h, w, tonemap="reinhard", ids_format=True, gamma=0.9)
    for k in range(3):
        exp = eager.process_packed12(cu, tonemap="reinhard", gamma=0.9, ids_format=True)
        got = [o.clone() for o in gs.step()]
        host = pipe.process(RigPipeline.pin(ids))
        torch.cuda.synchronize()
        for x, y, z in zip(exp, got, host):
            assert_close_int(to_np(x), to_np(y), 1, f"graphed ids step {k}")
            assert np.array_equal(to_np(x), z.numpy()), f"pipeline ids step {k}"
