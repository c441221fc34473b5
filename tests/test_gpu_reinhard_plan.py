"""GPU check of the scratch size the library reports (b200isp_reinhard_scratch_bytes, csrc/fused_isp.cuh reinhard_plan) for
every one-sweep Reinhard form: b200isp_process_packed12 is called directly with the ISP's parameter block and a canary-filled
scratch of exactly that size inside guard bands.

* exact size: nothing outside the scratch changes, every frame's map is written, and the outputs equal those of the same
  call with a generous scratch;
* one byte less: the map forms leave the scratch alone and run the exact form (Camera32: the outputs of the
  ``reinhard_exact=True`` ISP); YUV 4:2:0, resizing ISPs and the transposing transforms refuse the call (E_ARG); the Camera16
  table pass falls back to the arithmetic pass, which is bit-identical, and leaves the tables alone.
"""
import pytest
import torch

from tests.util import rng, packed_frame, to_cuda

pytestmark = pytest.mark.gpu

N, H, W = 5, 32, 776               # H % 8 == 0 and H >= 16: the turned passes apply
PAD = 1 << 12
CANARY = 0xA5
E_ARG = -1

# name -> (ISP class, output dtype, gamma, ISP keyword arguments, yuv420, refused with one byte less)
CASES = {
    "resize_cam16": ("Camera16", "u8", 0.6, dict(scale=0.5), False, True),
    "resize_cam32": ("Camera32", "u16", 0.9, dict(scale=0.5), False, True),
    "cam16_turned_no_fallback": ("Camera16", "u8", 0.6, dict(transform="rotate_90"), False, True),
    "cam16_yuv": ("Camera16", "u8", 0.6, {}, True, True),
    "cam16_table": ("Camera16", "u8", 0.6, {}, False, False),
    "cam16_arith": ("Camera16", "u16", 0.6, {}, False, False),
    "cam32_map16": ("Camera32", "u8", 0.9, {}, False, False),
    "cam32_turned_no_fallback": ("Camera32", "u8", 0.9, dict(transform="rotate_90"), False, True),
}


def _isp(cam, kw, **extra):
    from taichi_image_b200 import camera_isp, bayer, interpolate
    kw = dict(kw)
    if "transform" in kw:
        kw["transform"] = interpolate.ImageTransform[kw["transform"]]
    return getattr(camera_isp, cam)(bayer.BayerPattern.RGGB, **kw, **extra)


def _call(isp, p, frames, outs, metrics, scratch):
    from taichi_image_b200 import _lib
    if scratch is not None:
        p.reinhard_scratch, p.reinhard_scratch_bytes = scratch.data_ptr(), scratch.numel()
    rc = _lib.lib.b200isp_process_packed12(_lib.ptr_array(frames), _lib.ptr_array(outs), len(frames), p, metrics.data_ptr(),
                                           _lib.workspace(isp.device).data_ptr(), _lib.stream_ptr(isp.device))
    torch.cuda.synchronize()
    return rc


@pytest.mark.parametrize("case", list(CASES))
def test_reported_scratch_size_is_exactly_what_the_call_uses(cuda, case):
    from taichi_image_b200 import _lib, dtypes
    cam, out, gamma, kw, yuv, refused = CASES[case]
    out_dtype = dtypes.as_dtype(out)
    r = rng(91)
    frames = [to_cuda(packed_frame(r, H, W)) for _ in range(N)]
    isp = _isp(cam, kw)
    isp._metrics_and_alpha()
    isp.meter_packed12(frames, 0.0)                       # metrics of these frames; every call below only reads them
    metrics = isp.metrics.clone()
    tm = dict(gamma=gamma)
    flip = isp._fused_flip(H, "reinhard", out_dtype, gamma, 0.0, yuv420=yuv)
    assert bool(flip) == ("transform" in kw), "a transposing transform must go into the call"
    p = isp._fused_params(frames, "reinhard", out_dtype, tm, yuv420=yuv, flip=flip)
    need = _lib.lib.b200isp_reinhard_scratch_bytes(p, N)
    assert need > 0 and p.reinhard_scratch_bytes == need
    if yuv:
        oshape = (H * 3 // 2, W)
    else:
        plan = isp._resize_plan(H, W)
        ho, wo = (H, W) if plan is None else (plan[0][1], plan[0][0])
        oshape = (wo, ho, 3) if flip & 4 else (ho, wo, 3)
    new_outs = lambda: [torch.empty(oshape, dtype=out_dtype.torch, device="cuda") for _ in frames]
    frame_map = need // N if "table" not in case else (need - N * 65536) // N

    # exactly the reported size
    buf = torch.full((need + 2 * PAD,), CANARY, dtype=torch.uint8, device="cuda")
    got = new_outs()
    _lib.check(_call(isp, p, frames, got, metrics, buf[PAD:PAD + need]), case)
    assert bool((buf[:PAD] == CANARY).all()) and bool((buf[PAD + need:] == CANARY).all()), "write outside the scratch"
    for f in range(N):
        assert not bool((buf[PAD + f * frame_map:PAD + (f + 1) * frame_map] == CANARY).all()), f"frame {f}: map not written"
    big = torch.full((2 * need,), CANARY, dtype=torch.uint8, device="cuda")
    ref = new_outs()
    _lib.check(_call(isp, p, frames, ref, metrics, big), case)
    for g, e in zip(got, ref):
        assert torch.equal(g, e), "outputs depend on the scratch size beyond the reported one"

    # one byte less
    buf.fill_(CANARY)
    less = new_outs()
    rc = _call(isp, p, frames, less, metrics, buf[PAD:PAD + need - 1])
    if refused:
        assert rc == E_ARG, rc
        assert bool((buf == CANARY).all()), "a refused call wrote to the scratch"
        return
    _lib.check(rc, case)
    if "table" in case:                                   # the maps are written, the tables are not; same outputs
        assert bool((buf[PAD + N * frame_map:] == CANARY).all()), "a table was written without room for all of them"
        for g, e in zip(less, ref):
            assert torch.equal(g, e), "the arithmetic pass differs from the table pass"
        return
    assert bool((buf == CANARY).all()), "the map form ran without room for its map"
    if cam == "Camera32":
        exact = _isp(cam, kw, reinhard_exact=True)
        pe = exact._fused_params(frames, "reinhard", out_dtype, tm, flip=flip)
        assert pe.reinhard_scratch_bytes == 0
        two = new_outs()
        _lib.check(_call(exact, pe, frames, two, metrics, None), case)
        for g, e in zip(less, two):
            assert torch.equal(g, e), "not the exact form"
