"""CPU-only: host logic, the C ABI surface and oracle properties (no GPU compute calls)."""
import ctypes
import os
import re

import numpy as np
import pytest

from oracle import isp_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_exports_every_declared_symbol_and_reports_abi_103():
    from taichi_image_b200 import _lib
    header = open(os.path.join(ROOT, "include", "b200isp.h")).read()
    declared = set(re.findall(r"\b(b200isp_[a-z0-9_]+)\s*\(", header))
    declared -= {"b200isp_fused_params"}
    assert declared, "no declarations found"
    lib = ctypes.CDLL(str(_lib.LIB_PATH))
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/b200isp.h but not exported"
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    assert _lib.lib.b200isp_version() == 103
    assert _lib.WORKSPACE_BYTES >= 4096


def test_fused_params_struct_matches_header():
    from taichi_image_b200 import _lib
    # 7 ints, 9 floats, 4 floats, int, float, 6 ints, 2 floats, 5 ints (35 x 4 bytes) + 4 bytes of padding before the first
    # pointer + 4 pointers + 2 size_t
    assert ctypes.sizeof(_lib.FusedParams) == 4 * (7 + 9 + 4 + 1 + 1 + 6 + 2 + 5) + 4 + 6 * ctypes.sizeof(ctypes.c_void_p)
    header = open(os.path.join(ROOT, "include", "b200isp.h")).read()
    body = header[header.index("typedef struct {"):header.index("} b200isp_fused_params;")]
    names = re.findall(r"\b(?:int|float|void\*|size_t)\s+([a-z_0-9, \[\]]+);", body)
    flat = [n.strip().split("[")[0] for group in names for n in group.split(",")]
    assert flat == [f[0] for f in _lib.FusedParams._fields_], flat


def test_error_paths_do_not_need_a_gpu():
    from taichi_image_b200 import _lib
    lib = _lib.lib
    assert lib.b200isp_decode12(None, 3, None, 1, 0, 0, None) == -3       # odd size
    assert b"even" in lib.b200isp_last_error()
    assert lib.b200isp_bayer_to_rgb(None, 0, None, 0, 3, 4, 0, None, None) == -3
    assert lib.b200isp_bayer_to_rgb(None, 0, None, 0, 4, 4, 9, None, None) == -1
    assert lib.b200isp_transform(None, None, 0, 4, 4, 99, None) == -1
    assert lib.b200isp_decode12(None, 0, None, 1, 0, 0, None) == 0        # empty input is a no-op
    p = _lib.FusedParams()
    p.height, p.width = 10, 12                                            # width % 8 != 0
    arr = (ctypes.c_void_p * 1)()
    assert lib.b200isp_process_packed12(arr, arr, 1, p, None, ctypes.c_void_p(8), None) == -3
    assert lib.b200isp_process_packed12(arr, arr, 65, p, None, ctypes.c_void_p(8), None) == -6


def test_no_cpu_fallback():
    import torch
    from taichi_image_b200 import packed, bayer, types
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        packed.encode12(np.zeros(4, np.uint16))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        bayer.bayer_to_rgb(np.zeros((4, 4), np.uint8))
    with pytest.raises(Exception):
        packed.decode12_kernel(types.u16)(torch.zeros(3, dtype=torch.uint8), torch.zeros(2, dtype=torch.uint16))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "taichi_image_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, f


def test_dtypes_and_types_tables():
    import torch
    from taichi_image_b200 import dtypes, types, u8, u16, f16, f32, uint8
    assert u8 is uint8 and dtypes.as_dtype(torch.float16) is f16 and dtypes.as_dtype(np.uint16) is u16
    assert dtypes.as_dtype("f32") is f32 and dtypes.as_dtype("float32") is f32 and dtypes.as_dtype(np.dtype("uint8")) is u8
    assert types.scale_factor[u8] == 255 and types.scale_factor[u16] == 65535 and types.scale_factor[dtypes.i16] == 32767
    assert types.ti_type(np.zeros(1, np.float16)) is f16 and types.ti_type(torch.zeros(1, dtype=torch.uint16)) is u16
    e = types.empty_like(np.zeros((2, 3), np.uint8), (4, 5), f32)
    assert e.shape == (4, 5) and e.dtype == np.float32
    with pytest.raises(KeyError):
        dtypes.as_dtype(torch.float64)
    with pytest.raises(ValueError):
        types.ti_type([1, 2, 3])


def test_shard_cameras_partition():
    from taichi_image_b200.distributed import shard_cameras
    for n, w in [(12, 8), (12, 2), (12, 4), (6, 1), (3, 8), (64, 8)]:
        parts = [list(shard_cameras(n, w, r)) for r in range(w)]
        assert sorted(sum(parts, [])) == list(range(n))
        assert max(map(len, parts)) - min(map(len, parts)) <= 1
    assert max(len(shard_cameras(12, 8, r)) for r in range(8)) == 2      # 12 cameras on 8 GPUs cap at 6x


def test_integer_demosaic_equals_floor_division():
    """The float quantisation chain of bayer.py:150-155 equals clamp(floor(S / t), 0, scale) for every
    reachable integer tap sum S and every border normaliser t -- the identity the CUDA integer path uses."""
    for s in (255, 65535, 32767):
        for t in (10, 11, 12, 13, 14, 15, 16, 17, 18, 20):
            S = np.arange(-64, t * s + 65, dtype=np.int64)
            f = np.clip(S.astype(np.float32) / np.float32(np.float32(s) * np.float32(t)), np.float32(0), np.float32(1))
            out = np.trunc(f * np.float32(s)).astype(np.int64)
            assert np.array_equal(out, np.clip(S // t, 0, s)), (s, t)


def test_border_normaliser_never_zero_and_constant_images():
    for p in O.PATTERNS:
        for shape in [(2, 2), (2, 4), (4, 2), (4, 6), (6, 6), (8, 10)]:
            b = np.full(shape, 200, np.uint8)
            assert np.all(O.bayer_to_rgb(b, p) == 200), (p, shape)


def test_malvar_matches_published_coefficients():
    from scipy.ndimage import correlate
    r = np.random.default_rng(0)
    cfa = (r.integers(0, 4096, size=(16, 20)) / 4095).astype(np.float32)
    rgb = O.demosaic_unit(cfa, "RGGB")
    g_at_rb = np.array([[0, 0, -1, 0, 0], [0, 0, 2, 0, 0], [-1, 2, 4, 2, -1], [0, 0, 2, 0, 0], [0, 0, -1, 0, 0]]) / 8
    r_at_g_rrow = np.array([[0, 0, .5, 0, 0], [0, -1, 0, -1, 0], [-1, 4, 5, 4, -1], [0, -1, 0, -1, 0], [0, 0, .5, 0, 0]]) / 8
    r_at_b = np.array([[0, 0, -1.5, 0, 0], [0, 2, 0, 2, 0], [-1.5, 0, 6, 0, -1.5], [0, 2, 0, 2, 0], [0, 0, -1.5, 0, 0]]) / 8
    f = lambda k: np.clip(correlate(cfa.astype(np.float64), k, mode="constant"), 0, 1)
    assert np.abs(f(g_at_rb)[2:-2:2, 2:-2:2] - rgb[2:-2:2, 2:-2:2, 1]).max() < 1e-6
    assert np.abs(f(r_at_g_rrow)[2:-2:2, 3:-2:2] - rgb[2:-2:2, 3:-2:2, 0]).max() < 1e-6
    assert np.abs(f(r_at_g_rrow.T)[3:-2:2, 2:-2:2] - rgb[3:-2:2, 2:-2:2, 0]).max() < 1e-6
    assert np.abs(f(r_at_b)[3:-2:2, 3:-2:2] - rgb[3:-2:2, 3:-2:2, 0]).max() < 1e-6


def test_packed_roundtrip_and_ids_quirk():
    r = np.random.default_rng(1)
    for _ in range(20):                                   # reference test/packed.py:6-15
        x = r.integers(0, 4096, size=int(r.integers(1000)) * 2).astype(np.uint16)
        assert np.array_equal(O.decode12(O.encode12(x)), x)
    x = r.integers(0, 4096, size=64).astype(np.uint16)
    y = O.decode12(O.encode12(x, ids_format=True), ids_format=True)
    exp = x.copy()                                        # the reference's IDS encode swaps the low nibbles
    exp[0::2] = (x[0::2] & 0xFF0) | (x[1::2] & 0xF)
    exp[1::2] = (x[1::2] & 0xFF0) | (x[0::2] & 0xF)
    assert np.array_equal(y, exp)


def test_c_abi_rejects_bad_arguments_without_touching_the_gpu():
    """Every entry point validates its arguments before the first CUDA call and reports through the status code +
    b200isp_last_error (include/b200isp.h conventions): exercised on the CPU with arguments that must be refused."""
    import ctypes as C
    from taichi_image_b200 import _lib
    lib = _lib.lib
    E_ARG, E_DTYPE, E_SHAPE, E_FRAMES = -1, -2, -3, -6
    dummy = C.c_void_p(0x1000)                                  # never dereferenced: validation fails first
    f9 = (C.c_float * 9)()
    assert lib.b200isp_bayer_to_rgb(dummy, 0, dummy, 0, 5, 8, 0, None, None) == E_SHAPE             # odd height
    assert b"even size" in lib.b200isp_last_error()
    assert lib.b200isp_bayer_to_rgb(dummy, 0, dummy, 0, 4, 8, 7, None, None) == E_ARG               # unknown pattern
    assert lib.b200isp_bayer_to_rgb(dummy, 9, dummy, 0, 4, 8, 0, None, None) == E_DTYPE
    assert lib.b200isp_bayer_to_rgb(None, 0, None, 0, 0, 0, 0, None, None) == 0                      # empty image: no-op
    assert lib.b200isp_rgb_to_bayer(dummy, dummy, 0, 4, 4, 9, None) == E_ARG
    assert lib.b200isp_rgb_yuv420(dummy, 0, dummy, 0, 5, 4, f9, None) == E_SHAPE
    assert lib.b200isp_transform(dummy, dummy, 0, 4, 4, 42, None) == E_ARG
    assert lib.b200isp_metering_update(None, 1, 4, 8, 8, 8, 0.0, None, None, None) == E_ARG
    p = _lib.FusedParams()
    p.height, p.width, p.pattern, p.isp_dtype, p.out_dtype, p.tonemap, p.gamma = 8, 16, 0, 4, 0, 0, 1.0
    ptrs = (C.c_void_p * 1)(0x1000)
    assert lib.b200isp_process_packed12(ptrs, ptrs, 0, p, dummy, dummy, None) == E_FRAMES           # no frames
    assert lib.b200isp_process_packed12(ptrs, ptrs, 65, p, dummy, dummy, None) == E_FRAMES          # > B200ISP_MAX_FRAMES
    p.width = 12
    assert lib.b200isp_process_packed12(ptrs, ptrs, 1, p, dummy, dummy, None) == E_SHAPE            # width % 8 != 0
    p.width, p.isp_dtype = 16, 0
    assert lib.b200isp_process_packed12(ptrs, ptrs, 1, p, dummy, dummy, None) == E_DTYPE            # ISP dtype must be f16 / f32
    p.isp_dtype, p.gamma = 4, 0.0
    ptrs16 = (C.c_void_p * 1)(0x1000)
    assert lib.b200isp_process_packed12(ptrs16, ptrs16, 1, p, dummy, dummy, None) == E_ARG          # gamma must be positive
    # transposing transforms (flip 4..7) only where the normalise pass of a one-sweep Reinhard -> u8 form turns the image
    from taichi_image_b200 import dtypes
    h, w = 32, 64
    f16, f32, u8, u16 = (d.code for d in (dtypes.f16, dtypes.f32, dtypes.u8, dtypes.u16))
    pitched = 3 * h + 48                                 # elements per row of the (W, H) output, a multiple of 16 bytes
    for isp, what, fields in ((f16, "linear", dict(tonemap=0, gamma=1.0)), (f32, "linear", dict(tonemap=0, gamma=1.0)),
                              (f16, "RGB16 Reinhard", dict(out_dtype=u16)), (f32, "RGB16 Reinhard", dict(out_dtype=u16)),
                              (f16, "IDS Reinhard", dict(ids_layout=1)), (f32, "IDS Reinhard", dict(ids_layout=1)),
                              (f32, "pitched Reinhard, gamma > 1", dict(out_pitch=pitched, gamma=1.2)),
                              (f32, "pitched Reinhard, color_adapt", dict(out_pitch=pitched, color_adapt=0.5))):
        for flip in range(4, 8):
            q = _lib.FusedParams()
            q.height, q.width, q.isp_dtype, q.out_dtype, q.tonemap, q.gamma, q.flip = h, w, isp, u8, 1, 0.9, flip
            for name, value in fields.items():
                setattr(q, name, value)
            assert lib.b200isp_process_packed12(ptrs, ptrs, 1, q, dummy, dummy, None) == E_ARG, (isp, what, flip)
            assert b"transposing" in lib.b200isp_last_error()
            assert lib.b200isp_reinhard_scratch_bytes(q, 1) == 0
            q.out_dtype, q.tonemap, q.gamma, q.color_adapt, q.ids_layout = u8, 1, 0.9, 0.0, 0
            assert lib.b200isp_reinhard_scratch_bytes(q, 1) > 0, (isp, what, flip)     # Reinhard -> u8: a turned form
    assert lib.b200isp_mailbox_bytes(0) == 0 and lib.b200isp_mailbox_bytes(8) > 0
    assert lib.b200isp_mailbox_exchange(dummy, 3, ptrs, 1, 0, dummy, None) == E_ARG                  # kind must be 1 | 2
    assert lib.b200isp_sample_histogram(dummy, 10, 0, dummy, None) == E_ARG
    with pytest.raises(_lib.B200ISPError, match="bad shape"):
        _lib.check(E_SHAPE, "demo")



def test_fused_call_turns_images_only_in_the_one_sweep_reinhard_forms(monkeypatch):
    """host logic of ISP._fused_flip (no GPU): which ISP transforms the fused call applies itself -- flips in the sweep's
    store on every path, transposing transforms (interpolate.py:36-56) in the normalise pass of the one-sweep Reinhard -> u8
    forms only; everything else returns 0 = the transform kernel runs behind the call"""
    import torch
    from taichi_image_b200 import camera_isp, bayer
    from taichi_image_b200.dtypes import u8, u16, f16
    from taichi_image_b200.interpolate import ImageTransform as T
    monkeypatch.delenv("B200ISP_REINHARD_EXACT", raising=False)
    cpu = torch.device("cpu")
    codes = {T.flip_horiz: 1, T.flip_vert: 2, T.rotate_180: 3, T.transpose: 4, T.rotate_270: 5, T.rotate_90: 6, T.transverse: 7}
    for cam in (camera_isp.Camera16, camera_isp.Camera32):
        for t, code in codes.items():
            isp = cam(bayer.BayerPattern.RGGB, transform=t, device=cpu)
            assert isp._fused_flip(3000, "reinhard", u8, 0.9, 0.0) == code
            turning = code & 4
            assert isp._fused_flip(3000, "linear", u16, 1.0, 0.0) == (0 if turning else code)        # the sweep writes the output itself
            assert isp._fused_flip(3000, "reinhard", f16, 0.9, 0.0) == (0 if turning else code)
            assert isp._fused_flip(3004, "reinhard", u8, 0.9, 0.0) == (0 if turning else code)       # height % 8 != 0
            assert isp._fused_flip(3000, "reinhard", u8, 0.9, 0.0, ids_format=True) == (0 if turning else code)
            assert isp._fused_flip(3000, "reinhard", u8, 0.9, 0.0, yuv420=True) == 0
        assert cam(bayer.BayerPattern.RGGB, device=cpu)._fused_flip(3000, "reinhard", u8, 0.9, 0.0) == 0
        assert cam(bayer.BayerPattern.RGGB, transform=T.rotate_90, resize_width=1920, device=cpu)._fused_flip(3000, "reinhard", u8, 0.9, 0.0) == 0
    # Camera32: only where the one-sweep u16 map applies (color_adapt == 0, 0.3 <= gamma <= 1, not reinhard_exact)
    isp = camera_isp.Camera32(bayer.BayerPattern.RGGB, transform=T.rotate_90, device=cpu)
    assert isp._fused_flip(3000, "reinhard", u8, 1.2, 0.0) == 0 and isp._fused_flip(3000, "reinhard", u8, 0.9, 0.5) == 0
    assert camera_isp.Camera32(bayer.BayerPattern.RGGB, transform=T.rotate_90, reinhard_exact=True, device=cpu)._fused_flip(3000, "reinhard", u8, 0.9, 0.0) == 0
    assert camera_isp.Camera16(bayer.BayerPattern.RGGB, transform=T.rotate_90, device=cpu)._fused_flip(3000, "reinhard", u8, 1.2, 0.5) == 6


def _expected_reinhard_scratch(isp, out, tonemap, gamma, ca, mode, flip, yuv, ids, pitched, resize, n, h, w, ho, wo):
    """the bytes of reinhard_scratch with which b200isp_process_packed12 takes its one-sweep Reinhard form (the plan of
    csrc/fused_isp.cuh reinhard_plan, restated); 0 where it uses no scratch or refuses the parameter block"""
    f16, u8 = "f16", "u8"
    if tonemap != "reinhard" or out == "f32":
        return 0
    refused = ((yuv and (isp != f16 or out != u8 or resize or flip or pitched)) or (flip and resize)
               or (flip & 4 and h % 8) or (ids and resize) or (pitched and resize))
    if refused:
        return 0
    g = np.float32(gamma)                 # the library sees the float32 of the parameter block
    if resize:
        return n * ho * wo * 3 * (2 if isp == f16 else 4)
    if isp == f16:
        if out == u8 and flip & 4 and not ids and not yuv:
            return n * h * w * 6                                      # f16 map + turned pass
        if yuv:
            return n * h * w * 6                                      # f16 map + YUV pass
        if not pitched and flip == 0:
            return n * h * w * 6 + (n * 65536 if out == u8 and g != np.float32(1) else 0)   # table / arithmetic pass
        return 0                                                      # exact two sweeps
    if (out == u8 and mode == 0 and ca == 0 and np.float32(0.3) <= g <= np.float32(1) and not yuv and not ids
            and (flip == 0 or flip & 4)):
        return n * h * w * 6                                          # u16 map + map16 / turned pass + gated sweeps
    return 0


def test_reinhard_scratch_query_matches_the_plan_and_sizes_the_isp_scratch():
    """b200isp_reinhard_scratch_bytes (no GPU) over every parameter that selects a Reinhard form, against the plan restated
    above; ISP._fused_params asks it for exactly that scratch, and allocates none where the call runs the exact form"""
    import itertools
    import torch
    from taichi_image_b200 import _lib, camera_isp, bayer, dtypes
    query = _lib.lib.b200isp_reinhard_scratch_bytes
    n, w, ho, wo = 3, 4096, 1080, 1920
    pitch = 3 * w + 48                    # >= 3 * (output row) for both orientations, a multiple of 16 elements
    tms = {"linear": 0, "reinhard": 1, "none": 2}
    grid = itertools.product(("f16", "f32"), ("u8", "u16", "f16", "f32"), tms, (0.29, 0.3, 0.9, 1.0, 1.2), (0.0, 0.5),
                             (0, 1, 2), range(8), (0, 1), (0, 1), (0, 1), (0, 1), (3000, 3004))
    checked = 0
    for isp, out, tm, gamma, ca, mode, flip, yuv, ids, pitched, resize, h in grid:
        p = _lib.FusedParams()
        p.height, p.width, p.isp_dtype, p.out_dtype = h, w, dtypes.as_dtype(isp).code, dtypes.as_dtype(out).code
        p.tonemap, p.gamma, p.color_adapt, p.reinhard_mode = tms[tm], gamma, ca, mode
        p.flip, p.out_yuv420, p.ids_layout, p.out_pitch = flip, yuv, ids, pitch if pitched else 0
        if resize:
            p.out_height, p.out_width, p.scale_r, p.scale_c = ho, wo, ho / h, wo / w
        exp = _expected_reinhard_scratch(isp, out, tm, gamma, ca, mode, flip, yuv, ids, pitched, resize, n, h, w, ho, wo)
        assert query(p, n) == exp, (isp, out, tm, gamma, ca, mode, flip, yuv, ids, pitched, resize, h)
        checked += exp > 0
    assert checked > 0
    p = _lib.FusedParams()
    p.height, p.width, p.isp_dtype, p.out_dtype, p.tonemap, p.gamma = 3000, w, dtypes.f16.code, dtypes.u8.code, 1, 0.9
    assert query(p, n) == n * 3000 * w * 6 + n * 65536
    assert query(p, 0) == 0 and query(p, 65) == 0 and query(None, n) == 0     # frame counts the call refuses, no block

    # the ISP's parameter blocks (CPU tensors: _fused_params only reads their shape and allocates the scratch it is told)
    cpu = torch.device("cpu")
    T = camera_isp.interpolate.ImageTransform
    for cam, exact, resize in itertools.product((camera_isp.Camera16, camera_isp.Camera32), (False, True), (False, True)):
        isp = cam(bayer.BayerPattern.RGGB, device=cpu, reinhard_exact=exact, resize_size=(wo, ho) if resize else None)
        for h in (3000, 3004):
            frames = [torch.empty((h, w * 3 // 2), dtype=torch.uint8)] * n
            for out, tm, gamma, ca, flip, yuv, ids, pitched in itertools.product(
                    ("u8", "u16", "f16"), ("linear", "reinhard"), (0.29, 0.9, 1.0), (0.0, 0.5), (0, 3, 6), (0, 1), (0, 1), (0, 1)):
                isp._reinhard_scratch = None
                p = isp._fused_params(frames, tm, dtypes.as_dtype(out), dict(gamma=gamma, color_adapt=ca), yuv420=yuv,
                                      ids_format=ids, flip=flip, out_pitch=pitch if pitched else 0)
                exp = _expected_reinhard_scratch(isp.dtype.name, out, tm, gamma, ca, int(exact), flip, yuv, ids, pitched, resize,
                                                 n, h, w, ho, wo)
                assert p.reinhard_scratch_bytes == exp == query(p, n), (cam.__name__, exact, resize, h, out, tm, gamma, ca, flip, yuv, ids, pitched)
                assert (isp._reinhard_scratch is None) == (exp == 0)
