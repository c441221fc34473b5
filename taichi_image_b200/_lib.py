"""ctypes binding of ``libb200isp.so`` (C ABI declared in ``include/b200isp.h``).

The library is the product: if it is missing the import fails loudly -- there is no CPU or PyTorch
fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import torch

import os

_HERE = Path(__file__).resolve().parent
# B200ISP_LIB selects an experimental build of the same library (build.py --out); default: the in-tree product
LIB_PATH = Path(os.environ["B200ISP_LIB"]).resolve() if os.environ.get("B200ISP_LIB") else _HERE / "libb200isp.so"

MAX_FRAMES = 64

ERRORS = {-1: "bad argument", -2: "bad dtype", -3: "bad shape", -4: "misaligned", -5: "CUDA error",
          -6: "too many frames", -7: "workspace too small"}


class B200ISPError(RuntimeError):
    pass


class FusedParams(C.Structure):
    """mirror of b200isp_fused_params (include/b200isp.h)"""
    _fields_ = [("height", C.c_int), ("width", C.c_int), ("pattern", C.c_int), ("isp_dtype", C.c_int),
                ("out_dtype", C.c_int), ("tonemap", C.c_int), ("has_ccm", C.c_int), ("ccm", C.c_float * 9),
                ("gamma", C.c_float), ("intensity", C.c_float), ("light_adapt", C.c_float),
                ("color_adapt", C.c_float), ("metering_stride", C.c_int), ("alpha", C.c_float),
                ("update_metering", C.c_int), ("rows_per_task", C.c_int), ("demosaic", C.c_int), ("out_yuv420", C.c_int),
                ("out_height", C.c_int), ("out_width", C.c_int),
                ("scale_r", C.c_float), ("scale_c", C.c_float), ("resize_gather", C.c_int), ("out_pitch", C.c_int), ("flip", C.c_int), ("reinhard_mode", C.c_int), ("ids_layout", C.c_int),
                ("profile_start", C.c_void_p), ("profile_stop", C.c_void_p),
                ("meter_cache", C.c_void_p), ("meter_cache_bytes", C.c_size_t),
                ("reinhard_scratch", C.c_void_p), ("reinhard_scratch_bytes", C.c_size_t)]


_vp, _i, _i64, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float

# name -> argtypes; every function returns int status unless listed in _SPECIAL
SIGNATURES = {
    "b200isp_encode12": [_vp, _i, _i64, _vp, _i, _i, _vp],
    "b200isp_decode12": [_vp, _i64, _vp, _i, _i, _i, _vp],
    "b200isp_repack12_ids": [_vp, _vp, _i64, _vp],
    "b200isp_decode16": [_vp, _i64, _vp, _i, _i, _vp],
    "b200isp_decode10": [_vp, _i64, _vp, _i, _i, _vp],
    "b200isp_encode10": [_vp, _i, _i64, _vp, _i, _vp],
    "b200isp_rgb_to_bayer": [_vp, _vp, _i, _i, _i, _i, _vp],
    "b200isp_bayer_to_rgb": [_vp, _i, _vp, _i, _i, _i, _i, C.POINTER(C.c_float), _vp],
    "b200isp_bayer_to_rgb_bilinear": [_vp, _i, _vp, _i, _i, _i, _i, C.POINTER(C.c_float), _vp],
    "b200isp_bounds": [_vp, _i, _i64, _vp, _vp, _vp],
    "b200isp_linear": [_vp, _i, _vp, _i, _i64, _vp, _f, _vp],
    "b200isp_reinhard_standalone": [_vp, _i, _vp, _vp, _i, _i64, _f, _f, _f, _f, _vp, _vp],
    "b200isp_resize_bilinear": [_vp, _i, _i, _i, _vp, _i, _i, _i, _f, _f, _vp],
    "b200isp_resize_area": [_vp, _i, _i, _i, _vp, _i, _i, _i, _vp],
    "b200isp_transform": [_vp, _vp, _i, _i, _i, _i, _vp],
    "b200isp_load_convert": [_vp, _vp, _i, _i64, _i, _vp],
    "b200isp_metering_update": [C.POINTER(_vp), _i, _i, _i, _i, _i, _f, _vp, _vp, _vp],
    "b200isp_isp_reinhard": [_vp, _i, _vp, _i, _i64, _vp, _f, _f, _f, _f, _vp, _vp],
    "b200isp_isp_reinhard_batch": [_vp, _vp, _i, _i, _i, _i64, _vp, _f, _f, _f, _f, _vp, _vp],
    "b200isp_process_packed12": [C.POINTER(_vp), C.POINTER(_vp), _i, C.POINTER(FusedParams), _vp, _vp, _vp],
    "b200isp_metering_phase1": [C.POINTER(_vp), _i, _i, _i, _i, _i, _vp, _vp, _vp],
    "b200isp_metering_phase2": [C.POINTER(_vp), _i, _i, _i, _i, _i, _vp, _i, _f, _vp, _vp, _vp, _vp],
    "b200isp_metering_finalize": [_vp, _vp, _i, _f, _vp, _vp, _vp],
    "b200isp_meter_packed12": [C.POINTER(_vp), _i, C.POINTER(FusedParams), _vp, _vp, _i, _vp, _vp],
    "b200isp_sample_histogram": [_vp, _i64, _i, _vp, _vp],
    "b200isp_histogram_percentiles": [_vp, _i, _vp, _i, _vp, _vp],
    "b200isp_rgb_yuv420": [_vp, _i, _vp, _i, _i, _i, C.POINTER(C.c_float), _vp],
    "b200isp_yuv420_rgb": [_vp, _i, _vp, _i, _i, _i, C.POINTER(C.c_float), _vp],
    "b200isp_mailbox_create": [_i, C.POINTER(_vp), _vp],
    "b200isp_mailbox_open": [_vp, C.POINTER(_vp)],
    "b200isp_mailbox_close": [_vp, _i],
    "b200isp_mailbox_post": [_vp, _i, C.POINTER(_vp), _i, _i, _vp],
    "b200isp_mailbox_wait": [_vp, _i, _i, _vp, _vp],
    "b200isp_mailbox_exchange": [_vp, _i, C.POINTER(_vp), _i, _i, _vp, _vp],
    "b200isp_mailbox_error": [_vp, _i, _vp],
    "b200isp_meter_packed12_shared": [C.POINTER(_vp), _i, C.POINTER(FusedParams), C.POINTER(_vp), _i, _i, _vp, _vp, _vp, _vp],
    "b200isp_meter_packed12_phase1": [C.POINTER(_vp), _i, C.POINTER(FusedParams), _vp, _vp, _vp],
    "b200isp_meter_packed12_phase2": [C.POINTER(_vp), _i, C.POINTER(FusedParams), _vp, _i, _vp, _vp, _vp, _vp],
}
_SPECIAL = {"b200isp_version": ([], C.c_int), "b200isp_last_error": ([], C.c_char_p),
            "b200isp_workspace_bytes": ([], C.c_size_t), "b200isp_mailbox_bytes": ([_i], C.c_size_t),
            "b200isp_reinhard_scratch_bytes": ([C.POINTER(FusedParams), _i], C.c_size_t)}
EXPORTS = tuple(SIGNATURES) + tuple(_SPECIAL)


def _load():
    if not LIB_PATH.exists():
        raise ImportError(
            f"{LIB_PATH} is missing: taichi_image_b200 has no CPU fallback. Build the sm_100a kernels with "
            f"`python build.py` (or `python -c 'import __graft_entry__ as g; g.build()'`) from the repo root.")
    lib = C.CDLL(str(LIB_PATH))
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = argtypes, C.c_int
    for name, (argtypes, restype) in _SPECIAL.items():
        fn = getattr(lib, name)
        fn.argtypes, fn.restype = argtypes, restype
    return lib


lib = _load()
WORKSPACE_BYTES = int(lib.b200isp_workspace_bytes())


def check(status: int, what: str):
    if status != 0:
        msg = lib.b200isp_last_error().decode(errors="replace")
        raise B200ISPError(f"{what}: {ERRORS.get(status, status)}: {msg}")


def require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise B200ISPError(f"{what}: expected a CUDA tensor, got device {t.device} (no CPU fallback)")


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


_workspaces: dict = {}


def workspace(device) -> torch.Tensor:
    """Per (device, stream) scratch buffer, zeroed once (the kernels leave it zeroed)."""
    device = torch.device(device)
    key = (device.index if device.index is not None else torch.cuda.current_device(), stream_ptr(device))
    ws = _workspaces.get(key)
    if ws is None:
        ws = torch.zeros(WORKSPACE_BYTES, dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def ptr_array(tensors):
    arr = (C.c_void_p * len(tensors))()
    for i, t in enumerate(tensors):
        arr[i] = t.data_ptr()
    return arr
