"""ctypes wrapper of oracle/c/isp_oracle.c (TEST INFRASTRUCTURE ONLY: CPU baseline + cross-check)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "c", "isp_oracle.c")
LIB = os.path.join(HERE, "_build", "libisp_oracle.so")
PATTERN_CODE = {"RGGB": 0, "GRBG": 1, "GBRG": 2, "BGGR": 3}


def build(force=False) -> str:
    """The library build.py left in the tree when it is current; otherwise a fresh build in a temporary directory
    that lives as long as this process, so that running the oracle (tests, bench.py's CPU baseline) never writes
    into a tree that may be read-only."""
    global _tmp
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= os.path.getmtime(SRC):
        return LIB
    _tmp = tempfile.TemporaryDirectory(prefix="isp_oracle_")
    out = os.path.join(_tmp.name, os.path.basename(LIB))
    subprocess.run(["gcc", "-O2", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC",
                    "-o", out, SRC, "-lm"], check=True)
    return out


_lib = None
_tmp = None


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(build())
        _lib.isp_oracle_process.restype = C.c_int
        _lib.isp_oracle_process_resized.restype = C.c_int
        _lib.isp_oracle_max_threads.restype = C.c_int
    return _lib


def max_threads() -> int:
    return int(lib().isp_oracle_max_threads())


def process(frames, pattern="RGGB", cam16=False, out_dtype="u8", tonemap="reinhard", ccm=None, gamma=1.0,
            intensity=1.0, light_adapt=1.0, color_adapt=0.0, stride=8, alpha=0.0, metrics=None, nthreads=0,
            resize=None):
    """frames: list of (H, 1.5 W) uint8 arrays -> (list of (H, W, 3) outputs, metrics[9]).
    resize = ((width, height), (scale_row, scale_col)): the ISP's bilinear resize (camera_isp.py:302-315) before
    metering / tone map; outputs are then (height, width, 3)."""
    h, w3 = frames[0].shape
    w = w3 * 2 // 3
    frames = [np.ascontiguousarray(f) for f in frames]
    ho, wo = (h, w) if resize is None else (int(resize[0][1]), int(resize[0][0]))
    outs = [np.empty((ho, wo, 3), np.uint16 if out_dtype == "u16" else np.uint8) for _ in frames]
    m = np.zeros(9, np.float32) if metrics is None else np.array(metrics, np.float32)
    inp = (C.c_void_p * len(frames))(*[f.ctypes.data for f in frames])
    outp = (C.c_void_p * len(frames))(*[o.ctypes.data for o in outs])
    ccm_arr = None if ccm is None else np.asarray(ccm, np.float64).reshape(-1).astype(np.float32)
    args = [inp, outp, len(frames), h, w, PATTERN_CODE[pattern], int(cam16), int(out_dtype == "u16"),
            int(tonemap == "reinhard"), None if ccm_arr is None else ccm_arr.ctypes.data_as(C.c_void_p),
            C.c_float(gamma), C.c_float(intensity), C.c_float(light_adapt), C.c_float(color_adapt),
            int(stride), C.c_float(alpha), m.ctypes.data_as(C.c_void_p), int(nthreads)]
    if resize is None:
        st = lib().isp_oracle_process(*args)
    else:
        st = lib().isp_oracle_process_resized(*args, ho, wo, C.c_float(resize[1][0]), C.c_float(resize[1][1]))
    assert st == 0
    return outs, m
