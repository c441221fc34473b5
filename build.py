#!/usr/bin/env python
"""Build the in-tree native artefacts.

* ``taichi_image_b200/libb200isp.so``  -- the hand-written sm_100a CUDA kernels behind the C ABI of
  ``include/b200isp.h`` (nvcc cross-compiles without a GPU; no -use_fast_math: IEEE division is part
  of the bit-exact contract, SURVEY 7.3 H2).
* ``oracle/_build/libisp_oracle.so``   -- the plain-C restatement used as the timed CPU baseline
  (test infrastructure, never loaded by the product).

Usage: python build.py [--force] [--jobs N] [--no-oracle]
"""
from __future__ import annotations

import argparse
import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent
CSRC = ROOT / "taichi_image_b200" / "csrc"
OBJ = ROOT / "build" / "obj"
LIB = ROOT / "taichi_image_b200" / "libb200isp.so"
ORACLE_SRC = ROOT / "oracle" / "c" / "isp_oracle.c"
ORACLE_LIB = ROOT / "oracle" / "_build" / "libisp_oracle.so"

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--threads", "1", "-Xfatbin", "-compress-all"] + os.environ.get("B200ISP_NVCC_EXTRA", "").split()

FUSED_OUT = {"u8": "uint8_t", "u16": "uint16_t", "f16": "__half", "f32": "float"}


def translation_units():
    """(object name, source, extra defines)"""
    tus = [(n, CSRC / f"{n}.cu", []) for n in ("api", "pack", "demosaic", "tonemap", "resize", "fused_api", "fused_resize", "normalise", "exchange", "yuv420")]
    for name, ctype in (("u8", "uint8_t"), ("u16", "uint16_t"), ("i16", "int16_t"), ("f16", "__half"), ("f32", "float")):
        tus.append((f"demosaic_{name}", CSRC / "demosaic_inst.cu", [f"-DISP_PLANE_T={ctype}"]))
    for cam in (0, 1):
        for mode, mname in ((0, "rgb"), (1, "linear"), (2, "rstore")):
            tus.append((f"resize_cam{16 if cam else 32}_{mname}", CSRC / "resize_inst.cu", [f"-DISP_RZ_CAM16={cam}", f"-DISP_RZ_MODE={mode}"]))
        tus.append((f"fused_rmax_cam{16 if cam else 32}", CSRC / "fused_inst.cu",
                    [f"-DISP_INST_CAM16={cam}", "-DISP_INST_RMAX"]))
        for name, ctype in FUSED_OUT.items():
            if cam and name == "f32":
                continue
            tus.append((f"fused_cam{16 if cam else 32}_{name}", CSRC / "fused_inst.cu",
                        [f"-DISP_INST_CAM16={cam}", f"-DISP_INST_OUT={ctype}"]))
    tus.append(("fused_gated_cam32", CSRC / "fused_inst.cu", ["-DISP_INST_CAM16=0", "-DISP_INST_GATED"]))
    return tus


def _digest(paths, extra=""):
    h = hashlib.sha256(extra.encode())
    for p in sorted(paths):
        h.update(p.name.encode())
        h.update(p.read_bytes())
    return h.hexdigest()


def nvcc_path() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built")


def build_cuda(force=False, jobs=None, verbose=False, out: Path | None = None) -> Path:
    """out: alternative output path for an experimental variant (objects go to build/obj_<stem>); the variant's
    flags come from B200ISP_NVCC_EXTRA and it is selected at run time with B200ISP_LIB=<path>."""
    global OBJ, LIB
    if out is not None:
        LIB = Path(out).resolve()
        OBJ = ROOT / "build" / f"obj_{LIB.stem}"
    sources = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [ROOT / "include" / "b200isp.h"]
    stamp = _digest(sources, " ".join(NVCC_FLAGS))
    stamp_file = OBJ / "stamp"
    if not force and LIB.exists() and stamp_file.exists() and stamp_file.read_text() == stamp:
        return LIB
    OBJ.mkdir(parents=True, exist_ok=True)
    nvcc = nvcc_path()
    tus = translation_units()

    headers = list(CSRC.glob("*.cuh")) + [ROOT / "include" / "b200isp.h"]

    def compile_one(tu):
        name, src, defs = tu
        obj = OBJ / f"{name}.o"
        # per-unit stamp: a change to one .cu file recompiles that unit only (any header change recompiles everything)
        tu_stamp, tu_stamp_file = _digest([Path(src)] + headers, " ".join([*NVCC_FLAGS, *defs])), OBJ / f"{name}.stamp"
        if not force and not verbose and obj.exists() and tu_stamp_file.exists() and tu_stamp_file.read_text() == tu_stamp:
            return obj
        cmd = [nvcc, *NVCC_FLAGS, *defs, "-c", str(src), "-o", str(obj)]
        if verbose:
            cmd += ["-Xptxas", "-v"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {name}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            (OBJ / f"{name}.ptxas.log").write_text(r.stderr)
        tu_stamp_file.write_text(tu_stamp)
        return obj

    with ThreadPoolExecutor(max_workers=jobs or min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, tus))
    cmd = [nvcc, "-shared", "-o", str(LIB), *map(str, objs), "-gencode", "arch=compute_100a,code=sm_100a",
           "-cudart", "static", "-Xcompiler", "-fPIC"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    stamp_file.write_text(stamp)
    return LIB


def build_oracle(force=False) -> Path | None:
    if not ORACLE_SRC.exists():
        return None
    if not force and ORACLE_LIB.exists() and ORACLE_LIB.stat().st_mtime >= ORACLE_SRC.stat().st_mtime:
        return ORACLE_LIB
    ORACLE_LIB.parent.mkdir(parents=True, exist_ok=True)
    cmd = ["gcc", "-O2", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-shared", "-fPIC",
           "-o", str(ORACLE_LIB), str(ORACLE_SRC), "-lm"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"oracle C build failed:\n{r.stdout}\n{r.stderr}")
    return ORACLE_LIB


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--force", action="store_true")
    ap.add_argument("--jobs", type=int, default=None)
    ap.add_argument("--verbose", action="store_true", help="keep ptxas -v logs under build/obj")
    ap.add_argument("--no-oracle", action="store_true")
    ap.add_argument("--out", default=None, help="build an experimental variant into this .so (see build_cuda)")
    a = ap.parse_args(argv)
    print("built", build_cuda(a.force, a.jobs, a.verbose, a.out))
    if not a.no_oracle:
        print("built", build_oracle(a.force))


if __name__ == "__main__":
    sys.exit(main())
