"""Build the C-ABI shared library (libyx_b200.so) with nvcc for sm_100a, in-tree.

Usage: python -m pixeltable_yolox_b200.build [--force]
The library is a plain `extern "C"` .so (no torch / pybind dependency); it links cudart
statically and resolves the one driver entry point it needs (cuTensorMapEncodeTiled) at run
time, so it loads on a GPU-less host (for the symbol checks) and fails loudly only when a
kernel is requested without an sm_100 device.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libyx_b200.so"
OBJ_DIR = PKG / "build"
SOURCES = ["yx_api.cu", "yx_conv_tc.cu", "yx_bneck_tc.cu", "yx_stem_tc.cu", "yx_conv_simt.cu", "yx_misc.cu", "yx_postprocess.cu", "yx_simota.cu", "yx_losses.cu", "yx_train.cu", "yx_preproc.cu", "yx_wgrad_tc.cu", "yx_allreduce_sgd.cu",
           "yx_dwconv_train.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")


def _digest() -> str:
    h = hashlib.sha256()
    for f in sorted(list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "yx_b200.h"]):
        h.update(f.name.encode())
        h.update(f.read_bytes())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build_lib(force: bool = False, verbose: bool = False) -> Path:
    stamp = LIB.with_suffix(".stamp")          # next to the library, so it travels with it when the tree is copied
    digest = _digest()
    if not force and LIB.exists() and stamp.exists() and stamp.read_text().strip() == digest:
        return LIB
    nvcc = _nvcc()
    OBJ_DIR.mkdir(exist_ok=True)

    def compile_one(src: str) -> Path:
        obj = OBJ_DIR / (src + ".o")
        cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            print(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as ex:
        objs = list(ex.map(compile_one, SOURCES))
    cmd = [nvcc, "-shared", "-o", str(LIB), *map(str, objs), "-cudart", "static",
           "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    stamp.write_text(digest)
    return LIB


if __name__ == "__main__":
    print(build_lib(force="--force" in sys.argv, verbose="-v" in sys.argv))
