"""Builds/loads oracle/_build/liboracle.so (gcc). Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from pathlib import Path

HERE = Path(__file__).resolve().parent
SO = HERE / "_build" / "liboracle.so"
GCC = ["gcc", "-O2", "-ffp-contract=off", "-shared", "-fPIC"]
_lib = None


def _built(so: Path, digest: str) -> bool:
    stamp = so.with_suffix(".stamp")
    return so.exists() and stamp.exists() and stamp.read_text().strip() == digest


def build(force: bool = False) -> Path:
    """Staleness is decided by the source's content, not by file times (a copied tree does not keep them). When the tree
    is read-only and the library there is missing or stale, it is built into a temporary directory instead."""
    src = HERE / "oracle.c"
    digest = hashlib.sha256(src.read_bytes() + " ".join(GCC).encode()).hexdigest()
    if not force and _built(SO, digest):
        return SO
    so = SO
    try:
        so.parent.mkdir(exist_ok=True)
    except OSError:
        pass
    if not os.access(so.parent, os.W_OK):
        so = Path(tempfile.mkdtemp(prefix="yx_oracle_")) / SO.name
    subprocess.run([*GCC, str(src), "-o", str(so), "-lm"], check=True)
    so.with_suffix(".stamp").write_text(digest)
    return so


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = C.CDLL(str(build()))
        _lib.oracle_nms.restype = C.c_int
        _lib.oracle_nms.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p]
        _lib.oracle_simota_matching.restype = C.c_int
        _lib.oracle_simota_matching.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    return _lib
