"""ctypes binding of the ray-casting oracle (oracle/oracle_rays.cpp -> liboracle_rays.so): the CPU restatement's whole
C surface plus orc_cast_rays.  TEST INFRASTRUCTURE ONLY.  The reference has no ray query, so this oracle is always the
restatement."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

from mlmapping_b200.capi import RAY_HIT_DTYPE, RAY_INFLATED, MlmConfig
from oracle_binding import Oracle, _prototypes

_ORACLE_DIR = Path(__file__).resolve().parent.parent / "oracle"
_SOURCES = [_ORACLE_DIR / "oracle_rays.cpp", _ORACLE_DIR / "oracle_capi.cpp", _ORACLE_DIR / "mlmap_oracle.hpp",
            _ORACLE_DIR.parent / "include" / "mlmap_b200.h"]
# the flags of oracle/Makefile (the reference's CMakeLists.txt:4): no -march, so no fused multiply-add
_CXXFLAGS = ["-std=c++17", "-O3", "-Wall", "-pthread", "-fPIC", "-shared"]
_lib = None


def library_path() -> Path:
    """next to the other oracle library, or in the temporary directory when the tree is not writable"""
    if os.access(_ORACLE_DIR, os.W_OK):
        return _ORACLE_DIR / "liboracle_rays.so"
    return Path(tempfile.gettempdir()) / f"liboracle_rays_{os.getuid()}.so"


def build() -> Path:
    out = library_path()
    cmd = [os.environ.get("CXX", "g++"), *_CXXFLAGS, "-o", str(out), str(_ORACLE_DIR / "oracle_rays.cpp")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("ray oracle build failed:\n" + res.stdout + res.stderr)
    return out


def load():
    global _lib
    if _lib is not None:
        return _lib
    out = library_path()
    if not out.exists() or any(p.stat().st_mtime > out.stat().st_mtime for p in _SOURCES):
        build()
    lib = _prototypes(C.CDLL(str(out)))
    lib.orc_cast_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]
    _lib = lib
    return lib


class RayOracle(Oracle):
    """oracle_binding.Oracle (the restatement) over liboracle_rays.so, with cast_rays"""

    def __init__(self, cfg: MlmConfig, bookkeeping: bool = True):
        self.impl = "port"
        self.lib = load()
        self.cfg = cfg.copy()
        self.h = C.c_void_p(self.lib.orc_create(C.byref(self.cfg)))
        self.lib.orc_set_bookkeeping(self.h, 1 if bookkeeping else 0)
        self.cells = cfg.subbox_n ** 3
        self.last_seconds = 0.0

    def cast_rays(self, from_, to, inflated=False) -> np.ndarray:
        """mlm_cast_rays restated: one RAY_HIT_DTYPE record per segment from_[i] -> to[i]"""
        a, b = self._pos(from_), self._pos(to)
        if a.shape != b.shape:
            raise ValueError(f"from_ and to differ in shape: {a.shape} vs {b.shape}")
        out = np.empty(a.shape[0], dtype=RAY_HIT_DTYPE)
        self.lib.orc_cast_rays(self.h, a.ctypes.data, b.ctypes.data, a.shape[0], RAY_INFLATED if inflated else 0,
                               out.ctypes.data)
        return out
