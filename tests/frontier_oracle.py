"""ctypes binding of the frontier-clustering oracle (oracle/oracle_frontier.cpp -> liboracle_frontier.so): the CPU
restatement's whole C surface plus orc_cast_rays plus orc_frontier_clusters.  TEST INFRASTRUCTURE ONLY.  The reference
has no clustering, so this oracle is always the restatement."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
import time
from pathlib import Path

import numpy as np

from mlmapping_b200.capi import FRONTIER_CLUSTER_DTYPE, FRONTIER_CONN6, MlmConfig, MlmError
from oracle_binding import _prototypes, create_handle
from ray_oracle import RayOracle

_ORACLE_DIR = Path(__file__).resolve().parent.parent / "oracle"
_SOURCES = [_ORACLE_DIR / "oracle_frontier.cpp", _ORACLE_DIR / "oracle_rays.cpp", _ORACLE_DIR / "oracle_capi.cpp",
            _ORACLE_DIR / "mlmap_oracle.hpp", _ORACLE_DIR.parent / "include" / "mlmap_b200.h"]
# the flags of oracle/Makefile (the reference's CMakeLists.txt:4): no -march, so no fused multiply-add
_CXXFLAGS = ["-std=c++17", "-O3", "-Wall", "-pthread", "-fPIC", "-shared"]
_lib = None


def library_path() -> Path:
    """next to the other oracle libraries, or in the temporary directory when the tree is not writable"""
    if os.access(_ORACLE_DIR, os.W_OK):
        return _ORACLE_DIR / "liboracle_frontier.so"
    return Path(tempfile.gettempdir()) / f"liboracle_frontier_{os.getuid()}.so"


def build() -> Path:
    out = library_path()
    cmd = [os.environ.get("CXX", "g++"), *_CXXFLAGS, "-o", str(out), str(_ORACLE_DIR / "oracle_frontier.cpp")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("frontier oracle build failed:\n" + res.stdout + res.stderr)
    return out


def load():
    global _lib
    if _lib is not None:
        return _lib
    out = library_path()
    if not out.exists() or any(p.stat().st_mtime > out.stat().st_mtime for p in _SOURCES):
        build()
    lib = _prototypes(C.CDLL(str(out)))
    vp, sz = C.c_void_p, C.c_size_t
    lib.orc_cast_rays.argtypes = [vp, vp, vp, sz, C.c_int, vp]
    lib.orc_frontier_clusters.argtypes = [vp, vp, vp, C.c_int32, C.c_int, vp, sz, C.POINTER(sz), vp, vp, sz, C.POINTER(sz)]
    lib.orc_frontier_clusters.restype = C.c_int
    _lib = lib
    return lib


class FrontierOracle(RayOracle):
    """RayOracle (the restatement with cast_rays) over liboracle_frontier.so, with the frontier clustering"""

    def __init__(self, cfg: MlmConfig, bookkeeping: bool = True):
        self.impl = "port"
        self.lib = load()
        self.cfg = cfg.copy()
        self.h = create_handle(self.lib, self.cfg)
        self.lib.orc_set_bookkeeping(self.h, 1 if bookkeeping else 0)
        self.cells = cfg.subbox_n ** 3
        self.last_seconds = 0.0

    def frontier_clusters(self, box_min=None, box_max=None, min_cells=1, conn6=False, labels=False):
        """MLMap.frontier_clusters restated (labels in the oracle's order: cluster by cluster); the call's wall time on
        one core in last_seconds"""
        a = None if box_min is None else (C.c_double * 3)(*[float(v) for v in box_min])
        b = None if box_max is None else (C.c_double * 3)(*[float(v) for v in box_max])
        n, m = C.c_size_t(), C.c_size_t()
        flags = FRONTIER_CONN6 if conn6 else 0
        rc = self.lib.orc_frontier_clusters(self.h, a, b, int(min_cells), flags, None, 0, C.byref(n), None, None, 0,
                                            C.byref(m))
        if rc != 0:
            raise MlmError(rc, f"oracle orc_frontier_clusters returned {rc}")
        out = np.empty(n.value, dtype=FRONTIER_CLUSTER_DTYPE)
        cells = np.empty((m.value if labels else 0, 3), dtype=np.int32)
        of = np.empty(cells.shape[0], dtype=np.int32)
        t0 = time.perf_counter()
        self.lib.orc_frontier_clusters(self.h, a, b, int(min_cells), flags, out.ctypes.data, out.size, C.byref(n),
                                       cells.ctypes.data if labels else None, of.ctypes.data if labels else None,
                                       of.size, C.byref(m))
        self.last_seconds = time.perf_counter() - t0
        return (out, cells, of) if labels else out
