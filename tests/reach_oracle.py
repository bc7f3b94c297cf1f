"""ctypes binding of the reachability-field oracle (oracle/oracle_reach.cpp -> liboracle_reach.so): the CPU
restatement's whole C surface plus orc_cast_rays, the view gain and its crafted-map setter, plus orc_reach_*.  TEST
INFRASTRUCTURE ONLY.  The reference has no path search, so this oracle is always the restatement."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
import time
from pathlib import Path

import numpy as np

from mlmapping_b200.capi import REACH_INFLATED, REACH_UNKNOWN, MlmConfig, MlmError, ViewSensor
from oracle_binding import _prototypes, create_handle
from view_oracle import ViewOracle

_ORACLE_DIR = Path(__file__).resolve().parent.parent / "oracle"
_SOURCES = [_ORACLE_DIR / "oracle_reach.cpp", _ORACLE_DIR / "oracle_views.cpp", _ORACLE_DIR / "oracle_rays.cpp",
            _ORACLE_DIR / "oracle_capi.cpp", _ORACLE_DIR / "mlmap_oracle.hpp",
            _ORACLE_DIR.parent / "include" / "mlmap_b200.h"]
# the flags of oracle/Makefile (the reference's CMakeLists.txt:4): no -march, so no fused multiply-add
_CXXFLAGS = ["-std=c++17", "-O3", "-Wall", "-pthread", "-fPIC", "-shared"]
_lib = None


def library_path() -> Path:
    """next to the other oracle libraries, or in the temporary directory when the tree is not writable"""
    if os.access(_ORACLE_DIR, os.W_OK):
        return _ORACLE_DIR / "liboracle_reach.so"
    return Path(tempfile.gettempdir()) / f"liboracle_reach_{os.getuid()}.so"


def build() -> Path:
    out = library_path()
    cmd = [os.environ.get("CXX", "g++"), *_CXXFLAGS, "-o", str(out), str(_ORACLE_DIR / "oracle_reach.cpp")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("reach oracle build failed:\n" + res.stdout + res.stderr)
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
    lib.orc_view_gain.argtypes = [vp, vp, sz, C.POINTER(ViewSensor), vp, C.c_int, vp, vp]
    lib.orc_view_gain.restype = C.c_int
    lib.orc_view_set_map.argtypes = [vp, sz, vp, vp, vp, vp, vp, vp]
    lib.orc_view_set_map.restype = None
    lib.orc_reach_build.argtypes = [vp, vp, vp, vp, sz, C.c_double, C.c_int, vp]
    lib.orc_reach_build.restype = C.c_int
    lib.orc_reach_release.argtypes = [vp]
    lib.orc_reach_release.restype = None
    lib.orc_reach_grid.argtypes = [vp, vp, vp, sz, C.c_int64, C.c_int, vp]
    lib.orc_reach_grid.restype = None
    lib.orc_reach_cost.argtypes = [vp, vp, sz, vp]
    lib.orc_reach_cost.restype = C.c_int
    lib.orc_reach_paths.argtypes = [vp, vp, sz, sz, vp, vp]
    lib.orc_reach_paths.restype = C.c_int
    lib.orc_reach_export.argtypes = [vp, vp, sz, vp, vp]
    lib.orc_reach_export.restype = C.c_int
    _lib = lib
    return lib


def reach_flags(inflated=False, unknown=False) -> int:
    return (REACH_INFLATED if inflated else 0) | (REACH_UNKNOWN if unknown else 0)


def reach_grid(cls: np.ndarray, sources, K: int, unknown: bool = False) -> np.ndarray:
    """the oracle's solve alone on a class grid [N_z, N_y, N_x] (0 free, 1 blocking, 2 unknown) with box-relative source
    cells (x, y, z): int64 costs, -1 unreachable"""
    lib = load()
    m = np.ascontiguousarray(cls, dtype=np.int8)
    dims = (C.c_int32 * 3)(m.shape[2], m.shape[1], m.shape[0])
    s = np.ascontiguousarray(np.asarray(sources, dtype=np.int32).reshape(-1, 3))
    out = np.empty(m.shape, dtype=np.int64)
    lib.orc_reach_grid(m.ctypes.data, dims, s.ctypes.data, s.shape[0], int(K), reach_flags(unknown=unknown),
                       out.ctypes.data)
    return out


class ReachOracle(ViewOracle):
    """the restatement (a RayOracle, with the view oracle's crafted-map setter) over liboracle_reach.so, with the
    reachability field"""

    def __init__(self, cfg: MlmConfig, bookkeeping: bool = True):
        self.impl = "port"
        self.lib = load()
        self.cfg = cfg.copy()
        self.h = create_handle(self.lib, self.cfg)
        self.lib.orc_set_bookkeeping(self.h, 1 if bookkeeping else 0)
        self.cells = cfg.subbox_n ** 3
        self.last_seconds = 0.0
        self.last_work = (0, 0)

    def close(self):
        if self.h:
            self.lib.orc_reach_release(self.h)
        super().close()

    def _rc(self, rc, what):
        if rc != 0:
            raise MlmError(rc, f"oracle {what} returned {rc}")

    def build_reach(self, box_min, box_max, starts, max_dist, inflated=False, unknown=False) -> int:
        """mlm_reach_build restated: the number of distinct sources; the build's wall time on one core in last_seconds"""
        a = (C.c_double * 3)(*[float(v) for v in box_min])
        b = (C.c_double * 3)(*[float(v) for v in box_max])
        s = self._pos(starts)
        n = C.c_int32()
        t0 = time.perf_counter()
        rc = self.lib.orc_reach_build(self.h, a, b, s.ctypes.data, s.shape[0], float(max_dist),
                                      reach_flags(inflated, unknown), C.byref(n))
        self.last_seconds = time.perf_counter() - t0
        self._rc(rc, "orc_reach_build")
        return n.value

    def reach_cost(self, pos):
        p = self._pos(pos)
        out = np.empty(p.shape[0], dtype=np.float64)
        self._rc(self.lib.orc_reach_cost(self.h, p.ctypes.data, p.shape[0], out.ctypes.data), "orc_reach_cost")
        return out

    def reach_paths(self, goals, max_cells: int):
        g = self._pos(goals)
        cells = np.zeros((g.shape[0], max_cells, 3), dtype=np.int32)
        ln = np.empty(g.shape[0], dtype=np.int32)
        self._rc(self.lib.orc_reach_paths(self.h, g.ctypes.data, g.shape[0], max_cells, cells.ctypes.data,
                                          ln.ctypes.data), "orc_reach_paths")
        return cells, ln

    def export_reach(self):
        lo, dims = (C.c_int32 * 3)(), (C.c_int32 * 3)()
        self._rc(self.lib.orc_reach_export(self.h, None, 0, lo, dims), "orc_reach_export")
        out = np.empty((dims[2], dims[1], dims[0]), dtype=np.int32)
        self._rc(self.lib.orc_reach_export(self.h, out.ctypes.data, out.size, lo, dims), "orc_reach_export")
        return out, np.array(lo[:], dtype=np.int32)
