"""ctypes binding of the signed-distance-field oracle (oracle/oracle_esdf.cpp -> liboracle_esdf.so): the CPU
restatement's whole C surface plus orc_cast_rays plus orc_esdf_*.  TEST INFRASTRUCTURE ONLY.  The reference has no
distance field, so this oracle is always the restatement."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
import time
from pathlib import Path

import numpy as np

from mlmapping_b200.capi import ESDF_INFLATED, MlmConfig, MlmError
from oracle_binding import _prototypes
from ray_oracle import RayOracle

_ORACLE_DIR = Path(__file__).resolve().parent.parent / "oracle"
_SOURCES = [_ORACLE_DIR / "oracle_esdf.cpp", _ORACLE_DIR / "oracle_rays.cpp", _ORACLE_DIR / "oracle_capi.cpp",
            _ORACLE_DIR / "mlmap_oracle.hpp", _ORACLE_DIR.parent / "include" / "mlmap_b200.h"]
# the flags of oracle/Makefile (the reference's CMakeLists.txt:4): no -march, so no fused multiply-add
_CXXFLAGS = ["-std=c++17", "-O3", "-Wall", "-pthread", "-fPIC", "-shared"]
_lib = None


def library_path() -> Path:
    """next to the other oracle libraries, or in the temporary directory when the tree is not writable"""
    if os.access(_ORACLE_DIR, os.W_OK):
        return _ORACLE_DIR / "liboracle_esdf.so"
    return Path(tempfile.gettempdir()) / f"liboracle_esdf_{os.getuid()}.so"


def build() -> Path:
    out = library_path()
    cmd = [os.environ.get("CXX", "g++"), *_CXXFLAGS, "-o", str(out), str(_ORACLE_DIR / "oracle_esdf.cpp")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("ESDF oracle build failed:\n" + res.stdout + res.stderr)
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
    lib.orc_esdf_build.argtypes = [vp, vp, vp, C.c_double, C.c_int]
    lib.orc_esdf_build.restype = C.c_int
    lib.orc_esdf_release.argtypes = [vp]
    lib.orc_esdf_release.restype = None
    lib.orc_esdf_distance.argtypes = [vp, vp, sz, vp, vp]
    lib.orc_esdf_distance.restype = C.c_int
    lib.orc_esdf_export.argtypes = [vp, vp, sz, vp, vp]
    lib.orc_esdf_export.restype = C.c_int
    lib.orc_esdf_export_exact.argtypes = [vp, vp, vp, vp]
    lib.orc_esdf_export_exact.restype = C.c_int
    lib.orc_esdf_squared.argtypes = [vp, vp, C.c_int, vp]
    lib.orc_esdf_squared.restype = None
    _lib = lib
    return lib


def squared_edt(mask: np.ndarray):
    """the oracle's transform alone on a boolean grid [N_z, N_y, N_x]: (D+, D-) int64, -1 for an empty set"""
    lib = load()
    m = np.ascontiguousarray(mask, dtype=np.int8)
    dims = (C.c_int32 * 3)(m.shape[2], m.shape[1], m.shape[0])
    out = []
    for want in (1, 0):
        o = np.empty(m.shape, dtype=np.int64)
        lib.orc_esdf_squared(m.ctypes.data, dims, want, o.ctypes.data)
        out.append(o)
    return out[0], out[1]


class EsdfOracle(RayOracle):
    """RayOracle (the restatement with cast_rays) over liboracle_esdf.so, with the signed distance field"""

    def __init__(self, cfg: MlmConfig, bookkeeping: bool = True):
        self.impl = "port"
        self.lib = load()
        self.cfg = cfg.copy()
        self.h = C.c_void_p(self.lib.orc_create(C.byref(self.cfg)))
        self.lib.orc_set_bookkeeping(self.h, 1 if bookkeeping else 0)
        self.cells = cfg.subbox_n ** 3
        self.last_seconds = 0.0

    def close(self):
        if self.h:
            self.lib.orc_esdf_release(self.h)
        super().close()

    def _rc(self, rc, what):
        if rc != 0:
            raise MlmError(rc, f"oracle {what} returned {rc}")

    def build_esdf(self, box_min, box_max, max_dist, inflated=False) -> float:
        """mlm_esdf_build restated; returns the build's wall time in seconds (one core)"""
        a = (C.c_double * 3)(*[float(v) for v in box_min])
        b = (C.c_double * 3)(*[float(v) for v in box_max])
        t0 = time.perf_counter()
        rc = self.lib.orc_esdf_build(self.h, a, b, float(max_dist), ESDF_INFLATED if inflated else 0)
        seconds = time.perf_counter() - t0
        self._rc(rc, "orc_esdf_build")
        return seconds

    def esdf_distance(self, pos):
        p = self._pos(pos)
        dist = np.empty(p.shape[0], dtype=np.float64)
        grad = np.empty((p.shape[0], 3), dtype=np.float64)
        self._rc(self.lib.orc_esdf_distance(self.h, p.ctypes.data, p.shape[0], dist.ctypes.data, grad.ctypes.data),
                 "orc_esdf_distance")
        return dist, grad

    def _box(self):
        lo, dims = (C.c_int32 * 3)(), (C.c_int32 * 3)()
        self._rc(self.lib.orc_esdf_export(self.h, None, 0, lo, dims), "orc_esdf_export")
        return np.array(lo[:], dtype=np.int32), tuple(int(v) for v in dims)

    def export_esdf(self):
        """(grid[N_z, N_y, N_x] float32, lo[3]) as MLMap.export_esdf"""
        lo, dims = self._box()
        out = np.empty((dims[2], dims[1], dims[0]), dtype=np.float32)
        self._rc(self.lib.orc_esdf_export(self.h, out.ctypes.data, out.size, (C.c_int32 * 3)(), (C.c_int32 * 3)()),
                 "orc_esdf_export")
        return out, lo

    def export_esdf_exact(self):
        """(values float64, D+ int64, D- int64 (-1: +inf)), each [N_z, N_y, N_x], and lo[3]"""
        lo, dims = self._box()
        shape = (dims[2], dims[1], dims[0])
        val, dp, dm = np.empty(shape), np.empty(shape, dtype=np.int64), np.empty(shape, dtype=np.int64)
        self._rc(self.lib.orc_esdf_export_exact(self.h, val.ctypes.data, dp.ctypes.data, dm.ctypes.data),
                 "orc_esdf_export_exact")
        return val, dp, dm, lo
