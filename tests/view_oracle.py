"""ctypes binding of the candidate-view-gain oracle (oracle/oracle_views.cpp -> liboracle_views.so): the CPU
restatement's whole C surface plus orc_cast_rays plus orc_view_gain.  TEST INFRASTRUCTURE ONLY.  The reference has no
view scoring, so this oracle is always the restatement."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile
import time
from pathlib import Path

import numpy as np

from mlmapping_b200.capi import VIEW_FRONTIER, VIEW_GAIN_DTYPE, VIEW_INFLATED, MlmConfig, MlmError, ViewSensor
from oracle_binding import _prototypes, create_handle
from ray_oracle import RayOracle

_ORACLE_DIR = Path(__file__).resolve().parent.parent / "oracle"
_SOURCES = [_ORACLE_DIR / "oracle_views.cpp", _ORACLE_DIR / "oracle_rays.cpp", _ORACLE_DIR / "oracle_capi.cpp",
            _ORACLE_DIR / "mlmap_oracle.hpp", _ORACLE_DIR.parent / "include" / "mlmap_b200.h"]
# the flags of oracle/Makefile (the reference's CMakeLists.txt:4): no -march, so no fused multiply-add
_CXXFLAGS = ["-std=c++17", "-O3", "-Wall", "-pthread", "-fPIC", "-shared"]
_lib = None


def library_path() -> Path:
    """next to the other oracle libraries, or in the temporary directory when the tree is not writable"""
    if os.access(_ORACLE_DIR, os.W_OK):
        return _ORACLE_DIR / "liboracle_views.so"
    return Path(tempfile.gettempdir()) / f"liboracle_views_{os.getuid()}.so"


def build() -> Path:
    out = library_path()
    cmd = [os.environ.get("CXX", "g++"), *_CXXFLAGS, "-o", str(out), str(_ORACLE_DIR / "oracle_views.cpp")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("view oracle build failed:\n" + res.stdout + res.stderr)
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
    lib.orc_view_set_map.argtypes = [vp, sz, vp, vp, vp, vp, vp]
    lib.orc_view_set_map.restype = None
    _lib = lib
    return lib


class ViewOracle(RayOracle):
    """RayOracle (the restatement with cast_rays) over liboracle_views.so, with the view gain"""

    def __init__(self, cfg: MlmConfig, bookkeeping: bool = True):
        self.impl = "port"
        self.lib = load()
        self.cfg = cfg.copy()
        self.h = create_handle(self.lib, self.cfg)
        self.lib.orc_set_bookkeeping(self.h, 1 if bookkeeping else 0)
        self.cells = cfg.subbox_n ** 3
        self.last_seconds = 0.0
        self.last_work = (0, 0)

    def view_gain(self, poses, sensor: ViewSensor, boxes=None, frontier=False, inflated=False) -> np.ndarray:
        """MLMap.view_gain restated; the call's wall time on one core in last_seconds, and (cells of the AABBs tested,
        cells the line-of-sight walks visited) in last_work"""
        p = np.ascontiguousarray(np.asarray(poses, dtype=np.float64).reshape(-1, 7))
        b = None if boxes is None else np.ascontiguousarray(np.asarray(boxes, dtype=np.int32).reshape(-1, 6))
        out = np.zeros(p.shape[0], dtype=VIEW_GAIN_DTYPE)
        work = np.zeros(2, dtype=np.int64)
        flags = (VIEW_FRONTIER if frontier else 0) | (VIEW_INFLATED if inflated else 0)
        t0 = time.perf_counter()
        rc = self.lib.orc_view_gain(self.h, p.ctypes.data, p.shape[0], C.byref(sensor),
                                    None if b is None else b.ctypes.data, flags, out.ctypes.data, work.ctypes.data)
        self.last_seconds = time.perf_counter() - t0
        if rc != 0:
            raise MlmError(rc, f"oracle orc_view_gain returned {rc}")
        self.last_work = (int(work[0]), int(work[1]))
        return out

    def set_map(self, ex):
        """replace the map with the subboxes of an export-like dict (glb, collapsed, occupancy, inflate, frontier bytes)"""
        glb = np.ascontiguousarray(ex["glb"], dtype=np.int32)
        col = np.ascontiguousarray(ex["collapsed"], dtype=np.uint8)
        occ = np.ascontiguousarray(ex["occupancy"]).view(np.uint8)
        inf = np.ascontiguousarray(ex["inflate"]).view(np.uint8)
        fr = np.ascontiguousarray(ex["frontier"], dtype=np.uint8)
        self.lib.orc_view_set_map(self.h, glb.shape[0], glb.ctypes.data, col.ctypes.data, occ.ctypes.data,
                                  inf.ctypes.data, fr.ctypes.data)
