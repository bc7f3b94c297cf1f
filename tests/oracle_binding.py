"""ctypes binding of the CPU oracle (oracle/liboracle.so).  TEST INFRASTRUCTURE ONLY: imported by
tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs, never by the
product package."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from mlmapping_b200.capi import FrameStats, MlmConfig  # noqa: E402  (struct layouts only)

_ORACLE_DIR = ROOT / "oracle"
_LIB = _ORACLE_DIR / "liboracle.so"
_REF_LIB = _ORACLE_DIR / "_ref" / "libmlmap_ref.so"  # the UNMODIFIED reference sources (oracle/ref_build/Makefile)
# a checkout of the original MLMapping sources (the repository does not ship them): MLMAPPING_REFERENCE, else the
# documented place
_REFERENCE = Path(os.environ.get("MLMAPPING_REFERENCE") or "/root/reference")
_lib = None
_ref_lib = None


def build_oracle():
    res = subprocess.run(["make", "-C", str(_ORACLE_DIR)], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + res.stdout + res.stderr)
    return _LIB


def build_reference():
    """compile the reference's own mapping sources (_REFERENCE) into oracle/_ref"""
    res = subprocess.run(["make", "-C", str(_ORACLE_DIR / "ref_build"), "-j8", f"REF={_REFERENCE}"], capture_output=True,
                         text=True)
    if res.returncode != 0:
        raise RuntimeError("oracle/_ref build failed:\n" + res.stdout[-3000:] + res.stderr[-3000:])
    return _REF_LIB


def reference_sources() -> bool:
    """the original sources are there and readable (os.path.isdir is False, not an error, where a user may not look)"""
    return os.path.isdir(_REFERENCE)


def reference_available() -> bool:
    """a library built earlier, or the sources to build it from"""
    return _REF_LIB.exists() or reference_sources()


def load_reference():
    global _ref_lib
    if _ref_lib is not None:
        return _ref_lib
    if reference_sources():
        build_reference()  # make: a no-op when up to date
    if not _REF_LIB.exists():
        raise FileNotFoundError(f"{_REF_LIB} missing and no original sources at {_REFERENCE} (MLMAPPING_REFERENCE)")
    _ref_lib = _prototypes(C.CDLL(str(_REF_LIB)))
    _ref_lib.orc_get_odd_at.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    return _ref_lib


def load_oracle():
    global _lib
    if _lib is not None:
        return _lib
    src_newer = (not _LIB.exists()) or any(
        p.stat().st_mtime > _LIB.stat().st_mtime for p in [_ORACLE_DIR / "mlmap_oracle.hpp", _ORACLE_DIR / "oracle_capi.cpp"])
    if src_newer:
        build_oracle()
    _lib = _prototypes(C.CDLL(str(_LIB)))
    return _lib


def _prototypes(lib):
    vp, sz, dp = C.c_void_p, C.c_size_t, C.POINTER(C.c_double)
    lib.orc_create.argtypes, lib.orc_create.restype = [C.POINTER(MlmConfig)], vp
    lib.orc_destroy.argtypes = [vp]
    lib.orc_set_bookkeeping.argtypes = [vp, C.c_int]
    lib.orc_integrate_depth_u16.argtypes = [vp, vp, C.c_int, C.c_int, sz, dp]
    lib.orc_integrate_depth_u16.restype = C.c_double
    lib.orc_integrate_points_f64.argtypes = [vp, vp, C.c_int, dp]
    lib.orc_integrate_points_f64.restype = C.c_double
    lib.orc_frame_stats.argtypes = [vp, C.POINTER(FrameStats)]
    lib.orc_num_points.argtypes, lib.orc_num_points.restype = [vp], sz
    lib.orc_get_points.argtypes, lib.orc_get_points.restype = [vp, vp, sz], sz
    lib.orc_last_hits.argtypes, lib.orc_last_hits.restype = [vp, vp, vp, sz], sz
    lib.orc_last_misses.argtypes, lib.orc_last_misses.restype = [vp, vp, sz], sz
    lib.orc_set_free_in_bound.argtypes = [vp, dp, dp]
    lib.orc_set_log_inserts.argtypes = [vp, C.c_int]
    lib.orc_insert_log.argtypes, lib.orc_insert_log.restype = [vp, vp, sz], sz
    lib.orc_inflate_map.argtypes = [vp, dp]
    lib.orc_get_occupancy.argtypes = [vp, vp, sz, vp]
    lib.orc_get_occupancy_inflate.argtypes = [vp, vp, sz, C.c_float, vp]
    lib.orc_get_inflate_occupancy.argtypes = [vp, vp, sz, vp]
    lib.orc_get_odd.argtypes = [vp, vp, sz, vp]
    lib.orc_get_odd_grad.argtypes = [vp, vp, sz, sz, vp]
    lib.orc_export_map_count.argtypes, lib.orc_export_map_count.restype = [vp], sz
    lib.orc_export_map.argtypes, lib.orc_export_map.restype = [vp, sz, vp, vp, vp, vp, vp], sz
    lib.orc_export_frontier.argtypes, lib.orc_export_frontier.restype = [vp, sz, vp], sz
    lib.orc_released_last.argtypes, lib.orc_released_last.restype = [vp], C.c_int
    lib.orc_export_cloud.argtypes, lib.orc_export_cloud.restype = [vp, C.c_int, vp, sz], sz
    lib.orc_export_odds_slice.argtypes, lib.orc_export_odds_slice.restype = [vp, C.c_double, vp, sz], sz
    lib.orc_odds_table.argtypes, lib.orc_odds_table.restype = [vp, C.c_int, C.c_int], C.c_float
    lib.orc_three_sigma.argtypes, lib.orc_three_sigma.restype = [vp, C.c_int], C.c_float
    lib.orc_fast_atan2.argtypes, lib.orc_fast_atan2.restype = [vp, C.c_double, C.c_double], C.c_double
    lib.orc_logit.argtypes, lib.orc_logit.restype = [C.c_float], C.c_float
    lib.orc_logit_inv.argtypes, lib.orc_logit_inv.restype = [C.c_float], C.c_float
    lib.orc_log10f_array.argtypes = [vp, sz, vp]
    lib.orc_pow2.argtypes, lib.orc_pow2.restype = [C.c_double], C.c_double
    lib.orc_vector_hash.argtypes, lib.orc_vector_hash.restype = [C.c_int, C.c_int, C.c_int], C.c_int
    lib.orc_transform_point.argtypes = [dp, dp, dp, dp]
    lib.orc_T_ls.argtypes = [dp, dp, dp]
    lib.orc_next_bucket_count.argtypes, lib.orc_next_bucket_count.restype = [sz], sz
    lib.orc_compensate_pose.argtypes = [dp, dp, dp, dp, C.c_double, C.c_double, C.c_double, dp]
    return lib


def best_oracle(cfg, **kw):
    """the checker the GPU parity tests use: the reference's own sources (oracle/_ref) when that library is available
    (built from _REFERENCE), else the restatement"""
    return Oracle(cfg, impl="reference" if reference_available() else "port", **kw)


K_DIFF_RANGE = 10  # rows either side of the odds table (awareness_map_cylindrical::diff_range)


def k_reach(cfg) -> np.ndarray:
    """K(rho): the last diff_r of update_hits' loop `diff_r < 3 * sigma_in_dr(rho)`, with the float arithmetic of
    build_awareness_tables (mlmap_capi.cu): dis = (float)(rho * dRho), sigma = (float)(coe * dis * dis / dRho)"""
    out = np.zeros(cfg.am_n_rho, dtype=np.int64)
    for r in range(cfg.am_n_rho):
        dis = float(np.float32(r * cfg.am_d_rho))
        bound = np.float32(3) * np.float32(cfg.depth_noise_coe * dis * dis / cfg.am_d_rho)
        k, d = 0, 1
        while np.float32(d) < bound:
            k = d
            if d > 4 * K_DIFF_RANGE:
                break
            d += 1
        out[r] = k
    return out


def update_hits_ok(cfg) -> bool:
    """mlm_create's precondition of update_hits: K(rho) <= min(10, rho) for every rho, so that the odds-table row
    diff_r + 10 stays within its 21 rows and the neighbour rho - diff_r stays >= 0"""
    k = k_reach(cfg)
    return bool((k <= np.minimum(K_DIFF_RANGE, np.arange(cfg.am_n_rho))).all())


def create_handle(lib, cfg) -> C.c_void_p:
    """orc_create, for configurations the library accepts: update_hits (the reference's code, restated) reads outside
    the odds table and the awareness map when 3 sigma(rho) reaches past them, so such a configuration is refused here
    instead of crashing the process"""
    if not (cfg.am_n_rho >= 2 and cfg.am_d_rho > 0 and cfg.depth_noise_coe >= 0) or not update_hits_ok(cfg):
        raise ValueError("configuration outside update_hits' preconditions: K(rho) <= min(10, rho) fails "
                         f"(am_d_rho {cfg.am_d_rho}, am_n_rho {cfg.am_n_rho}, depth_noise_coe {cfg.depth_noise_coe})")
    return C.c_void_p(lib.orc_create(C.byref(cfg)))


def _d7(a):
    a = np.asarray(a, dtype=np.float64).reshape(-1)
    return (C.c_double * len(a))(*a.tolist())


class Oracle:
    """CPU restatement of the reference's mlmap (oracle/mlmap_oracle.hpp) with the same surface as
    mlmapping_b200.MLMap so parity tests read symmetrically."""

    def __init__(self, cfg: MlmConfig, bookkeeping: bool = True, impl: str = "port"):
        """impl "port": the restatement (oracle/mlmap_oracle.hpp); "reference": the reference's own sources (oracle/_ref)"""
        self.impl = impl
        self.lib = load_reference() if impl == "reference" else load_oracle()
        self.cfg = cfg.copy()
        self.h = create_handle(self.lib, self.cfg)
        self.lib.orc_set_bookkeeping(self.h, 1 if bookkeeping else 0)
        self.cells = cfg.subbox_n ** 3
        self.last_seconds = 0.0

    def close(self):
        if self.h:
            self.lib.orc_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def integrate_depth(self, img, T_wb) -> FrameStats:
        img = np.ascontiguousarray(img, dtype=np.uint16)
        self.last_seconds = self.lib.orc_integrate_depth_u16(self.h, img.ctypes.data, img.shape[0], img.shape[1],
                                                             img.strides[0], _d7(T_wb))
        return self.frame_stats()

    def integrate_points(self, xyz, T_wb) -> FrameStats:
        pts = np.ascontiguousarray(np.asarray(xyz, dtype=np.float64).reshape(-1, 3))
        self.last_seconds = self.lib.orc_integrate_points_f64(self.h, pts.ctypes.data, pts.shape[0], _d7(T_wb))
        return self.frame_stats()

    def frame_stats(self) -> FrameStats:
        st = FrameStats()
        self.lib.orc_frame_stats(self.h, C.byref(st))
        return st

    def points(self):
        n = self.lib.orc_num_points(self.h)
        out = np.empty((n, 3), dtype=np.float64)
        self.lib.orc_get_points(self.h, out.ctypes.data, n)
        return out

    def last_frame_hits(self):
        n = self.lib.orc_last_hits(self.h, None, None, 0)
        keys = np.empty((n, 3), dtype=np.int32)
        p = np.empty(n, dtype=np.float32)
        self.lib.orc_last_hits(self.h, keys.ctypes.data, p.ctypes.data, n)
        return keys, p

    def set_log_inserts(self, on=True):
        self.lib.orc_set_log_inserts(self.h, 1 if on else 0)

    def insert_log(self):
        n = self.lib.orc_insert_log(self.h, None, 0)
        keys = np.empty((n, 3), dtype=np.int32)
        self.lib.orc_insert_log(self.h, keys.ctypes.data, n)
        return keys

    def last_frame_misses(self, sort=True):
        n = self.lib.orc_last_misses(self.h, None, 0)
        idx = np.empty(n, dtype=np.uint64)
        self.lib.orc_last_misses(self.h, idx.ctypes.data, n)
        return np.sort(idx) if sort else idx

    def setFree_map_in_bound(self, box_min, box_max):
        self.lib.orc_set_free_in_bound(self.h, _d7(box_min), _d7(box_max))

    def inflate_map(self, ct_pos):
        self.lib.orc_inflate_map(self.h, _d7(ct_pos))

    @staticmethod
    def _pos(p):
        return np.ascontiguousarray(np.asarray(p, dtype=np.float64).reshape(-1, 3))

    def getOccupancy(self, pos_w, inflate=None):
        p = self._pos(pos_w)
        out = np.empty(p.shape[0], dtype=np.int32)
        if inflate is None:
            self.lib.orc_get_occupancy(self.h, p.ctypes.data, p.shape[0], out.ctypes.data)
        else:
            self.lib.orc_get_occupancy_inflate(self.h, p.ctypes.data, p.shape[0], float(inflate), out.ctypes.data)
        return out

    def getInflateOccupancy(self, pos_w):
        p = self._pos(pos_w)
        out = np.empty(p.shape[0], dtype=np.int32)
        self.lib.orc_get_inflate_occupancy(self.h, p.ctypes.data, p.shape[0], out.ctypes.data)
        return out

    def getOdd(self, pos_w):
        p = self._pos(pos_w)
        out = np.empty(p.shape[0], dtype=np.float32)
        self.lib.orc_get_odd(self.h, p.ctypes.data, p.shape[0], out.ctypes.data)
        return out

    def getOddGrad(self, pos_w, max_iter=5):
        p = self._pos(pos_w)
        out = np.empty((p.shape[0], 3), dtype=np.float64)
        self.lib.orc_get_odd_grad(self.h, p.ctypes.data, p.shape[0], max_iter, out.ctypes.data)
        return out

    def export_cloud(self, kind: int) -> np.ndarray:
        """[n,4] float32 x,y,z,1 of the cells the reference would publish (0 inflated, 1 occupied, 2 frontier)"""
        n = self.lib.orc_export_cloud(self.h, kind, None, 0)
        out = np.zeros((n, 4), dtype=np.float32)
        if n:
            self.lib.orc_export_cloud(self.h, kind, out.ctypes.data, n)
        return out

    def export_odds_slice(self, height: float) -> np.ndarray:
        n = self.lib.orc_export_odds_slice(self.h, float(height), None, 0)
        out = np.zeros((n, 4), dtype=np.float32)
        if n:
            self.lib.orc_export_odds_slice(self.h, float(height), out.ctypes.data, n)
        return out

    def export_map(self):
        n = self.lib.orc_export_map_count(self.h)
        glb = np.zeros((n, 3), dtype=np.int32)
        col = np.zeros(n, dtype=np.uint8)
        occ = np.zeros((n, self.cells), dtype="S1")
        inf = np.zeros((n, self.cells), dtype="S1")
        lo = np.zeros((n, self.cells), dtype=np.float32)
        if n:
            self.lib.orc_export_map(self.h, n, glb.ctypes.data, col.ctypes.data, occ.ctypes.data, inf.ctypes.data,
                                    lo.ctypes.data)
        nb = (self.cells + 7) // 8
        fr = np.zeros((n, nb), dtype=np.uint8)
        if n:
            self.lib.orc_export_frontier(self.h, n, fr.ctypes.data)
        order = np.lexsort((glb[:, 2], glb[:, 1], glb[:, 0]))
        return {"glb": glb[order], "collapsed": col[order], "occupancy": occ[order], "inflate": inf[order],
                "log_odds": lo[order], "frontier": fr[order]}
