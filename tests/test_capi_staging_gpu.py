"""GPU: the host-pointer entry points of the C ABI stage their inputs and outputs through stream-ordered temporaries.
Host variants of the point queries equal their device variants bit for bit; every host call leaves the stream-ordered
pool's used bytes where they were, after a success and after a refused allocation; and a refused call leaves no error
behind for the next call on the thread."""
import ctypes as C

import numpy as np
import pytest

from mlmapping_b200 import MLMap, config_cfg_a, scenes
from test_frontier_host import build_map, explore_cfg_a

pytestmark = pytest.mark.gpu
CU_MEMPOOL_ATTR_USED_MEM_CURRENT = 7  # CUmemPool_attribute, cuda.h
MLM_ERR_CUDA = 3


class _PoolUsage:
    """used bytes of device 0's current stream-ordered memory pool.  Read through the driver API: the library links the
    CUDA runtime statically, so the driver is what this process and the library share."""

    def __init__(self, device: int = 0):
        self._cu = C.CDLL("libcuda.so.1")
        self._cu.cuDeviceGetMemPool.argtypes = [C.POINTER(C.c_void_p), C.c_int]
        self._cu.cuMemPoolGetAttribute.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
        assert self._cu.cuInit(0) == 0
        dev = C.c_int()
        assert self._cu.cuDeviceGet(C.byref(dev), device) == 0
        self._pool = C.c_void_p()
        assert self._cu.cuDeviceGetMemPool(C.byref(self._pool), dev.value) == 0

    def used(self) -> int:
        v = C.c_uint64()
        assert self._cu.cuMemPoolGetAttribute(self._pool, CU_MEMPOOL_ATTR_USED_MEM_CURRENT, C.byref(v)) == 0
        return v.value


def _cfg_a_map(frames: int = 6) -> MLMap:
    cfg = config_cfg_a()
    m = MLMap(cfg)
    for k in range(frames):
        pose = scenes.corridor_trajectory_pose(k * 10)
        m.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    return m


def _points(m: MLMap, n: int, seed: int = 3) -> np.ndarray:
    g = m.export_map()["glb"]
    d = m.cfg.subbox_n * m.cfg.subbox_d_xyz
    return scenes.query_positions(n, g.min(0) * d, (g.max(0) + 1) * d, seed=seed, inflate=2.0)


def _cells(m: MLMap, n: int):
    """(glb[n, 3], sub[n]): cells of allocated subboxes, with every tenth subbox index shifted off the allocated ones"""
    rs = np.random.RandomState(7)
    g = m.export_map()["glb"]
    glb = g[rs.randint(0, g.shape[0], n)].copy()
    glb[::10] += 1000
    return np.ascontiguousarray(glb, dtype=np.int32), rs.randint(0, m.cells, n).astype(np.int32)


def test_host_point_queries_equal_device_variants():
    m = _cfg_a_map()
    pos = _points(m, 50000)
    n = pos.shape[0]
    d_pos, d_out = m.to_device(pos), m.device_alloc(n * 24)
    try:
        m.getOccupancy_device(d_pos, n, d_out)
        assert m.to_host(d_out, n, np.int32).tobytes() == m.getOccupancy(pos).tobytes()
        m.getOdd_device(d_pos, n, d_out)
        assert m.to_host(d_out, n, np.float32).tobytes() == m.getOdd(pos).tobytes()
        m.getOddGrad_device(d_pos, n, d_out, max_iter=5)
        assert m.to_host(d_out, (n, 3), np.float64).tobytes() == m.getOddGrad(pos, max_iter=5).tobytes()
    finally:
        m.device_free(d_pos)
        m.device_free(d_out)
    glb, sub = _cells(m, 20000)
    k = glb.shape[0]
    d_g, d_s, d_o = m.to_device(glb), m.to_device(sub), m.device_alloc(k * 4)
    try:
        m._check(m._lib.mlm_get_odd_at_device(m._h, d_g, d_s, k, d_o))
        assert m.to_host(d_o, k, np.float32).tobytes() == m.getOdd_at(glb, sub).tobytes()
    finally:
        for p in (d_g, d_s, d_o):
            m.device_free(p)


def test_host_calls_return_their_temporaries_to_the_pool():
    pool = _PoolUsage()
    m, replica = _cfg_a_map(), MLMap(config_cfg_a())
    e = MLMap(explore_cfg_a())
    build_map("cfg-a-14", e)
    pos = _points(m, 20000)
    glb, sub = _cells(m, 5000)
    lo = pos.min(0)
    m.sync()
    e.sync()
    base = pool.used()

    def dirty_round_trip():
        n, rb = C.c_int32(), C.c_size_t()
        m._check(m._lib.mlm_dirty_count(m._h, C.byref(n), C.byref(rb)))
        assert n.value > 0
        buf = m.device_alloc(n.value * rb.value)
        m._check(m._lib.mlm_dirty_export(m._h, buf, n.value))
        replica._check(replica._lib.mlm_dirty_import(replica._h, buf, n.value))
        m.device_free(buf)

    def device_cloud():
        buf = e.device_alloc(1024 * 16)
        e.export_cloud_device(e.CLOUD_FRONTIER, buf, 1024)
        e.device_free(buf)

    calls = {
        "mlm_dirty_import": dirty_round_trip,  # first: the dirty blocks are the last frame's
        "mlm_get_occupancy": lambda: m.getOccupancy(pos),
        "mlm_get_occupancy_inflate": lambda: m.getOccupancy(pos, inflate=0.3),
        "mlm_get_inflate_occupancy": lambda: m.getInflateOccupancy(pos),
        "mlm_get_odd": lambda: m.getOdd(pos),
        "mlm_get_odd_grad": lambda: m.getOddGrad(pos, max_iter=5),
        "mlm_get_odd_at": lambda: m.getOdd_at(glb, sub),
        "mlm_last_frame_hits": m.last_frame_hits,
        "mlm_last_frame_misses": m.last_frame_misses,
        "mlm_export_map": m.export_map,
        "mlm_export_frontier": e.export_map,
        "mlm_export_cloud": lambda: [m.export_cloud(kind) for kind in (m.CLOUD_INFLATED, m.CLOUD_OCCUPIED)],
        "mlm_export_cloud_device": device_cloud,
        "mlm_export_odds_slice": lambda: m.export_odds_slice(1.0),
        "mlm_cast_rays": lambda: m.cast_rays(pos[:5000], pos[5000:10000]),
        "mlm_esdf_distance": lambda: (m.build_esdf(lo, lo + 8.0, 2.0), m.esdf_distance(pos)),
        "mlm_esdf_export": m.export_esdf,
        "mlm_frontier_clusters": lambda: e.frontier_clusters(labels=True),
        "mlm_debug_log10f": lambda: m.debug_log10f(np.linspace(0.01, 100.0, 4096, dtype=np.float32)),
        "mlm_checkpoint_save / restore": lambda: m.restore(m.checkpoint()),
        "mlm_set_free_in_bound": lambda: m.setFree_map_in_bound(lo, lo + 2.0),
        "mlm_inflate_map": lambda: m.inflate_map(pos[0]),
    }
    for name, call in calls.items():
        call()
        m.sync()
        e.sync()
        assert pool.used() == base, name


def test_refused_allocations_release_what_they_took_and_leave_no_error():
    pool = _PoolUsage()
    m = _cfg_a_map()
    lib, h = m._lib, m._h
    pts = _points(m, 1000)
    before = m.getOdd(pts)
    m.sync()
    base = pool.used()
    huge = 1 << 40  # the second temporary of each call asks for terabytes: refused before anything runs
    small = [np.zeros(64, dtype=np.uint8) for _ in range(5)]
    n = C.c_size_t()
    refused = {
        "mlm_export_map": lambda: lib.mlm_export_map(h, huge, *[a.ctypes.data for a in small], C.byref(n)),
        "mlm_last_frame_misses": lambda: lib.mlm_last_frame_misses(h, small[0].ctypes.data, huge, C.byref(n)),
        "mlm_export_cloud": lambda: lib.mlm_export_cloud(h, 0, small[0].ctypes.data, huge, C.byref(n)),
    }
    for name, call in refused.items():
        assert call() == MLM_ERR_CUDA, name
        m.sync()
        assert pool.used() == base, name
        assert m.getOdd(pts).tobytes() == before.tobytes(), name
