"""GPU: the signed distance field (mlm_esdf_*, k_esdf_*) against the oracle's restatement of the spec (orc_esdf_*), bit
for bit on the exported grid and on distances and gradients, on both layers.  Each map is first checked against the
oracle's, so that a map mismatch is told apart from a field mismatch."""
import ctypes as C

import numpy as np
import pytest

from mlmapping_b200 import MLMap, config_cfg_a, scenes
from mlmapping_b200.capi import MlmError
from esdf_oracle import EsdfOracle
from esdf_spec import first_difference, query_points, same_bits
from parity_utils import assert_map_parity
from raycast_spec import OCCUPIED
from test_parity_gpu import _lidar_small_cfg

pytestmark = pytest.mark.gpu
LO_TOL = 1e-6


def _boxes(ex, cfg, occupied_cell):
    """the map's AABB padded by 1 m, a box reaching 5 m into unmapped space, an all-unknown box, one occupied cell"""
    n, d = cfg.subbox_n, cfg.subbox_d_xyz
    lo, hi = ex["glb"].min(0) * n * d, (ex["glb"].max(0) + 1) * n * d
    mid = (lo + hi) / 2
    far = lo - 50.0
    cell = (np.asarray(occupied_cell) + 0.5) * d
    return {"aabb": (lo - 1.0, hi + 1.0), "partly_unmapped": (mid, np.maximum(hi + 5.0, mid + 1.0)),
            "unknown": (far, far + 3.0), "one_cell": (cell, cell)}


def _an_occupied_cell(ex, n):
    rows, subs = np.nonzero((ex["occupancy"] == b"o") & (ex["collapsed"][:, None] == 0))
    sub = subs[0]
    return ex["glb"][rows[0]] * n + np.array([sub % n, (sub // n) % n, sub // (n * n)])


def _assert_field_matches(gpu, orc, cfg, n_query, seed, tag):
    """every box on both layers: export bit for bit, queries bit for bit, blocking cells = ray-blocking cells"""
    ex = orc.export_map()
    d = cfg.subbox_d_xyz
    out = {}
    for name, (bmin, bmax) in _boxes(ex, cfg, _an_occupied_cell(ex, cfg.subbox_n)).items():
        for inflated in (False, True):
            key = (tag, name, inflated)
            gpu.build_esdf(bmin, bmax, 2.0, inflated=inflated)
            orc.build_esdf(bmin, bmax, 2.0, inflated=inflated)
            g, glo = gpu.export_esdf()
            o, olo = orc.export_esdf()
            assert np.array_equal(glo, olo) and g.shape == o.shape, key
            assert same_bits(g, o), (key, first_difference(g, o))
            dims = np.array(g.shape[::-1])
            pts = query_points(glo.astype(np.int64), dims, d, n_query if name == "aabb" else 5000, seed)
            gd, gg = gpu.esdf_distance(pts)
            od, og = orc.esdf_distance(pts)
            assert same_bits(gd, od), (key, first_difference(gd, od))
            assert same_bits(gg, og), (key, first_difference(gg, og))
            # v <= 0 exactly where a zero-length ray at the cell centre stops at once, on the same layer
            zz, yy, xx = np.meshgrid(*[np.arange(k) for k in g.shape], indexing="ij")
            centres = (np.stack([xx, yy, zz], -1).reshape(-1, 3) + glo + 0.5) * d
            rec = gpu.cast_rays(centres, centres, inflated=inflated)
            assert np.array_equal(g.reshape(-1) <= 0, rec["status"] == OCCUPIED), key
            out[key] = (g, pts, gd, gg)
    return out


def test_esdf_cfg_a_trajectory_with_inflation():
    """CFG-A, 40 frames at stride 5, inflate_map; the device variants give the host variants' results"""
    cfg = config_cfg_a()
    gpu, orc = MLMap(cfg), EsdfOracle(cfg)
    for k in range(40):
        pose = scenes.corridor_trajectory_pose(k * 5)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    gpu.inflate_map(pose[:3])
    orc.inflate_map(pose[:3])
    assert_map_parity(gpu, orc, LO_TOL, tag="cfg-a")
    res = _assert_field_matches(gpu, orc, cfg, 200_000, seed=51, tag="cfg-a")
    g, pts, gd, gg = res[("cfg-a", "aabb", True)]
    assert (g <= 0).sum() > 1000 and (g == 2.0).sum() > 1000 and np.isnan(gd).sum() > 100
    # device variants against the host variants (the field of the last build: one_cell, inflated -> rebuild aabb)
    ex = orc.export_map()
    bmin, bmax = _boxes(ex, cfg, _an_occupied_cell(ex, cfg.subbox_n))["aabb"]
    gpu.build_esdf(bmin, bmax, 2.0, inflated=True)
    n = pts.shape[0]
    d_p, d_d, d_g = gpu.to_device(pts), gpu.device_alloc(8 * n), gpu.device_alloc(24 * n)
    gpu.esdf_distance_device(d_p, n, d_d, d_g)
    assert same_bits(gpu.to_host(d_d, (n,), np.float64), gd) and same_bits(gpu.to_host(d_g, (n, 3), np.float64), gg)
    gpu.esdf_distance_device(d_p, n, d_d)                          # without gradients
    assert same_bits(gpu.to_host(d_d, (n,), np.float64), gd)
    cells = g.size
    d_o = gpu.device_alloc(4 * cells)
    lo, dims = gpu.export_esdf_device(d_o, cells)
    assert np.array_equal(dims, g.shape[::-1]) and same_bits(gpu.to_host(d_o, g.shape, np.float32), g)
    with pytest.raises(MlmError) as ei:
        gpu.export_esdf_device(d_o, cells - 1)
    assert ei.value.code == 5
    for p in (d_p, d_d, d_g, d_o):
        gpu.device_free(p)


def test_esdf_through_collapsed_subboxes_in_exploration_mode():
    """the exploration-mode map (14 frames, collapsed subboxes)"""
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    gpu, orc = MLMap(cfg), EsdfOracle(cfg)
    for k in range(14):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    assert_map_parity(gpu, orc, LO_TOL, tag="explore")
    assert (orc.export_map()["collapsed"] == 1).sum() >= 10
    _assert_field_matches(gpu, orc, cfg, 100_000, seed=61, tag="explore")


def test_esdf_on_the_lidar_map():
    """the reduced LiDAR configuration (2 m subboxes)"""
    cfg = _lidar_small_cfg()
    gpu, orc = MLMap(cfg), EsdfOracle(cfg)
    for k in range(6):
        pose = scenes.lidar_loop_pose(k * 3)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512)
        gpu.integrate_points(pts, pose)
        orc.integrate_points(pts, pose)
    assert_map_parity(gpu, orc, LO_TOL, tag="lidar")
    _assert_field_matches(gpu, orc, cfg, 100_000, seed=71, tag="lidar")


def test_esdf_arguments_lifetime_and_rebuilds():
    cfg = config_cfg_a()
    gpu, orc = MLMap(cfg), EsdfOracle(cfg)
    d = cfg.subbox_d_xyz
    # query / export before any build
    with pytest.raises(MlmError) as ei:
        gpu.esdf_distance([[0.0, 0.0, 0.0]])
    assert ei.value.code == 1 and "mlm_esdf_build" in str(ei.value)
    with pytest.raises(MlmError) as ei:
        gpu.export_esdf()
    assert ei.value.code == 1
    lib, h = gpu._lib, gpu._h
    a, b = (C.c_double * 3)(0.0, 0.0, 0.0), (C.c_double * 3)(1.0, 1.0, 1.0)
    nan, inf = float("nan"), float("inf")
    assert lib.mlm_esdf_build(h, a, b, 1.0, 2) == 1                       # flags
    for md in (0.0, -1.0, nan, inf):                                       # max_dist
        assert lib.mlm_esdf_build(h, a, b, md, 0) == 1
    for bad in ((nan, 0, 0), (0, inf, 0), (0, 0, 2.0 ** 30 * d), (2.0, 0, 0)):   # corners; box_min > box_max
        assert lib.mlm_esdf_build(h, (C.c_double * 3)(*bad), b, 1.0, 0) == 1
    assert lib.mlm_esdf_build(h, None, b, 1.0, 0) == 1
    # 4097 cells on one axis; more than 2^28 cells
    x0 = 0.05
    assert lib.mlm_esdf_build(h, (C.c_double * 3)(x0, 0.05, 0.05), (C.c_double * 3)(x0 + 4096 * d, 0.05, 0.05), 1.0, 0) == 5
    assert lib.mlm_esdf_build(h, (C.c_double * 3)(x0, 0.05, 0.05), (C.c_double * 3)(x0 + 4095 * d, 0.05, 0.05), 1.0, 0) == 0
    big = 4095.5 * d                                                      # 4096 x 4096 x 21 cells
    assert lib.mlm_esdf_build(h, a, (C.c_double * 3)(big, big, 20.5 * d), 1.0, 0) == 5
    for k in range(10):
        pose = scenes.corridor_trajectory_pose(k * 5)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    c = pose[:3]
    # a rebuild with a smaller box, then a larger one (the buffers grow), each equal to the oracle
    for half in (3.0, 1.0, 6.0):
        gpu.build_esdf(c - half, c + half, 1.5)
        orc.build_esdf(c - half, c + half, 1.5)
        g, o = gpu.export_esdf()[0], orc.export_esdf()[0]
        assert same_bits(g, o), (half, first_difference(g, o))
    # the field is a snapshot: later frames leave it as it is until the next build
    before = gpu.export_esdf()[0]
    pts = c + np.random.RandomState(3).uniform(-5.0, 5.0, (5000, 3))
    d0, g0 = gpu.esdf_distance(pts)
    for k in range(10, 14):
        pose = scenes.corridor_trajectory_pose(k * 5)
        gpu.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    gpu.inflate_map(pose[:3])
    d1, g1 = gpu.esdf_distance(pts)
    assert same_bits(gpu.export_esdf()[0], before) and same_bits(d0, d1) and same_bits(g0, g1)
    # null pointers with n > 0, n == 0, size query and capacity of the host export
    out = (C.c_double * 3)()
    assert lib.mlm_esdf_distance(h, None, 1, out, None) == 1
    assert lib.mlm_esdf_distance(h, out, 1, None, None) == 1
    assert lib.mlm_esdf_distance(h, None, 0, None, None) == 0
    assert lib.mlm_esdf_distance_device(h, None, 1, out, None) == 1
    lo3, dims3 = (C.c_int32 * 3)(), (C.c_int32 * 3)()
    assert lib.mlm_esdf_export(h, None, 0, lo3, dims3) == 0 and tuple(dims3) == before.shape[::-1]
    small = (C.c_float * 4)()
    assert lib.mlm_esdf_export(h, small, 4, lo3, dims3) == 5
    assert lib.mlm_esdf_export(h, None, 0, None, dims3) == 1


@pytest.mark.parametrize("world", [1, 2])
def test_sharded_rank_refuses_esdf_unless_it_owns_the_whole_map(world):
    """a rank of a world-2 sharded map holds only its own subboxes: MLM_ERR_UNSUPPORTED; a world-1 shard answers"""
    from mlmapping_b200.sharded import sharded_group_in_process
    cfg = _lidar_small_cfg()
    ranks = sharded_group_in_process(cfg, world)
    try:
        for r in ranks:
            if world == 1:
                r.map.build_esdf([0.0, 0.0, 0.0], [4.0, 4.0, 2.0], 1.0)
                dist, _ = r.map.esdf_distance([[1.0, 1.0, 1.0]])
                assert abs(dist[0] - 1.0) < 1e-12                    # an empty map: max_dist everywhere
                continue
            with pytest.raises(MlmError) as ei:
                r.map.build_esdf([0.0, 0.0, 0.0], [4.0, 4.0, 2.0], 1.0)
            assert ei.value.code == 6
            with pytest.raises(MlmError) as ei:
                r.map.esdf_distance([[1.0, 1.0, 1.0]])
            assert ei.value.code == 6
    finally:
        for r in ranks:
            r.close()
