"""GPU: mlm_cast_rays (k_cast_rays) against the oracle's restatement of the spec (orc_cast_rays), bit for bit on every
record field, on both layers.  Each map is first checked against the oracle's, so that a map mismatch is told apart from
a ray mismatch."""
import ctypes as C

import numpy as np
import pytest

from mlmapping_b200 import MLMap, capi, config_cfg_a, scenes
from mlmapping_b200.capi import MlmError
from ray_oracle import RayOracle
from parity_utils import assert_map_parity
from raycast_spec import FREE, OCCUPIED, edge_segments, first_difference, random_segments
from test_parity_gpu import _lidar_small_cfg

pytestmark = pytest.mark.gpu
LO_TOL = 1e-6


def _assert_rays_match(gpu, orc, f, t, tag):
    out = {}
    for inflated in (False, True):
        g, o = gpu.cast_rays(f, t, inflated=inflated), orc.cast_rays(f, t, inflated=inflated)
        assert first_difference(g, o) is None, (tag, inflated, first_difference(g, o))
        out[inflated] = g
    return out


def _segments(orc, cfg, n_random, seed, max_len):
    ex = orc.export_map()
    n, d = cfg.subbox_n, cfg.subbox_d_xyz
    f1, t1 = random_segments(n_random, ex["glb"].min(0) * n * d, (ex["glb"].max(0) + 1) * n * d, seed=seed, max_len=max_len)
    f2, t2 = edge_segments(ex, n, d, seed=seed + 7, n_each=500)
    return ex, np.ascontiguousarray(np.concatenate([f1, f2])), np.ascontiguousarray(np.concatenate([t1, t2]))


def test_rays_cfg_a_trajectory_with_inflation():
    """CFG-A, 40 frames at stride 5, inflate_map: 200 k segments of 0-8 m plus the edge cases, both layers; the device
    variant gives the host variant's records; n == 0 and bad arguments"""
    cfg = config_cfg_a()
    gpu, orc = MLMap(cfg), RayOracle(cfg)
    for k in range(40):
        pose = scenes.corridor_trajectory_pose(k * 5)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    gpu.inflate_map(pose[:3])
    orc.inflate_map(pose[:3])
    assert_map_parity(gpu, orc, LO_TOL, tag="cfg-a")
    ex, f, t = _segments(orc, cfg, 200_000, seed=21, max_len=8.0)
    # one segment of exactly 2^20 cells: the longest valid walk
    d = cfg.subbox_d_xyz
    f = np.concatenate([f, [[0.05, 0.05, 0.05]]])
    t = np.concatenate([t, [[0.05 + 2 ** 20 * d, 0.05, 0.05]]])
    recs = _assert_rays_match(gpu, orc, f, t, "cfg-a")
    st = recs[False]["status"]
    assert (st == FREE).sum() > 20_000 and (st == OCCUPIED).sum() > 20_000 and (st == capi.RAY_INVALID).sum() >= 13
    assert recs[False]["n_unknown"][-1] == 2 ** 20 + 1 or recs[False]["status"][-1] == OCCUPIED
    assert (recs[True]["status"] == OCCUPIED).sum() > (st == OCCUPIED).sum()
    # device variant, the same records
    n = f.shape[0]
    d_f, d_t, d_o = gpu.to_device(f), gpu.to_device(t), gpu.device_alloc(32 * n)
    for inflated in (False, True):
        gpu.cast_rays_device(d_f, d_t, n, d_o, inflated=inflated)
        dev = gpu.to_host(d_o, (n,), capi.RAY_HIT_DTYPE)
        assert first_difference(dev, recs[inflated]) is None
    # n == 0 on both variants; bad flags and null pointers with n > 0
    assert gpu.cast_rays(np.zeros((0, 3)), np.zeros((0, 3))).shape == (0,)
    gpu.cast_rays_device(0, 0, 0, 0)
    lib, h = gpu._lib, gpu._h
    assert lib.mlm_cast_rays_device(h, d_f, d_t, n, 2, d_o) == 1
    assert lib.mlm_cast_rays_device(h, None, d_t, 1, 0, d_o) == 1
    assert lib.mlm_cast_rays_device(h, d_f, d_t, 1, 0, None) == 1
    out = (capi.RayHit * 1)()
    p = (C.c_double * 3)(1.0, 0.0, 1.0)
    assert lib.mlm_cast_rays(h, p, None, 1, 0, out) == 1
    assert lib.mlm_cast_rays(h, p, p, 1, -1, out) == 1
    for ptr in (d_f, d_t, d_o):
        gpu.device_free(ptr)


def test_rays_through_collapsed_subboxes_in_exploration_mode():
    """the exploration-mode map of test_exploration_frontiers_and_memory_release (14 frames, collapsed subboxes)"""
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    gpu, orc = MLMap(cfg), RayOracle(cfg)
    for k in range(14):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    assert_map_parity(gpu, orc, LO_TOL, tag="explore")
    ex, f, t = _segments(orc, cfg, 100_000, seed=31, max_len=8.0)
    # segments between centres of collapsed subboxes and random points nearby: they cross collapsed subboxes
    col = ex["glb"][ex["collapsed"] == 1]
    assert col.shape[0] >= 10
    rs = np.random.RandomState(32)
    g = (col[rs.randint(0, col.shape[0], 20_000)] + rs.uniform(0.0, 1.0, (20_000, 3))) * cfg.subbox_n * cfg.subbox_d_xyz
    f = np.ascontiguousarray(np.concatenate([f, g]))
    t = np.ascontiguousarray(np.concatenate([t, g + rs.uniform(-2.0, 2.0, g.shape)]))
    _assert_rays_match(gpu, orc, f, t, "explore")


def test_view_rays_on_the_lidar_map():
    """the reduced LiDAR configuration (2 m subboxes): view rays from a scan pose out to 24 m"""
    cfg = _lidar_small_cfg()
    gpu, orc = MLMap(cfg), RayOracle(cfg)
    for k in range(6):
        pose = scenes.lidar_loop_pose(k * 3)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512)
        gpu.integrate_points(pts, pose)
        orc.integrate_points(pts, pose)
    assert_map_parity(gpu, orc, LO_TOL, tag="lidar")
    el = np.deg2rad(np.linspace(-30.0, 30.0, 64))
    az = np.linspace(0.0, 2 * np.pi, 1024, endpoint=False)
    ee, aa = np.meshgrid(el, az, indexing="ij")
    dirs = np.stack([np.cos(ee) * np.cos(aa), np.cos(ee) * np.sin(aa), np.sin(ee)], -1).reshape(-1, 3)
    o = np.broadcast_to(pose[:3], dirs.shape)
    f = np.ascontiguousarray(np.concatenate([o, o + 0.01 * dirs]))
    t = np.ascontiguousarray(np.concatenate([o + 24.0 * dirs, o + 24.0 * dirs]))
    ex, f2, t2 = _segments(orc, cfg, 50_000, seed=41, max_len=24.0)
    recs = _assert_rays_match(gpu, orc, np.concatenate([f, f2]), np.concatenate([t, t2]), "lidar")
    st = recs[False]["status"][:f.shape[0]]
    assert (st == OCCUPIED).sum() > 1000 and (st == FREE).sum() > 100


@pytest.mark.parametrize("world", [1, 2])
def test_sharded_rank_refuses_rays_unless_it_owns_the_whole_map(world):
    """a rank of a world-2 sharded map holds only its own subboxes: MLM_ERR_UNSUPPORTED; a world-1 shard answers"""
    from mlmapping_b200.sharded import sharded_group_in_process
    cfg = _lidar_small_cfg()
    ranks = sharded_group_in_process(cfg, world)
    f, t = np.array([[0.0, 0.0, 1.0]]), np.array([[5.0, 1.0, 1.0]])
    try:
        for r in ranks:
            if world == 1:
                assert r.map.cast_rays(f, t)["status"][0] == FREE
                continue
            with pytest.raises(MlmError) as ei:
                r.map.cast_rays(f, t)
            assert ei.value.code == 6
            d_f, d_o = r.map.to_device(f), r.map.device_alloc(32)
            assert r.map._lib.mlm_cast_rays_device(r.map._h, d_f, d_f, 1, 0, d_o) == 6
            r.map.device_free(d_f)
            r.map.device_free(d_o)
    finally:
        for r in ranks:
            r.close()
