"""GPU: the candidate-view gain (mlm_view_gain, k_view_*) against the oracle's restatement (orc_view_gain) bit for bit on
the records, each map first checked against the oracle's; against mlm_cast_rays and getOccupancy without the oracle; on
crafted maps restored from checkpoint images, against the oracle and the Python restatement; a large batch, views at the
depth limit, the device variant, repeatability, errors and sharded ranks."""
import ctypes as C

import numpy as np
import pytest

from mlmapping_b200 import MLMap, config_cfg_a, scenes
from mlmapping_b200.capi import VIEW_GAIN_DTYPE, MlmError
from frontier_spec import decode_frontier
from parity_utils import assert_map_parity
from test_frontier_host import build_map, cfg_of, explore_cfg_a
from test_parity_gpu import _lidar_small_cfg
from test_view_host import FLAGS, crafted_cases, identity_cfg, spec_gain
from view_oracle import ViewOracle
from view_spec import candidates_around, sensor, view_cells, write_map_checkpoint

pytestmark = pytest.mark.gpu
LO_TOL = 1e-6


def sensor_of(kind, max_depth):
    if kind == "lidar":  # a synthetic 90 x 74 degree camera on the LiDAR map (T_bs = identity: optical axis body z)
        return sensor(fx=160.0, cx=159.5, cy=119.5, cols=320, rows=240, min_depth=0.2, max_depth=max_depth)
    return sensor(min_depth=0.1, max_depth=max_depth)


def fuel_views(gpu, cfg, seed, n_clusters=12, per_cluster=4):
    """candidates around the largest frontier clusters of mlm_frontier_clusters, looking at the centroids, and each
    view's box = its cluster's lo / hi"""
    rec = gpu.frontier_clusters()
    top = rec[np.argsort(-rec["n_cells"], kind="stable")[:n_clusters]]
    poses, of = candidates_around(top["centroid"], list(cfg.T_bs), seed, per_cluster)
    boxes = np.concatenate([top["lo"][of], top["hi"][of]], 1).astype(np.int32)
    return poses, boxes


@pytest.mark.parametrize("kind", ["cfg-a-14", "cfg-a-40", "lidar"])
def test_view_gain_equals_the_oracle(kind):
    cfg = cfg_of(kind)
    gpu, orc = MLMap(cfg), ViewOracle(cfg)
    build_map(kind, gpu)
    build_map(kind, orc)
    assert_map_parity(gpu, orc, LO_TOL, tag=kind)
    poses, boxes = fuel_views(gpu, cfg, seed=3)
    S = sensor_of(kind, 4.0 if kind == "lidar" else 2.5)
    launches = gpu.kernel_launch_count()
    for frontier, inflated in FLAGS:
        for b in (None, boxes):
            g = gpu.view_gain(poses, S, b, frontier, inflated)
            o = orc.view_gain(poses, S, b, frontier, inflated)
            assert g.tobytes() == o.tobytes(), (kind, frontier, inflated, b is None)
            assert gpu.view_gain(poses, S, b, frontier, inflated).tobytes() == g.tobytes()  # repeatable
            assert (g["status"] == 0).all() and g["n_target"].sum() > 0
    assert gpu.kernel_launch_count() > launches
    # the map is left as it was: later queries and the export still equal the oracle's
    rs = np.random.RandomState(5)
    ex = orc.export_map()
    lo, hi = ex["glb"].min(0) * cfg.subbox_n * cfg.subbox_d_xyz, (ex["glb"].max(0) + 1) * cfg.subbox_n * cfg.subbox_d_xyz
    pts = rs.uniform(lo, hi, (20000, 3))
    assert np.array_equal(gpu.getOccupancy(pts), orc.getOccupancy(pts))
    assert gpu.cast_rays(pts[:5000], pts[5000:10000]).tobytes() == orc.cast_rays(pts[:5000], pts[5000:10000]).tobytes()
    assert_map_parity(gpu, orc, LO_TOL, tag=kind + " after")


def test_view_gain_equals_cast_rays_and_get_occupancy():
    """without the oracle: frustum cells enumerated in numpy (view_spec.view_cells), targets by getOccupancy, visibility
    by cast_rays from the origin to each target centre: visible exactly when the stop cell is the target and every cell
    before it is free (n_free == |c - cell(o)|_1, plus 1 when the ray reaches a free end cell)"""
    kind = "cfg-a-40"
    cfg = cfg_of(kind)
    gpu = MLMap(cfg)
    build_map(kind, gpu)
    d = cfg.subbox_d_xyz
    poses, _ = fuel_views(gpu, cfg, seed=4, n_clusters=16, per_cluster=4)
    traj = np.array([scenes.corridor_trajectory_pose(k) for k in (30, 90, 150)])
    poses = np.concatenate([poses, traj])
    S = sensor_of(kind, 3.5)
    # the views that see the most (so that visible targets are checked too) and a few others
    order = np.argsort(-gpu.view_gain(poses, S)["n_visible"], kind="stable")
    poses = poses[np.concatenate([order[:8], order[-4:]])]
    got = gpu.view_gain(poses, S)
    fcells = {tuple(c) for c in decode_frontier(gpu.export_map(), cfg.subbox_n).tolist()}
    for i, pose in enumerate(poses):
        o, co, cells = view_cells(pose, S, d, list(cfg.T_bs))
        x = (cells + 0.5) * d
        occ = gpu.getOccupancy(x)
        for frontier in (False, True):
            tgt = cells[np.array([tuple(c) in fcells for c in cells.tolist()], bool)] if frontier else cells[occ == -1]
            rec = gpu.cast_rays(np.tile(np.array(o), (len(tgt), 1)), (tgt + 0.5) * d)
            l1 = np.abs(tgt - np.array(co)).sum(1)
            end_free = (rec["status"] == 1) & (gpu.getOccupancy((tgt + 0.5) * d) == 1)
            vis = (rec["cell"] == tgt).all(1) & (rec["n_free"] - end_free == l1)
            want = gpu.view_gain(pose[None], S, frontier=frontier)[0] if frontier else got[i]
            assert (want["n_target"], want["n_visible"]) == (len(tgt), int(vis.sum())), (i, frontier)
    assert got["n_visible"].sum() > 0


@pytest.fixture(scope="module")
def restore_to():
    """an exploration handle (T_bs = identity) with one frame behind it (a valid header); load(ex) restores a crafted map"""
    cfg = identity_cfg()
    gpu = MLMap(cfg)
    pose = [0.0, 0.0, 1.0, 0.5, -0.5, 0.5, -0.5]
    gpu.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=0), pose)
    template = gpu.checkpoint()

    def load(ex):
        gpu.restore(write_map_checkpoint(template, cfg, ex))
        return gpu

    return cfg, load


@pytest.mark.parametrize("name", ["wall_hole", "closed_room", "eight_subboxes", "eight_subboxes_boxed"])
def test_crafted_maps(restore_to, name):
    cfg, load = restore_to
    ex, poses, S, boxes = crafted_cases(cfg.subbox_n)[name]
    gpu = load(ex)
    orc = ViewOracle(cfg)
    orc.set_map(ex)
    for frontier, inflated in FLAGS:
        g = gpu.view_gain(poses, S, boxes, frontier, inflated)
        assert g.tobytes() == orc.view_gain(poses, S, boxes, frontier, inflated).tobytes(), (name, frontier, inflated)
        assert g.tobytes() == spec_gain(ex, cfg, poses, S, boxes, frontier, inflated).tobytes(), (name, frontier, inflated)


@pytest.fixture(scope="module")
def explored_30():
    """the CFG-A exploration map of 30 corridor frames, on the GPU and in the oracle"""
    cfg = explore_cfg_a()
    gpu, orc = MLMap(cfg), ViewOracle(cfg)
    for m in (gpu, orc):
        for k in range(30):
            pose = scenes.corridor_trajectory_pose(k * 5)
            m.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    assert_map_parity(gpu, orc, LO_TOL, tag="explore-30")
    return cfg, gpu, orc


def test_batch_of_4096_views_and_the_depth_limit(explored_30):
    cfg, gpu, orc = explored_30
    d = cfg.subbox_d_xyz
    rec = gpu.frontier_clusters()
    poses, _ = candidates_around(rec["centroid"], list(cfg.T_bs), seed=9, per_cluster=4096 // rec.size + 1)
    poses = poses[:4096]
    S = sensor_of("cfg-a", 5.0)
    rs = np.random.RandomState(2)
    sub = rs.choice(poses.shape[0], 12, replace=False)
    for frontier in (False, True):
        g = gpu.view_gain(poses, S, frontier=frontier)
        assert g.shape == (4096,) and (g["status"] == 0).all()
        assert g[sub].tobytes() == orc.view_gain(poses[sub], S, frontier=frontier).tobytes(), frontier
    lim = sensor_of("cfg-a", 256 * d)
    lim.fx = lim.fy = 400.0  # a far corner off axis by 0.8 * 25.6 m: within the limit
    g = gpu.view_gain(poses[sub[:2]], lim)
    assert g.tobytes() == orc.view_gain(poses[sub[:2]], lim).tobytes()
    assert g["n_target"].min() > 1_000_000
    over = sensor_of("cfg-a", np.nextafter(256 * d, np.inf))
    with pytest.raises(MlmError) as ei:
        gpu.view_gain(poses[:1], over)
    assert ei.value.code == 5


def test_device_variant_equals_host_variant(explored_30):
    cfg, gpu, _ = explored_30
    rec = gpu.frontier_clusters()
    poses, of = candidates_around(rec["centroid"], list(cfg.T_bs), seed=5, per_cluster=3)
    boxes = np.concatenate([rec["lo"][of], rec["hi"][of]], 1).astype(np.int32)
    S = sensor_of("cfg-a", 3.0)
    d_p, d_b = gpu.to_device(poses), gpu.to_device(boxes)
    d_o = gpu.device_alloc(16 * poses.shape[0])
    for b in (None, boxes):
        for frontier, inflated in FLAGS:
            gpu.view_gain_device(d_p, poses.shape[0], S, d_o, 0 if b is None else d_b, frontier, inflated)
            dev = gpu.to_host(d_o, poses.shape[0], VIEW_GAIN_DTYPE)
            assert dev.tobytes() == gpu.view_gain(poses, S, b, frontier, inflated).tobytes()
    for p in (d_p, d_b, d_o):
        gpu.device_free(p)


def test_errors_and_unsupported():
    cfg = explore_cfg_a()
    gpu = MLMap(cfg)
    lib, h = gpu._lib, gpu._h
    pose = np.array([[1.0, 0.0, 1.0, 1.0, 0.0, 0.0, 0.0]])
    out = np.zeros(1, dtype=VIEW_GAIN_DTYPE)
    S = sensor()
    assert lib.mlm_view_gain(h, pose.ctypes.data, 1, C.byref(S), None, 0, out.ctypes.data) == 0
    assert lib.mlm_view_gain(h, pose.ctypes.data, 0, C.byref(S), None, 0, out.ctypes.data) == 0
    assert lib.mlm_view_gain(h, None, 1, C.byref(S), None, 0, out.ctypes.data) == 1
    assert lib.mlm_view_gain(h, pose.ctypes.data, 1, None, None, 0, out.ctypes.data) == 1
    assert lib.mlm_view_gain(h, pose.ctypes.data, 1, C.byref(S), None, 0, None) == 1
    assert lib.mlm_view_gain(h, pose.ctypes.data, 1, C.byref(S), None, 4, out.ctypes.data) == 1
    for kw in (dict(fx=-1.0), dict(fy=0.0), dict(cx=float("nan")), dict(rows=0), dict(cols=-3), dict(min_depth=-1.0),
               dict(min_depth=2.0, max_depth=1.0), dict(max_depth=float("inf"))):
        assert lib.mlm_view_gain(h, pose.ctypes.data, 1, C.byref(sensor(**kw)), None, 0, out.ctypes.data) == 1, kw
    assert lib.mlm_view_gain(h, pose.ctypes.data, 1, C.byref(sensor(fx=10.0, max_depth=20.0)), None, 0,
                             out.ctypes.data) == 5
    plain = MLMap(config_cfg_a())
    with pytest.raises(MlmError) as ei:
        plain.view_gain(pose, S, frontier=True)
    assert ei.value.code == 6
    assert plain.view_gain(pose, S)["status"][0] == 0


def test_sharded_ranks_refuse():
    from mlmapping_b200.sharded import sharded_group_in_process
    ranks = sharded_group_in_process(_lidar_small_cfg(), 2)
    try:
        for r in ranks:
            with pytest.raises(MlmError) as ei:
                r.map.view_gain(np.array([[0.0, 0, 0, 1, 0, 0, 0]]), sensor())
            assert ei.value.code == 6
    finally:
        for r in ranks:
            r.close()
