"""CPU: the restatement (oracle/mlmap_oracle.hpp) against the reference's OWN sources compiled into
oracle/_ref/libmlmap_ref.so (oracle/ref_build/Makefile: /root/reference src/map_awareness.cpp, src/map_local.cpp,
src/mlmap.cpp, src/rviz_vis.cpp, include/*.h, vendored Sophus, built where they lie with g++ -std=c++17 -O3).
Same seeded inputs into both; everything the reference exposes must be identical bit for bit: the hit map in its
iteration order with its probabilities, the miss set in ITS iteration order, the counters, the whole local map, the
queries, box fill, inflation, frontiers, collapsed subboxes, the published clouds and the forwarded pose.
Every test first holds the restatement (and the reference build, where it is available) to the stored outputs in
tests/golden/reference_pin.json (make_golden_pin.py: counters and digests of everything compared below, same inputs), so
the comparisons hold where the reference's own build is not available; the live comparisons follow where it is
(oracle/_ref prebuilt, or the sources at MLMAPPING_REFERENCE, else /root/reference)."""
import ctypes as C
import json
from pathlib import Path

import numpy as np
import pytest

from mlmapping_b200 import config_cfg_a, config_cfg_b, config_cfg_c, scenes
from oracle_binding import Oracle, _d7, load_oracle, load_reference, reference_available

PIN = json.loads((Path(__file__).parent / "golden" / "reference_pin.json").read_text())["cases"]


def _pinned(name):
    """the restatement, and the reference build where it is available, against the stored outputs; True where the live
    comparison can follow"""
    from golden.make_golden_pin import run_case
    assert run_case(name) == PIN[name], ("restatement differs from the stored reference outputs", name)
    if not reference_available():
        return False
    assert run_case(name, impl="reference") == PIN[name], ("reference build differs from the stored outputs", name)
    return True


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8) if a.dtype.kind in "fS" else a


def assert_same_frame(p, r, tag):
    sp, sr = p.frame_stats(), r.frame_stats()
    for f in ("n_points", "n_inside", "n_cast", "n_hit_cells", "n_miss_cells", "n_touched_voxels", "hit_bucket_count",
              "ram_expand_cnt", "obs_cnt"):
        assert getattr(sp, f) == getattr(sr, f), (tag, f, getattr(sp, f), getattr(sr, f))
    kp, pp = p.last_frame_hits()
    kr, pr = r.last_frame_hits()
    assert np.array_equal(kp, kr), (tag, "hit keys / iteration order")
    assert np.array_equal(pp.view(np.uint32), pr.view(np.uint32)), (tag, "hit probabilities")
    assert np.array_equal(p.last_frame_misses(sort=False), r.last_frame_misses(sort=False)), (tag, "miss set / iteration order")


def assert_same_map(p, r, tag):
    mp, mr = p.export_map(), r.export_map()
    for k in mp:
        assert np.array_equal(_bits(mp[k]), _bits(mr[k])), (tag, k)
    return mp




def test_golden_vectors_come_from_the_reference_and_the_restatement_reproduces_them():
    from golden.make_golden import CASES, run_case
    meta = json.loads((Path(__file__).parent / "golden" / "golden.json").read_text())
    assert "UNMODIFIED reference sources" in meta["provenance"]
    for name in CASES:
        want = meta["cases"][name]
        if reference_available():
            assert run_case(name, impl="reference") == want, ("reference build no longer reproduces its golden vectors", name)
        assert run_case(name, impl="port") == want, ("restatement differs from the reference", name)


def test_depth_trajectory_with_rolled_poses_queries_and_clouds():
    if not _pinned("depth_trajectory"):
        return
    from golden.make_golden_pin import rolled as _rolled
    cfg = config_cfg_a()
    cfg.inflate_n, cfg.inflate_global_n = 2, 2
    p, r = Oracle(cfg), Oracle(cfg, impl="reference")
    for k in range(6):
        pose = _rolled(scenes.corridor_trajectory_pose(35 * k), k)
        img = scenes.corridor_depth_frame(cfg, pose, rows=240, cols=320, frame_idx=k)
        p.integrate_depth(img, pose), r.integrate_depth(img, pose)
        assert_same_frame(p, r, f"frame{k}")
    m = assert_same_map(p, r, "trajectory")
    lo, hi = m["glb"].min(0) * 1.0, (m["glb"].max(0) + 1) * 1.0
    pos = scenes.query_positions(30000, lo, hi, seed=5, inflate=2.0)
    assert np.array_equal(p.getOccupancy(pos), r.getOccupancy(pos))
    assert np.array_equal(p.getOdd(pos).view(np.uint32), r.getOdd(pos).view(np.uint32))
    assert np.array_equal(p.getOddGrad(pos[:8000]).view(np.uint64), r.getOddGrad(pos[:8000]).view(np.uint64))
    assert np.array_equal(p.getOccupancy(pos[:3000], inflate=0.2), r.getOccupancy(pos[:3000], inflate=0.2))
    for o in (p, r):
        o.inflate_map(pose[:3])
        o.setFree_map_in_bound([pose[0] + 0.5, -0.4, 0.8], [pose[0] + 1.5, 0.4, 1.6])
    assert_same_map(p, r, "after inflate + setFree")
    assert np.array_equal(p.getInflateOccupancy(pos[:5000]), r.getInflateOccupancy(pos[:5000]))
    # clouds: the reference's own publishers (rviz_vis::pub_global_local_map, mlmap::visualize_odds) captured as messages;
    # both iterate the same unordered_map, so even the point ORDER agrees
    for kind in (0, 1):
        assert np.array_equal(p.export_cloud(kind).view(np.uint32), r.export_cloud(kind).view(np.uint32)), kind
    assert r.export_cloud(0).shape[0] > 100
    sp, sr = p.export_odds_slice(1.25), r.export_odds_slice(1.25)
    assert sr.shape[0] > 100 and np.array_equal(sp.view(np.uint32), sr.view(np.uint32))


def test_exploration_mode_frontiers_and_release():
    if not _pinned("exploration"):
        return
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    p, r = Oracle(cfg), Oracle(cfg, impl="reference")
    released = 0
    for k in range(10):
        pose = scenes.corridor_trajectory_pose(12 * k)
        img = scenes.corridor_depth_frame(cfg, pose, rows=240, cols=320, frame_idx=k)
        p.integrate_depth(img, pose), r.integrate_depth(img, pose)
        assert_same_frame(p, r, f"explore{k}")
        assert p.lib.orc_released_last(p.h) == r.lib.orc_released_last(r.h)
        released += r.lib.orc_released_last(r.h)
    m = assert_same_map(p, r, "explore")
    assert np.unpackbits(m["frontier"]).sum() > 100
    assert np.array_equal(p.export_cloud(2).view(np.uint32), r.export_cloud(2).view(np.uint32))
    assert r.export_cloud(2).shape[0] == int(np.unpackbits(m["frontier"]).sum())


def test_lidar_points_and_the_large_configs():
    if not _pinned("lidar_and_cfg_b"):
        return
    cfg = config_cfg_c()
    cfg.am_n_rho, cfg.am_n_z_below, cfg.am_n_z_over = 120, 30, 30
    p, r = Oracle(cfg), Oracle(cfg, impl="reference")
    for k in range(2):
        pose = scenes.lidar_loop_pose(5 * k)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512)
        p.integrate_points(pts, pose), r.integrate_points(pts, pose)
        assert_same_frame(p, r, f"lidar{k}")
    assert_same_map(p, r, "lidar")
    cfg = config_cfg_b()  # 0.05 m cells, n_Rho 180: one reduced-size frame
    p, r = Oracle(cfg), Oracle(cfg, impl="reference")
    pose = scenes.corridor_trajectory_pose(3, step=0.1)
    img = scenes.corridor_depth_frame(cfg, pose, rows=192, cols=256, frame_idx=3, length=200.0)
    p.integrate_depth(img, pose), r.integrate_depth(img, pose)
    assert_same_frame(p, r, "cfg_b")
    assert_same_map(p, r, "cfg_b")


def test_sampled_projection_is_the_references_own_project_depth():
    """mlmapping_sample_cnt > 0: here the reference's own mlmap::project_depth (src/mlmap.cpp:311-349) runs on its cv::Mat"""
    if not _pinned("sampled_projection"):
        return
    cfg = config_cfg_a()
    cfg.sample_cnt = 400
    libc = C.CDLL("libc.so.6")
    pose = scenes.corridor_trajectory_pose(7)
    img = scenes.corridor_depth_frame(cfg, pose, frame_idx=7)
    outs = []
    for impl in ("port", "reference"):
        libc.srand(1)
        o = Oracle(cfg, impl=impl)
        for _ in range(3):
            o.integrate_depth(img, pose)
        outs.append((o.points().copy(), o))
    assert outs[0][0].shape[0] > 300 and np.array_equal(outs[0][0].view(np.uint64), outs[1][0].view(np.uint64))
    assert_same_frame(outs[0][1], outs[1][1], "sampled")
    assert_same_map(outs[0][1], outs[1][1], "sampled")


def test_prologue_transform_and_pose_forwarding_bit_for_bit():
    """T_ls = T_wa^-1 * (T_wb * T_bs), T_ls * p and the callback's pose forwarding: restatement == reference build ==
    the product's host code (mlm_compensate_pose), on general (rolled, pitched, unnormalised) quaternions"""
    from mlmapping_b200 import compensate_pose
    from golden.make_golden_pin import d, prologue_inputs
    _, fwd = prologue_inputs()
    assert d(np.array([compensate_pose(*f) for f in fwd])) == PIN["prologue"]["compensate_pose"]
    if not _pinned("prologue"):
        return
    a, b = load_oracle(), load_reference()
    rng = np.random.default_rng(0)
    for i in range(1500):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        if i % 3 == 0:
            q = q * rng.uniform(0.5, 2)
        Twb = np.r_[rng.uniform(-50, 50, 3), q]
        q2 = rng.normal(size=4)
        Tbs = np.r_[rng.uniform(-1, 1, 3), q2 / np.linalg.norm(q2)] if i % 2 else np.r_[0.12, 0, 0, 0.5, -0.5, 0.5, -0.5]
        oa, ob = (C.c_double * 7)(), (C.c_double * 7)()
        a.orc_T_ls(_d7(Twb), _d7(Tbs), oa), b.orc_T_ls(_d7(Twb), _d7(Tbs), ob)
        assert list(oa) == list(ob), i
        pt = rng.uniform(-10, 10, 3)
        pa, pb = (C.c_double * 3)(), (C.c_double * 3)()
        a.orc_transform_point(_d7(Twb), _d7(Tbs), _d7(pt), pa), b.orc_transform_point(_d7(Twb), _d7(Tbs), _d7(pt), pb)
        assert list(pa) == list(pb), i
    for i in range(300):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        pos, lv, av = rng.uniform(-5, 5, 3), rng.uniform(-2, 2, 3), rng.uniform(-1, 1, 3)
        go, gi, lat = rng.uniform(0, 0.05), rng.uniform(0, 0.05), rng.uniform(0, 0.01)
        oa, ob = (C.c_double * 7)(), (C.c_double * 7)()
        a.orc_compensate_pose(_d7(pos), _d7(q), _d7(lv), _d7(av), go, gi, lat, oa)
        b.orc_compensate_pose(_d7(pos), _d7(q), _d7(lv), _d7(av), go, gi, lat, ob)
        assert list(oa) == list(ob), i
        assert list(compensate_pose(pos, q, lv, av, go, gi, lat)) == list(ob), i


def test_get_odd_by_index_overload():
    """getOdd(const Vec3I&, size_t) (mlmap.h:128,227-235) of the reference on lattice indices"""
    if not _pinned("odd_by_index"):
        return
    cfg = config_cfg_a()
    r = Oracle(cfg, impl="reference")
    pose = scenes.corridor_trajectory_pose(0)
    r.integrate_depth(scenes.corridor_depth_frame(cfg, pose, rows=120, cols=160), pose)
    m = r.export_map()
    rs = np.random.RandomState(3)
    sel = rs.randint(0, m["glb"].shape[0], 2000)
    sub = rs.randint(0, 1000, 2000).astype(np.int32)
    glb = np.ascontiguousarray(m["glb"][sel].astype(np.int32))
    out = np.empty(2000, dtype=np.float32)
    r.lib.orc_get_odd_at(r.h, glb.ctypes.data, sub.ctypes.data, 2000, out.ctypes.data)
    lo = m["log_odds"][sel, sub].astype(np.float64)
    want = (np.power(10.0, lo) / (1 + np.power(10.0, lo))).astype(np.float32)
    assert np.abs(out.astype(np.float64) - want).max() <= 1.2e-7
