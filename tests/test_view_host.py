"""CPU: the C++ oracle's candidate-view gain (orc_view_gain) equals the Python restatement of the spec
(tests/view_spec.py) record for record, on the first frames of the CFG-A exploration map and on crafted maps, for both
target kinds, with and without MLM_VIEW_INFLATED and boxes; the borders of the frustum and degenerate views; argument
errors; and the C ABI rejects bad arguments without a device."""
import ctypes as C

import numpy as np
import pytest

import mlmapping_b200 as mlm
from mlmapping_b200 import config_cfg_a, scenes
from mlmapping_b200.capi import VIEW_GAIN_DTYPE, VIEW_INVALID, MlmError
from frontier_spec import clusters, decode_frontier
from raycast_spec import MapStates
from test_frontier_host import explore_cfg_a
from view_oracle import ViewOracle
from view_spec import candidates_around, crafted_map, frontier_set, gain, sensor, view_cells

FLAGS = [(False, False), (False, True), (True, False), (True, True)]  # (frontier, inflated)


def spec_gain(ex, cfg, poses, S, boxes=None, frontier=False, inflated=False):
    n, d = cfg.subbox_n, cfg.subbox_d_xyz
    return gain(MapStates(ex, n), frontier_set(ex, n), poses, S, d, list(cfg.T_bs), boxes, frontier, inflated)


def corridor_views(cfg, ex, seed, per_cluster=3, n_clusters=4):
    """candidates around the largest frontier clusters, plus poses of the corridor trajectory (views out of free space)"""
    d = cfg.subbox_d_xyz
    rec = clusters(decode_frontier(ex, cfg.subbox_n), d)[0]
    top = rec[np.argsort(-rec["n_cells"], kind="stable")[:n_clusters]]
    poses, of = candidates_around(top["centroid"], list(cfg.T_bs), seed, per_cluster)
    traj = np.array([scenes.corridor_trajectory_pose(k) for k in (0, 7, 15, 22)], dtype=np.float64)
    boxes = np.concatenate([np.concatenate([top["lo"][of], top["hi"][of]], 1),
                            np.tile(np.array([[0, -15, 0, 60, 15, 12]]), (traj.shape[0], 1))]).astype(np.int32)
    return np.concatenate([poses, traj]), boxes


@pytest.fixture(scope="module")
def corridor():
    cfg = explore_cfg_a()
    orc = ViewOracle(cfg)
    for k in range(4):
        pose = scenes.corridor_trajectory_pose(k * 10)
        orc.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    return cfg, orc, orc.export_map()


@pytest.mark.parametrize("frontier,inflated", FLAGS)
def test_oracle_equals_spec_on_the_corridor_map(corridor, frontier, inflated):
    cfg, orc, ex = corridor
    poses, boxes = corridor_views(cfg, ex, seed=1)
    for S in (sensor(max_depth=1.0), sensor(min_depth=0.3, max_depth=1.5, cols=320, rows=240, cx=160.0, cy=120.0,
                                            fx=200.0)):
        for b in (None, boxes):
            got = orc.view_gain(poses, S, b, frontier, inflated)
            want = spec_gain(ex, cfg, poses, S, b, frontier, inflated)
            assert got.tobytes() == want.tobytes(), (S.max_depth, b is None, got, want)
            assert (got["status"] == 0).all() and got["n_target"].sum() > 0
    if not frontier:
        assert got["n_visible"].sum() > 0  # views from the trajectory see unknown cells past the free corridor


# ---- crafted maps (shared with the GPU tests, which restore them through checkpoints) -------------------------------
def identity_cfg():
    cfg = explore_cfg_a()
    cfg.T_bs[:] = [0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0]
    return cfg


def box_cells(lo, hi):
    g = np.indices(tuple(np.array(hi) - np.array(lo) + 1)).reshape(3, -1).T + np.array(lo)
    return [tuple(c) for c in g.tolist()]


def crafted_cases(n):
    """name -> (export-like map, poses, sensor, boxes or None); all with T_bs = identity (sensor axis = body z)"""
    look_z = lambda x, y, z: [x, y, z, 1.0, 0.0, 0.0, 0.0]
    S = sensor(fx=40.0, cx=31.5, cy=23.5, cols=64, rows=48, min_depth=0.0, max_depth=2.0)
    out = {}
    # a wall at z = 10 with a one-cell hole at (0, 0), free space in front of it, unknown behind
    st = {c: b"f" for c in box_cells((-8, -8, 0), (8, 8, 9))}
    st.update({c: b"o" for c in box_cells((-8, -8, 10), (8, 8, 10))})
    st[(0, 0, 10)] = b"f"
    out["wall_hole"] = (crafted_map(st, n, frontier=[(0, 0, 11), (3, 3, 11)]), [look_z(0.05, 0.05, 0.05)], S, None)
    # a closed free room: the cells beyond its occupied walls are unknown and none is visible
    st = {c: b"o" for c in box_cells((-6, -6, -2), (6, 6, 14))}
    st.update({c: b"f" for c in box_cells((-5, -5, -1), (5, 5, 13))})
    out["closed_room"] = (crafted_map(st, n), [look_z(0.05, 0.05, 0.05), look_z(-0.23, 0.17, 0.31)], S, None)
    # a view whose frustum spans the 8 subboxes around the origin, inflation on a free cell in the way, collapsed
    # subboxes (a free one and an occupied one), negative coordinates
    st = {c: b"f" for c in box_cells((-n, -n, -n), (n - 1, n - 1, n - 1))}
    col = {(-2, -1, 0): b"f", (1, 1, 1): b"o", (-1, -2, 1): b"f"}
    fr = [(-3, -4, 5), (4, 4, 8), (-12, -5, 9)]
    m = crafted_map(st, n, inflated=[(0, 0, 3), (-1, -1, 2)], frontier=fr, collapsed=col)
    poses = [look_z(-0.01, -0.01, -0.35), look_z(-1.15, -0.72, -0.5), [-0.4, -0.3, 0.2, 0.9, 0.1, -0.3, 0.2]]
    out["eight_subboxes"] = (m, poses, S, None)
    out["eight_subboxes_boxed"] = (m, poses, S, np.array([[-5, -5, 0, 4, 4, 9]] * 3, dtype=np.int32))
    return out


@pytest.mark.parametrize("name", ["wall_hole", "closed_room", "eight_subboxes", "eight_subboxes_boxed"])
def test_oracle_equals_spec_on_crafted_maps(name):
    cfg = identity_cfg()
    ex, poses, S, boxes = crafted_cases(cfg.subbox_n)[name]
    orc = ViewOracle(cfg)
    orc.set_map(ex)
    for frontier, inflated in FLAGS:
        got = orc.view_gain(poses, S, boxes, frontier, inflated)
        want = spec_gain(ex, cfg, poses, S, boxes, frontier, inflated)
        assert got.tobytes() == want.tobytes(), (name, frontier, inflated, got, want)
    plain = orc.view_gain(poses, S, boxes)
    if name == "wall_hole":  # through the hole: the line of cells behind it, and nothing else behind the wall
        assert 0 < plain["n_visible"][0] < plain["n_target"][0]
        assert orc.view_gain(poses, S, boxes, frontier=True)["n_visible"][0] == 1  # (0, 0, 11) but not (3, 3, 11)
    if name == "closed_room":
        assert (plain["n_target"] > 0).all() and (plain["n_visible"] == 0).all()
    if name == "eight_subboxes":
        assert orc.view_gain(poses, S, boxes, inflated=True)["n_visible"][0] < plain["n_visible"][0]


def test_frustum_borders_are_exact():
    """a cell centre exactly on u = -0.5 is in view, one on u = cols - 0.5 is not; p_z exactly min_depth or max_depth is
    in view (T_bs and the body rotation are the identity, so p = x - o exactly)"""
    cfg = identity_cfg()
    d = cfg.subbox_d_xyz
    S = sensor(fx=100.0, cx=99.5, cy=99.5, cols=200, rows=200, min_depth=(2 + 0.5) * d, max_depth=(7 + 0.5) * d)
    pose = [0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0]
    _, co, cells = view_cells(pose, S, d, list(cfg.T_bs))
    got = set(map(tuple, cells.tolist()))
    for cz in (2, 5, 7):
        assert (-cz - 1, 0, cz) in got and (cz, 0, cz) not in got        # u = -0.5 in, u = cols - 0.5 out
        assert (0, -cz - 1, cz) in got and (0, cz, cz) not in got
    assert min(c[2] for c in got) == 2 and max(c[2] for c in got) == 7  # both depth limits included
    orc = ViewOracle(cfg)
    orc.set_map(crafted_map({c: b"f" for c in box_cells((-9, -9, -1), (9, 9, 5))}, cfg.subbox_n))
    ex = orc.export_map()
    for flags in FLAGS:
        a = orc.view_gain([pose], S, None, *flags)
        assert a.tobytes() == spec_gain(ex, cfg, [pose], S, None, *flags).tobytes(), flags
    assert orc.view_gain([pose], S)["n_target"][0] == sum(1 for c in got if c[2] > 5)


def test_degenerate_views():
    cfg = explore_cfg_a()
    d = cfg.subbox_d_xyz
    orc = ViewOracle(cfg)
    occ = (3, 4, 5)
    orc.set_map(crafted_map({occ: b"o", (3, 4, 6): b"f"}, cfg.subbox_n))
    ex = orc.export_map()
    S = sensor(max_depth=1.0)
    nan, big = float("nan"), 2.0 ** 30 * d
    # the origin is T_wb.t + R_wb * T_bs.t, T_bs.t = (0.12, 0, 0): body poses that put it in the occupied cell
    in_occ = [(occ[0] + 0.5) * d - 0.12, (occ[1] + 0.5) * d, (occ[2] + 0.5) * d, 1.0, 0.0, 0.0, 0.0]
    poses = [[nan, 0, 0, 1, 0, 0, 0], [0, 0, 0, 0, 0, 0, 0], [0, 0, 0, 1, float("inf"), 0, 0], [big, 0, 0, 1, 0, 0, 0],
             [0, 0, 0, 1e200, 1e200, 0, 0], in_occ, [0.3, 0.4, 0.5, 1, 0, 0, 0]]
    boxes = np.array([[0, 0, 0, 5, 5, 5]] * 6 + [[0, 3, 0, 5, 2, 5]], dtype=np.int32)  # the last: lo > hi in y
    for b in (None, boxes):
        got = orc.view_gain(poses, S, b)
        assert got.tobytes() == spec_gain(ex, cfg, poses, S, b).tobytes()
        assert (got["status"][:5] == VIEW_INVALID).all() and (got["n_target"][:5] == 0).all()
        assert got["status"][5] == 0 and got["n_target"][5] > 0 and got["n_visible"][5] == 0  # occupied origin
    assert orc.view_gain(poses, S, boxes)["status"][6] == VIEW_INVALID
    assert orc.view_gain(poses, S)["status"][6] == 0


def test_argument_errors_of_the_oracle():
    cfg = config_cfg_a()
    orc = ViewOracle(cfg)
    pose = [[0, 0, 0, 1, 0, 0, 0]]
    lim = 256 * cfg.subbox_d_xyz
    bad = [dict(fx=0.0), dict(fx=float("nan")), dict(cols=0), dict(min_depth=-0.1), dict(min_depth=1.0, max_depth=1.0),
           dict(max_depth=float("inf"))]
    for kw in bad:
        with pytest.raises(MlmError) as ei:
            orc.view_gain(pose, sensor(**kw))
        assert ei.value.code == 1, kw
    assert orc.view_gain(pose, sensor(max_depth=lim))["status"][0] == 0
    for kw in (dict(max_depth=np.nextafter(lim, np.inf)), dict(max_depth=lim * 0.9, fx=100.0)):
        with pytest.raises(MlmError) as ei:
            orc.view_gain(pose, sensor(**kw))
        assert ei.value.code == 5, kw
    with pytest.raises(MlmError) as ei:
        orc.view_gain(pose, sensor(), frontier=True)  # a handle without the exploration mode
    assert ei.value.code == 6


def test_view_abi_rejects_bad_arguments_without_a_device():
    if not mlm.library_path().exists():
        mlm.build_library()
    lib = mlm.load_library()
    assert lib.mlm_sizeof_view_gain() == 16 == VIEW_GAIN_DTYPE.itemsize
    pose = (C.c_double * 7)(0, 0, 0, 1, 0, 0, 0)
    out = np.zeros(1, dtype=VIEW_GAIN_DTYPE)
    S = sensor()
    for fn in (lib.mlm_view_gain, lib.mlm_view_gain_device):
        assert fn(None, pose, 1, C.byref(S), None, 0, out.ctypes.data) == 1
        assert fn(None, None, 0, None, None, 0, None) == 1
