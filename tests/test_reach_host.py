"""CPU: the C++ oracle's reachability field (orc_reach_*) equals the written spec (tests/reach_spec.py, scipy's Dijkstra
over the vectorised move graph) on random class grids under every flag combination, gives the known answers of
corridors, diagonals, corners, walls, a maze and the budget, and every path it returns passes the spec's checker; the
C ABI rejects bad arguments without a device."""
import ctypes as C

import numpy as np
import pytest

import mlmapping_b200 as mlm
from mlmapping_b200 import config_cfg_a, scenes
from reach_oracle import ReachOracle, reach_grid
from reach_spec import (BLOCKING, FREE, UNKNOWN, box_classes, budget, check_path, cost_query, field, path,
                        source_cells)

BIG = 1 << 30


def _grid(shape, p_block, p_unknown, rs):
    u = rs.uniform(size=shape)
    return np.where(u < p_block, BLOCKING, np.where(u < p_block + p_unknown, UNKNOWN, FREE)).astype(np.int8)


def _sources(shape, k, rs):
    return [(int(rs.randint(shape[2])), int(rs.randint(shape[1])), int(rs.randint(shape[0]))) for _ in range(k)]


def test_oracle_equals_spec_on_random_grids():
    """20-60 % blocking, line-shaped and thin boxes, one and several sources, unknown traversable or not"""
    rs = np.random.RandomState(7)
    shapes = [(6, 7, 5), (9, 4, 11), (1, 1, 1), (1, 13, 1), (1, 1, 17), (15, 1, 1), (2, 9, 9), (12, 12, 2), (8, 8, 8)]
    n = 0
    for s in shapes:
        for pb in (0.2, 0.4, 0.6):
            cls = _grid(s, pb, 0.2, rs)
            for k in (1, 3):
                src = _sources(s, k, rs)
                for unknown in (False, True):
                    for K in (BIG, 4000):
                        o = reach_grid(cls, src, K, unknown)
                        assert np.array_equal(o, field(cls, src, K, unknown)), (s, pb, k, unknown, K)
                        n += int((o > 0).sum())
    assert n > 5000


def test_oracle_equals_spec_on_a_larger_grid():
    rs = np.random.RandomState(8)
    cls = _grid((20, 40, 50), 0.25, 0.15, rs)
    src = _sources(cls.shape, 4, rs)
    for unknown in (False, True):
        o = reach_grid(cls, src, BIG, unknown)
        assert np.array_equal(o, field(cls, src, BIG, unknown))
        reach = np.argwhere(o > 0)
        for z, y, x in reach[rs.choice(len(reach), 50, replace=False)]:
            check_path(path(o, cls, src, (x, y, z), unknown), o, cls, src, unknown)


def _free(shape):
    return np.full(shape, FREE, dtype=np.int8)


def test_known_answers_corridor_and_diagonals():
    c = _free((1, 1, 12))
    assert reach_grid(c, [(0, 0, 0)], BIG)[0, 0].tolist() == [1000 * i for i in range(12)]
    # pure face and body diagonals in an open box
    o = reach_grid(_free((7, 7, 7)), [(0, 0, 0)], BIG)
    for i in range(7):
        assert o[0, i, i] == 1414 * i and o[i, i, i] == 1732 * i
    # 2D: one blocking cell of the 2 x 2 block makes the diagonal illegal; the detour is two face moves
    g = _free((1, 2, 2))
    g[0, 0, 1] = BLOCKING
    o = reach_grid(g, [(0, 0, 0)], BIG)
    assert o[0, 1, 1] == 2000 and o[0, 0, 1] == -1
    g[0, 1, 0] = BLOCKING
    assert reach_grid(g, [(0, 0, 0)], BIG)[0, 1, 1] == -1
    # 3D: one blocking cell of the 2 x 2 x 2 block forbids the body diagonal, and the face / edge moves through it
    g = _free((2, 2, 2))
    g[1, 0, 0] = BLOCKING
    o = reach_grid(g, [(0, 0, 0)], BIG)
    assert o[1, 1, 1] == 1414 + 1000 and o[1, 0, 1] == 2000 and o[1, 1, 0] == 2000 and o[1, 0, 0] == -1
    for unknown in (False, True):
        assert np.array_equal(o, field(g, [(0, 0, 0)], BIG, unknown))


def test_known_answers_wall_gap_and_maze():
    # a wall at x = 5 with a one-cell gap at y = 8: everything beyond it goes through the gap
    g = _free((1, 11, 11))
    g[0, :, 5] = BLOCKING
    g[0, 8, 5] = FREE
    o = reach_grid(g, [(0, 0, 0)], BIG)
    # the gap is entered only by the face move from (4, 8) (a diagonal into it cuts the wall): (0, 0) -> (4, 8) is four
    # diagonals and four straight moves
    assert o[0, 8, 5] == 4 * 1414 + 4000 + 1000
    assert np.array_equal(o, field(g, [(0, 0, 0)], BIG)) and (o[0, :, 6:] > 0).all()
    # a serpentine maze: corridors along x joined at alternate ends; the cost is the corridor length
    w, rows = 9, 5
    g = np.full((1, 2 * rows - 1, w), BLOCKING, dtype=np.int8)
    for r in range(rows):
        g[0, 2 * r, :] = FREE
        if r + 1 < rows:
            g[0, 2 * r + 1, w - 1 if r % 2 == 0 else 0] = FREE
    o = reach_grid(g, [(0, 0, 0)], BIG)
    end = (0 if (rows - 1) % 2 == 1 else w - 1)
    assert o[0, 2 * rows - 2, end] == 1000 * (rows * w + rows - 1 - 1)
    assert np.array_equal(o, field(g, [(0, 0, 0)], BIG))
    p = path(o, g, [(0, 0, 0)], (end, 2 * rows - 2, 0))
    assert len(p) == rows * w + rows - 1
    check_path(p, o, g, [(0, 0, 0)])


def test_budget_cut_off_and_sources():
    c = _free((1, 1, 10))
    assert reach_grid(c, [(0, 0, 0)], 5000)[0, 0].tolist() == [0, 1000, 2000, 3000, 4000, 5000, -1, -1, -1, -1]
    assert reach_grid(c, [(0, 0, 0)], 4999)[0, 0].tolist() == [0, 1000, 2000, 3000, 4000, -1, -1, -1, -1, -1]
    # sources outside the box are ignored; a source on a blocking cell is seeded and may be left
    g = _free((1, 1, 5))
    g[0, 0, 2] = BLOCKING
    assert (reach_grid(g, [(-1, 0, 0), (5, 0, 0), (0, 1, 0)], BIG) == -1).all()
    assert reach_grid(g, [(2, 0, 0)], BIG)[0, 0].tolist() == [2000, 1000, 0, 1000, 2000]
    # an empty T: only the sources
    e = np.full((3, 3, 3), BLOCKING, dtype=np.int8)
    o = reach_grid(e, [(1, 1, 1), (0, 2, 1)], BIG)
    assert (o == 0).sum() == 2 and (o > 0).sum() == 0
    # two adjacent sources, both blocking otherwise: a face move between them is allowed
    o = reach_grid(e, [(1, 1, 1), (1, 1, 2)], BIG)
    assert (o == 0).sum() == 2
    # unknown cells are traversable only with the flag
    u = np.full((1, 1, 4), UNKNOWN, dtype=np.int8)
    assert reach_grid(u, [(0, 0, 0)], BIG)[0, 0].tolist() == [0, -1, -1, -1]
    assert reach_grid(u, [(0, 0, 0)], BIG, unknown=True)[0, 0].tolist() == [0, 1000, 2000, 3000]


@pytest.fixture(scope="module")
def corridor():
    """CFG-A, 10 corridor frames, then inflate_map at the last pose"""
    cfg = config_cfg_a()
    orc = ReachOracle(cfg)
    for k in range(10):
        pose = scenes.corridor_trajectory_pose(k * 5)
        orc.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    orc.inflate_map(pose[:3])
    return cfg, orc, orc.export_map(), pose


@pytest.mark.parametrize("inflated", [False, True])
@pytest.mark.parametrize("unknown", [False, True])
def test_oracle_map_field_equals_the_spec(corridor, inflated, unknown):
    """a box around the last pose, starts at the pose and one outside the box: field, queries and paths"""
    cfg, orc, ex, pose = corridor
    d = cfg.subbox_d_xyz
    c = pose[:3]
    bmin, bmax = c - [3.0, 3.0, 1.0], c + [3.0, 3.0, 1.0]
    starts = np.array([c, c + [0.4, 0.0, 0.0], c + [10.0, 0.0, 0.0]])
    ns = orc.build_reach(bmin, bmax, starts, 4.0, inflated=inflated, unknown=unknown)
    lo, dims, cls = box_classes(ex, cfg.subbox_n, d, bmin, bmax, inflated)
    src = source_cells(starts, lo, dims, d)
    assert ns == len(src) == 2
    want = field(cls, src, budget(4.0, d), unknown)
    got, glo = orc.export_reach()
    assert np.array_equal(glo, lo) and np.array_equal(got, want)
    assert (got > 0).sum() > 500 and (got == -1).sum() > 100
    rs = np.random.RandomState(3)
    pts = np.concatenate([rs.uniform(bmin - 0.5, bmax + 0.5, (3000, 3)), [[np.nan, 0, 0], [0, np.inf, 0]]])
    q = orc.reach_cost(pts)
    assert np.array_equal(q.view(np.uint64), cost_query(got, lo, d, pts).view(np.uint64))
    assert np.isnan(q).sum() > 100 and np.isinf(q).sum() > 10
    cells, ln = orc.reach_paths(pts, 64)
    rel = cells.astype(np.int64) - lo
    for i in np.flatnonzero((ln > 0) & (ln <= 64))[:300]:
        check_path(rel[i, :ln[i]], got, cls, src, unknown)
    assert ((ln == -2) == np.isnan(q)).all() and ((ln == -1) == np.isinf(q)).all()


def test_reach_abi_rejects_bad_arguments_without_a_device():
    if not mlm.library_path().exists():
        mlm.build_library()
    lib = mlm.load_library()
    a, b = (C.c_double * 3)(0.0, 0.0, 0.0), (C.c_double * 3)(1.0, 1.0, 1.0)
    s = (C.c_double * 3)(0.5, 0.5, 0.5)
    n = C.c_int32()
    assert lib.mlm_reach_build(None, a, b, s, 1, 1.0, 0, C.byref(n)) == 1
    assert lib.mlm_reach_build(None, a, b, s, 1, 1.0, 4, None) == 1
    p, out = (C.c_double * 3)(), (C.c_double * 3)()
    for fn in (lib.mlm_reach_cost, lib.mlm_reach_cost_device):
        assert fn(None, p, 1, out) == 1
        assert fn(None, None, 0, None) == 1
    cells, ln = (C.c_int32 * 3)(), (C.c_int32 * 1)()
    for fn in (lib.mlm_reach_paths, lib.mlm_reach_paths_device):
        assert fn(None, p, 1, 1, cells, ln) == 1
        assert fn(None, None, 0, 0, None, None) == 1
    lo, dims = (C.c_int32 * 3)(), (C.c_int32 * 3)()
    for fn in (lib.mlm_reach_export, lib.mlm_reach_export_device):
        assert fn(None, None, 0, lo, dims) == 1
