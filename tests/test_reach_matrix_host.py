"""CPU: the path-cost matrix's restatement (reach_matrix_spec.matrix, one scipy Dijkstra per row) equals a loop of
the C++ oracle's single-start fields bit for bit, on random class grids under every flag combination and on a crafted
map through the oracle's world-point calls (build_reach + reach_cost per row); it covers starts in occupied, unknown
and inflated cells, on tile faces, duplicated, outside the box and failing rule 1, and an asymmetric pair.  The C ABI
refuses bad matrix arguments without a device."""
import ctypes as C

import numpy as np
import pytest

import mlmapping_b200 as mlm
from mlmapping_b200 import config_cfg_a
from esdf_spec import cells_of
from reach_oracle import ReachOracle, reach_grid
from reach_matrix_spec import matrix
from reach_spec import BLOCKING, FREE, UNKNOWN, box_classes, budget
from view_spec import crafted_map

BIG = 1 << 30
FLAGS = [(False, False), (True, False), (False, True), (True, True)]


def _grid(shape, p_block, p_unknown, rs):
    u = rs.uniform(size=shape)
    return np.where(u < p_block, BLOCKING, np.where(u < p_block + p_unknown, UNKNOWN, FREE)).astype(np.int8)


def _oracle_loop(cls, starts, goals, K, unknown):
    """the definition: one oracle field per start, read at the goals (-2 outside the box)"""
    goals = np.asarray(goals, dtype=np.int64)
    dims = np.array(cls.shape[::-1])
    inside = ((goals >= 0) & (goals < dims)).all(1)
    g = np.where(inside[:, None], goals, 0)
    out = np.empty((len(starts), goals.shape[0]), dtype=np.int64)
    for i, s in enumerate(starts):
        f = reach_grid(cls, [s], K, unknown)
        out[i] = np.where(inside, f[g[:, 2], g[:, 1], g[:, 0]], -2)
    return out


def _special_starts(cls, rs):
    """a free, a blocking and an unknown cell, cells on tile faces (7 and 8 mod 8), a duplicate, cells outside the
    box"""
    nz, ny, nx = cls.shape
    out = []
    for kind in (FREE, BLOCKING, UNKNOWN):
        w = np.argwhere(cls == kind)
        if len(w):
            z, y, x = w[rs.randint(len(w))]
            out.append((int(x), int(y), int(z)))
    for face in (7, 8):
        out.append((min(face, nx - 1), min(face, ny - 1), min(face, nz - 1)))
    out.append(out[0])
    out += [(-1, 0, 0), (nx, 0, 0), (0, 0, nz + 3)]
    return out


def test_matrix_spec_equals_the_oracle_loop_on_random_grids():
    """20-60 % blocking, every flag combination (the inflated flag acts on the class grid, so it is the same grid here),
    unlimited and tight budgets; goals are the starts plus random cells, some outside the box"""
    rs = np.random.RandomState(17)
    asym = 0
    for shape in [(9, 10, 11), (3, 17, 16), (12, 12, 12)]:
        for pb in (0.2, 0.4, 0.6):
            cls = _grid(shape, pb, 0.2, rs)
            starts = _special_starts(cls, rs) + [(int(rs.randint(shape[2])), int(rs.randint(shape[1])),
                                                  int(rs.randint(shape[0]))) for _ in range(6)]
            extra = [(int(rs.randint(-2, shape[2] + 2)), int(rs.randint(-2, shape[1] + 2)),
                      int(rs.randint(-2, shape[0] + 2))) for _ in range(40)]
            goals = starts + extra
            for _, unknown in FLAGS:
                for K in (BIG, 5000):
                    want = _oracle_loop(cls, starts, goals, K, unknown)
                    got = matrix(cls, starts, goals, K, unknown)
                    assert np.array_equal(got, want), (shape, pb, unknown, K)
                    # rows of starts outside the box: -1 in the box, -2 outside
                    for i, s in enumerate(starts):
                        if not all(0 <= s[k] < shape[2 - k] for k in range(3)):
                            assert set(np.unique(got[i])) <= {-1, -2}
                    n = len(starts)
                    sq = got[:, :n]
                    asym += int(((sq >= 0) & (sq.T == -1)).sum())
    assert asym > 0


def test_blocked_start_makes_the_matrix_asymmetric():
    """a start inside a wall reaches the free cells next to it, but as a goal of the other row it is unreachable"""
    cls = np.full((1, 1, 6), FREE, dtype=np.int8)
    cls[0, 0, 3] = BLOCKING
    starts = [(3, 0, 0), (1, 0, 0)]
    got = matrix(cls, starts, starts, BIG)
    assert got[0, 1] == 2000 and got[1, 0] == -1 and got[0, 0] == 0 and got[1, 1] == 0
    assert np.array_equal(got, _oracle_loop(cls, starts, starts, BIG, False))


@pytest.fixture(scope="module")
def crafted_oracle():
    """a 20 x 18 x 10 crafted map: free with 30 % occupied and 15 % unknown cells, inflation on 10 % of the free ones"""
    cfg = config_cfg_a()
    rs = np.random.RandomState(5)
    origin = np.array([-6, 3, -2])
    cells, infl = {}, []
    for z in range(10):
        for y in range(18):
            for x in range(20):
                u = rs.uniform()
                s = b"o" if u < 0.3 else (b"u" if u < 0.45 else b"f")
                c = (int(origin[0] + x), int(origin[1] + y), int(origin[2] + z))
                cells[c] = s
                if s == b"f" and rs.uniform() < 0.1:
                    infl.append(c)
    ex = crafted_map(cells, cfg.subbox_n, inflated=infl)
    orc = ReachOracle(cfg)
    orc.set_map(ex)
    yield cfg, orc, ex, origin, infl
    orc.close()


@pytest.mark.parametrize("inflated,unknown", FLAGS)
def test_matrix_spec_equals_oracle_world_points(crafted_oracle, inflated, unknown):
    """world points through rule 1: the oracle's build_reach + reach_cost per row against the restatement with rule 6,
    starts in occupied, unknown and inflated cells, a NaN start, starts outside the box and a duplicate"""
    cfg, orc, ex, origin, infl = crafted_oracle
    d = cfg.subbox_d_xyz
    bmin, bmax = (origin + 0.5) * d, (origin + np.array([20, 18, 10]) - 0.5) * d
    lo, dims, cls = box_classes(ex, cfg.subbox_n, d, bmin, bmax, inflated)
    rs = np.random.RandomState(6)
    starts = []
    for kind in (FREE, BLOCKING, UNKNOWN):
        for z, y, x in np.argwhere(cls == kind)[:2]:
            starts.append((lo + [x, y, z] + 0.5) * d)
    starts.append((np.array(infl[0]) + 0.5) * d)
    starts.append((lo + [7, 8, 7] + 0.5) * d)                # tile faces
    starts.append(starts[0])
    starts += [[np.nan, 0, 0], (lo - 3 + 0.5) * d, [1e12, 0, 0]]
    starts = np.array(starts, dtype=np.float64)
    goals = np.concatenate([starts, rs.uniform(bmin - 0.6, bmax + 0.6, (120, 3))])
    max_dist = 6.0
    K = budget(max_dist, d)
    want = np.empty((starts.shape[0], goals.shape[0]))
    for i, s in enumerate(starts):
        orc.build_reach(bmin, bmax, [s], max_dist, inflated=inflated, unknown=unknown)
        want[i] = orc.reach_cost(goals)
    # the restatement: cells by rule 1 (an invalid start or goal gets a cell outside the box)
    def rel(p):
        valid, c = cells_of(p, d)
        return np.where(valid.all(1)[:, None], c - lo, -1)
    m = matrix(cls, [tuple(r) for r in rel(starts)], rel(goals), K, unknown)
    with np.errstate(invalid="ignore"):
        got = np.where(m == -2, np.nan, np.where(m == -1, np.inf, (m.astype(np.float64) / 1000.0) * d))
    assert np.array_equal(got.view(np.uint64), want.view(np.uint64))
    assert np.isnan(want).any() and np.isinf(want).any() and (np.isfinite(want) & (want > 0)).sum() > 50
    n = starts.shape[0]
    sq = want[:, :n]
    assert (np.isfinite(sq) & np.isinf(sq.T)).any()           # the asymmetry, not assumed


def test_matrix_abi_rejects_bad_arguments_without_a_device():
    if not mlm.library_path().exists():
        mlm.build_library()
    lib = mlm.load_library()
    a, b = (C.c_double * 3)(0.0, 0.0, 0.0), (C.c_double * 3)(1.0, 1.0, 1.0)
    s, out = (C.c_double * 3)(0.5, 0.5, 0.5), (C.c_double * 1)()
    for fn in (lib.mlm_reach_matrix, lib.mlm_reach_matrix_device):
        assert fn(None, a, b, s, 1, s, 1, 1.0, 0, out) == 1
        assert fn(None, a, b, None, 0, None, 0, 1.0, 0, None) == 1
