"""CPU: the C++ oracle's frontier clustering (orc_frontier_clusters) equals the numpy restatement of the spec
(tests/frontier_spec.py) bit for bit, records compared as bytes, on the exploration maps of the GPU tests, both
connectivities, min_cells 1 and 10 and several boxes; the restatement's labellers agree with each other and with brute
force; the checkpoint writer's images parse back; and the C ABI rejects bad arguments without a device."""
import ctypes as C

import numpy as np
import pytest

import mlmapping_b200 as mlm
from mlmapping_b200 import config_cfg_a, scenes
from frontier_oracle import FrontierOracle
from frontier_spec import (box_cells, clusters, decode_frontier, export_of, fresh_header, frontier_words,
                           label_scipy, label_union_find, read_checkpoint, sort_labels, write_checkpoint)
from test_parity_gpu import _lidar_small_cfg


def explore_cfg_a():
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    return cfg


def explore_lidar():
    cfg = _lidar_small_cfg()
    cfg.use_exploration_frontiers = 1
    return cfg


def build_map(kind, m):
    """integrate one of the three exploration maps into m (an MLMap or an oracle); returns m's config"""
    if kind == "lidar":
        for k in range(6):
            pose = scenes.lidar_loop_pose(k * 3)
            m.integrate_points(scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512, max_range=20.0), pose)
        return
    frames, stride = (14, 10) if kind == "cfg-a-14" else (40, 5)
    for k in range(frames):
        pose = scenes.corridor_trajectory_pose(k * stride)
        m.integrate_depth(scenes.corridor_depth_frame(m.cfg, pose, frame_idx=k), pose)


def cfg_of(kind):
    return explore_lidar() if kind == "lidar" else explore_cfg_a()


def boxes(cells, d):
    """whole map; a box through the middle of the largest 26-connected cluster (it cuts it); a box without frontier;
    one frontier cell"""
    rec, lab_cells, lab_of = clusters(cells, d)
    big = lab_cells[lab_of == int(np.argmax(rec["n_cells"]))]
    lo, hi = big.min(0), big.max(0)
    mid = (lo + hi) // 2
    cut_lo, cut_hi = lo.copy(), hi.copy()
    cut_hi[0] = mid[0]
    far = cells.min(0) - 40
    one = cells[len(cells) // 2]
    return {"whole": None, "cut": ((cut_lo + 0.5) * d, (cut_hi + 0.5) * d), "empty": ((far + 0.5) * d, (far + 5.5) * d),
            "one_cell": ((one + 0.25) * d, (one + 0.75) * d)}


def assert_oracle_equals_spec(orc, ex, cfg, tag):
    d, n = cfg.subbox_d_xyz, cfg.subbox_n
    cells = decode_frontier(ex, n)
    assert cells.shape[0] > 0
    seen = {}
    for name, box in boxes(cells, d).items():
        for conn6 in (False, True):
            for min_cells in (1, 10):
                key = (tag, name, conn6, min_cells)
                bmin, bmax = (None, None) if box is None else box
                rec, lc, lo = orc.frontier_clusters(bmin, bmax, min_cells, conn6, labels=True)
                srec, slc, slo = clusters(cells, d, None if box is None else box_cells(d, *box), min_cells, conn6)
                assert rec.tobytes() == srec.tobytes(), (key, rec.size, srec.size)
                lc, lo = sort_labels(lc, lo)
                assert np.array_equal(lc, slc) and np.array_equal(lo, slo), key
                seen[key] = rec
    whole = seen[(tag, "whole", False, 1)]
    assert whole["n_cells"].sum() == cells.shape[0]
    cut = seen[(tag, "cut", False, 1)]
    assert cut["n_cells"].max() < whole["n_cells"].max()
    assert seen[(tag, "empty", False, 1)].size == 0 and seen[(tag, "one_cell", True, 1)]["n_cells"].tolist() == [1]
    assert seen[(tag, "whole", True, 1)].size >= whole.size
    return seen


@pytest.fixture(scope="module", params=["cfg-a-14", "cfg-a-40", "lidar"])
def explored(request):
    cfg = cfg_of(request.param)
    orc = FrontierOracle(cfg)
    build_map(request.param, orc)
    return request.param, cfg, orc


def test_oracle_equals_spec_on_the_exploration_maps(explored):
    kind, cfg, orc = explored
    seen = assert_oracle_equals_spec(orc, orc.export_map(), cfg, kind)
    if kind == "lidar":  # the map where one component spans most of the frontier
        whole = seen[(kind, "whole", False, 1)]
        assert whole["n_cells"].max() > 10_000 and whole["n_cells"].max() > whole["n_cells"].sum() // 2


def test_oracle_equals_spec_after_set_free_in_bound():
    """cells that set_free_in_bound made free keep their frontier bits (cell state is not looked at)"""
    cfg = cfg_of("cfg-a-14")
    orc = FrontierOracle(cfg)
    build_map("cfg-a-14", orc)
    before = orc.frontier_clusters()
    orc.setFree_map_in_bound([2.0, -1.0, 0.0], [4.0, 1.0, 1.5])
    after = orc.frontier_clusters()
    assert after.tobytes() == before.tobytes()
    assert_oracle_equals_spec(orc, orc.export_map(), cfg, "set-free")


def _synthetic_sets():
    rs = np.random.RandomState(7)
    out = [np.zeros((0, 3), np.int64), np.array([[0, 0, 0]]), np.array([[-1, -1, -1], [0, 0, 0]]),
           np.array([[0, 0, 0], [1, 1, 0], [5, 5, 5], [5, 5, 6]])]
    for shape, p in (((6, 7, 5), 0.3), ((9, 4, 11), 0.5), ((12, 12, 12), 0.15), ((3, 3, 3), 1.0)):
        m = rs.uniform(size=shape) < p
        out.append(np.argwhere(m)[:, ::-1] - np.array(shape[::-1]) // 2)  # x, y, z around the origin
    g = np.indices((8, 8, 8)).reshape(3, -1).T
    out.append(g[g.sum(1) % 2 == 0] - 4)  # a checkerboard: 26 -> one cluster, 6 -> singletons
    return out


def _brute_force(cells, d, conn6, min_cells):
    """components by repeated flood fill over a Python set, records by the rules' formulas"""
    left = {tuple(c) for c in np.asarray(cells).tolist()}
    recs = []
    while left:
        comp, stack = [], [min(left, key=lambda c: (c[2], c[1], c[0]))]
        left.discard(stack[0])
        while stack:
            c = stack.pop()
            comp.append(c)
            for dz in (-1, 0, 1):
                for dy in (-1, 0, 1):
                    for dx in (-1, 0, 1):
                        l1 = abs(dx) + abs(dy) + abs(dz)
                        b = (c[0] + dx, c[1] + dy, c[2] + dz)
                        if l1 and (l1 == 1 or not conn6) and b in left:
                            left.discard(b)
                            stack.append(b)
        a = np.array(comp, dtype=np.int64)
        if len(comp) >= min_cells:
            key = min(comp, key=lambda c: (c[2], c[1], c[0]))
            cen = tuple(((float(s) / len(comp)) + 0.5) * d for s in a.sum(0))
            recs.append((len(comp), key, tuple(a.min(0)), tuple(a.max(0)), cen))
    return sorted(recs, key=lambda r: (r[1][2], r[1][1], r[1][0]))


def test_spec_labellers_and_records_equal_brute_force():
    d = 0.1
    for cells in _synthetic_sets():
        for conn6 in (False, True):
            for min_cells in (1, 3):
                a = clusters(cells, d, None, min_cells, conn6)
                b = clusters(cells, d, None, min_cells, conn6, labeller=label_union_find)
                assert all(np.array_equal(x, y) for x, y in zip(a[1:], b[1:])) and a[0].tobytes() == b[0].tobytes()
                want = _brute_force(cells, d, conn6, min_cells)
                got = [(int(r["n_cells"]), tuple(r["key"].tolist()), tuple(r["lo"].tolist()), tuple(r["hi"].tolist()),
                        tuple(r["centroid"].tolist())) for r in a[0]]
                assert got == want, (cells.shape, conn6, min_cells)
    g = np.indices((8, 8, 8)).reshape(3, -1).T
    board = g[g.sum(1) % 2 == 0]
    assert clusters(board, d)[0].size == 1 and clusters(board, d, conn6=True)[0].size == board.shape[0]
    assert np.unique(label_scipy(board, True)).size == board.shape[0]


def test_checkpoint_writer_round_trips_through_its_parser():
    cfg = explore_cfg_a()
    n = cfg.subbox_n
    rs = np.random.RandomState(11)
    cells = np.unique(rs.randint(-25, 25, (3000, 3)), axis=0)
    glb, words = frontier_words(cells, n)
    col = np.zeros(glb.shape[0], bool)
    col[::7] = True
    image = write_checkpoint(fresh_header(cfg), cfg, glb, words, col)
    hd, g2, c2, w2 = read_checkpoint(image, n)
    assert hd.n_records == glb.shape[0] and np.array_equal(g2, glb) and np.array_equal(c2, col.astype(np.int32))
    assert np.array_equal(w2[~col], words[~col]) and not w2[col].any()  # a collapsed record carries no frontier
    back = decode_frontier(export_of(g2, w2, c2, n), n)
    keep = ~col[np.unique(np.floor_divide(cells, n), axis=0, return_inverse=True)[1].reshape(-1)]
    order = lambda a: a[np.lexsort((a[:, 0], a[:, 1], a[:, 2]))]
    assert np.array_equal(order(back), order(cells[keep]))
    with pytest.raises(AssertionError):
        read_checkpoint(image[:-16] + bytes(16) if image[-16:] != bytes(16) else image[:-16] + b"\1" * 16, n)


def test_frontier_abi_rejects_bad_arguments_without_a_device():
    if not mlm.library_path().exists():
        mlm.build_library()
    lib = mlm.load_library()
    n, m = C.c_size_t(), C.c_size_t()
    assert lib.mlm_sizeof_frontier_cluster() == 64
    for fn in (lib.mlm_frontier_clusters, lib.mlm_frontier_clusters_device):
        assert fn(None, None, None, 1, 0, None, 0, C.byref(n), None, None, 0, C.byref(m)) == 1
