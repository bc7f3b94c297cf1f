"""GPU: frontier clustering (mlm_frontier_clusters, k_fc_*) against the oracle's restatement (orc_frontier_clusters) bit
for bit on the records, labels compared after sorting; each map first checked against the oracle's, so that a map
mismatch is told apart from a clustering mismatch.  Crafted frontier sets go onto the device through restored checkpoint
images and are checked against the numpy restatement (tests/frontier_spec.py)."""
import ctypes as C

import numpy as np
import pytest

from mlmapping_b200 import MLMap, config_cfg_a, scenes
from mlmapping_b200.capi import FRONTIER_CLUSTER_DTYPE, MlmError
from frontier_oracle import FrontierOracle
from frontier_spec import box_cells, clusters, decode_frontier, frontier_words, sort_labels, write_checkpoint
from parity_utils import assert_map_parity
from test_frontier_host import boxes, build_map, cfg_of, explore_cfg_a
from test_parity_gpu import _lidar_small_cfg

pytestmark = pytest.mark.gpu
LO_TOL = 1e-6


def _assert_gpu_equals_oracle(gpu, orc, cfg, tag):
    cells = decode_frontier(orc.export_map(), cfg.subbox_n)
    for name, box in boxes(cells, cfg.subbox_d_xyz).items():
        bmin, bmax = (None, None) if box is None else box
        for conn6 in (False, True):
            for min_cells in (1, 10):
                key = (tag, name, conn6, min_cells)
                g, gc, go = gpu.frontier_clusters(bmin, bmax, min_cells, conn6, labels=True)
                o, oc, oo = orc.frontier_clusters(bmin, bmax, min_cells, conn6, labels=True)
                assert g.tobytes() == o.tobytes(), (key, g.size, o.size)
                gc, go = sort_labels(gc, go)
                oc, oo = sort_labels(oc, oo)
                assert np.array_equal(gc, oc) and np.array_equal(go, oo), key
                assert gpu.frontier_clusters(bmin, bmax, min_cells, conn6).tobytes() == g.tobytes(), key  # repeatable


@pytest.mark.parametrize("kind", ["cfg-a-14", "cfg-a-40", "lidar"])
def test_frontier_clusters_equal_the_oracle(kind):
    cfg = cfg_of(kind)
    gpu, orc = MLMap(cfg), FrontierOracle(cfg)
    build_map(kind, gpu)
    build_map(kind, orc)
    assert_map_parity(gpu, orc, LO_TOL, tag=kind)
    launches = gpu.kernel_launch_count()
    _assert_gpu_equals_oracle(gpu, orc, cfg, kind)
    assert gpu.kernel_launch_count() > launches
    # the clustering left the map as it was: later queries still equal the oracle's
    rs = np.random.RandomState(5)
    ex = orc.export_map()
    lo, hi = ex["glb"].min(0) * cfg.subbox_n * cfg.subbox_d_xyz, (ex["glb"].max(0) + 1) * cfg.subbox_n * cfg.subbox_d_xyz
    pts = rs.uniform(lo, hi, (20000, 3))
    assert np.array_equal(gpu.getOccupancy(pts), orc.getOccupancy(pts))
    a, b = pts[:5000], pts[5000:10000]
    assert gpu.cast_rays(a, b).tobytes() == orc.cast_rays(a, b).tobytes()
    assert_map_parity(gpu, orc, LO_TOL, tag=kind + " after")


def test_device_variant_equals_host_variant_and_checkpoint_round_trip():
    cfg = cfg_of("cfg-a-14")
    gpu = MLMap(cfg)
    build_map("cfg-a-14", gpu)
    rec, cells, of = gpu.frontier_clusters(labels=True)
    d_out, d_cells, d_of = gpu.device_alloc(64 * rec.size), gpu.device_alloc(12 * of.size), gpu.device_alloc(4 * of.size)
    n, m = gpu.frontier_clusters_device(d_out, rec.size, d_cells, d_of, of.size)
    assert (n, m) == (rec.size, of.size)
    assert gpu.to_host(d_out, rec.size, FRONTIER_CLUSTER_DTYPE).tobytes() == rec.tobytes()
    assert np.array_equal(gpu.to_host(d_cells, (m, 3), np.int32), cells) and np.array_equal(gpu.to_host(d_of, m, np.int32), of)
    for p in (d_out, d_cells, d_of):
        gpu.device_free(p)
    other = MLMap(cfg)
    other.restore(gpu.checkpoint())
    r2, c2, o2 = other.frontier_clusters(labels=True)
    # the label order is repeatable on one handle only: a restore inserts the subboxes concurrently, so two of them that
    # probe the same hash slots can swap slots and with them their cells' place in the list
    (c2, o2), (cells, of) = sort_labels(c2, o2), sort_labels(cells, of)
    assert r2.tobytes() == rec.tobytes() and np.array_equal(c2, cells) and np.array_equal(o2, of)


@pytest.fixture(scope="module")
def crafted():
    """an exploration handle with one frame behind it (a valid header) and a way to replace its frontier sets"""
    cfg = explore_cfg_a()
    gpu = MLMap(cfg)
    pose = scenes.corridor_trajectory_pose(0)
    gpu.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=0), pose)
    template = gpu.checkpoint()

    def load(cells):
        glb, words = frontier_words(cells, cfg.subbox_n)
        gpu.restore(write_checkpoint(template, cfg, glb, words))
        return gpu

    return cfg, load


def _assert_crafted(cfg, gpu, cells, box=None, min_cells=(1, 10)):
    d = cfg.subbox_d_xyz
    out = {}
    for conn6 in (False, True):
        for mc in min_cells:
            bmin, bmax = (None, None) if box is None else box
            g, gc, go = gpu.frontier_clusters(bmin, bmax, mc, conn6, labels=True)
            s, sc, so = clusters(cells, d, None if box is None else box_cells(d, *box), mc, conn6)
            assert g.tobytes() == s.tobytes(), (conn6, mc, g.size, s.size)
            gc, go = sort_labels(gc, go)
            assert np.array_equal(gc, sc) and np.array_equal(go, so), (conn6, mc)
            out[(conn6, mc)] = g
    return out


def test_crafted_corner_negative_and_checkerboard(crafted):
    cfg, load = crafted
    n = cfg.subbox_n
    # two blobs that touch only at the corner shared by the 8 subboxes around the origin, and at a corner of 8 subboxes
    # around (n, n, n)
    a = np.indices((3, 3, 3)).reshape(3, -1).T
    cells = np.concatenate([a - 3, a, a + n - 3 + np.array([0, 0, 0]), a + n])
    out = _assert_crafted(cfg, load(cells), cells)
    assert out[(False, 1)].size == 2 and out[(True, 1)].size == 4
    # a 3-D checkerboard over 27 subboxes, negative coordinates
    g = np.indices((3 * n, 3 * n, 3 * n)).reshape(3, -1).T - 2 * n + 3
    board = g[g.sum(1) % 2 == 0]
    out = _assert_crafted(cfg, load(board), board, min_cells=(1,))
    assert out[(False, 1)].size == 1 and out[(True, 1)].size == board.shape[0]
    box = ((board.min(0) + 4.5) * cfg.subbox_d_xyz, (board.min(0) + 20.5) * cfg.subbox_d_xyz)
    _assert_crafted(cfg, load(board), board, box=box, min_cells=(1,))


def test_crafted_snake_and_full_subboxes(crafted):
    cfg, load = crafted
    # a snake of > 100 k cells: x runs on every other y row, joined at alternating ends; layers on every other z, joined
    L, rows, layers = 100, 50, 25
    parts = []
    for zi in range(layers):
        for yi in range(rows):
            y = 2 * yi if zi % 2 == 0 else 2 * (rows - 1 - yi)
            parts.append(np.stack([np.arange(L), np.full(L, y), np.full(L, 2 * zi)], 1))
            if yi + 1 < rows:
                end = L - 1 if yi % 2 == 0 else 0
                parts.append(np.array([[end, y + (1 if zi % 2 == 0 else -1), 2 * zi]]))
        if zi + 1 < layers:
            last = parts[-1][-1]
            parts.append(np.array([[last[0], last[1], 2 * zi + 1]]))
    snake = np.concatenate(parts) - np.array([37, 41, 13])
    assert snake.shape[0] > 100_000
    out = _assert_crafted(cfg, load(snake), snake, min_cells=(1,))
    assert out[(False, 1)]["n_cells"].tolist() == [snake.shape[0]]
    # 512 subboxes with every bit set: one cluster of 512 k cells
    full = np.indices((80, 80, 80)).reshape(3, -1).T - 40
    out = _assert_crafted(cfg, load(full), full, min_cells=(1,))
    assert out[(True, 1)]["n_cells"].tolist() == [512_000]


def test_caps_smaller_than_the_result(crafted):
    cfg, load = crafted
    rs = np.random.RandomState(3)
    cells = np.unique(rs.randint(-30, 30, (4000, 3)), axis=0)
    gpu = load(cells)
    rec, lc, lo = clusters(cells, cfg.subbox_d_xyz, conn6=True)
    assert rec.size > 100
    lib, h = gpu._lib, gpu._h
    out = np.zeros(rec.size, dtype=FRONTIER_CLUSTER_DTYPE)
    c3, of = np.full((lo.size, 3), -7, np.int32), np.full(lo.size, -7, np.int32)
    n, m = C.c_size_t(), C.c_size_t()
    assert lib.mlm_frontier_clusters(h, None, None, 1, 1, out.ctypes.data, 10, C.byref(n), c3.ctypes.data,
                                     of.ctypes.data, 100, C.byref(m)) == 0
    assert (n.value, m.value) == (rec.size, lo.size)
    assert out[:10].tobytes() == rec[:10].tobytes() and not out[10:].tobytes().strip(b"\0")
    assert (of[:100] >= 0).all() and (of[100:] == -7).all() and (c3[100:] == -7).all()
    assert lib.mlm_frontier_clusters(h, None, None, 1, 1, None, 0, C.byref(n), None, None, 0, None) == 0
    assert n.value == rec.size


def test_errors():
    cfg = explore_cfg_a()
    gpu = MLMap(cfg)
    lib, h = gpu._lib, gpu._h
    n = C.c_size_t()
    a, b = (C.c_double * 3)(0.0, 0.0, 0.0), (C.c_double * 3)(1.0, 1.0, 1.0)
    nan = float("nan")
    assert lib.mlm_frontier_clusters(h, a, b, 1, 0, None, 0, C.byref(n), None, None, 0, None) == 0 and n.value == 0
    assert lib.mlm_frontier_clusters(h, a, None, 1, 0, None, 0, C.byref(n), None, None, 0, None) == 1
    assert lib.mlm_frontier_clusters(h, None, b, 1, 0, None, 0, C.byref(n), None, None, 0, None) == 1
    assert lib.mlm_frontier_clusters(h, b, a, 1, 0, None, 0, C.byref(n), None, None, 0, None) == 1   # min > max
    for bad in ((nan, 0, 0), (0, float("inf"), 0), (0, 0, 2.0 ** 30 * cfg.subbox_d_xyz)):
        assert lib.mlm_frontier_clusters(h, (C.c_double * 3)(*bad), b, 1, 0, None, 0, C.byref(n), None, None, 0, None) == 1
    assert lib.mlm_frontier_clusters(h, None, None, 0, 0, None, 0, C.byref(n), None, None, 0, None) == 1  # min_cells
    assert lib.mlm_frontier_clusters(h, None, None, 1, 2, None, 0, C.byref(n), None, None, 0, None) == 1  # flags
    assert lib.mlm_frontier_clusters(h, None, None, 1, 0, None, 4, C.byref(n), None, None, 0, None) == 1  # null out
    assert lib.mlm_frontier_clusters(h, None, None, 1, 0, None, 0, C.byref(n), None, None, 4, None) == 1  # null cells
    assert lib.mlm_frontier_clusters(h, None, None, 1, 0, None, 0, None, None, None, 0, None) == 1         # null n_out
    plain = MLMap(config_cfg_a())
    with pytest.raises(MlmError) as ei:
        plain.frontier_clusters()
    assert ei.value.code == 6


def test_sharded_ranks_refuse():
    """sharded maps run without the exploration mode (mlm_shard_open refuses it), so every rank of a world-2 map has no
    frontier sets to cluster: MLM_ERR_UNSUPPORTED"""
    from mlmapping_b200.sharded import sharded_group_in_process
    ranks = sharded_group_in_process(_lidar_small_cfg(), 2)
    try:
        for r in ranks:
            with pytest.raises(MlmError) as ei:
                r.map.frontier_clusters()
            assert ei.value.code == 6
    finally:
        for r in ranks:
            r.close()
