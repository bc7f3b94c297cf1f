"""GPU: the reachability field (mlm_reach_*, k_reach_*) against the oracle's restatement of the spec (orc_reach_*), bit
for bit on the exported field, the cost queries (NaN and +inf included) and the paths, on frame-built maps under every
flag combination and on crafted maps restored from checkpoint images (a 3D serpentine maze, a checkerboard only
diagonal leaks could connect, an all-free box, an all-unknown box, negative coordinates).  Each frame-built map is first
checked against the oracle's, so that a map mismatch is told apart from a field mismatch."""
import ctypes as C

import numpy as np
import pytest

from mlmapping_b200 import MLMap, config_cfg_a, scenes
from mlmapping_b200.capi import MlmError
from esdf_spec import first_difference, query_points, same_bits
from parity_utils import assert_map_parity
from reach_oracle import ReachOracle
from reach_spec import box_classes, check_path, source_cells
from test_parity_gpu import _lidar_small_cfg
from view_spec import crafted_map, write_map_checkpoint

pytestmark = pytest.mark.gpu
LO_TOL = 1e-6
FLAGS = [(False, False), (True, False), (False, True), (True, True)]


def _assert_same(gpu, orc, bmin, bmax, starts, max_dist, inflated, unknown, n_query, seed, tag, max_cells=256):
    """build on both, then field, queries and paths bit for bit; returns (field, lo)"""
    key = (tag, inflated, unknown)
    ng = gpu.build_reach(bmin, bmax, starts, max_dist, inflated=inflated, unknown=unknown)
    no = orc.build_reach(bmin, bmax, starts, max_dist, inflated=inflated, unknown=unknown)
    assert ng == no, key
    g, glo = gpu.export_reach()
    o, olo = orc.export_reach()
    assert np.array_equal(glo, olo) and g.shape == o.shape, key
    assert np.array_equal(g, o), (key, first_difference(g, o))
    d = orc.cfg.subbox_d_xyz
    pts = query_points(glo.astype(np.int64), np.array(g.shape[::-1]), d, n_query, seed)
    assert same_bits(gpu.reach_cost(pts), orc.reach_cost(pts)), key
    goals = pts[:: max(1, pts.shape[0] // 4000)]
    gc, gl = gpu.reach_paths(goals, max_cells)
    oc, ol = orc.reach_paths(goals, max_cells)
    assert np.array_equal(gl, ol), (key, first_difference(gl, ol))
    for i in np.flatnonzero(gl > 0):
        k = min(int(gl[i]), max_cells)
        assert np.array_equal(gc[i, :k], oc[i, :k]), (key, i)
    return g, glo, pts, goals


def _boxes(ex, cfg, centre):
    """the map's AABB padded by 1 m, a box reaching 5 m into unmapped space, one cell"""
    n, d = cfg.subbox_n, cfg.subbox_d_xyz
    lo, hi = ex["glb"].min(0) * n * d, (ex["glb"].max(0) + 1) * n * d
    mid = (lo + hi) / 2
    cell = (np.floor(centre / d) + 0.5) * d
    return {"aabb": (lo - 1.0, hi + 1.0), "partly_unmapped": (mid, np.maximum(hi + 5.0, mid + 1.0)),
            "one_cell": (cell, cell)}


def test_reach_cfg_a_trajectory_with_inflation_all_flags():
    """CFG-A, 40 frames at stride 5, inflate_map; every box and flag combination; device variants = host variants;
    truncated paths; export caps; a frame after the build leaves the field as it is"""
    cfg = config_cfg_a()
    gpu, orc = MLMap(cfg), ReachOracle(cfg)
    for k in range(40):
        pose = scenes.corridor_trajectory_pose(k * 5)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    gpu.inflate_map(pose[:3])
    orc.inflate_map(pose[:3])
    assert_map_parity(gpu, orc, LO_TOL, tag="cfg-a")
    ex = orc.export_map()
    c = pose[:3]
    starts = np.array([c, scenes.corridor_trajectory_pose(50)[:3], c + [1000.0, 0, 0]])
    for name, (bmin, bmax) in _boxes(ex, cfg, c).items():
        for inflated, unknown in FLAGS:
            g, lo, _, _ = _assert_same(gpu, orc, bmin, bmax, starts, 30.0, inflated, unknown,
                                       100_000 if name == "aabb" else 3000, 11, name)
            if name == "aabb":
                assert (g > 0).sum() > 10_000 and (g == -1).sum() > 1000, (inflated, unknown)
    # device variants against the host variants, on the last aabb build (inflated + unknown)
    bmin, bmax = _boxes(ex, cfg, c)["aabb"]
    gpu.build_reach(bmin, bmax, starts, 30.0, inflated=True, unknown=True)
    g, lo = gpu.export_reach()
    pts = query_points(lo.astype(np.int64), np.array(g.shape[::-1]), cfg.subbox_d_xyz, 20_000, 12)
    want = gpu.reach_cost(pts)
    n = pts.shape[0]
    d_p, d_o = gpu.to_device(pts), gpu.device_alloc(8 * n)
    gpu.reach_cost_device(d_p, n, d_o)
    assert same_bits(gpu.to_host(d_o, (n,), np.float64), want)
    mc = 64
    hc, hl = gpu.reach_paths(pts, mc)
    d_c, d_l = gpu.device_alloc(12 * n * mc), gpu.device_alloc(4 * n)
    gpu.reach_paths_device(d_p, n, mc, d_c, d_l)
    dl, dc = gpu.to_host(d_l, (n,), np.int32), gpu.to_host(d_c, (n, mc, 3), np.int32)
    assert np.array_equal(dl, hl)
    for i in np.flatnonzero(hl > 0):
        assert np.array_equal(dc[i, :min(hl[i], mc)], hc[i, :min(hl[i], mc)])
    # truncated paths: the first cells of a longer walk, the full length reported
    long_ = np.flatnonzero(hl > 8)
    assert long_.size > 100
    tc, tl = gpu.reach_paths(pts[long_], 8)
    assert np.array_equal(tl, hl[long_]) and np.array_equal(tc, hc[long_, :8])
    zc, zl = gpu.reach_paths(pts[long_], 0)
    assert np.array_equal(zl, hl[long_])
    cells = g.size
    d_e = gpu.device_alloc(4 * cells)
    lo2, dims = gpu.export_reach_device(d_e, cells)
    assert np.array_equal(dims, g.shape[::-1]) and np.array_equal(gpu.to_host(d_e, g.shape, np.int32), g)
    with pytest.raises(MlmError) as ei:
        gpu.export_reach_device(d_e, cells - 1)
    assert ei.value.code == 5
    lib, h = gpu._lib, gpu._h
    lo3, dims3 = (C.c_int32 * 3)(), (C.c_int32 * 3)()
    assert lib.mlm_reach_export(h, None, 0, lo3, dims3) == 0 and tuple(dims3) == g.shape[::-1]
    assert lib.mlm_reach_export(h, (C.c_int32 * 4)(), 4, lo3, dims3) == 5
    # the field is a snapshot
    for k in range(40, 44):
        p = scenes.corridor_trajectory_pose(k * 5)
        gpu.integrate_depth(scenes.corridor_depth_frame(cfg, p, frame_idx=k), p)
    gpu.inflate_map(p[:3])
    assert np.array_equal(gpu.export_reach()[0], g) and same_bits(gpu.reach_cost(pts), want)
    for q in (d_p, d_o, d_c, d_l, d_e):
        gpu.device_free(q)


def test_reach_on_the_lidar_map():
    cfg = _lidar_small_cfg()
    gpu, orc = MLMap(cfg), ReachOracle(cfg)
    for k in range(6):
        pose = scenes.lidar_loop_pose(k * 3)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512)
        gpu.integrate_points(pts, pose)
        orc.integrate_points(pts, pose)
    assert_map_parity(gpu, orc, LO_TOL, tag="lidar")
    ex = orc.export_map()
    c = pose[:3]
    for name, (bmin, bmax) in _boxes(ex, cfg, c).items():
        for inflated, unknown in FLAGS:
            _assert_same(gpu, orc, bmin, bmax, [c], 60.0, inflated, unknown, 50_000 if name == "aabb" else 3000, 21,
                         name)


# ---- crafted maps ---------------------------------------------------------------------------------------------------
def _explore_cfg():
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    return cfg


@pytest.fixture(scope="module")
def crafted():
    cfg = _explore_cfg()
    gpu = MLMap(cfg)
    yield cfg, gpu, gpu.checkpoint()
    gpu.close()


def _restore(cfg, gpu, template, states, origin, inflated=()):
    """states[Z, Y, X] of b'f' / b'o' / b'u' placed at cell origin, inflation 'o' on the pattern cells (x, y, z) of
    `inflated`; returns the oracle holding the same map"""
    cells = {}
    for (z, y, x), s in np.ndenumerate(states):
        cells[(origin[0] + x, origin[1] + y, origin[2] + z)] = s
    ex = crafted_map(cells, cfg.subbox_n, inflated=[tuple(int(v) for v in np.add(origin, c)) for c in inflated])
    gpu.restore(write_map_checkpoint(template, cfg, ex))
    back = gpu.export_map()
    assert np.array_equal(back["glb"], ex["glb"]) and np.array_equal(back["occupancy"], ex["occupancy"])
    orc = ReachOracle(cfg)
    orc.set_map(ex)
    return orc, ex


def _serpentine(nx, ny, nz):
    """corridors along x on every other y row, joined at alternate ends; layers joined the same way along z"""
    s = np.full((nz, ny, nx), b"o", dtype="S1")
    for z in range(0, nz, 2):
        for y in range(0, ny, 2):
            s[z, y, :] = b"f"
            if y + 2 < ny:
                s[z, y + 1, nx - 1 if (y // 2) % 2 == 0 else 0] = b"f"
        if z + 2 < nz:
            last = ((ny - 1) // 2) % 2
            s[z + 1, ny - 1 if ny % 2 else ny - 2, 0 if last else nx - 1] = b"f"
    return s


CRAFTED = {
    "maze": (lambda: _serpentine(40, 41, 5), (3, -2, 1)),
    "checkerboard": (lambda: np.where(np.indices((6, 20, 20)).sum(0) % 2 == 0, b"f", b"o").astype("S1"), (0, 0, 0)),
    "all_free": (lambda: np.full((24, 64, 64), b"f", dtype="S1"), (-10, -10, -4)),
    "negative": (lambda: _serpentine(17, 23, 3), (-1000, -507, -33)),
}


@pytest.mark.parametrize("name", sorted(CRAFTED))
def test_reach_crafted_maps(crafted, name):
    cfg, gpu, template = crafted
    d = cfg.subbox_d_xyz
    make, origin = CRAFTED[name]
    states = make()
    orc, ex = _restore(cfg, gpu, template, states, origin)
    o = np.array(origin)
    bmin = (o + 0.5) * d
    bmax = (o + np.array(states.shape[::-1]) - 0.5) * d
    start = (o + 0.5) * d                                     # cell (0, 0, 0) of the pattern: free in every pattern
    for inflated, unknown in FLAGS:
        g, lo, pts, goals = _assert_same(gpu, orc, bmin, bmax, [start], 1e4, inflated, unknown, 20_000, 31, name,
                                         max_cells=1024)
    lo_, dims, cls = box_classes(ex, cfg.subbox_n, d, bmin, bmax)
    src = source_cells([start], lo_, dims, d)
    if name in ("maze", "negative"):
        assert (g >= 0).sum() == (states == b"f").sum()       # the maze is one corridor: every free cell reached
        far = np.unravel_index(np.argmax(g), g.shape)
        gc, gl = gpu.reach_paths((np.array(far[::-1]) + lo + 0.5) * d, 1 << 14)
        assert gl[0] > 500 if name == "maze" else gl[0] > 150
        check_path(gc[0, :gl[0]].astype(np.int64) - lo, g, cls, src)
    if name == "checkerboard":
        assert (g >= 0).sum() == 1                            # no face move exists and every diagonal cuts a corner
    if name == "all_free":
        assert (g >= 0).all() and g[0, 0, 1] == 1000 and g[1, 1, 1] == 1732
    # an all-unknown box next to the crafted map: only the source, or everything with unknown cells traversable
    far_lo = (o + np.array([200, 200, 0]) + 0.5) * d
    far_hi = far_lo + np.array([20, 20, 8]) * d
    for unknown in (False, True):
        g, *_ = _assert_same(gpu, orc, far_lo, far_hi, [far_lo], 1e4, False, unknown, 5000, 41, "unknown")
        assert (g >= 0).sum() == (g.size if unknown else 1)
    orc.close()


def _pattern_box(origin, states, d):
    """the box whose cells are exactly those of the pattern: box-relative coordinates are pattern coordinates, so the
    solve's 8-cell tiles start at pattern cell 0"""
    o = np.asarray(origin)
    return (o + 0.5) * d, (o + np.array(states.shape[::-1]) - 0.5) * d


@pytest.mark.parametrize("axis", [0, 1, 2])
def test_reach_corridor_start_swept_across_tile_faces(crafted, axis):
    """a 1-cell corridor of 24 cells along one axis, walled in on every side, the start on each cell from 5 to 18: at 7,
    8, 15 and 16 the start sits on a tile face, and half of the corridor lies only across that face.  Every corridor
    cell is reached at its exact distance, equal to the oracle's bit for bit"""
    cfg, gpu, template = crafted
    d, n = cfg.subbox_d_xyz, 24
    shape = [3, 3, 3]
    shape[2 - axis] = n                                       # states are [Z, Y, X]
    states = np.full(tuple(shape), b"o", dtype="S1")
    line = [1, 1, 1]
    line[2 - axis] = slice(None)
    states[tuple(line)] = b"f"
    origin = np.array([-13, 4, 2])
    orc, _ = _restore(cfg, gpu, template, states, origin)
    bmin, bmax = _pattern_box(origin, states, d)
    for p in range(5, 19):
        cell = origin + 1
        cell[axis] = origin[axis] + p
        for inflated, unknown in ((False, False), (True, True)):
            g, *_ = _assert_same(gpu, orc, bmin, bmax, [(cell + 0.5) * d], 1e3, inflated, unknown, 500, p,
                                 ("corridor", axis, p))
            assert (g >= 0).sum() == n and g.max() == 1000 * max(p, n - 1 - p), (axis, p, inflated, unknown)
    orc.close()


@pytest.mark.parametrize("wall", [7, 8])
@pytest.mark.parametrize("kind", ["occupied", "unknown", "inflation"])
def test_reach_source_inside_a_wall_on_a_tile_face(crafted, wall, kind):
    """a 16^3 free box cut by a wall at x = 7 or 8 (the last cell of tile 0 or the first of tile 1), the start inside the
    wall at y = 7 (a second tile face): occupied, unknown (not traversable) or free but in the inflation layer (with the
    inflated flag).  The start is a source whatever its state, and both sides of the wall are reached through it"""
    cfg, gpu, template = crafted
    d = cfg.subbox_d_xyz
    states = np.full((16, 16, 16), b"f", dtype="S1")
    inflated_cells = ()
    if kind == "inflation":
        inflated_cells = [(wall, y, z) for z in range(16) for y in range(16)]
    else:
        states[:, :, wall] = b"o" if kind == "occupied" else b"u"
    origin = np.array([5, -9, 3])
    orc, _ = _restore(cfg, gpu, template, states, origin, inflated=inflated_cells)
    bmin, bmax = _pattern_box(origin, states, d)
    start = (origin + np.array([wall, 7, 8]) + 0.5) * d
    g, *_ = _assert_same(gpu, orc, bmin, bmax, [start], 1e3, kind == "inflation", False, 3000, wall, (kind, wall))
    assert (g >= 0).sum() == 16 ** 3 - 16 ** 2 + 1, (kind, wall)
    assert (g[:, :, :wall] >= 0).all() and (g[:, :, wall + 1:] >= 0).all()
    orc.close()
    orc.close()


def test_reach_arguments_and_lifetime():
    cfg = config_cfg_a()
    gpu = MLMap(cfg)
    with pytest.raises(MlmError) as ei:
        gpu.reach_cost([[0.0, 0.0, 0.0]])
    assert ei.value.code == 1 and "mlm_reach_build" in str(ei.value)
    for call in (lambda: gpu.export_reach(), lambda: gpu.reach_paths([[0.0, 0.0, 0.0]], 4)):
        with pytest.raises(MlmError) as ei:
            call()
        assert ei.value.code == 1
    lib, h = gpu._lib, gpu._h
    d = cfg.subbox_d_xyz
    a, b = (C.c_double * 3)(0.0, 0.0, 0.0), (C.c_double * 3)(1.0, 1.0, 1.0)
    s = (C.c_double * 3)(0.5, 0.5, 0.5)
    nan, inf = float("nan"), float("inf")
    assert lib.mlm_reach_build(h, a, b, s, 1, 1.0, 4, None) == 1                  # flags
    assert lib.mlm_reach_build(h, a, b, s, 0, 1.0, 0, None) == 1                  # no starts
    assert lib.mlm_reach_build(h, a, b, None, 1, 1.0, 0, None) == 1
    for md in (0.0, -1.0, nan, inf):
        assert lib.mlm_reach_build(h, a, b, s, 1, md, 0, None) == 1
    for bad in ((nan, 0, 0), (0, inf, 0), (2.0, 0, 0)):
        assert lib.mlm_reach_build(h, (C.c_double * 3)(*bad), b, s, 1, 1.0, 0, None) == 1
    x0 = 0.05
    assert lib.mlm_reach_build(h, (C.c_double * 3)(x0, 0.05, 0.05), (C.c_double * 3)(x0 + 4096 * d, 0.05, 0.05), s, 1,
                               1.0, 0, None) == 5
    big = 4095.5 * d
    assert lib.mlm_reach_build(h, a, (C.c_double * 3)(big, big, 20.5 * d), s, 1, 1.0, 0, None) == 5
    # the budget: K <= 2^30 is accepted, K > 2^30 is not
    k_max = float(1 << 30) / 1000.0 * d
    seen = set()
    for md in (k_max * (1 - 1e-9), k_max, np.nextafter(k_max, inf), k_max * (1 + 1e-9), k_max * 2):
        ok = np.floor((md / d) * 1000.0) <= float(1 << 30)
        seen.add(ok)
        n = C.c_int32(-1)
        assert lib.mlm_reach_build(h, a, b, s, 1, md, 0, C.byref(n)) == (0 if ok else 5), md
        assert n.value == (1 if ok else -1)
    assert seen == {True, False}
    out = (C.c_double * 3)()
    assert lib.mlm_reach_cost(h, None, 1, out) == 1
    assert lib.mlm_reach_cost(h, out, 1, None) == 1
    assert lib.mlm_reach_cost(h, None, 0, None) == 0
    ln = (C.c_int32 * 1)()
    assert lib.mlm_reach_paths(h, out, 1, 4, None, ln) == 1
    assert lib.mlm_reach_paths(h, s, 1, 0, None, ln) == 0 and ln[0] == 1       # the source cell itself
    # an empty map, starts outside the box: nothing reachable, 0 sources
    assert gpu.build_reach([0, 0, 0], [1, 1, 1], [[5.0, 5.0, 5.0]], 2.0) == 0
    g, _ = gpu.export_reach()
    assert (g == -1).all()
    # rebuild with a smaller then a larger box (the buffers grow) and several starts in one cell
    assert gpu.build_reach([0, 0, 0], [3, 3, 1], [[0.5, 0.5, 0.5], [0.51, 0.55, 0.5]], 2.0, unknown=True) == 1
    g, _ = gpu.export_reach()
    assert g.max() <= int(np.floor((2.0 / d) * 1000.0)) and (g == 0).sum() == 1 and (g > 0).sum() > 100
    gpu.close()


@pytest.mark.parametrize("world", [1, 2])
def test_sharded_ranks_refuse_reach(world):
    """a rank of a world-2 sharded map holds only its own subboxes: MLM_ERR_UNSUPPORTED; a world-1 shard answers"""
    from mlmapping_b200.sharded import sharded_group_in_process
    cfg = _lidar_small_cfg()
    ranks = sharded_group_in_process(cfg, world)
    try:
        for r in ranks:
            if world == 1:
                assert r.map.build_reach([0.0, 0.0, 0.0], [4.0, 4.0, 2.0], [[1.0, 1.0, 1.0]], 3.0, unknown=True) == 1
                assert r.map.reach_cost([[1.0, 1.0, 1.0]])[0] == 0.0
                continue
            with pytest.raises(MlmError) as ei:
                r.map.build_reach([0.0, 0.0, 0.0], [4.0, 4.0, 2.0], [[1.0, 1.0, 1.0]], 3.0)
            assert ei.value.code == 6
            with pytest.raises(MlmError) as ei:
                r.map.reach_cost([[1.0, 1.0, 1.0]])
            assert ei.value.code == 6
    finally:
        for r in ranks:
            r.close()
