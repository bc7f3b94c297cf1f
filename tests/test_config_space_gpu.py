"""GPU parity across the configuration space that mlm_create accepts (tests/config_space.py): every named case against
the oracle (the reference's own sources when oracle/_ref is available, else the restatement) frame by frame with
bit-exact log-odds, then queries on random positions and on the voxel lattice, box clearing, inflation and the clouds;
the derived features at subbox sizes 3, 7 and 16; checkpoint, dirty-block replication and sharding at n = 7; the
frame kernel at small SM budgets; the pool and subbox-range limits of the library."""
import ctypes as C

import numpy as np
import pytest

import config_space as cs
from mlmapping_b200 import MLMap, config_cfg_a, scenes
from mlmapping_b200.capi import MlmError
from oracle_binding import best_oracle as Oracle
from parity_utils import assert_cloud_parity, assert_frame_parity, assert_map_parity

pytestmark = pytest.mark.gpu
POOL_EXHAUSTED, INVALID_ARG, INVALID_CONFIG = 4, 1, 2


def _bit_exact(gpu, orc, tag):
    info = assert_map_parity(gpu, orc, 0.0, tag=tag)
    assert info["log_odds_bit_exact"], (tag, info)
    return info


def _run(case, cfg, gpu, orc, tag):
    """the case's frames in lock step, frame sets and the whole map compared after every frame"""
    stats = []
    for k, (kind, data, pose) in enumerate(cs.frames(case, cfg)):
        st_g, st_o = cs.integrate(gpu, kind, data, pose), cs.integrate(orc, kind, data, pose)
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"{tag}-frame{k}")
        _bit_exact(gpu, orc, f"{tag}-frame{k}")
        stats.append((st_o, data, pose))
    return stats


def _aabb(m, cfg):
    dg = cfg.subbox_n * cfg.subbox_d_xyz
    return m["glb"].min(0) * dg, (m["glb"].max(0) + 1) * dg


def _lattice(lo, hi, d, rs, n=4000):
    """k * d on every axis inside [lo, hi], the doubles one ulp to either side, and the negatives of all of them"""
    k = np.stack([rs.randint(int(np.floor(lo[i] / d)), int(np.ceil(hi[i] / d)) + 1, n) for i in range(3)], 1)
    p = k * d
    pts = np.concatenate([p, np.nextafter(p, np.inf), np.nextafter(p, -np.inf)])
    return np.concatenate([pts, -pts])


def _check_queries(gpu, orc, cfg, tag):
    m = orc.export_map()
    lo, hi = _aabb(m, cfg)
    d = cfg.subbox_d_xyz
    pos = np.concatenate([scenes.query_positions(50000, lo, hi, seed=5, inflate=2.0),
                          _lattice(lo, hi, d, np.random.RandomState(7))])
    og, oo = gpu.getOccupancy(pos), orc.getOccupancy(pos)
    assert np.array_equal(og, oo), (tag, "getOccupancy", int((og != oo).sum()))
    assert (oo == 0).sum() > 0 and ((oo == 1).sum() > 0 or not cfg.use_raycasting), (tag, "no occupied / free cell")
    g, o = gpu.getOdd(pos), orc.getOdd(pos)
    ulps = np.abs(g.view(np.int32).astype(np.int64) - o.view(np.int32).astype(np.int64))
    assert ulps.max() <= 1, (tag, "getOdd", int(ulps.max()))
    n = cfg.subbox_n
    for it in sorted({1, 5, n // 2 + 1, n + 1, 2 * n + 1}):
        sub = pos[::4]
        dg = np.abs(gpu.getOddGrad(sub, it) - orc.getOddGrad(sub, it)).max()
        assert dg <= 1e-6, (tag, "getOddGrad", it, dg)
    r = 1.5 * d
    assert np.array_equal(gpu.getOccupancy(pos, inflate=r), orc.getOccupancy(pos, inflate=r)), (tag, "inflate query")
    return pos


def _check_edits(gpu, orc, cfg, pose, pos, tag):
    m = orc.export_map()
    lo, hi = _aabb(m, cfg)
    d = cfg.subbox_d_xyz
    # corners inside subboxes (and off the voxel lattice)
    mid, ext = (lo + hi) / 2, (hi - lo)
    b0, b1 = mid - 0.23 * ext + 0.37 * d, mid + 0.19 * ext + 0.61 * d
    gpu.setFree_map_in_bound(b0, b1)
    orc.setFree_map_in_bound(b0, b1)
    _bit_exact(gpu, orc, f"{tag}-setfree")
    gpu.inflate_map(pose[:3])
    orc.inflate_map(pose[:3])
    _bit_exact(gpu, orc, f"{tag}-inflate")
    assert np.array_equal(gpu.getInflateOccupancy(pos), orc.getInflateOccupancy(pos)), (tag, "getInflateOccupancy")
    # odds slices at cell-centre heights of this lattice
    heights = tuple((np.floor(z / d) + 0.5) * d for z in (0.35, 0.95, 1.45))
    sizes = assert_cloud_parity(gpu, orc, kinds=(0, 1, 2) if cfg.use_exploration_frontiers else (0, 1),
                                heights=heights, tag=tag)
    assert sizes[1] > 0 and sum(sizes[("slice", h)] for h in heights) > 0, (tag, sizes)
    return sizes


def _edge(case, cfg, stats, orc, sizes):
    """each case proves it reached the edge it names"""
    m = orc.export_map()
    name = case.name
    assert m["glb"].shape[0] > 0 and all(st.n_inside > 0 for st, _, _ in stats), name
    if name == "no_raycast":
        assert all(st.n_miss_cells == 0 and st.n_cast == 0 for st, _, _ in stats)
    else:
        assert sum(st.n_miss_cells for st, _, _ in stats) > 0, name
    if name == "default_yaml":
        assert all(st.n_points == cfg.sample_cnt == 500 for st, _, _ in stats)
    if name == "fine_cells":
        # the oracle's hit list of the last frame, counted per voxel: the fusion's list-walk branch (> 16 per voxel)
        keys, _ = orc.last_frame_hits()
        assert cs.hits_per_voxel(cfg, keys, stats[-1][2]).max() > 16
    if name.startswith("explore_"):
        nbytes = m["frontier"].shape[1]
        assert np.unpackbits(m["frontier"]).sum() > 100
        if name == "explore_n7":
            assert m["collapsed"].sum() > 0
            assert np.unpackbits(m["frontier"][:, (nbytes - 1) // 4 * 4:]).sum() > 0   # the partial last word
        assert sizes[2] > 0
    if name == "far_origin":
        assert m["glb"][:, 1].max() < -4000 / (cfg.subbox_n * cfg.subbox_d_xyz)
    if name == "log_odds":
        lo = m["log_odds"][m["collapsed"] == 0]
        assert lo.max() == np.float32(cfg.log_odds_max)   # the clamp is reached
        assert (m["occupancy"] == b"o").sum() > 0
    if name in ("inflate_n1", "inflate_n3"):
        assert (m["inflate"] == b"o").sum() > (m["occupancy"] == b"o").sum()


@pytest.mark.parametrize("name", [c.name for c in cs.CASES])
def test_case_matches_the_oracle(name):
    case = cs.BY_NAME[name]
    cfg = cs.config_of(case)
    if name == "default_yaml":
        libc = C.CDLL("libc.so.6")
        libc.srand(1)   # the oracle draws from libc's global stream like the reference; the handle owns a seed-1 stream
    gpu, orc = MLMap(cfg), Oracle(cfg)
    stats = _run(case, cfg, gpu, orc, name)
    pos = _check_queries(gpu, orc, cfg, name)
    sizes = _check_edits(gpu, orc, cfg, stats[-1][2], pos, name)
    _edge(case, cfg, stats, orc, sizes)


def test_refusals_match_the_python_precondition():
    """the configurations for which K(rho) <= min(10, rho) fails are refused by mlm_create; noise_wide's value is the
    largest accepted one.  Also the device-side limit of the projection: its per-column histogram holds at most about
    3000 work columns, so 0.1 degree sectors (3600 columns) are refused where 0.125 degrees (2880) run."""
    cfg = cs.BY_NAME["noise_wide"].make()
    MLMap(cfg).close()
    bad = cfg.copy()
    bad.depth_noise_coe = np.nextafter(cfg.depth_noise_coe, np.inf) * (1 + 1e-9)
    crash = config_cfg_a()
    crash.am_d_rho, crash.am_n_rho = 0.02, 300
    for c in (bad, crash):
        with pytest.raises(MlmError) as e:
            MLMap(c)
        assert e.value.code == INVALID_CONFIG and "depth_noise_coe" in str(e.value)
    phi = cs.BY_NAME["phi0_125"].make()
    phi.am_d_phi_deg = 0.1
    with pytest.raises(MlmError) as e:
        MLMap(phi)
    assert e.value.code == INVALID_CONFIG and "shared-memory histogram" in str(e.value)


# ---- derived features at other subbox sizes ---------------------------------------------------------------------

def _explore_n(n):
    cfg = config_cfg_a()
    cfg.subbox_n, cfg.use_exploration_frontiers = n, 1
    return cfg


@pytest.mark.parametrize("n", [3, 7, 16])
def test_derived_features_at_subbox_size(n):
    from esdf_oracle import EsdfOracle
    from esdf_spec import first_difference as esdf_diff, query_points, same_bits
    from frontier_oracle import FrontierOracle
    from raycast_spec import FREE, OCCUPIED, edge_segments, first_difference, random_segments
    from test_frontier_gpu import _assert_gpu_equals_oracle
    from test_view_gpu import fuel_views, sensor_of
    from view_oracle import ViewOracle
    cfg = _explore_n(n)
    gpu, eo, fo, vo = MLMap(cfg), EsdfOracle(cfg), FrontierOracle(cfg), ViewOracle(cfg)
    for k in range(6):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, rows=240, cols=320, frame_idx=k)
        for m in (gpu, eo, fo, vo):
            m.integrate_depth(img, pose)
    for m in (gpu, eo, fo, vo):
        m.inflate_map(pose[:3])
    _bit_exact(gpu, eo, f"n{n}")
    ex = eo.export_map()
    d = cfg.subbox_d_xyz
    lo, hi = _aabb(ex, cfg)
    # rays on both layers
    f1, t1 = random_segments(20000, lo, hi, seed=n, max_len=4.0)
    f2, t2 = edge_segments(ex, n, d, seed=n + 7, n_each=200)
    f, t = np.concatenate([f1, f2]), np.concatenate([t1, t2])
    for inflated in (False, True):
        g, o = gpu.cast_rays(f, t, inflated=inflated), eo.cast_rays(f, t, inflated=inflated)
        assert first_difference(g, o) is None, (n, inflated, first_difference(g, o))
        assert (g["status"] == FREE).sum() > 100 and (g["status"] == OCCUPIED).sum() > 100
    # distance field on a box whose faces cut through subboxes
    c = pose[:3]
    b0, b1 = c - [0.37 * n * d, 1.43, 1.31], c + [2.0 + 0.41 * n * d, 1.39, 1.29]
    for inflated in (False, True):
        gpu.build_esdf(b0, b1, 1.0, inflated=inflated)
        eo.build_esdf(b0, b1, 1.0, inflated=inflated)
        g, glo = gpu.export_esdf()
        o, olo = eo.export_esdf()
        assert np.array_equal(glo, olo) and same_bits(g, o), (n, inflated, esdf_diff(g, o))
        assert (g <= 0).sum() > 0 and (g > 0).sum() > 0
        pts = query_points(glo.astype(np.int64), np.array(g.shape[::-1]), d, 20000, n)
        gd, gg = gpu.esdf_distance(pts)
        od, og = eo.esdf_distance(pts)
        assert same_bits(gd, od) and same_bits(gg, og), (n, inflated)
    # frontier clusters, 6- and 26-connected
    _bit_exact(gpu, fo, f"n{n}-frontier")
    _assert_gpu_equals_oracle(gpu, fo, cfg, f"n{n}")
    assert gpu.frontier_clusters()["n_cells"].sum() > 0
    # view gain
    poses, boxes = fuel_views(gpu, cfg, seed=n)
    S = sensor_of("cfg-a", 2.5)
    for frontier in (False, True):
        for b in (None, boxes):
            g, o = gpu.view_gain(poses, S, b, frontier, False), vo.view_gain(poses, S, b, frontier, False)
            assert g.tobytes() == o.tobytes(), (n, frontier, b is None)
            assert g["n_target"].sum() > 0


# ---- checkpoint, replication and sharding at n = 7 ------------------------------------------------------------

def test_dirty_records_at_n7():
    """dirty-block shipping at n = 7: the record sizes of the dirty blocks and of the checkpoint follow the cell count
    (343 cells, not a multiple of 16), and export / import rebuilds the owner's map bit for bit.  Exploration mode refuses it (frontier sets and collapses
    are not shipped)."""
    cfg = cs.BY_NAME["n7"].make()
    a, rep, orc = MLMap(cfg), MLMap(cfg), Oracle(cfg)
    lib = a._lib
    sizes = []
    for k in range(6):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        a.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
        n, rb = C.c_int32(), C.c_size_t()
        a._check(lib.mlm_dirty_count(a._h, C.byref(n), C.byref(rb)))
        assert n.value > 0
        buf = a.device_alloc(n.value * rb.value)
        a._check(lib.mlm_dirty_export(a._h, buf, n.value))
        rep._check(lib.mlm_dirty_import(rep._h, buf, n.value))
        a.device_free(buf)
        sizes.append((a.export_map()["glb"].shape[0], len(a.checkpoint()), rb.value))
    # records of 6 bytes per cell behind a 16-byte dirty header / a 32-byte checkpoint header, padded to 16 bytes
    (s0, c0, _), (s1, c1, rb) = sizes[0], sizes[-1]
    cells = cfg.subbox_n ** 3
    assert rb == (16 + 6 * cells + 15) // 16 * 16 == 2080
    assert s1 > s0 and (c1 - c0) == (s1 - s0) * ((32 + 6 * cells + 15) // 16 * 16), sizes
    ma, mr = a.export_map(), rep.export_map()
    for name in ma:
        assert np.array_equal(ma[name].view(np.uint8), mr[name].view(np.uint8)), ("replica", name)
    _bit_exact(rep, orc, "n7-replica")
    ex = MLMap(_explore_n(7))
    n, rb = C.c_int32(), C.c_size_t()
    assert lib.mlm_dirty_count(ex._h, C.byref(n), C.byref(rb)) == 6 and b"exploration" in lib.mlm_last_error()


def test_checkpoint_restore_at_n7_with_exploration():
    """checkpoint / restore into a handle with another pool size, two more frames in lock step with the oracle"""
    cfg = _explore_n(7)
    a, orc = MLMap(cfg), Oracle(cfg)
    for k in range(8):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        a.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    ma = a.export_map()
    _bit_exact(a, orc, "n7-before")
    assert ma["collapsed"].sum() > 0
    cfg_b = cfg.copy()
    cfg_b.pool_submaps = ma["glb"].shape[0] + 37
    b = MLMap(cfg_b)
    b.restore(a.checkpoint())
    mb = b.export_map()
    for name in ma:
        assert np.array_equal(ma[name].view(np.uint8), mb[name].view(np.uint8)), ("restored", name)
    for k in range(8, 10):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        st_b, st_o = b.integrate_depth(img, pose), orc.integrate_depth(img, pose)
        assert_frame_parity(b, orc, st_b, st_o, tag=f"n7-restored{k}")
        _bit_exact(b, orc, f"n7-restored{k}")


def test_sharded_lidar_map_at_n7():
    """2 ranks of one process on one GPU: subbox ownership goes through a floor division by n = 7"""
    from mlmapping_b200.sharded import sharded_group_in_process
    from test_parity_gpu import assert_union_equals_oracle
    cfg = cs.BY_NAME["phi5"].make()
    cfg.am_d_phi_deg, cfg.subbox_n = 1.0, 7
    ranks, orc = sharded_group_in_process(cfg, 2), Oracle(cfg)
    for k in range(4):
        pose = scenes.lidar_loop_pose(k * 3)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512)
        for r in ranks:
            r.submit(pts, pose)
        stats = [r.finish() for r in ranks]
        st_o = orc.integrate_points(pts, pose)
        assert all(st.n_hit_cells == st_o.n_hit_cells for st in stats)
        owned = assert_union_equals_oracle(ranks, orc, f"n7-shard{k}")
    assert min(owned) > 0
    for r in ranks:
        r.close()


# ---- launch shape -----------------------------------------------------------------------------------------------

@pytest.mark.parametrize("scenario", ["cfg_a", "lidar", "explore"])
def test_small_sm_budgets(scenario):
    """the frame kernel with 1, 2, 3, 7 CTAs and with one per SM: the work queue, the light-column merge and the
    device-wide barrier with several items per CTA give the same map bit for bit (the budget applies to the fused
    frame kernel of both modes; frames that settle a rehash run the stand-alone passes, which do not take it)"""
    if scenario == "lidar":
        case = cs.Case("lidar", lambda: _with(cs.BY_NAME["phi5"].make(), am_d_phi_deg=1.0), scene="lidar", frames=3)
    elif scenario == "explore":
        case = cs.Case("explore", lambda: _with(config_cfg_a(), use_exploration_frontiers=1), rows=480, cols=640,
                       frames=4)
    else:
        case = cs.Case("cfg_a", config_cfg_a, rows=480, cols=640, frames=3)
    cfg = case.make()
    maps = []
    for b in (1, 2, 3, 7, 0):
        gpu, orc = MLMap(cfg), Oracle(cfg)
        gpu.set_sm_budget(b)
        _run(case, cfg, gpu, orc, f"{scenario}-sms{b}")
        maps.append(gpu.export_map())
    for m in maps[1:]:
        for name in m:
            assert np.array_equal(m[name].view(np.uint8), maps[0][name].view(np.uint8)), (scenario, name)


def _with(cfg, **kw):
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


# ---- pool and range limits --------------------------------------------------------------------------------------

def _pool_frames(cfg):
    out = []
    for k in range(6):
        pose = scenes.corridor_trajectory_pose(k * 10)
        out.append((scenes.corridor_depth_frame(cfg, pose, rows=240, cols=320, frame_idx=k), pose))
    return out


def test_pool_of_exactly_the_subbox_count():
    """without exploration no block is ever returned: a pool of the oracle's final subbox count runs the scenario; one
    block less fails on the first frame whose cumulative allocation exceeds it, and not earlier; the handle stays
    usable, its blocks hold the oracle's values, and a later frame that touches the unusable subbox fails again"""
    cfg = cs.BY_NAME["n7"].make()
    frames = _pool_frames(cfg)
    orc = Oracle(cfg)
    expand = [orc.integrate_depth(img, pose).ram_expand_cnt for img, pose in frames]
    total = orc.export_map()["glb"].shape[0]
    assert expand[-1] == total and expand[0] < total
    cfg.pool_submaps = total
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k, (img, pose) in enumerate(frames):
        assert_frame_parity(gpu, orc, gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose), tag=f"exact{k}")
    _bit_exact(gpu, orc, "exact-pool")
    cfg.pool_submaps = total - 1
    gpu, orc = MLMap(cfg), Oracle(cfg)
    first_over = next(k for k, e in enumerate(expand) if e > total - 1)
    for k, (img, pose) in enumerate(frames[:first_over]):
        assert_frame_parity(gpu, orc, gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose), tag=f"short{k}")
    img, pose = frames[first_over]
    orc.integrate_depth(img, pose)
    with pytest.raises(MlmError) as e:
        gpu.integrate_depth(img, pose)
    assert e.value.code == POOL_EXHAUSTED
    # still usable: queries and the export return, and every subbox that holds a block has the oracle's values
    m = orc.export_map()
    gpu.getOccupancy(scenes.query_positions(10000, *_aabb(m, cfg), seed=3))
    g = gpu.export_map()
    assert g["glb"].shape[0] == total - 1
    idx = {tuple(r): i for i, r in enumerate(m["glb"])}
    rows = np.array([idx[tuple(r)] for r in g["glb"]])
    for name in ("collapsed", "occupancy", "inflate"):
        assert np.array_equal(g[name], m[name][rows]), name
    assert np.array_equal(g["log_odds"].view(np.uint32), m["log_odds"][rows].view(np.uint32))
    with pytest.raises(MlmError) as e:
        gpu.integrate_depth(img, pose)
    assert e.value.code == POOL_EXHAUSTED


def test_pool_that_only_recycling_makes_enough():
    """exploration mode returns the blocks of collapsed subboxes: a pool of the peak live-block count (from the oracle:
    live blocks after the previous frame + the frame's new subboxes), below the number of subboxes ever created, runs
    the scenario bit for bit, frontier words of reused blocks included"""
    cfg = _explore_n(7)
    frames = [(scenes.corridor_depth_frame(cfg, p, frame_idx=k), p)
              for k, p in enumerate(scenes.corridor_trajectory_pose(k * 10) for k in range(14))]
    orc = Oracle(cfg)
    live_prev = peak = prev = 0
    for img, pose in frames:
        st = orc.integrate_depth(img, pose)
        m = orc.export_map()
        peak = max(peak, live_prev + st.ram_expand_cnt - prev)
        live_prev, prev = int(m["glb"].shape[0] - m["collapsed"].sum()), st.ram_expand_cnt
    created = m["glb"].shape[0]
    cfg.pool_submaps = peak + 4
    assert cfg.pool_submaps < created, (peak, created)
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k, (img, pose) in enumerate(frames):
        st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"recycle{k}")
        _bit_exact(gpu, orc, f"recycle{k}")
    assert orc.export_map()["collapsed"].sum() > 0


def test_subbox_index_range():
    """subbox indices are limited to +-2^20 per axis: at n = 2, d_sub = 0.1 the limit is y = -209715.2 m.  The first
    corridor frame maps y0 .. y0 + 1.2 m: with y0 half a metre below the limit the frame straddles it and fails with
    MLM_ERR_INVALID_ARG instead of aliasing keys; half a metre above it the frame matches the oracle"""
    cfg = cs.BY_NAME["n2"].make()
    limit = -(2 ** 20) * cfg.subbox_n * cfg.subbox_d_xyz
    cfg.pool_submaps = 1 << 14
    for y0, ok in ((limit + 0.5, True), (limit - 0.5, False)):
        case = cs.Case("range", lambda: cfg, frames=1, y_offset=y0)
        gpu, orc = MLMap(cfg), Oracle(cfg)
        (kind, img, pose), = cs.frames(case, cfg)
        st_o = orc.integrate_depth(img, pose)
        g = orc.export_map()["glb"][:, 1]
        if ok:
            assert g.min() >= -(2 ** 20)
            assert_frame_parity(gpu, orc, gpu.integrate_depth(img, pose), st_o, tag="inside")
            _bit_exact(gpu, orc, "inside")
        else:
            assert g.min() < -(2 ** 20) <= g.max()
            with pytest.raises(MlmError) as e:
                gpu.integrate_depth(img, pose)
            assert e.value.code == INVALID_ARG
