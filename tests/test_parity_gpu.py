"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on identical seeded
inputs.  Bar (BASELINE.json north_star): per-frame hit/miss cell sets, allocated subboxes and
occupancy states bit-exact; log-odds within 1e-6 absolute (tolerance written here: LO_TOL)."""
import numpy as np
import pytest

from mlmapping_b200 import MLMap, config_cfg_a, config_cfg_c, scenes
from mlmapping_b200.capi import MlmError
from oracle_binding import best_oracle as Oracle  # the reference's own sources when oracle/_ref is there, else the restatement
from parity_utils import assert_cloud_parity, assert_frame_parity, assert_map_parity

pytestmark = pytest.mark.gpu
LO_TOL = 1e-6


def _small_cfg():
    c = config_cfg_a()
    return c


def test_single_frame_cfg_a():
    """BASELINE config 1: one 640x480 frame of the box corridor, body at (5,0,1.2), yaw 0"""
    cfg = config_cfg_a()
    pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0)
    img = scenes.corridor_depth_frame(cfg, pose)
    gpu, orc = MLMap(cfg), Oracle(cfg)
    st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
    assert st_g.ordering_slow_path == 1  # first frame of a fresh map always crosses libstdc++ rehashes
    assert_frame_parity(gpu, orc, st_g, st_o, tag="frame0")
    info = assert_map_parity(gpu, orc, LO_TOL)
    assert info["subboxes"] > 0
    # same frame again: steady-state (no rehash) ordering path, saturating updates
    st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
    assert st_g.ordering_slow_path == 0
    assert_frame_parity(gpu, orc, st_g, st_o, tag="frame0-again")
    assert_map_parity(gpu, orc, LO_TOL)


def test_trajectory_cfg_a():
    """BASELINE config 2 (first 40 frames): streaming allocate as the body moves and yaws"""
    cfg = config_cfg_a()
    gpu, orc = MLMap(cfg), Oracle(cfg)
    exact = []
    for k in range(40):
        pose = scenes.corridor_trajectory_pose(k * 5)  # stride 5 -> 0.25 m steps, new subboxes every few frames
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"frame{k}")
        if k % 10 == 9:
            exact.append(assert_map_parity(gpu, orc, LO_TOL, tag=f"frame{k}"))
    assert exact[-1]["subboxes"] > 100


def test_strided_image_and_rotated_pose():
    """row stride != cols*2 and a pose with roll/pitch (phi columns no longer follow image columns)"""
    cfg = config_cfg_a()
    pose = np.array([7.0, 0.2, 1.0, 0.9, 0.1, -0.15, 0.3])
    img_full = np.zeros((480, 704), dtype=np.uint16)
    img_full[:, :640] = scenes.corridor_depth_frame(cfg, pose, frame_idx=3)
    view = img_full[:, :640]
    gpu, orc = MLMap(cfg), Oracle(cfg)
    st_g, st_o = gpu.integrate_depth(view, pose), orc.integrate_depth(np.ascontiguousarray(view), pose)
    assert_frame_parity(gpu, orc, st_g, st_o)
    assert_map_parity(gpu, orc, LO_TOL)


def test_point_cloud_input_lidar_small():
    """input_pc_pose on sensor-frame points (LiDAR-like), reduced CFG-C grid"""
    cfg = config_cfg_c()
    cfg.am_n_rho, cfg.am_n_z_below, cfg.am_n_z_over = 120, 30, 30
    cfg.max_points = 32 * 512
    cfg.pool_submaps = 8192
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k in range(3):
        pose = scenes.lidar_loop_pose(k * 3)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512)
        st_g, st_o = gpu.integrate_points(pts, pose), orc.integrate_points(pts, pose)
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"scan{k}")
    assert_map_parity(gpu, orc, LO_TOL)


def test_empty_and_degenerate_frames():
    cfg = config_cfg_a()
    gpu, orc = MLMap(cfg), Oracle(cfg)
    pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0)
    zero = np.zeros((480, 640), dtype=np.uint16)
    st_g, st_o = gpu.integrate_depth(zero, pose), orc.integrate_depth(zero, pose)
    assert st_g.n_points == 0 and st_o.n_points == 0
    assert_frame_parity(gpu, orc, st_g, st_o)
    # a single valid pixel, then a ragged small image
    one = zero.copy()
    one[240, 320] = 2500
    st_g, st_o = gpu.integrate_depth(one, pose), orc.integrate_depth(one, pose)
    assert_frame_parity(gpu, orc, st_g, st_o)
    small = scenes.corridor_depth_frame(cfg, pose, rows=37, cols=53)
    st_g, st_o = gpu.integrate_depth(small, pose), orc.integrate_depth(small, pose)
    assert_frame_parity(gpu, orc, st_g, st_o)
    # maximum depth everywhere: every ray is outside the awareness range and is clamped
    far = np.full((480, 640), 65535, dtype=np.uint16)
    st_g, st_o = gpu.integrate_depth(far, pose), orc.integrate_depth(far, pose)
    assert st_g.n_inside == 0
    assert_frame_parity(gpu, orc, st_g, st_o)
    assert_map_parity(gpu, orc, LO_TOL)
    with pytest.raises(MlmError):
        gpu.integrate_depth(np.zeros((481, 640), dtype=np.uint16), pose)  # exceeds cfg.max_points


def test_queries_and_set_free():
    cfg = config_cfg_a()
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k in range(6):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    m = orc.export_map()
    lo = m["glb"].min(0) * cfg.subbox_d_xyz * cfg.subbox_n
    hi = (m["glb"].max(0) + 1) * cfg.subbox_d_xyz * cfg.subbox_n
    pos = scenes.query_positions(200000, lo, hi, seed=5, inflate=2.0)
    # cell-boundary and exact-lattice positions exercise the floor()/division quirks
    lattice = np.round(pos[:20000] / cfg.subbox_d_xyz) * cfg.subbox_d_xyz
    pos = np.concatenate([pos, lattice, -lattice[:100]])
    assert np.array_equal(gpu.getOccupancy(pos), orc.getOccupancy(pos))
    og, oo = gpu.getOdd(pos), orc.getOdd(pos)
    assert np.abs(og.astype(np.float64) - oo.astype(np.float64)).max() <= 1.2e-7  # <= 1 float ulp of odds in [0.5,1]
    gg, go = gpu.getOddGrad(pos[:100000]), orc.getOddGrad(pos[:100000])
    assert np.abs(gg - go).max() <= 1e-6
    # one-step walks, walks that stay inside a subbox less often, and walks longer than a subbox (several borders crossed)
    for it in (1, 3, cfg.subbox_n + 3, 2 * cfg.subbox_n + 1):
        q = pos[100000:140000]
        assert np.abs(gpu.getOddGrad(q, it) - orc.getOddGrad(q, it)).max() <= 1e-6, it
    assert np.array_equal(gpu.getOccupancy(pos[:50000], 0.15), orc.getOccupancy(pos[:50000], 0.15))
    # setFree_map_in_bound, then everything again
    bmin, bmax = [5.0, -0.5, 0.3], [8.0, 0.5, 2.0]
    gpu.setFree_map_in_bound(bmin, bmax)
    orc.setFree_map_in_bound(bmin, bmax)
    assert_map_parity(gpu, orc, LO_TOL)
    assert np.array_equal(gpu.getOccupancy(pos), orc.getOccupancy(pos))


def test_log10f_matches_host_glibc():
    """device log10f == this box's glibc log10f on every float in [2^-14, 2^27) (the logit() domain
    p/(1-p), p in [0.001, 1)) plus a strided sweep of all positive floats"""
    from oracle_binding import load_oracle
    lib = load_oracle()
    cfg = config_cfg_a()
    gpu = MLMap(cfg)
    lo_bits, hi_bits = np.float32(2.0 ** -14).view(np.uint32), np.float32(2.0 ** 27).view(np.uint32)
    total_bad = 0
    chunk = 1 << 24
    for start in range(int(lo_bits), int(hi_bits), chunk):
        bits = np.arange(start, min(start + chunk, int(hi_bits)), dtype=np.uint32)
        x = bits.view(np.float32)
        ref = np.empty_like(x)
        lib.orc_log10f_array(x.ctypes.data, x.size, ref.ctypes.data)
        got = gpu.debug_log10f(x)
        total_bad += int((got.view(np.uint32) != ref.view(np.uint32)).sum())
    assert total_bad == 0
    bits = np.arange(1, 0x7F800000, 997, dtype=np.uint32)  # subnormals .. max finite
    x = bits.view(np.float32)
    ref = np.empty_like(x)
    lib.orc_log10f_array(x.ctypes.data, x.size, ref.ctypes.data)
    got = gpu.debug_log10f(x)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_fallback_paths_global_sort_spill_and_oversized_columns(monkeypatch):
    """shrink the shared-memory capacities (debug env hooks) so columns take the global-memory sort
    spill and the record-copy path; results must not change"""
    cfg = config_cfg_a()
    frames = []
    for k in range(3):
        pose = scenes.corridor_trajectory_pose(40 * k)
        frames.append((scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose))
    for env in ({"MLM_DEBUG_SORT_CAP": "256"}, {"MLM_DEBUG_MAP_CAP": "64"},
                {"MLM_DEBUG_SORT_CAP": "128", "MLM_DEBUG_MAP_CAP": "1"}):
        for k_, v_ in env.items():
            monkeypatch.setenv(k_, v_)
        gpu, orc = MLMap(cfg), Oracle(cfg)
        for k_ in env:
            monkeypatch.delenv(k_)
        for i, (img, pose) in enumerate(frames):
            st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
            assert_frame_parity(gpu, orc, st_g, st_o, tag=f"{env} frame{i}")
        assert_map_parity(gpu, orc, LO_TOL)


def test_alternative_launch_paths_give_the_same_map(monkeypatch):
    """the frame runs as one cooperative k_frame launch by default; the three stand-alone kernels (graph or direct
    launches, the latter as profiling runs them) and whole-column work items (no split at the sensor row) must give the
    same cell sets and map"""
    cfg = config_cfg_a()
    frames = []
    for k in range(3):
        pose = scenes.corridor_trajectory_pose(35 * k)
        frames.append((scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose))
    for env, direct in (({"MLM_NO_FUSED": "1"}, False), ({"MLM_DEBUG_NO_SPLIT": "1"}, False),
                        ({"MLM_NO_FUSED": "1"}, True), ({"MLM_NO_FUSED": "1", "MLM_DEBUG_NO_SPLIT": "1"}, False)):
        for k_, v_ in env.items():
            monkeypatch.setenv(k_, v_)
        gpu, orc = MLMap(cfg), Oracle(cfg)
        for k_ in env:
            monkeypatch.delenv(k_)
        gpu.set_profiling(direct)
        for i, (img, pose) in enumerate(frames):
            st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
            assert_frame_parity(gpu, orc, st_g, st_o, tag=f"{env} direct={direct} frame{i}")
        expected_launches = 3 * len(frames) if "MLM_NO_FUSED" in env else len(frames)
        assert gpu.kernel_launch_count() >= expected_launches
        assert_map_parity(gpu, orc, LO_TOL)


def test_full_size_cfg_b_l515_like():
    """BASELINE config 3 geometry at full size: 1024x768 @ 0.05 m, n_Rho 180, n_Z 81 (3 frames)"""
    from mlmapping_b200 import config_cfg_b
    cfg = config_cfg_b()
    cfg.pool_submaps = 32768
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k in range(3):
        pose = scenes.corridor_trajectory_pose(k * 20, step=0.1)
        img = scenes.corridor_depth_frame(cfg, pose, rows=768, cols=1024, frame_idx=k, length=200.0)
        st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"cfgB frame{k}")
    assert_map_parity(gpu, orc, LO_TOL)


def test_full_size_cfg_c_lidar():
    """BASELINE config 4 geometry at full size: 128x2048 LiDAR scan, n_Rho 250, n_Z 201, 0.2 m voxels"""
    cfg = config_cfg_c()
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k in range(2):
        pose = scenes.lidar_loop_pose(k * 5)
        pts = scenes.lidar_scan(pose, frame_idx=k)
        st_g, st_o = gpu.integrate_points(pts, pose), orc.integrate_points(pts, pose)
        assert st_g.n_points > 200000
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"cfgC scan{k}")
    assert_map_parity(gpu, orc, LO_TOL)


def test_inflate_map_and_inflate_occupancy():
    """inflate_map (src/mlmap.cpp:286-309) incl. the wipe-by-later-reset order rule, cross-subbox stamps that
    allocate neighbours, repeated calls at moving centres, getInflateOccupancy"""
    cfg = config_cfg_a()
    cfg.inflate_n, cfg.inflate_global_n = 2, 2
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k in range(8):
        pose = scenes.corridor_trajectory_pose(k * 12)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
        if k % 3 == 2:
            gpu.inflate_map(pose[:3])
            orc.inflate_map(pose[:3])
            assert_map_parity(gpu, orc, LO_TOL, tag=f"inflate@{k}")
    st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
    assert st_g.ram_expand_cnt == st_o.ram_expand_cnt   # inflate_atpos allocations are counted too
    m = orc.export_map()
    assert (m["inflate"] == b"o").sum() > 1000
    lo = m["glb"].min(0) * 1.0
    hi = (m["glb"].max(0) + 1) * 1.0
    pos = scenes.query_positions(200000, lo, hi, seed=7, inflate=1.0)
    assert np.array_equal(gpu.getInflateOccupancy(pos), orc.getInflateOccupancy(pos))
    # centre far from the data: empty window, nothing may change
    gpu.inflate_map([100.0, 0.0, 0.0])
    orc.inflate_map([100.0, 0.0, 0.0])
    assert_map_parity(gpu, orc, LO_TOL, tag="inflate-empty-window")
    # the clouds the reference publishes from this map: inflated / occupied cells and two odds slices
    sizes = assert_cloud_parity(gpu, orc, kinds=(0, 1), tag="inflate")
    assert sizes[0] > 1000 and sizes[1] > 100 and sizes[("slice", 0.75)] > 1000
    cap = 64  # truncated export reports the full count and writes only `cap` points
    dptr = gpu.device_alloc(16 * cap)
    assert gpu.export_cloud_device(0, dptr, cap) == sizes[0]
    gpu.device_free(dptr)


def test_sampled_project_depth_matches_glibc_rand_stream():
    """mlmapping_sample_cnt = 500 (the reference's live configuration, config_sim.yaml:37): pixels drawn with
    rand() % rows / rand() % cols, at most 2*cnt draws, zero pixels skipped (src/mlmap.cpp:321-346)"""
    import ctypes as C
    cfg = config_cfg_a()
    cfg.sample_cnt = 500
    libc = C.CDLL("libc.so.6")
    gpu, orc = MLMap(cfg), Oracle(cfg)
    libc.srand(1)  # the oracle draws from libc's global stream like the reference; the handle owns a seed-1 stream
    for k in range(12):
        pose = scenes.corridor_trajectory_pose(k * 7)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        if k == 5:
            img[::2, :] = 0          # many invalid pixels: fewer than 500 points after 1000 draws
        st_o = orc.integrate_depth(img, pose)
        st_g = gpu.integrate_depth(img, pose)
        assert st_g.n_points == st_o.n_points and (st_g.n_points == 500 or k == 5)
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"sampled{k}")
    assert_map_parity(gpu, orc, LO_TOL)


@pytest.mark.parametrize("one_launch", [True, False])
def test_exploration_frontiers_and_memory_release(one_launch, monkeypatch):
    """use_exploration_frontiers = true (config2.yaml:36): update_observation in miss-set iteration order,
    frontier sets, neighbour subbox allocation, release pass (collapse to element 0), queries on collapsed
    subboxes — SURVEY §8a a14-a15.  Once as the single cooperative launch per frame (k_frame_explore; the frames
    that cross a rehash of the hit map or the miss set fall back to the stand-alone passes), once with the
    stand-alone passes for every frame."""
    if not one_launch:
        monkeypatch.setenv("MLM_NO_FUSED", "1")
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k in range(14):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"explore{k}")
        info = assert_map_parity(gpu, orc, LO_TOL, tag=f"explore{k}")
    m = orc.export_map()
    assert m["collapsed"].sum() >= 10 and np.unpackbits(m["frontier"]).sum() > 300
    lo = m["glb"].min(0) * 1.0
    hi = (m["glb"].max(0) + 1) * 1.0
    pos = scenes.query_positions(200000, lo, hi, seed=9, inflate=1.0)
    assert np.array_equal(gpu.getOccupancy(pos), orc.getOccupancy(pos))
    assert np.abs(gpu.getOdd(pos).astype(np.float64) - orc.getOdd(pos)).max() <= 1.2e-7
    assert np.abs(gpu.getOddGrad(pos[:50000]) - orc.getOddGrad(pos[:50000])).max() <= 1e-6
    # box fill and inflation must skip collapsed subboxes like the reference
    gpu.setFree_map_in_bound([5.0, -1.0, 0.2], [9.0, 1.0, 2.2])
    orc.setFree_map_in_bound([5.0, -1.0, 0.2], [9.0, 1.0, 2.2])
    gpu.inflate_map(pose[:3])
    orc.inflate_map(pose[:3])
    assert_map_parity(gpu, orc, LO_TOL, tag="explore-setfree-inflate")
    sizes = assert_cloud_parity(gpu, orc, kinds=(0, 1, 2), tag="explore")   # incl. the frontier cloud and collapsed subboxes
    assert sizes[2] > 100


def _lidar_small_cfg():
    cfg = config_cfg_c()
    cfg.am_n_rho, cfg.am_n_z_below, cfg.am_n_z_over = 120, 30, 30
    cfg.max_points = 32 * 512
    cfg.pool_submaps = 8192
    return cfg


def _union_of_ranks(ranks):
    parts = [r.export_map() for r in ranks]
    glb = np.concatenate([p["glb"] for p in parts])
    order = np.lexsort((glb[:, 2], glb[:, 1], glb[:, 0]))
    out = {k: np.concatenate([p[k] for p in parts])[order] for k in parts[0]}
    return out, [int(p["glb"].shape[0]) for p in parts]


def assert_union_equals_oracle(ranks, orc, tag):
    """every subbox is owned by exactly one rank and the union of the owned subboxes equals the oracle map bit for bit"""
    u, owned = _union_of_ranks(ranks)
    o = orc.export_map()
    assert np.array_equal(u["glb"], o["glb"]), (tag, "union of owned subboxes differs", u["glb"].shape, o["glb"].shape, owned)
    for name in ("collapsed", "occupancy", "inflate"):
        assert np.array_equal(u[name], o[name]), (tag, name)
    assert np.array_equal(u["log_odds"].view(np.uint32), o["log_odds"].view(np.uint32)), (tag, "log_odds")
    return owned


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 4])
def test_sharded_map_ranks_on_one_gpu_match_oracle(world):
    """the sharded LiDAR map with `world` ranks: stage by phi column -> keys and update records stored straight into the
    owners' exchange arenas (peer-memory stores + system-scope flags, csrc/shard_kernels.cuh) -> device-side wait ->
    ingest + fuse.  All ranks are handles of this process on ONE GPU, so the whole exchange protocol (double-buffered
    arenas, epochs, the rehash path of the first scans, stats) runs on a single-GPU box; across processes / GPUs the
    only difference is how the arenas are mapped (tests/multi_gpu/sharded_check.py)."""
    from mlmapping_b200.sharded import sharded_group_in_process
    cfg = _lidar_small_cfg()
    ranks, orc = sharded_group_in_process(cfg, world), Oracle(cfg)
    rehash_scans = 0
    for k in range(6):
        pose = scenes.lidar_loop_pose(k * 3)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512)
        for r in ranks:
            r.submit(pts, pose)  # all ranks enqueue before any waits: their wait kernels need each other's flags
        stats = [r.finish() for r in ranks]
        st_o = orc.integrate_points(pts, pose)
        assert all(st.n_hit_cells == st_o.n_hit_cells for st in stats), (k, [st.n_hit_cells for st in stats], st_o.n_hit_cells)
        assert all(st.hit_bucket_count == st_o.hit_bucket_count for st in stats)
        assert sum(st.n_touched_voxels for st in stats) == st_o.n_touched_voxels
        assert sum(st.n_miss_cells for st in stats) == st_o.n_miss_cells and all(st.n_inside == st_o.n_inside for st in stats)
        assert sum(r.last["n_hit_local"] for r in ranks) == st_o.n_hit_cells
        assert len({r.last["rehash_path"] for r in ranks}) == 1   # every rank takes the same decision
        rehash_scans += ranks[0].last["rehash_path"]
        assert stats[0].ordering_slow_path == ranks[0].last["rehash_path"]
        assert_union_equals_oracle(ranks, orc, f"world{world}-scan{k}")
    assert 1 <= rehash_scans < 6    # the first scan(s) grow the emulated bucket array, later ones take the device-only path
    assert sum(st.ram_expand_cnt for st in stats) == st_o.ram_expand_cnt and sum(st.obs_cnt for st in stats) == st_o.obs_cnt
    owned = assert_union_equals_oracle(ranks, orc, f"world{world}")
    assert min(owned) > 0
    # a rank's answers are the oracle's wherever it owns the subbox, UNKNOWN elsewhere
    m = orc.export_map()
    pos = scenes.query_positions(50000, m["glb"].min(0) * 2.0, (m["glb"].max(0) + 1) * 2.0, seed=4)
    occ = np.stack([r.map.getOccupancy(pos) for r in ranks])
    want = orc.getOccupancy(pos)
    assert np.array_equal(occ.max(axis=0), want) and ((occ != -1).sum(axis=0) <= 1).all()
    for r in ranks:
        r.close()


@pytest.mark.gpu
def test_sharded_map_scan_handed_over_in_slices():
    """mlm_shard_submit_points_slice_f64: every rank copies only its slice of the scan from the host, the slices reach
    the other ranks' arenas through the library's scatter kernel; the map must equal the oracle's like with whole scans
    (3 ranks on one GPU; uneven and empty slices)"""
    from mlmapping_b200.sharded import sharded_group_in_process
    cfg = _lidar_small_cfg()
    world = 3
    ranks = sharded_group_in_process(cfg, world)
    orc = Oracle(cfg)
    for k in range(5):
        pose = scenes.lidar_loop_pose(k * 3)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512)
        n = pts.shape[0]
        cuts = [0, n // 5, n // 5, n] if k == 2 else [0, n // 3, (2 * n) // 3 + 7, n]   # k == 2: rank 1 has nothing to copy
        st_o = orc.integrate_points(pts, pose)
        for r, sh in enumerate(ranks):
            sh.submit_slice(pts[cuts[r]:cuts[r + 1]], cuts[r], n, pose)
        for sh in ranks:
            st = sh.finish()
            assert st.n_hit_cells == st_o.n_hit_cells and st.n_inside == st_o.n_inside
        assert_union_equals_oracle(ranks, orc, f"slices-scan{k}")
    for sh in ranks:
        sh.close()


def test_sharded_map_empty_and_tiny_scans():
    from mlmapping_b200.sharded import sharded_group_in_process
    cfg = _lidar_small_cfg()
    ranks, orc = sharded_group_in_process(cfg, 2), Oracle(cfg)
    pose = scenes.lidar_loop_pose(0)
    full = scenes.lidar_scan(pose, frame_idx=0, beams=32, azimuths=512)
    for pts in (full[:0], full[:1], full[:37], full, full[:0], full[5:9]):
        for r in ranks:
            r.submit(pts, pose)
        stats = [r.finish() for r in ranks]
        st_o = orc.integrate_points(pts, pose)
        assert all(st.n_hit_cells == st_o.n_hit_cells for st in stats)
        assert_union_equals_oracle(ranks, orc, f"n={len(pts)}")
    for r in ranks:
        r.close()


@pytest.mark.gpu
def test_sharded_map_processes_on_separate_gpus_match_oracle():
    """ranks as PROCESSES, one GPU each (arenas mapped with CUDA IPC over NVLink): tests/multi_gpu/sharded_check.py under
    torchrun on every GPU of the box (2, 4 or 8).  Skipped on a single-GPU box."""
    import subprocess
    import sys
    import torch
    n = torch.cuda.device_count()
    if n < 2:
        pytest.skip("needs at least 2 GPUs")
    world = 8 if n >= 8 else (4 if n >= 4 else 2)
    script = str(__import__("pathlib").Path(__file__).resolve().parent / "multi_gpu" / "sharded_check.py")
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
                          "--master-addr", "127.0.0.1", "--master-port", "29533", script], capture_output=True, text=True,
                         timeout=600)
    assert res.returncode == 0 and '"sharded_check": "ok"' in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]


@pytest.mark.gpu
def test_replicated_map_dirty_block_shipping_single_gpu():
    """replica kept coherent by shipping the subbox blocks each frame touched (two handles on one GPU stand in
    for two ranks; the NCCL broadcast in between is exercised by tests/multi_gpu/replicated_check.py)"""
    import ctypes as C
    cfg = config_cfg_a()
    owner, replica, orc = MLMap(cfg), MLMap(cfg), Oracle(cfg)
    lib = owner._lib
    for k in range(6):
        pose = scenes.corridor_trajectory_pose(k * 15)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        owner.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
        n, rb = C.c_int32(), C.c_size_t()
        owner._check(lib.mlm_dirty_count(owner._h, C.byref(n), C.byref(rb)))
        assert n.value > 0 and rb.value == 6016
        buf = owner.device_alloc(n.value * rb.value)
        owner._check(lib.mlm_dirty_export(owner._h, buf, n.value))
        replica._check(lib.mlm_dirty_import(replica._h, buf, n.value))
        owner.device_free(buf)
    assert_map_parity(replica, orc, LO_TOL, tag="replica")
    m = orc.export_map()
    pos = scenes.query_positions(100000, m["glb"].min(0) * 1.0, (m["glb"].max(0) + 1) * 1.0, seed=3, inflate=2.0)
    assert np.array_equal(replica.getOccupancy(pos), orc.getOccupancy(pos))
    assert np.array_equal(replica.getOddGrad(pos[:20000]), owner.getOddGrad(pos[:20000]))


@pytest.mark.gpu
def test_replicated_map_over_peer_memory_in_process():
    """mlm_replica_*: the source's kernel stores each frame's dirty blocks into the replicas' inboxes and raises the
    frame's flag, the replicas' kernels wait on the device, apply and acknowledge (three handles on one GPU stand in
    for three ranks; tests/multi_gpu/replicated_check.py runs the same over CUDA IPC between processes)"""
    from mlmapping_b200.sharded import replicated_group_in_process
    cfg = config_cfg_a()
    ranks = replicated_group_in_process(cfg, 3, src=1)
    orc = Oracle(cfg)
    for k in range(9):   # more frames than inbox halves: the acknowledgements are exercised
        pose = scenes.corridor_trajectory_pose(k * 12)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        orc.integrate_depth(img, pose)
        ranks[1].integrate_depth(img, pose)
        assert ranks[1].last["dirty_blocks"] > 0
        for r in (0, 2):
            ranks[r].integrate_depth(None, pose)
            assert ranks[r].last["dirty_blocks"] == ranks[1].last["dirty_blocks"]
    for r in (0, 2):
        assert_map_parity(ranks[r].map, orc, LO_TOL, tag=f"replica{r}")
    m = orc.export_map()
    pos = scenes.query_positions(100000, m["glb"].min(0) * 1.0, (m["glb"].max(0) + 1) * 1.0, seed=3, inflate=2.0)
    assert np.array_equal(ranks[2].map.getOccupancy(pos), orc.getOccupancy(pos))
    # out of lock step: a replica that applies without a published frame times out on the device and reports it
    import os
    os.environ["MLM_SHARD_TIMEOUT_MS"] = "50"
    try:
        lone = replicated_group_in_process(cfg, 2, src=0)
        with pytest.raises(MlmError):
            lone[1].integrate_depth(None, pose)
        for r in lone:
            r.close()
    finally:
        del os.environ["MLM_SHARD_TIMEOUT_MS"]
    for r in ranks:
        r.close()


def test_replicated_map_two_gpus_matches_oracle():
    """dirty-block broadcast over NCCL + split query stream on 2 ranks.  Skipped on a single-GPU box."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    script = str(__import__("pathlib").Path(__file__).resolve().parent / "multi_gpu" / "replicated_check.py")
    res = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                          "--master-addr", "127.0.0.1", "--master-port", "29537", script], capture_output=True, text=True,
                         timeout=600)
    assert res.returncode == 0 and '"replicated_check": "ok"' in res.stdout, res.stdout[-2000:] + res.stderr[-4000:]


@pytest.mark.gpu
def test_checkpoint_restore_round_trip_and_continuation():
    """checkpoint / restore (SURVEY 8f-4): the image restored into a second handle gives the same map bit for bit,
    and frames integrated after the restore keep matching the oracle (bucket counts, counters and the rand() stream
    travel in the header); exploration mode so that collapsed subboxes and frontier sets are covered"""
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    cfg.inflate_n, cfg.inflate_global_n = 2, 2
    a, orc = MLMap(cfg), Oracle(cfg)
    for k in range(8):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        a.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    a.inflate_map(pose[:3])
    orc.inflate_map(pose[:3])
    image = a.checkpoint()
    ma = a.export_map()
    assert ma["collapsed"].sum() > 0 and len(image) > 6000 * ma["glb"].shape[0]
    cfg_b = cfg.copy()
    cfg_b.pool_submaps = cfg.pool_submaps // 2 + 7  # another pool size that still holds the map
    b = MLMap(cfg_b)
    b.restore(image)
    mb = b.export_map()
    for name in ma:
        assert np.array_equal(ma[name].view(np.uint8), mb[name].view(np.uint8)), name
    assert b.checkpoint()[-4096:] is not None and len(b.checkpoint()) == len(image)
    # both handles and the oracle continue in lock step
    for k in range(8, 12):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        st_a, st_b, st_o = a.integrate_depth(img, pose), b.integrate_depth(img, pose), orc.integrate_depth(img, pose)
        assert_frame_parity(b, orc, st_b, st_o, tag=f"restored{k}")
        assert st_a.ram_expand_cnt == st_b.ram_expand_cnt == st_o.ram_expand_cnt and st_a.obs_cnt == st_b.obs_cnt
    assert_map_parity(b, orc, LO_TOL, tag="restored")
    assert_map_parity(a, orc, LO_TOL, tag="original")
    # roll the first handle back to the checkpoint, foreign bytes and a different configuration are refused
    a.restore(image)
    m2 = a.export_map()
    for name in ma:
        assert np.array_equal(ma[name].view(np.uint8), m2[name].view(np.uint8)), name
    with pytest.raises(MlmError) as e:
        a.restore(b"\0" * len(image))
    assert e.value.code == 1
    cfg_c = config_cfg_a()
    c = MLMap(cfg_c)  # exploration mode off: not the same map configuration
    with pytest.raises(MlmError) as e:
        c.restore(image)
    assert e.value.code == 2


def test_two_call_layer_interface_equals_the_fused_frame():
    """awareness_map->input_pc_pose then local_map->input_pc_pose_direct (src/mlmap.cpp:382-386) as two calls: the frame's
    sets are readable in between, and the map afterwards equals the oracle's (and the one-launch path's)"""
    cfg = config_cfg_a()
    two, one, orc = MLMap(cfg), MLMap(cfg), Oracle(cfg)
    for k in range(5):
        pose = scenes.corridor_trajectory_pose(k * 20)
        img = scenes.corridor_depth_frame(cfg, pose, rows=240, cols=320, frame_idx=k)
        st_a = two.awareness_input_depth(img, pose)
        st_o = orc.integrate_depth(img, pose)
        assert (st_a.n_points, st_a.n_inside, st_a.n_cast, st_a.n_hit_cells, st_a.n_miss_cells) == \
               (st_o.n_points, st_o.n_inside, st_o.n_cast, st_o.n_hit_cells, st_o.n_miss_cells)
        kg, pg = two.last_frame_hits()          # between the calls: the awareness layer's containers
        ko, po = orc.last_frame_hits()
        assert np.array_equal(kg, ko) and np.array_equal(pg.view(np.uint32), po.view(np.uint32))
        assert np.array_equal(two.last_frame_misses(), orc.last_frame_misses())
        with pytest.raises(MlmError):
            two.integrate_depth(img, pose)      # a staged update must be fused first
        st_g = two.local_input_pc_pose_direct()
        one.integrate_depth(img, pose)
        assert_frame_parity(two, orc, st_g, st_o, tag=f"two-call{k}")
    assert_map_parity(two, orc, LO_TOL, tag="two-call")
    a, b = two.export_map(), one.export_map()
    for name in a:
        assert np.array_equal(a[name].view(np.uint8), b[name].view(np.uint8)), name
    # point-cloud entry + exploration mode through the same two calls
    cfg = _lidar_small_cfg()
    cfg.use_exploration_frontiers = 1
    two, orc = MLMap(cfg), Oracle(cfg)
    for k in range(3):
        pose = scenes.lidar_loop_pose(k * 3)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512, max_range=20.0)
        two.awareness_input_pc_pose(pts, pose)
        st_g, st_o = two.local_input_pc_pose_direct(), orc.integrate_points(pts, pose)
        assert_frame_parity(two, orc, st_g, st_o, tag=f"two-call-explore{k}")
    assert_map_parity(two, orc, LO_TOL, tag="two-call-explore")


def test_sampled_projection_of_a_device_image():
    """mlmapping_sample_cnt > 0 with the image already in device memory: same pixels, same number of rand() draws consumed
    as mlmap::project_depth on the host image (src/mlmap.cpp:321-346), frame after frame"""
    import ctypes as C
    cfg = config_cfg_a()
    cfg.sample_cnt = 300
    dev, host, orc = MLMap(cfg), MLMap(cfg), Oracle(cfg)
    C.CDLL("libc.so.6").srand(1)
    for k in range(6):
        pose = scenes.corridor_trajectory_pose(k * 11)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        if k == 3:
            img[:, ::2] = 0      # many invalid pixels: the quota is not reached, all 2*cnt tries are consumed
            img[::2, :] = 0
        d_img = dev.to_device(img)
        st_d, st_h, st_o = dev.integrate_depth_device(d_img, 480, 640, pose), host.integrate_depth(img, pose), orc.integrate_depth(img, pose)
        dev.device_free(d_img)
        assert st_d.n_points == st_h.n_points == st_o.n_points, (k, st_d.n_points, st_h.n_points, st_o.n_points)
        assert_frame_parity(dev, orc, st_d, st_o, tag=f"sampled-device{k}")
    assert_map_parity(dev, orc, LO_TOL, tag="sampled-device")


def test_get_odd_by_subbox_index():
    """getOdd(const Vec3I &glb_id, size_t subbox_id) (mlmap.h:128,227-235): allocated, absent and collapsed subboxes"""
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k in range(14):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
    m = orc.export_map()
    rs = np.random.RandomState(3)
    sel = rs.randint(0, m["glb"].shape[0], 4000)
    glb = m["glb"][sel].copy()
    glb[:200] += 1000                      # absent subboxes -> 0.5
    sub = rs.randint(0, 1000, 4000).astype(np.int32)
    got = gpu.getOdd_at(glb, sub)
    lo = np.where(m["collapsed"][sel] == 1, m["log_odds"][sel, 0], m["log_odds"][sel, sub]).astype(np.float64)
    want = (np.power(10.0, lo) / (1 + np.power(10.0, lo)))
    want[:200] = 0.5
    assert m["collapsed"].sum() > 0 and np.abs(got.astype(np.float64) - want).max() <= 1.2e-7
    if getattr(orc, "impl", "port") == "reference":   # the reference's own overload
        ref = np.empty(4000, dtype=np.float32)
        g32 = np.ascontiguousarray(glb.astype(np.int32))
        orc.lib.orc_get_odd_at(orc.h, g32.ctypes.data, sub.ctypes.data, 4000, ref.ctypes.data)
        assert np.abs(got.astype(np.float64) - ref).max() <= 1.2e-7


def test_asynchronous_frames_of_several_maps_on_one_gpu():
    """BASELINE config 5 on one GPU: frames of several agent maps submitted together, each handle with a share of the SMs
    so that their cooperative launches are co-resident; every map equals its oracle"""
    cfg = config_cfg_a()
    n = 4
    maps, orcs = [MLMap(cfg) for _ in range(n)], [Oracle(cfg) for _ in range(n)]
    for m in maps:
        m.set_sm_budget(148 // n)
    for k in range(6):
        dev, poses, imgs = [], [], []
        for a in range(n):
            pose = scenes.corridor_trajectory_pose(9 * k, y_offset=20.0 * a)
            img = scenes.corridor_depth_frame(cfg, pose, rows=240, cols=320, frame_idx=k, seed_drop=1 + 10 * a, seed_noise=2 + 10 * a,
                                              y_offset=20.0 * a)
            dev.append(maps[a].to_device(img)), poses.append(pose), imgs.append(img)
        for a in range(n):
            maps[a].submit_depth_device(dev[a], 240, 320, poses[a])
        for a in range(n):
            st_g, st_o = maps[a].finish_frame(), orcs[a].integrate_depth(imgs[a], poses[a])
            assert_frame_parity(maps[a], orcs[a], st_g, st_o, tag=f"async-agent{a}-frame{k}")
            maps[a].device_free(dev[a])
    for a in range(n):
        assert_map_parity(maps[a], orcs[a], LO_TOL, tag=f"async-agent{a}")


def test_cpp_mirror_harness_runs_on_the_device():
    """examples/corridor_harness: the C++ mirror of class mlmap (mlmapping_b200/include/mlmap.hpp) over the C ABI, built by
    __graft_entry__.build(); its own checks must pass on a device"""
    import subprocess
    from pathlib import Path
    exe = Path(__file__).resolve().parent.parent / "examples" / "corridor_harness"
    if not exe.exists():
        pytest.skip("examples/corridor_harness not built (run __graft_entry__.build())")
    res = subprocess.run([str(exe)], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
    assert "frame" in res.stdout.lower() or "rays" in res.stdout.lower(), res.stdout[-500:]
