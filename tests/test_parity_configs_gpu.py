"""GPU parity at the sizes and corners BASELINE.json's configs name (SURVEY §8d), against the reference's own sources
when oracle/_ref is available (else the restatement): the whole 1000-frame CFG-A trajectory, CFG-B and CFG-C series,
the far agents of CFG-D, exploration mode on point-cloud input, and an adversarial cloud that sits on the cell borders
of the cylindrical index (the guarded float fast path of the projection must never disagree with the exact chain)."""
import numpy as np
import pytest

from mlmapping_b200 import MLMap, config_cfg_a, config_cfg_b, config_cfg_c, scenes
from oracle_binding import best_oracle as Oracle
from parity_utils import assert_frame_parity, assert_map_parity

pytestmark = pytest.mark.gpu
LO_TOL = 1e-6


def _counters_equal(st_g, st_o, tag):
    for f in ("n_points", "n_inside", "n_cast", "n_hit_cells", "n_miss_cells", "n_touched_voxels", "hit_bucket_count",
              "ram_expand_cnt", "obs_cnt"):
        assert getattr(st_g, f) == getattr(st_o, f), (tag, f, getattr(st_g, f), getattr(st_o, f))


def _replay_against_golden(name, make_cfg):
    """runs the named series (tests/golden/make_golden_long.py) on the GPU and compares with the vectors the REFERENCE
    produced for the same seeded inputs: counters every frame, the frame's hit map (iteration order, probabilities) and
    miss set and a digest of the WHOLE map (subbox set, states, log-odds bits) at the recorded checkpoints"""
    import json
    from pathlib import Path
    from golden.make_golden_long import COUNTERS, frame_digest, map_digest, series
    gold = json.loads((Path(__file__).parent / "golden" / "golden_long.json").read_text())
    assert "UNMODIFIED reference sources" in gold["provenance"] and gold["counters"] == list(COUNTERS)
    g = gold["series"][name]
    gpu = MLMap(make_cfg())
    n_frames = n_maps = 0
    for k, kind, data, pose in series(name):
        st = gpu.integrate_depth(data, pose) if kind == "depth" else gpu.integrate_points(data, pose)
        got = [int(getattr(st, f)) for f in COUNTERS]
        assert got == g["counters"][k], (name, k, dict(zip(COUNTERS, got)), dict(zip(COUNTERS, g["counters"][k])))
        if str(k) in g["frames"]:
            assert frame_digest(gpu) == g["frames"][str(k)], (name, k, "per-frame hit map / miss set differs from the reference")
            n_frames += 1
        if str(k) in g["maps"]:
            m = gpu.export_map()
            assert m["glb"].shape[0] == g["maps"][str(k)]["subboxes"], (name, k)
            assert map_digest(m) == g["maps"][str(k)]["digest"], (name, k, "map differs from the reference (bit-level digest)")
            n_maps += 1
    assert k + 1 == len(g["counters"]) and n_frames == len(g["frames"]) and n_maps == len(g["maps"])
    return g


def test_cfg_a_full_1000_frame_trajectory():
    """BASELINE config 2 in full: 1000 frames, x = 5 + 0.05 k, streaming subbox allocation"""
    g = _replay_against_golden("cfg_a_1000", config_cfg_a)
    assert g["maps"]["999"]["subboxes"] > 500 and len(g["maps"]) == 10 and len(g["frames"]) == 20


def test_cfg_b_series_of_50_frames():
    """BASELINE config 3: L515-like 1024x768 @ 0.05 m, 200 m corridor, 0.1 m steps (50 consecutive frames)"""
    g = _replay_against_golden("cfg_b_50", config_cfg_b)
    assert g["maps"]["49"]["subboxes"] > 300


def test_cfg_c_series_of_12_full_scans():
    """BASELINE config 4: 128 x 2048 LiDAR scans along the loop, one GPU"""
    g = _replay_against_golden("cfg_c_12", config_cfg_c)
    assert g["maps"]["11"]["subboxes"] > 5000


@pytest.mark.parametrize("agent", [0, 7])
def test_cfg_d_agent_maps(agent):
    """BASELINE config 5: agent a lives on the corridor shifted by y = 20 a (agent 7 at y ~ 140 m: other hash slots,
    other lattice rounding, outside the exploration bounds) with seeds + 10 a; 12 frames + the planner query mix"""
    cfg = config_cfg_a()
    gpu, orc = MLMap(cfg), Oracle(cfg)
    y0 = 20.0 * agent
    for k in range(12):
        pose = scenes.corridor_trajectory_pose(7 * k, y_offset=y0)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=7 * k, seed_drop=1 + 10 * agent, seed_noise=2 + 10 * agent, y_offset=y0)
        st_g, st_o = gpu.integrate_depth(img, pose), orc.integrate_depth(img, pose)
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"agent{agent}-frame{k}")
    assert_map_parity(gpu, orc, LO_TOL, tag=f"agent{agent}")
    m = orc.export_map()
    assert abs(m["glb"][:, 1].mean() - y0) < 3
    pos = scenes.query_positions(200000, m["glb"].min(0) * 1.0, (m["glb"].max(0) + 1) * 1.0, seed=5)
    assert np.array_equal(gpu.getOccupancy(pos[:80000]), orc.getOccupancy(pos[:80000]))
    assert np.array_equal(gpu.getOdd(pos[80000:160000]).view(np.uint32), orc.getOdd(pos[80000:160000]).view(np.uint32))
    assert np.array_equal(gpu.getOddGrad(pos[160000:]).view(np.uint64), orc.getOddGrad(pos[160000:]).view(np.uint64))


def test_exploration_mode_on_point_cloud_input():
    """use_exploration_frontiers with input_pc_pose fed directly (LiDAR-like points inside the exploration bounds):
    frontier sets, neighbour allocation and the release pass against the reference"""
    cfg = config_cfg_c()
    cfg.am_n_rho, cfg.am_n_z_below, cfg.am_n_z_over = 100, 20, 20   # 20 m range, z within +-4 m
    cfg.use_exploration_frontiers = 1
    cfg.max_points = 32 * 512
    cfg.pool_submaps = 16384
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for k in range(6):
        pose = scenes.lidar_loop_pose(k * 2)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512, max_range=25.0)
        st_g, st_o = gpu.integrate_points(pts, pose), orc.integrate_points(pts, pose)
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"explore-pc{k}")
        assert_map_parity(gpu, orc, LO_TOL, tag=f"explore-pc{k}")
    m = orc.export_map()
    assert np.unpackbits(m["frontier"]).sum() > 1000


def _border_cloud(cfg, rs):
    """sensor-frame points (T_bs = identity, pose = identity => p_l == p_s bit for bit) whose cylindrical coordinates sit
    on, or a few ulps beside, the borders of the rho / phi / z cells, plus the quirks of xyz2RhoPhiZwithBoderCheck"""
    d_rho, d_z = cfg.am_d_rho, cfg.am_d_z
    d_phi = cfg.am_d_phi_deg * np.pi / 180
    n_rho = cfg.am_n_rho
    z_min = -(cfg.am_n_z_below * d_z) - 0.5 * d_z
    nz = cfg.am_n_z_below + cfg.am_n_z_over + 1

    def ulps(v, j):
        v = np.asarray(v, dtype=np.float64).copy()
        for _ in range(abs(j)):
            v = np.nextafter(v, np.inf if j > 0 else -np.inf)
        return v

    pts = []
    # (1) axis points: rho == |x| exactly, so rho / dRho lands on k or one ulp beside it; phi is 0, pi or the x == 0 quirk
    ks = np.r_[np.arange(0, n_rho + 3), n_rho * 5, 325, 650]
    for j in (-2, -1, 0, 1, 2):
        r = ulps(ks * d_rho, j)
        z = rs.uniform(z_min + 0.3, z_min + nz * d_z - 0.3, r.size)
        pts += [np.c_[r, np.zeros_like(r), z], np.c_[-r, np.zeros_like(r), z], np.c_[np.zeros_like(r), r, z],
                np.c_[np.zeros_like(r), -r, z], np.c_[r, -0.0 * r, z]]
    # (2) z borders: z - z_border_min == k dZ (and beside), incl. the bottom / top of the range and beyond
    kz = np.arange(-2, nz + 3)
    for j in (-2, -1, 0, 1, 2):
        z = ulps(z_min + kz * d_z, j)
        a = rs.uniform(0, 2 * np.pi, z.size)
        rr = rs.uniform(0.5, (n_rho - 1) * d_rho, z.size)
        pts.append(np.c_[rr * np.cos(a), rr * np.sin(a), z])
    # (3) rho borders at arbitrary azimuths: x, y = rho (cos a, sin a) is within a few ulps of the border
    for j in range(-4, 5):
        k = rs.randint(1, n_rho + 2, 3000)
        rho = ulps(k * d_rho, j)
        a = rs.uniform(0, 2 * np.pi, k.size)
        pts.append(np.c_[rho * np.cos(a), rho * np.sin(a), rs.uniform(z_min + 0.2, z_min + nz * d_z - 0.2, k.size)])
    # (4) phi borders: fast_atan2 (a cubic, include/map_awareness.h:86-118) is piecewise, so aim at phi = m dPhi through
    # the inverse of its first octant by bisection, mirror into all octants, then jitter by ulps
    def fast_atan_deg(t):
        return t * (45 - (t - 1) * (14 + 3.83 * t))
    m_deg = np.arange(0, 46, 1.0) * cfg.am_d_phi_deg
    lo, hi = np.zeros_like(m_deg), np.ones_like(m_deg)
    for _ in range(80):
        mid = 0.5 * (lo + hi)
        too_small = fast_atan_deg(mid) < m_deg
        lo, hi = np.where(too_small, mid, lo), np.where(too_small, hi, mid)
    for t in (lo, hi):
        for j in (-3, -1, 0, 1, 3):
            tt = ulps(t, j)
            rr = rs.uniform(1.0, (n_rho - 2) * d_rho, tt.size)
            x, y = rr / np.sqrt(1 + tt * tt), rr * tt / np.sqrt(1 + tt * tt)
            z = rs.uniform(z_min + 0.3, z_min + nz * d_z - 0.3, tt.size)
            for sx, sy, swap in ((1, 1, 0), (1, 1, 1), (-1, 1, 0), (-1, 1, 1), (1, -1, 0), (1, -1, 1), (-1, -1, 0), (-1, -1, 1)):
                a, b = (y, x) if swap else (x, y)
                pts.append(np.c_[sx * a, sy * b, z])
    # (5) far and degenerate points: 65 m, beyond int range, infinities, NaN
    far = np.array([[65.0, 1e-3, 0.1], [-65.0, 0.5, -0.2], [1e9, 2e9, 0.0], [3e10, 1.0, 0.0], [np.inf, 1.0, 0.0], [1.0, -np.inf, 0.3],
                    [np.nan, 1.0, 0.0], [1.0, 1.0, np.nan], [1.0, 2.0, 1e12], [1.0, 2.0, -1e12], [1e-300, 1e-300, 0.0],
                    [5e-324, 0.0, 0.0], [2.0 ** -30, -2.0 ** -30, 0.05]])
    pts.append(far)
    cloud = np.concatenate(pts, 0)
    rs.shuffle(cloud)
    return np.ascontiguousarray(cloud)


@pytest.mark.parametrize("which", ["lidar_0.2m", "depth_like_0.1m"])
def test_adversarial_cell_border_cloud(which):
    """the projection's guarded float fast path accepts an index only when it is farther than a guard band from the next
    integer; everything inside the band runs the exact double chain.  This cloud lives on the borders: hit map (iteration
    order + probabilities), miss set, counters and the map must equal the reference's bit for bit."""
    cfg = config_cfg_c()
    if which == "depth_like_0.1m":
        cfg.am_d_rho = cfg.am_d_z = cfg.subbox_d_xyz = 0.1
        cfg.am_n_rho, cfg.am_n_z_below, cfg.am_n_z_over = 65, 20, 20
        cfg.depth_noise_coe = 0.00375
    else:
        cfg.am_n_rho, cfg.am_n_z_below, cfg.am_n_z_over = 120, 30, 30
    cloud = _border_cloud(cfg, np.random.RandomState(11))
    cfg.max_points = int(cloud.shape[0])
    cfg.pool_submaps = 32768
    gpu, orc = MLMap(cfg), Oracle(cfg)
    for rep, pose in enumerate([np.array([0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0]), np.array([0.5, -0.25, 0.125, 1.0, 0.0, 0.0, 0.0])]):
        st_g, st_o = gpu.integrate_points(cloud, pose), orc.integrate_points(cloud, pose)
        assert st_o.n_inside > 20000 and st_o.n_cast >= st_o.n_inside
        assert_frame_parity(gpu, orc, st_g, st_o, tag=f"{which}-border{rep}")
        assert_map_parity(gpu, orc, LO_TOL, tag=f"{which}-border{rep}")
