"""CPU: pins for the oracle.  The reference has no tests or golden vectors (SURVEY §4), so these are
first-principles known answers for the reference's formulas, quirks the SURVEY derived from the cited
lines, and the libstdc++ container model the CUDA path emulates.  Every test runs twice: on the
restatement (oracle/mlmap_oracle.hpp, "port") and on the reference's OWN sources compiled into
oracle/_ref ("reference", oracle/ref_build/Makefile)."""
import math

import numpy as np
import pytest

from mlmapping_b200 import config_cfg_a, scenes
from oracle_binding import Oracle as _Oracle, load_oracle, load_reference, reference_available
from order_model import BUCKET_CHAIN, iteration_order, vector_hash


@pytest.fixture(scope="module", params=["port", "reference"])
def impl(request):
    if request.param == "reference" and not reference_available():
        pytest.skip("needs the reference build: oracle/_ref, or the original sources (MLMAPPING_REFERENCE)")
    return request.param


@pytest.fixture(scope="module")
def Oracle(impl):
    return lambda cfg, **kw: _Oracle(cfg, impl=impl, **kw)


@pytest.fixture(scope="module")
def lib(impl):
    return load_reference() if impl == "reference" else load_oracle()


@pytest.fixture(scope="module")
def orc(Oracle):
    return Oracle(config_cfg_a())


def test_logit_known_values(lib):
    # SURVEY §4 [probe]: logit(0.999f) = 2.99957108, logit(1.0f) = +inf (include/map_local.h:8)
    assert lib.orc_logit(np.float32(0.999)) == pytest.approx(2.99957108, abs=2e-7)
    assert math.isinf(lib.orc_logit(np.float32(1.0)))
    assert lib.orc_logit(np.float32(0.5)) == 0.0
    # logit_inv (include/mlmap.h:40): double pow, float result
    assert lib.orc_logit_inv(np.float32(0.0)) == 0.5
    assert lib.orc_logit_inv(np.float32(-2.0)) == pytest.approx(0.00990099, abs=1e-8)
    assert lib.orc_logit_inv(np.float32(4.2)) == pytest.approx(1 - 1 / (1 + 10 ** 4.2), abs=1e-7)


def test_fast_atan2_quirks(lib, orc):
    # include/map_awareness.h:86-113: (y>0, x=0) -> 3*pi/2 (sic); (y<0, x=0) -> -3pi/2 + ... = pi/2 after wrap
    assert lib.orc_fast_atan2(orc.h, 1.0, 0.0) == pytest.approx(1.5 * math.pi, abs=1e-12)
    v = lib.orc_fast_atan2(orc.h, -1.0, 0.0)
    assert (v + 2 * math.pi if v < 0 else v) == pytest.approx(0.5 * math.pi, abs=1e-12)
    # cubic approximation error stays below 0.1 degree
    ang = np.linspace(-3.1, 3.1, 2001)
    err = [abs(lib.orc_fast_atan2(orc.h, math.sin(a), math.cos(a)) - a) for a in ang]
    assert max(err) < math.radians(0.1)


def test_odds_table_clamps_and_reach(lib, orc):
    cfg = orc.cfg
    tab = np.array([[lib.orc_odds_table(orc.h, d, r) for r in range(cfg.am_n_rho)] for d in range(-10, 11)])
    assert tab.min() >= np.float32(0.001) and tab.max() <= np.float32(0.999)   # map_awareness.cpp:128-129
    assert tab[10, 1] == np.float32(0.999)        # near field: all mass in the centre cell
    assert np.all(tab[10] >= tab[11]) and np.all(tab[10] >= tab[9])
    assert tab[0, 0] == tab[0, 1] and tab[10, 0] == tab[10, 1]   # r == 0 treated as 1
    # 3*sigma_in_dr(64) = 3*0.00375*6.4^2/0.1 = 4.608 (SURVEY §8d)
    assert lib.orc_three_sigma(orc.h, 64) == pytest.approx(4.608, abs=1e-5)
    assert lib.orc_three_sigma(orc.h, 0) == 0.0


def test_pow2_is_exact_square(lib):
    rs = np.random.RandomState(0)
    for x in rs.uniform(-100, 100, 2000):
        assert lib.orc_pow2(x) == x * x


def test_vector_hasher_matches_model(lib):
    rs = np.random.RandomState(1)
    keys = rs.randint(-5, 700, size=(4000, 3))
    keys[:10] = [[0, 0, 0], [64, 359, 40], [-1, 0, 0], [2 ** 20, 3, 7], [1, 2, 3], [3, 2, 1], [65, 0, 20],
                 [0, 359, 0], [7, 7, 7], [-3, -2, -1]]
    model = vector_hash(keys)
    for k, m in zip(keys, model):
        assert lib.orc_vector_hash(int(k[0]), int(k[1]), int(k[2])) == int(m)


def test_bucket_chain_matches_this_libstdcxx(lib):
    # _Prime_rehash_policy: first insert -> 13 buckets, then next_bkt(2*B) (SURVEY Appendix B)
    assert lib.orc_next_bucket_count(12) == 13
    for b, nb in zip(BUCKET_CHAIN[1:20], BUCKET_CHAIN[2:21]):
        assert lib.orc_next_bucket_count(2 * b) == nb, (b, nb)


def test_T_ls_prologue(lib):
    # input_pc_pose prologue (map_awareness.cpp:184-186): T_ls = T_wa^-1 * T_wb * T_bs; yaw-only body
    import ctypes as C
    T_bs = (C.c_double * 7)(0.12, 0, 0, 0.5, -0.5, 0.5, -0.5)
    out = (C.c_double * 3)()
    T_wb = (C.c_double * 7)(*scenes.pose_from_xyz_yaw(5.0, -1.0, 1.2, 0.0))
    lib.orc_transform_point(T_wb, T_bs, (C.c_double * 3)(0.3, -0.2, 2.0), out)
    # optical frame (x right, y down, z forward) -> awareness frame (x forward, y left, z up), + 0.12 forward
    assert list(out) == pytest.approx([2.12, -0.3, 0.2], abs=1e-12)
    T_wb = (C.c_double * 7)(*scenes.pose_from_xyz_yaw(5.0, -1.0, 1.2, math.pi / 2))
    lib.orc_transform_point(T_wb, T_bs, (C.c_double * 3)(0.0, 0.0, 1.0), out)
    assert list(out) == pytest.approx([0.0, 1.12, 0.0], abs=1e-12)


def test_single_point_hit_miss_sets(Oracle):
    """one pixel, straight ahead at 1.0 m: hit cell + ray walk follow map_awareness.cpp:135-171,241-275"""
    cfg = config_cfg_a()
    o = Oracle(cfg)
    img = np.zeros((480, 640), dtype=np.uint16)
    img[240, 320] = 1000
    pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0)
    st = o.integrate_depth(img, pose)
    assert (st.n_points, st.n_inside, st.n_cast) == (1, 1, 1)
    keys, p = o.last_frame_hits()
    # p_l = (1.12, 0, 0): rho_idx 11, phi_idx 0, z_idx floor(2.05/0.1) = 20; sigma(11) = 0.045 cells:
    # the whole mass falls in the centre cell -> clamped to 0.999; 3*sigma < 1 -> no neighbours
    assert keys.tolist() == [[11, 0, 20]] and p[0] == np.float32(0.999)
    miss = o.last_frame_misses()
    nrho, nphi = cfg.am_n_rho, 360
    expect = sorted(20 * nrho * nphi + 0 * nrho + r for r in range(1, 11))  # r = 10..1, same z row (rate 0)
    assert miss.tolist() == expect
    m = o.export_map()
    assert (m["occupancy"] == b"o").sum() == 0          # logit(0.999) = 2.9996 < 3.0 threshold
    assert (m["occupancy"] == b"f").sum() == 10
    lo = m["log_odds"][m["occupancy"] == b"f"]
    assert np.all(lo == np.float32(-0.9))
    assert m["log_odds"].max() == pytest.approx(2.99957108, abs=3e-7)
    # second identical frame: hit cell 2*2.9996 -> clamps to 4.2 and turns 'o'; free cells go to -1.8
    o.integrate_depth(img, pose)
    m = o.export_map()
    assert (m["occupancy"] == b"o").sum() == 1
    assert m["log_odds"].max() == np.float32(4.2)
    assert m["log_odds"].min() == pytest.approx(-1.8, abs=1e-6)
    # the occupied voxel holds the hit cell centre (5 + 1.15 cos 0.5deg, 1.15 sin 0.5deg, 1.2 + 0) in the world
    si, ci = np.argwhere(m["occupancy"] == b"o")[0]
    g = m["glb"][si]
    xyz = np.array([ci % 10, (ci // 10) % 10, ci // 100])
    centre = g * 1.0 + xyz * 0.1 + 0.05
    assert abs(centre[0] - 6.15) < 0.051 and abs(centre[1] - 0.01) < 0.051 and abs(centre[2] - 1.2) < 0.051
    assert o.getOccupancy([centre])[0] == 0
    assert o.getOccupancy([centre - [0.6, 0, 0]])[0] == 1
    assert o.getOdd([centre])[0] == pytest.approx(1 - 1 / (1 + 10 ** 4.2), abs=1e-7)
    grad = o.getOddGrad([centre + [0.01, 0.0, 0.0]])[0]
    assert np.abs(grad).sum() > 0   # some neighbour has lower odds -> non-zero pseudo-gradient
    assert o.getOccupancy([[6.0, 5.0, 1.2]])[0] == -1
    assert o.getOdd([[100.0, 0.0, 0.0]])[0] == 0.5
    # third frame: free cells saturate at log_odds_min (-2.0), still 'f'
    o.integrate_depth(img, pose)
    assert o.export_map()["log_odds"].min() == np.float32(-2.0)


def test_out_of_range_ray_is_clamped_not_dropped(Oracle):
    """rho beyond n_Rho: no hit, ray cast from rho = n_Rho-1 with the stale rate (map_awareness.cpp:261-265)"""
    cfg = config_cfg_a()
    o = Oracle(cfg)
    img = np.zeros((480, 640), dtype=np.uint16)
    img[240, 320] = 20000  # 20 m
    st = o.integrate_depth(img, scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0))
    assert (st.n_inside, st.n_cast, st.n_hit_cells) == (0, 1, 0)
    assert st.n_miss_cells == cfg.am_n_rho - 2   # r = 63..1


def test_iteration_order_model_with_rehashes(Oracle, impl):
    """the data-parallel ordering scheme (stamp -> sort -> re-sequence per rehash) reproduces
    std::unordered_map's iteration order, including frames that cross several rehashes"""
    if impl == "reference":
        pytest.skip("needs the insert log, an instrumentation of the restatement")
    cfg = config_cfg_a()
    o = Oracle(cfg)
    o.set_log_inserts(True)
    B = 1
    sizes = [(60, 80), (120, 160), (480, 640), (20, 20), (480, 640)]
    for k, (r, c) in enumerate(sizes):
        pose = scenes.corridor_trajectory_pose(30 * k)
        img = scenes.corridor_depth_frame(cfg, pose, rows=r, cols=c, frame_idx=k)
        st = o.integrate_depth(img, pose)
        model, B = iteration_order(o.insert_log(), B)
        keys, _ = o.last_frame_hits()
        assert np.array_equal(model, keys), k
        assert B == st.hit_bucket_count


def test_set_free_and_grad(Oracle):
    cfg = config_cfg_a()
    o = Oracle(cfg)
    pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0)
    img = scenes.corridor_depth_frame(cfg, pose, rows=120, cols=160)
    c = cfg.copy()
    o.integrate_depth(img, pose)
    o.integrate_depth(img, pose)
    before = o.export_map()
    o.setFree_map_in_bound([5.0, -0.5, 0.5], [7.0, 0.5, 1.5])
    after = o.export_map()
    changed = (before["occupancy"] != after["occupancy"]) | (before["log_odds"] != after["log_odds"])
    assert changed.any()
    assert np.all(after["occupancy"][changed] == b"f") and np.all(after["log_odds"][changed] == 0.0)
    g = o.getOddGrad([[100.0, 100.0, 100.0]])
    assert np.all(g == 0.0)   # unknown space everywhere: no lower neighbour -> zero vector (mlmap.h:293)


def test_inflate_map_known_answer(Oracle):
    """one occupied cell in the middle of a subbox -> L1 ball of radius inflate_n in inflate_occupancy
    (src/mlmap.cpp:286-309, include/map_local.h:233-264); cells at or below flate_height do not inflate"""
    cfg = config_cfg_a()
    cfg.inflate_n, cfg.inflate_global_n, cfg.inflate_height = 2, 1, 0.1
    o = Oracle(cfg)
    img = np.zeros((480, 640), dtype=np.uint16)
    img[240, 320] = 1000
    pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0)
    o.integrate_depth(img, pose)
    o.integrate_depth(img, pose)          # second hit clamps to 4.2 and turns the cell 'o'
    m = o.export_map()
    assert (m["occupancy"] == b"o").sum() == 1 and (m["inflate"] == b"o").sum() == 0
    o.inflate_map(pose[:3])
    m = o.export_map()
    assert (m["inflate"] == b"o").sum() == 25   # |dx|+|dy|+|dz| <= 2 has 25 lattice points
    assert o.getInflateOccupancy([[6.15, 0.02, 1.25]])[0] == 0      # the occupied voxel itself (OCCUPIED)
    assert o.getInflateOccupancy([[6.15, 0.02, 1.55]])[0] == -1     # 3 cells above: outside the ball
    # the same scene 1.2 m lower: the hit cell centre is at z = 0.05 <= flate_height -> no inflation
    o2 = Oracle(cfg)
    low = scenes.pose_from_xyz_yaw(5.0, 0.0, 0.0, 0.0)
    o2.integrate_depth(img, low)
    o2.integrate_depth(img, low)
    o2.inflate_map(low[:3])
    assert (o2.export_map()["inflate"] == b"o").sum() == 0


def test_exploration_frontier_known_answer(Oracle):
    """one free cell in unknown space inside the exploration bounds: update_observation puts exactly one
    frontier cell on the first 'u' neighbour in the order +z,-z,+y,-y,+x,-x (src/map_local.cpp:7-33,78-83)"""
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    o = Oracle(cfg)
    img = np.zeros((480, 640), dtype=np.uint16)
    img[240, 320] = 300                    # hit at rho 4 (0.42 m): the walk frees rho 3..1 along phi 0
    pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0)
    st = o.integrate_depth(img, pose)
    m = o.export_map()
    n_free = int((m["occupancy"] == b"f").sum())
    n_front = int(np.unpackbits(m["frontier"]).sum())
    assert n_free == 3
    assert 1 <= n_front <= 3               # every freed cell nominates its +z neighbour (still 'u')
    # frontier cells are 'u' cells
    bits = np.unpackbits(m["frontier"], axis=1, bitorder="little")[:, :1000].astype(bool)
    assert np.all(m["occupancy"][bits] == b"u")
    # outside the hard-coded bounds {-30,30,-30,30,0,5} nothing is observed
    o2 = Oracle(cfg)
    far = scenes.pose_from_xyz_yaw(100.0, 0.0, 1.2, 0.0)
    o2.integrate_depth(img, far)
    assert np.unpackbits(o2.export_map()["frontier"]).sum() == 0


def test_sampled_projection_uses_libc_rand_stream(Oracle):
    """mlmapping_sample_cnt > 0: v = rand() % rows, u = rand() % cols, up to 2*cnt draws (src/mlmap.cpp:321-326)"""
    import ctypes as C
    cfg = config_cfg_a()
    cfg.sample_cnt = 50
    libc = C.CDLL("libc.so.6")
    img = np.full((480, 640), 2000, dtype=np.uint16)
    pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0)
    libc.srand(1)
    o = Oracle(cfg)
    st = o.integrate_depth(img, pose)
    assert st.n_points == 50
    pts = o.points()
    libc.srand(1)
    seq = [libc.rand() for _ in range(100)]
    v0, u0 = seq[0] % 480, seq[1] % 640
    fx = np.float32(347.99755859375)
    assert pts[0, 2] == 2000 * (1.0 / 1000.0)
    assert pts[0, 0] == float(np.float32(u0) - np.float32(320.0)) * pts[0, 2] / float(fx)
    assert pts[0, 1] == float(np.float32(v0) - np.float32(240.0)) * pts[0, 2] / float(fx)
    # three quarters of the image invalid: fewer than cnt points after 2*cnt draws
    img[:, ::2] = 0
    img[::2, :] = 0
    st = o.integrate_depth(img, pose)
    assert st.n_points < 50


def test_map_clouds_follow_subbox_id2xyz_glb(Oracle):
    """map clouds (rviz_vis.cpp:267-327): one float point per selected cell at origin*d_glb + xyz*d_sub + d_sub/2
    (map_local.h:201-206), cell ids x-fastest; the odds slice (mlmap.cpp:200-284) keeps the cells within 1e-3 of the height"""
    cfg = config_cfg_a()
    orc = Oracle(cfg)
    pose = scenes.corridor_trajectory_pose(0)
    for k in range(3):
        orc.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    m = orc.export_map()
    n = cfg.subbox_n
    occ = orc.export_cloud(1)
    assert occ.shape[0] == int((m["occupancy"] == b"o").sum()) > 100 and np.all(occ[:, 3] == 1.0)
    # rebuild the expected set from the exported arrays
    sb, cell = np.nonzero(m["occupancy"] == b"o")
    xyz = np.stack([cell % n, (cell // n) % n, cell // (n * n)], 1)
    d_sub, d_glb = cfg.subbox_d_xyz, cfg.subbox_d_xyz * n
    exp = (m["glb"][sb] * d_glb + xyz * d_sub + d_sub / 2).astype(np.float32)
    key = lambda a: a[np.lexsort((a[:, 2], a[:, 1], a[:, 0]))]
    assert np.array_equal(key(occ[:, :3]), key(exp))
    assert orc.export_cloud(0).shape[0] == int((m["inflate"] == b"o").sum())
    assert orc.export_cloud(2).shape[0] == 0  # frontiers are off in this configuration
    sl = orc.export_odds_slice(0.75)
    assert sl.shape[0] > 0 and np.all(np.abs(sl[:, 2] - 0.75) < 1e-3)
    assert orc.export_odds_slice(0.7).shape[0] == 0  # cell centres sit at k*0.1 + 0.05: nothing within 1e-3 of 0.7
    lo = m["log_odds"][(m["glb"][:, 2] == 0)][:, 7 * n * n:8 * n * n]
    assert sl.shape[0] == lo.size
    assert np.all((sl[:, 3] > 0) & (sl[:, 3] < 1))
    orc.close()


def test_far_hit_spreads_over_neighbours_along_the_ray(lib, Oracle):
    """update_hits (map_awareness.cpp:135-171): at 5.8 m the depth noise reaches 3*sigma = 0.001125*rho^2 > 3 cells, so one
    point marks the centre cell and, for d = 1..K, the cells (rho+d, round(z + d*rate)) and (rho-d, round(z - d*rate))
    with rate = (z - n_below) / rho, each with the tabulated odds of its offset; a second identical point folds
    p <- 1 - (1-p)(1-odd) in float"""
    import ctypes as C
    cfg = config_cfg_a()
    o = Oracle(cfg)
    img = np.zeros((480, 640), dtype=np.uint16)
    v, u = 200, 400
    img[v, u] = 5500
    pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.1)
    st = o.integrate_depth(img, pose)
    assert (st.n_points, st.n_inside) == (1, 1)
    # the point in the awareness frame, from the documented projection + T_ls (checked separately above)
    fx = np.float32(cfg.cam_fx)
    d = 5500 * (1.0 / 1000.0)
    ps = (C.c_double * 3)(float(np.float32(u) - np.float32(cfg.cam_cx)) * d / float(fx),
                          float(np.float32(v) - np.float32(cfg.cam_cy)) * d / float(np.float32(cfg.cam_fy)), d)
    pl = (C.c_double * 3)()
    lib.orc_transform_point((C.c_double * 7)(*pose), (C.c_double * 7)(*cfg.T_bs), ps, pl)
    x, y, z = pl[0], pl[1], pl[2]
    rho0 = int(math.sqrt(x * x + y * y) / cfg.am_d_rho)
    phi = math.degrees(math.atan2(y, x)) % 360.0
    z0 = int(math.floor((z + cfg.am_n_z_below * cfg.am_d_z + 0.5 * cfg.am_d_z) / cfg.am_d_z))
    keys, p = o.last_frame_hits()
    got = {tuple(k): float(pp) for k, pp in zip(keys.tolist(), p)}
    phis = {k[1] for k in got}
    assert len(phis) == 1 and abs(phis.pop() + 0.5 - phi) < 0.6           # fast_atan2 is within 0.09 deg of atan2
    phi0 = keys[0][1]
    K = 0
    while K + 1 < 3 * float(lib.orc_three_sigma(o.h, rho0)) / 3 and rho0 + K + 1 < cfg.am_n_rho:
        K += 1
    assert K >= 3
    rate = (z0 - cfg.am_n_z_below) / (rho0 * 1.0)
    rnd = lambda t: int(math.floor(abs(t) + 0.5) * (1 if t >= 0 else -1))   # std::round: half away from zero
    expect = {(rho0, phi0, z0): np.float32(lib.orc_odds_table(o.h, 0, rho0))}
    for dd in range(1, K + 1):
        expect[(rho0 + dd, phi0, rnd(z0 + dd * rate))] = np.float32(lib.orc_odds_table(o.h, dd, rho0))
        expect[(rho0 - dd, phi0, rnd(z0 - dd * rate))] = np.float32(lib.orc_odds_table(o.h, -dd, rho0))
    assert set(got) == set(expect), (sorted(got), sorted(expect))
    for k, pp in expect.items():
        assert np.float32(got[k]) == pp, (k, got[k], pp)
    assert abs(sum(got.values()) - 1.0) < 0.02                               # the offsets' odds are a discretised Gaussian
    # two identical points in one frame: every key folds once more, in float
    img[v, u + 1] = 0
    o2 = Oracle(cfg)
    pts = np.array([[ps[0], ps[1], ps[2]], [ps[0], ps[1], ps[2]]])
    o2.integrate_points(pts, pose)
    keys2, p2 = o2.last_frame_hits()
    got2 = {tuple(k): np.float32(pp) for k, pp in zip(keys2.tolist(), p2)}
    one = np.float32(1.0)
    for k, pp in expect.items():
        assert got2[k] == one - (one - pp) * (one - pp), k
    o.close()
    o2.close()


def test_inflated_occupancy_query_probes_19_points(Oracle):
    """getOccupancy(pos, inflate) (mlmap.h:142-169): OCCUPIED iff the point itself, one of the 6 axis offsets or one of
    the 12 planar diagonals (+-inflate on two axes) is occupied; never UNKNOWN; the 8 space diagonals are not probed"""
    cfg = config_cfg_a()
    o = Oracle(cfg)
    img = np.zeros((480, 640), dtype=np.uint16)
    img[240, 320] = 1000
    pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0)
    o.integrate_depth(img, pose)
    o.integrate_depth(img, pose)                       # second frame turns the hit voxel 'o' (see the single-point test)
    m = o.export_map()
    si, ci = np.argwhere(m["occupancy"] == b"o")[0]
    c = m["glb"][si] * 1.0 + np.array([ci % 10, (ci // 10) % 10, ci // 100]) * 0.1 + 0.05
    r = 0.3
    assert o.getOccupancy([c])[0] == 0 and o.getOccupancy([c], inflate=r)[0] == 0
    probes, expect = [], []
    for dx in (-r, 0.0, r):
        for dy in (-r, 0.0, r):
            for dz in (-r, 0.0, r):
                probes.append(c + [dx, dy, dz])        # querying from here, the occupied cell sits at offset (-dx,-dy,-dz)
                expect.append(0 if (dx == 0) + (dy == 0) + (dz == 0) >= 1 else 1)
    got = o.getOccupancy(np.array(probes), inflate=r)
    assert got.tolist() == expect
    assert o.getOccupancy([c + [0.0, 0.0, r]])[0] != 0                      # the plain query there is not occupied
    assert o.getOccupancy([[100.0, 0.0, 0.0]], inflate=r)[0] == 1           # unknown everywhere -> FREE, never UNKNOWN
    o.close()


def test_odd_gradient_picks_the_strictly_lowest_neighbour(Oracle):
    """getOddGrad (mlmap.h:237-295): the six axis probes are compared in the order +z,-z,+y,-y,+x,-x and a probe wins only
    if it is strictly lower than the running minimum; the result is (centre(best) - pos) * (float)(ori - min)"""
    cfg = config_cfg_a()
    o = Oracle(cfg)
    img = np.zeros((480, 640), dtype=np.uint16)
    img[240, 320] = 1000
    pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0)
    o.integrate_depth(img, pose)
    o.integrate_depth(img, pose)     # hit voxel: lo 4.2 'o'; the ten voxels of the ray in front of it: lo -1.8 'f'
    m = o.export_map()
    si, ci = np.argwhere(m["occupancy"] == b"o")[0]
    c = m["glb"][si] * 1.0 + np.array([ci % 10, (ci // 10) % 10, ci // 100]) * 0.1 + 0.05
    ori = np.float32(10.0 ** float(np.float32(4.2)) / (1 + 10.0 ** float(np.float32(4.2))))
    free = np.float32(10.0 ** float(np.float32(-1.8)) / (1 + 10.0 ** float(np.float32(-1.8))))
    assert o.getOdd([c])[0] == ori and o.getOdd([c - [0.1, 0, 0]])[0] == pytest.approx(float(free), abs=1e-7)
    # at the occupied cell: +z is unknown (0.5 < ori) and becomes the minimum first, ..., -x (free, 0.0156) wins at the end
    g = o.getOddGrad([c])[0]
    assert g[0] == pytest.approx(-0.1 * float(ori - o.getOdd([c - [0.1, 0, 0]])[0]), abs=1e-9) and abs(g[1]) < 1e-12 and abs(g[2]) < 1e-12
    # two cells above it everything within one step is unknown (0.5) except nothing lower: the search widens; the occupied
    # cell below has HIGHER odds, so the first strictly lower value is found only where the free ray cells come into reach
    up = c + [0.0, 0.0, 0.2]
    assert o.getOdd([up])[0] == 0.5
    g_up = o.getOddGrad([up], max_iter=1)[0]
    assert np.all(g_up == 0.0)                        # one step: all six neighbours are unknown, none is lower than 0.5
    # from a free ray cell, the cell behind it (towards the sensor) is equally free and the occupied one is higher:
    # no strictly lower neighbour within 5 steps along the axes except none -> zero vector at the second ray cell
    mid = c - [0.5, 0.0, 0.0]
    g_mid = o.getOddGrad([mid])[0]
    assert np.all(g_mid == 0.0)
    o.close()
