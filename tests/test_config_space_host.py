"""CPU: the configuration-space table (tests/config_space.py) holds only configurations that mlm_create accepts and
that the oracle runs; the Python statement of K(rho) matches the oracle's 3 sigma(rho); validate_config's limits are
exact; the oracle refuses a configuration outside update_hits' preconditions with an exception instead of crashing;
and at subbox sizes 3, 7 and 16 the restatement's rays, distance field, frontier clusters and view gains equal the
plain statements of those specs."""
import ctypes as C

import numpy as np
import pytest

import mlmapping_b200 as mlm
from mlmapping_b200 import config_cfg_a
import config_space as cs
from oracle_binding import Oracle, k_reach, update_hits_ok

MLM_OK, INVALID_CONFIG, NO_DEVICE = 0, 2, 7


@pytest.fixture(scope="module")
def lib():
    if not mlm.library_path().exists():
        mlm.build_library()
    return mlm.load_library()


def _create_rc(lib, cfg):
    """mlm_create's verdict: MLM_OK (handle destroyed again) on a machine with a device, MLM_ERR_NO_DEVICE without one
    for a configuration that validate_config accepts, MLM_ERR_INVALID_CONFIG for one it refuses"""
    h = C.c_void_p()
    rc = lib.mlm_create(C.byref(cfg), 0, C.byref(h))
    if rc == MLM_OK:
        lib.mlm_destroy(h)
    return rc


@pytest.mark.parametrize("name", [c.name for c in cs.CASES])
def test_table_entry_is_accepted_and_runs_through_the_oracle(lib, name):
    case = cs.BY_NAME[name]
    cfg = cs.config_of(case)
    assert _create_rc(lib, cfg) in (MLM_OK, NO_DEVICE), mlm.capi.load_library().mlm_last_error()
    assert update_hits_ok(cfg)
    orc = Oracle(cfg)
    for kind, data, pose in cs.frames(case, cfg):
        st = cs.integrate(orc, kind, data, pose)
        assert st.n_inside > 0, (name, "no point reaches the awareness map")
    m = orc.export_map()
    assert m["glb"].shape[0] > 0 and (m["occupancy"] == b"o").sum() > 0
    if case.pool_from_oracle:
        assert cfg.pool_submaps > m["glb"].shape[0]


def test_table_reaches_the_derived_constants_it_names():
    """the host rules of mlm_create, restated: the cases aimed at whole-column work items get split = 0, the others keep
    the half columns; noise_wide reaches maxK = 10; the phi cases get the sector counts they name"""
    split = {c.name: cs.split_of(c.make()) for c in cs.CASES if c.name != "default_yaml"}
    for name in ("phi0_125", "below0", "over0", "noise_wide_short"):
        assert split.pop(name) == 0, name
    assert all(v == 1 for v in split.values()), split
    for name in ("noise_wide", "noise_wide_short"):
        assert k_reach(cs.BY_NAME[name].make()).max() == 10
    assert [cs.n_phi(cs.BY_NAME[n].make()) for n in ("phi5", "phi7", "phi0_125", "phi360")] == [72, 51, 2880, 1]
    assert 51 * 7 < 360   # phi7: the last sector is partial


def _refused_by_k():
    """configurations that break K(rho) <= min(10, rho): the one that crashed the oracle, and noise_wide's largest
    accepted depth_noise_coe times 1 + 1e-9"""
    a = config_cfg_a()
    a.am_d_rho, a.am_n_rho = 0.02, 300
    b = cs.BY_NAME["noise_wide"].make()
    b.depth_noise_coe *= 1 + 1e-9
    return [a, b]


def test_k_reach_matches_the_oracles_three_sigma():
    """the Python K(rho) against the oracle's own sigma_in_dr: K = the last integer below 3 sigma"""
    for case in cs.CASES:
        cfg = case.make()
        orc = Oracle(cfg)
        ts = np.array([orc.lib.orc_three_sigma(orc.h, r) for r in range(cfg.am_n_rho)], dtype=np.float32)
        want = np.array([max(0, min(int(np.ceil(t)) - 1, 41)) for t in ts])
        assert np.array_equal(k_reach(cfg), want), case.name
    for cfg in _refused_by_k():
        assert not update_hits_ok(cfg)


def test_oracle_refuses_what_update_hits_cannot_run():
    """Oracle(cfg) used to run update_hits off the odds table at am_d_rho = 0.02, am_n_rho = 300 and crash the process;
    it raises instead, for every oracle class"""
    from esdf_oracle import EsdfOracle
    from frontier_oracle import FrontierOracle
    from ray_oracle import RayOracle
    from view_oracle import ViewOracle
    for cfg in _refused_by_k():
        for cls in (Oracle, RayOracle, EsdfOracle, FrontierOracle, ViewOracle):
            with pytest.raises(ValueError, match="update_hits"):
                cls(cfg)


def test_validate_config_boundaries(lib):
    """the limits of validate_config, exactly, on both sides.  A configuration it accepts reaches the device check (and
    runs on a B200); every configuration-dependent refusal happens here, with or without a device.  On sm_100 the
    shared memory of the frame kernels (227 KB per block) is tighter than the index ranges: the projection's
    per-column histogram bounds the work columns (3045: n_Phi 1522 with half columns, 3045 without), the column item's
    bitmaps and odds table bound n_Z * n_Rho and n_Rho."""
    base = config_cfg_a()

    def rc(**kw):
        c = base.copy()
        for k, v in kw.items():
            setattr(c, k, v)
        return _create_rc(lib, c)

    def refused(r, why):
        return r == INVALID_CONFIG and why in lib.mlm_last_error()

    ok = (MLM_OK, NO_DEVICE)
    assert refused(rc(subbox_n=0), b"subbox size") and refused(rc(subbox_n=65), b"subbox size")
    # one cell per subbox is refused: the reference reads a one-element subbox as collapsed and never updates it again
    assert refused(rc(subbox_n=1), b"collapsed")
    assert rc(subbox_n=2) in ok and rc(subbox_n=64, pool_submaps=8) in ok

    def phi(n):  # a sector size with int(360 / d) == n
        d = 360 / (n + 0.5)
        assert int(360 / d) == n
        return d
    hist = b"shared-memory histogram"
    assert rc(am_d_phi_deg=phi(1522)) in ok and refused(rc(am_d_phi_deg=phi(1523)), hist)     # 2 columns per sector
    assert refused(rc(am_d_phi_deg=phi(2048)), hist) and rc(am_d_phi_deg=phi(2049)) in ok    # > 2048: not split
    assert rc(am_d_phi_deg=phi(3045)) in ok and refused(rc(am_d_phi_deg=phi(3046)), hist)
    assert refused(rc(am_d_phi_deg=phi(4096)), hist) and refused(rc(am_d_phi_deg=phi(4097)), b"[1,4096]")
    # n_Rho: the range check first, the column's shared memory (odds table + bitmaps) binds first at n_Z = 41
    column = b"does not fit shared memory"
    far = dict(depth_noise_coe=0.0, subbox_d_xyz=1.0)   # K(rho) = 0 and a frame-local grid well below 2^31 cells
    assert rc(am_n_rho=2) in ok and refused(rc(am_n_rho=1), b"awareness extents")
    assert rc(am_n_rho=1494, **far) in ok and refused(rc(am_n_rho=1495, **far), column)
    assert refused(rc(am_n_rho=4096, **far), b"n_Rho must be < 4096")
    # n_Z * n_Rho < 2^20 (the cell index bits) is looser than the column bitmaps: n_Z <= 224 at n_Rho = 1024
    assert rc(am_n_rho=1024, am_n_z_below=0, am_n_z_over=223, **far) in ok
    assert refused(rc(am_n_rho=1024, am_n_z_below=0, am_n_z_over=224, **far), column)
    assert refused(rc(am_n_rho=2048, am_n_z_below=255, am_n_z_over=256, **far), b"2^20")
    assert refused(rc(am_n_rho=1025, am_n_z_below=511, am_n_z_over=511, **far), column)   # 2^20 - 1 cells
    # the frame-local voxel grid (< 2^31 cells): 0.005 m voxels over CFG-A's 6.5 m range make 5.8e9
    assert refused(rc(subbox_d_xyz=0.005), b"voxel grid too large")
    assert rc(am_n_z_below=0) in ok and rc(am_n_z_over=0) in ok and refused(rc(am_n_z_below=-1), b"awareness extents")
    # update_hits' preconditions: K(rho) <= min(10, rho)
    for cfg in _refused_by_k():
        assert refused(_create_rc(lib, cfg), b"depth_noise_coe too large")


# ---- the derived-feature specs at other subbox sizes -------------------------------------------------------------

def _explore_n(n):
    cfg = config_cfg_a()
    cfg.subbox_n, cfg.use_exploration_frontiers = n, 1
    return cfg


def _build(orc, frames=6):
    from mlmapping_b200 import scenes
    for k in range(frames):
        pose = scenes.corridor_trajectory_pose(k * 10)
        orc.integrate_depth(scenes.corridor_depth_frame(orc.cfg, pose, rows=240, cols=320, frame_idx=k), pose)
    return pose


@pytest.mark.parametrize("n", [3, 7, 16])
def test_rays_and_distance_field_equal_the_spec(n):
    from esdf_oracle import EsdfOracle
    from raycast_spec import FREE, OCCUPIED, MapStates, cast_rays, edge_segments, first_difference, random_segments
    from test_esdf_host import _check_box
    cfg = _explore_n(n)
    orc = EsdfOracle(cfg)
    pose = _build(orc)
    orc.inflate_map(pose[:3])
    ex = orc.export_map()
    d = cfg.subbox_d_xyz
    f1, t1 = random_segments(600, ex["glb"].min(0) * n * d, (ex["glb"].max(0) + 1) * n * d, seed=n, max_len=4.0)
    f2, t2 = edge_segments(ex, n, d, seed=n + 7, n_each=40)
    f, t = np.concatenate([f1, f2]), np.concatenate([t1, t2])
    states = MapStates(ex, n)
    for inflated in (False, True):
        want, _ = cast_rays(f, t, d, states, inflated)
        got = orc.cast_rays(f, t, inflated=inflated)
        assert first_difference(got, want) is None, (n, inflated, first_difference(got, want))
        assert (got["status"] == FREE).sum() > 10 and (got["status"] == OCCUPIED).sum() > 10
    # a box whose faces cut through subboxes
    c = pose[:3]
    lo, hi = c - [0.37 * n * d, 1.43, 1.31], c + [2.0 + 0.41 * n * d, 1.39, 1.29]
    for inflated in (False, True):
        val, blk, *_ = _check_box(cfg, orc, ex, lo, hi, 1.0, inflated, n_query=2000, seed=n)
        assert blk.sum() > 0 and (~blk).sum() > 0


@pytest.mark.parametrize("n", [3, 7, 16])
def test_frontier_clusters_and_view_gain_equal_the_spec(n):
    from frontier_oracle import FrontierOracle
    from test_frontier_host import assert_oracle_equals_spec
    from test_view_host import corridor_views, spec_gain
    from view_oracle import ViewOracle
    from view_spec import sensor
    cfg = _explore_n(n)
    orc = FrontierOracle(cfg)
    _build(orc)
    ex = orc.export_map()
    assert_oracle_equals_spec(orc, ex, cfg, f"n{n}")
    vo = ViewOracle(cfg)
    _build(vo)
    poses, boxes = corridor_views(cfg, ex, seed=n)
    S = sensor(max_depth=1.5)
    for frontier in (False, True):
        for b in (None, boxes):
            got = vo.view_gain(poses, S, b, frontier, False)
            want = spec_gain(ex, cfg, poses, S, b, frontier, False)
            assert got.tobytes() == want.tobytes(), (n, frontier, b is None)
            assert got["n_target"].sum() > 0
