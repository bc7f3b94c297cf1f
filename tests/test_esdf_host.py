"""CPU: the C++ oracle's signed distance field (orc_esdf_*) equals the written spec (tests/esdf_spec.py): exact squared
distances against brute force and scipy, cell values and queries bit for bit on both layers, the max_dist clamp, NaN
outside the box, the clamped stencil of the border half cell; and the C ABI rejects bad arguments without a device."""
import ctypes as C

import numpy as np
import pytest

import mlmapping_b200 as mlm
from mlmapping_b200 import config_cfg_a, scenes
from esdf_oracle import EsdfOracle, squared_edt
from esdf_spec import (box_blocking, brute_force, cell_values, first_difference, query, query_points, same_bits,
                       scipy_squared)


def _random_masks():
    rs = np.random.RandomState(3)
    shapes = [(6, 7, 5), (9, 4, 11), (1, 1, 1), (1, 8, 9), (7, 1, 6), (5, 6, 1), (1, 1, 23), (1, 17, 1), (13, 1, 1)]
    out = []
    for s in shapes:
        for p in (0.0, 0.03, 0.3, 0.8, 1.0):
            out.append(rs.uniform(size=s) < p)
    return out


def test_oracle_transform_equals_brute_force_and_scipy():
    """random blocking sets incl. empty, all-blocking, one cell, flat and line-shaped boxes"""
    for m in _random_masks():
        dp, dm = squared_edt(m)
        bp, bm = brute_force(m)
        assert np.array_equal(dp, bp) and np.array_equal(dm, bm), m.shape
        sp, sm = scipy_squared(m)
        assert np.array_equal(dp, sp) and np.array_equal(dm, sm), m.shape
    # larger boxes: scipy only
    rs = np.random.RandomState(4)
    for s, p in (((40, 64, 50), 0.01), ((20, 30, 128), 0.2), ((64, 3, 64), 0.002)):
        m = rs.uniform(size=s) < p
        dp, dm = squared_edt(m)
        sp, sm = scipy_squared(m)
        assert np.array_equal(dp, sp) and np.array_equal(dm, sm), s


@pytest.fixture(scope="module")
def corridor():
    """CFG-A, 10 corridor frames, then inflate_map at the last pose"""
    cfg = config_cfg_a()
    orc = EsdfOracle(cfg)
    for k in range(10):
        pose = scenes.corridor_trajectory_pose(k * 5)
        orc.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    orc.inflate_map(pose[:3])
    return cfg, orc, orc.export_map(), pose


def _check_box(cfg, orc, ex, box_min, box_max, max_dist, inflated, brute=False, n_query=3000, seed=0):
    d = cfg.subbox_d_xyz
    orc.build_esdf(box_min, box_max, max_dist, inflated=inflated)
    val, dp, dm, lo = orc.export_esdf_exact()
    slo, dims, blk = box_blocking(ex, cfg.subbox_n, d, box_min, box_max, inflated)
    assert np.array_equal(lo, slo) and val.shape == (dims[2], dims[1], dims[0])
    sp, sm = brute_force(blk) if brute else scipy_squared(blk)
    assert np.array_equal(dp, sp) and np.array_equal(dm, sm)
    want = cell_values(blk, sp, sm, d, max_dist)
    assert same_bits(val, want), first_difference(val, want)
    grid, glo = orc.export_esdf()
    assert np.array_equal(glo, lo) and same_bits(grid, val.astype(np.float32))
    pts = query_points(lo, dims, d, n_query, seed)
    dist, grad = orc.esdf_distance(pts)
    sdist, sgrad = query(val, lo, d, pts)
    assert same_bits(dist, sdist), first_difference(dist, sdist)
    assert same_bits(grad, sgrad), first_difference(grad, sgrad)
    return val, blk, lo, dims, pts, dist, grad


@pytest.mark.parametrize("inflated", [False, True])
def test_oracle_field_equals_the_spec(corridor, inflated):
    """a local-planner box around the last pose (scipy), a small box (brute force), both layers"""
    cfg, orc, ex, pose = corridor
    c = pose[:3]
    val, blk, lo, dims, pts, dist, grad = _check_box(cfg, orc, ex, c - [3.0, 3.0, 1.0], c + [3.0, 3.0, 1.0], 2.0,
                                                     inflated, n_query=20000, seed=1)
    assert blk.sum() > 100 and (~blk).sum() > 1000
    assert (val == 0).any() and (val == 2.0).any() and (val > 0.1).sum() > 1000
    assert np.isnan(dist).sum() >= 5 and np.isfinite(dist).sum() > 20000
    occ = np.argwhere(blk)[0][::-1] + lo                          # a small box around an obstacle cell
    d = cfg.subbox_d_xyz
    _check_box(cfg, orc, ex, (occ - [4, 5, 3]) * d + 0.01, (occ + [5, 4, 3]) * d + 0.01, 0.6, inflated, brute=True,
               seed=2)


def test_inflation_layer_blocks_more(corridor):
    cfg, orc, ex, pose = corridor
    c = pose[:3]
    orc.build_esdf(c - 2.0, c + 2.0, 1.0)
    a, _ = orc.export_esdf()
    orc.build_esdf(c - 2.0, c + 2.0, 1.0, inflated=True)
    b, _ = orc.export_esdf()
    assert (b <= 0).sum() > (a <= 0).sum() and ((a <= 0) <= (b <= 0)).all()


def test_max_dist_clamp(corridor):
    """free cells stop at max_dist, obstacle cells at d_sub - max_dist; a max_dist under one cell"""
    cfg, orc, ex, pose = corridor
    d, c = cfg.subbox_d_xyz, pose[:3]
    for md in (0.35, 0.05, 100.0):
        val, blk, *_ = _check_box(cfg, orc, ex, c - 1.5, c + 1.5, md, False, n_query=500, seed=5)
        assert val[~blk].max() <= md and val[blk].min() >= d - md
        if md < 1.0:
            assert (val[~blk] == md).any()
        if md < d:                                               # every cell of B sits one cell from a free one or more
            assert (val[blk] == d - md).all() and (val[~blk] == md).all()


def test_empty_and_full_boxes(corridor):
    """an all-unknown box: max_dist everywhere; a one-cell box on an occupied cell: d_sub - max_dist"""
    cfg, orc, ex, pose = corridor
    d = cfg.subbox_d_xyz
    orc.build_esdf([-40.0, -40.0, -40.0], [-38.0, -39.0, -39.5], 1.5)
    val, dp, dm, _ = orc.export_esdf_exact()
    assert (val == 1.5).all() and (dp == -1).all()
    i = np.argwhere(box_blocking(ex, cfg.subbox_n, d, pose[:3] - 2, pose[:3] + 2)[2])[0][::-1]
    lo = np.floor((pose[:3] - 2) / d).astype(np.int64)
    p = (lo + i + 0.5) * d
    orc.build_esdf(p, p, 1.5)
    val, dp, dm, glo = orc.export_esdf_exact()
    assert val.shape == (1, 1, 1) and val[0, 0, 0] == d - 1.5 and dp[0, 0, 0] == 0 and dm[0, 0, 0] == -1
    dist, grad = orc.esdf_distance(p[None])
    assert dist[0] == d - 1.5 and (grad == 0).all()


def test_outside_and_border_half_cell(corridor):
    """NaN and a zero gradient outside the box and for non-finite points; in the outer half cell of a face the two
    corners along that axis are the same cell, so the gradient along it is exactly 0"""
    cfg, orc, ex, pose = corridor
    d, c = cfg.subbox_d_xyz, pose[:3]
    orc.build_esdf(c - 1.0, c + 1.0, 1.0)
    val, _, _, lo = orc.export_esdf_exact()
    dims = np.array(val.shape[::-1])
    lo_w, hi_w = lo * d, (lo + dims) * d
    bad = np.array([[np.nan, c[1], c[2]], [c[0], np.inf, c[2]], [c[0], c[1], -np.inf], lo_w - d * 0.01, hi_w,
                    [2.0 ** 30 * d, c[1], c[2]]])
    dist, grad = orc.esdf_distance(bad)
    assert np.isnan(dist).all() and (grad == 0).all()
    assert same_bits(dist, query(val, lo, d, bad)[0])
    rs = np.random.RandomState(9)
    for k in range(3):
        p = rs.uniform(lo_w + d, hi_w - d, (200, 3))
        p[:100, k] = lo_w[k] + rs.uniform(0.0, 0.49, 100) * d
        p[100:, k] = hi_w[k] - rs.uniform(0.01, 0.5, 100) * d
        dist, grad = orc.esdf_distance(p)
        assert np.isfinite(dist).all() and (grad[:, k] == 0).all()
        sdist, sgrad = query(val, lo, d, p)
        assert same_bits(dist, sdist) and same_bits(grad, sgrad)


def test_esdf_abi_rejects_bad_arguments_without_a_device():
    if not mlm.library_path().exists():
        mlm.build_library()
    lib = mlm.load_library()
    a = (C.c_double * 3)(0.0, 0.0, 0.0)
    b = (C.c_double * 3)(1.0, 1.0, 1.0)
    assert lib.mlm_esdf_build(None, a, b, 1.0, 0) == 1
    assert lib.mlm_esdf_build(None, a, b, 1.0, 2) == 1
    p, out = (C.c_double * 3)(), (C.c_double * 3)()
    lo, dims = (C.c_int32 * 3)(), (C.c_int32 * 3)()
    for fn in (lib.mlm_esdf_distance, lib.mlm_esdf_distance_device):
        assert fn(None, p, 1, out, out) == 1
        assert fn(None, None, 0, None, None) == 1
    for fn in (lib.mlm_esdf_export, lib.mlm_esdf_export_device):
        assert fn(None, None, 0, lo, dims) == 1
