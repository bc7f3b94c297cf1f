"""GPU: the path-cost matrix (mlm_reach_matrix, k_reach_matrix_*) equals, bit for bit with its NaN and +inf patterns, a
loop of single-start builds (mlm_reach_build + mlm_reach_cost) on every row, and the oracle's loop on a subset of rows:
on the CFG-A trajectory map after inflate_map under every flag combination, on crafted maps (maze, checkerboard,
all-free, all-unknown, negative coordinates), and over a box large enough for several solve launches.  It leaves the
field of the last build untouched, needs no build, its host and device variants agree and the host variant returns its
temporaries to the pool; bad arguments are refused with the stated codes; a world-2 sharded rank refuses it; the C++
mirror's getReachMatrix gives the same matrix."""
import ctypes as C
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

from mlmapping_b200 import MLMap, config_cfg_a, scenes
from mlmapping_b200.capi import MlmError
from esdf_spec import same_bits
from parity_utils import assert_map_parity
from reach_oracle import ReachOracle
from test_capi_staging_gpu import _PoolUsage
from test_parity_gpu import _lidar_small_cfg
from test_reach_gpu import CRAFTED, _restore, crafted  # noqa: F401  (crafted is a fixture)

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
LO_TOL = 1e-6
FLAGS = [(False, False), (True, False), (False, True), (True, True)]


def _loop(m, bmin, bmax, starts, goals, max_dist, inflated=False, unknown=False):
    """the definition: one single-start build per row, its cost query at the goals"""
    out = np.empty((len(starts), len(goals)))
    for i, s in enumerate(starts):
        m.build_reach(bmin, bmax, [s], max_dist, inflated=inflated, unknown=unknown)
        out[i] = m.reach_cost(goals)
    return out


@pytest.fixture(scope="module")
def cfg_a_map():
    """CFG-A, 40 corridor frames at stride 5, inflate_map at the last pose, checked against the oracle's map"""
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
    yield cfg, gpu, orc, pose
    orc.close()
    gpu.close()


def _w1_starts(cfg, gpu, c, bmin, bmax, n_free=30, seed=4):
    """free cells of the box plus a start in an occupied, an unknown and an inflated cell, starts on tile faces, a
    duplicate, one outside the box and one failing rule 1"""
    d = cfg.subbox_d_xyz
    rs = np.random.RandomState(seed)
    pts = rs.uniform(bmin, bmax, (20000, 3))
    occ = gpu.getOccupancy(pts)
    free = pts[occ == 1][:n_free]                              # MLM_FREE
    special = []
    for state in (0, -1):                                      # MLM_OCCUPIED, MLM_UNKNOWN
        w = pts[occ == state]
        if len(w):
            special.append(w[0])
    lo = np.floor(bmin / d)
    special += [(lo + [7, 8, 7] + 0.5) * d, (lo + [8, 15, 16] + 0.5) * d, free[0], c + [1000.0, 0, 0], [np.nan, 0, 0]]
    return np.concatenate([free, np.array(special)]), pts


def test_matrix_cfg_a_w1_box_all_flags(cfg_a_map):
    """about 40 starts against the starts plus 200 random goals, some outside the box: equal to the loop of single GPU
    builds on every row and to the oracle's loop on 6 rows, under every flag combination"""
    cfg, gpu, orc, pose = cfg_a_map
    c = pose[:3]
    half = np.array([6.4, 6.4, 1.6])
    bmin, bmax = c - half, c + half
    starts, pts = _w1_starts(cfg, gpu, c, bmin, bmax)
    n_special = len(starts) - 7                                # occupied, unknown, two tile faces, duplicate, outside
    # starts in free cells of the inflation layer
    infl = pts[(gpu.getOccupancy(pts) == 1) & (gpu.getInflateOccupancy(pts) == 0)]
    starts = np.concatenate([starts, infl[:2]])
    rs = np.random.RandomState(9)
    goals = np.concatenate([starts, rs.uniform(bmin - 1.0, bmax + 1.0, (200, 3))])
    asym = 0
    for inflated, unknown in FLAGS:
        key = (inflated, unknown)
        got = gpu.reach_matrix(bmin, bmax, starts, goals, 30.0, inflated=inflated, unknown=unknown)
        assert got.shape == (len(starts), len(goals))
        want = _loop(gpu, bmin, bmax, starts, goals, 30.0, inflated, unknown)
        assert same_bits(got, want), key
        rows = [0, 7, n_special, n_special + 1, n_special + 5, len(starts) - 1]
        assert same_bits(got[rows], _loop(orc, bmin, bmax, starts[rows], goals, 30.0, inflated, unknown)), key
        assert np.isnan(got).any() and np.isinf(got).any() and (np.isfinite(got) & (got > 0)).sum() > 1000, key
        sq = got[:, :len(starts)]
        asym += int((np.isfinite(sq) & np.isinf(sq.T)).sum())
        # the rows without a source (outside the box, rule 1): +inf in the box, NaN outside
        for i in (n_special + 5, n_special + 6):
            assert set(np.unique(np.where(np.isnan(got[i]), 0, got[i]))) <= {0.0, np.inf}, key
    assert asym > 0


@pytest.mark.parametrize("name", sorted(CRAFTED))
def test_matrix_crafted_maps(crafted, name):  # noqa: F811
    """maze (the most rounds), checkerboard, all-free, negative coordinates, and an all-unknown box beside each: equal
    to the loop of single GPU builds"""
    cfg, gpu, template = crafted
    d = cfg.subbox_d_xyz
    make, origin = CRAFTED[name]
    states = make()
    orc, _ = _restore(cfg, gpu, template, states, origin)
    orc.close()
    o = np.array(origin)
    bmin, bmax = (o + 0.5) * d, (o + np.array(states.shape[::-1]) - 0.5) * d
    rs = np.random.RandomState(3)
    fz, fy, fx = np.nonzero(states == b"f")
    pick = rs.choice(len(fx), min(12, len(fx)), replace=False)
    starts = np.concatenate([(o + np.stack([fx[pick], fy[pick], fz[pick]], 1) + 0.5) * d,
                             (o + np.array([[1, 0, 0], [0, 1, 0]]) + 0.5) * d])   # blocked cells in most patterns
    goals = np.concatenate([starts, rs.uniform(bmin - 0.5, bmax + 0.5, (150, 3))])
    for inflated, unknown in FLAGS:
        got = gpu.reach_matrix(bmin, bmax, starts, goals, 1e4, inflated=inflated, unknown=unknown)
        assert same_bits(got, _loop(gpu, bmin, bmax, starts, goals, 1e4, inflated, unknown)), (name, inflated, unknown)
    if name == "maze":
        assert np.nanmax(np.where(np.isinf(got), np.nan, got)) > 500 * d
    far_lo = (o + np.array([200, 200, 0]) + 0.5) * d
    far_hi = far_lo + np.array([20, 20, 8]) * d
    s2 = np.array([far_lo, far_lo + 3 * d, far_hi])
    for unknown in (False, True):
        got = gpu.reach_matrix(far_lo, far_hi, s2, s2, 1e4, unknown=unknown)
        assert same_bits(got, _loop(gpu, far_lo, far_hi, s2, s2, 1e4, unknown=unknown)), ("unknown box", unknown)
        assert np.isfinite(got).all() if unknown else (np.isfinite(got) == np.eye(3, dtype=bool)).all()


def test_matrix_over_several_launches(cfg_a_map):
    """a 480 x 480 x 160 box with unknown cells traversable: at most 2^28 / 36.9 M = 7 fields per launch, so 15 starts
    take 3 launches; equal to the loop of single builds"""
    cfg, gpu, _, pose = cfg_a_map
    c = pose[:3]
    d = cfg.subbox_d_xyz
    half = np.array([240, 240, 80]) * d
    bmin, bmax = c - half, c + half - d
    rs = np.random.RandomState(12)
    starts = np.concatenate([[c], rs.uniform(bmin, bmax, (14, 3))])
    goals = np.concatenate([starts, rs.uniform(bmin - 1.0, bmax + 1.0, (100, 3))])
    l0 = gpu.kernel_launch_count()
    got = gpu.reach_matrix(bmin, bmax, starts, goals, 80.0, unknown=True)
    assert gpu.kernel_launch_count() - l0 == 1 + 3 * 3               # one gather, three batches of seed / solve / rows
    assert same_bits(got, _loop(gpu, bmin, bmax, starts, goals, 80.0, unknown=True))
    assert (np.isfinite(got) & (got > 10.0)).sum() > 100


def test_matrix_lifetime_and_variants(cfg_a_map):
    """the matrix leaves the built field as it was; a fresh handle needs no build; host = device variant; the host
    variant's temporaries go back to the stream-ordered pool"""
    cfg, gpu, _, pose = cfg_a_map
    c = pose[:3]
    bmin, bmax = c - [5.0, 5.0, 1.5], c + [5.0, 5.0, 1.5]
    rs = np.random.RandomState(21)
    pts = rs.uniform(bmin - 0.3, bmax + 0.3, (3000, 3))
    gpu.build_reach(bmin, bmax, [c], 20.0, inflated=True)
    cost0, (cells0, len0), (g0, lo0) = gpu.reach_cost(pts), gpu.reach_paths(pts[:500], 64), gpu.export_reach()
    starts = np.concatenate([[c], rs.uniform(bmin, bmax, (9, 3))])
    # a larger box than the field's: the matrix grows its own scratch, never the field's
    m1 = gpu.reach_matrix(c - [8.0, 8.0, 2.0], c + [8.0, 8.0, 2.0], starts, pts[:300], 25.0, unknown=True)
    assert same_bits(gpu.reach_cost(pts), cost0)
    cells1, len1 = gpu.reach_paths(pts[:500], 64)
    assert np.array_equal(len1, len0) and np.array_equal(cells1, cells0)
    g1, lo1 = gpu.export_reach()
    assert np.array_equal(g1, g0) and np.array_equal(lo1, lo0)
    # host = device variant
    ns, ng = starts.shape[0], 300
    d_s, d_g, d_o = gpu.to_device(starts), gpu.to_device(np.ascontiguousarray(pts[:300])), gpu.device_alloc(8 * ns * ng)
    gpu.reach_matrix_device(c - [8.0, 8.0, 2.0], c + [8.0, 8.0, 2.0], d_s, ns, d_g, ng, 25.0, d_o, unknown=True)
    assert same_bits(gpu.to_host(d_o, (ns, ng), np.float64), m1)
    for p in (d_s, d_g, d_o):
        gpu.device_free(p)
    pool = _PoolUsage()
    gpu.sync()
    base = pool.used()
    gpu.reach_matrix(bmin, bmax, starts, pts[:300], 25.0)
    assert pool.used() == base
    # a fresh handle with the same map and no build
    fresh = MLMap(cfg)
    fresh.restore(gpu.checkpoint())
    with pytest.raises(MlmError):
        fresh.reach_cost([c])
    m2 = fresh.reach_matrix(c - [8.0, 8.0, 2.0], c + [8.0, 8.0, 2.0], starts, pts[:300], 25.0, unknown=True)
    assert same_bits(m2, m1)
    with pytest.raises(MlmError):                                     # still no field
        fresh.reach_cost([c])
    fresh.close()


def test_matrix_arguments(cfg_a_map):
    """every refusal returns its code and leaves the earlier field usable; the empty matrix is MLM_OK"""
    cfg, gpu, _, pose = cfg_a_map
    c = pose[:3]
    d = cfg.subbox_d_xyz
    gpu.build_reach(c - 2.0, c + 2.0, [c], 10.0)
    want = gpu.reach_cost([c + 0.5, c])
    lib, h = gpu._lib, gpu._h
    a = (C.c_double * 3)(*(c - 1.0))
    b = (C.c_double * 3)(*(c + 1.0))
    s = (C.c_double * 3)(*c)
    out = (C.c_double * 4)()
    nan, inf = float("nan"), float("inf")
    for fn in (lib.mlm_reach_matrix, lib.mlm_reach_matrix_device):
        dev = fn is lib.mlm_reach_matrix_device
        if dev:
            d_s, d_o = gpu.to_device(np.array([c])), gpu.device_alloc(8)
            s_, o_ = C.c_void_p(d_s), C.c_void_p(d_o)
        else:
            s_, o_ = s, out
        assert fn(None, a, b, s_, 1, s_, 1, 10.0, 0, o_) == 1
        assert fn(h, None, b, s_, 1, s_, 1, 10.0, 0, o_) == 1
        assert fn(h, a, None, s_, 1, s_, 1, 10.0, 0, o_) == 1
        assert fn(h, a, b, None, 1, s_, 1, 10.0, 0, o_) == 1
        assert fn(h, a, b, s_, 1, None, 1, 10.0, 0, o_) == 1
        assert fn(h, a, b, s_, 1, s_, 1, 10.0, 0, None) == 1
        assert fn(h, a, b, s_, 1 << 40, s_, 1 << 40, 10.0, 0, o_) == 1          # n_starts * n_goals overflows
        assert fn(h, a, b, s_, 1, s_, 1, 10.0, 4, o_) == 1                      # flags
        for md in (0.0, -1.0, nan, inf):
            assert fn(h, a, b, s_, 1, s_, 1, md, 0, o_) == 1
        for bad in ((nan, 0, 0), (0, inf, 0), tuple(c + [5.0, 0, 0])):
            assert fn(h, (C.c_double * 3)(*bad), b, s_, 1, s_, 1, 10.0, 0, o_) == 1
        x0 = 0.05
        assert fn(h, (C.c_double * 3)(x0, 0.05, 0.05), (C.c_double * 3)(x0 + 4096 * d, 0.05, 0.05), s_, 1, s_, 1, 10.0,
                  0, o_) == 5
        big = 4095.5 * d
        assert fn(h, (C.c_double * 3)(0, 0, 0), (C.c_double * 3)(big, big, 20.5 * d), s_, 1, s_, 1, 10.0, 0, o_) == 5
        assert fn(h, a, b, s_, 1, s_, 1, float(1 << 30) / 1000.0 * d * 2, 0, o_) == 5   # K > 2^30
        # the empty matrix
        assert fn(h, a, b, None, 0, s_, 1, 10.0, 0, None) == 0
        assert fn(h, a, b, s_, 1, None, 0, 10.0, 0, None) == 0
        if dev:
            gpu.device_free(d_s)
            gpu.device_free(d_o)
        assert same_bits(gpu.reach_cost([c + 0.5, c]), want)
    assert gpu.reach_matrix(c - 1.0, c + 1.0, np.zeros((0, 3)), [c], 10.0).shape == (0, 1)
    assert gpu.reach_matrix(c - 1.0, c + 1.0, [c], np.zeros((0, 3)), 10.0).shape == (1, 0)
    assert same_bits(gpu.reach_cost([c + 0.5, c]), want)


@pytest.mark.parametrize("world", [1, 2])
def test_sharded_ranks_refuse_reach_matrix(world):
    """a rank of a world-2 sharded map holds only its own subboxes: MLM_ERR_UNSUPPORTED; a world-1 shard answers"""
    from mlmapping_b200.sharded import sharded_group_in_process
    cfg = _lidar_small_cfg()
    ranks = sharded_group_in_process(cfg, world)
    try:
        for r in ranks:
            s = [[1.0, 1.0, 1.0], [2.0, 1.0, 1.0]]
            if world == 1:
                m = r.map.reach_matrix([0.0, 0.0, 0.0], [4.0, 4.0, 2.0], s, s, 3.0, unknown=True)
                assert m[0, 0] == 0.0 and m[1, 1] == 0.0 and np.isfinite(m).all()
                continue
            with pytest.raises(MlmError) as ei:
                r.map.reach_matrix([0.0, 0.0, 0.0], [4.0, 4.0, 2.0], s, s, 3.0)
            assert ei.value.code == 6
    finally:
        for r in ranks:
            r.close()


_CPP = r"""
#include <cstdio>
#include <cstring>
#include <fstream>
#include <iterator>
#include <vector>
#include "mlmap.hpp"
using namespace mlmap_b200;
static std::vector<unsigned char> slurp(const char *p) {
  std::ifstream f(p, std::ios::binary);
  return std::vector<unsigned char>(std::istreambuf_iterator<char>(f), {});
}
int main(int argc, char **argv) {  // config image, checkpoint, starts, goals, box + max_dist, out
  std::vector<unsigned char> cfg = slurp(argv[1]), img = slurp(argv[2]), s = slurp(argv[3]), g = slurp(argv[4]),
                             bx = slurp(argv[5]);
  if (cfg.size() != sizeof(mlm_config)) return 2;
  mlm_config c;
  std::memcpy(&c, cfg.data(), sizeof c);
  mlmap m;
  m.init_map(c);
  m.restore(img);
  const double *b = reinterpret_cast<const double *>(bx.data());
  const size_t ns = s.size() / 24, ng = g.size() / 24;
  std::vector<double> out(ns * ng);
  m.getReachMatrix(Vec3(b[0], b[1], b[2]), Vec3(b[3], b[4], b[5]), reinterpret_cast<const Vec3 *>(s.data()), ns,
                   reinterpret_cast<const Vec3 *>(g.data()), ng, b[6], out.data(), true, false);
  FILE *f = std::fopen(argv[6], "wb");
  std::fwrite(out.data(), sizeof(double), out.size(), f);
  std::fclose(f);
  std::printf("matrix %zu x %zu\n", ns, ng);
  return 0;
}
"""


def test_cpp_mirror_get_reach_matrix(cfg_a_map):
    """getReachMatrix on a handle restored from this map's checkpoint equals the Python result"""
    cfg, gpu, _, pose = cfg_a_map
    c = pose[:3]
    bmin, bmax = c - [4.0, 4.0, 1.5], c + [4.0, 4.0, 1.5]
    rs = np.random.RandomState(31)
    starts = np.concatenate([[c], rs.uniform(bmin, bmax, (7, 3))])
    goals = np.concatenate([starts, rs.uniform(bmin - 0.5, bmax + 0.5, (40, 3))])
    want = gpu.reach_matrix(bmin, bmax, starts, goals, 15.0, inflated=True)
    lib_dir = ROOT / "mlmapping_b200" / "lib"
    with tempfile.TemporaryDirectory() as t:
        t = Path(t)
        (t / "m.cpp").write_text(_CPP)
        exe = t / "m"
        res = subprocess.run(["g++", "-std=c++17", "-O2", str(t / "m.cpp"), "-o", str(exe),
                              "-I" + str(ROOT / "mlmapping_b200" / "include"), "-I" + str(ROOT / "include"),
                              "-L" + str(lib_dir), "-lmlmap_b200", "-Wl,-rpath," + str(lib_dir)],
                             capture_output=True, text=True)
        assert res.returncode == 0, res.stderr[-3000:]
        (t / "cfg").write_bytes(bytes(cfg))
        (t / "img").write_bytes(gpu.checkpoint())
        (t / "s").write_bytes(np.ascontiguousarray(starts).tobytes())
        (t / "g").write_bytes(np.ascontiguousarray(goals).tobytes())
        (t / "b").write_bytes(np.concatenate([bmin, bmax, [15.0]]).tobytes())
        res = subprocess.run([str(exe), *(str(t / n) for n in ("cfg", "img", "s", "g", "b", "out"))],
                             capture_output=True, text=True, timeout=300, env=dict(os.environ))
        assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-2000:]
        got = np.fromfile(t / "out", dtype=np.float64).reshape(want.shape)
    assert same_bits(got, want)
