"""CPU: the C++ oracle's ray casting (orc_cast_rays) equals the written spec (tests/raycast_spec.py) bit for bit on both
layers, the records satisfy the spec's invariants, and the C ABI rejects bad arguments without a device."""
import ctypes as C

import numpy as np
import pytest

import mlmapping_b200 as mlm
from mlmapping_b200 import capi, config_cfg_a, scenes
from ray_oracle import RayOracle
from raycast_spec import FREE, OCCUPIED, MapStates, cast_rays, edge_segments, first_difference, random_segments


@pytest.fixture(scope="module")
def corridor():
    """CFG-A, 10 corridor frames, then inflate_map at the last pose"""
    cfg = config_cfg_a()
    orc = RayOracle(cfg)
    for k in range(10):
        pose = scenes.corridor_trajectory_pose(k * 5)
        orc.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    orc.inflate_map(pose[:3])
    ex = orc.export_map()
    n, d = cfg.subbox_n, cfg.subbox_d_xyz
    f1, t1 = random_segments(2000, ex["glb"].min(0) * n * d, (ex["glb"].max(0) + 1) * n * d, seed=11, max_len=8.0)
    f2, t2 = edge_segments(ex, n, d, seed=12, n_each=100)
    return cfg, orc, ex, np.concatenate([f1, f2]), np.concatenate([t1, t2])


@pytest.mark.parametrize("inflated", [False, True])
def test_oracle_rays_equal_the_spec(corridor, inflated):
    cfg, orc, ex, f, t = corridor
    assert f.shape[0] >= 3000
    states = MapStates(ex, cfg.subbox_n)
    want, paths = cast_rays(f, t, cfg.subbox_d_xyz, states, inflated)
    got = orc.cast_rays(f, t, inflated=inflated)
    assert first_difference(got, want) is None, first_difference(got, want)
    st = got["status"]
    # the set covers every outcome, walks through several subboxes, and blocks at the start cell
    assert (st == FREE).sum() > 300 and (st == OCCUPIED).sum() > 300 and (st == capi.RAY_INVALID).sum() >= 13
    assert max(len(p) for p in paths) > 3 * cfg.subbox_n
    assert sum(1 for p, s in zip(paths, st) if s == OCCUPIED and len(p) == 1) >= 50
    # invariants
    for i in range(f.shape[0]):
        r, path = got[i], paths[i]
        if r["status"] == capi.RAY_INVALID:
            assert not path and r["n_free"] == r["n_unknown"] == 0 and tuple(r["cell"]) == (0, 0, 0) and r["t"] == 0.0
            continue
        c0 = [int(np.floor(v / cfg.subbox_d_xyz)) for v in f[i]]
        e = [int(np.floor(v / cfg.subbox_d_xyz)) for v in t[i]]
        assert list(path[0]) == c0 and tuple(r["cell"]) == path[-1]
        assert all(sum(abs(a - b) for a, b in zip(p, q)) == 1 for p, q in zip(path, path[1:]))   # 6-connected
        assert 0.0 <= r["t"] <= 1.0 and (len(path) > 1 or r["t"] == 0.0)
        blocking = [states(c)[0] == b"o" or (inflated and states(c)[1] == b"o") for c in path]
        assert not any(blocking[:-1])
        if r["status"] == FREE:
            assert list(path[-1]) == e and not blocking[-1]
            assert r["n_free"] + r["n_unknown"] == sum(abs(a - b) for a, b in zip(e, c0)) + 1
        else:
            assert blocking[-1] and r["n_free"] + r["n_unknown"] == len(path) - 1
        assert r["n_free"] == sum(states(c)[0] == b"f" for c in path[:len(path) - (r["status"] == OCCUPIED)])


def test_inflation_layer_blocks_earlier(corridor):
    cfg, orc, ex, f, t = corridor
    a, b = orc.cast_rays(f, t), orc.cast_rays(f, t, inflated=True)
    assert (b["status"] == OCCUPIED).sum() > (a["status"] == OCCUPIED).sum()
    both = (a["status"] == OCCUPIED) & (b["status"] == OCCUPIED)
    assert (b["t"][both] <= a["t"][both]).all()


def test_ray_abi_rejects_bad_arguments_without_a_device():
    if not mlm.library_path().exists():
        mlm.build_library()
    lib = mlm.load_library()
    assert lib.mlm_sizeof_ray_hit() == C.sizeof(capi.RayHit) == capi.RAY_HIT_DTYPE.itemsize == 32
    out = (capi.RayHit * 1)()
    p = (C.c_double * 3)(0.0, 0.0, 0.0)
    for fn in (lib.mlm_cast_rays, lib.mlm_cast_rays_device):
        assert fn(None, p, p, 1, 0, out) == 1           # null handle
        assert fn(None, None, None, 0, 0, None) == 1
        assert fn(None, None, p, 1, 0, out) == 1
        assert fn(None, p, p, 1, 2, out) == 1           # flags other than 0 / MLM_RAY_INFLATED
