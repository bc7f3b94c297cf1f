"""Generates tests/golden/reference_pin.json: counters and sha256 digests of everything tests/test_reference_pin.py compares,
on the same seeded inputs, so that those comparisons also hold where the reference's own build is not available.
tests/test_reference_pin.py checks the restatement (and, for the pose forwarding, the product's host code) against these
records on every run, and the reference build against the same records wherever it is available.
Run:  python tests/golden/make_golden_pin.py   (from the reference build when it is available, else from the restatement;
the file records which)"""
import ctypes as C
import hashlib
import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent))

from mlmapping_b200 import config_cfg_a, config_cfg_b, config_cfg_c, scenes  # noqa: E402
from oracle_binding import Oracle, _d7, load_oracle, load_reference  # noqa: E402

from golden.make_golden import _quat_mul  # noqa: E402

COUNTERS = ("n_points", "n_inside", "n_cast", "n_hit_cells", "n_miss_cells", "n_touched_voxels", "hit_bucket_count",
            "ram_expand_cnt", "obs_cnt")


def d(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:20]


def rolled(pose, k):
    a, b = 0.05 * np.sin(0.7 * k), 0.04 * np.cos(0.9 * k)
    q = _quat_mul(pose[3:7], _quat_mul([np.cos(a / 2), np.sin(a / 2), 0, 0], [np.cos(b / 2), 0, np.sin(b / 2), 0]))
    return np.r_[pose[:3], q]


def frame(o):
    """counters, the hit map in its iteration order with its probabilities, the miss set in ITS iteration order"""
    st = o.frame_stats()
    keys, p = o.last_frame_hits()
    return {"counters": [int(getattr(st, f)) for f in COUNTERS], "hits_in_order": d(keys), "hit_p": d(p),
            "miss_in_order": d(o.last_frame_misses(sort=False))}


def whole_map(o):
    m = o.export_map()
    return {k: d(m[k]) for k in sorted(m)} | {"subboxes": int(m["glb"].shape[0])}, m


def cloud(a):
    return {"n": int(a.shape[0]), "in_order": d(a)}


def depth_trajectory(impl):
    cfg = config_cfg_a()
    cfg.inflate_n, cfg.inflate_global_n = 2, 2
    o = Oracle(cfg, impl=impl)
    out = {"frames": []}
    for k in range(6):
        pose = rolled(scenes.corridor_trajectory_pose(35 * k), k)
        o.integrate_depth(scenes.corridor_depth_frame(cfg, pose, rows=240, cols=320, frame_idx=k), pose)
        out["frames"].append(frame(o))
    out["map"], m = whole_map(o)
    lo, hi = m["glb"].min(0) * 1.0, (m["glb"].max(0) + 1) * 1.0
    pos = scenes.query_positions(30000, lo, hi, seed=5, inflate=2.0)
    out["getOccupancy"], out["getOdd"] = d(o.getOccupancy(pos)), d(o.getOdd(pos))
    out["getOddGrad"] = d(o.getOddGrad(pos[:8000]))
    out["getOccupancy_inflate"] = d(o.getOccupancy(pos[:3000], inflate=0.2))
    o.inflate_map(pose[:3])
    o.setFree_map_in_bound([pose[0] + 0.5, -0.4, 0.8], [pose[0] + 1.5, 0.4, 1.6])
    out["map_after_inflate_set_free"], _ = whole_map(o)
    out["getInflateOccupancy"] = d(o.getInflateOccupancy(pos[:5000]))
    out["cloud_inflated"], out["cloud_occupied"] = cloud(o.export_cloud(0)), cloud(o.export_cloud(1))
    out["odds_slice_1.25"] = cloud(o.export_odds_slice(1.25))
    return out


def exploration(impl):
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    o = Oracle(cfg, impl=impl)
    out = {"frames": [], "released": []}
    for k in range(10):
        pose = scenes.corridor_trajectory_pose(12 * k)
        o.integrate_depth(scenes.corridor_depth_frame(cfg, pose, rows=240, cols=320, frame_idx=k), pose)
        out["frames"].append(frame(o))
        out["released"].append(int(o.lib.orc_released_last(o.h)))
    out["map"], m = whole_map(o)
    out["frontier_cells"] = int(np.unpackbits(m["frontier"]).sum())
    out["cloud_frontier"] = cloud(o.export_cloud(2))
    return out


def lidar_and_cfg_b(impl):
    cfg = config_cfg_c()
    cfg.am_n_rho, cfg.am_n_z_below, cfg.am_n_z_over = 120, 30, 30
    o = Oracle(cfg, impl=impl)
    out = {"lidar_frames": []}
    for k in range(2):
        pose = scenes.lidar_loop_pose(5 * k)
        o.integrate_points(scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512), pose)
        out["lidar_frames"].append(frame(o))
    out["lidar_map"], _ = whole_map(o)
    cfg = config_cfg_b()
    o = Oracle(cfg, impl=impl)
    pose = scenes.corridor_trajectory_pose(3, step=0.1)
    o.integrate_depth(scenes.corridor_depth_frame(cfg, pose, rows=192, cols=256, frame_idx=3, length=200.0), pose)
    out["cfg_b_frame"] = frame(o)
    out["cfg_b_map"], _ = whole_map(o)
    return out


def sampled_projection(impl):
    """mlmapping_sample_cnt > 0: pixels drawn from glibc's rand() stream after srand(1)"""
    cfg = config_cfg_a()
    cfg.sample_cnt = 400
    pose = scenes.corridor_trajectory_pose(7)
    img = scenes.corridor_depth_frame(cfg, pose, frame_idx=7)
    C.CDLL("libc.so.6").srand(1)
    o = Oracle(cfg, impl=impl)
    for _ in range(3):
        o.integrate_depth(img, pose)
    pts = o.points()
    out = {"points": {"n": int(pts.shape[0]), "in_order": d(pts)}, "frame": frame(o)}
    out["map"], _ = whole_map(o)
    return out


def prologue_inputs():
    """the random poses, points and callback states of the prologue / pose-forwarding comparison"""
    rng = np.random.default_rng(0)
    tls = []
    for i in range(1500):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        if i % 3 == 0:
            q = q * rng.uniform(0.5, 2)
        Twb = np.r_[rng.uniform(-50, 50, 3), q]
        q2 = rng.normal(size=4)
        Tbs = np.r_[rng.uniform(-1, 1, 3), q2 / np.linalg.norm(q2)] if i % 2 else np.r_[0.12, 0, 0, 0.5, -0.5, 0.5, -0.5]
        tls.append((Twb, Tbs, rng.uniform(-10, 10, 3)))
    fwd = []
    for i in range(300):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        pos, lv, av = rng.uniform(-5, 5, 3), rng.uniform(-2, 2, 3), rng.uniform(-1, 1, 3)
        fwd.append((pos, q, lv, av, rng.uniform(0, 0.05), rng.uniform(0, 0.05), rng.uniform(0, 0.01)))
    return tls, fwd


def prologue_outputs(lib):
    """T_ls = T_wa^-1 * (T_wb * T_bs), T_ls * p and the callback's pose forwarding of one library, as arrays"""
    tls, fwd = prologue_inputs()
    T, P, F = np.empty((len(tls), 7)), np.empty((len(tls), 3)), np.empty((len(fwd), 7))
    for i, (Twb, Tbs, pt) in enumerate(tls):
        o7, o3 = (C.c_double * 7)(), (C.c_double * 3)()
        lib.orc_T_ls(_d7(Twb), _d7(Tbs), o7)
        lib.orc_transform_point(_d7(Twb), _d7(Tbs), _d7(pt), o3)
        T[i], P[i] = list(o7), list(o3)
    for i, (pos, q, lv, av, go, gi, lat) in enumerate(fwd):
        o7 = (C.c_double * 7)()
        lib.orc_compensate_pose(_d7(pos), _d7(q), _d7(lv), _d7(av), go, gi, lat, o7)
        F[i] = list(o7)
    return T, P, F


def prologue(impl):
    T, P, F = prologue_outputs(load_reference() if impl == "reference" else load_oracle())
    return {"T_ls": d(T), "transform_point": d(P), "compensate_pose": d(F)}


def odd_by_index_cells(o):
    """the map after one frame and 2000 (subbox, cell) pairs of it, with their log-odds"""
    cfg = o.cfg
    pose = scenes.corridor_trajectory_pose(0)
    o.integrate_depth(scenes.corridor_depth_frame(cfg, pose, rows=120, cols=160), pose)
    m = o.export_map()
    rs = np.random.RandomState(3)
    sel = rs.randint(0, m["glb"].shape[0], 2000)
    sub = rs.randint(0, 1000, 2000).astype(np.int32)
    return m, np.ascontiguousarray(m["glb"][sel].astype(np.int32)), sub, m["log_odds"][sel, sub]


def odd_by_index(impl):
    o = Oracle(config_cfg_a(), impl=impl)
    m, glb, sub, lo = odd_by_index_cells(o)
    return {"map": whole_map(o)[0], "cells": d(glb) + d(sub), "log_odds": d(lo)}


CASES = {"depth_trajectory": depth_trajectory, "exploration": exploration, "lidar_and_cfg_b": lidar_and_cfg_b,
         "sampled_projection": sampled_projection, "prologue": prologue, "odd_by_index": odd_by_index}


def run_case(name, impl="port"):
    return json.loads(json.dumps(CASES[name](impl)))  # the shape the file stores (tuples as lists)


if __name__ == "__main__":
    from oracle_binding import reference_available
    impl = "reference" if reference_available() else "port"
    out = {"generator": "tests/golden/make_golden_pin.py", "impl": impl,
           "provenance": ("outputs of the reference's own build (oracle/_ref)" if impl == "reference" else
                          "outputs of the restatement (oracle/mlmap_oracle.hpp, unchanged since it was checked bit for bit "
                          "against the reference's own build on these inputs by tests/test_reference_pin.py); the "
                          "reference build is held to the same records wherever it is available"),
           "cases": {c: run_case(c, impl) for c in CASES}}
    (HERE / "reference_pin.json").write_text(json.dumps(out, indent=1) + "\n")
    print({c: len(json.dumps(v)) for c, v in out["cases"].items()})
