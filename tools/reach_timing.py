"""Reachability-field timing (mlm_reach_build: k_esdf_gather / k_reach_seed / k_reach_solve; mlm_reach_cost_device:
k_reach_cost; mlm_reach_paths_device: k_reach_paths), L2 flushed before every timed pass, CUDA events on the handle's
stream, 3 warm-up passes then 10 timed, medians reported.  The per-kernel split of a build is not measured.

  W1  the distance field's W1 box: the CFG-A map of the bench (200 corridor frames, then inflate_map), box = last pose
      +- (6.4, 6.4, 1.6) m, the source at the last pose, max_dist 30 m, both layers.  The field is checked against the
      oracle's restatement in the same run; the oracle's single-core Dijkstra and scipy's Dijkstra over the same class
      grid are the CPU baselines.
  W2  the CFG-C hall after its 100 scans: 600 x 600 x 60 cells, the source at the last scan pose, unknown cells
      traversable (the optimistic mode), max_dist 200 m.
  W3  the crafted serpentine maze of tests/test_reach_gpu.py at 96 x 97 x 9 cells: one corridor through every tile,
      the worst case for the number of rounds.
  W4  2 M cost queries and 10 k paths (at most 512 cells each) on the W1 inflated field.
Writes one JSON file (--out)."""
import argparse
import json
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))
from mlmapping_b200 import MLMap, config_cfg_a, config_cfg_c, scenes  # noqa: E402
from ray_timing import card  # noqa: E402

REPS, WARM = 13, 3


def timed(m, fn):
    ms = []
    for rep in range(REPS):
        m.flush_l2()
        m.timer_start()
        fn()
        t = m.timer_stop_ms()
        if rep >= WARM:
            ms.append(t)
    return {"ms_median": float(np.median(ms)), "ms_min": float(np.min(ms)), "ms_max": float(np.max(ms))}


def build_leg(m, box, starts, max_dist, inflated=False, unknown=False):
    r = timed(m, lambda: m.build_reach(box[0], box[1], starts, max_dist, inflated=inflated, unknown=unknown))
    g, lo = m.export_reach()
    r.update({"box_min": np.asarray(box[0]).tolist(), "box_max": np.asarray(box[1]).tolist(),
              "dims": list(g.shape[::-1]), "cells": int(g.size), "reached": int((g >= 0).sum()),
              "max_cost": int(g.max()), "inflated": inflated, "unknown": unknown})
    r["cells_per_s"] = g.size / (r["ms_median"] * 1e-3)
    return r, g, lo


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "reach_timing.json"))
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--scans", type=int, default=100)
    args = ap.parse_args()
    res = {"tool": "tools/reach_timing.py", **card(), "timed_passes": REPS - WARM, "l2_flushed": True,
           "per_kernel_split": "not measured", "legs": {}}

    # ---- W1 and W4
    cfg = config_cfg_a()
    m = MLMap(cfg)
    for k in range(args.frames):
        pose = scenes.corridor_trajectory_pose(k)
        m.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    m.inflate_map(pose[:3])
    c = pose[:3]
    half = np.array([6.4, 6.4, 1.6])
    w1 = (c - half, c + half)
    grids = {}
    for inflated in (False, True):
        r, g, lo = build_leg(m, w1, [c], 30.0, inflated=inflated)
        grids[inflated] = (g, lo)
        res["legs"]["w1_inflated" if inflated else "w1"] = r
    nq, npaths, mc = 2_000_000, 10_000, 512
    q = np.ascontiguousarray(scenes.query_positions(nq, w1[0], w1[1], seed=5, frac_inside=1.0))
    d_q, d_o = m.to_device(q), m.device_alloc(8 * nq)
    r = timed(m, lambda: m.reach_cost_device(d_q, nq, d_o))
    r["points_per_s"] = nq / (r["ms_median"] * 1e-3)
    res["legs"]["w4_cost_queries"] = {"points": nq, "field": "w1_inflated", **r}
    g, lo = grids[True]
    reach = np.argwhere(g > 0)[np.random.RandomState(2).choice(int((g > 0).sum()), npaths)]
    goals = np.ascontiguousarray(((reach[:, ::-1] + lo) + 0.5) * cfg.subbox_d_xyz)
    d_g, d_c, d_l = m.to_device(goals), m.device_alloc(12 * npaths * mc), m.device_alloc(4 * npaths)
    r = timed(m, lambda: m.reach_paths_device(d_g, npaths, mc, d_c, d_l))
    ln = m.to_host(d_l, (npaths,), np.int32)
    res["legs"]["w4_paths"] = {"goals": npaths, "max_cells": mc, "mean_length": float(ln.mean()),
                               "max_length": int(ln.max()), "field": "w1_inflated", **r}
    for p in (d_q, d_o, d_g, d_c, d_l):
        m.device_free(p)
    m.close()
    from reach_oracle import ReachOracle
    from reach_spec import box_classes, field, source_cells, budget
    orc = ReachOracle(cfg)
    for k in range(args.frames):
        pose = scenes.corridor_trajectory_pose(k)
        orc.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    orc.inflate_map(pose[:3])
    ex = orc.export_map()
    bad = []
    for inflated in (False, True):
        key = "w1_inflated" if inflated else "w1"
        secs = []
        for _ in range(3):
            orc.build_reach(w1[0], w1[1], [c], 30.0, inflated=inflated)
            secs.append(orc.last_seconds)
        o, _ = orc.export_reach()
        if not np.array_equal(o, grids[inflated][0]):
            bad.append((key, int((o != grids[inflated][0]).sum())))
        lo_, dims, cls = box_classes(ex, cfg.subbox_n, cfg.subbox_d_xyz, w1[0], w1[1], inflated)
        src = source_cells([c], lo_, dims, cfg.subbox_d_xyz)
        t0 = time.perf_counter()
        field(cls, src, budget(30.0, cfg.subbox_d_xyz))
        leg = res["legs"][key]
        leg["oracle_build_ms_one_core"] = float(np.median(secs)) * 1e3
        leg["scipy_ms_one_core"] = (time.perf_counter() - t0) * 1e3
        leg["speedup_vs_oracle"] = leg["oracle_build_ms_one_core"] / leg["ms_median"]
    res["w1_parity"] = "ok" if not bad else f"MISMATCH {bad}"
    orc.close()

    # ---- W2: the CFG-C hall
    cfg = config_cfg_c()
    m = MLMap(cfg)
    for k in range(args.scans):
        pose = scenes.lidar_loop_pose(k)
        m.integrate_points(scenes.lidar_scan(pose, frame_idx=k), pose)
    d = cfg.subbox_d_xyz
    w2 = (np.array([-60.0, -60.0, 0.0]), np.array([60.0 - d / 2, 60.0 - d / 2, 12.0 - d / 2]))
    res["legs"]["w2"], _, _ = build_leg(m, w2, [pose[:3]], 200.0, unknown=True)
    m.close()

    # ---- W3: the serpentine maze
    from test_reach_gpu import _serpentine
    from view_spec import crafted_map, write_map_checkpoint
    cfg = config_cfg_a()
    cfg.use_exploration_frontiers = 1
    m = MLMap(cfg)
    states = _serpentine(96, 97, 9)
    cells = {(x, y, z): s for (z, y, x), s in np.ndenumerate(states)}
    m.restore(write_map_checkpoint(m.checkpoint(), cfg, crafted_map(cells, cfg.subbox_n)))
    d = cfg.subbox_d_xyz
    w3 = (np.array([0.5, 0.5, 0.5]) * d, (np.array(states.shape[::-1]) - 0.5) * d)
    res["legs"]["w3_maze"], g, _ = build_leg(m, w3, [w3[0]], 1e5)
    res["legs"]["w3_maze"]["corridor_cells"] = int((states == b"f").sum())
    m.close()
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(res, indent=1, default=str) + "\n")
    print(json.dumps(res, default=str))


if __name__ == "__main__":
    main()
