"""Candidate-view gain on one B200: mlm_view_gain for 256 and 2048 FUEL-style candidates (rings of 1-3 m around the
frontier clusters, looking at their centroids) at max_depth 3 m and 5 m on the CFG-A exploration map (30 corridor frames
at stride 5, the CFG-A camera 640 x 480, fx 348), both target kinds, and on the small LiDAR exploration map with a
synthetic 320 x 240 camera (fx 160, 0.2-4 m).  Against the oracle on one core (a subset, scaled per view) and the composed
host path a planner has without it (frustum cells enumerated in numpy, getOccupancy, one cast_rays segment per target).
Cells tested and walk steps come from the oracle.  L2 flushed before every timed call, median of 10.  Writes
profiles/view_timing.json (or --out)."""
import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from mlmapping_b200 import MLMap, scenes  # noqa: E402
from test_frontier_host import explore_cfg_a, explore_lidar  # noqa: E402
from view_oracle import ViewOracle  # noqa: E402
from view_spec import candidates_around, sensor, view_cells  # noqa: E402

REPS = 10
ORACLE_VIEWS = 8
HOST_VIEWS = 4


def gpu_info():
    q = "name,power.limit,clocks.max.sm,clocks.sm,clocks.mem"
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), [v.strip() for v in r.stdout.strip().splitlines()[0].split(",")])) if r.returncode == 0 else {}


def median_ms(gpu, fn):
    ts = []
    fn()  # warm-up: scratch allocation, module load
    for _ in range(REPS):
        gpu.flush_l2()
        gpu.sync()
        t0 = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return {"median": round(statistics.median(ts), 4), "min": round(min(ts), 4), "max": round(max(ts), 4)}


def events_ms(gpu, d_p, n, S, d_o, frontier):
    """CUDA events on the handle's stream around the device variant (kernels only, no staging)"""
    gpu.view_gain_device(d_p, n, S, d_o, frontier=frontier)
    ev = []
    for _ in range(REPS):
        gpu.flush_l2()
        gpu.timer_start()
        gpu.view_gain_device(d_p, n, S, d_o, frontier=frontier)
        ev.append(gpu.timer_stop_ms())
    return {"median": round(statistics.median(ev), 4), "min": round(min(ev), 4)}


def composed_host_path(gpu, cfg, poses, S):
    """per view: frustum cells in numpy, their state by getOccupancy, one cast_rays segment per unknown target"""
    d = cfg.subbox_d_xyz
    vis = 0
    for pose in poses:
        o, co, cells = view_cells(pose, S, d, list(cfg.T_bs))
        x = (cells + 0.5) * d
        tgt = cells[gpu.getOccupancy(x) == -1]
        rec = gpu.cast_rays(np.tile(np.array(o), (len(tgt), 1)), (tgt + 0.5) * d)
        vis += int(((rec["cell"] == tgt).all(1) & (rec["n_free"] == np.abs(tgt - np.array(co)).sum(1))).sum())
    return vis


def measure(name, gpu, orc, cfg, S_of, depths, sizes):
    rec = gpu.frontier_clusters()
    rows = {"frontier_cells": int(rec["n_cells"].sum()), "clusters": int(rec.size)}
    rs = np.random.RandomState(7)
    for depth in depths:
        S = S_of(depth)
        for n in sizes:
            poses, _ = candidates_around(rec["centroid"], list(cfg.T_bs), seed=n, per_cluster=n // rec.size + 1)
            poses = poses[rs.permutation(poses.shape[0])[:n]]
            d_p, d_o = gpu.to_device(poses), gpu.device_alloc(16 * n)
            for frontier in (False, True):
                key = f"{n}_views_{depth}m_{'frontier' if frontier else 'unknown'}"
                g = gpu.view_gain(poses, S, frontier=frontier)
                row = {"n_target_mean": round(float(g["n_target"].mean()), 1),
                       "n_visible_mean": round(float(g["n_visible"].mean()), 1),
                       "host_variant_ms": median_ms(gpu, lambda: gpu.view_gain(poses, S, frontier=frontier)),
                       "device_variant_events_ms": events_ms(gpu, d_p, n, S, d_o, frontier)}
                sub = rs.choice(n, ORACLE_VIEWS, replace=False)
                o = orc.view_gain(poses[sub], S, frontier=frontier)
                row["oracle_equal_on_subset"] = o.tobytes() == g[sub].tobytes()
                per_view_s = orc.last_seconds / ORACLE_VIEWS
                tested, steps = (v / ORACLE_VIEWS for v in orc.last_work)
                row["oracle_one_core_ms_per_view"] = round(1e3 * per_view_s, 3)
                row["oracle_one_core_ms_scaled_to_batch"] = round(1e3 * per_view_s * n, 1)
                row["cells_tested_per_view"] = round(tested)
                row["walk_steps_per_view"] = round(steps)
                t = row["device_variant_events_ms"]["median"] * 1e-3
                row["gpu_cells_tested_per_s"] = float(f"{tested * n / t:.4g}")
                row["gpu_walk_steps_per_s"] = float(f"{steps * n / t:.4g}")
                if not frontier and n == sizes[0]:
                    t0 = time.perf_counter()
                    composed_host_path(gpu, cfg, poses[:HOST_VIEWS], S)
                    row["composed_host_path_ms_per_view"] = round(1e3 * (time.perf_counter() - t0) / HOST_VIEWS, 1)
                rows[key] = row
                print(name, key, json.dumps(row), flush=True)
            gpu.device_free(d_p)
            gpu.device_free(d_o)
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "view_timing.json"))
    args = ap.parse_args()
    out = {"gpu": gpu_info(), "reps": REPS,
           "statistic": "median of 10 calls, L2 flushed before each: host variant by host clock (pose upload, three "
                        "kernels, record copy, stream sync), device variant by CUDA events on the handle's stream",
           "oracle": f"one core, {ORACLE_VIEWS} views of each batch, scaled per view; cells tested and walk steps are "
                     "the oracle's counts per view (its AABB cells and the cells its walks visit), over the GPU's "
                     "event time for the rates",
           "composed_host_path": f"{HOST_VIEWS} views: numpy frustum enumeration over a cube around the origin, "
                                 "getOccupancy, cast_rays per unknown target, per view"}
    cfg = explore_cfg_a()
    gpu, orc = MLMap(cfg), ViewOracle(cfg, bookkeeping=False)
    for k in range(30):
        pose = scenes.corridor_trajectory_pose(k * 5)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    out["cfg_a_exploration_30_frames"] = measure("cfg-a", gpu, orc, cfg, lambda m: sensor(max_depth=m), (3.0, 5.0),
                                                 (256, 2048))
    gpu.close()
    orc.close()
    cfg = explore_lidar()
    gpu, orc = MLMap(cfg), ViewOracle(cfg, bookkeeping=False)
    for k in range(6):
        pose = scenes.lidar_loop_pose(k * 3)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512, max_range=20.0)
        gpu.integrate_points(pts, pose)
        orc.integrate_points(pts, pose)
    lidar_S = lambda m: sensor(fx=160.0, cx=159.5, cy=119.5, cols=320, rows=240, min_depth=0.2, max_depth=m)
    out["lidar_sensor"] = "320 x 240, fx = fy = 160, cx 159.5, cy 119.5, 0.2-4 m, optical axis = body z (T_bs identity)"
    out["lidar_exploration_6_scans"] = measure("lidar", gpu, orc, cfg, lidar_S, (4.0,), (256, 2048))
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(json.dumps(out["gpu"]))


if __name__ == "__main__":
    main()
