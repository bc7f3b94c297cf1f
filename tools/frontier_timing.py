"""Frontier clustering on one B200: mlm_frontier_clusters on the CFG-A exploration map (30 corridor frames at stride 5),
on the small LiDAR exploration map and on a crafted map of ~5 M frontier cells (restored from a checkpoint image),
against the host path a planner has without it (export_frontier + bitmask decode + scipy.ndimage.label) and the oracle on
one core.  L2 flushed before every timed call, median of 10.  Writes profiles/frontier_timing.json (or --out)."""
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

from mlmapping_b200 import MLMap  # noqa: E402
from frontier_oracle import FrontierOracle  # noqa: E402
from frontier_spec import clusters, decode_frontier, frontier_words, label_scipy, write_checkpoint  # noqa: E402
from test_frontier_host import explore_cfg_a, explore_lidar  # noqa: E402
from mlmapping_b200 import scenes  # noqa: E402

REPS = 10


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
    return statistics.median(ts), min(ts), max(ts)


def host_path(gpu, cfg):
    """what a planner does today: the frontier bitmasks to the host (export_frontier), decoded, labelled on the CPU"""
    import ctypes as C
    n = C.c_size_t()
    gpu._lib.mlm_export_map_count(gpu._h, C.byref(n))
    cap, fw = n.value, (cfg.subbox_n ** 3 + 31) // 32
    glb = np.zeros((cap, 3), np.int32)
    words = np.zeros((cap, fw), np.uint32)
    gpu._check(gpu._lib.mlm_export_frontier(gpu._h, cap, glb.ctypes.data, words.ctypes.data, C.byref(n)))
    ex = {"glb": glb, "collapsed": np.zeros(cap, np.uint8), "frontier": words.view(np.uint8)[:, :(cfg.subbox_n ** 3 + 7) // 8]}
    return label_scipy(decode_frontier(ex, cfg.subbox_n))


def measure(name, gpu, cfg, orc=None):
    rec = gpu.frontier_clusters()
    rec6 = gpu.frontier_clusters(conn6=True)
    row = {"frontier_cells": int(rec["n_cells"].sum()), "clusters_26": int(rec.size), "clusters_6": int(rec6.size),
           "largest": int(rec["n_cells"].max(initial=0)), "clusters_ge_10": int((rec["n_cells"] >= 10).sum())}
    t0 = gpu.kernel_launch_count()
    gpu.frontier_clusters()
    row["launches_per_call"] = gpu.kernel_launch_count() - t0
    for key, fn in (("gpu_26_ms", lambda: gpu.frontier_clusters()),
                    ("gpu_6_ms", lambda: gpu.frontier_clusters(conn6=True)),
                    ("gpu_26_min10_labels_ms", lambda: gpu.frontier_clusters(min_cells=10, labels=True)),
                    ("host_export_frontier_decode_scipy_ms", lambda: host_path(gpu, cfg))):
        med, lo, hi = median_ms(gpu, fn)
        row[key] = {"median": round(med, 4), "min": round(lo, 4), "max": round(hi, 4)}
    ev = []
    for _ in range(REPS):  # CUDA events on the handle's stream around the same call (includes the sync bubbles)
        gpu.flush_l2()
        gpu.timer_start()
        gpu.frontier_clusters()
        ev.append(gpu.timer_stop_ms())
    row["gpu_26_events_ms"] = {"median": round(statistics.median(ev), 4), "min": round(min(ev), 4)}
    if orc is not None:
        o = orc.frontier_clusters()
        row["oracle_equal"] = o.tobytes() == rec.tobytes()
        ts = []
        for _ in range(3):
            orc.frontier_clusters()
            ts.append(orc.last_seconds * 1e3)
        row["oracle_one_core_ms"] = round(statistics.median(ts), 3)
    print(name, json.dumps(row), flush=True)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "frontier_timing.json"))
    ap.add_argument("--big-cells", type=int, default=5_000_000)
    args = ap.parse_args()
    out = {"gpu": gpu_info(), "reps": REPS, "statistic": "median of 10 host-clock calls, L2 flushed before each",
           "note": "each call includes its two stream synchronisations and, for the host variant, the record copy"}
    # CFG-A exploration map
    cfg = explore_cfg_a()
    gpu, orc = MLMap(cfg), FrontierOracle(cfg, bookkeeping=False)
    for k in range(30):
        pose = scenes.corridor_trajectory_pose(k * 5)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        gpu.integrate_depth(img, pose)
        orc.integrate_depth(img, pose)
    out["cfg_a_exploration_30_frames"] = measure("cfg-a", gpu, cfg, orc)
    gpu.close()
    orc.close()
    # LiDAR exploration map
    cfg = explore_lidar()
    gpu, orc = MLMap(cfg), FrontierOracle(cfg, bookkeeping=False)
    for k in range(6):
        pose = scenes.lidar_loop_pose(k * 3)
        pts = scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512, max_range=20.0)
        gpu.integrate_points(pts, pose)
        orc.integrate_points(pts, pose)
    out["lidar_exploration_6_scans"] = measure("lidar", gpu, cfg, orc)
    gpu.close()
    orc.close()
    # crafted: random cells at density 1/2 in a box of 2 * big_cells cells (subboxes of 10^3 cells)
    cfg = explore_cfg_a()
    gpu = MLMap(cfg)
    pose = scenes.corridor_trajectory_pose(0)
    gpu.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=0), pose)
    side = int(round((2 * args.big_cells) ** (1 / 3) / 10)) * 10
    rs = np.random.RandomState(1)
    g = np.indices((side, side, side)).reshape(3, -1).T - side // 2
    cells = g[rs.uniform(size=g.shape[0]) < 0.5]
    glb, words = frontier_words(cells, cfg.subbox_n)
    gpu.restore(write_checkpoint(gpu.checkpoint(), cfg, glb, words))
    row = measure("crafted", gpu, cfg)
    t0 = time.perf_counter()
    spec = clusters(cells, cfg.subbox_d_xyz)[0]
    row["numpy_spec_s"] = round(time.perf_counter() - t0, 3)
    row["spec_equal"] = spec.tobytes() == gpu.frontier_clusters().tobytes()
    row["subboxes"] = int(glb.shape[0])
    out["crafted_random_half_density"] = row
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(json.dumps(out["gpu"]))


if __name__ == "__main__":
    main()
