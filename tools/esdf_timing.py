"""Signed-distance-field timing (mlm_esdf_build: k_esdf_gather / k_esdf_x / k_esdf_y / k_esdf_z; mlm_esdf_distance_device:
k_esdf_query), L2 flushed before every timed pass, CUDA events on the handle's stream, 3 warm-up passes then 10 timed,
medians reported.

  W1  local planner box: the CFG-A map of the bench (200 corridor frames, then inflate_map), box = last pose
      +- (6.4, 6.4, 1.6) m, max_dist 2 m, both layers.  The grid is checked against the oracle's restatement in the same
      run; the oracle's single-core build of the same box is the CPU baseline.
  W2  whole map: the CFG-C LiDAR map after its 100 scans, box = the 120 x 120 x 12 m hall (600 x 600 x 60 cells), both
      layers.
  W3  queries: 2 M scenes.query_positions inside the W1 box with gradients, alternated in the same loop with
      mlm_get_odd_grad_device on the same points (the gradient planners use today; the two answer different questions,
      so only their cost is compared).

Algorithmic bytes of a build: 1 B per box cell read (2 B with the inflated layer), 12 B per subbox probed, the grid
written once at 8 B per cell.  Of a query: 24 B in, 32 B out, 64 B gathered (8 corners).  Each as a share of bench.py's
measured_peak_gbs().  Writes one JSON file (--out)."""
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
from bench import measured_peak_gbs  # noqa: E402
from mlmapping_b200 import MLMap, config_cfg_a, config_cfg_c, scenes  # noqa: E402
from ray_timing import card  # noqa: E402

REPS, WARM = 13, 3


def subboxes_probed(lo, dims, n):
    g0, g1 = np.floor_divide(lo, n), np.floor_divide(lo + dims - 1, n)
    return int(np.prod(g1 - g0 + 1))


def build_bytes(lo, dims, n, inflated):
    cells = int(np.prod(dims))
    return cells * (2 if inflated else 1) + 12 * subboxes_probed(lo, dims, n) + 8 * cells


def timed_build(m, box, max_dist, inflated):
    m.flush_l2()
    m.timer_start()
    m.build_esdf(box[0], box[1], max_dist, inflated=inflated)
    return m.timer_stop_ms()


def stats(ms, nbytes, peak):
    med = float(np.median(ms))
    return {"ms_median": med, "ms_min": float(np.min(ms)), "ms_max": float(np.max(ms)), "algorithmic_bytes": nbytes,
            "gbs": nbytes / (med * 1e-3) / 1e9, "share_of_peak": nbytes / (med * 1e-3) / 1e9 / peak}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "esdf_timing.json"))
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--scans", type=int, default=100)
    ap.add_argument("--queries", type=int, default=2_000_000)
    ap.add_argument("--no-oracle", action="store_true", help="skip the W1 oracle check and CPU baseline")
    args = ap.parse_args()
    peak, peak_src = measured_peak_gbs()
    res = {"tool": "tools/esdf_timing.py", **card(), "peak_gbs": peak, "peak_source": peak_src, "timed_passes": REPS - WARM,
           "l2_flushed": True, "max_dist_m": 2.0, "legs": {}}

    # ---- W1: CFG-A bench map, local planner box
    cfg = config_cfg_a()
    m = MLMap(cfg)
    for k in range(args.frames):
        pose = scenes.corridor_trajectory_pose(k)
        m.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    m.inflate_map(pose[:3])
    c = pose[:3]
    half = np.array([6.4, 6.4, 1.6])
    w1 = (c - half, c + half)
    d, n = cfg.subbox_d_xyz, cfg.subbox_n
    times = {False: [], True: [], "query": [], "odd_grad": []}
    nq = args.queries
    q = np.ascontiguousarray(scenes.query_positions(nq, w1[0], w1[1], seed=5, frac_inside=1.0))
    d_q, d_dist, d_grad, d_og = m.to_device(q), m.device_alloc(8 * nq), m.device_alloc(24 * nq), m.device_alloc(24 * nq)
    for rep in range(REPS):
        for inflated in (False, True):
            ms = timed_build(m, w1, 2.0, inflated)
            if rep >= WARM:
                times[inflated].append(ms)
        # W3 on the inflated W1 field, alternating with getOddGrad on the same points
        m.flush_l2()
        m.timer_start()
        m.esdf_distance_device(d_q, nq, d_dist, d_grad)
        ms_q = m.timer_stop_ms()
        m.flush_l2()
        m.timer_start()
        m.getOddGrad_device(d_q, nq, d_og)
        ms_g = m.timer_stop_ms()
        if rep >= WARM:
            times["query"].append(ms_q)
            times["odd_grad"].append(ms_g)
    grids = {}
    for inflated in (False, True):
        m.build_esdf(w1[0], w1[1], 2.0, inflated=inflated)
        g, lo = m.export_esdf()
        grids[inflated] = g
        dims = np.array(g.shape[::-1])
        key = "w1_inflated" if inflated else "w1"
        res["legs"][key] = {"box_min": w1[0].tolist(), "box_max": w1[1].tolist(), "dims": dims.tolist(),
                            "cells": int(g.size), "subboxes_probed": subboxes_probed(lo, dims, n),
                            "blocking_cells": int((g <= 0).sum()),
                            **stats(times[inflated], build_bytes(lo, dims, n, inflated), peak)}
        res["legs"][key]["cells_per_s"] = g.size / (res["legs"][key]["ms_median"] * 1e-3)
    res["legs"]["w3_esdf_query"] = {"points": nq, "gradient": True, "field": "w1_inflated",
                                    **stats(times["query"], nq * (24 + 32 + 64), peak)}
    res["legs"]["w3_esdf_query"]["points_per_s"] = nq / (res["legs"]["w3_esdf_query"]["ms_median"] * 1e-3)
    res["legs"]["w3_getOddGrad"] = {"points": nq, "max_iter": 5, "ms_median": float(np.median(times["odd_grad"])),
                                    "ms_min": float(np.min(times["odd_grad"])), "ms_max": float(np.max(times["odd_grad"]))}
    res["w3_esdf_query_vs_getOddGrad"] = res["legs"]["w3_getOddGrad"]["ms_median"] / res["legs"]["w3_esdf_query"]["ms_median"]
    res["cfg_a_frame_us_reference"] = 85.0
    if not args.no_oracle:
        from esdf_oracle import EsdfOracle
        from esdf_spec import first_difference, same_bits
        orc = EsdfOracle(cfg)
        for k in range(args.frames):
            pose = scenes.corridor_trajectory_pose(k)
            orc.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
        orc.inflate_map(pose[:3])
        bad = []
        for inflated in (False, True):
            secs = [orc.build_esdf(w1[0], w1[1], 2.0, inflated=inflated) for _ in range(3)]
            o, _ = orc.export_esdf()
            if not same_bits(grids[inflated], o):
                bad.append((inflated, first_difference(grids[inflated], o)))
            key = "w1_inflated" if inflated else "w1"
            res["legs"][key]["oracle_build_ms_one_core"] = float(np.median(secs)) * 1e3
            res["legs"][key]["speedup_vs_oracle"] = res["legs"][key]["oracle_build_ms_one_core"] / res["legs"][key]["ms_median"]
        res["w1_parity"] = "ok" if not bad else f"MISMATCH {bad}"
        orc.close()
    for p in (d_q, d_dist, d_grad, d_og):
        m.device_free(p)
    m.close()

    # ---- W2: CFG-C LiDAR map after its scans, the whole hall
    cfg = config_cfg_c()
    m = MLMap(cfg)
    t0 = time.time()
    for k in range(args.scans):
        pose = scenes.lidar_loop_pose(k)
        m.integrate_points(scenes.lidar_scan(pose, frame_idx=k), pose)
    res["w2_map_seconds"] = time.time() - t0
    d, n = cfg.subbox_d_xyz, cfg.subbox_n
    w2 = (np.array([-60.0, -60.0, 0.0]), np.array([60.0 - d / 2, 60.0 - d / 2, 12.0 - d / 2]))
    times = {False: [], True: []}
    for rep in range(REPS):
        for inflated in (False, True):
            ms = timed_build(m, w2, 2.0, inflated)
            if rep >= WARM:
                times[inflated].append(ms)
    for inflated in (False, True):
        m.build_esdf(w2[0], w2[1], 2.0, inflated=inflated)
        g, lo = m.export_esdf()
        dims = np.array(g.shape[::-1])
        key = "w2_inflated" if inflated else "w2"
        res["legs"][key] = {"box_min": w2[0].tolist(), "box_max": w2[1].tolist(), "dims": dims.tolist(),
                            "cells": int(g.size), "subboxes_probed": subboxes_probed(lo, dims, n),
                            "blocking_cells": int((g <= 0).sum()),
                            **stats(times[inflated], build_bytes(lo, dims, n, inflated), peak)}
        res["legs"][key]["cells_per_s"] = g.size / (res["legs"][key]["ms_median"] * 1e-3)
    m.close()
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(res, indent=1, default=str) + "\n")
    print(json.dumps(res, default=str))


if __name__ == "__main__":
    main()
