"""Path-cost matrix timing: mlm_reach_matrix_device (one class gather, then per batch of fields k_reach_matrix_seed /
k_reach_matrix_solve / k_reach_matrix_gather) against the loop a caller would otherwise write, K x (mlm_reach_build +
mlm_reach_cost_device) with one start per build.  Goals are the starts.  The L2 is flushed before every timed pass; the
matrix and the loop alternate, 3 warm-up passes then 10 timed, medians reported; CUDA events on the handle's stream.
Every leg checks matrix == loop bit for bit.

  M1  the W1 box of tools/reach_timing.py (CFG-A bench map: 200 corridor frames, inflate_map; last pose +- (6.4, 6.4,
      1.6) m), inflated, max_dist 30 m; K = 16, 64, 256 seeded free-cell starts.  At K = 16 also the oracle's loop of
      single-core Dijkstra builds.
  M2  the CFG-C hall after its 100 scans (600 x 600 x 60 cells), unknown cells traversable, max_dist 200 m, K = 16:
      12 fields per launch, so two launches.
  M3  the serpentine maze of tests/test_reach_gpu.py at 96 x 97 x 9 cells, max_dist 1e5 m, K = 32.
The single build of W1 (one start, inflated) is timed again in the same run for comparison with reach_timing.json.
Writes one JSON file (--out)."""
import argparse
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
sys.path.insert(0, str(ROOT / "tools"))
from mlmapping_b200 import MLMap, config_cfg_a, config_cfg_c, scenes  # noqa: E402
from ray_timing import card  # noqa: E402

REPS, WARM = 13, 3


def _ms(m, fn):
    m.flush_l2()
    m.timer_start()
    fn()
    return m.timer_stop_ms()


def free_starts(m, box, k, seed):
    """k seeded points in distinct free cells of the box"""
    rs = np.random.RandomState(seed)
    d = m.cfg.subbox_d_xyz
    pts = rs.uniform(box[0], box[1], (200 * k + 20000, 3))
    pts = pts[m.getOccupancy(pts) == 1]
    _, first = np.unique(np.floor(pts / d).astype(np.int64), axis=0, return_index=True)
    pts = pts[np.sort(first)]
    assert len(pts) >= k, (len(pts), k)
    return np.ascontiguousarray(pts[:k])


def matrix_leg(m, box, starts, max_dist, inflated=False, unknown=False):
    """matrix and loop alternately; parity of the two"""
    k = starts.shape[0]
    d_s, d_m, d_l = m.to_device(starts), m.device_alloc(8 * k * k), m.device_alloc(8 * k * k)

    def mat():
        m.reach_matrix_device(box[0], box[1], d_s, k, d_s, k, max_dist, d_m, inflated=inflated, unknown=unknown)

    def loop():
        for i in range(k):
            m.build_reach(box[0], box[1], starts[i:i + 1], max_dist, inflated=inflated, unknown=unknown)
            m.reach_cost_device(d_s, k, d_l + 8 * k * i)

    tm, tl = [], []
    for rep in range(REPS):
        a, b = _ms(m, mat), _ms(m, loop)
        if rep >= WARM:
            tm.append(a)
            tl.append(b)
    same = np.array_equal(m.to_host(d_m, (k, k), np.float64).view(np.uint64),
                          m.to_host(d_l, (k, k), np.float64).view(np.uint64))
    mat_h = m.to_host(d_m, (k, k), np.float64)
    for p in (d_s, d_m, d_l):
        m.device_free(p)
    r = {"k": k, "inflated": inflated, "unknown": unknown, "max_dist": max_dist,
         "matrix_ms_median": float(np.median(tm)), "matrix_ms_min": float(np.min(tm)),
         "matrix_ms_max": float(np.max(tm)), "loop_ms_median": float(np.median(tl)), "loop_ms_min": float(np.min(tl)),
         "loop_ms_max": float(np.max(tl)), "finite_entries": int(np.isfinite(mat_h).sum()),
         "parity": "ok" if same else "MISMATCH"}
    r["speedup"] = r["loop_ms_median"] / r["matrix_ms_median"]
    return r, mat_h


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "reach_matrix_timing.json"))
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--scans", type=int, default=100)
    args = ap.parse_args()
    res = {"tool": "tools/reach_matrix_timing.py", **card(), "timed_passes": REPS - WARM, "l2_flushed": True,
           "alternated": True, "per_kernel_split": "not measured", "legs": {}}

    # ---- M1: the W1 box on the CFG-A bench map
    cfg = config_cfg_a()
    m = MLMap(cfg)
    for k in range(args.frames):
        pose = scenes.corridor_trajectory_pose(k)
        m.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    m.inflate_map(pose[:3])
    c = pose[:3]
    half = np.array([6.4, 6.4, 1.6])
    w1 = (c - half, c + half)
    single = []
    for rep in range(REPS):
        t = _ms(m, lambda: m.build_reach(w1[0], w1[1], [c], 30.0, inflated=True))
        if rep >= WARM:
            single.append(t)
    res["w1_single_build_inflated"] = {"ms_median": float(np.median(single)), "ms_min": float(np.min(single)),
                                       "ms_max": float(np.max(single))}
    starts_all = free_starts(m, w1, 256, 1)
    m1 = {}
    for k in (16, 64, 256):
        r, mat = matrix_leg(m, w1, starts_all[:k], 30.0, inflated=True)
        m1[k] = mat
        res["legs"][f"m1_k{k}"] = r
    m.close()
    from reach_oracle import ReachOracle
    orc = ReachOracle(cfg)
    for k in range(args.frames):
        pose = scenes.corridor_trajectory_pose(k)
        orc.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    orc.inflate_map(pose[:3])
    secs, rows = 0.0, []
    for s in starts_all[:16]:
        orc.build_reach(w1[0], w1[1], [s], 30.0, inflated=True)
        secs += orc.last_seconds
        rows.append(orc.reach_cost(starts_all[:16]))
    orc.close()
    leg = res["legs"]["m1_k16"]
    leg["oracle_loop_ms_one_core"] = secs * 1e3
    leg["oracle_parity"] = "ok" if np.array_equal(np.array(rows).view(np.uint64), m1[16].view(np.uint64)) else "MISMATCH"

    # ---- M2: the CFG-C hall
    cfg = config_cfg_c()
    m = MLMap(cfg)
    for k in range(args.scans):
        pose = scenes.lidar_loop_pose(k)
        m.integrate_points(scenes.lidar_scan(pose, frame_idx=k), pose)
    d = cfg.subbox_d_xyz
    w2 = (np.array([-60.0, -60.0, 0.0]), np.array([60.0 - d / 2, 60.0 - d / 2, 12.0 - d / 2]))
    res["legs"]["m2_k16"], _ = matrix_leg(m, w2, free_starts(m, w2, 16, 2), 200.0, unknown=True)
    m.close()

    # ---- M3: the serpentine maze
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
    res["legs"]["m3_maze_k32"], _ = matrix_leg(m, w3, free_starts(m, w3, 32, 3), 1e5)
    m.close()

    res["parity"] = "ok" if all(v["parity"] == "ok" for v in res["legs"].values()) and \
        res["legs"]["m1_k16"]["oracle_parity"] == "ok" else "MISMATCH"
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(res, indent=1, default=str) + "\n")
    print(json.dumps(res, default=str))


if __name__ == "__main__":
    main()
