"""Ray-casting timing (mlm_cast_rays_device, k_cast_rays) on the CFG-A map of the bench (200 corridor frames, then
inflate_map), L2 flushed before every timed pass, CUDA events on the handle's stream, 3 warm-up passes then 10 timed.

  W1  planner segments: 1 M segments, starts from scenes.query_positions(seed=5) over the map's AABB, uniformly random
      directions, lengths uniform in 0.5-5 m; both layers.  In the same loop, alternating, the same segments answered
      the way a caller without a ray query does it: points every d_sub/2 along each segment (end point included) through
      mlm_get_occupancy_device, timing that kernel only.
  W2  view rays: 16 viewpoints along the corridor x the 640x480 pixel directions of the CFG-A camera (intrinsics,
      T_bs) out to 6.5 m (4.9 M rays); both layers.

Algorithmic bytes per call: 48 B of endpoints in and 32 B out per ray, 1 B per visited cell (2 B with the inflated layer)
and 12 B (hash key + value) per subbox entered; as a share of bench.py's measured_peak_gbs().  W1's first 100 k records
(both layers) are checked against the oracle's restatement of the spec.  Writes one JSON file (--out)."""
import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from bench import measured_peak_gbs  # noqa: E402
from mlmapping_b200 import MLMap, capi, config_cfg_a, scenes  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in q.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:  # the number stays tied to what could be read
        import torch
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": f"unread ({e})"}


def view_rays(cfg, n_views=16, rows=480, cols=640, rng=6.5):
    T_bs = np.array(list(cfg.T_bs))
    R_bs = scenes.quat_to_rot(T_bs[3:7])
    uu, vv = np.meshgrid(np.arange(cols, dtype=np.float64), np.arange(rows, dtype=np.float64))
    d_s = np.stack([(uu - cfg.cam_cx) / cfg.cam_fx, (vv - cfg.cam_cy) / cfg.cam_fy, np.ones_like(uu)], -1).reshape(-1, 3)
    d_s /= np.linalg.norm(d_s, axis=1, keepdims=True)
    F, T = [], []
    for k in np.linspace(0, 199, n_views).round().astype(int):
        T_wb = scenes.corridor_trajectory_pose(int(k))
        R_wb = scenes.quat_to_rot(T_wb[3:7])
        o = T_wb[:3] + R_wb @ T_bs[:3]
        d_w = d_s @ (R_wb @ R_bs).T
        F.append(np.broadcast_to(o, d_w.shape))
        T.append(o + rng * d_w)
    return np.ascontiguousarray(np.concatenate(F)), np.ascontiguousarray(np.concatenate(T))


def traffic(rec, f, cfg, inflated):
    """algorithmic bytes and visited cells of one call, from its records"""
    d, n = cfg.subbox_d_xyz, cfg.subbox_n
    ok = rec["status"] != capi.RAY_INVALID
    cells = rec["n_free"].astype(np.int64) + rec["n_unknown"] + (rec["status"] == capi.OCCUPIED)
    g0 = np.floor(np.floor(f / d) / n)
    g1 = np.floor(rec["cell"] / n)
    subboxes = np.where(ok, 1 + np.abs(g1 - g0).sum(axis=1), 0).astype(np.int64)   # per-axis walks are monotone
    nbytes = 80 * rec.shape[0] + (2 if inflated else 1) * int(cells.sum()) + 12 * int(subboxes.sum())
    return nbytes, int(cells.sum()), int(subboxes.sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "ray_timing.json"))
    ap.add_argument("--n-w1", type=int, default=1_000_000)
    ap.add_argument("--frames", type=int, default=200)
    ap.add_argument("--parity", type=int, default=100_000, help="W1 records checked against the oracle (0: none)")
    args = ap.parse_args()
    import torch

    cfg = config_cfg_a()
    m = MLMap(cfg)
    for k in range(args.frames):
        pose = scenes.corridor_trajectory_pose(k)
        m.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
    m.inflate_map(pose[:3])
    ex = m.export_map()
    d, nsub = cfg.subbox_d_xyz, cfg.subbox_n
    lo, hi = ex["glb"].min(0) * nsub * d, (ex["glb"].max(0) + 1) * nsub * d
    nq = args.n_w1
    a = scenes.query_positions(nq, lo, hi, seed=5)
    rs = np.random.RandomState(6)
    v = rs.normal(size=(nq, 3))
    v /= np.linalg.norm(v, axis=1, keepdims=True)
    w1 = (a, np.ascontiguousarray(a + v * rs.uniform(0.5, 5.0, (nq, 1))))
    w2 = view_rays(cfg)

    # the sampled-getOccupancy path on W1: points every d_sub/2 from `from` (end point appended), built on the device
    dev = torch.device("cuda", 0)
    fa, ta = torch.from_numpy(w1[0]).to(dev), torch.from_numpy(w1[1]).to(dev)
    seg = ta - fa
    length = seg.norm(dim=1)
    per = torch.floor(length / (d / 2)).to(torch.int64) + 2
    idx = torch.repeat_interleave(torch.arange(nq, device=dev), per)
    first = torch.cumsum(per, 0) - per
    j = torch.arange(idx.numel(), device=dev) - first[idx]
    s = torch.clamp(j.to(torch.float64) * (d / 2) / torch.clamp(length[idx], min=1e-300), max=1.0)
    s = torch.where(j == per[idx] - 1, torch.ones_like(s), s)
    samples = (fa[idx] + seg[idx] * s[:, None]).contiguous()
    occ_out = torch.empty(samples.shape[0], dtype=torch.int32, device=dev)
    n_samples = int(samples.shape[0])
    torch.cuda.synchronize()

    bufs = {}
    for name, (f, t) in (("w1", w1), ("w2", w2)):
        bufs[name] = (m.to_device(f), m.to_device(t), m.device_alloc(32 * f.shape[0]), f.shape[0])

    def run_rays(name, inflated):
        d_f, d_t, d_o, n = bufs[name]
        m.flush_l2()
        m.timer_start()
        m.cast_rays_device(d_f, d_t, n, d_o, inflated=inflated)
        return m.timer_stop_ms()

    def run_sampled():
        m.flush_l2()
        m.timer_start()
        m.getOccupancy_device(samples.data_ptr(), n_samples, occ_out.data_ptr())
        return m.timer_stop_ms()

    legs = [("w1", False), ("w1", True), ("w2", False), ("w2", True)]
    times = {f"{w}{'_inflated' if i else ''}": [] for w, i in legs}
    times["w1_sampled_getOccupancy"] = []
    for rep in range(13):
        for w, i in legs:
            ms = run_rays(w, i)
            if w == "w1" and not i:   # the comparison alternates with the plain W1 pass
                ms_s = run_sampled()
                if rep >= 3:
                    times["w1_sampled_getOccupancy"].append(ms_s)
            if rep >= 3:
                times[f"{w}{'_inflated' if i else ''}"].append(ms)

    peak, peak_src = measured_peak_gbs()
    res = {"tool": "tools/ray_timing.py", **card(), "peak_gbs": peak, "peak_source": peak_src,
           "map_subboxes": int(ex["glb"].shape[0]), "frames": args.frames, "timed_passes": 10, "l2_flushed": True,
           "legs": {}}
    recs = {}
    for w, i in legs:
        key = f"{w}{'_inflated' if i else ''}"
        d_f, d_t, d_o, n = bufs[w]
        m.cast_rays_device(d_f, d_t, n, d_o, inflated=i)
        rec = m.to_host(d_o, (n,), capi.RAY_HIT_DTYPE)
        recs[key] = rec
        ms = float(np.median(times[key]))
        nbytes, cells, subs = traffic(rec, (w1 if w == "w1" else w2)[0], cfg, i)
        st = rec["status"]
        res["legs"][key] = {
            "rays": n, "ms_median": ms, "ms_min": float(np.min(times[key])), "ms_max": float(np.max(times[key])),
            "rays_per_s": n / (ms * 1e-3), "cells_per_s": cells / (ms * 1e-3), "visited_cells": cells,
            "subboxes_entered": subs, "algorithmic_bytes": nbytes, "gbs": nbytes / (ms * 1e-3) / 1e9,
            "share_of_peak": nbytes / (ms * 1e-3) / 1e9 / peak,
            "occupied": int((st == capi.OCCUPIED).sum()), "free": int((st == capi.FREE).sum()),
            "invalid": int((st == capi.RAY_INVALID).sum())}
    ms_s = float(np.median(times["w1_sampled_getOccupancy"]))
    res["legs"]["w1_sampled_getOccupancy"] = {
        "points": n_samples, "points_per_segment": n_samples / nq, "ms_median": ms_s,
        "ms_min": float(np.min(times["w1_sampled_getOccupancy"])), "ms_max": float(np.max(times["w1_sampled_getOccupancy"])),
        "segments_per_s": nq / (ms_s * 1e-3)}
    res["w1_speedup_vs_sampled"] = ms_s / res["legs"]["w1"]["ms_median"]

    if args.parity:
        from ray_oracle import RayOracle
        from raycast_spec import first_difference
        t0 = time.time()
        orc = RayOracle(cfg)
        for k in range(args.frames):
            pose = scenes.corridor_trajectory_pose(k)
            orc.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose)
        orc.inflate_map(pose[:3])
        k = args.parity
        bad = [first_difference(recs["w1_inflated" if i else "w1"][:k], orc.cast_rays(w1[0][:k], w1[1][:k], inflated=i))
               for i in (False, True)]
        res["ray_parity"] = "ok" if bad == [None, None] else f"MISMATCH {bad}"
        res["ray_parity_records"] = 2 * k
        res["oracle_seconds"] = time.time() - t0
    out = Path(args.out)
    out.parent.mkdir(parents=True, exist_ok=True)
    out.write_text(json.dumps(res, indent=1, default=str) + "\n")
    print(json.dumps(res, default=str))


if __name__ == "__main__":
    main()
