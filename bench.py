#!/usr/bin/env python
"""bench.py — rays integrated / second of the MLMapping per-frame map update on B200.

Workload (BASELINE.json configs[1], SURVEY §8d CFG-A config 2): the synthetic corridor trajectory,
640x480 uint16 depth @ 0.1 m voxels, streaming global-map submap allocation.  One "step" = one
depth frame integrated end to end (projection + awareness ray cast + log-odds fusion).  With
--gpus N each rank owns an independent agent map on its own trajectory (CFG-D style sharding:
no data-path collective), so scaling is weak.

  value  : valid rays / s over the K timed steps with the frames already resident in HBM
           (CUDA events on the library's stream around each step, L2 flushed between steps)
  e2e    : same metric through the host-buffer C-ABI call mlm_integrate_depth_u16
           (pinned staging + H2D copy + kernels + D2H stats inside the timed region)
  roofline / cpu_baseline : see DESIGN.md "Measurement"

`--impl reference` times the CPU oracle (the reference's algorithm restated, single-threaded like
the reference) on the same frames and prints the same JSON shape.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

METRIC = "rays_integrated_per_sec"
UNIT = "rays/s"
ROWS, COLS = 480, 640
WORKLOAD = "cfg_a_corridor_trajectory_640x480_d0.1m_streaming_submaps"
TRAJ_STRIDE = 1  # frame k of the 1000-frame trajectory


def gen_frames(cfg, n, agent=0):
    from mlmapping_b200 import scenes
    frames, poses = [], []
    for k in range(n):
        kk = (k * TRAJ_STRIDE) % 1000
        pose = scenes.corridor_trajectory_pose(kk, y_offset=20.0 * agent)
        frames.append(scenes.corridor_depth_frame(cfg, pose, frame_idx=kk, seed_drop=1 + 10 * agent,
                                                  seed_noise=2 + 10 * agent, y_offset=20.0 * agent))
        poses.append(pose)
    return frames, poses


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region"""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "10",
                 "-i", str(self.gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                smax.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def algorithmic_bytes(stats) -> int:
    """SURVEY §8d: B_frame = 2*W*H + 56 + 10*N_touch + 6000*N_new"""
    return 2 * ROWS * COLS + 56 + 10 * stats.n_touched_voxels + 6000 * stats.n_new_submaps


def measured_peak_gbs():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


def cpu_impl():
    """the CPU arm: the reference's OWN sources (oracle/_ref/libmlmap_ref.so, built from $MLMAPPING_REFERENCE by
    oracle/ref_build/Makefile) when available, else the restatement"""
    from oracle_binding import reference_available
    return "reference" if reference_available() else "port"


def dump_outputs(out_dir, m, st, exported, budget=64 << 20):
    """what the timed path computed in its last step, as float32 / float64 .npy files under out_dir: the frame's FrameStats
    (field order of mlmapping_b200.capi.FrameStats), its hit cells (rho, phi, z in the reference's iteration order) with
    their probabilities, its miss cells (flat indices, sorted) and the whole map sorted by subbox index (occupancy and
    inflate as the byte codes 'u' / 'f' / 'o').  A map larger than the budget is cut to a fixed, seeded sample of
    subboxes."""
    keys, p = m.last_frame_hits()
    arrays = {"frame_stats": np.array([getattr(st, f) for f, _ in st._fields_], dtype=np.float64),
              "hit_keys": keys.astype(np.float64), "hit_p": p.astype(np.float32),
              "miss_cells": np.sort(m.last_frame_misses()).astype(np.float64)}
    cells = exported["log_odds"].shape[1]
    rows = exported["glb"].shape[0]
    left = budget - sum(a.nbytes for a in arrays.values())
    keep = max(0, min(rows, left // (3 * 8 + 4 + 3 * 4 * cells)))
    sel = np.arange(rows) if keep == rows else np.sort(np.random.default_rng(0).choice(rows, keep, replace=False))
    arrays.update({"map_glb": exported["glb"][sel].astype(np.float64),
                   "map_collapsed": exported["collapsed"][sel].astype(np.float32),
                   "map_occupancy": exported["occupancy"][sel].view(np.uint8).astype(np.float32),
                   "map_inflate": exported["inflate"][sel].view(np.uint8).astype(np.float32),
                   "map_log_odds": exported["log_odds"][sel].astype(np.float32)})
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


def run_cpu_sample(cfg, frames, poses, n_frames):
    """the reference's mapping code (cpu_impl()) timed on the first n_frames of the workload, 1 core"""
    from oracle_binding import Oracle
    orc = Oracle(cfg, bookkeeping=False, impl=cpu_impl())
    rays, secs = 0, 0.0
    for k in range(n_frames):
        st = orc.integrate_depth(frames[k], poses[k])
        rays += st.n_points
        secs += orc.last_seconds
    orc.close()
    return rays, secs


def run_reference(args, rank, world):
    """CPU arm: the reference's own mapping sources (oracle/_ref) when that library is present, else the restatement.
    One map is single-threaded like the reference; with --gpus N the N independent agent maps of the GPU arm run on
    N host threads (ctypes releases the GIL), one map each."""
    import threading
    from mlmapping_b200 import config_cfg_a
    if rank != 0:
        return
    cfg = config_cfg_a()
    total = args.steps + args.warmup
    n_agents = max(1, args.gpus)
    from oracle_binding import Oracle
    data = [gen_frames(cfg, total, agent=a) for a in range(n_agents)]
    res = [None] * n_agents
    impl = cpu_impl()
    orcs = [Oracle(cfg, bookkeeping=False, impl=impl) for _ in range(n_agents)]  # created one after the other (init is not re-entrant)

    def work(a):
        frames, poses = data[a]
        orc = orcs[a]
        for k in range(args.warmup):
            orc.integrate_depth(frames[k], poses[k])
        rays, secs = 0, 0.0
        for k in range(args.warmup, total):
            st = orc.integrate_depth(frames[k], poses[k])
            rays += st.n_points
            secs += orc.last_seconds
        res[a] = (rays, secs)
        orc.close()

    th = [threading.Thread(target=work, args=(a,)) for a in range(n_agents)]
    [t.start() for t in th]
    [t.join() for t in th]
    rays = sum(r for r, _ in res)
    secs = max(s_ for _, s_ in res)
    value = rays / secs
    sample = (f"{args.steps} frames of {WORKLOAD} after {args.warmup} warm-up frames, {n_agents} agent map(s) on "
              f"{n_agents} host thread(s), one map per thread ({os.cpu_count()} host cores present)")
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * secs / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rows": ROWS, "cols": COLS, "agents": n_agents,
                   "timing": "steady_clock around project_depth+update_map (the region the reference times, src/mlmap.cpp:474-511)",
                   "cpu_code": "oracle/_ref: the reference's own sources" if impl == "reference" else "oracle/: restatement of the reference"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": n_agents, "kind": impl, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def run_lidar(rank, world, local_rank, barrier, scans=12, warm=4):
    """BASELINE config 4 (CFG-C): 128 x 2048 LiDAR scans into ONE map.  At every N the scan goes through the sharded
    path (stage by phi column, keys + update records stored into the owners' arenas over NVLink peer memory, owner-side
    fusion; world 1 = the same kernels without peers); at N = 1 the fused single-GPU frame (k_frame) is timed beside it
    and is the N = 1 figure.  Timed on the device: CUDA events on the library's stream around submit..finish, barrier
    before every scan, sum over the timed scans, max over ranks.  The first two scans are checked against the CPU
    oracle (union of the ranks' subboxes == the oracle map, bit for bit)."""
    import torch
    from mlmapping_b200 import MLMap, config_cfg_c, scenes
    from mlmapping_b200.sharding import split_range
    from mlmapping_b200.sharded import ShardedMLMap
    cfg = config_cfg_c()
    data = []
    for k in range(scans):
        pose = scenes.lidar_loop_pose(k)
        data.append((scenes.lidar_scan(pose, frame_idx=k), pose))
    out = {"workload": "cfg_c_128beam_lidar_2048az_d0.2m_50m (BASELINE config 4)", "scans": scans - warm, "n_gpus": world,
           "scaling": "strong"}
    peak, _ = measured_peak_gbs()

    def reduce_max(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    fused = None
    if world == 1:
        m = MLMap(cfg, device=local_rank)
        dev = [(m.to_device(p), p.shape[0], pose) for p, pose in data]
        ms, rays, touched, new = 0.0, 0, 0, 0
        for k, (dp, n, pose) in enumerate(dev):
            m.flush_l2()
            m.timer_start()
            st = m.integrate_points_device(dp, n, pose)
            t = m.timer_stop_ms()
            if k >= warm:
                ms += t
                rays += st.n_points
                touched += st.n_touched_voxels
                new += st.n_new_submaps
        alg = 24 * rays + 56 * (scans - warm) + 10 * touched + 6000 * new  # SURVEY 8d frame bytes with point input
        fused = {"mode": "one map on one GPU, ONE cooperative launch per scan (k_frame), points resident in HBM, L2 flushed",
                 "rays_per_s": rays / (ms * 1e-3), "us_per_scan": 1e3 * ms / (scans - warm),
                 "alg_GB_per_s": alg / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": alg / (ms * 1e-3) / 1e9 / peak}
        m.close()

    sh = ShardedMLMap(cfg, rank=rank, world=world, device=local_rank)
    dev = [(sh.map.to_device(p), p.shape[0], pose) for p, pose in data]
    parity = "not checked"
    ms, rays, wait_ns, rehash = 0.0, 0, 0, 0
    sh_hits = []
    for k, (dp, n, pose) in enumerate(dev):
        sh.map.flush_l2()
        barrier()
        sh.map.timer_start()
        sh.submit_device(dp, n, pose)
        sh_hits.append(sh.finish().n_hit_cells)
        t = sh.map.timer_stop_ms()
        rehash += sh.last["rehash_path"]
        if k >= warm:
            ms += t
            rays += n
            wait_ns += sh.last["wait_ns"]
        if k == 1:  # parity of the sharded map against the CPU oracle after two scans
            mine = sh.export_map()
            gathered = [mine]
            if world > 1:
                gathered = [None] * world
                torch.distributed.all_gather_object(gathered, mine)
            if rank == 0:
                from oracle_binding import Oracle
                oc = Oracle(cfg, bookkeeping=False, impl=cpu_impl())
                for p, ps in data[:2]:
                    oc.integrate_points(p, ps)
                o = oc.export_map()
                oc.close()
                glb = np.concatenate([g["glb"] for g in gathered])
                order = np.lexsort((glb[:, 2], glb[:, 1], glb[:, 0]))
                ok = np.array_equal(glb[order], o["glb"])
                for name in ("occupancy", "log_odds", "collapsed"):
                    u = np.concatenate([g[name] for g in gathered])[order]
                    ok = ok and u.shape == o[name].shape and np.array_equal(u.view(np.uint8), o[name].view(np.uint8))
                parity = "ok" if ok else "MISMATCH"
                out["parity_subboxes"] = int(glb.shape[0])
                out["subboxes_owned_per_rank"] = [int(g["glb"].shape[0]) for g in gathered]
    ms = reduce_max(ms)
    sharded = {"mode": "ONE map sharded by subbox ownership over the ranks: keys and update records stored into the owners' "
                       "arenas over NVLink peer memory by the library's kernels, device-side wait; points resident in HBM, "
                       "L2 flushed, CUDA events around submit..finish, max over ranks",
               "rays_per_s": rays / (ms * 1e-3), "us_per_scan": 1e3 * ms / (scans - warm),
               "wait_us_per_scan_this_rank": 1e-3 * wait_ns / (scans - warm), "rehash_scans": rehash,
               "last_exchange": sh.last}
    # per-stage device times (events between the launches; a separate pass so that the events do not sit in the timed one)
    sh.map.set_profiling(True)
    acc = {}
    for k, (dp, n, pose) in enumerate(dev[warm:]):
        sh.map.flush_l2()
        barrier()
        sh.submit_device(dp, n, pose)
        sh.finish()
        for k_, v_ in sh.last_kernel_us().items():
            acc[k_] = acc.get(k_, 0.0) + v_ / (scans - warm)
    sh.map.set_profiling(False)
    sharded["stage_us_this_rank"] = {k_: round(v_, 1) for k_, v_ in acc.items()}
    # e2e: the scan starts in pinned host memory, the H2D copy is inside the timed region (wall clock, max over ranks)
    buf = sh.pinned_points(max(p.shape[0] for p, _ in data))
    secs, e_rays, h2d_us, t_submit = 0.0, 0, 0.0, 0.0
    slices_ok = True
    sh.map.set_profiling(world == 1)   # (the stage events are only read at N = 1; they cost host time in the submit)
    for k, (pts, pose) in enumerate(data):  # the first `warm` scans are not timed (staging buffers are allocated on first use)
        b = buf[:pts.shape[0]]
        b[...] = pts
        sh.map.flush_l2()
        barrier()
        t0 = time.perf_counter()
        if world > 1:   # every rank copies its 1/world of the scan; the slices travel over NVLink inside the library
            lo, hi = split_range(pts.shape[0], rank, world)
            sh.submit_slice(b[lo:hi], lo, pts.shape[0], pose)
        else:
            sh.submit(b, pose)
        t1 = time.perf_counter()
        st_e = sh.finish()
        t2 = time.perf_counter()
        slices_ok = slices_ok and st_e.n_hit_cells == sh_hits[k]   # the frame's hit set does not depend on the map's state
        if k < warm:
            continue
        secs += t2 - t0
        t_submit += t1 - t0
        e_rays += pts.shape[0]
        if world == 1:
            h2d_us += sh.last_kernel_us()["resets_h2d"] / (scans - warm)
    sh.map.set_profiling(False)
    secs = reduce_max(secs)
    sharded["e2e"] = {"rays_per_s": e_rays / secs, "us_per_scan": 1e6 * secs / (scans - warm),
                      "h2d_bytes_per_scan_and_rank": int(24 * e_rays / (scans - warm) / world),
                      "resets_and_h2d_us_this_rank": round(h2d_us, 1) if world == 1 else None,
                      "host_submit_us_this_rank": round(1e6 * t_submit / (scans - warm), 1),
                      "hit_cells_equal_whole_scan_submission": bool(slices_ok),
                      "note": "every rank copies 1/world of the scan from pinned host memory (mlm_shard_submit_points_slice_f64); "
                              "the slices reach the other ranks over NVLink peer memory"}
    if world > 1:
        barrier()
    sh.close()
    if world > 1:
        barrier()
    best = fused if fused is not None and fused["us_per_scan"] <= sharded["us_per_scan"] else sharded
    out.update({"parity": parity, "rays_per_s": best["rays_per_s"], "us_per_scan": best["us_per_scan"], "sharded": sharded})
    if fused is not None:
        out["fused_single_gpu"] = fused
    return out


def run_agents(rank, world, local_rank, barrier, steps, warm, n_queries, n_agents=8):
    """BASELINE config 5 (CFG-D) as written: 8 independent agent maps (agent a: corridor shifted by y = 20 a, seeds + 10 a)
    distributed round-robin over the N ranks, plus the 10 M planner queries per step.  A step advances EVERY agent by one
    frame, so the total work is fixed: strong scaling (8 handles on one GPU at N = 1, one per GPU at N = 8).  Device time
    per step = sum of the rank's frame times (CUDA events on each handle's stream, L2 flushed once per step), max over
    ranks.  The query stream is answered twice: split over the ranks against each rank's own agent maps, and against
    ONE map replicated on every rank (dirty subbox blocks of each frame broadcast over NCCL, ReplicatedMLMap)."""
    import torch
    from mlmapping_b200 import MLMap, config_cfg_a, scenes
    from mlmapping_b200.sharding import agents_for_rank, reduce_timing, split_range
    cfg = config_cfg_a()
    mine = agents_for_rank(n_agents, rank, world)
    total = steps + warm
    maps, dev = {}, {}
    for a in mine:
        frames, poses = gen_frames(cfg, total, agent=a)
        maps[a] = MLMap(cfg, device=local_rank)
        dev[a] = [(maps[a].to_device(f), p) for f, p in zip(frames, poses)]
    first = maps[mine[0]] if mine else None
    step_ms, rays, frame_us = [], 0, []
    for k in range(total):
        if first is not None:
            first.flush_l2()
        t_step = 0.0
        for a in mine:
            m = maps[a]
            m.timer_start()
            st = m.integrate_depth_device(dev[a][k][0], ROWS, COLS, dev[a][k][1])
            t = m.timer_stop_ms()
            t_step += t
            if k >= warm:
                rays += st.n_points
                frame_us.append(1e3 * t)
        if k >= warm:
            step_ms.append(t_step)
    barrier()
    (ms_sum,), (rays_all,) = reduce_timing([float(np.sum(step_ms))], [float(rays)], device="cuda" if world > 1 else None)
    out = {"workload": "cfg_d_8_agent_maps_640x480_d0.1m (BASELINE config 5)", "agents": n_agents, "n_gpus": world,
           "agents_this_rank": mine, "scaling": "strong", "steps": steps,
           "rays_per_s": rays_all / (ms_sum * 1e-3), "ms_per_step": ms_sum / steps,
           "mode": "a rank's maps one after the other, each frame ONE cooperative launch on all SMs",
           "us_per_frame_this_rank": {"median": float(np.median(frame_us)) if frame_us else None,
                                      "max": float(np.max(frame_us)) if frame_us else None}}
    # ---- the same steps with the rank's maps in flight TOGETHER: every map gets a share of the SMs (its cooperative frame
    # kernel uses that many CTAs), frames are submitted on all handles and then finished; fresh maps, same frames ----
    if len(mine) > 1:
        for m in maps.values():
            m.close()
        share = max(8, 148 // len(mine))
        maps = {}
        for a in mine:
            maps[a] = MLMap(cfg, device=local_rank)
            maps[a].set_sm_budget(share)
            dev[a] = [(maps[a].to_device(f), p) for f, p in zip(*gen_frames(cfg, total, agent=a))]
        first = maps[mine[0]]
        c_secs, c_rays = 0.0, 0
        for k in range(total):
            first.flush_l2()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for a in mine:
                maps[a].submit_depth_device(dev[a][k][0], ROWS, COLS, dev[a][k][1])
            sts = [maps[a].finish_frame() for a in mine]
            dt = time.perf_counter() - t0
            if k >= warm:
                c_secs += dt
                c_rays += sum(st.n_points for st in sts)
        barrier()
        (c_max,), (c_rays_all,) = reduce_timing([1e3 * c_secs], [float(c_rays)], device="cuda" if world > 1 else None)
        out["concurrent"] = {"mode": f"{len(mine)} maps of a rank in flight together, {share} SMs each (wall clock around submit-all / finish-all)",
                             "rays_per_s": c_rays_all / (c_max * 1e-3), "ms_per_step": c_max / steps}
        if out["concurrent"]["rays_per_s"] > out["rays_per_s"]:
            out["best"] = "concurrent"
    # ---- queries against the agents' own maps: the stream is split over the ranks, each rank's share over its maps ----
    if n_queries and mine:
        qb, qe = split_range(n_queries, rank, world)
        per = (qe - qb) // len(mine)
        q_ms = 0.0
        d = cfg.subbox_d_xyz * cfg.subbox_n
        for a in mine:
            m = maps[a]
            ex = m.export_map()
            pos = scenes.query_positions(per, ex["glb"].min(0) * d, (ex["glb"].max(0) + 1) * d, seed=5 + a)
            n_odd, n_occ = int(0.4 * per), int(0.4 * per)
            n_grad = per - n_odd - n_occ
            d_pos = m.to_device(pos)
            o1, o2, o3 = m.device_alloc(4 * n_odd), m.device_alloc(4 * n_occ), m.device_alloc(24 * n_grad)
            for rep in range(4):
                m.flush_l2()
                m.timer_start()
                m.getOdd_device(d_pos, n_odd, o1)
                m.getOccupancy_device(d_pos + 24 * n_odd, n_occ, o2)
                m.getOddGrad_device(d_pos + 24 * (n_odd + n_occ), n_grad, o3, 5)
                t = m.timer_stop_ms()
            q_ms += t
            for pp in (d_pos, o1, o2, o3):
                m.device_free(pp)
        (q_max,), _ = reduce_timing([q_ms], [0.0], device="cuda" if world > 1 else None)
        out["queries_own_maps"] = {"n_queries": n_queries, "ms_per_step": q_max, "queries_per_s": n_queries / (q_max * 1e-3),
                                   "split": "evenly over ranks, a rank's share evenly over its agent maps"}
    for m in maps.values():
        m.close()
    # ---- the same stream against ONE map replicated on every rank ----
    if n_queries:
        from mlmapping_b200.sharded import ReplicatedMLMap
        rep = ReplicatedMLMap(cfg, rank=rank, world=world, src=0, device=local_rank)
        frames, poses = gen_frames(cfg, min(total, 30), agent=0)
        t_rep, nb = 0.0, 0
        for k, (f, p) in enumerate(zip(frames, poses)):
            barrier()
            t0 = time.perf_counter()
            rep.integrate_depth(f if rank == 0 else None, p)
            torch.cuda.synchronize()
            if k >= 5:
                t_rep += time.perf_counter() - t0
                nb += rep.last["broadcast_bytes"]
        nrep = max(1, len(frames) - 5)
        ex = rep.map.export_map()
        d = cfg.subbox_d_xyz * cfg.subbox_n
        qb, qe = split_range(n_queries, rank, world)
        pos = scenes.query_positions(n_queries, ex["glb"].min(0) * d, (ex["glb"].max(0) + 1) * d, seed=5)[qb:qe]
        n_odd, n_occ = int(0.4 * len(pos)), int(0.4 * len(pos))
        n_grad = len(pos) - n_odd - n_occ
        m = rep.map
        d_pos = m.to_device(pos)
        o1, o2, o3 = m.device_alloc(4 * n_odd), m.device_alloc(4 * n_occ), m.device_alloc(24 * n_grad)
        for r_ in range(4):
            m.flush_l2()
            m.timer_start()
            m.getOdd_device(d_pos, n_odd, o1)
            m.getOccupancy_device(d_pos + 24 * n_odd, n_occ, o2)
            m.getOddGrad_device(d_pos + 24 * (n_odd + n_occ), n_grad, o3, 5)
            t = m.timer_stop_ms()
        (q_max, t_rep_max), _ = reduce_timing([t, 1e3 * t_rep / nrep], [0.0], device="cuda" if world > 1 else None)
        out["queries_replicated_map"] = {"n_queries": n_queries, "ms_per_step": q_max, "queries_per_s": n_queries / (q_max * 1e-3),
                                         "replication_ms_per_frame": t_rep_max, "broadcast_bytes_per_frame": nb / nrep,
                                         "note": "rank 0 integrates, then its kernel stores the frame's dirty subbox blocks into every replica's "
                                                 "inbox over NVLink peer memory (mlm_replica_publish / apply); wall clock incl. the "
                                                 "update on rank 0"}
        rep.close()
    return out


def run_other_configs(local_rank):
    """what BASELINE.json's other single-GPU configurations cost (SURVEY 8d): CFG-B frames (L515-like 1024x768 @ 0.05 m),
    exploration-mode frames, and the first frame of a fresh map (libstdc++ rehash path, ~70 launches).  Device-resident
    inputs, CUDA events on the library's stream, L2 flushed between frames; the CPU reference on a short sample."""
    from mlmapping_b200 import MLMap, config_cfg_a, config_cfg_b, scenes
    from oracle_binding import Oracle
    peak, _ = measured_peak_gbs()
    out = {}
    # ---- CFG-B ----
    cfg = config_cfg_b()
    n, warm = 24, 6
    frames, poses = [], []
    for k in range(n):
        pose = scenes.corridor_trajectory_pose(k, step=0.1)
        frames.append(scenes.corridor_depth_frame(cfg, pose, rows=768, cols=1024, frame_idx=k, length=200.0))
        poses.append(pose)
    m = MLMap(cfg, device=local_rank)
    dev = [m.to_device(f) for f in frames]
    ms, rays, alg = 0.0, 0, 0
    for k in range(n):
        m.flush_l2()
        m.timer_start()
        st = m.integrate_depth_device(dev[k], 768, 1024, poses[k])
        t = m.timer_stop_ms()
        if k >= warm:
            ms += t
            rays += st.n_points
            alg += 2 * 768 * 1024 + 56 + 10 * st.n_touched_voxels + 6000 * st.n_new_submaps
    pin = m.pinned_array(frames[0].shape, np.uint16)
    pin[...] = frames[warm - 1]
    m.integrate_depth_ptr(pin.ctypes.data, 768, 1024, 2 * 1024, poses[warm - 1])  # first host-buffer call allocates the staging
    e_s = 0.0
    for k in range(warm, n):
        pin[...] = frames[k]
        m.flush_l2()
        t0 = time.perf_counter()
        m.integrate_depth_ptr(pin.ctypes.data, 768, 1024, 2 * 1024, poses[k])
        e_s += time.perf_counter() - t0
    m.close()
    orc = Oracle(cfg, bookkeeping=False, impl=cpu_impl())
    c_rays, c_s = 0, 0.0
    for k in range(4):
        st = orc.integrate_depth(frames[k], poses[k])
        if k >= 1:
            c_rays += st.n_points
            c_s += orc.last_seconds
    orc.close()
    out["cfg_b_l515_1024x768_d0.05m"] = {
        "us_per_frame": 1e3 * ms / (n - warm), "rays_per_s": rays / (ms * 1e-3), "e2e_us_per_frame": 1e6 * e_s / (n - warm),
        "alg_GB_per_s": alg / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": alg / (ms * 1e-3) / 1e9 / peak,
        "cpu_baseline": {"value": c_rays / c_s, "unit": UNIT, "cores": 1, "kind": cpu_impl(), "us_per_frame": 1e6 * c_s / 3,
                         "sample": "frames 1-3 of the same series on the CPU oracle, single thread"}}
    # ---- exploration mode (use_exploration_frontiers) and the first frame of a fresh map, CFG-A ----
    cfg = config_cfg_a()
    fr, ps = gen_frames(cfg, 30)
    cfg_e = config_cfg_a()
    cfg_e.use_exploration_frontiers = 1
    m = MLMap(cfg_e, device=local_rank)
    dev = [m.to_device(f) for f in fr]
    ms, slow_e = 0.0, 0
    for k in range(30):
        m.flush_l2()
        m.timer_start()
        st_e = m.integrate_depth_device(dev[k], ROWS, COLS, ps[k])
        t = m.timer_stop_ms()
        if k >= 10:
            ms += t
            slow_e += st_e.ordering_slow_path
    m.close()
    out["cfg_a_exploration_mode"] = {"us_per_frame": 1e3 * ms / 20, "rehash_frames_in_timed_region": slow_e,
                                     "note": "frontier sets + release pass: one cooperative launch per frame (k_frame_explore)"}
    firsts = []
    for rep in range(3):
        m = MLMap(cfg, device=local_rank)
        d0 = m.to_device(fr[0])
        m.flush_l2()
        m.timer_start()
        st = m.integrate_depth_device(d0, ROWS, COLS, ps[0])
        firsts.append(1e3 * m.timer_stop_ms())
        assert st.ordering_slow_path == 1
        m.close()
    out["cfg_a_first_frame_of_a_fresh_map"] = {"us": float(np.median(firsts)),
                                               "note": "crosses the libstdc++ rehash chain 1 -> 13 -> ... (staged re-sequencing, ~70 launches)"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--cpu-frames", type=int, default=60, help="frames of the workload timed on the CPU oracle")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-queries", action="store_true")
    ap.add_argument("--no-lidar", action="store_true")
    ap.add_argument("--lidar-only", action="store_true", help="run only the LiDAR section and print its JSON (tooling)")
    ap.add_argument("--agents-only", action="store_true", help="run only the CFG-D agents section and print its JSON (tooling)")
    ap.add_argument("--no-agents", action="store_true")
    ap.add_argument("--queries", type=int, default=10_000_000, help="planner queries per step (4:4:2 odd/occupancy/grad)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy "
                    "(frame stats, hit and miss cells, the map) for comparing two builds on the same inputs")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the CUDA path computed: it needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the mlmap_b200 hot path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime
        # a stuck collective should fail the run in minutes, not hold the box for NCCL's default ten
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=180))

    from mlmapping_b200 import MLMap, config_cfg_a
    import ctypes as C
    from mlmapping_b200.capi import FrameStats

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.lidar_only:
        res = run_lidar(rank, world, local_rank, barrier)
        if rank == 0:
            print(json.dumps({"lidar": res}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    if args.agents_only:
        res = run_agents(rank, world, local_rank, barrier, min(args.steps, 40), 5, args.queries)
        if rank == 0:
            print(json.dumps({"agents": res}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    cfg = config_cfg_a()
    total = args.steps + args.warmup
    frames, poses = gen_frames(cfg, total, agent=rank)

    # ---------------- pass 1: device-resident inputs ("value") ----------------
    m = MLMap(cfg, device=local_rank)
    d_frames = [m.to_device(f) for f in frames]
    for k in range(args.warmup):
        m.integrate_depth_device(d_frames[k], ROWS, COLS, poses[k])
    sampler = ClockSampler(local_rank)
    launches0 = m.kernel_launch_count()
    barrier()
    sampler.start()
    try:
        wall0 = time.perf_counter()
        dev_ms, rays, alg_bytes, slow_frames = 0.0, 0, 0, 0
        for k in range(args.warmup, total):
            m.flush_l2()
            m.timer_start()
            st = m.integrate_depth_device(d_frames[k], ROWS, COLS, poses[k])
            dev_ms += m.timer_stop_ms()
            rays += st.n_points
            alg_bytes += algorithmic_bytes(st)
            slow_frames += st.ordering_slow_path
        barrier()
        wall1 = time.perf_counter()
    finally:  # the sampler's nvidia-smi child must not outlive a failed run
        clocks = sampler.stop()
    launches = m.kernel_launch_count() - launches0  # the library counts its map kernels only (the L2 flush is not one)
    exported = m.export_map()
    submaps = exported["glb"].shape[0]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, m, st, exported)

    # ---------------- batched planner queries against the map just built (BASELINE config 5 mix) ----------------
    queries = None
    if not args.no_queries:
        from mlmapping_b200 import scenes
        from mlmapping_b200.sharding import split_range
        nq = args.queries
        qb, qe = split_range(nq, rank, world)
        d = cfg.subbox_d_xyz * cfg.subbox_n
        lo, hi = exported["glb"].min(0) * d, (exported["glb"].max(0) + 1) * d
        pos = scenes.query_positions(nq, lo, hi, seed=5)[qb:qe]
        n_odd, n_occ = int(0.4 * len(pos)), int(0.4 * len(pos))
        n_grad = len(pos) - n_odd - n_occ
        d_pos = m.to_device(pos)
        d_o1, d_o2, d_o3 = m.device_alloc(4 * n_odd), m.device_alloc(4 * n_occ), m.device_alloc(24 * n_grad)
        off_occ, off_grad = 24 * n_odd, 24 * (n_odd + n_occ)

        def run_queries():
            t = {}
            m.flush_l2(); m.timer_start(); m.getOdd_device(d_pos, n_odd, d_o1); t["getOdd"] = m.timer_stop_ms()
            m.flush_l2(); m.timer_start(); m.getOccupancy_device(d_pos + off_occ, n_occ, d_o2); t["getOccupancy"] = m.timer_stop_ms()
            m.flush_l2(); m.timer_start(); m.getOddGrad_device(d_pos + off_grad, n_grad, d_o3, 5); t["getOddGrad"] = m.timer_stop_ms()
            return t
        for _ in range(3):
            run_queries()
        reps = 10
        acc = {"getOdd": 0.0, "getOccupancy": 0.0, "getOddGrad": 0.0}
        for _ in range(reps):
            for k_, v_ in run_queries().items():
                acc[k_] += v_ / reps
        q_ms = sum(acc.values())
        # SURVEY 8d algorithmic bytes: getOdd 32 B, getOccupancy 29 B, getOddGrad 76 B (one search round)
        q_bytes = 32 * n_odd + 29 * n_occ + 76 * n_grad
        queries = {"n_local": len(pos), "ms": acc, "total_ms": q_ms, "alg_bytes": q_bytes}
        for pp in (d_pos, d_o1, d_o2, d_o3):
            m.device_free(pp)

    # ---------------- LiDAR-scale integration (BASELINE config 4, CFG-C): 128 x 2048 scans ----------------
    # ONE logical map sharded over the ranks by subbox ownership (stage by phi column; hit keys all-gathered and update
    # records sent to their owners by the library's kernels over NVLink peer memory); N = 1 also times the fused frame.
    lidar = None
    if not args.no_lidar:
        if world == 1:
            try:
                lidar = run_lidar(rank, world, local_rank, barrier)
            except Exception as e:  # no peers at N = 1: an error here must not cost the headline line
                lidar = {"error": f"{type(e).__name__}: {e}"[:300]}
        else:
            lidar = run_lidar(rank, world, local_rank, barrier)

    # ---------------- CFG-D as written: 8 agent maps over the N ranks + the query stream (own maps / replicated map) ----
    agents = None
    if not args.no_agents:
        try:
            agents = run_agents(rank, world, local_rank, barrier, min(args.steps, 40), 5, 0 if args.no_queries else args.queries)
        except Exception as e:
            if world > 1:
                raise
            agents = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---------------- pass 2: per-kernel events on the same frames (roofline share) ----------------
    m.close()
    m = MLMap(cfg, device=local_rank)
    m.set_profiling(True)
    for k in range(args.warmup):
        m.integrate_depth(frames[k], poses[k])
    kern = {}
    for k in range(args.warmup, total):
        m.flush_l2()
        m.integrate_depth(frames[k], poses[k])
        for name, ms in m.last_frame_kernel_ms().items():
            kern[name] = kern.get(name, 0.0) + ms
    m.set_profiling(False)
    m.close()

    # ---------------- pass 3: end to end through the host-buffer C-ABI call ("e2e") ----------------
    m = MLMap(cfg, device=local_rank)
    pinned = []
    for f in frames:  # inputs live in pinned host memory (bench contract); the H2D copy is inside the call
        pf = m.pinned_array(f.shape, np.uint16)
        pf[...] = f
        pinned.append(pf)
    ptrs = [pf.ctypes.data for pf in pinned]  # the C-ABI call takes the host address, as a C/C++ caller passes it
    for k in range(args.warmup):
        m.integrate_depth_ptr(ptrs[k], ROWS, COLS, 2 * COLS, poses[k])
    barrier()
    e2e_s, e2e_rays = 0.0, 0
    for k in range(args.warmup, total):
        m.flush_l2()  # synchronous: the flush is not part of the step
        t0 = time.perf_counter()
        st = m.integrate_depth_ptr(ptrs[k], ROWS, COLS, 2 * COLS, poses[k])
        e2e_s += time.perf_counter() - t0
        e2e_rays += st.n_points
    barrier()
    m.close()

    # ---------------- reduce over ranks: max time, sum of rays ----------------
    from mlmapping_b200.sharding import reduce_timing
    q_ms_local = queries["total_ms"] if queries else 0.0
    # per-rank device time of the timed steps (every rank integrates ITS agent's trajectory: other walls, other seeds, so
    # the frames of different ranks are not the same work; the headline takes the max, the spread is reported next to it)
    per_rank_us = [1e3 * dev_ms / args.steps]
    if world > 1:
        import torch.distributed as dist
        tt = torch.zeros(world, dtype=torch.float64, device="cuda")
        tt[rank] = per_rank_us[0]
        dist.all_reduce(tt)
        per_rank_us = tt.tolist()
    (dev_ms, e2e_s, q_ms_max), (rays, e2e_rays, launches) = reduce_timing(
        [dev_ms, e2e_s, q_ms_local], [rays, e2e_rays, launches], device="cuda" if world > 1 else None)
    rays, e2e_rays, launches = int(rays), int(e2e_rays), int(launches)

    if rank == 0:
        value = rays / (dev_ms * 1e-3)
        # a timed step is ONE launch of the cooperative kernel k_frame (projection, work columns and fusion behind
        # device-wide barriers), so it is the dominant kernel and its launch duration is the device time of the step;
        # `kern` holds the same three phases run as stand-alone kernels (profiling path) to show where the time goes
        top = "k_frame" if launches == args.steps * world else max(kern, key=kern.get)
        top_ms = dev_ms / args.steps if top == "k_frame" else kern[top] / args.steps
        peak, peak_src = measured_peak_gbs()
        per_rank_bytes = alg_bytes / args.steps
        achieved = per_rank_bytes / (top_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        try:  # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu --set full capture
            prof = json.loads((ROOT / "profiles" / "ncu_full_summary_r02.json").read_text())[top][0]

            def _bytes(v):
                num, unit = v.split()
                return float(num) * {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[unit]
            traffic = _bytes(prof["dram__bytes_read.sum"]) + _bytes(prof["dram__bytes_write.sum"])
            traffic_src = "profiles/ncu_full_summary_r02.json (bytes per launch, cold-cache ncu capture)"
        except Exception:
            pass
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "rows": ROWS, "cols": COLS, "voxel_m": 0.1, "frames_per_step": 1,
                       "l2": "flushed between timed steps (256 MiB write)", "agents": world,
                       "slow_ordering_frames": slow_frames, "submaps_allocated_rank0": submaps,
                       "wall_s_timed_loop": wall1 - wall0},
            "us_per_frame": 1e3 * dev_ms / args.steps,
            "us_per_frame_over_ranks": {"min": float(np.min(per_rank_us)), "median": float(np.median(per_rank_us)),
                                        "max": float(np.max(per_rank_us)), "per_rank": [round(v, 2) for v in per_rank_us],
                                        "note": "rank r integrates agent r's own trajectory (different geometry and seeds): "
                                                "the max over ranks is the heaviest trajectory, not a slower GPU"},
            "e2e": {"value": e2e_rays / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 2 * ROWS * COLS + 136,
                    "d2h_bytes_per_step": 64 + 24, "us_per_frame": 1e6 * e2e_s / args.steps},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": top, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": per_rank_bytes, "kernel_us": 1e3 * top_ms,
                         "phase_us_per_frame_standalone_kernels": {k: 1e3 * v / args.steps for k, v in kern.items()},
                         "traffic_source": traffic_src,
                         "note": "latency/issue-bound stage: ~1 MB of algorithmic traffic per frame (SURVEY 8d); "
                                 "the bandwidth-shaped stage is the query batch, see 'queries'"},
        }
        if queries:
            qpeak, _ = measured_peak_gbs()
            per = {k_: {"ms": v_} for k_, v_ in queries["ms"].items()}
            n_loc = queries["n_local"]
            sizes = {"getOdd": (int(0.4 * n_loc), 32), "getOccupancy": (int(0.4 * n_loc), 29)}
            sizes["getOddGrad"] = (n_loc - 2 * int(0.4 * n_loc), 76)
            for k_, (cnt, bpq) in sizes.items():
                gbs = cnt * bpq / (per[k_]["ms"] * 1e-3) / 1e9
                per[k_].update({"queries": cnt, "queries_per_s": cnt / (per[k_]["ms"] * 1e-3), "alg_GB_per_s": gbs,
                                "frac_of_hbm_peak": gbs / qpeak})
            out["queries"] = {"metric": "queries_per_sec", "value": args.queries / (q_ms_max * 1e-3), "unit": "queries/s",
                              "n_queries": args.queries, "mix": "40% getOdd, 40% getOccupancy, 20% getOddGrad(max_iter=5)",
                              "ms_per_step": q_ms_max, "per_kernel_rank0": per, "inputs": "device-resident, L2 flushed",
                              "split": "evenly over ranks, each rank queries its own agent map"}
        if lidar:
            out["lidar"] = lidar
        if agents:
            out["agents"] = agents
        if world == 1 and not args.no_cpu:
            try:
                out["other_configs"] = run_other_configs(local_rank)
            except Exception as e:
                out["other_configs"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        if not args.no_cpu:
            nf = min(args.cpu_frames, total)
            c_rays, c_s = run_cpu_sample(cfg, frames, poses, nf)
            if queries:
                from mlmapping_b200 import scenes as _sc
                from oracle_binding import Oracle
                orc = Oracle(cfg, bookkeeping=False, impl=cpu_impl())
                for k in range(min(20, total)):
                    orc.integrate_depth(frames[k], poses[k])
                mo = orc.export_map()
                dd = cfg.subbox_d_xyz * cfg.subbox_n
                qp = _sc.query_positions(300000, mo["glb"].min(0) * dd, (mo["glb"].max(0) + 1) * dd, seed=5)
                t0 = time.perf_counter(); orc.getOdd(qp[:120000]); orc.getOccupancy(qp[120000:240000]); orc.getOddGrad(qp[240000:])
                tq = time.perf_counter() - t0
                out["queries"]["cpu_baseline"] = {"value": 300000 / tq, "unit": "queries/s", "cores": 1, "kind": cpu_impl(),
                                                  "sample": "300k queries (same 4:4:2 mix) on a 20-frame oracle map"}
                # all host cores: getOddGrad keeps its search state in members of the map (like the reference, mlmap.h:100-101),
                # so every thread integrates its own copy of the map and answers one slice of the same stream
                import threading
                ncore = min(os.cpu_count() or 1, 32)
                chunks = np.array_split(np.arange(300000), ncore)
                ready, go = threading.Barrier(ncore + 1), threading.Barrier(ncore + 1)
                done_t = [0.0] * ncore

                o2s = [Oracle(cfg, bookkeeping=False, impl=cpu_impl()) for _ in range(ncore)]

                def _q(i, ix):
                    o2 = o2s[i]
                    for k in range(min(20, total)):
                        o2.integrate_depth(frames[k], poses[k])
                    a = ix[ix < 120000]
                    b = ix[(ix >= 120000) & (ix < 240000)]
                    c = ix[ix >= 240000]
                    ready.wait()
                    go.wait()
                    if len(a): o2.getOdd(qp[a])
                    if len(b): o2.getOccupancy(qp[b])
                    if len(c): o2.getOddGrad(qp[c])
                    done_t[i] = time.perf_counter()
                    o2.close()
                th = [threading.Thread(target=_q, args=(i, ix)) for i, ix in enumerate(chunks)]
                [t_.start() for t_ in th]
                ready.wait()
                t0 = time.perf_counter()
                go.wait()
                [t_.join() for t_ in th]
                tq_all = max(done_t) - t0
                out["queries"]["cpu_baseline_all_cores"] = {"value": 300000 / tq_all, "unit": "queries/s", "cores": ncore, "kind": cpu_impl(),
                                                            "sample": "the same 300k queries split over the host cores, one map copy per thread"}
                orc.close()
            if lidar and "error" not in lidar:
                from mlmapping_b200 import config_cfg_c, scenes as _sc2
                from oracle_binding import Oracle as _Orc
                cfg_c = config_cfg_c()
                oc = _Orc(cfg_c, bookkeeping=False, impl=cpu_impl())
                l_rays, l_s = 0, 0.0
                for k in range(3):
                    pose = _sc2.lidar_loop_pose(k)
                    st_l = oc.integrate_points(_sc2.lidar_scan(pose, frame_idx=k), pose)
                    if k >= 1:
                        l_rays += st_l.n_points
                        l_s += oc.last_seconds
                oc.close()
                out["lidar"]["cpu_baseline"] = {"value": l_rays / l_s, "unit": UNIT, "cores": 1, "kind": cpu_impl(),
                                                "sample": "scans 1-2 of the same loop on the CPU oracle, single thread"}
            out["cpu_baseline"] = {"value": c_rays / c_s, "unit": UNIT, "cores": 1, "kind": cpu_impl(),
                                   "sample": f"first {nf} frames of {WORKLOAD} on the CPU oracle, single thread "
                                             f"({os.cpu_count()} host cores present)",
                                   "us_per_frame": 1e6 * c_s / nf}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
