"""Generates tests/golden/golden_long.json: per-frame counters and digests of the long series of SURVEY §8d (the whole
1000-frame CFG-A trajectory, 50 CFG-B frames, 12 full CFG-C scans), produced by the REFERENCE ITSELF (oracle/_ref, the
unmodified sources of /root/reference; see make_golden.py).  The GPU tests replay the same seeded inputs and compare
with these vectors, so the GPU box does not spend minutes in the CPU reference while it holds a B200.
Run where the reference exists:  python tests/golden/make_golden_long.py   (about ten minutes of CPU)"""
import hashlib
import json
import sys
import time
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent))

from mlmapping_b200 import config_cfg_a, config_cfg_b, config_cfg_c, scenes  # noqa: E402
from oracle_binding import Oracle, reference_available  # noqa: E402

COUNTERS = ("n_points", "n_inside", "n_cast", "n_hit_cells", "n_miss_cells", "n_touched_voxels", "hit_bucket_count",
            "ram_expand_cnt", "obs_cnt")


def d(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:20]


def map_digest(m):
    h = hashlib.sha256()
    for k in ("glb", "collapsed", "occupancy", "inflate", "log_odds"):
        h.update(np.ascontiguousarray(m[k]).tobytes())
    return h.hexdigest()[:20]


def frame_digest(o):
    keys, p = o.last_frame_hits()
    return {"hits_in_order": d(keys), "hit_p": d(p), "miss": d(o.last_frame_misses())}


def series(name):
    """yields (k, kind, data, pose) of the named series; shared with the GPU tests"""
    if name == "cfg_a_1000":
        cfg = config_cfg_a()
        for k in range(1000):
            pose = scenes.corridor_trajectory_pose(k)
            yield k, "depth", scenes.corridor_depth_frame(cfg, pose, frame_idx=k), pose
    elif name == "cfg_b_50":
        cfg = config_cfg_b()
        for k in range(50):
            pose = scenes.corridor_trajectory_pose(k, step=0.1)
            yield k, "depth", scenes.corridor_depth_frame(cfg, pose, rows=768, cols=1024, frame_idx=k, length=200.0), pose
    elif name == "cfg_c_12":
        for k in range(12):
            pose = scenes.lidar_loop_pose(k)
            yield k, "points", scenes.lidar_scan(pose, frame_idx=k), pose
    else:
        raise KeyError(name)


SERIES = {"cfg_a_1000": (config_cfg_a, 50, 100), "cfg_b_50": (config_cfg_b, 10, 25), "cfg_c_12": (config_cfg_c, 4, 6)}


def run(name, impl):
    make_cfg, frame_every, map_every = SERIES[name]
    o = Oracle(make_cfg(), impl=impl)
    out = {"counters": [], "frames": {}, "maps": {}}
    t0 = time.time()
    for k, kind, data, pose in series(name):
        st = o.integrate_depth(data, pose) if kind == "depth" else o.integrate_points(data, pose)
        out["counters"].append([int(getattr(st, f)) for f in COUNTERS])
        if k % frame_every == frame_every - 1:
            out["frames"][str(k)] = frame_digest(o)
        if k % map_every == map_every - 1:
            m = o.export_map()
            out["maps"][str(k)] = {"digest": map_digest(m), "subboxes": int(m["glb"].shape[0])}
    out["seconds"] = round(time.time() - t0, 1)
    return out


if __name__ == "__main__":
    if not reference_available():
        raise SystemExit("generated from the reference's own build: oracle/_ref or its sources are needed")
    res = {"generator": "tests/golden/make_golden_long.py", "counters": list(COUNTERS),
           "provenance": "outputs of the UNMODIFIED reference sources built into oracle/_ref/libmlmap_ref.so (see golden.json)",
           "series": {n: run(n, "reference") for n in SERIES}}
    (HERE / "golden_long.json").write_text(json.dumps(res, separators=(",", ":")))
    print({n: (v["seconds"], len(v["counters"])) for n, v in res["series"].items()})
