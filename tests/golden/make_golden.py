"""Generates tests/golden/golden.json: digests + counters on the seeded inputs of SURVEY §8d, produced by
the REFERENCE ITSELF: the unmodified sources of /root/reference compiled into oracle/_ref/libmlmap_ref.so
(oracle/ref_build/Makefile; Eigen / ROS / PCL / OpenCV replaced by the stand-ins of oracle/ref_build/shim).
tests/test_host_logic.py checks the restatement (oracle/mlmap_oracle.hpp) against these digests, so the
restatement stays pinned to the reference on boxes where /root/reference does not exist.
Run where the reference exists:  python tests/golden/make_golden.py"""
import hashlib
import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent))

from mlmapping_b200 import config_cfg_a, config_cfg_c, scenes  # noqa: E402
from oracle_binding import Oracle  # noqa: E402


def _d(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def _summ(o, st, extra=None):
    keys, p = o.last_frame_hits()
    miss = o.last_frame_misses()
    m = o.export_map()
    out = {"n_points": st.n_points, "n_inside": st.n_inside, "n_cast": st.n_cast, "n_hit": st.n_hit_cells,
           "n_miss": st.n_miss_cells, "n_touched": st.n_touched_voxels, "buckets": st.hit_bucket_count,
           "ram_expand_cnt": st.ram_expand_cnt, "obs_cnt": st.obs_cnt,
           "hits_in_order": _d(keys), "hit_p": _d(p), "miss": _d(miss), "subboxes": _d(m["glb"]),
           "occupancy": _d(m["occupancy"]), "log_odds": _d(m["log_odds"]),
           "n_occupied": int((m["occupancy"] == b"o").sum()), "n_free": int((m["occupancy"] == b"f").sum())}
    if extra:
        out.update(extra)
    return out


def run_case(name, impl="port"):
    global Oracle
    base = Oracle
    Oracle = lambda cfg: base(cfg, impl=impl)  # noqa: E731
    try:
        return _run_case(name)
    finally:
        Oracle = base


def _run_case(name):
    if name == "cfg_a_config1_single_frame":
        cfg = config_cfg_a()
        pose = scenes.pose_from_xyz_yaw(5.0, 0.0, 1.2, 0.0)
        img = scenes.corridor_depth_frame(cfg, pose)
        o = Oracle(cfg)
        st = o.integrate_depth(img, pose)
        return _summ(o, st, {"image": _d(img)})
    if name == "cfg_a_config2_first_8_frames_stride_25":
        cfg = config_cfg_a()
        o = Oracle(cfg)
        for k in range(8):
            pose = scenes.corridor_trajectory_pose(25 * k)
            st = o.integrate_depth(scenes.corridor_depth_frame(cfg, pose, frame_idx=25 * k), pose)
        m = o.export_map()
        lo = m["glb"].min(0) * 1.0
        hi = (m["glb"].max(0) + 1) * 1.0
        pos = scenes.query_positions(20000, lo, hi, seed=5, inflate=2.0)
        return _summ(o, st, {"occ_q": _d(o.getOccupancy(pos)), "odd_q": _d(o.getOdd(pos)),
                             "grad_q": _d(o.getOddGrad(pos[:5000]))})
    if name == "cfg_c_small_lidar_3_scans":
        cfg = config_cfg_c()
        cfg.am_n_rho, cfg.am_n_z_below, cfg.am_n_z_over = 120, 30, 30
        o = Oracle(cfg)
        for k in range(3):
            pose = scenes.lidar_loop_pose(3 * k)
            st = o.integrate_points(scenes.lidar_scan(pose, frame_idx=k, beams=32, azimuths=512), pose)
        return _summ(o, st)
    if name == "cfg_a_exploration_6_frames_rolled_poses":
        # exploration mode (update_observation + release pass), poses with roll / pitch, inflation, box fill and the
        # map clouds: the rows of SURVEY 8a a14-a16 and 8f-1/2 in one case
        cfg = config_cfg_a()
        cfg.use_exploration_frontiers = 1
        cfg.inflate_n, cfg.inflate_global_n = 2, 2
        o = Oracle(cfg)
        for k in range(6):
            pose = scenes.corridor_trajectory_pose(40 * k)
            a = 0.05 * np.sin(0.7 * k)
            b = 0.04 * np.cos(0.9 * k)
            q = _quat_mul(pose[3:7], _quat_mul([np.cos(a / 2), np.sin(a / 2), 0, 0], [np.cos(b / 2), 0, np.sin(b / 2), 0]))
            pose = np.r_[pose[:3], q]
            st = o.integrate_depth(scenes.corridor_depth_frame(cfg, pose, rows=240, cols=320, frame_idx=k), pose)
        o.inflate_map(pose[:3])
        o.setFree_map_in_bound([pose[0] + 0.5, -0.4, 0.8], [pose[0] + 1.5, 0.4, 1.6])
        m = o.export_map()

        def rows(a):
            a = np.ascontiguousarray(a).view(np.uint32).reshape(a.shape[0], -1)
            return a[np.lexsort(tuple(a[:, c] for c in range(a.shape[1] - 1, -1, -1)))]
        return _summ(o, st, {"frontier": _d(m["frontier"]), "inflate": _d(m["inflate"]), "collapsed": int(m["collapsed"].sum()),
                             "cloud_inflated": _d(rows(o.export_cloud(0))), "cloud_occupied": _d(rows(o.export_cloud(1))),
                             "cloud_frontier": _d(rows(o.export_cloud(2))), "slice_1.25": _d(rows(o.export_odds_slice(1.25)))})
    raise KeyError(name)


def _quat_mul(a, b):
    aw, ax, ay, az = a
    bw, bx, by, bz = b
    return np.array([aw * bw - ax * bx - ay * by - az * bz, aw * bx + ax * bw + ay * bz - az * by,
                     aw * by - ax * bz + ay * bw + az * bx, aw * bz + ax * by - ay * bx + az * bw])


CASES = ["cfg_a_config1_single_frame", "cfg_a_config2_first_8_frames_stride_25", "cfg_c_small_lidar_3_scans",
         "cfg_a_exploration_6_frames_rolled_poses"]

if __name__ == "__main__":
    from oracle_binding import reference_available
    if not reference_available():
        raise SystemExit("the golden vectors are generated from the reference's own build: oracle/_ref or its sources are needed")
    out = {"generator": "tests/golden/make_golden.py",
           "provenance": "outputs of the UNMODIFIED reference sources (/root/reference src/map_awareness.cpp, src/map_local.cpp, "
                         "src/mlmap.cpp, src/rviz_vis.cpp, include/*.h, 3rdPartLib/Sophus/sophus/{so3,se3}.cpp) built by "
                         "oracle/ref_build/Makefile into oracle/_ref/libmlmap_ref.so with g++ -std=c++17 -O3 (reference "
                         "CMakeLists.txt:4) against the Eigen subset / inert ROS-PCL-OpenCV stand-ins of oracle/ref_build/shim",
           "cases": {c: run_case(c, impl="reference") for c in CASES}}
    (HERE / "golden.json").write_text(json.dumps(out, indent=1))
    print(json.dumps(out, indent=1))
