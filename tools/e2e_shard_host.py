"""host-side cost of mlm_shard_submit and mlm_shard_finish"""
import sys, time
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from mlmapping_b200 import config_cfg_c, scenes
from mlmapping_b200.sharded import sharded_group_in_process
cfg = config_cfg_c()
sh = sharded_group_in_process(cfg, 1)[0]
data = []
for k in range(6):
    pose = scenes.lidar_loop_pose(k)
    data.append((scenes.lidar_scan(pose, frame_idx=k), pose))
buf = sh.pinned_points(max(p.shape[0] for p, _ in data))
for k, (pts, pose) in enumerate(data):
    b = buf[:pts.shape[0]]
    b[...] = pts
    sh.map.sync()
    t0 = time.perf_counter()
    sh.submit(b, pose)
    t1 = time.perf_counter()
    sh.finish()
    t2 = time.perf_counter()
    print(k, f"submit {1e6*(t1-t0):.1f} us, finish {1e6*(t2-t1):.1f} us")
