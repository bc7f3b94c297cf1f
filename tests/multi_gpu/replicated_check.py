"""Run under torchrun on N GPUs: rank 0 integrates the CFG-A trajectory; after every frame the dirty subbox blocks
reach the replicas (stored into their inboxes over NVLink peer memory by the library; `--nccl`: broadcast by the caller); the query stream is split evenly over the ranks and the
concatenated answers must equal the CPU oracle's."""
import json
import os
import sys
import time
from pathlib import Path

import numpy as np
import torch
import torch.distributed as dist

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from mlmapping_b200 import config_cfg_a, scenes  # noqa: E402
from mlmapping_b200.sharded import ReplicatedMLMap  # noqa: E402
from mlmapping_b200.sharding import split_range  # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cfg = config_cfg_a()
    rm = ReplicatedMLMap(cfg, rank=rank, world=world, src=0, device=local, transport="nccl" if "--nccl" in sys.argv else "p2p")
    orc = None
    if rank == 0:
        from oracle_binding import Oracle
        orc = Oracle(cfg)
    shipped = []
    for k in range(10):
        pose = scenes.corridor_trajectory_pose(k * 10)
        img = scenes.corridor_depth_frame(cfg, pose, frame_idx=k)
        rm.integrate_depth(img, pose)
        shipped.append(rm.last["broadcast_bytes"])
        if orc is not None:
            orc.integrate_depth(img, pose)
    nq = 2_000_000
    pos = scenes.query_positions(nq, [0.0, -3.0, -1.0], [20.0, 3.0, 4.0], seed=5, inflate=2.0)
    b, e = split_range(nq, rank, world)
    mine = pos[b:e]
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    occ = rm.map.getOccupancy(mine)
    odd = rm.map.getOdd(mine)
    t1 = time.perf_counter() - t0
    parts = [None] * world
    dist.all_gather_object(parts, (occ, odd, t1))
    if rank == 0:
        occ_all = np.concatenate([p[0] for p in parts])
        odd_all = np.concatenate([p[1] for p in parts])
        assert np.array_equal(occ_all, orc.getOccupancy(pos)), "replica occupancy differs from the oracle"
        assert np.array_equal(odd_all.view(np.uint32), orc.getOdd(pos).view(np.uint32))
        print(json.dumps({"replicated_check": "ok", "world": world, "queries": 2 * nq,
                          "host_path_queries_per_s": 2 * nq / max(p[2] for p in parts),
                          "broadcast_bytes_per_frame": shipped}))
    dist.barrier()
    rm.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
