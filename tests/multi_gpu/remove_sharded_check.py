"""ekf_remove_lines on a row-sharded filter returns EKF_EINVAL (compaction would move rows between ranks) and leaves the
state alone.  Launch:  python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
                           --master-port 29531 tests/multi_gpu/remove_sharded_check.py"""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from slam_ros_b200 import EkfFilter, scenario as sc  # noqa: E402
from slam_ros_b200.ekf import EkfError, EKF_EINVAL, nccl_unique_id  # noqa: E402


def main():
    rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"]); local = int(os.environ["LOCAL_RANK"])
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    uid = torch.zeros(128, dtype=torch.uint8, device=dev)
    if rank == 0:
        uid = torch.tensor(list(nccl_unique_id()), dtype=torch.uint8, device=dev)
    dist.broadcast(uid, 0)
    N = 200
    f = EkfFilter(capacity_lines=N + 64, device=local, shard=(rank, world, bytes(uid.cpu().tolist())))
    scn = sc.map_scenario(N, 2, m=8, seed=5)
    f.scan(np.zeros(3), scn["seed_z"], scn["seed_R"])
    f.scan(scn["u"][0], scn["z"][0], scn["R"][0])
    y0 = f.download_y()
    try:
        f.remove_lines([0, 5])
        raise AssertionError("a row-sharded filter accepted ekf_remove_lines")
    except EkfError as e:
        assert e.code == EKF_EINVAL, e
    assert f.lines == N and np.array_equal(f.download_y(), y0)
    print("rank %d: remove_lines refused" % rank, flush=True)
    dist.barrier()
    f.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
