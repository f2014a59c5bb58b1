"""liodom_scan_lanes on a point-sharded context (needs >= 2 GPUs; launched by torchrun, one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29534 \
        tests/run_sharded_lanes_check.py

Every rank's liodom_scan_lanes must return LIODOM_E_INVALID without enqueueing anything; the next liodom_scan_batch
must then give the pose of the single-GPU path (within 1e-9 m / 1e-10 rad).  Prints one JSON line on rank 0."""
import ctypes
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from liodom_b200 import api, synth  # noqa: E402
from conftest import pose_err  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    scans, _ = synth.sequence("hdl64_small", 1000, 2)
    kw = dict(prev_frames=15, max_points=32768, device=local)
    uid = [api.shard_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    single = api.Context(batch=1, **kw)
    shard = api.Context(batch=1, **kw)
    shard.shard_init(rank, world, uid[0])
    s = np.ascontiguousarray(scans[0], dtype=np.float32)
    before = shard.launch_count
    rc = shard.lib.liodom_scan_lanes(shard.h, (ctypes.c_int32 * 1)(0), 1, (ctypes.c_void_p * 1)(s.ctypes.data),
                                     (ctypes.c_int * 1)(len(s)), 16, 0, 0, 0)
    rejected = rc == -1 and shard.launch_count == before
    worst = [0.0, 0.0]
    for f in scans:
        single.scan_batch([f])
        shard.scan_batch([f])
        dt, dr = pose_err(single.results()[0][0], shard.results()[0][0])
        worst = [max(worst[0], dt), max(worst[1], dr)]
    ok = rejected and worst[0] < 1e-9 and worst[1] < 1e-10
    flags = [None] * world
    dist.all_gather_object(flags, ok)
    if rank == 0:
        print(json.dumps({"check": "sharded_scan_lanes", "world": world, "status": "ok" if all(flags) else "fail",
                          "rejected": bool(rejected), "worst_pose_diff_m": worst[0], "worst_rot_diff_rad": worst[1]}))
    single.close()
    shard.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
