"""Worker of tests/test_gpu_multi.py (run under torchrun, one process per rank): the multi-GPU paths of cpuvox_b200/parallel.py on
real devices, each compared bit for bit with a single-GPU render on rank 0:
  * one view, rays sharded, CUDA-IPC peer-store gather ("p2p");
  * a stream of views, rays sharded, frame ring with device-side flow control ("ring"), more views than ring slots;
  * batched views, views sharded.
With fewer devices than ranks every rank runs on device 0 and gloo carries the rendezvous (NCCL needs a device per rank): the
IPC mappings, the peer stores into another process's memory and the ring's flags between processes are then exercised on one GPU."""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    import torch.distributed as dist

    import cpuvox_b200 as cv

    rank, local, n = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"]), int(os.environ["WORLD_SIZE"])
    shared = torch.cuda.device_count() < n
    local = 0 if shared else local
    torch.cuda.set_device(local)
    if shared:
        dist.init_process_group("gloo")
    else:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    world = cv.World.from_obj(os.path.join(ROOT, "tests", "data", "mill.obj"), 256) if rank == 0 else None
    world = cv.broadcast_world(world, src=0, device=None if shared else torch.device(f"cuda:{local}"))
    poses = cv.benchmark_path(world.dims, 12, far_clip=2.0 * world.max_dimension)
    ok = True
    ref = None
    if rank == 0:
        ref = cv.RenderManager(local)
        ref.upload_world(world)

    def want(pose, W, H):
        ref.set_resolution(W, H)
        ref.draw_world(pose)
        return ref.read_frame()

    srm = cv.ShardedRenderManager(local, rank, n, gather="p2p")
    srm.upload_world(world)
    for (W, H) in ((640, 360), (1920, 1080)):
        srm.set_resolution(W, H)
        for i, pose in enumerate(poses[::2]):
            srm.draw_world_sharded(pose)
            if rank == 0:
                same = np.array_equal(srm.read_frame(), want(pose, W, H))
                ok &= same
                if not same:
                    print(f"MISMATCH gather=p2p {W}x{H} pose {i}", flush=True)
    srm.destroy()

    # frame ring: 12 views through 3 ring slots, twice (the view counter keeps running), at two resolutions
    srm = cv.ShardedRenderManager(local, rank, n, gather="ring", ring_slots=3)
    srm.upload_world(world)
    for (W, H) in ((640, 360), (1920, 1080)):
        srm.set_resolution(W, H)
        dst = cv.alloc_pinned((len(poses), H, W)) if rank == 0 else None
        for rep in range(2):
            if rank == 0:
                dst[:] = 0
            # rep 0: rays dealt in chunks of 32 (interleaved); rep 1: one contiguous, weight-balanced range per rank
            srm.draw_views_sharded(poses, dst, chunk=32 if rep == 0 else 0)
            if rank == 0:
                for i, pose in enumerate(poses):
                    same = np.array_equal(dst[i], want(pose, W, H))
                    ok &= same
                    if not same:
                        print(f"MISMATCH ring {W}x{H} rep {rep} view {i}: {int((dst[i] != want(pose, W, H)).sum())} pixels", flush=True)
    srm.destroy()

    # views sharded
    srm = cv.ShardedRenderManager(local, rank, n)
    srm.upload_world(world)
    W, H = 1280, 720
    srm.set_resolution(W, H)
    mine = cv.partition_views(len(poses), n, rank)
    dst = cv.alloc_pinned((len(mine), H, W))
    got_idx = srm.draw_views(poses, dst)
    frames = [None] * n
    dist.all_gather_object(frames, (got_idx, np.array(dst)))
    if rank == 0:
        for idx, fr in frames:
            for j, i in enumerate(idx):
                same = np.array_equal(want(poses[i], W, H), fr[j])
                ok &= same
                if not same:
                    print(f"MISMATCH views sharded: view {i}", flush=True)
        print("MULTI-GPU CHECK " + ("PASSED" if ok else "FAILED"), flush=True)
        ref.destroy()
    srm.destroy()
    dist.barrier()
    dist.destroy_process_group()
    if rank == 0 and not ok:
        sys.exit(1)


if __name__ == "__main__":
    main()
