"""Multi-GPU plumbing: one process per GPU, `torch.distributed` for rendezvous, world broadcast and barriers.

The path shards by independent units (SURVEY.md §8(e)): every ray reads the shared read-only world and writes only its own
raybuffer row (DrawSegmentRayJob.cs:106,199), so
  * batched views (BASELINE config 5) are dealt round-robin to ranks, no per-frame exchange at all;
  * a single large view (configs 3, 4) is cut into contiguous flat-ray ranges in RaySetupJob order (DrawSegmentRayJob.cs:12-40);
    each rank runs Phase 1 for its rays and Phase 2 only for the screen pixels those rays feed, storing them straight into
    the root's framebuffer through a CUDA-IPC mapping (NVLink peer stores; the gather is the kernel's own stores).
torch is used for process-group plumbing only; all rendering goes through the C ABI.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import numpy as np

from .host import CameraPose, RenderManager, World
from .native import FrameSetup


def partition_rays(total_rays: int, world_size: int, weights: Optional[Sequence[float]] = None) -> List[Tuple[int, int]]:
    """Contiguous flat-ray ranges, one per rank, balanced by `weights` (per-ray cost estimates; equal if None)."""
    if world_size < 1:
        raise ValueError("world_size < 1")
    if total_rays <= 0:
        return [(0, 0)] * world_size
    if weights is None:
        cuts = [(total_rays * r) // world_size for r in range(world_size + 1)]
    else:
        w = np.asarray(weights, dtype=np.float64)
        if w.shape != (total_rays,) or (w < 0).any():
            raise ValueError("weights must be one non-negative value per ray")
        cum = np.concatenate([[0.0], np.cumsum(w)])
        if cum[-1] <= 0:
            return partition_rays(total_rays, world_size)
        targets = cum[-1] * np.arange(1, world_size) / world_size
        inner = np.searchsorted(cum, targets, side="left")
        inner = [i - 1 if i > 0 and (i > total_rays or t - cum[i - 1] < cum[i] - t) else i for i, t in zip(inner, targets)]  # nearest cut
        cuts = [0] + [int(min(max(c, 0), total_rays)) for c in inner] + [total_rays]
        for i in range(1, len(cuts)):
            cuts[i] = max(cuts[i], cuts[i - 1])
    return [(cuts[r], cuts[r + 1]) for r in range(world_size)]


def ray_weights(setup: FrameSetup, width: int, height: int) -> np.ndarray:
    """Default per-ray cost estimate: the writable pixels of the ray's row (RenderManager.cs:298-316)."""
    vx, vy = setup.vanishing_point_screen
    out = []
    for k in range(4):
        rc = setup.segments[k].ray_count
        if rc <= 0:
            continue
        if k < 2:
            v = int(min(max(np.rint(np.float32(vy)), 0), height - 1))
            n = height - v if k == 0 else v + 1
        else:
            v = int(min(max(np.rint(np.float32(vx)), 0), width - 1))
            n = v + 1 if k == 3 else width - v
        out.append(np.full(rc, float(n)))
    return np.concatenate(out) if out else np.zeros(0)


def partition_views(n_views: int, world_size: int, rank: int) -> List[int]:
    """Views dealt round-robin: view i -> rank i mod world_size."""
    return list(range(rank, n_views, world_size))


def broadcast_world(world: Optional[World], src: int = 0, device=None, group=None) -> World:
    """World broadcast once from `src` and replicated per rank (blobs travel as uint8 tensors: NCCL when `device` is a
    CUDA device, gloo on CPU)."""
    import torch
    import torch.distributed as dist

    rank = dist.get_rank(group)
    meta = [None]
    if rank == src:
        meta = [(tuple(world.dims), list(world.column_counts), list(world.voxel_counts), [int(b.nbytes) for b in world.blobs])]
    dist.broadcast_object_list(meta, src=src, group=group)
    dims, cols, vox, sizes = meta[0]
    blobs = []
    for i, n in enumerate(sizes):
        if rank == src:
            t = torch.from_numpy(np.ascontiguousarray(world.blobs[i]))
            if device is not None:
                t = t.to(device)
        else:
            t = torch.empty(n, dtype=torch.uint8, device=device if device is not None else "cpu")
        dist.broadcast(t, src=src, group=group)
        blobs.append(world.blobs[i] if rank == src else t.cpu().numpy())
    return world if rank == src else World(tuple(dims), blobs, list(cols), list(vox))


class ShardedRenderManager:
    """One rank's share of a multi-GPU render. Wraps a RenderManager on `device`.

    gather: "p2p"    one view at a time: peer stores into the root's framebuffer, a host barrier per view;
            "ring"   a stream of views: peer stores into a ring of framebuffers on the root, all ordering between ranks on the
                     device (flag words polled by tiny kernels), no host barrier and no collective between views."""

    def __init__(self, device: int, rank: int, world_size: int, gather: str = "p2p", group=None, ring_slots: int = 4):
        if gather not in ("p2p", "ring"):
            raise ValueError("gather must be 'p2p' or 'ring'")
        self.rm = RenderManager(device)
        self.device, self.rank, self.world_size, self.gather, self.group = device, rank, world_size, gather, group
        self.ring_slots = ring_slots
        self._root_frame_ptr = 0      # mapped pointer to rank 0's framebuffer (p2p, rank != 0)
        self._next_view = 0           # ring: running view index, the same on every rank
        self._ring_ready = False

    def upload_world(self, world: World):
        self.rm.upload_world(world)

    def set_resolution(self, width: int, height: int):
        import torch.distributed as dist

        same = width == self.rm.width and height == self.rm.height
        if same and (self._root_frame_ptr or self._ring_ready or self.world_size == 1):
            return
        if self.world_size > 1 and not same:
            # peers close their mappings of the root's memory BEFORE the root reallocates it (CUDA IPC rule), then everyone moves on
            if self._root_frame_ptr:
                self.rm.ipc_close(self._root_frame_ptr)
                self._root_frame_ptr = 0
            if self._ring_ready and self.rank != 0:
                self.rm.ring_close()
            self._ring_ready = False
            dist.barrier(group=self.group)
        self.rm.set_resolution(width, height)
        if self.world_size == 1:
            if self.gather == "ring":   # a ring of one rank: the same code path, no mapping to exchange
                self.rm.ring_create(self.ring_slots, 1)
                self._ring_ready = True
                self._next_view = 0
            return
        if self.gather == "p2p":
            handle = [self.rm.ipc_export_frame() if self.rank == 0 else None]
            dist.broadcast_object_list(handle, src=0, group=self.group)
            if self.rank != 0:
                self._root_frame_ptr = self.rm.ipc_open(handle[0])
        else:
            handle = [self.rm.ring_create(self.ring_slots, self.world_size) if self.rank == 0 else None]
            dist.broadcast_object_list(handle, src=0, group=self.group)
            if self.rank != 0:
                self.rm.ring_open(handle[0], self.ring_slots, self.world_size)
            self._ring_ready = True
            self._next_view = 0

    def draw_world_sharded(self, pose: CameraPose, weights: Optional[Sequence[float]] = None) -> FrameSetup:
        """Single view, rays sharded: after the call (and its barrier) rank 0's framebuffer holds the whole frame."""
        import torch.distributed as dist

        rm = self.rm
        setup = rm.make_setup(pose)
        total = sum(max(0, setup.segments[k].ray_count) for k in range(4))
        if weights is None:
            weights = ray_weights(setup, rm.width, rm.height)
        begin, end = partition_rays(total, self.world_size, weights)[self.rank]
        if self.world_size == 1 and self.gather != "ring":
            rm.draw_setup(setup)
            return setup
        if self.gather == "ring":
            self.draw_views_sharded([pose], weights=[weights])
            return setup
        # the previous view is final on the root only after the barrier that ended it; whoever reads or presents it there must do
        # so before entering this call — this barrier keeps a fast rank from storing into it any earlier than that
        dist.barrier(group=self.group)
        rm.draw_rays(setup, begin, end)
        rm.blit_owned(setup, begin, end, self._root_frame_ptr)
        rm.sync()
        dist.barrier(group=self.group)  # every rank's peer stores have landed
        return setup

    def draw_views_sharded(self, poses: Sequence[CameraPose], dst: Optional[np.ndarray] = None, weights: Optional[Sequence] = None,
                           barrier: bool = True, chunk: int = 512, sync: bool = True) -> List[FrameSetup]:
        """A stream of views, each with its rays sharded over all ranks (gather="ring"). Every rank enqueues its share of every
        view without waiting for anyone; the root consumes view v (into dst[v] if given: pinned host memory, one frame per view)
        as soon as all shares of it have arrived and thereby frees its ring slot. Returns when this rank's work is done
        (and, with `barrier`, when every rank's is); with sync=False it returns as soon as the work is enqueued (sync_views waits). Rays are dealt to the ranks in chunks of `chunk` rays unless `weights`
        (per-ray cost estimates, one array per view) are given or chunk == 0: then each rank takes one contiguous, weight-balanced range."""
        import torch.distributed as dist

        if self.gather != "ring" or not self._ring_ready:
            raise RuntimeError("draw_views_sharded needs gather='ring' and a resolution")
        rm = self.rm
        setups = []
        base = self._next_view
        lag = self.ring_slots - 1
        for i, pose in enumerate(poses):
            setup = rm.make_setup(pose)
            setups.append(setup)
            if weights is None and chunk > 0:
                # rays dealt in chunks of `chunk` (chunk c -> rank c mod N): balanced without a cost estimate
                rm.draw_sharded(setup, -1, chunk, base + i, self.rank)
            else:
                total = sum(max(0, setup.segments[k].ray_count) for k in range(4))
                w = weights[i] if weights is not None else ray_weights(setup, rm.width, rm.height)
                begin, end = partition_rays(total, self.world_size, w)[self.rank]
                rm.draw_sharded(setup, begin, end, base + i, self.rank)
            if self.rank == 0 and i >= lag:
                rm.ring_consume(base + i - lag, dst[i - lag] if dst is not None else None)
        if self.rank == 0:
            for i in range(max(0, len(poses) - lag), len(poses)):
                rm.ring_consume(base + i, dst[i] if dst is not None else None)
        self._next_view = base + len(poses)
        if sync:
            self.sync_views(barrier)
        return setups

    def sync_views(self, barrier: bool = True):
        """Wait for everything draw_views_sharded(sync=False) enqueued on this rank (and, with `barrier`, on every rank)."""
        import torch.distributed as dist

        self.rm.sync()
        if self.rank == 0:
            self.rm.ring_status()
        if barrier and self.world_size > 1:
            dist.barrier(group=self.group)

    def draw_views(self, poses: Sequence[CameraPose], dst: Optional[np.ndarray] = None) -> List[int]:
        """Batched views: this rank renders views rank, rank+N, ...; returns their indices (frames land in `dst`, one
        W*H slab per local view, if given)."""
        mine = partition_views(len(poses), self.world_size, self.rank)
        setups = [self.rm.make_setup(poses[i]) for i in mine]
        if setups:
            self.rm.draw_batch(setups, dst)
        return mine

    def read_frame(self) -> np.ndarray:
        """The last single view on the root (p2p). Ring views are delivered through draw_views_sharded(dst=...)."""
        return self.rm.read_frame()

    def destroy(self):
        import torch.distributed as dist

        if self._root_frame_ptr:
            self.rm.ipc_close(self._root_frame_ptr)
            self._root_frame_ptr = 0
        if self._ring_ready and self.world_size > 1:
            if self.rank != 0:
                self.rm.ring_close()
            dist.barrier(group=self.group)   # mappings are closed before the root frees the ring
            self._ring_ready = False
        self.rm.destroy()
