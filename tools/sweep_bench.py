"""Throughput of cvx_sweep on mill 1024^3 built resident (cvx_world_build_from_mesh), LOD 0. Prints one JSON line.

(a) 1 M character boxes (half extents 0.3, 0.9, 0.3) at random free positions, random directions, max_distance 16;
(b) 1 M boxes of half extent 0.5 along the 3840x2160 pick rays of 6 benchmark-path poses (every 48th ray), max_distance +inf;
(c) 1 M 4-cell boxes (half extent 2) at random free positions, random directions, max_distance 64.
A position is free when a sweep there with max_distance 0 reports no overlap. For each set: boxes/s and headers/s (headers = the
`steps` the kernel counts) on the device path (boxes and hits in device memory, CUDA events on the context's stream), on the host
path (host arrays in and out, wall clock of the returning call), and of the cell-by-cell definition (tools/raycast_oracle) on 16
host threads over a subset. The device hits are checked against the host path on every field, and the subset against the
definition on every field but `steps`.

    python tools/sweep_bench.py [--reps 5] [--oracle-stride 4096]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

N = 1 << 20


def free_boxes(cv, rm, rng, dims, half, max_distance):
    """N boxes of half extents `half` at random positions where they overlap no solid cell, random directions."""
    out = []
    while sum(len(b) for b in out) < N:
        c = rng.random((2 * N, 3)) * np.array(dims)
        probe = cv.make_boxes(c, half, rng.normal(size=(2 * N, 3)), 0.0)
        out.append(probe[rm.sweep_boxes(probe)["hit"] == 0])
    boxes = np.concatenate(out)[:N]
    boxes["max_distance"] = max_distance
    return boxes


def measure(cv, rm, boxes, reps, oracle_world, oracle_stride):
    import torch
    import sweep_oracle as swo
    stream = torch.cuda.current_stream()
    n = len(boxes)
    t_boxes = torch.from_numpy(boxes.view(np.uint8)).cuda()
    t_hits = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
    rm.sweep_device(t_boxes.data_ptr(), t_hits.data_ptr(), n)        # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        rm.sweep_device(t_boxes.data_ptr(), t_hits.data_ptr(), n)
    e1.record(stream)
    e1.synchronize()
    dev_s = e0.elapsed_time(e1) / 1e3 / reps
    dev_hits = t_hits.cpu().numpy().view(cv.RAY_HIT_DTYPE)
    rm.sweep_boxes(boxes)                                             # warm-up (scratch growth)
    t0 = time.perf_counter()
    for _ in range(reps):
        hits = rm.sweep_boxes(boxes)
    host_s = (time.perf_counter() - t0) / reps
    exact = bool(np.array_equal(hits.view(np.uint8), dev_hits.view(np.uint8)))
    headers = int(hits["steps"].astype(np.int64).sum())
    sub = boxes[::oracle_stride]
    t0 = time.perf_counter()
    ref = swo.sweep(oracle_world, sub, threads=16)
    o_s = time.perf_counter() - t0
    got = hits[::oracle_stride].copy()
    got["steps"] = 0
    exact &= bool(np.array_equal(got.view(np.uint8), ref.view(np.uint8)))
    return {"boxes": n, "headers": headers, "device_ms": dev_s * 1e3, "device_boxes_per_s": n / dev_s,
            "device_headers_per_s": headers / dev_s, "host_ms": host_s * 1e3, "host_boxes_per_s": n / host_s,
            "host_headers_per_s": headers / host_s, "oracle_boxes": len(sub), "oracle_boxes_per_s": len(sub) / o_s,
            "oracle_threads": 16, "hit_share": float(np.mean(hits["hit"] == 1)),
            "face6_share": float(np.mean(hits["face"] == 6)), "bit_exact": exact}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--oracle-stride", type=int, default=4096)
    ap.add_argument("--max-dimension", type=int, default=1024)
    args = ap.parse_args()
    import torch
    import cpuvox_b200 as cv
    import raycast_oracle as rco
    from conftest import MILL, parse_obj
    from raycast_bench import gpu_info, pick_grid
    torch.cuda.init()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    rm = cv.RenderManager(0)
    rm.set_stream(stream.cuda_stream)   # the context runs on this stream, so the CUDA events below are on the context's stream
    P, Cc = parse_obj(MILL)
    host_world = rm.build_world_from_mesh(P, Cc, args.max_dimension, flips=(True, False, False))   # blobs for the definition
    world = rm.build_resident_world_from_mesh(P, Cc, args.max_dimension, flips=(True, False, False))
    ow = rco.RayWorld(host_world)
    rng = np.random.default_rng(1)
    W, H = 3840, 2160
    poses = [cv.benchmark_pose(cv.benchmark_length() * k / 5, world.dims, far_clip=2.0 * max(world.dims)) for k in range(6)]
    rays = np.concatenate([pick_grid(cv, p, W, H)[::48] for p in poses])[:N]
    along = cv.make_boxes(rays["origin"], (0.5, 0.5, 0.5), rays["direction"], np.inf)
    out = {"tool": "sweep_bench", "world": f"mill {world.dims[0]}x{world.dims[1]}x{world.dims[2]}", "lod": 0,
           "regular": rm.world_is_regular(), **gpu_info(), "reps": args.reps,
           "character_1m_free_16": measure(cv, rm, free_boxes(cv, rm, rng, world.dims, (0.3, 0.9, 0.3), 16.0), args.reps, ow,
                                           args.oracle_stride),
           "half05_1m_pick_rays_6_poses_inf": measure(cv, rm, along, args.reps, ow, args.oracle_stride),
           "cell4_1m_free_64": measure(cv, rm, free_boxes(cv, rm, rng, world.dims, (2.0, 2.0, 2.0), 64.0), args.reps, ow,
                                       args.oracle_stride)}
    rm.set_stream(0)
    rm.destroy()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
