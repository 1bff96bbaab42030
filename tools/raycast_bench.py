"""Throughput of cvx_raycast on mill 1024^3 built resident (cvx_world_build_from_mesh). Prints one JSON line.

(a) pick grids: every pixel of a 3840x2160 frame (8.3 M rays) from 6 poses of the benchmark path;
(b) 1 M random rays starting inside the world.
For each: rays/s and cells/s (cells = the `steps` the definition counts) on the device path (rays and hits in device memory,
CUDA events on the context's stream), on the host path (host arrays in and out, wall clock of the returning call), and of the
per-cell definition (tools/raycast_oracle) on all host threads over a subset. The device hits of every ray are checked against
the host path, and a subset against the definition, bit for bit.

    python tools/raycast_bench.py [--reps 5] [--oracle-stride 64]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def quat_rotate(q, v):
    """Quaternion * Vector3 (host_setup.cpp rotate) in fp32 on arrays of vectors."""
    x, y, z, w = (np.float32(a) for a in q)
    two = np.float32(2)
    x2, y2, z2 = x * two, y * two, z * two
    xx, yy, zz, xy, xz, yz = x * x2, y * y2, z * z2, x * y2, x * z2, y * z2
    wx, wy, wz = w * x2, w * y2, w * z2
    one = np.float32(1)
    px, py, pz = v[:, 0], v[:, 1], v[:, 2]
    return np.stack([(one - (yy + zz)) * px + (xy - wz) * py + (xz + wy) * pz,
                     (xy + wz) * px + (one - (xx + zz)) * py + (yz - wx) * pz,
                     (xz - wy) * px + (yz + wx) * py + (one - (xx + yy)) * pz], axis=1)


def pick_grid(cv, pose, W, H):
    """cvx_host_screen_ray for the centre of every pixel, vectorised (same formulas; the benchmark needs 8.3 M rays per pose)."""
    ys, xs = np.mgrid[0:H, 0:W]
    px = xs.ravel().astype(np.float32) + np.float32(0.5)
    py = ys.ravel().astype(np.float32) + np.float32(0.5)
    tan_half = np.float32(np.tan(np.float64(np.float32(pose.fov_y_degrees) * np.float32(0.017453292) * np.float32(0.5))))
    aspect = np.float32(W) / np.float32(H)
    cam = np.stack([(np.float32(2) * px / np.float32(W) - np.float32(1)) * aspect * tan_half,
                    (np.float32(2) * py / np.float32(H) - np.float32(1)) * tan_half, np.ones_like(px)], axis=1)
    near = np.float32(pose.near_clip)
    origin = np.asarray(pose.position, dtype=np.float32) + quat_rotate(pose.rotation, cam * near)
    unit = cam / np.sqrt(np.sum(cam * cam, axis=1, dtype=np.float32))[:, None]
    return cv.make_rays(origin, quat_rotate(pose.rotation, unit.astype(np.float32)))


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit_clocks_max_sm_clocks_sm"] = out
    except Exception as e:  # noqa: BLE001
        info["nvidia_smi"] = str(e)
    return info


def measure(cv, rm, sets, reps, oracle_world, oracle_stride):
    import torch
    import raycast_oracle as rco
    stream = torch.cuda.current_stream()
    res = {"rays": int(sum(len(r) for r in sets))}
    dev_s = host_s = 0.0
    cells = 0
    exact = True
    for rays in sets:
        n = len(rays)
        t_rays = torch.from_numpy(rays.view(np.uint8)).cuda()
        t_hits = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
        rm.raycast_device(t_rays.data_ptr(), t_hits.data_ptr(), n)    # warm-up
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            rm.raycast_device(t_rays.data_ptr(), t_hits.data_ptr(), n)
        e1.record(stream)
        e1.synchronize()
        dev_s += e0.elapsed_time(e1) / 1e3 / reps
        dev_hits = t_hits.cpu().numpy().view(cv.RAY_HIT_DTYPE)
        rm.raycast_rays(rays)                                           # warm-up (scratch growth)
        t0 = time.perf_counter()
        for _ in range(reps):
            hits = rm.raycast_rays(rays)
        host_s += (time.perf_counter() - t0) / reps
        exact &= bool(np.array_equal(hits.view(np.uint8), dev_hits.view(np.uint8)))
        cells += int(hits["steps"].astype(np.int64).sum())
    res.update(cells=cells, device_rays_per_s=res["rays"] / dev_s, device_cells_per_s=cells / dev_s,
               host_rays_per_s=res["rays"] / host_s, host_cells_per_s=cells / host_s, device_ms=dev_s * 1e3, host_ms=host_s * 1e3)
    sub = np.concatenate([r[::oracle_stride] for r in sets])
    t0 = time.perf_counter()
    ref = rco.raycast(oracle_world, sub)
    o_s = time.perf_counter() - t0
    got = rm.raycast_rays(sub)
    exact &= bool(np.array_equal(got.view(np.uint8), ref.view(np.uint8)))
    o_cells = int(ref["steps"].astype(np.int64).sum())
    res.update(oracle_rays=len(sub), oracle_rays_per_s=len(sub) / o_s, oracle_cells_per_s=o_cells / o_s,
               oracle_threads=os.cpu_count(), hit_share=float(np.mean(got["hit"] == 1)), bit_exact=exact)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--oracle-stride", type=int, default=64)
    ap.add_argument("--max-dimension", type=int, default=1024)
    args = ap.parse_args()
    import torch
    import cpuvox_b200 as cv
    import raycast_oracle as rco
    from conftest import MILL, parse_obj
    torch.cuda.init()
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    rm = cv.RenderManager(0)
    rm.set_stream(stream.cuda_stream)   # the context runs on this stream, so the CUDA events below are on the context's stream
    P, Cc = parse_obj(MILL)
    host_world = rm.build_world_from_mesh(P, Cc, args.max_dimension, flips=(True, False, False))   # blobs for the definition
    t0 = time.perf_counter()
    world = rm.build_resident_world_from_mesh(P, Cc, args.max_dimension, flips=(True, False, False))
    build_s = time.perf_counter() - t0
    ow = rco.RayWorld(host_world)
    W, H = 3840, 2160
    poses = [cv.benchmark_pose(cv.benchmark_length() * k / 5, world.dims, far_clip=2.0 * max(world.dims)) for k in range(6)]
    grids = [pick_grid(cv, p, W, H) for p in poses]
    rng = np.random.default_rng(1)
    n = 1 << 20
    dirs = rng.normal(size=(n, 3)).astype(np.float32)
    rand = cv.make_rays((rng.random((n, 3)) * np.array(world.dims)).astype(np.float32), dirs)
    out = {"tool": "raycast_bench", "world": f"mill {world.dims[0]}x{world.dims[1]}x{world.dims[2]}", "resident_build_s": build_s,
           "regular": rm.world_is_regular(), **gpu_info(), "reps": args.reps,
           "pick_4k_6_poses": measure(cv, rm, grids, args.reps, ow, args.oracle_stride),
           "random_1m_inside": measure(cv, rm, [rand], args.reps, ow, args.oracle_stride)}
    rm.set_stream(0)
    rm.destroy()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
