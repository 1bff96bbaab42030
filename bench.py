"""bench.py — the headline benchmark of the raybuffer path (BASELINE.json: frames/sec on mill 1024^3 at 1080p & 4K).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config 1..5] [--mode views|rays] [--res WxH] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

Workloads (config.workload; BASELINE.json `configs`, made concrete in SURVEY.md §8(d)):
  1 (default, the line the driver records) datasets/mill.obj voxelized to 1024^3 (+5 LOD mips), rendered along the reference's own
    benchmark camera path (BenchmarkPath.anim sampled at 60 evenly spaced times, UnityManager.cs:86-87) at 3840x2160 — the
    north_star's headline resolution; 1080p is reported beside it under "at_1080p". A step = one pass over the 60 poses.
  2 fBm terrain 2048^3 (seed 1234), 1920x1080, camera at the centre, y 1700, pitch 60 down, 16 yaws (vanishing point on screen, 4 segments)
  3 the same terrain, 3840x2160, 40 above the ground, pitch 3 and pitch 0 (LimitRotationHorizon), 8 yaws each (clamped segments)
  4 boxes/pipes/slabs 4096x1024x4096 (seed 7), 7680x4320, far 8192, 4 views; with N > 1 the RAYS of every view are sharded (--mode rays)
  5 256 cameras (seed 99) at 1280x720 over the terrain; with N > 1 the VIEWS are sharded
A step = one pass over the config's views.

value    frames/s with everything resident in HBM: per frame one Phase-1 and one Phase-2 launch; a step is one
         cvx_draw_batch over the views (device only), which keeps up to `frames_in_flight` views in flight, each on its own
         stream with its own raybuffers and framebuffer (the reference double-buffers its raybuffers for the same overlap,
         RenderManager.cs:14,53-56). "at_inflight" repeats the measurement with 1 and 2 views in flight (the interactive case).
e2e      frames/s through the public C ABI with HOST buffers (cvx_draw_world_batch_async = RenderManager.DrawWorld per camera): per
         frame the host computes the segment/VP setup from the camera pose, passes it by value (kernel parameters are the only
         host->device bytes) and receives the finished frame in pinned host memory (copies overlapped with the next frames' kernels;
         two pinned destinations, the host waits for step k - 1 while step k renders; --e2e-sync: one synchronous call per step).
         "d2h_ceiling" is a probe of the box: every rank copying framebuffer-sized pinned blocks at the same time, nothing else running.
roofline Phase-1 kernel (dominant): algorithmic bytes of SURVEY.md §8(d) per launch / launch duration against the measured
         HBM copy bandwidth of MEASURED_PEAKS.json. Launches of different views overlap, so the duration used is the timed
         region's wall time per frame times Phase 1's share of the kernel time; the share comes from the "exclusive" pass, which
         repeats the launches with one view in flight (each launch alone on the GPU, CUDA events around every launch).
cpu_baseline / --impl reference: the reference's own CPU code (oracle/_ref: its C# translated to C++, see oracle/ref.py) on all
         host threads; the hand restatement ("port") only when that library is missing.
N > 1    --mode views (default, configs 1-3, 5): views are sharded (each rank renders the whole path for its own share of a global
         batch of N x views), the world is built on rank 0, broadcast once over NCCL and replicated; no collective on the data path
         ("weak"). --mode rays (default for config 4): every view's rays are cut into N flat-ray ranges; each rank renders its range
         and stores the pixels it feeds straight into a ring of framebuffers on rank 0 over NVLink peer memory, ordered by
         device-side flags (cvx_draw_sharded); total work is fixed ("strong"). The default line at N > 1 also carries a short
         "rays_sharded" measurement of that mode on the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the tree it runs from may be read-only: bench.py leaves nothing in it

MILL = os.path.join(ROOT, "tests", "data", "mill.obj")
FRAMES_PER_STEP = 60
METRIC = "frames/sec @4K, mill 1024^3, BenchmarkPath 60 poses"
L2_FLUSH_BYTES = 256 << 20
DUMP_BYTES = 48 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=[1, 2, 3, 4, 5], help="BASELINE.json config (1 = the headline workload)")
    ap.add_argument("--mode", default="auto", choices=["auto", "views", "rays"], help="N > 1: shard views (weak) or the rays of every view (strong)")
    ap.add_argument("--res", default=None, help="WxH; default: the config's resolution (config 1: 3840x2160)")
    ap.add_argument("--maxdim", type=int, default=1024)
    ap.add_argument("--group", type=int, default=0, help="Phase-1 lanes per ray (0 = library default)")
    ap.add_argument("--inflight", type=int, default=6, help="views in flight per cvx_draw_batch (1..16)")
    ap.add_argument("--inflight-e2e", type=int, default=6, help="views in flight for the e2e leg (frames leave through the library's framebuffer pool: a slot does not wait for its copy)")
    ap.add_argument("--ring-slots", type=int, default=8, help="framebuffers of the gather ring (--mode rays)")
    ap.add_argument("--shard-chunk", type=int, default=512, help="--mode rays: rays are dealt to the ranks in chunks of this many (power of two)")
    ap.add_argument("--e2e-sync", action="store_true", help="e2e leg through the synchronous cvx_draw_world_batch (one call per step, returns when its frames are on the host) instead of double-buffered asynchronous batches")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-1080p", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip at_inflight, d2h_ceiling and rays_sharded (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write the frames of the last step to DIR/frames.npy (views mode, rank 0): float64 pixel "
                         "values (the packed 32-bit colours, exact) of every view at a fixed seeded sample of pixel positions, "
                         f"at most {DUMP_BYTES >> 20} MiB; the inputs are the same from run to run, so two builds compare output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.res is None:
        a.res = {1: "3840x2160", 2: "1920x1080", 3: "3840x2160", 4: "7680x4320", 5: "1280x720"}[a.config]
    if a.mode == "auto":
        a.mode = "rays" if a.config == 4 else "views"
    if a.dump_outputs and (a.mode != "views" or a.impl != "b200"):
        ap.error("--dump-outputs writes the frames of the GPU views path (--impl b200, --mode views)")
    return a


def workload_name(maxdim, W, H):
    return (f"datasets/mill.obj voxelized to {maxdim}^3 (+5 LODs), {W}x{H}, {FRAMES_PER_STEP}-pose BenchmarkPath.anim camera path, "
            "FOV 85, near 0.05, far 2*maxdim, lodError 1")


def ground_height(world, x, z):
    """worldMax of LOD-0 column (x, z): uint16 at byte 8 of its 12-byte RLEColumn header (World.cs:163-168)."""
    hdr = np.asarray(world.blobs[0])[: 12 * world.column_counts[0]].view(np.uint32).reshape(-1, 3)
    return int(hdr[int(x) * world.dims[2] + int(z), 2] & 0xFFFF)


def make_workload(cv, a, build_world=True):
    """(world or None, poses, name, metric) of a BASELINE config; worlds of configs 2-5 come from the library's seeded generators."""
    W, H = [int(x) for x in a.res.split("x")]
    if a.config == 1:
        world = cv.World.from_obj(MILL, a.maxdim) if build_world else None
        dims = world.dims if world else (a.maxdim,) * 3
        poses = cv.benchmark_path(dims, FRAMES_PER_STEP, far_clip=2.0 * max(dims))
        return world, poses, workload_name(a.maxdim, W, H), METRIC
    if a.config in (2, 3, 5):
        world = cv.World.synthetic(0, (2048, 2048, 2048), seed=1234)   # poses of 3 and 5 need the ground height: always built
        if a.config == 2:
            poses = [cv.CameraPose.from_euler((1024.0, 1700.0, 1024.0), (60.0, 30.0 + 22.5 * i, 0.0), far_clip=4096.0) for i in range(16)]
            name = f"fBm terrain 2048^3 (seed 1234), {W}x{H}, camera (1024,1700,1024) pitch 60 down, 16 yaws, vanishing point on screen (4 segments)"
        elif a.config == 3:
            h = ground_height(world, 1024, 1024)
            poses = [cv.CameraPose.from_euler((1024.5, h + 40.0, 1024.5), (pitch, 30.0 + 45.0 * i, 0.0), far_clip=4096.0) for pitch in (3.0, 0.0) for i in range(8)]
            name = f"fBm terrain 2048^3 (seed 1234), {W}x{H}, camera 40 above the ground, pitch 3 and pitch 0 (LimitRotationHorizon), 8 yaws each (clamped segments)"
        else:
            rng = np.random.default_rng(99)
            poses = []
            for _ in range(256):
                x, z = rng.uniform(0, 2048, 2)
                hh = ground_height(world, min(2047, x), min(2047, z))
                y = rng.uniform(hh + 20.0, max(hh + 21.0, 1900.0))
                poses.append(cv.CameraPose.from_euler((float(x), float(y), float(z)), (float(rng.uniform(-30, 80)), float(rng.uniform(0, 360)), 0.0), far_clip=4096.0))
            name = f"256 cameras (seed 99) at {W}x{H} over the fBm terrain 2048^3, y in [ground+20, 1900], pitch in [-30, 80], no roll"
        return world, poses, name, f"frames/sec, BASELINE config {a.config}"
    world = cv.World.synthetic(1, (4096, 1024, 4096), seed=7) if build_world else None
    poses = [cv.CameraPose.from_euler((2048.5, 700.5, 2048.5), (35.0, 20.0, 0.0), far_clip=8192.0),
             cv.CameraPose.from_euler((500.5, 400.5, 700.5), (12.0, 50.0, 0.0), far_clip=8192.0),
             cv.CameraPose.from_euler((3000.5, 950.5, 1000.5), (70.0, 200.0, 10.0), far_clip=8192.0),
             cv.CameraPose.from_euler((2048.5, 300.5, 100.5), (-10.0, 0.0, 0.0), far_clip=8192.0)]
    return world, poses, f"boxes/pipes/slabs 4096x1024x4096 (seed 7), {W}x{H}, 4 views, far 8192", "frames/sec, BASELINE config 4"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1 and len(r) >= 9] or [r for _, r in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = [float(r[1]) for r in rows]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][2]), "power_w_max": max(float(r[3]) for r in rows),
                "samples": len(rows), "reasons": reasons}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(W):
    """DRAM bytes of ONE Phase-1 launch from the committed ncu --set full capture (which pose: see the note), if one exists."""
    p = os.path.join(ROOT, "profiles", "phase1_traffic.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if str(W) in d:
            return {"dram_bytes": d[str(W)], "note": d.get("_source")}
    return None


def ncu_instructions(W):
    """Mean warp instructions per Phase-1 launch over the 60 poses, from the committed ncu pass (profiles/phase1_inst.json)."""
    p = os.path.join(ROOT, "profiles", "phase1_inst.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if str(W) in d:
            return {"mean": d[str(W)], "commit": d.get("_source")}
    return None


def phase1_bytes(c):
    """Phase-1 share of the algorithmic bytes (SURVEY.md §8(d)): headers, runs, colour gather, raybuffer writes."""
    return 12 * c["dda_steps"] + 4 * c["runs_visited"] + 4 * c["px_voxel"] + 4 * (c["px_voxel"] + c["px_sky"])


# ---------------------------------------------------------------------------------------------------------------------
def parse_obj_soup(path):
    """ObjModel.Import (ObjModel.cs:10-167) for `v x y z [r g b]` / `f a b c` files: the triangle soup it builds (one vertex per
    face corner, indices 0..n-1), colours through Unity's Color -> Color32 rounding. Pure Python: the CPU arm must not need the product."""
    vs, cs, tri = [], [], []
    with open(path) as f:
        for line in f:
            if line.startswith("v "):
                q = line.split()
                vs.append([float(q[1]), float(q[2]), float(q[3])])
                cs.append([float(q[4]), float(q[5]), float(q[6])] if len(q) > 6 else [1.0, 1.0, 1.0])
            elif line.startswith("f "):
                tri.append([int(x.split("/")[0]) - 1 for x in line.split()[1:4]])
    vs, cs, tri = np.array(vs, dtype=np.float32), np.array(cs, dtype=np.float32), np.array(tri).ravel()
    col = np.rint(np.clip(cs, 0, 1) * np.float32(255)).astype(np.uint8)
    col = np.concatenate([col, np.full((len(col), 1), 255, np.uint8)], 1)
    return vs[tri], col[tri]


class CpuPath:
    """The reference's CPU implementation of the path, for `--impl reference` and the cpu_baseline leg.
    kind "reference": oracle/_ref — the reference's own C# (voxelizer, RLE builder, DownSample, segment setup, DrawSegments + the four
        jobs of DrawSegmentRayJob) translated to C++ and compiled (oracle/ref.py; no C# toolchain exists here), jobs spread over
        all host threads with a shared batch counter like Unity's IJobParallelFor;
    kind "port": oracle/cpuvox_oracle.cpp (hand restatement), only when the prebuilt oracle/_ref library is missing.
    Phase 2 is a GPU shader in the reference (RayBufferBlit.shader); on the CPU arm it is the oracle's per-pixel restatement
    (threaded), so that a CPU "frame" is the same product as a GPU frame. Camera path, LOD distances and LimitRotationHorizon
    (UnityEngine / MonoBehaviour code) come from the oracle library's restatements.
    Config 1 needs no product code at all (mill.obj parsed here, world built by the reference's own builder); the synthetic worlds
    and camera sets of configs 2-5 have no reference analogue and come from the library's host-side generators (no GPU involved)."""

    def __init__(self, a, W, H, workload=None):
        from oracle import oracle as orc
        from oracle import ref
        self.orc, self.W, self.H = orc, W, H
        self.kind = "reference" if ref.build() else "port"
        self.ref = ref if self.kind == "reference" else None
        self.threads = orc.hardware_threads()
        if a.config == 1:
            P, C = parse_obj_soup(MILL)
            if self.kind == "reference":
                dims, blobs, ccs, _ = ref.build_world_from_mesh(P, C, np.arange(P.shape[0]), a.maxdim)   # flip X only: the UI default
            else:
                import cpuvox_b200 as cv  # fallback only: the oracle has no world builder of its own
                w = cv.World.from_obj(MILL, a.maxdim)
                dims, blobs, ccs = w.dims, w.blobs, w.column_counts
            cams = [orc.benchmark_pose(1.15 * i / (FRAMES_PER_STEP - 1), dims) + (2.0 * max(dims),) for i in range(FRAMES_PER_STEP)]  # clip length 1.15
        else:
            if workload is None:
                import cpuvox_b200 as cv
                workload = make_workload(cv, a)
            world, poses = workload[0], workload[1]
            dims, blobs, ccs = world.dims, world.blobs, world.column_counts
            cams = [(p.position, p.rotation, p.far_clip) for p in poses]
        self.dims = dims
        if self.kind == "reference":
            self.world = ref.RefWorld(dims, blobs, ccs)
            self.buffers = ref.alloc_raybuffers(W, H)
        else:
            self.buffers = (np.zeros((W + 2 * H, H), dtype=np.uint32), np.zeros((2 * W + H, W), dtype=np.uint32))
        self.oworld = orc.OracleWorld(dims, blobs, ccs)
        lods = orc.setup_lods(max(dims), W, H)
        self.setups = []
        for pos, rot, far in cams:
            if self.kind == "reference":
                rot = orc.limit_rotation_horizon(pos, rot)
                self.setups.append(ref.frame_setup(pos, rot, W, H, lods, dims[1], far=far))
            else:
                self.setups.append(orc.frame_setup(pos, rot, W, H, lods, dims[1], far=far))
        self.frame = np.zeros((H, W), dtype=np.uint32)

    def render(self, i):
        s = self.setups[i]
        if self.kind == "reference":
            td, lr = self.ref.render_raybuffers(self.world, s, self.W, self.H, threads=0, buffers=self.buffers)
            s = self.orc.copy_setup(s)
        else:
            td, lr, _ = self.orc.render_raybuffers(self.oworld, s, self.W, self.H, threads=0, td=self.buffers[0], lr=self.buffers[1])
        self.orc.blit(s, self.W, self.H, td, lr, threads=0, frame=self.frame)

    def describe(self):
        what = ("reference C# translated to C++ (oracle/_ref: cs2cpp.py, g++ -O2 -ffp-contract=off; not .NET, not Burst)" if self.kind == "reference"
                else "hand C++ restatement (oracle/cpuvox_oracle.cpp)")
        return f"Phase 1 = {what}, Phase 2 = per-pixel restatement of the blit shader; {self.threads} host threads"


def dump_frames(directory, cv, N, rm, setups, W, H):
    """--dump-outputs, right after the timed steps: every view's frame of the step, as cvx_draw_batch hands them to a caller.
    The device-only timed steps keep only the last view's frame readable, so the same batch is drawn once more into host memory;
    its last frame must equal the one the timed steps left behind. A 4K step is 2 GB of frames: a seeded sample of pixel
    positions (the same for every view) is written as float64, which holds the 32-bit colours exactly."""
    last = rm.read_frame()
    frames = cv.alloc_pinned((len(setups), H, W))
    try:
        rm.draw_batch(setups, frames)
        if not np.array_equal(frames[-1], last):
            raise SystemExit("--dump-outputs: drawing the step again gave a different last frame")
        per_view = min(W * H, DUMP_BYTES // (8 * len(setups)))
        idx = np.sort(np.random.default_rng(0).choice(W * H, per_view, replace=False))
        out = frames.reshape(len(setups), -1)[:, idx].astype(np.float64)
    finally:
        N.lib.cvx_free_pinned(frames.ctypes.data)
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "frames.npy"), out)


def config_block(a, name, W, H, frames_per_step, extra=None):
    c = {"workload": name, "baseline_config": a.config, "resolution": [W, H], "frames_per_step": frames_per_step}
    if extra:
        c.update(extra)
    return c


def run_reference(a, rank, world_size):
    """--impl reference: the reference's own CPU implementation on all host threads, the same views per step as the repo arm."""
    if rank != 0:
        return
    W, H = [int(x) for x in a.res.split("x")]
    workload = None
    if a.config != 1:
        import cpuvox_b200 as cv   # host-side generators of the synthetic configs only
        workload = make_workload(cv, a)
        name, metric = workload[2], workload[3]
    else:
        name, metric = workload_name(a.maxdim, W, H), METRIC
    cpu = CpuPath(a, W, H, workload)
    n = len(cpu.setups)

    def step():
        for i in range(n):
            cpu.render(i)

    for _ in range(a.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        step()
    dt = time.perf_counter() - t0
    fps = n * a.steps / dt
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": fps, "unit": "frames/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": 1000.0 * dt / a.steps, "higher_is_better": True, "scaling": "strong" if a.mode == "rays" else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "datasets/mill.obj (reference dataset) voxelized in-process, fixed 60-pose camera path" if a.config == 1 else "synthetic (seeded generators)",
        "config": config_block(a, name, W, H, n),
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cpu.threads, "kind": cpu.kind,
                         "sample": f"all {n} views of the workload per step; " + cpu.describe()},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
def time_path(torch, dist, rm, setups, steps, warmup, device, flush, world_size, profile=True):
    """W warm-up steps, then exactly `steps` steps between barrier+synchronize pairs; CUDA events on the launching stream."""
    def one_step():
        flush.zero_()            # L2 flush between steps: 256 MiB written on the same stream
        rm.draw_batch(setups)    # device only: enqueues all views, joined back into this stream

    for _ in range(warmup):
        one_step()
    torch.cuda.synchronize(device)
    if world_size > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    if profile:
        rm.profile_begin(steps * len(setups))
    launches0 = rm.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        one_step()
    e1.record()
    torch.cuda.synchronize(device)
    t1 = time.perf_counter()
    if world_size > 1:
        dist.barrier()
    torch.cuda.synchronize(device)
    ms = e0.elapsed_time(e1)
    p1 = p2 = 0.0
    n = 0
    if profile:
        p1, p2, n = rm.profile_end()
    return ms, p1, p2, n, rm.launch_count() - launches0, (t0, t1)


def time_e2e(torch, dist, cv, rm, poses, steps, warmup, device, world_size, pinned, sync_calls=False):
    """Public-API path with host buffers: host setup per frame, frames delivered to pinned host memory. `pinned` holds two destinations:
    step k goes into pinned[k % 2] through cvx_draw_world_batch_async and the host waits for step k - 1 while step k renders (a consumer
    that double-buffers its frames; every frame's copy lies inside the timed region, which ends when the last step's frames have landed).
    sync_calls: the synchronous cvx_draw_world_batch per step instead (returns when the step's frames are on the host)."""
    def run(n):
        # RenderManager.DrawWorld per camera: the host part (LimitRotationHorizon, vanishing point, segments, CameraData) is computed
        # inside the call from the poses; kernels + device->host frame copies
        prev = None
        batch = rm.pose_batch(poses)    # marshalled once (the poses of a step are the same every step)
        for k in range(n):
            if sync_calls:
                rm.draw_world_batch(poses, pinned[k % 2])
                continue
            cur = rm.draw_world_batch_async(batch, pinned[k % 2])
            if prev is not None:
                rm.batch_wait(prev)      # the frames of step k - 1 are on the host; its buffer is free for step k + 1
            prev = cur
        if prev is not None:
            rm.batch_wait(prev)

    run(max(2, warmup // 2))
    torch.cuda.synchronize(device)
    if world_size > 1:
        dist.barrier()
    t0 = time.perf_counter()
    run(steps)
    torch.cuda.synchronize(device)
    dt = time.perf_counter() - t0
    if world_size > 1:
        dist.barrier()
    return dt


def d2h_ceiling(torch, dist, device, world_size, bytes_per_copy, blocks, copies=None):
    """Probe of the box, not of the library: every rank copies framebuffer-sized blocks device -> pinned host memory at the same
    time with nothing else running (torch tensors, 4 streams per rank), into as many distinct host blocks as a step of the e2e leg
    delivers (a few small destinations would stay in the host's last-level cache and overstate what streaming frames can reach).
    The e2e number cannot exceed job GB/s / frame bytes."""
    copies = copies or 2 * blocks
    src = torch.empty(bytes_per_copy, dtype=torch.uint8, device=f"cuda:{device}")
    dst = torch.empty((blocks, bytes_per_copy), dtype=torch.uint8, pin_memory=True)
    streams = [torch.cuda.Stream(device) for _ in range(4)]

    def run(n):
        for i in range(n):
            with torch.cuda.stream(streams[i % 4]):
                dst[i % blocks].copy_(src, non_blocking=True)
        torch.cuda.synchronize(device)

    run(blocks)
    if world_size > 1:
        dist.barrier()
    t0 = time.perf_counter()
    run(copies)
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device=f"cuda:{device}")
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    worst = float(t.item())
    return {"job_gbs": world_size * copies * bytes_per_copy / worst / 1e9, "slowest_rank_gbs": copies * bytes_per_copy / worst / 1e9,
            "block_bytes": bytes_per_copy, "host_blocks": blocks,
            "note": "all ranks copying device -> pinned host at once, 4 streams each, nothing else running"}


def time_rays(torch, dist, srm, poses, steps, warmup, device, world_size, dst=None, chunk=512):
    """--mode rays: a step = draw_views_sharded over the views (every view's rays cut over the ranks, frames gathered in the ring on
    rank 0). Host clock between synchronize+barrier pairs: all device work of the steps lies inside; max over ranks."""
    for _ in range(warmup):
        srm.draw_views_sharded(poses, dst, chunk=chunk)
    torch.cuda.synchronize(device)
    if world_size > 1:
        dist.barrier()
    launches0 = srm.rm.launch_count()
    t0 = time.perf_counter()
    for _ in range(steps):
        srm.draw_views_sharded(poses, dst, barrier=False, sync=False, chunk=chunk)   # the ring's device-side flags order the steps: no drain between them
    srm.sync_views(barrier=False)
    torch.cuda.synchronize(device)
    dt = time.perf_counter() - t0
    if world_size > 1:
        dist.barrier()
    t = torch.tensor([dt], dtype=torch.float64, device=f"cuda:{device}")
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), srm.rm.launch_count() - launches0, (t0, t0 + dt)


def cpu_baseline_leg(a, W, H, workload, frames_per_step):
    cpu = CpuPath(a, W, H, workload)   # the checker as the timed CPU arm (oracle/_ref), never on the product path
    t0 = time.perf_counter()
    done = 0
    for _ in range(8):
        for i in range(len(cpu.setups)):
            cpu.render(i)
            done += 1
            if time.perf_counter() - t0 > 25.0:
                break
        if time.perf_counter() - t0 > 12.0:
            break
    dt = time.perf_counter() - t0
    return {"value": done / dt, "unit": "frames/s", "cores": cpu.threads, "kind": cpu.kind,
            "sample": f"{done} frames ({'whole passes over' if done % len(cpu.setups) == 0 else 'the first views of'} the same {frames_per_step}-view workload at {W}x{H}); " + cpu.describe()}


def run_rays(a, rank, local_rank, world_size, torch, dist, cv, N, world, poses, name, metric):
    """--mode rays: every view's rays sharded over the ranks, frame ring on rank 0 (cvx_draw_sharded / cvx_ring_consume)."""
    device = local_rank
    W, H = [int(x) for x in a.res.split("x")]
    srm = cv.ShardedRenderManager(device, rank, world_size, gather="ring", ring_slots=a.ring_slots)
    srm.upload_world(world)
    srm.rm.set_group_size(a.group)
    srm.rm.set_frames_in_flight(a.inflight)
    srm.set_resolution(W, H)
    per = None
    if rank == 0:   # work counters of the whole views (single-GPU draws), for the algorithmic bytes
        rm = srm.rm
        rm.set_counters(True)
        rm.counters()
        per = []
        for p in poses:
            rm.draw_setup(rm.make_setup(p))
            per.append(rm.counters())
        rm.set_counters(False)
        rm.sync()
    sampler = ClockSampler(device) if rank == 0 else None
    dt, launches, span = time_rays(torch, dist, srm, poses, a.steps, a.warmup, device, world_size, chunk=a.shard_chunk)
    clocks = sampler.stop(*span) if sampler else None
    pinned = cv.alloc_pinned((len(poses), H, W)) if rank == 0 else None
    e2e_dt, _, _ = time_rays(torch, dist, srm, poses, max(2, a.steps // 2), 1, device, world_size, dst=pinned, chunk=a.shard_chunk)
    e2e_steps = max(2, a.steps // 2)
    if rank == 0:
        frames = len(poses) * a.steps
        fps = frames / dt
        peak, peak_src = measured_hbm_peak()
        p1_bytes = sum(phase1_bytes(c) for c in per) / len(per)
        frame_bytes = sum(cv.algorithmic_bytes(c, W, H) for c in per) / len(per)
        line = {
            "metric": metric, "value": fps, "unit": "frames/s", "n_gpus": world_size, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1000.0 * dt / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic (seeded generators)" if a.config != 1 else "datasets/mill.obj (reference dataset) voxelized in-process, fixed 60-pose camera path",
            "config": config_block(a, name, W, H, len(poses), {
                "parallelism": f"rays of every view sharded over {world_size} GPU(s); pixels stored into a ring of {a.ring_slots} framebuffers on rank 0 over NVLink "
                               "peer memory, device-side flags between ranks, no host barrier or collective between views; world broadcast once and replicated",
                "l2": "inputs larger than L2: the raybuffers + frame of one view are 1.0 GB at 8K (no flush)" if W * H > 20e6 else "no flush: successive views differ",
                "frames_in_flight": a.inflight, "ring_slots": a.ring_slots, "shard_chunk_rays": a.shard_chunk,
                "timing": "host clock between synchronize+barrier pairs around the steps (all device work inside), max over ranks"}),
            "runs_per_s": sum(c["runs_visited"] for c in per) / len(per) * fps,
            "ms_per_frame": {"total": 1000.0 * dt / frames},
            "roofline": {"bound": "hbm", "kernel": "phase1_kernel", "achieved": p1_bytes * fps / 1e9, "peak": peak * world_size, "unit": "GB/s",
                         "frac": p1_bytes * fps / 1e9 / (peak * world_size), "peak_source": peak_src + f" x {world_size} GPUs", "algorithmic_bytes_per_launch": p1_bytes,
                         "traffic": None,
                         "note": "Phase-1 algorithmic bytes of the whole view x views/s (the per-rank launches overlap across views); see the views-mode line for per-launch figures",
                         "whole_frame": {"algorithmic_bytes": frame_bytes, "achieved": frame_bytes * fps / 1e9, "frac": frame_bytes * fps / 1e9 / (peak * world_size)}},
            "e2e": {"value": len(poses) * e2e_steps / e2e_dt, "unit": "frames/s", "h2d_bytes_per_step": len(poses) * __import__("ctypes").sizeof(N.FrameSetup),
                    "d2h_bytes_per_step": len(poses) * W * H * 4, "note": "frames copied from the ring to pinned host memory on rank 0 by cvx_ring_consume"},
            "gpu_launches": launches, "clocks": clocks,
        }
        if world_size == 1 and not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_leg(a, W, H, (world, poses, name, metric), len(poses))
        print(json.dumps(line), flush=True)
        N.lib.cvx_free_pinned(pinned.ctypes.data)
    srm.destroy()


def run_b200(a, rank, local_rank, world_size):
    import torch
    import torch.distributed as dist

    import cpuvox_b200 as cv
    from cpuvox_b200 import native as N

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: cpuvox_b200 has no CPU fallback (use --impl reference for the CPU baseline)")
    device = local_rank
    torch.cuda.set_device(device)
    if world_size > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{device}"))

    W, H = [int(x) for x in a.res.split("x")]
    world, poses, name, metric = make_workload(cv, a, build_world=(rank == 0))
    if world_size > 1:
        world = cv.broadcast_world(world if rank == 0 else None, src=0, device=torch.device(f"cuda:{device}"))  # once, then replicated per GPU
    if a.mode == "rays":
        run_rays(a, rank, local_rank, world_size, torch, dist, cv, N, world, poses, name, metric)
        if world_size > 1:
            dist.destroy_process_group()
        return
    nviews = len(poses)
    rm = cv.RenderManager(device)
    # one explicit stream for everything that is timed: the library's launches, the L2 flush and the torch events
    # (torch's default stream is the NULL handle, which cvx_set_stream reads as "use the context's own stream")
    stream = torch.cuda.Stream(device)
    torch.cuda.set_stream(stream)
    rm.set_stream(stream.cuda_stream)
    rm.upload_world(world)
    rm.set_group_size(a.group)
    rm.set_frames_in_flight(a.inflight)
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=f"cuda:{device}")

    def counters_for(setups):
        rm.set_counters(True)
        rm.counters()
        per = []
        for s in setups:
            rm.draw_setup(s)
            per.append(rm.counters())
        rm.set_counters(False)
        return per

    results = {}
    resolutions = [(W, H)] + ([] if a.no_1080p or a.config != 1 or (W, H) == (1920, 1080) else [(1920, 1080)])
    clocks = None
    at_inflight = {}
    for ri, (w, h) in enumerate(resolutions):
        rm.set_resolution(w, h)
        setups = [rm.make_setup(p) for p in poses]
        per = counters_for(setups)
        sampler = ClockSampler(device) if (ri == 0 and rank == 0) else None
        steps = a.steps if ri == 0 else max(2, a.steps // 2)
        ms, p1, p2, n, launches, span = time_path(torch, dist, rm, setups, steps, a.warmup, device, flush, world_size)
        if sampler:
            clocks = sampler.stop(*span)
        if ri == 0 and rank == 0 and a.dump_outputs:
            dump_frames(a.dump_outputs, cv, N, rm, setups, w, h)
        # the same launches one view at a time: exclusive kernel durations (outside the timed region, reported beside it)
        rm.set_frames_in_flight(1)
        _, x1, x2, xn, _, _ = time_path(torch, dist, rm, setups, 1, 1, device, flush, world_size)
        if ri == 0 and not a.no_extras:
            # the interactive case: one view at a time, and two (the reference's double buffering, RenderManager.cs:14,53-56)
            for k in (1, 2):
                rm.set_frames_in_flight(k)
                kms, _, _, _, _, _ = time_path(torch, dist, rm, setups, max(2, a.steps // 3), 2, device, flush, world_size, profile=False)
                t = torch.tensor([kms], dtype=torch.float64, device=f"cuda:{device}")
                if world_size > 1:
                    dist.all_reduce(t, op=dist.ReduceOp.MAX)
                at_inflight[str(k)] = {"value": nviews * max(2, a.steps // 3) * world_size / (float(t.item()) / 1000.0), "unit": "frames/s"}
        rm.set_frames_in_flight(a.inflight)
        pinned = cv.alloc_pinned((2, nviews, h, w))
        rm.set_frames_in_flight(a.inflight_e2e)   # frames leave through the framebuffer pool (cvx_draw_batch): the slots do not wait for the copies
        e2e_s = time_e2e(torch, dist, cv, rm, poses, steps, a.warmup, device, world_size, pinned, sync_calls=a.e2e_sync)
        rm.set_frames_in_flight(a.inflight)
        N.lib.cvx_free_pinned(pinned.ctypes.data)
        t = torch.tensor([ms, e2e_s * 1000.0, p1, p2, x1, x2], dtype=torch.float64, device=f"cuda:{device}")
        if world_size > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)  # max over ranks
        ms, e2e_ms, p1, p2, x1, x2 = [float(x) for x in t.cpu()]
        results[(w, h)] = dict(ms=ms, e2e_ms=e2e_ms, p1=p1, p2=p2, n=n, launches=launches, steps=steps, per=per, x1=x1, x2=x2, xn=xn)

    ceiling = None
    if not a.no_extras:
        ceiling = d2h_ceiling(torch, dist, device, world_size, W * H * 4, min(nviews, 64))

    # a short measurement of the other split on the same workload: every view's rays sharded over the ranks (frame ring)
    rays_sharded = None
    if world_size > 1 and not a.no_extras:
        rm.destroy()
        rm = None
        try:   # an extra: its failure must not cost the main line (every measurement above is already taken)
            srm = cv.ShardedRenderManager(device, rank, world_size, gather="ring", ring_slots=a.ring_slots)
            srm.upload_world(world)
            srm.rm.set_frames_in_flight(a.inflight)
            srm.set_resolution(W, H)
            sub = poses[:60]
            rdt, _, _ = time_rays(torch, dist, srm, sub, 3, 1, device, world_size, chunk=a.shard_chunk)
            rays_sharded = {"value": len(sub) * 3 / rdt, "unit": "frames/s", "views": len(sub), "scaling": "strong",
                            "note": f"{len(sub)} views of the same workload, every view's rays dealt over the {world_size} ranks in chunks of {a.shard_chunk}, frames gathered in a ring "
                                    "on rank 0 over NVLink peer memory (device-side flags, no host barrier between views); the same total work as ONE rank's share of `value`"}
            srm.destroy()
        except Exception as e:  # noqa: BLE001
            rays_sharded = {"error": str(e)[:300]}

    main = results[(W, H)]
    steps = main["steps"]
    frames = nviews * steps * world_size
    fps = frames / (main["ms"] / 1000.0)
    e2e_fps = frames / (main["e2e_ms"] / 1000.0)
    per = main["per"]
    runs_per_frame = sum(c["runs_visited"] for c in per) / len(per)
    p1_bytes = sum(phase1_bytes(c) for c in per) / len(per)             # mean algorithmic bytes per Phase-1 launch
    p1_ev = main["p1"] / max(1, main["n"])                              # mean Phase-1 launch duration by CUDA events (launches overlap)
    p2_ev = main["p2"] / max(1, main["n"])
    frame_ms = main["ms"] / (steps * nviews)                            # timed-region wall time per frame on this rank
    x1_ms, x2_ms = main["x1"] / max(1, main["xn"]), main["x2"] / max(1, main["xn"])   # one view in flight: each launch alone
    # Phase 1's share of the step: from the EXCLUSIVE durations (the overlapped event durations of the short Phase-2 launches are
    # inflated by the Phase-1 launches of the other views they share the GPU with, which would flatter Phase 1)
    share = x1_ms / (x1_ms + x2_ms) if x1_ms + x2_ms > 0 else (p1_ev / (p1_ev + p2_ev) if p1_ev + p2_ev > 0 else 1.0)
    p1_ms, p2_ms = frame_ms * share, frame_ms * (1.0 - share)           # effective duration per launch under overlap
    peak, peak_src = measured_hbm_peak()
    achieved = p1_bytes / (p1_ms * 1e-3) / 1e9 if p1_ms > 0 else 0.0
    frame_bytes = sum(cv.algorithmic_bytes(c, W, H) for c in per) / len(per)
    # what actually bounds Phase 1: issue slots (148 SMs x 4 schedulers x SM clock); instruction counts come from the committed ncu pass
    inst = ncu_instructions(W) if a.config == 1 else None
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    issue = None
    if inst and p1_ms > 0:
        slots_per_s = 148 * 4 * sm_mhz * 1e6
        issue = {"warp_instructions_per_launch": inst["mean"] if isinstance(inst, dict) else inst,
                 "source": "profiles/phase1_inst.json (refreshed by tools/gpu_round.sh): " + str(inst.get("commit")),
                 "issue_slot_utilisation": (inst["mean"] if isinstance(inst, dict) else inst) / (p1_ms * 1e-3) / slots_per_s,
                 "note": "Phase 1 is latency/issue bound (DESIGN.md §7): this, not the HBM fraction, tracks kernel quality"}
    traffic = ncu_traffic(W) if a.config == 1 else None

    if rank != 0:
        if rm:
            rm.destroy()
        if world_size > 1:
            dist.destroy_process_group()
        return

    line = {
        "metric": metric, "value": fps, "unit": "frames/s", "n_gpus": world_size, "steps": steps, "warmup": a.warmup,
        "ms_per_step": main["ms"] / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "datasets/mill.obj (reference dataset) voxelized in-process, fixed 60-pose camera path" if a.config == 1 else "synthetic (seeded generators)",
        "config": config_block(a, name, W, H, nviews * world_size, {
            "parallelism": "1 GPU" if world_size == 1 else f"views sharded over {world_size} GPUs, world broadcast once and replicated, no data-path collective",
            "l2": "flushed between steps (256 MiB device write inside the timed region); frames of one step run back to back",
            "phase1_lanes_per_ray": a.group or 32, "frames_in_flight": a.inflight, "frames_in_flight_e2e": a.inflight_e2e}),
        "runs_per_s": runs_per_frame * fps,
        "ms_per_frame": {"total": frame_ms, "phase1_kernel": p1_ms, "phase2_kernel": p2_ms,
                         "basis": "wall time of the timed region per frame, split by the kernels' share of the exclusive CUDA-event durations "
                                  f"(up to {a.inflight} views in flight, launches overlap)",
                         "event_mean_overlapped": {"phase1_kernel": p1_ev, "phase2_kernel": p2_ev},
                         "exclusive_one_view_in_flight": {"phase1_kernel": x1_ms, "phase2_kernel": x2_ms}},
        "roofline": {
            "bound": "hbm", "kernel": "phase1_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "peak_source": peak_src, "algorithmic_bytes_per_launch": p1_bytes,
            "traffic": traffic["dram_bytes"] if isinstance(traffic, dict) else traffic,
            "traffic_note": (traffic.get("note") if isinstance(traffic, dict) else None),
            "exclusive": {"launch_ms": x1_ms, "achieved": p1_bytes / (x1_ms * 1e-3) / 1e9 if x1_ms > 0 else 0.0,
                          "note": "same launches with one view in flight (each alone on the GPU), measured after the timed region"},
            "issue": issue,
            "phase2_kernel": {"algorithmic_bytes_per_launch": 8 * W * H, "exclusive_launch_ms": x2_ms,
                              "achieved": 8 * W * H / (x2_ms * 1e-3) / 1e9 if x2_ms > 0 else 0.0,
                              "frac": 8 * W * H / (x2_ms * 1e-3) / 1e9 / peak if x2_ms > 0 else 0.0,
                              "note": "8 B per screen pixel (one raybuffer read, one frame write) / CUDA-event duration of a launch alone (launch gaps included)"},
            "whole_frame": {"algorithmic_bytes": frame_bytes, "achieved": frame_bytes * fps / world_size / 1e9,
                            "frac": frame_bytes * fps / world_size / 1e9 / peak},
        },
        "e2e": {"value": e2e_fps, "unit": "frames/s",
                "h2d_bytes_per_step": nviews * world_size * __import__("ctypes").sizeof(N.FrameSetup),
                "d2h_bytes_per_step": nviews * world_size * W * H * 4,
                "call": "cvx_draw_world_batch (synchronous, one call per step)" if a.e2e_sync else
                        "cvx_draw_world_batch_async + cvx_batch_wait, two pinned destinations: step k renders while step k - 1's frames finish landing"},
        "gpu_launches": main["launches"],
        "clocks": clocks,
    }
    if at_inflight:
        at_inflight[str(a.inflight)] = {"value": fps, "unit": "frames/s"}
        line["at_inflight"] = at_inflight
        line["at_inflight"]["note"] = ("device-resident frames/s with that many views in flight; 1 = one interactive view at a time (bounded by its slowest "
                                       "ray's serial chain), 2 = the reference's double buffering (RenderManager.cs:14,53-56)")
    if ceiling:
        ceiling["frames_per_s_ceiling"] = ceiling["job_gbs"] * 1e9 / (W * H * 4)
        ceiling["e2e_fraction_of_ceiling"] = e2e_fps / ceiling["frames_per_s_ceiling"]
        line["e2e"]["d2h_ceiling"] = ceiling
    if rays_sharded:
        line["rays_sharded"] = rays_sharded
    if (1920, 1080) in results and (W, H) != (1920, 1080):
        r = results[(1920, 1080)]
        fr = nviews * r["steps"] * world_size
        line["at_1080p"] = {"value": fr / (r["ms"] / 1000.0), "unit": "frames/s", "e2e": fr / (r["e2e_ms"] / 1000.0),
                            "phase1_kernel_ms_exclusive": r["x1"] / max(1, r["xn"]), "phase2_kernel_ms_exclusive": r["x2"] / max(1, r["xn"]),
                            "runs_per_s": sum(c["runs_visited"] for c in r["per"]) / len(r["per"]) * fr / (r["ms"] / 1000.0)}

    if world_size == 1 and not a.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_leg(a, W, H, (world, poses, name, metric), nviews)
    print(json.dumps(line), flush=True)
    if rm:
        rm.destroy()
    if world_size > 1:
        dist.destroy_process_group()


def main():
    a = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    if a.impl == "reference":
        run_reference(a, rank, world_size)
        return
    if world_size != a.gpus and world_size == 1 and a.gpus > 1:
        raise SystemExit(f"--gpus {a.gpus} needs torchrun: python -m torch.distributed.run --nnodes=1 --nproc-per-node {a.gpus} "
                         f"--master-addr 127.0.0.1 --master-port 29511 bench.py --gpus {a.gpus} ...")
    run_b200(a, rank, local_rank, world_size)


if __name__ == "__main__":
    main()
