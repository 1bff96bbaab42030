"""Host-side mirror of the reference's managed surface for the raybuffer path, over the C ABI.

Names follow the reference: `RenderManager.set_resolution / draw_world` (Assets/Code/RenderManager.cs:94-194),
`World` with its LOD blobs (Assets/Code/World.cs), `setup_lods` / `limit_rotation_horizon`
(Assets/Code/UnityManager.cs:193-201,417-458), the `BenchmarkPath.anim` sampler (UnityManager.cs:86-87).
All arithmetic happens inside libcpuvox_b200.so (C++ host helpers + CUDA kernels); this file only moves
buffers. A C# host does the same through P/Invoke (INTEGRATION.md, csharp/).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import native as N
from .native import LOD_LEVELS, CvxError, FrameSetup, Pose, check, lib

SKYBOX_ARGB = 0x191919FF  # ColorARGB32(25,25,25), DrawSegmentRayJob.cs:702


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


@dataclass
class World:
    """LOD blobs in the reference's WorldAllocator layout (World.cs:285-313)."""

    dims: Tuple[int, int, int]
    blobs: List[np.ndarray]          # uint8, one per LOD
    column_counts: List[int]
    voxel_counts: List[int] = field(default_factory=list)

    @property
    def max_dimension(self) -> int:
        return max(self.dims)

    @staticmethod
    def _from_builder(b, lods: int) -> "World":
        try:
            dims = (C.c_int32 * 3)()
            check(lib.cvx_builder_dims(b, C.byref(dims)))
            blobs, cols, vox = [], [], []
            for lod in range(lods):
                if min(dims[0] >> lod, dims[1] >> lod, dims[2] >> lod) < 1:
                    break
                p, nbytes, cc, vc = C.c_void_p(), C.c_int64(), C.c_int32(), C.c_int64()
                check(lib.cvx_builder_lod(b, lod, C.byref(p), C.byref(nbytes), C.byref(cc), C.byref(vc)))
                blobs.append(np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(nbytes.value,)).copy())
                cols.append(cc.value)
                vox.append(vc.value)
            return World((dims[0], dims[1], dims[2]), blobs, cols, vox)
        finally:
            lib.cvx_builder_free(b)

    @staticmethod
    def from_obj(path: str, max_dimension: int = 1024, flips: Sequence[bool] = (True, False, False),
                 swap_yz: bool = False, lods: int = LOD_LEVELS, threads: int = 0) -> "World":
        """ObjModel.Import -> SimpleMesh.Rescale -> WorldBuilder -> ToLOD0World -> DownSample (UnityManager.cs:297-331)."""
        pos, col, n = C.c_void_p(), C.c_void_p(), C.c_int32()
        check(lib.cvx_obj_parse(path.encode(), int(swap_yz), C.byref(pos), C.byref(col), C.byref(n)))
        try:
            fl = (C.c_int32 * 3)(*[int(bool(f)) for f in flips])
            b = C.c_void_p()
            check(lib.cvx_builder_from_mesh(pos, col, n.value, max_dimension, C.byref(fl), threads, C.byref(b)))
        finally:
            lib.cvx_host_free(pos)
            lib.cvx_host_free(col)
        return World._from_builder(b, lods)

    @staticmethod
    def from_mesh(positions: np.ndarray, colors32: np.ndarray, max_dimension: int,
                  flips: Sequence[bool] = (False, False, False), lods: int = LOD_LEVELS, threads: int = 0) -> "World":
        positions = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3)
        colors32 = np.ascontiguousarray(colors32, dtype=np.uint8).reshape(-1, 4)
        fl = (C.c_int32 * 3)(*[int(bool(f)) for f in flips])
        b = C.c_void_p()
        check(lib.cvx_builder_from_mesh(_ptr(positions), _ptr(colors32), positions.shape[0], max_dimension, C.byref(fl), threads, C.byref(b)))
        return World._from_builder(b, lods)

    @staticmethod
    def synthetic(kind: int, dims: Tuple[int, int, int], seed: int, lods: int = LOD_LEVELS, threads: int = 0) -> "World":
        """kind 0: fBm heightmap shell (BASELINE config 2/3/5); kind 1: boxes/pipes/slabs (config 4)."""
        b = C.c_void_p()
        check(lib.cvx_builder_synthetic(kind, dims[0], dims[1], dims[2], seed, threads, C.byref(b)))
        return World._from_builder(b, lods)

    def save(self, path: str) -> None:
        """WorldSaveFile.Serialize (WorldSaveFile.cs:8-55)."""
        dims = (C.c_int32 * 3)(*self.dims)
        n = len(self.blobs)
        ptrs = (C.c_void_p * n)(*[b.ctypes.data for b in self.blobs])
        sizes = (C.c_int64 * n)(*[b.nbytes for b in self.blobs])
        check(lib.cvx_world_file_write(path.encode(), C.byref(dims), n, ptrs, sizes))

    @staticmethod
    def load(path: str) -> "World":
        """WorldSaveFile.Deserialize (WorldSaveFile.cs:57-94); column counts follow World.ColumnCount (World.cs:17)."""
        dims, n = (C.c_int32 * 3)(), C.c_int32()
        ptrs, sizes = (C.c_void_p * LOD_LEVELS)(), (C.c_int64 * LOD_LEVELS)()
        check(lib.cvx_world_file_read(path.encode(), C.byref(dims), C.byref(n), C.byref(ptrs), C.byref(sizes)))
        blobs, cols = [], []
        for i in range(n.value):
            blobs.append(np.ctypeslib.as_array(C.cast(ptrs[i], C.POINTER(C.c_uint8)), shape=(sizes[i],)).copy())
            lib.cvx_host_free(ptrs[i])
            cols.append((dims[0] * dims[2]) // ((i + 1) * (i + 1)))
        return World((dims[0], dims[1], dims[2]), blobs, cols, [])


@dataclass
class CameraPose:
    """What RenderManager.DrawWorld reads from UnityEngine.Camera / Transform."""

    position: Tuple[float, float, float]
    rotation: Tuple[float, float, float, float]  # quaternion x, y, z, w
    fov_y_degrees: float = 85.0   # Assets/Scenes/SampleScene.unity:178
    near_clip: float = 0.05       # SampleScene.unity:176
    far_clip: float = 2048.0      # UnityManager.SetupLods: 2 * world max dimension

    @staticmethod
    def from_euler(position, euler_deg, **kw) -> "CameraPose":
        q = (C.c_float * 4)()
        lib.cvx_host_quat_euler(euler_deg[0], euler_deg[1], euler_deg[2], C.byref(q))
        return CameraPose(tuple(position), tuple(q), **kw)

    def to_native(self, width: int, height: int) -> Pose:
        p = Pose()
        p.position[:] = self.position
        p.rotation[:] = self.rotation
        p.fov_y_degrees, p.near_clip, p.far_clip = self.fov_y_degrees, self.near_clip, self.far_clip
        p.pixel_width, p.pixel_height = width, height
        return p


def setup_lods(world_max_dimension: int, res_x: int, res_y: int, fov_y_degrees: float = 85.0, lod_error: float = 1.0) -> np.ndarray:
    """UnityManager.SetupLods (UnityManager.cs:417-458)."""
    out = (C.c_float * LOD_LEVELS)()
    lib.cvx_host_setup_lods(world_max_dimension, res_x, res_y, fov_y_degrees, lod_error, C.byref(out))
    return np.array(out[:], dtype=np.float32)


def benchmark_pose(clip_time: float, world_dims: Sequence[int], **kw) -> CameraPose:
    """BenchmarkPath.SampleAnimation(clip_time) * world dimensions (UnityManager.cs:86-87)."""
    p = Pose()
    dims = (C.c_int32 * 3)(*world_dims)
    lib.cvx_host_benchmark_pose(clip_time, C.byref(dims), C.byref(p))
    return CameraPose(tuple(p.position), tuple(p.rotation), **kw)


def benchmark_length() -> float:
    return float(lib.cvx_host_benchmark_length())


def benchmark_path(world_dims: Sequence[int], frames: int = 60, **kw) -> List[CameraPose]:
    """BASELINE config 1: the clip sampled at `frames` evenly spaced times."""
    length = benchmark_length()
    return [benchmark_pose(length * i / (frames - 1), world_dims, **kw) for i in range(frames)]


def frame_setup(pose: CameraPose, width: int, height: int, lod_distances: np.ndarray, world_dim_y: int,
                limit_horizon: bool = True) -> FrameSetup:
    """LimitRotationHorizon + RenderManager.DrawWorld up to the DrawSegments call (RenderManager.cs:119-152)."""
    p = pose.to_native(width, height)
    if limit_horizon:
        lib.cvx_host_limit_rotation_horizon(C.byref(p))
    lods = (C.c_float * LOD_LEVELS)(*[float(x) for x in lod_distances])
    out = FrameSetup()
    check(lib.cvx_host_frame_setup(C.byref(p), C.byref(lods), world_dim_y, C.byref(out)))
    return out


# cvx_ray / cvx_ray_hit as numpy records (include/cpuvox_b200.h)
RAY_DTYPE = np.dtype([("origin", "<f4", 3), ("max_distance", "<f4"), ("direction", "<f4", 3), ("reserved", "<i4")])
RAY_HIT_DTYPE = np.dtype([("hit", "<i4"), ("face", "<i4"), ("cell", "<i4", 3), ("distance", "<f4"), ("color", "<u4"), ("steps", "<i4")])


def make_rays(origins, directions, max_distance=np.inf) -> np.ndarray:
    """Pack origins (n, 3), directions (n, 3) and max_distance (scalar or (n,)) into a cvx_ray array."""
    origins = np.asarray(origins, dtype=np.float32).reshape(-1, 3)
    directions = np.asarray(directions, dtype=np.float32).reshape(-1, 3)
    if origins.shape != directions.shape:
        raise ValueError(f"origins {origins.shape} and directions {directions.shape} differ")
    rays = np.zeros(origins.shape[0], dtype=RAY_DTYPE)
    rays["origin"] = origins
    rays["direction"] = directions
    rays["max_distance"] = max_distance
    return rays


# cvx_box as a numpy record (include/cpuvox_b200.h); cvx_sweep returns RAY_HIT_DTYPE records
BOX_DTYPE = np.dtype([("center", "<f4", 3), ("max_distance", "<f4"), ("direction", "<f4", 3), ("reserved0", "<i4"),
                      ("half_extent", "<f4", 3), ("reserved1", "<i4")])


def make_boxes(centers, half_extents, directions, max_distance=np.inf) -> np.ndarray:
    """Pack centers (n, 3), half_extents ((n, 3) or (3,)), directions (n, 3) and max_distance (scalar or (n,)) into a cvx_box array."""
    centers = np.asarray(centers, dtype=np.float32).reshape(-1, 3)
    directions = np.asarray(directions, dtype=np.float32).reshape(-1, 3)
    if centers.shape != directions.shape:
        raise ValueError(f"centers {centers.shape} and directions {directions.shape} differ")
    boxes = np.zeros(centers.shape[0], dtype=BOX_DTYPE)
    boxes["center"] = centers
    boxes["half_extent"] = np.asarray(half_extents, dtype=np.float32)
    boxes["direction"] = directions
    boxes["max_distance"] = max_distance
    return boxes


def screen_ray(pose: CameraPose, px: float, py: float, width: int, height: int) -> Tuple[np.ndarray, np.ndarray]:
    """Camera.ScreenPointToRay (cvx_host_screen_ray): pixel (px, py) in Unity screen space (bottom-left origin) of a width x height
    camera; returns (origin on the near plane, normalised direction), float32 (3,) each."""
    p = pose.to_native(width, height)
    o, d = (C.c_float * 3)(), (C.c_float * 3)()
    lib.cvx_host_screen_ray(C.byref(p), px, py, C.byref(o), C.byref(d))
    return np.array(o[:], dtype=np.float32), np.array(d[:], dtype=np.float32)


class RenderManager:
    """RenderManager (Assets/Code/RenderManager.cs) with its Phase-1 jobs and Phase-2 blit on the GPU."""

    def __init__(self, device: int = 0, counters: bool = False):
        self._ctx = C.c_void_p()
        cfg = N.Config(device, N.FLAG_COUNTERS if counters else 0)
        check(lib.cvx_create(C.byref(cfg), C.byref(self._ctx)))
        self.width = self.height = 0
        self.world: Optional[World] = None
        self.lod_distances: Optional[np.ndarray] = None
        self.fov_y_degrees = 85.0
        self.lod_error = 1.0

    # -- lifetime ---------------------------------------------------------------------------------
    def destroy(self):  # RenderManager.Destroy, RenderManager.cs:43-51
        if self._ctx:
            lib.cvx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass

    def _ck(self, code):
        return check(code, self._ctx)

    # -- world ------------------------------------------------------------------------------------
    def upload_world(self, world: World):
        self._ck(lib.cvx_world_free(self._ctx))
        for lod, blob in enumerate(world.blobs):
            self._ck(lib.cvx_world_upload(self._ctx, lod, world.dims[0], world.dims[1], world.dims[2], _ptr(blob), blob.nbytes, world.column_counts[lod]))
        self.world = world
        self._refresh_lods()

    def _refresh_lods(self):
        if self.world is not None and self.width > 0:
            self.lod_distances = setup_lods(self.world.max_dimension, self.width, self.height, self.fov_y_degrees, self.lod_error)

    def build_world_from_mesh(self, positions: np.ndarray, colors32: np.ndarray, max_dimension: int,
                              flips: Sequence[bool] = (False, False, False), lods: int = LOD_LEVELS) -> World:
        """World production on this context's GPU (cvx_gpu_builder_from_mesh): voxelizer + RLE + LOD mips as CUDA kernels; the
        blobs equal World.from_mesh's byte for byte. The world is returned to the host (upload it with upload_world)."""
        positions = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3)
        colors32 = np.ascontiguousarray(colors32, dtype=np.uint8).reshape(-1, 4)
        fl = (C.c_int32 * 3)(*[int(bool(f)) for f in flips])
        b = C.c_void_p()
        self._ck(lib.cvx_gpu_builder_from_mesh(self._ctx, _ptr(positions), _ptr(colors32), positions.shape[0], max_dimension, C.byref(fl), lods, C.byref(b)))
        return World._from_builder(b, lods)

    def build_resident_world_from_mesh(self, positions: np.ndarray, colors32: np.ndarray, max_dimension: int,
                                       flips: Sequence[bool] = (False, False, False), lods: int = LOD_LEVELS) -> World:
        """cvx_world_build_from_mesh: mesh -> LOD blobs -> Phase-1 tables without leaving the device; the result becomes this
        context's world. Returns a World that carries only dimensions and voxel counts (the blobs exist on the GPU only)."""
        positions = np.ascontiguousarray(positions, dtype=np.float32).reshape(-1, 3)
        colors32 = np.ascontiguousarray(colors32, dtype=np.uint8).reshape(-1, 4)
        fl = (C.c_int32 * 3)(*[int(bool(f)) for f in flips])
        dims, vox = (C.c_int32 * 3)(), (C.c_int64 * LOD_LEVELS)()
        self._ck(lib.cvx_world_build_from_mesh(self._ctx, _ptr(positions), _ptr(colors32), positions.shape[0], max_dimension, C.byref(fl), lods,
                                               C.byref(dims), C.byref(vox)))
        # the build stops at the first LOD where an axis reaches 0, as World._from_builder does
        built = next((lod for lod in range(lods) if min(dims[0] >> lod, dims[1] >> lod, dims[2] >> lod) < 1), lods)
        self.world = World((dims[0], dims[1], dims[2]), [], [], [int(v) for v in vox][:built])
        self._refresh_lods()
        return self.world

    def build_world_from_obj(self, path: str, max_dimension: int = 1024, flips: Sequence[bool] = (True, False, False),
                             swap_yz: bool = False, lods: int = LOD_LEVELS) -> World:
        """ObjModel.Import on the host, then the conversion pipeline of UnityManager.cs:297-331 on the GPU."""
        pos, col, n = C.c_void_p(), C.c_void_p(), C.c_int32()
        check(lib.cvx_obj_parse(path.encode(), int(swap_yz), C.byref(pos), C.byref(col), C.byref(n)))
        try:
            fl = (C.c_int32 * 3)(*[int(bool(f)) for f in flips])
            b = C.c_void_p()
            self._ck(lib.cvx_gpu_builder_from_mesh(self._ctx, pos, col, n.value, max_dimension, C.byref(fl), lods, C.byref(b)))
        finally:
            lib.cvx_host_free(pos)
            lib.cvx_host_free(col)
        return World._from_builder(b, lods)

    # -- resolution -------------------------------------------------------------------------------
    def set_resolution(self, width: int, height: int) -> bool:  # RenderManager.SetResolution :94-109
        if width == self.width and height == self.height:
            return False
        self._ck(lib.cvx_set_resolution(self._ctx, width, height))
        self.width, self.height = width, height
        self._refresh_lods()  # UnityManager.LateUpdate :173-176
        return True

    # -- drawing ----------------------------------------------------------------------------------
    def make_setup(self, pose: CameraPose) -> FrameSetup:
        return frame_setup(pose, self.width, self.height, self.lod_distances, self.world.dims[1])

    def draw_world(self, pose: CameraPose) -> FrameSetup:  # RenderManager.DrawWorld :111-194
        s = self.make_setup(pose)
        self._ck(lib.cvx_draw(self._ctx, C.byref(s)))
        return s

    def draw_setup(self, setup: FrameSetup):
        self._ck(lib.cvx_draw(self._ctx, C.byref(setup)))

    def draw_rays(self, setup: FrameSetup, ray_begin: int = 0, ray_end: int = -1):
        self._ck(lib.cvx_draw_rays(self._ctx, C.byref(setup), ray_begin, ray_end))

    def blit_rows(self, setup: FrameSetup, row_begin: int = 0, row_end: int = -1):
        self._ck(lib.cvx_blit_rows(self._ctx, C.byref(setup), row_begin, row_end))

    def blit_owned(self, setup: FrameSetup, ray_begin: int, ray_end: int, device_frame: int = 0):
        self._ck(lib.cvx_blit_owned(self._ctx, C.byref(setup), ray_begin, ray_end, C.c_void_p(device_frame)))

    def draw_batch(self, setups: Sequence[FrameSetup], dst: Optional[np.ndarray] = None):
        """cvx_draw_batch: with `dst` (pinned host array, one frame per view) returns when all frames are on the host; without,
        only enqueues (the frames stay on the device; read_frame / read_raybuffers return the last view)."""
        arr = (FrameSetup * len(setups))(*setups)
        self._ck(lib.cvx_draw_batch(self._ctx, arr, len(setups), _ptr(dst) if dst is not None else None))

    def draw_world_batch(self, poses: Sequence[CameraPose], dst: Optional[np.ndarray] = None, limit_horizon: bool = True):
        """cvx_draw_world_batch: RenderManager.DrawWorld for a batch of cameras — the host part of every view (vanishing point,
        segments, CameraData) is computed inside the library, one FFI call per batch."""
        arr = (Pose * len(poses))(*[p.to_native(self.width, self.height) for p in poses])
        lods = (C.c_float * LOD_LEVELS)(*[float(x) for x in self.lod_distances])
        self._ck(lib.cvx_draw_world_batch(self._ctx, arr, len(poses), C.byref(lods), int(limit_horizon), _ptr(dst) if dst is not None else None))

    def draw_batch_async(self, setups: Sequence[FrameSetup], dst: np.ndarray) -> int:
        """cvx_draw_batch_async: enqueue the batch and return its number at once; batch_wait(number) returns when its frames are in `dst`
        (pinned host array, one frame per view). A further asynchronous batch (into another destination) renders while this one's frames
        are still being copied out."""
        arr = (FrameSetup * len(setups))(*setups)
        b = C.c_int64(-1)
        self._ck(lib.cvx_draw_batch_async(self._ctx, arr, len(setups), _ptr(dst), C.byref(b)))
        return b.value

    def draw_world_batch_async(self, poses, dst: np.ndarray, limit_horizon: bool = True) -> int:
        """cvx_draw_world_batch_async. `poses` may be what pose_batch() returned (marshalled once, reused every call)."""
        arr = poses if not isinstance(poses, (list, tuple)) else self.pose_batch(poses)
        lods = (C.c_float * LOD_LEVELS)(*[float(x) for x in self.lod_distances])
        b = C.c_int64(-1)
        self._ck(lib.cvx_draw_world_batch_async(self._ctx, arr, len(arr), C.byref(lods), int(limit_horizon), _ptr(dst), C.byref(b)))
        return b.value

    def pose_batch(self, poses: Sequence[CameraPose]):
        """The poses as the C array cvx_draw_world_batch(_async) takes."""
        return (Pose * len(poses))(*[p.to_native(self.width, self.height) for p in poses])

    def batch_wait(self, batch: int):
        self._ck(lib.cvx_batch_wait(self._ctx, batch))

    def sync(self):
        self._ck(lib.cvx_sync(self._ctx))

    # -- ray queries (cvx_raycast) --------------------------------------------------------------------
    def raycast_rays(self, rays: np.ndarray, lod: int = 0) -> np.ndarray:
        """cvx_raycast over a RAY_DTYPE array (host path): returns the RAY_HIT_DTYPE hits."""
        rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
        hits = np.zeros(rays.shape[0], dtype=RAY_HIT_DTYPE)
        self._ck(lib.cvx_raycast(self._ctx, _ptr(rays), rays.shape[0], lod, _ptr(hits), 0))
        return hits

    def raycast(self, origins, directions, max_distance=np.inf, lod: int = 0) -> np.ndarray:
        """First voxel each ray hits at LOD `lod`: origins / directions (n, 3) in world units (directions need not be normalised),
        max_distance a scalar or (n,). Returns a RAY_HIT_DTYPE array (hit 1 / 0 / -1 invalid, face, cell, distance, color, steps)."""
        return self.raycast_rays(make_rays(origins, directions, max_distance), lod)

    def raycast_device(self, rays_ptr: int, hits_ptr: int, n: int, lod: int = 0):
        """cvx_raycast on device arrays (n cvx_ray in, n cvx_ray_hit out; e.g. torch tensors' data_ptr()), ordered on the context's
        stream; returns at once."""
        self._ck(lib.cvx_raycast(self._ctx, C.c_void_p(rays_ptr), n, lod, C.c_void_p(hits_ptr), 1))

    def pick(self, pose: CameraPose, px: float, py: float, lod: int = 0, max_distance: float = np.inf) -> np.void:
        """The voxel under screen pixel (px, py) (bottom-left origin) of `pose` at this context's resolution: one RAY_HIT_DTYPE record."""
        o, d = screen_ray(pose, px, py, self.width, self.height)
        return self.raycast(o, d, max_distance, lod)[0]

    # -- swept-box queries (cvx_sweep) ---------------------------------------------------------------
    def sweep_boxes(self, boxes: np.ndarray, lod: int = 0) -> np.ndarray:
        """cvx_sweep over a BOX_DTYPE array (host path): returns the RAY_HIT_DTYPE hits."""
        boxes = np.ascontiguousarray(boxes, dtype=BOX_DTYPE)
        hits = np.zeros(boxes.shape[0], dtype=RAY_HIT_DTYPE)
        self._ck(lib.cvx_sweep(self._ctx, _ptr(boxes), boxes.shape[0], lod, _ptr(hits), 0))
        return hits

    def sweep(self, centers, half_extents, directions, max_distance=np.inf, lod: int = 0) -> np.ndarray:
        """How far each axis-aligned box moves along its direction before it touches a solid cell of LOD `lod`: centers /
        directions (n, 3) and half_extents (n, 3) or (3,) in world units, max_distance a scalar or (n,). Returns a RAY_HIT_DTYPE
        array (hit 1 / 0 / -1 invalid, face of the cell entered or 6 = overlapping at the start, cell, distance, color, steps)."""
        return self.sweep_boxes(make_boxes(centers, half_extents, directions, max_distance), lod)

    def sweep_device(self, boxes_ptr: int, hits_ptr: int, n: int, lod: int = 0):
        """cvx_sweep on device arrays (n cvx_box in, n cvx_ray_hit out), ordered on the context's stream; returns at once."""
        self._ck(lib.cvx_sweep(self._ctx, C.c_void_p(boxes_ptr), n, lod, C.c_void_p(hits_ptr), 1))

    # -- outputs ----------------------------------------------------------------------------------
    def read_frame(self, out: Optional[np.ndarray] = None) -> np.ndarray:
        if out is None:
            out = np.empty((self.height, self.width), dtype=np.uint32)
        self._ck(lib.cvx_read_frame(self._ctx, _ptr(out), out.nbytes))
        return out

    def read_raybuffers(self) -> Tuple[np.ndarray, np.ndarray]:
        W, H = self.width, self.height
        td = np.empty((W + 2 * H, H), dtype=np.uint32)
        lr = np.empty((2 * W + H, W), dtype=np.uint32)
        self._ck(lib.cvx_read_raybuffer(self._ctx, 0, _ptr(td), td.nbytes))
        self._ck(lib.cvx_read_raybuffer(self._ctx, 1, _ptr(lr), lr.nbytes))
        return td, lr

    def clear_raybuffers(self, argb: int = 0):
        self._ck(lib.cvx_clear_raybuffers(self._ctx, argb))

    def blit_raybuffer(self, which: int):
        """Debug view of the last view's raybuffer (0 = top/down, 1 = left/right): the shader's COPY_MAIN1 / COPY_MAIN2 variants
        (RayBufferBlit.shader:48-53), written into the framebuffer."""
        self._ck(lib.cvx_blit_raybuffer(self._ctx, which))

    def present(self, fmt: int = 0, top_down: bool = True, out: Optional[np.ndarray] = None) -> np.ndarray:
        """cvx_present to host memory: the frame as RGBA8 (fmt 0), BGRA8 (fmt 1) or packed RGB8 (fmt 2) bytes, rows top-down or bottom-up."""
        if out is None:
            out = np.empty((self.height, self.width, 3 if fmt == 2 else 4), dtype=np.uint8)
        self._ck(lib.cvx_present(self._ctx, fmt, int(top_down), _ptr(out), 0))
        return out

    def present_jpeg(self, quality: int = 90, subsampling: int = 0) -> bytes:
        """cvx_present_jpeg: the frame encoded on the device as a baseline JPEG (subsampling 0 = 4:4:4, 1 = 4:2:0); returns the bitstream."""
        n = C.c_int64(0)
        cap = self.width * self.height * 3 + 65536  # an upper bound no baseline JPEG of the frame exceeds in practice
        buf = np.empty(cap, dtype=np.uint8)
        self._ck(lib.cvx_present_jpeg(self._ctx, quality, subsampling, _ptr(buf), cap, C.byref(n)))
        return buf[: n.value].tobytes()

    def present_device(self, device_ptr: int, fmt: int = 0, top_down: bool = True):
        """cvx_present into a caller-owned W*H*4 device buffer (graphics interop resource, encoder surface), on the context's stream."""
        self._ck(lib.cvx_present(self._ctx, fmt, int(top_down), C.c_void_p(device_ptr), 1))

    def counters(self, reset: bool = True) -> dict:
        c = N.Counters()
        self._ck(lib.cvx_get_counters(self._ctx, C.byref(c), int(reset)))
        return c.as_dict()

    def last_draw_ms(self) -> Tuple[float, float]:
        a, b = C.c_float(), C.c_float()
        self._ck(lib.cvx_last_draw_ms(self._ctx, C.byref(a), C.byref(b)))
        return a.value, b.value

    def set_option(self, option: int, value: int):
        self._ck(lib.cvx_set_option(self._ctx, option, value))

    def set_group_size(self, lanes: int):
        """Lanes cooperating on one ray in Phase 1: 0 = auto (from the frame's ray count), 8, 16 or 32."""
        self.set_option(N.OPT_GROUP_SIZE, lanes)

    def set_counters(self, on: bool):
        self.set_option(N.OPT_COUNTERS, int(on))

    def set_frames_in_flight(self, k: int):
        """Views of one draw_batch rendered concurrently (1..16, default 6), each on its own stream and buffer set."""
        self.set_option(N.OPT_FRAMES_IN_FLIGHT, k)

    def set_general_path(self, on: bool):
        """True = always run the general Phase-1 kernel; False (default) = boundary-table kernel for regular worlds."""
        self.set_option(N.OPT_GENERAL_PATH, int(on))

    def world_is_regular(self) -> bool:
        r = lib.cvx_world_is_regular(self._ctx)
        self._ck(min(r, 0))
        return bool(r)

    def profile_begin(self, max_draws: int):
        self._ck(lib.cvx_profile_begin(self._ctx, max_draws))

    def profile_end(self) -> Tuple[float, float, int]:
        a, b, n = C.c_double(), C.c_double(), C.c_int32()
        self._ck(lib.cvx_profile_end(self._ctx, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    def launch_count(self) -> int:
        return int(lib.cvx_launch_count(self._ctx))

    def ray_setup(self, setup: FrameSetup) -> np.ndarray:
        total = sum(max(0, setup.segments[k].ray_count) for k in range(4))
        out = (N.RayState * max(1, total))()
        self._ck(lib.cvx_debug_ray_setup(self._ctx, C.byref(setup), out, total))
        return np.frombuffer(out, dtype=RAY_STATE_DTYPE, count=total).copy()

    def ray_timing(self, setup: FrameSetup) -> np.ndarray:
        """Debug: cycles per code region per ray, shape (rays, 16) — see cvx_debug_ray_timing."""
        total = sum(max(0, setup.segments[k].ray_count) for k in range(4))
        out = np.zeros((max(1, total), 16), dtype=np.int64)
        self._ck(lib.cvx_debug_ray_timing(self._ctx, C.byref(setup), _ptr(out), total))
        return out[:total]

    def device_frame_ptr(self) -> Tuple[int, int]:
        p, n = C.c_void_p(), C.c_int64()
        self._ck(lib.cvx_device_frame(self._ctx, C.byref(p), C.byref(n)))
        return p.value, n.value

    def set_stream(self, cuda_stream: int):
        """Run on a caller-owned cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream); 0 restores the own stream."""
        self._ck(lib.cvx_set_stream(self._ctx, C.c_void_p(cuda_stream)))

    def ipc_export_frame(self) -> bytes:
        h = (C.c_uint8 * 64)()
        self._ck(lib.cvx_ipc_export_frame(self._ctx, C.byref(h)))
        return bytes(h)

    def ipc_open(self, handle: bytes) -> int:
        h = (C.c_uint8 * 64)(*handle)
        p = C.c_void_p()
        self._ck(lib.cvx_ipc_open(self._ctx, C.byref(h), C.byref(p)))
        return p.value

    def ipc_close(self, device_ptr: int):
        self._ck(lib.cvx_ipc_close(self._ctx, C.c_void_p(device_ptr)))

    # -- frame ring: pipelined gather of ray-sharded views (cvx_ring_*) ----------------------------------------------
    def ring_create(self, slots: int, world_size: int) -> bytes:
        h = (C.c_uint8 * 64)()
        self._ck(lib.cvx_ring_create(self._ctx, slots, world_size, C.byref(h)))
        return bytes(h)

    def ring_open(self, handle: bytes, slots: int, world_size: int):
        h = (C.c_uint8 * 64)(*handle)
        self._ck(lib.cvx_ring_open(self._ctx, C.byref(h), slots, world_size))

    def ring_close(self):
        self._ck(lib.cvx_ring_close(self._ctx))

    def draw_sharded(self, setup: FrameSetup, ray_begin: int, ray_end: int, view_index: int, rank: int):
        self._ck(lib.cvx_draw_sharded(self._ctx, C.byref(setup), ray_begin, ray_end, view_index, rank))

    def ring_consume(self, view_index: int, dst: Optional[np.ndarray] = None) -> int:
        p = C.c_void_p()
        self._ck(lib.cvx_ring_consume(self._ctx, view_index, _ptr(dst) if dst is not None else None, C.byref(p)))
        return p.value

    def ring_status(self):
        self._ck(lib.cvx_ring_status(self._ctx))

    def set_external_frame(self, device_ptr: int):
        self._ck(lib.cvx_set_external_frame(self._ctx, C.c_void_p(device_ptr)))


RAY_STATE_DTYPE = np.dtype([
    ("segment", "<i4"), ("plane_ray_index", "<i4"), ("status", "<i4"), ("lod", "<i4"),
    ("position", "<i4", 2), ("step", "<i4", 2), ("start", "<f4", 2), ("dir", "<f4", 2),
    ("t_delta", "<f4", 2), ("t_max", "<f4", 2), ("intersection_distances", "<f4", 2),
])


def write_bmp(path: str, frame: np.ndarray) -> None:
    """A frame as returned by read_frame (uint32 ColorARGB32, row 0 = bottom) as a 32-bit .bmp."""
    frame = np.ascontiguousarray(frame, dtype=np.uint32)
    check(lib.cvx_host_write_bmp(path.encode(), _ptr(frame), frame.shape[1], frame.shape[0]))


def alloc_pinned(shape, dtype=np.uint32) -> np.ndarray:
    """Page-locked host array (cudaHostAlloc) so cvx_draw_batch / cvx_read_frame copies run asynchronously."""
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    check(lib.cvx_alloc_pinned(nbytes, C.byref(p)))
    buf = (C.c_uint8 * nbytes).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype).reshape(shape)
    return arr


def algorithmic_bytes(counters: dict, width: int, height: int, frames: int = 1) -> int:
    """SURVEY.md §8(d): 12*dda_steps + 4*runs + 4*px_voxel (colour gather) + 4*(px_voxel+px_sky) (raybuffer write)
    + 8*W*H (Phase-2 read + framebuffer write), with the reference's element sizes."""
    return (12 * counters["dda_steps"] + 4 * counters["runs_visited"] + 4 * counters["px_voxel"]
            + 4 * (counters["px_voxel"] + counters["px_sky"]) + 8 * width * height * frames)
