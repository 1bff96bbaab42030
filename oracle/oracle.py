"""TEST INFRASTRUCTURE ONLY — ctypes wrapper of the CPU oracle (oracle/cpuvox_oracle.cpp).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import this.
PARITY UNPINNED (see cpuvox_oracle.h): a restatement of the reference source, not the Burst binary.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcpuvox_oracle.so")
LODS = 6


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "cpuvox_oracle.cpp")
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return LIB_PATH


class Segment(C.Structure):
    _fields_ = [("min_screen", C.c_float * 2), ("max_screen", C.c_float * 2),
                ("cam_local_plane_ray_min", C.c_float * 2), ("cam_local_plane_ray_max", C.c_float * 2),
                ("ray_count", C.c_int32)]


class Camera(C.Structure):
    _fields_ = [("world_to_screen", C.c_float * 16), ("position_xz", C.c_float * 2), ("position_y", C.c_float),
                ("inverse_element_iteration_direction", C.c_int32), ("far_clip", C.c_float),
                ("lod_distances", C.c_float * LODS)]


class FrameSetup(C.Structure):
    _fields_ = [("segments", Segment * 4), ("camera", Camera), ("vanishing_point_screen", C.c_float * 2)]


class Counters(C.Structure):
    _fields_ = [(k, C.c_uint64) for k in ("dda_steps", "columns_nonempty", "runs_visited", "px_voxel", "px_sky", "rays")]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class Pose(C.Structure):
    _fields_ = [("position", C.c_float * 3), ("rotation", C.c_float * 4), ("fov_y_degrees", C.c_float),
                ("near_clip", C.c_float), ("far_clip", C.c_float), ("pixel_width", C.c_int32), ("pixel_height", C.c_int32)]


RAY_STATE_DTYPE = np.dtype([
    ("segment", "<i4"), ("plane_ray_index", "<i4"), ("status", "<i4"), ("lod", "<i4"),
    ("position", "<i4", 2), ("step", "<i4", 2), ("start", "<f4", 2), ("dir", "<f4", 2),
    ("t_delta", "<f4", 2), ("t_max", "<f4", 2), ("intersection_distances", "<f4", 2),
])

_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(LIB_PATH)
        P = C.c_void_p
        L.orc_world_create.restype = P
        L.orc_world_create.argtypes = [C.c_int32] * 3
        L.orc_world_set_lod.argtypes = [P, C.c_int32, P, C.c_int64, C.c_int32]
        L.orc_world_free.argtypes = [P]
        L.orc_min_max.argtypes = [P, P, C.c_int32, P, P]
        L.orc_quat_euler.argtypes = [C.c_float] * 3 + [C.POINTER(C.c_float * 4)]
        L.orc_limit_rotation_horizon.argtypes = [C.POINTER(Pose)]
        L.orc_setup_lods.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float, C.POINTER(C.c_float * LODS)]
        L.orc_frame_setup_from_pose.argtypes = [C.POINTER(Pose), C.POINTER(C.c_float * LODS), C.c_int32, C.POINTER(FrameSetup)]
        L.orc_benchmark_pose.argtypes = [C.c_float, C.POINTER(C.c_int32 * 3), C.POINTER(Pose)]
        L.orc_render_raybuffers.argtypes = [P, C.POINTER(FrameSetup), C.c_int32, C.c_int32, P, P, C.c_int32, C.c_int32, C.c_int32, C.POINTER(Counters)]
        L.orc_blit.argtypes = [C.POINTER(FrameSetup), C.c_int32, C.c_int32, P, P, P, C.c_int32, C.c_int32, C.c_int32]
        L.orc_blit_raybuffer.argtypes = [P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, P]
        L.orc_blit_raybuffer.restype = C.c_int
        L.orc_ray_setup.argtypes = [P, C.POINTER(FrameSetup), C.c_int32, C.c_int32, P, C.c_int32]
        L.orc_ray_stats.argtypes = [P, C.POINTER(FrameSetup), C.c_int32, C.c_int32, P, C.c_int32]
        L.orc_dda_walk.argtypes = [C.POINTER(C.c_float * 2), C.POINTER(C.c_float * 2), C.POINTER(C.c_float * LODS), C.c_float, C.c_int32, P, P]
        L.orc_hardware_threads.restype = C.c_int
        _lib = L
    return _lib


class OracleWorld:
    """Borrowed view of reference-layout LOD blobs (numpy uint8 arrays must outlive this object)."""

    def __init__(self, dims, blobs, column_counts):
        L = lib()
        self.dims = tuple(dims)
        self._blobs = [np.ascontiguousarray(b) for b in blobs]
        self._w = C.c_void_p(L.orc_world_create(*self.dims))
        for lod, (b, cc) in enumerate(zip(self._blobs, column_counts)):
            assert L.orc_world_set_lod(self._w, lod, b.ctypes.data_as(C.c_void_p), b.nbytes, cc) == 0

    def __del__(self):
        if getattr(self, "_w", None):
            lib().orc_world_free(self._w)
            self._w = None


def copy_setup(src) -> FrameSetup:
    """Reinterpret a product-side FrameSetup (same layout by design) as the oracle's struct."""
    out = FrameSetup()
    assert C.sizeof(out) == C.sizeof(src)
    C.memmove(C.byref(out), C.byref(src), C.sizeof(out))
    return out


def frame_setup(position, rotation, width, height, lod_distances, world_dim_y, fov=85.0, near=0.05, far=2048.0, limit_horizon=True) -> FrameSetup:
    L = lib()
    p = Pose()
    p.position[:] = position
    p.rotation[:] = rotation
    p.fov_y_degrees, p.near_clip, p.far_clip, p.pixel_width, p.pixel_height = fov, near, far, width, height
    if limit_horizon:
        L.orc_limit_rotation_horizon(C.byref(p))
    lods = (C.c_float * LODS)(*[float(x) for x in lod_distances])
    out = FrameSetup()
    assert L.orc_frame_setup_from_pose(C.byref(p), C.byref(lods), world_dim_y, C.byref(out)) == 0
    return out


def limit_rotation_horizon(position, rotation):
    """UnityManager.LimitRotationHorizon (UnityManager.cs:193-201): the rotation DrawWorld receives."""
    p = Pose()
    p.position[:] = position
    p.rotation[:] = rotation
    p.pixel_width = p.pixel_height = 16
    lib().orc_limit_rotation_horizon(C.byref(p))
    return tuple(p.rotation)


def setup_lods(world_max_dimension, res_x, res_y, fov=85.0, lod_error=1.0) -> np.ndarray:
    out = (C.c_float * LODS)()
    lib().orc_setup_lods(world_max_dimension, res_x, res_y, fov, lod_error, C.byref(out))
    return np.array(out[:], dtype=np.float32)


def benchmark_pose(t, dims):
    p = Pose()
    d = (C.c_int32 * 3)(*dims)
    lib().orc_benchmark_pose(t, C.byref(d), C.byref(p))
    return tuple(p.position), tuple(p.rotation)


def quat_euler(x, y, z):
    q = (C.c_float * 4)()
    lib().orc_quat_euler(x, y, z, C.byref(q))
    return tuple(q)


def render_raybuffers(world: OracleWorld, setup: FrameSetup, width, height, ray_begin=0, ray_end=-1, threads=0, td=None, lr=None):
    W, H = width, height
    if td is None:
        td = np.zeros((W + 2 * H, H), dtype=np.uint32)
    if lr is None:
        lr = np.zeros((2 * W + H, W), dtype=np.uint32)
    cn = Counters()
    r = lib().orc_render_raybuffers(world._w, C.byref(setup), W, H, td.ctypes.data_as(C.c_void_p), lr.ctypes.data_as(C.c_void_p),
                                    ray_begin, ray_end, threads, C.byref(cn))
    assert r == 0
    return td, lr, cn.as_dict()


def blit(setup: FrameSetup, width, height, td, lr, threads=0, row_begin=0, row_end=-1, frame=None):
    if frame is None:
        frame = np.zeros((height, width), dtype=np.uint32)
    r = lib().orc_blit(C.byref(setup), width, height, td.ctypes.data_as(C.c_void_p), lr.ctypes.data_as(C.c_void_p),
                       frame.ctypes.data_as(C.c_void_p), row_begin, row_end, threads)
    assert r == 0
    return frame


def blit_raybuffer(buf: np.ndarray, width, height) -> np.ndarray:
    """Debug view COPY_MAIN1 / COPY_MAIN2 (RayBufferBlit.shader:48-53) of one raybuffer (rows x row_len)."""
    buf = np.ascontiguousarray(buf, dtype=np.uint32)
    frame = np.zeros((height, width), dtype=np.uint32)
    r = lib().orc_blit_raybuffer(buf.ctypes.data_as(C.c_void_p), buf.shape[0], buf.shape[1], width, height, frame.ctypes.data_as(C.c_void_p))
    assert r == 0
    return frame


def ray_setup(world: OracleWorld, setup: FrameSetup, width, height) -> np.ndarray:
    total = sum(max(0, setup.segments[k].ray_count) for k in range(4))
    out = np.zeros(max(1, total), dtype=RAY_STATE_DTYPE)
    n = lib().orc_ray_setup(world._w, C.byref(setup), width, height, out.ctypes.data_as(C.c_void_p), total)
    assert n == total
    return out[:total]


def min_max(a, b):
    """The renderer's math.min / math.max, elementwise over float32 arrays: (min, max)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    b = np.ascontiguousarray(b, dtype=np.float32)
    mn, mx = np.empty_like(a), np.empty_like(a)
    lib().orc_min_max(a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), a.size, mn.ctypes.data_as(C.c_void_p), mx.ctypes.data_as(C.c_void_p))
    return mn, mx


def dda_walk(start, direction, lod_distances, far_clip, max_steps=100000):
    """Cell sequence (x, z, lod) and (last, next) distances of one ray as ExecuteRay walks it."""
    cells = np.zeros((max_steps, 3), dtype=np.int32)
    dists = np.zeros((max_steps, 2), dtype=np.float32)
    n = lib().orc_dda_walk(C.byref((C.c_float * 2)(*start)), C.byref((C.c_float * 2)(*direction)),
                           C.byref((C.c_float * LODS)(*[float(x) for x in lod_distances])), far_clip, max_steps,
                           cells.ctypes.data_as(C.c_void_p), dists.ctypes.data_as(C.c_void_p))
    return cells[:n], dists[:n]


RAY_STAT_FIELDS = ("dda_steps", "columns_nonempty", "columns_entered", "renarrows", "runs_visited", "spans_tested",
                   "spans_committed", "spans_wrote", "px_voxel", "px_sky")


def ray_stats(world: OracleWorld, setup: FrameSetup, width, height) -> np.ndarray:
    """Diagnostics: per-ray work counts, shape (rays, len(RAY_STAT_FIELDS))."""
    total = sum(max(0, setup.segments[k].ray_count) for k in range(4))
    out = np.zeros((max(1, total), len(RAY_STAT_FIELDS)), dtype=np.uint64)
    n = lib().orc_ray_stats(world._w, C.byref(setup), width, height, out.ctypes.data_as(C.c_void_p), total)
    assert n == total
    return out[:total]


def hardware_threads() -> int:
    return int(lib().orc_hardware_threads())
