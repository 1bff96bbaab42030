"""ctypes binding of libcpuvox_b200.so (include/cpuvox_b200.h).

This is the same C ABI a C# host binds with [DllImport("cpuvox_b200")] (see INTEGRATION.md); the
Python layer above it only exists because the image has no .NET toolchain. There is no fallback of any
kind: if the shared library is missing this module raises at import, and every rendering entry point
fails with CVX_ERR_NO_DEVICE when no CUDA device is present.
"""
from __future__ import annotations

import ctypes as C
import os

LOD_LEVELS = 6  # UnityManager.LOD_LEVELS, Assets/Code/UnityManager.cs:42

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CPUVOX_B200_LIB") or os.path.join(_HERE, "libcpuvox_b200.so")  # the override is for kernel-variant A/B runs (tools/)


class CvxError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"cpuvox_b200 error {code}: {message}")
        self.code = code


class Segment(C.Structure):  # RenderManager.SegmentData, RenderManager.cs:503-510
    _fields_ = [
        ("min_screen", C.c_float * 2),
        ("max_screen", C.c_float * 2),
        ("cam_local_plane_ray_min", C.c_float * 2),
        ("cam_local_plane_ray_max", C.c_float * 2),
        ("ray_count", C.c_int32),
    ]


class Camera(C.Structure):  # CameraData, CameraData.cs:11-36
    _fields_ = [
        ("world_to_screen", C.c_float * 16),
        ("position_xz", C.c_float * 2),
        ("position_y", C.c_float),
        ("inverse_element_iteration_direction", C.c_int32),
        ("far_clip", C.c_float),
        ("lod_distances", C.c_float * LOD_LEVELS),
    ]


class FrameSetup(C.Structure):
    _fields_ = [
        ("segments", Segment * 4),
        ("camera", Camera),
        ("vanishing_point_screen", C.c_float * 2),
    ]


class Counters(C.Structure):
    _fields_ = [
        ("dda_steps", C.c_uint64),
        ("columns_nonempty", C.c_uint64),
        ("runs_visited", C.c_uint64),
        ("px_voxel", C.c_uint64),
        ("px_sky", C.c_uint64),
        ("rays", C.c_uint64),
    ]

    def as_dict(self):
        return {k: int(getattr(self, k)) for k, _ in self._fields_}


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("flags", C.c_int32)]


FLAG_COUNTERS = 1
OPT_GROUP_SIZE = 1
OPT_COUNTERS = 2
OPT_GENERAL_PATH = 3
OPT_FRAMES_IN_FLIGHT = 4


class Pose(C.Structure):
    _fields_ = [
        ("position", C.c_float * 3),
        ("rotation", C.c_float * 4),
        ("fov_y_degrees", C.c_float),
        ("near_clip", C.c_float),
        ("far_clip", C.c_float),
        ("pixel_width", C.c_int32),
        ("pixel_height", C.c_int32),
    ]


class RayState(C.Structure):
    _fields_ = [
        ("segment", C.c_int32),
        ("plane_ray_index", C.c_int32),
        ("status", C.c_int32),
        ("lod", C.c_int32),
        ("position", C.c_int32 * 2),
        ("step", C.c_int32 * 2),
        ("start", C.c_float * 2),
        ("dir", C.c_float * 2),
        ("t_delta", C.c_float * 2),
        ("t_max", C.c_float * 2),
        ("intersection_distances", C.c_float * 2),
    ]


class Ray(C.Structure):  # cvx_ray: a ray query (no reference analogue), 32 bytes
    _fields_ = [
        ("origin", C.c_float * 3),
        ("max_distance", C.c_float),
        ("direction", C.c_float * 3),
        ("reserved", C.c_int32),
    ]


class RayHit(C.Structure):  # cvx_ray_hit, 32 bytes
    _fields_ = [
        ("hit", C.c_int32),
        ("face", C.c_int32),
        ("cell", C.c_int32 * 3),
        ("distance", C.c_float),
        ("color", C.c_uint32),
        ("steps", C.c_int32),
    ]


# every symbol include/cpuvox_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I32, _I64, _U32, _F = C.c_int32, C.c_int64, C.c_uint32, C.c_float
SYMBOLS = {
    "cvx_create": (C.c_int, [C.POINTER(Config), C.POINTER(_P)]),
    "cvx_destroy": (C.c_int, [_P]),
    "cvx_last_error": (C.c_char_p, [_P]),
    "cvx_set_stream": (C.c_int, [_P, _P]),
    "cvx_world_upload": (C.c_int, [_P, _I32, _I32, _I32, _I32, _P, _I64, _I32]),
    "cvx_world_free": (C.c_int, [_P]),
    "cvx_set_resolution": (C.c_int, [_P, _I32, _I32]),
    "cvx_draw": (C.c_int, [_P, C.POINTER(FrameSetup)]),
    "cvx_draw_rays": (C.c_int, [_P, C.POINTER(FrameSetup), _I32, _I32]),
    "cvx_blit_rows": (C.c_int, [_P, C.POINTER(FrameSetup), _I32, _I32]),
    "cvx_blit_owned": (C.c_int, [_P, C.POINTER(FrameSetup), _I32, _I32, _P]),
    "cvx_draw_batch": (C.c_int, [_P, C.POINTER(FrameSetup), _I32, _P]),
    "cvx_draw_world_batch": (C.c_int, [_P, C.POINTER(Pose), _I32, C.POINTER(_F * LOD_LEVELS), _I32, _P]),
    "cvx_draw_batch_async": (C.c_int, [_P, C.POINTER(FrameSetup), _I32, _P, C.POINTER(C.c_int64)]),
    "cvx_draw_world_batch_async": (C.c_int, [_P, C.POINTER(Pose), _I32, C.POINTER(_F * LOD_LEVELS), _I32, _P, C.POINTER(C.c_int64)]),
    "cvx_batch_wait": (C.c_int, [_P, C.c_int64]),
    "cvx_sync": (C.c_int, [_P]),
    "cvx_read_frame": (C.c_int, [_P, _P, _I64]),
    "cvx_read_raybuffer": (C.c_int, [_P, _I32, _P, _I64]),
    "cvx_get_counters": (C.c_int, [_P, C.POINTER(Counters), _I32]),
    "cvx_clear_raybuffers": (C.c_int, [_P, _U32]),
    "cvx_blit_raybuffer": (C.c_int, [_P, _I32]),
    "cvx_present": (C.c_int, [_P, _I32, _I32, _P, _I32]),
    "cvx_present_jpeg": (C.c_int, [_P, _I32, _I32, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "cvx_alloc_pinned": (C.c_int, [_I64, C.POINTER(_P)]),
    "cvx_free_pinned": (C.c_int, [_P]),
    "cvx_device_frame": (C.c_int, [_P, C.POINTER(_P), C.POINTER(_I64)]),
    "cvx_device_raybuffer": (C.c_int, [_P, _I32, C.POINTER(_P), C.POINTER(_I64)]),
    "cvx_set_external_frame": (C.c_int, [_P, _P]),
    "cvx_last_draw_ms": (C.c_int, [_P, C.POINTER(_F), C.POINTER(_F)]),
    "cvx_launch_count": (_I64, [_P]),
    "cvx_set_option": (C.c_int, [_P, _I32, _I32]),
    "cvx_world_is_regular": (C.c_int, [_P]),
    "cvx_profile_begin": (C.c_int, [_P, _I32]),
    "cvx_profile_end": (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(_I32)]),
    "cvx_ipc_export_frame": (C.c_int, [_P, C.POINTER(C.c_uint8 * 64)]),
    "cvx_ipc_open": (C.c_int, [_P, C.POINTER(C.c_uint8 * 64), C.POINTER(_P)]),
    "cvx_ipc_close": (C.c_int, [_P, _P]),
    "cvx_ring_create": (C.c_int, [_P, C.c_int32, C.c_int32, C.POINTER(C.c_uint8 * 64)]),
    "cvx_ring_open": (C.c_int, [_P, C.POINTER(C.c_uint8 * 64), C.c_int32, C.c_int32]),
    "cvx_ring_close": (C.c_int, [_P]),
    "cvx_draw_sharded": (C.c_int, [_P, C.POINTER(FrameSetup), C.c_int32, C.c_int32, C.c_int64, C.c_int32]),
    "cvx_ring_consume": (C.c_int, [_P, C.c_int64, _P, C.POINTER(_P)]),
    "cvx_ring_status": (C.c_int, [_P]),
    "cvx_raycast": (C.c_int, [_P, _P, _I32, _I32, _P, _I32]),
    "cvx_debug_ray_setup": (C.c_int, [_P, C.POINTER(FrameSetup), C.POINTER(RayState), _I32]),
    "cvx_debug_ray_timing": (C.c_int, [_P, C.POINTER(FrameSetup), _P, _I32]),
    "cvx_host_quat_euler": (None, [_F, _F, _F, C.POINTER(_F * 4)]),
    "cvx_host_limit_rotation_horizon": (None, [C.POINTER(Pose)]),
    "cvx_host_setup_lods": (None, [_I32, _I32, _I32, _F, _F, C.POINTER(_F * LOD_LEVELS)]),
    "cvx_host_screen_ray": (None, [C.POINTER(Pose), _F, _F, C.POINTER(_F * 3), C.POINTER(_F * 3)]),
    "cvx_host_frame_setup": (C.c_int, [C.POINTER(Pose), C.POINTER(_F * LOD_LEVELS), _I32, C.POINTER(FrameSetup)]),
    "cvx_host_benchmark_pose": (None, [_F, C.POINTER(_I32 * 3), C.POINTER(Pose)]),
    "cvx_host_benchmark_length": (_F, []),
    "cvx_builder_from_mesh": (C.c_int, [_P, _P, _I32, _I32, C.POINTER(_I32 * 3), _I32, C.POINTER(_P)]),
    "cvx_gpu_builder_from_mesh": (C.c_int, [_P, _P, _P, _I32, _I32, C.POINTER(_I32 * 3), _I32, C.POINTER(_P)]),
    "cvx_world_build_from_mesh": (C.c_int, [_P, _P, _P, _I32, _I32, C.POINTER(_I32 * 3), _I32, C.POINTER(_I32 * 3), C.POINTER(_I64 * LOD_LEVELS)]),
    "cvx_obj_parse": (C.c_int, [C.c_char_p, _I32, C.POINTER(_P), C.POINTER(_P), C.POINTER(_I32)]),
    "cvx_host_free": (None, [_P]),
    "cvx_builder_synthetic": (C.c_int, [_I32, _I32, _I32, _I32, _U32, _I32, C.POINTER(_P)]),
    "cvx_builder_dims": (C.c_int, [_P, C.POINTER(_I32 * 3)]),
    "cvx_builder_lod": (C.c_int, [_P, _I32, C.POINTER(_P), C.POINTER(_I64), C.POINTER(_I32), C.POINTER(_I64)]),
    "cvx_builder_free": (None, [_P]),
    "cvx_world_file_write": (C.c_int, [C.c_char_p, C.POINTER(_I32 * 3), _I32, C.POINTER(_P), C.POINTER(_I64)]),
    "cvx_host_write_bmp": (C.c_int, [C.c_char_p, _P, _I32, _I32]),
    "cvx_world_file_read": (C.c_int, [C.c_char_p, C.POINTER(_I32 * 3), C.POINTER(_I32), C.POINTER(_P * LOD_LEVELS), C.POINTER(_I64 * LOD_LEVELS)]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C cpuvox_b200/csrc). cpuvox_b200 has no Python or CPU fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here means the .so is stale
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()


def check(code: int, ctx=None):
    if code < 0:
        msg = lib.cvx_last_error(ctx)
        raise CvxError(code, msg.decode() if msg else "")
    return code
