"""TEST INFRASTRUCTURE: ctypes binding of tools/simt_emu/libcvx_emu.so — the CUDA kernel source of Phase 1 compiled for the
CPU through a SIMT emulator (one fiber per lane). Lets `-m "not gpu"` tests compare kernel LOGIC with the oracle in a container
without a GPU. The product never loads this; the `-m gpu` tests call the real kernels through the C ABI."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_DIR = os.path.join(ROOT, "tools", "simt_emu")
_lib = None


def lib():
    global _lib
    if _lib is None:
        subprocess.check_call(["make", "-C", _DIR, "-s"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        L = C.CDLL(os.path.join(_DIR, "libcvx_emu.so"))
        L.emu_world_create.restype = C.c_void_p
        L.emu_world_create.argtypes = [C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_void_p), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]
        L.emu_world_destroy.argtypes = [C.c_void_p]
        L.emu_world_regular.argtypes = [C.c_void_p]
        L.emu_transcode_verdict.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_int, C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_int)]
        L.emu_phase1.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 5
        _lib = L
    return _lib


class EmuWorld:
    def __init__(self, world):
        n = len(world.blobs)
        self._blobs = [np.ascontiguousarray(b) for b in world.blobs]
        dims = (C.c_int32 * 3)(*world.dims)
        ptrs = (C.c_void_p * n)(*[b.ctypes.data for b in self._blobs])
        sizes = (C.c_int64 * n)(*[b.nbytes for b in self._blobs])
        counts = (C.c_int32 * n)(*world.column_counts)
        self._w = lib().emu_world_create(n, dims, ptrs, sizes, counts)
        assert self._w, "world blob rejected"

    @property
    def regular(self) -> bool:
        return bool(lib().emu_world_regular(self._w))

    def __del__(self):
        if getattr(self, "_w", None):
            lib().emu_world_destroy(self._w)
            self._w = None


def transcode_verdict(blob: np.ndarray, column_count: int, dims, lod: int = 0):
    """world_transcode.h on one LOD blob: (accepted, first bad column or -1, regular)."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    bad, regular = C.c_int64(-1), C.c_int(0)
    ok = lib().emu_transcode_verdict(blob.ctypes.data, blob.nbytes, column_count, lod, (C.c_int32 * 3)(*dims), C.byref(bad), C.byref(regular))
    return bool(ok), int(bad.value), bool(regular.value)


def render_raybuffers(world: EmuWorld, setup, W, H, variant=0, group=32, counters=True, fill=0, threads=0, ray_begin=0, ray_end=-1):
    """Phase 1 of `setup` (a cpuvox_b200 FrameSetup) through the emulated kernel. variant 0 = general kernel, 1 = fast kernel."""
    td = np.full((W + 2 * H, H), fill, dtype=np.uint32)
    lr = np.full((2 * W + H, W), fill, dtype=np.uint32)
    cn = np.zeros(6, dtype=np.uint64)
    lib().emu_phase1(world._w, C.addressof(setup), W, H, td.ctypes.data, lr.ctypes.data, cn.ctypes.data if counters else None,
                     variant, group, threads, ray_begin, ray_end)
    names = ("dda_steps", "columns_nonempty", "runs_visited", "px_voxel", "px_sky", "rays")
    return td, lr, ({k: int(v) for k, v in zip(names, cn)} if counters else None)
