"""TEST INFRASTRUCTURE: ctypes binding of tools/raycast_oracle/libraycast_oracle.so — the definition of cvx_raycast as a literal
per-cell walk over LOD blobs in the reference layout (DESIGN.md §3.5), and of the same traversal compiled for the CPU from the
kernel source (raycast.h through tools/simt_emu: emu_raycast). The product never loads either."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_DIR = os.path.join(ROOT, "tools", "raycast_oracle")
_lib = None
_emu = None

RAY_DTYPE = np.dtype([("origin", "<f4", 3), ("max_distance", "<f4"), ("direction", "<f4", 3), ("reserved", "<i4")])
RAY_HIT_DTYPE = np.dtype([("hit", "<i4"), ("face", "<i4"), ("cell", "<i4", 3), ("distance", "<f4"), ("color", "<u4"), ("steps", "<i4")])


def lib():
    global _lib
    if _lib is None:
        subprocess.check_call(["make", "-C", _DIR, "-s"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        L = C.CDLL(os.path.join(_DIR, "libraycast_oracle.so"))
        P = C.c_void_p
        L.rco_world_create.restype = P
        L.rco_world_create.argtypes = [C.c_int32] * 3
        L.rco_world_set_lod.argtypes = [P, C.c_int32, P, C.c_int64, C.c_int32]
        L.rco_world_free.argtypes = [P]
        L.rco_raycast.argtypes = [P, C.c_int32, P, C.c_int32, P, C.c_int32]
        _lib = L
    return _lib


def emu_lib():
    global _emu
    if _emu is None:
        import emu
        L = emu.lib()
        L.emu_raycast.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
        _emu = L
    return _emu


class RayWorld:
    """The per-cell definition's view of reference-layout LOD blobs (kept alive by this object)."""

    def __init__(self, world):
        L = lib()
        self.dims = tuple(world.dims)
        self.lods = len(world.blobs)
        self._blobs = [np.ascontiguousarray(b) for b in world.blobs]
        self._w = C.c_void_p(L.rco_world_create(*self.dims))
        for lod, (b, cc) in enumerate(zip(self._blobs, world.column_counts)):
            assert L.rco_world_set_lod(self._w, lod, b.ctypes.data_as(C.c_void_p), b.nbytes, cc) == 0

    def __del__(self):
        if getattr(self, "_w", None):
            lib().rco_world_free(self._w)
            self._w = None


def raycast(world: RayWorld, rays: np.ndarray, lod: int = 0, threads: int = 0) -> np.ndarray:
    rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
    hits = np.zeros(rays.shape[0], dtype=RAY_HIT_DTYPE)
    assert lib().rco_raycast(world._w, lod, rays.ctypes.data_as(C.c_void_p), rays.shape[0], hits.ctypes.data_as(C.c_void_p), threads) == 0
    return hits


def emu_raycast(emu_world, rays: np.ndarray, lod: int = 0, general: bool = False, threads: int = 0) -> np.ndarray:
    """raycast.h compiled for the CPU (the kernel's traversal); emu_world is a tests/emu.py EmuWorld."""
    rays = np.ascontiguousarray(rays, dtype=RAY_DTYPE)
    hits = np.zeros(rays.shape[0], dtype=RAY_HIT_DTYPE)
    assert emu_lib().emu_raycast(emu_world._w, lod, rays.ctypes.data, rays.shape[0], hits.ctypes.data, int(general), threads) == 0
    return hits
