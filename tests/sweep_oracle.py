"""TEST INFRASTRUCTURE: ctypes binding of the swept-box query in tools/raycast_oracle/libraycast_oracle.so — the definition of
cvx_sweep evaluated cell by cell (DESIGN.md §3.6, rco_sweep) — and of the kernel's traversal compiled for the CPU (raycast.h through
tools/simt_emu: emu_sweep). It shares the libraries and the world object of raycast_oracle.py. The product never loads either."""
from __future__ import annotations

import ctypes as C

import numpy as np

import raycast_oracle as rco
from raycast_oracle import RAY_HIT_DTYPE, RayWorld  # noqa: F401  (re-exported: the worlds and hits are those of the ray query)

BOX_DTYPE = np.dtype([("center", "<f4", 3), ("max_distance", "<f4"), ("direction", "<f4", 3), ("reserved0", "<i4"),
                      ("half_extent", "<f4", 3), ("reserved1", "<i4")])


def sweep(world: RayWorld, boxes: np.ndarray, lod: int = 0, threads: int = 0) -> np.ndarray:
    """The definition of cvx_sweep evaluated cell by cell (steps stays 0)."""
    L = rco.lib()
    L.rco_sweep.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]
    boxes = np.ascontiguousarray(boxes, dtype=BOX_DTYPE)
    hits = np.zeros(boxes.shape[0], dtype=RAY_HIT_DTYPE)
    assert L.rco_sweep(world._w, lod, boxes.ctypes.data_as(C.c_void_p), boxes.shape[0], hits.ctypes.data_as(C.c_void_p), threads) == 0
    return hits


def emu_sweep(emu_world, boxes: np.ndarray, lod: int = 0, general: bool = False, threads: int = 0) -> np.ndarray:
    """cvx_sweep's traversal (raycast.h compiled for the CPU); emu_world is a tests/emu.py EmuWorld."""
    L = rco.emu_lib()
    L.emu_sweep.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
    boxes = np.ascontiguousarray(boxes, dtype=BOX_DTYPE)
    hits = np.zeros(boxes.shape[0], dtype=RAY_HIT_DTYPE)
    assert L.emu_sweep(emu_world._w, lod, boxes.ctypes.data, boxes.shape[0], hits.ctypes.data, int(general), threads) == 0
    return hits
