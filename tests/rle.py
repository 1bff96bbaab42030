"""Test helper: numpy encoder/decoder of the reference's world blob layout (Assets/Code/World.cs:161-234,285-313):
column_count 12-byte RLEColumn headers {int32 elementOffset; uint16 runCount, worldMin, worldMax; pad}, then 4-byte cells;
per non-empty column [guard(0,0)] [RLEElement{int16 ColorsIndex, int16 Length}]*runCount [guard] [ColorARGB32]*solidCount,
runs stored top -> bottom, colours top-first, air runs have ColorsIndex < 0."""
from __future__ import annotations

import numpy as np


def column_count(dim_x: int, dim_z: int, lod: int = 0) -> int:
    return (dim_x * dim_z) // ((lod + 1) * (lod + 1))  # World.ColumnCount, World.cs:17 (an over-estimate for lod >= 2)


def encode_world(grid: np.ndarray, lod: int = 0):
    """grid[x, y, z] uint32: 0 = air, else the ColorARGB32 value. Returns (blob uint8, column_count)."""
    dx, dy, dz = grid.shape
    cc = column_count(dx << lod, dz << lod, lod)
    assert cc >= dx * dz
    headers = np.zeros((cc, 3), dtype=np.uint32)
    cells = []
    for x, z in zip(*np.nonzero(grid.any(axis=1))):  # the non-empty columns, in index order
        col = grid[x, :, z]
        runs, colors = [], []
        y = dy - 1
        while y >= 0:  # top -> bottom
            solid = col[y] != 0
            y0 = y
            while y >= 0 and (col[y] != 0) == solid:
                y -= 1
            length = y0 - y
            if solid:
                runs.append((len(colors), length))
                colors.extend(int(c) for c in col[y + 1:y0 + 1][::-1])
            else:
                runs.append((-1, length))
        ys = np.nonzero(col)[0]
        off = len(cells)
        cells.append(0)
        for ci, ln in runs:
            cells.append((ci & 0xFFFF) | ((ln & 0xFFFF) << 16))
        cells.append(0)
        cells.extend(colors)
        idx = x * dz + z
        headers[idx, 0] = off
        headers[idx, 1] = len(runs) | (((int(ys.min())) << lod) << 16)
        headers[idx, 2] = (int(ys.max()) + 1) << lod
    if not cells:
        cells = [0]
    blob = np.concatenate([headers.reshape(-1).view(np.uint8), np.array(cells, dtype=np.uint32).view(np.uint8)])
    return blob, cc


def decode_world(blob: np.ndarray, cc: int, dims, lod: int = 0) -> np.ndarray:
    """Inverse of encode_world for one LOD blob; also checks the layout invariants."""
    dx, dy, dz = dims[0] >> lod, dims[1] >> lod, dims[2] >> lod
    words = np.frombuffer(np.ascontiguousarray(blob).tobytes(), dtype=np.uint32)
    headers = words[:3 * cc].reshape(cc, 3)
    cells = words[3 * cc:]
    grid = np.zeros((dx, dy, dz), dtype=np.uint32)
    for x in range(dx):
        for z in range(dz):
            off, w1, w2 = (int(v) for v in headers[x * dz + z])
            rc = w1 & 0xFFFF
            if rc == 0:
                continue
            assert cells[off] == 0 and cells[off + rc + 1] == 0, "guards"
            colors = cells[off + rc + 2:]
            y = dy
            lo, hi = dy, 0
            for k in range(rc):
                e = int(cells[off + 1 + k])
                ci = e & 0xFFFF
                ci = ci - 0x10000 if ci >= 0x8000 else ci
                ln = (e >> 16) & 0xFFFF
                assert 0 < ln <= 0x7FFF
                if ci >= 0:
                    grid[x, y - ln:y, z] = colors[ci:ci + ln][::-1]
                    lo, hi = min(lo, y - ln), max(hi, y)
                y -= ln
            assert y == 0, "runs must cover the whole column height"
            assert (w1 >> 16) == lo << lod and (w2 & 0xFFFF) == hi << lod, "worldMin/worldMax"
    return grid
