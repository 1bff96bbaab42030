"""TEST INFRASTRUCTURE: world production restated in plain NumPy, independent of both builders (world_builder.cpp on the host,
world_builder_gpu.cu on the device). The product never loads this.

    remap     SimpleMesh.Remap_Internal (SimpleMesh.cs:64-106): fp32 scale to max_dimension, next_pow2 dims, flips p = dims - p
    voxelize  VoxelizerHelper.GetVoxelsInternal (VoxelizerHelper.cs:28-132) in float32, expression for expression and in the same
              order; NumPy float32 arithmetic rounds every operation and never contracts to FMA, as the builders' -fmad=false and
              -ffp-contract=off builds do. Scan order x, then z, then y; a triangle stops after VOXELIZE_BUFFER_MAX voxels
    merge     RLEColumnBuilder dedupe (WordBuilder.cs:203-228): per (x, y, z) the integer mean of each channel, alpha of the first
    lod       World.DownSample (World.cs:45-127): the unique LOD-0 voxels grouped by (x >> j, y >> j, z >> j), integer mean again
    blob      tests/rle.py::encode_world plus the WorldAllocator capacity rule (World.cs:295-373) and World.ColumnCount (World.cs:17)

NaN rules (DESIGN.md §3.4). A corner whose vertex lies exactly on the fp32 centroid of a non-degenerate triangle is pushed out by
normalize(0) * 0.5, which is NaN in every component. The bounding box ignores a NaN operand (math.min / math.max of the reference,
fminf / fmaxf), so it spans the other two corners. Every comparison with NaN is false, so no cell of that box is rejected, and
every colour channel is NaN; a NaN channel converts to the byte 0.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Sequence, Tuple

import numpy as np

from rle import column_count, encode_world

VOXELIZE_BUFFER_MAX = 1024 * 256  # WordBuilder.cs:37
F = np.float32


def next_pow2(n: int) -> int:
    """Mathf.NextPowerOfTwo: 0 for n <= 0."""
    if n <= 0:
        return 0
    p = 1
    while p < n:
        p <<= 1
    return p


def remap(positions: np.ndarray, max_dimension: int, flips: Sequence[bool] = (False, False, False)) -> Tuple[np.ndarray, Tuple[int, int, int]]:
    """Vertices in world units (float32 (n, 3)) and the world dimensions."""
    v = np.ascontiguousarray(positions, dtype=F).reshape(-1, 3)
    mn, mx = v.min(axis=0), v.max(axis=0)
    size = mx - mn
    scale = F(max_dimension) / max(size[0], size[1], size[2])
    dims = tuple(next_pow2(int(size[k] * scale)) for k in range(3))
    v = (v - mn) * scale
    for k in range(3):
        if flips[k]:
            v[:, k] = F(dims[k]) - v[:, k]
    return v.astype(F), dims


def _dot(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def _normalize(a):
    r = F(1.0) / np.sqrt(_dot(a, a))
    return [a[0] * r, a[1] * r, a[2] * r]


def _f2i(f: F) -> int:
    """(int)f as cvttss2si: out of range and NaN give INT_MIN."""
    return int(f) if -2147483648.0 <= f < 2147483648.0 else -2147483648


def to_byte(c: np.ndarray) -> np.ndarray:
    """Color -> Color32 channel: round(clamp01(c) * 255), half to even; NaN -> 0."""
    v = np.where(c > F(0.0), np.where(c < F(1.0), c, F(1.0)), F(0.0)).astype(F)
    return np.rint(v * F(255.0)).astype(np.uint32)


def voxelize_triangle(tri: np.ndarray, cols: np.ndarray, dims) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray, int]:
    """One triangle (float32 (3, 3) world units, uint8 (3, 4) Color32): (x, y, z, argb) of its voxels in scan order, after the
    VOXELIZE_BUFFER_MAX cut, and the number of voxels before the cut."""
    empty = np.zeros(0, dtype=np.int64)
    a, b, c = ([F(t) for t in tri[i]] for i in range(3))
    e1 = [b[k] - a[k] for k in range(3)]
    e2 = [c[k] - a[k] for k in range(3)]
    nc = [e1[1] * e2[2] - e1[2] * e2[1], e1[2] * e2[0] - e1[0] * e2[2], e1[0] * e2[1] - e1[1] * e2[0]]
    l2 = _dot(nc, nc)
    if l2 == F(0.0):
        return empty, empty, empty, np.zeros(0, dtype=np.uint32), 0
    inv = F(1.0) / np.sqrt(l2)
    n = [nc[k] * inv for k in range(3)]
    mid = [((a[k] + b[k]) + c[k]) * F(1.0) for k in range(3)]
    mid = [mid[k] / F(3.0) for k in range(3)]
    corners = []
    for p in (a, b, c):
        q = _normalize([p[k] - mid[k] for k in range(3)])
        corners.append([p[k] + q[k] * F(0.5) for k in range(3)])
    a, b, c = corners
    lo, hi = [], []
    for k in range(3):
        mn = np.fmin(a[k], np.fmin(b[k], c[k]))   # NaN operands ignored
        mx = np.fmax(a[k], np.fmax(b[k], c[k]))
        lo.append(min(max(_f2i(np.floor(mn)), 0), dims[k] - 1))
        hi.append(min(max(_f2i(np.ceil(mx)), 0), dims[k] - 1))
    xs, zs, ys = np.meshgrid(np.arange(lo[0], hi[0] + 1), np.arange(lo[2], hi[2] + 1), np.arange(lo[1], hi[1] + 1), indexing="ij")
    xs, ys, zs = xs.ravel(), ys.ravel(), zs.ravel()
    vox = [xs.astype(F) + F(0.5), ys.astype(F) + F(0.5), zs.astype(F) + F(0.5)]
    va = [vox[k] - a[k] for k in range(3)]
    d = _dot(va, n)
    p = [vox[k] - n[k] * d for k in range(3)]
    p2 = [p[k] - a[k] for k in range(3)]
    p0 = [b[k] - a[k] for k in range(3)]
    p1 = [c[k] - a[k] for k in range(3)]
    d00, d01, d11 = _dot(p0, p0), _dot(p0, p1), _dot(p1, p1)
    d20, d21 = _dot(p2, p0), _dot(p2, p1)
    denom = F(1.0) / (d00 * d11 - d01 * d01)
    by = (d11 * d20 - d01 * d21) * denom
    bz = (d00 * d21 - d01 * d20) * denom
    bx = F(1.0) - by - bz
    reject = (np.abs(d) > F(0.5)) | (bx < 0) | (by < 0) | (bz < 0) | (bx > 1) | (by > 1) | (bz > 1)
    keep = np.nonzero(~reject)[0]
    total = len(keep)
    keep = keep[:VOXELIZE_BUFFER_MAX]
    bx, by, bz = bx[keep], by[keep], bz[keep]
    cf = cols[:, :3].astype(F) / F(255.0)
    argb = np.full(len(keep), 255, dtype=np.uint32)
    for k in range(3):
        ch = cf[0, k] * bx + cf[1, k] * by + cf[2, k] * bz
        argb |= to_byte(ch) << np.uint32(8 * (k + 1))
    return xs[keep], ys[keep], zs[keep], argb, total


def voxelize(xyz: np.ndarray, colors32: np.ndarray, dims):
    """All triangles: voxel records (x, y, z, argb) and the per-triangle voxel counts before the VOXELIZE_BUFFER_MAX cut."""
    xyz = np.asarray(xyz, dtype=F).reshape(-1, 3, 3)
    colors32 = np.asarray(colors32, dtype=np.uint8).reshape(-1, 3, 4)
    parts, totals = [], []
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        for t in range(xyz.shape[0]):
            *rec, total = voxelize_triangle(xyz[t], colors32[t], dims)
            parts.append(rec)
            totals.append(total)
    cat = [np.concatenate([p[i] for p in parts]) if parts else np.zeros(0) for i in range(4)]
    return (cat[0].astype(np.int64), cat[1].astype(np.int64), cat[2].astype(np.int64), cat[3].astype(np.uint32)), np.array(totals, dtype=np.int64)


def merge(x, y, z, argb, dims):
    """Unique voxels sorted by (x, z, y): per channel the integer mean of the records, alpha of the first record."""
    key = (x.astype(np.int64) * dims[2] + z) * dims[1] + y
    order = np.argsort(key, kind="stable")
    key, argb = key[order], argb[order]
    uk, first, cnt = np.unique(key, return_index=True, return_counts=True)
    out = argb[first] & np.uint32(0xFF)
    for k in range(3):
        s = np.add.reduceat(((argb >> np.uint32(8 * (k + 1))) & np.uint32(0xFF)).astype(np.int64), first) if len(key) else np.zeros(0, np.int64)
        out |= ((s // cnt).astype(np.uint32) & np.uint32(0xFF)) << np.uint32(8 * (k + 1))
    y = uk % dims[1]
    col = uk // dims[1]
    return col // dims[2], y, col % dims[2], out


def lod_levels(dims, lods: int) -> int:
    """LODs both builders produce when `lods` are asked for: they stop at the first LOD where an axis reaches 0."""
    n = 0
    while n < lods and min(d >> n for d in dims) >= 1:
        n += 1
    return n


@dataclass
class RefWorld:
    dims: Tuple[int, int, int]
    voxels: List[tuple] = field(default_factory=list)       # per LOD: (x, y, z, argb) of the unique voxels
    blobs: List[np.ndarray] = field(default_factory=list)
    column_counts: List[int] = field(default_factory=list)
    voxel_counts: List[int] = field(default_factory=list)
    triangle_voxels: np.ndarray = None                      # per triangle, before the VOXELIZE_BUFFER_MAX cut


def grid_of(vox, dims, lod: int) -> np.ndarray:
    x, y, z, argb = vox
    g = np.zeros((dims[0] >> lod, dims[1] >> lod, dims[2] >> lod), dtype=np.uint32)
    g[x, y, z] = argb
    return g


def blob(vox, dims, lod: int) -> Tuple[np.ndarray, int]:
    """The LOD blob exactly as the builders write it: columns in index order, runs top -> bottom with ColorsIndex and Length
    stored as int16 (a 32768-voxel run wraps to Length -32768), the element area zero-filled to the WorldAllocator capacity
    (columnCount * 4 cells, doubled until the elements fit)."""
    enc, cc = encode_world(grid_of(vox, dims, lod), lod)
    assert cc == column_count(dims[0], dims[2], lod)
    cells = enc[12 * cc:]
    used = len(cells) // 4 if len(vox[0]) else 0
    capacity = cc * 4
    while capacity < used:
        capacity = min(capacity * 2, 2**31 - 1)
    out = np.zeros(12 * cc + 4 * capacity, dtype=np.uint8)
    out[:12 * cc] = enc[:12 * cc]
    out[12 * cc:12 * cc + 4 * used] = cells[:4 * used]
    return out, cc


def downsample(vox0, dims, lod: int):
    x, y, z, argb = vox0
    return merge(x >> lod, y >> lod, z >> lod, argb, (dims[0] >> lod, dims[1] >> lod, dims[2] >> lod))


def build(positions: np.ndarray, colors32: np.ndarray, max_dimension: int, flips=(False, False, False), lods: int = 6,
          blobs: bool = True) -> RefWorld:
    """The whole pipeline: remap, voxelize, merge, LOD mips, blobs (blobs=False keeps only the voxel sets)."""
    xyz, dims = remap(positions, max_dimension, flips)
    cols = np.ascontiguousarray(colors32, dtype=np.uint8).reshape(-1, 4)
    ntri = xyz.shape[0] // 3
    (x, y, z, argb), totals = voxelize(xyz[:3 * ntri], cols[:3 * ntri], dims)
    w = RefWorld(dims, triangle_voxels=totals)
    vox0 = merge(x, y, z, argb, dims)
    for lod in range(lod_levels(dims, lods)):
        v = vox0 if lod == 0 else downsample(vox0, dims, lod)
        w.voxels.append(v)
        w.voxel_counts.append(len(v[0]))
        w.column_counts.append(column_count(dims[0], dims[2], lod))
        if blobs:
            w.blobs.append(blob(v, dims, lod)[0])
    return w
