"""Swept-box queries against the resident world (cvx_sweep; DESIGN.md §3.6).

CPU: the cell-by-cell definition (tools/raycast_oracle) against an independent float64 brute force, the kernel's traversal (raycast.h
compiled for the CPU) against the definition bit for bit, properties that relate a sweep to ray queries and to itself, and invalid
boxes. GPU: cvx_sweep against the definition and the CPU build of its traversal, ordering and errors."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from conftest import MILL, comb_world, irregular_world, limited, parse_obj
import raycast_oracle as rco
import sweep_oracle as swo
from test_raycast import decode_cells, fuzz_worlds, pick_rays

# ---- fixtures and helpers ---------------------------------------------------------------------------------------------------


def random_boxes(rng, dims, n, cell=1.0, max_cells=None, snapped=0.0):
    """Boxes inside and around the world with half extents from 1/16 cell to 4 cells, random and axis-parallel directions,
    max_distance cut-offs (at most max_cells cells when given). A share `snapped` of them sits on a quarter-cell grid with quarter-cell
    extents and directions of components -1, 0, 1: faces that touch cell faces, and many cells entered at the same time."""
    dims = np.array(dims, dtype=np.float64)
    inside = rng.random(n) < 0.7
    c = np.where(inside[:, None], rng.uniform(0, 1, (n, 3)) * dims, rng.uniform(-0.3, 1.3, (n, 3)) * dims)
    d = rng.normal(size=(n, 3))
    par = rng.random(n)
    d[par < 0.15, rng.integers(0, 3)] = 0.0
    for i in np.nonzero((par >= 0.15) & (par < 0.25))[0]:
        k = rng.integers(0, 3)
        v = d[i, k]
        d[i] = 0.0
        d[i, k] = v if v != 0 else 1.0
    aim = (rng.random(n) < 0.3) & ~inside
    d[aim] = (rng.uniform(0, 1, (n, 3)) * dims - c)[aim]
    h = np.exp(rng.uniform(np.log(1 / 16), np.log(4), (n, 3))) * cell
    if max_cells is None:
        md = np.where(rng.random(n) < 0.5, np.inf, rng.uniform(0, 1.2, n) * dims.max())
    else:
        md = rng.uniform(0, max_cells, n) * cell
    boxes = np.zeros(n, dtype=swo.BOX_DTYPE)
    boxes["center"] = c
    boxes["direction"] = d
    boxes["half_extent"] = h
    boxes["max_distance"] = md
    snap = rng.random(n) < snapped
    q = 0.25 * cell
    boxes["center"][snap] = np.round(c[snap] / q) * q
    boxes["half_extent"][snap] = np.maximum(np.round(h[snap] / q), 1) * q
    boxes["direction"][snap] = rng.integers(-1, 2, (int(snap.sum()), 3))
    boxes["direction"][snap & ~np.any(boxes["direction"] != 0, axis=1), 1] = -1.0
    return boxes


def same(a, b, steps=True):
    """Bit-for-bit equality of two hit arrays; steps=False leaves `steps` (a cost figure of the kernel) out."""
    a, b = np.ascontiguousarray(a).copy(), np.ascontiguousarray(b).copy()
    if not steps:
        a["steps"] = 0
        b["steps"] = 0
    return a.view(np.uint8).tobytes() == b.view(np.uint8).tobytes()


def first_mismatch(boxes, a, b, steps=True):
    aa, bb = np.ascontiguousarray(a).view(np.uint32).reshape(-1, 8), np.ascontiguousarray(b).view(np.uint32).reshape(-1, 8)
    cols = slice(0, 8) if steps else slice(0, 7)
    bad = np.nonzero(np.any(aa[:, cols] != bb[:, cols], axis=1))[0]
    if len(bad) == 0:
        return None
    i = int(bad[0])
    return f"{len(bad)} boxes differ; first {i}: box {boxes[i]} -> {a[i]} vs {b[i]}"


def brute_force(solid, colours, box):
    """Independent float64 evaluation of §3.6 over the solid cells (n, 3) of a LOD-0 grid. Returns (hit, cell, face, colour,
    distance, ambiguous); ambiguous when a solid cell that could compete lies within 1e-4 of a window edge or a tie."""
    c = np.array(box["center"], dtype=np.float64)
    h = np.array(box["half_extent"], dtype=np.float64)
    dr = np.array(box["direction"], dtype=np.float64)
    md = float(box["max_distance"])
    d = dr / np.linalg.norm(dr)
    tol = lambda t: 1e-4 * (1 + np.abs(t))  # noqa: E731
    enter, exit_ = np.empty((3, len(solid))), np.empty((3, len(solid)))
    edge = np.zeros(len(solid), dtype=bool)
    for i in range(3):
        lo, hi = solid[:, i] - h[i], solid[:, i] + 1 + h[i]
        if d[i] == 0:
            reach = (lo < c[i]) & (c[i] < hi)
            enter[i] = np.where(reach, -np.inf, np.inf)
            exit_[i] = np.where(reach, np.inf, -np.inf)
            edge |= np.minimum(np.abs(lo - c[i]), np.abs(hi - c[i])) < 1e-4
        else:
            a, b = (lo - c[i]) / d[i], (hi - c[i]) / d[i]
            enter[i], exit_[i] = np.minimum(a, b), np.maximum(a, b)
    order = [0, 2, 1]
    e = enter[order]
    T = e.max(axis=0)
    Tp = exit_.min(axis=0)
    ts = np.maximum(T, 0.0)
    with np.errstate(invalid="ignore"):
        edge |= (np.abs(T - Tp) < tol(Tp)) | (np.abs(Tp) < tol(Tp)) | (np.abs(T) < tol(T))
        if np.isfinite(md):
            edge |= np.abs(ts - md) < tol(md)
    cand = (T < Tp) & (Tp > 0) & (ts <= md) & np.isfinite(ts)
    if not cand.any():
        return 0, None, None, None, None, bool(edge.any())
    ov = T < 0
    idx = np.nonzero(cand)[0]
    k = idx[np.lexsort((solid[idx, 1], solid[idx, 2], solid[idx, 0], ~ov[idx], ts[idx]))[0]]
    bt = ts[k]
    near = ts <= bt + tol(bt)
    amb = bool((edge & near).any()) or bool(np.any(cand & (ts != bt) & near))
    srt = np.sort(e[:, k])
    if np.isfinite(srt[1]) and srt[2] - srt[1] < tol(srt[2]):
        amb = True                                                    # entry axis
    axis = order[int(np.argmax(e[:, k]))]
    face = 6 if ov[k] else 2 * axis + (0 if d[axis] > 0 else 1)
    return 1, tuple(int(v) for v in solid[k]), face, int(colours[k]), float(bt), amb


def _check_against_brute_force(grid, world, boxes):
    hits = swo.sweep(rco.RayWorld(world), boxes)
    solid = np.argwhere(grid != 0)
    colours = grid[grid != 0]
    amb = 0
    for b, h in zip(boxes, hits):
        hit, cell, face, colour, dist, ambiguous = brute_force(solid, colours, b)
        if ambiguous:
            amb += 1
            continue
        assert h["hit"] == hit, (b, h, hit, cell, face, dist)
        if hit == 1:
            assert (tuple(h["cell"]), int(h["face"]), int(h["color"])) == (cell, face, colour), (b, h, cell, face, dist)
            assert abs(float(h["distance"]) - dist) <= 1e-4 * (1 + dist), (b, h, dist)
        else:
            assert h["face"] == 0 and h["distance"] == 0 and h["color"] == 0 and tuple(h["cell"]) == (0, 0, 0)
    return amb


def _emu_equals_definition(world, boxes, lods=None):
    from emu import EmuWorld
    ew, rw = EmuWorld(world), rco.RayWorld(world)
    for lod in range(len(world.blobs)) if lods is None else lods:
        ref = swo.sweep(rw, boxes, lod)
        assert np.any(ref["hit"] == 1) and np.any(ref["hit"] == 0)
        assert np.all(ref["steps"] == 0)
        for general in (False, True):
            got = swo.emu_sweep(ew, boxes, lod, general)
            assert same(got, ref, steps=False), (lod, general, first_mismatch(boxes, got, ref, steps=False))


def _lod_boxes(world, seed, n=10000, max_cells=64):
    """Per LOD, boxes whose sizes and cut-offs are in that LOD's cells (the definition is a brute force over the swept box)."""
    return [random_boxes(np.random.default_rng(seed + lod), world.dims, n, cell=float(1 << lod), max_cells=max_cells, snapped=0.3)
            for lod in range(len(world.blobs))]


def _flat_world(cv, dims=(16, 16, 16), floor=4):
    """A solid floor of `floor` cells (y < floor) under air."""
    from rle import encode_world
    grid = np.zeros(dims, dtype=np.uint32)
    grid[:, :floor, :] = 0xFF336699
    blob, cc = encode_world(grid)
    return cv.World(dims, [blob], [cc], [int((grid != 0).sum())])


# ---- CPU ----------------------------------------------------------------------------------------------------------------------

def test_box_struct_layout(cv):
    from cpuvox_b200 import native as N
    assert C.sizeof(N.Box) == 48
    assert [(f, getattr(N.Box, f).offset) for f, _ in N.Box._fields_] == [
        ("center", 0), ("max_distance", 12), ("direction", 16), ("reserved0", 28), ("half_extent", 32), ("reserved1", 44)]
    assert cv.BOX_DTYPE.itemsize == 48 and cv.BOX_DTYPE == swo.BOX_DTYPE
    b = cv.make_boxes([[1, 2, 3]], [0.5, 1.0, 1.5], [[0, -1, 0]], 7.0)
    assert b["half_extent"].tolist() == [[0.5, 1.0, 1.5]] and b["max_distance"][0] == 7.0 and b["direction"][0, 1] == -1.0


def test_definition_matches_float64_brute_force(cv):
    rng = np.random.default_rng(21)
    total = amb = 0
    for (world, blob, cc), n in ((comb_world(cv), 400), (irregular_world(cv), 2000)):
        boxes = random_boxes(rng, world.dims, n)
        amb += _check_against_brute_force(decode_cells(blob, cc, world.dims), world, boxes)
        total += n
    for world, blob, cc, _ in fuzz_worlds(cv):
        boxes = random_boxes(rng, world.dims, 200)
        amb += _check_against_brute_force(decode_cells(blob, cc, world.dims), world, boxes)
        total += len(boxes)
    print(f"skipped {amb} of {total}")
    assert amb < 0.01 * total, (amb, total)


def test_kernel_traversal_equals_definition_small_worlds(cv):
    rng = np.random.default_rng(22)
    for world, _, _ in (comb_world(cv), irregular_world(cv)):
        _emu_equals_definition(world, random_boxes(rng, world.dims, 10000, snapped=0.3))
    for world, _, _, _ in fuzz_worlds(cv):
        _emu_equals_definition(world, random_boxes(rng, world.dims, 200, snapped=0.3))


@pytest.mark.parametrize("name", ["mill_world", "terrain_world", "structure_world"])
def test_kernel_traversal_equals_definition_every_lod(cv, request, name):
    from emu import EmuWorld
    world = request.getfixturevalue(name)
    ew, rw = EmuWorld(world), rco.RayWorld(world)
    for lod, boxes in enumerate(_lod_boxes(world, 23)):
        ref = swo.sweep(rw, boxes, lod)
        assert np.any(ref["hit"] == 1) and np.any(ref["face"] == 6)
        for general in (False, True):
            got = swo.emu_sweep(ew, boxes, lod, general)
            assert same(got, ref, steps=False), (lod, general, first_mismatch(boxes, got, ref, steps=False))


def test_sweep_is_not_farther_than_the_centre_ray(cv, mill_world):
    rw = rco.RayWorld(mill_world)
    boxes = random_boxes(np.random.default_rng(24), mill_world.dims, 4000, max_cells=64)
    rays = cv.make_rays(boxes["center"], boxes["direction"], boxes["max_distance"])
    rh, sh = rco.raycast(rw, rays), swo.sweep(rw, boxes)
    ray_hit = rh["hit"] == 1
    assert ray_hit.sum() > 200
    assert np.all(sh["hit"][ray_hit] == 1)
    t = rh["distance"][ray_hit].astype(np.float64)
    assert np.all(sh["distance"][ray_hit] <= t + 1e-4 * (1 + t))
    inside = ray_hit & (rh["face"] == 6)
    assert inside.sum() > 10 and np.all(sh["face"][inside] == 6) and np.all(sh["distance"][inside] == 0)


def test_box_moved_to_its_hit_does_not_overlap(cv, mill_world, terrain_world):
    for world in (mill_world, terrain_world):
        rw = rco.RayWorld(world)
        for lod in (0, 2):
            s = float(1 << lod)
            boxes = random_boxes(np.random.default_rng(25 + lod), world.dims, 3000, cell=s, max_cells=64)
            hits = swo.sweep(rw, boxes, lod)
            moved = (hits["hit"] == 1) & (hits["face"] != 6) & (hits["distance"] > 1e-2 * s)
            assert moved.sum() > 100
            b = boxes[moved].copy()
            d = b["direction"].astype(np.float64)
            d /= np.linalg.norm(d, axis=1)[:, None]
            t = hits["distance"][moved].astype(np.float64) - 1e-3 * s
            b["center"] = b["center"] + t[:, None] * d
            b["max_distance"] = 0.0
            again = swo.sweep(rw, b, lod)
            assert not np.any(again["face"] == 6), np.nonzero(again["face"] == 6)[0][:5]


def test_box_resting_on_a_floor_slides(cv):
    world = _flat_world(cv)
    rw = rco.RayWorld(world)
    # bottom face exactly on y = 4 (fp-exact: 4.5 - 0.5), moving along the floor in every horizontal direction
    dirs = [(1, 0, 0), (-1, 0, 0), (0, 0, 1), (0, 0, -1), (1, 0, 1), (-0.3, 0, 0.7)]
    boxes = cv.make_boxes([(8.0, 4.5, 8.0)] * len(dirs), (0.5, 0.5, 0.5), dirs, np.inf)
    hits = swo.sweep(rw, boxes)
    assert np.all(hits["hit"] == 0), hits
    # moving down it touches at once: distance 0 through the top face of the floor cell under its lowest x, z
    down = swo.sweep(rw, cv.make_boxes([(8.25, 4.5, 8.75)], (0.5, 0.5, 0.5), [(0, -1, 0)]))[0]
    assert (down["hit"], down["face"], down["distance"], tuple(down["cell"])) == (1, 3, 0.0, (7, 3, 8))
    # the same box lowered by a hair overlaps the floor: face 6
    sunk = swo.sweep(rw, cv.make_boxes([(8.0, 4.49, 8.0)], (0.5, 0.5, 0.5), [(1, 0, 0)]))[0]
    assert sunk["hit"] == 1 and sunk["face"] == 6 and sunk["distance"] == 0.0
    from emu import EmuWorld
    all_boxes = np.concatenate([boxes, cv.make_boxes([(8.25, 4.5, 8.75), (8.0, 4.49, 8.0)], (0.5, 0.5, 0.5), [(0, -1, 0), (1, 0, 0)])])
    for general in (False, True):
        assert same(swo.emu_sweep(EmuWorld(world), all_boxes, 0, general), swo.sweep(rw, all_boxes), steps=False)


def test_height_not_divisible_stacks_from_zero(cv):
    """dim_y = 13 at LOD 2: 3 cells of 4 units stacked from y = 0 ([0, 12)), the band [12, 13) is outside the LOD (§3.5)."""
    from rle import encode_world
    from test_world_heights import lod_grid
    dims = (8, 13, 8)
    grid = np.full(dims, 0xFF00FF00, dtype=np.uint32)
    grids = [lod_grid(grid, j) for j in range(3)]
    enc = [encode_world(g, j) for j, g in enumerate(grids)]
    world = cv.World(dims, [b for b, _ in enc], [c for _, c in enc], [int((g != 0).sum()) for g in grids])
    rw = rco.RayWorld(world)
    assert world.dims[1] >> 2 == 3
    # a box falling from above touches the top of cell 2 at y = 12, not at 13
    h = swo.sweep(rw, cv.make_boxes([(4.0, 20.0, 4.0)], (1.0, 1.0, 1.0), [(0, -1, 0)]), 2)[0]
    assert (h["hit"], h["face"], h["cell"][1]) == (1, 3, 2) and h["distance"] == 20.0 - 1.0 - 12.0
    # a box inside the band [12, 13) overlaps nothing at LOD 2 but the top LOD-0 layer
    band = cv.make_boxes([(4.0, 12.6, 4.0)], (0.25, 0.25, 0.25), [(1, 0, 0)], 0.0)
    assert swo.sweep(rw, band, 2)[0]["hit"] == 0 and swo.sweep(rw, band, 0)[0]["face"] == 6
    from emu import EmuWorld
    boxes = random_boxes(np.random.default_rng(26), dims, 2000)
    for lod in range(len(world.blobs)):
        assert same(swo.emu_sweep(EmuWorld(world), boxes, lod), swo.sweep(rw, boxes, lod), steps=False)


def test_invalid_boxes(cv, mill_world):
    from emu import EmuWorld
    nan, inf = np.nan, np.inf
    good = dict(center=(100.0, 100.0, 100.0), half=(1.0, 1.0, 1.0), dir=(0.0, -1.0, 0.0), md=inf)
    cases = []
    for i in range(3):
        for v in (nan, inf, -inf):
            for key in ("center", "half", "dir"):
                x = dict(good)
                t = list(x[key])
                t[i] = v
                x[key] = tuple(t)
                cases.append(x)
        for v in (0.0, -0.0, -1.0):
            x = dict(good)
            t = list(x["half"])
            t[i] = v
            x["half"] = tuple(t)
            cases.append(x)
    cases += [dict(good, md=nan), dict(good, md=-inf), dict(good, dir=(0.0, 0.0, 0.0)), dict(good, dir=(1e30, 1e30, 0.0)),
              dict(good, dir=(1e-30, 0.0, -1e-30))]
    boxes = np.zeros(len(cases), dtype=swo.BOX_DTYPE)
    for k, x in enumerate(cases):
        boxes[k] = (x["center"], x["md"], x["dir"], 0, x["half"], 0)
    expect = np.zeros(len(cases), dtype=rco.RAY_HIT_DTYPE)
    expect["hit"] = -1
    ref = swo.sweep(rco.RayWorld(mill_world), boxes)
    assert same(ref, expect), first_mismatch(boxes, ref, expect)
    for general in (False, True):
        assert same(swo.emu_sweep(EmuWorld(mill_world), boxes, 0, general), expect)


# ---- GPU ----------------------------------------------------------------------------------------------------------------------

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def rm(cv):
    r = cv.RenderManager(0)
    yield r
    r.destroy()


def _device_sweep(rm, boxes, lod):
    import torch
    t_boxes = torch.from_numpy(np.ascontiguousarray(boxes).view(np.uint8).copy()).cuda()
    t_hits = torch.zeros(len(boxes) * 32, dtype=torch.uint8, device="cuda")
    rm.sweep_device(t_boxes.data_ptr(), t_hits.data_ptr(), len(boxes), lod)
    rm.sync()
    return t_hits.cpu().numpy().view(rco.RAY_HIT_DTYPE)


def _gpu_equals_definition(rm, world, boxes_per_lod):
    from emu import EmuWorld
    rm.upload_world(world)
    rw, ew = rco.RayWorld(world), EmuWorld(world)
    for lod, boxes in enumerate(boxes_per_lod):
        ref = swo.sweep(rw, boxes, lod)
        for general in (False, True):
            rm.set_general_path(general)
            emu = swo.emu_sweep(ew, boxes, lod, general)
            got = rm.sweep_boxes(boxes, lod)
            assert same(got, ref, steps=False), (lod, general, first_mismatch(boxes, got, ref, steps=False))
            assert same(got, emu), (lod, general, first_mismatch(boxes, got, emu))
            got = _device_sweep(rm, boxes, lod)
            assert same(got, emu), ("device", lod, general, first_mismatch(boxes, got, emu))
    rm.set_general_path(False)


@gpu
def test_gpu_sweep_equals_definition_small_worlds(cv, rm):
    rng = np.random.default_rng(22)
    for world, _, _ in (comb_world(cv), irregular_world(cv)):
        _gpu_equals_definition(rm, world, [random_boxes(rng, world.dims, 10000, snapped=0.3)])
    for world, _, _, _ in fuzz_worlds(cv, 30):
        _gpu_equals_definition(rm, world, [random_boxes(rng, world.dims, 200, snapped=0.3)])


@gpu
@pytest.mark.parametrize("name", ["mill_world", "terrain_world", "structure_world"])
def test_gpu_sweep_equals_definition_every_lod(cv, rm, request, name):
    world = request.getfixturevalue(name)
    _gpu_equals_definition(rm, world, _lod_boxes(world, 23))


@gpu
def test_gpu_sweep_mill1024_resident(cv):
    from emu import EmuWorld
    r = cv.RenderManager(0)
    try:
        P, Cc = parse_obj(MILL)
        host = r.build_world_from_mesh(P, Cc, 1024, flips=(True, False, False))
        r.build_resident_world_from_mesh(P, Cc, 1024, flips=(True, False, False))
        rw, ew = rco.RayWorld(host), EmuWorld(host)
        W, H = 640, 360
        for k in range(6):
            pose = limited(cv, cv.benchmark_pose(cv.benchmark_length() * k / 5, host.dims, far_clip=2048.0))
            _, _, rays = pick_rays(cv, pose, W, H, stride=9)
            n = len(rays)
            # start up to 32 units short of what the pick ray hits, so that most boxes reach the surface within max_distance
            t = rco.raycast(rw, rays)["distance"].astype(np.float64)
            d = rays["direction"] / np.linalg.norm(rays["direction"], axis=1)[:, None]
            start = rays["origin"] + np.maximum(t - 32.0, 0.0)[:, None] * d
            for half in ((0.3, 0.9, 0.3), (2.0, 2.0, 2.0)):        # a character, a box 4 cells across
                boxes = cv.make_boxes(start, np.tile(half, (n, 1)), rays["direction"], 64.0)
                got = r.sweep_boxes(boxes)
                assert same(got, swo.sweep(rw, boxes), steps=False), (k, half)
                assert same(got, swo.emu_sweep(ew, boxes)), (k, half)
                assert np.mean(got["hit"] == 1) > 0.05, (k, half)
    finally:
        r.destroy()


@gpu
def test_gpu_sweep_ordering_and_errors(cv, terrain_world, structure_world):
    from cpuvox_b200 import native as N
    r = cv.RenderManager(0)
    try:
        box = cv.make_boxes([[1.0, 300.0, 1.0]], (0.5, 0.5, 0.5), [[0.1, -1.0, 0.2]])
        hit = np.zeros(1, dtype=cv.RAY_HIT_DTYPE)
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        assert N.lib.cvx_sweep(r._ctx, p(box), 1, 0, p(hit), 0) == -5        # CVX_ERR_NO_WORLD
        w4 = cv.World(terrain_world.dims, terrain_world.blobs[:4], terrain_world.column_counts[:4])
        r.upload_world(w4)
        assert N.lib.cvx_sweep(r._ctx, p(box), 1, 4, p(hit), 0) == -1         # LOD 4 not uploaded
        assert N.lib.cvx_sweep(r._ctx, p(box), 1, 6, p(hit), 0) == -1
        assert N.lib.cvx_sweep(r._ctx, p(box), -1, 0, p(hit), 0) == -1
        assert N.lib.cvx_sweep(r._ctx, None, 1, 0, p(hit), 0) == -1
        assert N.lib.cvx_sweep(r._ctx, p(box), 1, 0, None, 1) == -1
        launches = r.launch_count()
        assert N.lib.cvx_sweep(r._ctx, None, 0, 0, None, 0) == 0 and r.launch_count() == launches
        rw = rco.RayWorld(w4)
        assert same(r.sweep_boxes(box), swo.sweep(rw, box), steps=False)
        assert r.sweep_boxes(box)["hit"][0] == 1
        # scratch growth alternating with cvx_raycast: 2 M boxes, 3 M rays, then small calls reusing the scratch
        big = random_boxes(np.random.default_rng(9), w4.dims, 2_000_000, max_cells=8)
        assert same(r.sweep_boxes(big, 1), swo.sweep(rw, big, 1), steps=False)
        rays = cv.make_rays(np.random.default_rng(8).uniform(0, 256, (3_000_000, 3)), np.random.default_rng(7).normal(size=(3_000_000, 3)))
        assert np.array_equal(r.raycast_rays(rays, 1), rco.raycast(rw, rays, 1))
        assert same(r.sweep_boxes(big[:1000], 2), swo.sweep(rw, big[:1000], 2), steps=False)
        assert np.array_equal(r.raycast_rays(rays[:1000], 2), rco.raycast(rw, rays[:1000], 2))
        # a sweep issued while two asynchronous batches are outstanding
        W, H = 640, 360
        r.set_resolution(W, H)
        poses = [cv.CameraPose.from_euler((128.0, 200.0 + 5 * i, 128.0), (50.0, 20.0 * i, 0.0), far_clip=512.0) for i in range(8)]
        setups = [r.make_setup(q) for q in poses]
        dst = [cv.alloc_pinned((len(setups), H, W)) for _ in range(2)]
        b0 = r.draw_batch_async(setups[:4], dst[0])
        b1 = r.draw_batch_async(setups[4:], dst[1])
        boxes = random_boxes(np.random.default_rng(10), w4.dims, 100000)
        got = r.sweep_boxes(boxes)
        r.batch_wait(b0)
        r.batch_wait(b1)
        assert same(got, swo.sweep(rw, boxes), steps=False)
        for i, s in enumerate(setups):
            r.draw_setup(s)
            r.sync()
            assert np.array_equal(r.read_frame(), dst[i // 4][i % 4]), i
        # a world replacement is seen by the next query (host and device paths)
        r.upload_world(structure_world)
        bs = random_boxes(np.random.default_rng(11), structure_world.dims, 20000, max_cells=64)
        ref = swo.sweep(rco.RayWorld(structure_world), bs)
        assert same(r.sweep_boxes(bs), ref, steps=False)
        assert same(_device_sweep(r, bs, 0), ref, steps=False)
        h = r.sweep([[256.0, 500.0, 128.0]], (2.0, 2.0, 2.0), [[0.0, -1.0, 0.0]])
        assert same(h, swo.sweep(rco.RayWorld(structure_world), cv.make_boxes([[256.0, 500.0, 128.0]], (2.0, 2.0, 2.0), [[0.0, -1.0, 0.0]])),
                    steps=False)
    finally:
        r.destroy()
