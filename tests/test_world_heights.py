"""Worlds whose height is not a power of two.

`cvx_world_upload` takes any height from 1 to 32768 (only X and Z must be powers of two), and `.world` files and host-built blobs
reach it, while the builders only make power-of-two worlds. Such heights run code nothing else runs: the boundary projection's
`unlerp(0, worldMaxY, y)` branch (`y_pow2 == 0`), and LODs whose cell size 2^j does not divide the height. A LOD-j column then
covers (dim_y >> j) << j world units, short of dim_y by dim_y mod 2^j, so the LOD is irregular (world_transcode.h) and the two run
iteration directions of the renderer place it differently: looking down (runs stacked from dim_y) it sits dim_y mod 2^j higher than
looking up (stacked from 0), as in the reference. A ray query stacks it from 0 (DESIGN.md §3.5).

Worlds are made here from numpy grids with one downsampling rule (`lod_grid`), one blob per LOD, and every implementation is
compared on the same blobs: the oracle against oracle/pyref.py and the reference's own code, the kernel source through the SIMT
emulator against the oracle, the transcode verdict against a numpy statement of the rule, the ray-query definition against a float64
brute force, and on the GPU the CUDA kernels against all of these."""
from __future__ import annotations

import itertools

import numpy as np
import pytest

import emu
import raycast_oracle as rco
from rle import encode_world
from test_degenerate_rays import MAGENTA, _assert_same, _gpu_frame, _oracle_frame
from test_raycast import _device_raycast, brute_force, first_mismatch, random_rays, same

F32 = np.float32
LODS = 6
# (dim_y, dim_x, dim_z): the heights under test, 32 and 256 as power-of-two controls; X != Z in both orders
BASES = [(3, 16, 8), (5, 8, 16), (7, 32, 32), (32, 16, 16), (96, 32, 16), (100, 16, 32), (127, 32, 32), (129, 8, 64),
         (255, 64, 8), (256, 16, 16), (257, 16, 8), (384, 32, 32), (1000, 16, 16), (4095, 16, 8), (32767, 8, 8)]
W, H = 20, 14          # screen of every case but the tiny ones
TINY = (3, 2)          # screen drawn at every group width, counters on and off


# ---- worlds ----------------------------------------------------------------------------------------------------------------------
def _colour(rng, n):
    return rng.integers(1, 2 ** 32 - 1, size=n, dtype=np.uint64).astype(np.uint32) | 0xFF


def lod_grid(grid, j):
    """LOD j of a LOD-0 grid: cell (x, y, z) covers the 2^j cube at (x, y, z) << j and takes the colour of the cube's first solid
    voxel in C order (x, then y, then z). The grid has dim >> j cells per axis, so voxels at or above (dim_y >> j) << j belong to
    no cell."""
    s = 1 << j
    nx, ny, nz = (d >> j for d in grid.shape)
    g = grid[:nx * s, :ny * s, :nz * s].reshape(nx, s, ny, s, nz, s).transpose(0, 2, 4, 1, 3, 5).reshape(nx, ny, nz, s ** 3)
    first = (g != 0).argmax(axis=-1)
    return np.take_along_axis(g, first[..., None], -1)[..., 0]


def lod_count(dims):
    """LODs that exist: every axis keeps at least one cell."""
    return next(j for j in range(LODS + 1) if j == LODS or min(d >> j for d in dims) < 1)


def divisible_lods(dims):
    """The LODs from 0 up to the first one whose 2^j does not divide dim_y (those a regular world may have)."""
    n = lod_count(dims)
    return next(j for j in range(n + 1) if j == n or dims[1] % (1 << j))


def boundary_level(dy, top):
    """An integer height in [1, top] at which y / dim_y and y * (1 / dim_y) round differently in fp32 (the boundary-table kernel
    must take the division there), else top // 2."""
    for y in range(max(1, top // 3), top + 1):
        if F32(y) / F32(dy) != F32(y) * (F32(1) / F32(dy)):
            return y
    return max(1, top // 2)


def make_grid(dims, seed):
    """Heightmap of a few terraces (one at `boundary_level`) in a band at most 48 high, sparse voxels over the whole height, three
    floating boxes (overhangs: columns of several runs, undersides to look up at), one full-height column and one run that ends in
    the top cell. Every voxel has its own colour, so a vertical shift of the geometry changes what a ray sees."""
    rng = np.random.default_rng(seed)
    dx, dy, dz = dims
    grid = np.zeros(dims, dtype=np.uint32)
    top = min(dy - 1, 48) if dy > 1 else 1
    level = boundary_level(dy, top)
    levels = np.unique(np.clip([level, level + 1, level - 2, top // 4, top, 1], 1, top))
    hm = rng.choice(levels, size=(dx, dz))
    mask = np.arange(dy)[None, :, None] < hm[:, None, :]
    grid[mask] = _colour(rng, int(mask.sum()))
    n = min(400, dx * dy * dz // 40)
    grid[rng.integers(0, dx, n), rng.integers(0, dy, n), rng.integers(0, dz, n)] = _colour(rng, n)
    for _ in range(3):
        x, z = rng.integers(0, dx - 2), rng.integers(0, dz - 2)
        y = int(rng.integers(0, dy))
        box = grid[x:x + 3, y:y + 4, z:z + 3]
        box[...] = _colour(rng, box.size).reshape(box.shape)
    grid[dx - 2, :, dz - 2] = _colour(rng, dy)
    grid[1, max(0, dy - 5):, dz - 2] = _colour(rng, min(dy, 5))
    if dy > 8:
        grid[1, dy - 7, dz - 2] = 0
    return grid, level


class Base:
    """One grid, every LOD that exists encoded once; `world(n)` is the world of LODs 0 .. n - 1."""

    def __init__(self, cv, dims, seed):
        self.dims = dims
        self.grid, self.level = make_grid(dims, seed)
        self.grids = [lod_grid(self.grid, j) for j in range(lod_count(dims))]
        enc = [encode_world(g, j) for j, g in enumerate(self.grids)]
        self.blobs = [b for b, _ in enc]
        self.ccs = [c for _, c in enc]
        self.vox = [int((g != 0).sum()) for g in self.grids]
        self.cv = cv

    def world(self, n):
        return self.cv.World(self.dims, self.blobs[:n], self.ccs[:n], self.vox[:n])


def lod_sets(dims):
    """LOD 0 only; the divisible LODs (regular); one past them (irregular); every LOD that exists. Duplicates dropped."""
    n, v = lod_count(dims), divisible_lods(dims)
    return sorted({1, v, min(v + 1, n), n})


@pytest.fixture(scope="module")
def bases(cv):
    return {dims_y: Base(cv, (dx, dims_y, dz), 100 + i) for i, (dims_y, dx, dz) in enumerate(BASES)}


# ---- cameras ---------------------------------------------------------------------------------------------------------------------
def lod_distances(dims, n):
    """Distances (XZ plane) that switch LODs inside the world: n LODs over the first 2/3 of its XZ extent."""
    step = max(dims[0], dims[2]) / 3.0 / max(1, n - 1)
    return np.array([step * (k + 1) for k in range(n - 1)] + [1e9] * (LODS - n + 1), dtype=F32)


def cameras(dims, level):
    """(name, position, euler, far clip, screen): above the top, below 0, exactly at dim_y, at a fractional and at an integer height
    (the terrace level) in between; pitched down and up (both run iteration directions); outside the world at yaw 0 and 90 (a
    still axis enters through a face); a far clip inside the world; and one tiny screen."""
    dx, dy, dz = dims
    xz = float(max(dx, dz))
    far = 4.0 * xz
    cx, cz = dx * 0.5 + 0.3, dz * 0.5 + 0.2
    return [
        ("above", (cx, dy + 0.5 * xz, cz), (60.0, 30.0, 0.0), far, (W, H)),
        ("below", (cx - 1.1, -2.5, cz + 0.7), (-50.0, 200.0, 0.0), far, (W, H)),
        ("at_dim_y", (dx * 0.3, float(dy), dz * 0.7), (20.0, 120.0, 0.0), far, (W, H)),
        ("fraction_up", (dx * 0.6, dy * 0.37 + 0.21, dz * 0.4), (-15.0, 300.0, 0.0), far, (W, H)),
        ("level_down", (cx, float(level), cz), (10.0, 45.0, 0.0), far, (W, H)),
        ("level_up", (dx * 0.25, float(level), dz * 0.25), (-10.0, 225.0, 0.0), far, (W, H)),
        ("outside_yaw90", (-3.0, level + 3.0, dz * 0.5 + 0.5), (30.0, 90.0, 0.0), far, (W, H)),
        ("outside_yaw0", (dx * 0.5, float(level), -3.0), (-20.0, 0.0, 0.0), far, (W, H)),
        ("near_far_clip", (cx, level + 2.5, cz), (35.0, 160.0, 0.0), 6.0, (W, H)),
        ("tiny", (cx, level + 4.0, cz - 1.0), (40.0, 70.0, 0.0), far, TINY),
    ]


def corpus(cv, bases):
    """(key, world, case name, W, H, FrameSetup) for every base x LOD set x camera; key = (dim_y, LOD count)."""
    out = []
    for dy, b in bases.items():
        for n in lod_sets(b.dims):
            world = b.world(n)
            for name, pos, euler, far, (w, h) in cameras(b.dims, b.level):
                pose = cv.CameraPose.from_euler(pos, euler, far_clip=far)
                out.append(((dy, n), world, name, w, h, cv.frame_setup(pose, w, h, lod_distances(b.dims, n), dy, limit_horizon=False)))
    return out


@pytest.fixture(scope="module")
def cases(cv, bases):
    return corpus(cv, bases)


@pytest.fixture(scope="module")
def oracle_worlds(orc, bases):
    return {(dy, n): orc.OracleWorld(b.dims, b.blobs[:n], b.ccs[:n]) for dy, b in bases.items() for n in lod_sets(b.dims)}


def _tag(case):
    (dy, n), world, name, w, h, _ = case
    return f"{world.dims} LODs 0..{n - 1} camera {name} {w}x{h}"


def regular_rule(grid, dim_y, j):
    """world_transcode.h's verdict on an encoder-made LOD, stated on the grid: regular when 2^j divides dim_y or no column is solid."""
    return dim_y % (1 << j) == 0 or not grid.any()


# ---- the corpus reaches its edges ------------------------------------------------------------------------------------------------
def test_corpus_reaches_its_edges(cv, orc, bases, oracle_worlds, cases):
    """Minimum counts of the inputs this file exists for: regular worlds with a height that is not a power of two, worlds irregular
    only through non-divisible LODs, both run iteration directions on such LODs, and rays that switch into a non-divisible LOD."""
    regular_npow2 = irregular_by_lod = 0
    for dy, b in bases.items():
        for n in lod_sets(b.dims):
            ew = emu.EmuWorld(b.world(n))
            verdicts = [emu.transcode_verdict(b.blobs[j], b.ccs[j], b.dims, j) for j in range(n)]
            assert all(ok for ok, _, _ in verdicts)
            if ew.regular and dy & (dy - 1):
                regular_npow2 += 1
            if not ew.regular and all(reg == (dy % (1 << j) == 0) for j, (_, _, reg) in enumerate(verdicts)):
                irregular_by_lod += 1
    directions = {0: 0, 1: 0}
    switched = 0
    for case in cases:
        (dy, n), world, name, w, h, s = case
        nondiv = [j for j in range(n) if dy % (1 << j)]
        if not nondiv:
            continue
        directions[s.camera.inverse_element_iteration_direction] += 1
        st = orc.ray_setup(oracle_worlds[(dy, n)], orc.copy_setup(s), w, h)
        for r in st[::3]:
            if not np.isfinite(r["dir"]).all() or r["status"] != 0:
                continue
            cells, _ = orc.dda_walk(r["start"], r["dir"], s.camera.lod_distances[:], s.camera.far_clip, 4096)
            lods = cells[:, 2]
            if len(lods) > 1 and np.any((lods[1:] != lods[:-1]) & np.isin(lods[1:], nondiv)):
                switched += 1
    assert regular_npow2 >= 10, f"regular worlds whose height is not a power of two: {regular_npow2}"
    assert irregular_by_lod >= 8, f"worlds irregular only through LODs whose 2^j does not divide the height: {irregular_by_lod}"
    assert min(directions.values()) >= 40, f"cases per iteration direction on worlds with such LODs: {directions}"
    assert switched >= 100, f"rays that switch into such a LOD inside the world: {switched}"


# ---- CPU legs --------------------------------------------------------------------------------------------------------------------
def test_transcode_verdict_follows_the_divisibility_rule(bases):
    """world_transcode.h on every LOD of every base: accepted, and regular exactly when 2^j divides dim_y or the LOD is empty; plus
    an empty LOD of a non-divisible height, which stays regular."""
    seen = {True: 0, False: 0}
    for dy, b in bases.items():
        for j, g in enumerate(b.grids):
            ok, bad, regular = emu.transcode_verdict(b.blobs[j], b.ccs[j], b.dims, j)
            assert ok and bad == -1, (b.dims, j, bad)
            assert regular == regular_rule(g, dy, j), f"{b.dims} LOD {j}: verdict regular={regular}"
            seen[regular] += 1
    for dims, j in (((16, 100, 16), 3), ((8, 7, 8), 1)):
        g = np.zeros((dims[0] >> j, dims[1] >> j, dims[2] >> j), dtype=np.uint32)
        blob, cc = encode_world(g, j)
        assert emu.transcode_verdict(blob, cc, dims, j) == (True, -1, True), (dims, j)
    assert seen[True] >= 20 and seen[False] >= 15, seen


def test_oracle_equals_python_restatement(cv, orc, bases, oracle_worlds, cases):
    """oracle/cpuvox_oracle.cpp == oracle/pyref.py, raybuffers and frame, on the tiny screens and on the heights up to 129."""
    from oracle import pyref
    n = 0
    for case in cases:
        (dy, nl), world, name, w, h, s = case
        if not (name == "tiny" or (dy <= 129 and name in ("level_down", "outside_yaw90", "below"))):
            continue
        pw = [pyref.PyWorldLod(world.dims, l, b, c) for l, (b, c) in enumerate(zip(world.blobs, world.column_counts))]
        os_ = orc.copy_setup(s)
        otd, olr, _ = orc.render_raybuffers(oracle_worlds[(dy, nl)], os_, w, h)
        ptd, plr = pyref.render_raybuffers(pw, s, w, h)
        assert np.array_equal(otd, ptd), f"{_tag(case)}: top/down raybuffer differs in {int((otd != ptd).sum())} pixels"
        assert np.array_equal(olr, plr), f"{_tag(case)}: left/right raybuffer differs in {int((olr != plr).sum())} pixels"
        assert np.array_equal(orc.blit(os_, w, h, otd, olr), pyref.blit(s, w, h, ptd, plr)), f"{_tag(case)}: frame"
        n += 1
    assert n >= 60


def test_emulated_kernel_equals_oracle(cv, orc, oracle_worlds, cases):
    """The Phase-1 kernel source through the SIMT emulator == the oracle, raybuffers and counters, on every case: the boundary-table
    kernel where the world is regular, the general kernel everywhere, and on the tiny screens at 32, 16 and 8 lanes with the counters
    compiled in and out."""
    ews = {}
    for case in cases:
        key, world, name, w, h, s = case
        if key not in ews:
            ews[key] = emu.EmuWorld(world)
        ew = ews[key]
        otd, olr, ocn, _ = _oracle_frame(orc, oracle_worlds[key], s, w, h, MAGENTA)
        tiny = name == "tiny"
        for variant, group, counters in itertools.product((1, 0) if ew.regular else (0,), (32, 16, 8) if tiny else (32,),
                                                          (True, False) if tiny else (True,)):
            td, lr, cn = emu.render_raybuffers(ew, s, w, h, variant=variant, group=group, counters=counters, fill=MAGENTA)
            tag = f"{_tag(case)} kernel={'boundary-table' if variant else 'general'} g{group} counters={counters}"
            assert np.array_equal(td, otd), f"{tag}: top/down raybuffer differs in {int((td != otd).sum())} pixels"
            assert np.array_equal(lr, olr), f"{tag}: left/right raybuffer differs in {int((lr != olr).sum())} pixels"
            assert cn is None or cn == ocn, f"{tag}: counters {cn} != {ocn}"


def test_oracle_equals_the_reference(cv, orc, ref, oracle_worlds, cases):
    """The reference's own code (oracle/_ref) == the oracle on these worlds: pins where a LOD whose 2^j does not divide the height is
    drawn, in both iteration directions, to the reference rather than to a restatement of it."""
    for case in cases:
        key, world, name, w, h, s = case
        rw = ref.RefWorld(world.dims, world.blobs, world.column_counts)
        td, lr, _ = orc.render_raybuffers(oracle_worlds[key], orc.copy_setup(s), w, h)
        rtd, rlr = ref.render_raybuffers(rw, ref.copy_setup(s), w, h)
        assert (td == rtd).all() and (lr == rlr).all(), _tag(case)


def upsampled(b, j):
    """LOD j of a base as a dense grid of world units, stacked from y = 0 (the ray query's placement, DESIGN.md §3.5)."""
    s = 1 << j
    g = b.grids[j]
    out = np.zeros(b.dims, dtype=np.uint32)
    out[:g.shape[0] * s, :g.shape[1] * s, :g.shape[2] * s] = g.repeat(s, 0).repeat(s, 1).repeat(s, 2)
    return out


def test_definition_matches_float64_brute_force(cv, bases):
    """The ray-query definition (tools/raycast_oracle) at every LOD == a float64 DDA over that LOD's grid from lod_grid, upsampled to
    world units from y = 0; rays within 1e-4 of a tie are skipped (under 2 %). Heights up to 1000 (the brute force steps unit cells)."""
    rng = np.random.default_rng(7)
    total = amb = hits = 0
    for dy, b in bases.items():
        if dy > 1000:
            continue
        rw = rco.RayWorld(b.world(len(b.blobs)))
        for j in range(len(b.blobs)):
            grid = upsampled(b, j)
            rays = random_rays(rng, b.dims, 60)
            got = rco.raycast(rw, rays, j)
            for r, h in zip(rays, got):
                hit, cell, face, color, ambiguous = brute_force(grid, r)
                total += 1
                if ambiguous:
                    amb += 1
                    continue
                assert h["hit"] == hit, (b.dims, j, r, h, hit, cell)
                if hit == 1:
                    hits += 1
                    want = tuple(c >> j for c in cell)
                    assert tuple(h["cell"]) == want and h["face"] == face and h["color"] == color, (b.dims, j, r, h, want, face, color)
                    t = _entry_distance(r, cell, face)
                    assert abs(float(h["distance"]) - t) <= 1e-3 + 1e-5 * t, (b.dims, j, r, h, t)
    assert amb < 0.02 * total and hits > 0.2 * total, (amb, hits, total)


def _entry_distance(ray, cell, face):
    """float64 distance along the normalised ray to the face of the unit cell it entered through (0 for a start inside it)."""
    if face == 6:
        return 0.0
    d = np.array(ray["direction"], dtype=np.float64)
    d /= np.linalg.norm(d)
    a = face // 2
    plane = cell[a] + (face & 1)          # even faces are entered moving up the axis (through the cell's low side)
    return (plane - float(ray["origin"][a])) / d[a]


def test_kernel_traversal_equals_definition(cv, bases):
    """raycast.h compiled for the CPU == the definition on every field and bit, at every LOD, on both run paths (boundary records
    and element area)."""
    rng = np.random.default_rng(8)
    for dy, b in bases.items():
        world = b.world(len(b.blobs))
        ew, rw = emu.EmuWorld(world), rco.RayWorld(world)
        rays = random_rays(rng, b.dims, 1500)
        for j in range(len(b.blobs)):
            want = rco.raycast(rw, rays, j)
            for general in (False, True):
                got = rco.emu_raycast(ew, rays, j, general)
                assert same(got, want), (b.dims, j, general, first_mismatch(rays, got, want))


def test_world_file_round_trip_keeps_the_height(cv, bases, tmp_path):
    """cvx_world_file_write / cvx_world_file_read at heights that are not powers of two: dimensions, blobs and column counts back."""
    for dy in (100, 4095):
        b = bases[dy]
        world = b.world(len(b.blobs))
        path = str(tmp_path / f"h{dy}.world")
        world.save(path)
        back = cv.World.load(path)
        assert tuple(back.dims) == b.dims and back.column_counts == world.column_counts
        assert all(np.array_equal(x, y) for x, y in zip(back.blobs, world.blobs))


# ---- ray queries against the frame -----------------------------------------------------------------------------------------------
PICK_W, PICK_H = 120, 90


def _pick_cases(cv):
    """(dims, LOD j, camera name, pose): LODs whose 2^j does not divide the height, cameras just outside a corner of the world looking
    down and up across it (rays enter the world at LOD j)."""
    out = []
    for dims, j in (((32, 127, 32), 1), ((32, 127, 32), 2), ((32, 100, 32), 3), ((16, 1000, 16), 4)):
        level = 30.5
        for name, pos, euler in (("down", (-2.3, level + 14.0, -2.6), (35.0, 45.0, 0.0)), ("up", (-2.3, level - 9.0, -2.6), (-25.0, 45.0, 0.0))):
            out.append((dims, j, name, cv.CameraPose.from_euler(pos, euler, far_clip=4.0 * max(dims[0], dims[2]))))
    return out


def _pick_world(dims):
    """Floating boxes with a colour per voxel over a terrace floor: side faces and caps at many heights to pick against."""
    rng = np.random.default_rng(dims[1])
    grid = np.zeros(dims, dtype=np.uint32)
    for _ in range(40):
        x, z = rng.integers(0, dims[0] - 4), rng.integers(0, dims[2] - 4)
        y = int(rng.integers(5, 60))
        box = grid[x:x + int(rng.integers(2, 5)), y:y + int(rng.integers(3, 10)), z:z + int(rng.integers(2, 5))]
        box[...] = _colour(rng, box.size).reshape(box.shape)
    grid[:, :3, :] = _colour(rng, dims[0] * 3 * dims[2]).reshape(dims[0], 3, dims[2])
    return grid


def test_picking_follows_the_bottom_up_placement(cv, orc):
    """At a LOD whose 2^j does not divide dim_y, a ray query stacks columns from y = 0 (DESIGN.md §3.5). A frame drawn looking up
    does too; a frame drawn looking down stacks them from dim_y, r = dim_y mod 2^j world units higher. Picks at pixel centres of
    frames drawn at LOD j alone agree best with the frame when their origins are lowered by exactly r looking down and by 0 looking
    up, among every shift 0 .. 2^j."""
    for dims, j, name, pose in _pick_cases(cv):
        grid = _pick_world(dims)
        blobs = [encode_world(lod_grid(grid, k), k) for k in range(j + 1)]
        world = cv.World(dims, [b for b, _ in blobs], [c for _, c in blobs])
        r = dims[1] % (1 << j)
        assert r
        lods = np.array([-1.0] * j + [1e9] * (LODS - j), dtype=F32)   # every ray starts at LOD j
        s = cv.frame_setup(pose, PICK_W, PICK_H, lods, dims[1], limit_horizon=False)
        assert s.camera.inverse_element_iteration_direction == (name == "up")
        ow = orc.OracleWorld(dims, world.blobs, world.column_counts)
        st = orc.ray_setup(ow, orc.copy_setup(s), PICK_W, PICK_H)
        assert (st["lod"][st["status"] == 0] == j).all()
        os_ = orc.copy_setup(s)
        td, lr, _ = orc.render_raybuffers(ow, os_, PICK_W, PICK_H)
        frame = orc.blit(os_, PICK_W, PICK_H, td, lr)
        ys, xs = np.mgrid[0:PICK_H:2, 0:PICK_W:2]
        xs, ys = xs.ravel(), ys.ravel()
        o = np.zeros((xs.size, 3), dtype=F32)
        d = np.zeros((xs.size, 3), dtype=F32)
        for k, (x, y) in enumerate(zip(xs, ys)):
            o[k], d[k] = cv.screen_ray(pose, x + 0.5, y + 0.5, PICK_W, PICK_H)
        px = frame[ys, xs]
        vox = px != cv.SKYBOX_ARGB
        assert vox.sum() > 0.2 * vox.size, (dims, j, name)
        rw = rco.RayWorld(world)
        agree = []
        for shift in range(0, (1 << j) + 1):
            hits = rco.raycast(rw, cv.make_rays(o - F32([0, shift, 0]), d), j)
            agree.append(float(np.mean((hits["hit"][vox] == 1) & (hits["color"][vox] == px[vox]))))
        want = r if name == "down" else 0
        best = int(np.argmax(agree))
        assert best == want, f"{dims} LOD {j} looking {name}: agreement per origin shift {np.round(agree, 3)}, best at {best}, want {want}"
        print(f"{dims} LOD {j} looking {name}: agreement per origin shift {np.round(agree, 3)}")
        assert agree[want] >= 0.65 and max(a for k, a in enumerate(agree) if k != want) < agree[want], (dims, j, name, agree)


# ---- GPU legs --------------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def rm(cv):
    m = cv.RenderManager(0, counters=True)
    yield m
    m.destroy()


def _by_world(cases):
    out = {}
    for case in cases:
        out.setdefault(case[0], []).append(case)
    return out


@gpu
@pytest.mark.parametrize("group", [0, 8, 16])
def test_cuda_equals_oracle(cv, orc, rm, bases, oracle_worlds, cases, group):
    """CUDA == oracle bit for bit over the whole corpus: raybuffers, work counters and frame, product and counter builds, and the
    general kernel forced where the world is regular; the regular flag equals the host verdict, and (at the default group width)
    every ray's setup state equals the oracle's on every field."""
    rm.set_group_size(group)
    try:
        for key, group_cases in _by_world(cases).items():
            dy, n = key
            b = bases[dy]
            rm.upload_world(group_cases[0][1])
            verdicts = [emu.transcode_verdict(b.blobs[j], b.ccs[j], b.dims, j)[2] for j in range(n)]
            assert rm.world_is_regular() == all(verdicts) == emu.EmuWorld(group_cases[0][1]).regular, key
            for case in group_cases:
                _, world, name, w, h, s = case
                rm.set_resolution(w, h)
                _assert_same(_gpu_frame(rm, s, MAGENTA), _oracle_frame(orc, oracle_worlds[key], s, w, h, MAGENTA), f"{_tag(case)} g{group}")
                if group == 0:
                    g = rm.ray_setup(s)
                    o = orc.ray_setup(oracle_worlds[key], orc.copy_setup(s), w, h)
                    assert len(g) == len(o), _tag(case)
                    for field in o.dtype.names:   # bit for bit, except that any NaN equals any NaN
                        gv, ov = g[field], o[field]
                        ok = gv.view(np.uint32) == ov.view(np.uint32)
                        if gv.dtype.kind == "f":
                            ok |= np.isnan(gv) & np.isnan(ov)
                        assert ok.all(), (_tag(case), field)
    finally:
        rm.set_group_size(0)


@gpu
def test_device_transcode_equals_the_host(cv, rm, bases):
    """The device transcode's accept/reject decision and regular flag == world_transcode.h's on every base at every LOD set, and on
    corrupted copies of one LOD made as the transcode fuzz of the world-production tests makes them."""
    from test_world_production import CVX_ERR_FORMAT, mutate, upload_error
    rng = np.random.default_rng(31)
    rejected = accepted = 0
    for dy, b in bases.items():
        for n in lod_sets(b.dims):
            world = b.world(n)
            assert upload_error(rm, cv, world) is None, (b.dims, n)
            assert rm.world_is_regular() == all(emu.transcode_verdict(b.blobs[j], b.ccs[j], b.dims, j)[2] for j in range(n)), (b.dims, n)
        for _ in range(6):
            j = int(rng.integers(0, len(b.blobs)))
            if not b.grids[j].any():
                continue
            blob, cc, what = mutate(b.blobs[j], b.ccs[j], b.dims, j, rng)
            blobs, ccs = list(b.blobs), list(b.ccs)
            blobs[j], ccs[j] = blob, cc
            world = cv.World(b.dims, blobs, ccs)
            verdicts = [emu.transcode_verdict(x, c, b.dims, k) for k, (x, c) in enumerate(zip(blobs, ccs))]
            ok, bad, _ = verdicts[j]
            err = upload_error(rm, cv, world)
            if not ok:
                assert err == (CVX_ERR_FORMAT, bad, j), f"{b.dims} {what} at LOD {j}: host rejects column {bad}, device {err}"
                rejected += 1
                continue
            assert err is None, f"{b.dims} {what} at LOD {j}: host accepts, device {err}"
            assert rm.world_is_regular() == all(v[2] for v in verdicts), f"{b.dims} {what} at LOD {j}: regular flag"
            accepted += 1
    assert rejected >= 10 and accepted >= 10, (rejected, accepted)


@gpu
def test_world_file_renders_like_the_direct_upload(cv, rm, bases, cases, tmp_path):
    """A .world written at a height that is not a power of two, read back and uploaded, draws the same frames as the direct upload."""
    for dy in (100, 257, 4095):
        b = bases[dy]
        world = b.world(len(b.blobs))
        path = str(tmp_path / f"h{dy}.world")
        world.save(path)
        back = cv.World.load(path)
        mine = [c for c in cases if c[0] == (dy, len(b.blobs))]
        assert mine
        frames = []
        for w in (world, back):
            rm.upload_world(w)
            for case in mine:
                rm.set_resolution(case[3], case[4])
                frames.append(_gpu_frame(rm, case[5], MAGENTA))
        for case, direct, from_file in zip(mine, frames[:len(mine)], frames[len(mine):]):
            _assert_same(direct, from_file, f"{_tag(case)}: file vs direct upload")


@gpu
def test_gpu_raycast_equals_definition(cv, rm, bases):
    """cvx_raycast == the definition on every field and bit, host and device arrays, both run paths, at every uploaded LOD."""
    rng = np.random.default_rng(9)
    for dy, b in bases.items():
        world = b.world(len(b.blobs))
        rm.upload_world(world)
        rw = rco.RayWorld(world)
        rays = random_rays(rng, b.dims, 4000)
        for j in range(len(b.blobs)):
            want = rco.raycast(rw, rays, j)
            for general in (False, True):
                rm.set_general_path(general)
                got = rm.raycast_rays(rays, j)
                assert same(got, want), (b.dims, j, general, first_mismatch(rays, got, want))
                got = _device_raycast(rm, rays, j)
                assert same(got, want), ("device", b.dims, j, general, first_mismatch(rays, got, want))
        rm.set_general_path(False)
