"""World production at its edges: the host builder (world_builder.cpp), the device builder (world_builder_gpu.cu: voxelize, sort +
merge, re-key, RLE) and the upload transcode (transcode_count_kernel / transcode_write_kernel) against tests/voxref.py, a plain
NumPy restatement of VoxelizerHelper / WorldBuilder / World.DownSample that uses neither builder.

CPU: the NumPy reference equals World.from_mesh on every case of an edge-mesh corpus, every LOD blob byte for byte.
GPU: the device builder equals the reference; the resident build ray-casts like the per-cell definition on the reference blobs at
every LOD and renders like the uploaded reference blobs and the oracle; refusals leave no world behind; and the device transcode's
accept / reject decision, rejected column and regular flag equal the host transcode's (world_transcode.h) on seeded corruptions of
builder blobs, compared before anything is drawn."""
from __future__ import annotations

import re

import numpy as np
import pytest

import emu
import raycast_oracle as rco
import voxref
from test_raycast import first_mismatch, random_rays, same

CVX_ERR_INVALID_ARGUMENT = -1
CVX_ERR_NO_WORLD = -5
CVX_ERR_FORMAT = -8
RNG_SEED = 20261020


# ---- the edge-mesh corpus ------------------------------------------------------------------------------------------------------
# Every case pins the remap box with a degenerate triangle from the origin to `hi` and uses max_dimension = max(hi), so the scale
# is exactly 1 and the vertices below are already in world units (a mesh's own coordinates reach the voxelizer unchanged).

class Case:
    def __init__(self, name, hi, tris, colors=None, flips=(False, False, False), lods=6, seed=0):
        rng = np.random.default_rng(seed)
        tris = np.asarray(tris, dtype=np.float32).reshape(-1, 3)
        self.name, self.flips, self.lods = name, tuple(flips), lods
        self.max_dimension = int(max(hi))
        self.positions = np.concatenate([np.array([(0, 0, 0), (0, 0, 0), hi], dtype=np.float32), tris])
        if colors is None:
            colors = rng.integers(0, 256, size=(len(tris), 4))
        colors = np.asarray(colors).reshape(-1, 4).astype(np.uint8)
        self.colors = np.concatenate([np.full((3, 4), 255, dtype=np.uint8), colors])
        self.colors[:, 3] = 255

    def __repr__(self):
        return self.name


def soup(rng, n, hi, size):
    """n triangles with vertices within `size` of a random centre, clipped to the box (some land exactly on its faces)."""
    hi = np.array(hi, dtype=np.float64)
    c = rng.uniform(0, 1, (n, 1, 3)) * hi
    v = c + rng.uniform(-size, size, (n, 3, 3))
    return np.clip(v, 0, hi).astype(np.float32)


def quad(p, u, v):
    p, u, v = (np.array(t, dtype=np.float32) for t in (p, u, v))
    return [p, p + u, p + u + v, p, p + u + v, p + v]


# a non-degenerate fp32 sliver whose vertex `a` lies exactly on its centroid: normalize(a - mid) is 0 * inf, a NaN corner
NAN_SLIVER = [(31.80664825, 26.96515083, 29.68316078), (17.53909684, 0.45387703, 41.32613754), (46.07419968, 53.47642899, 18.04018021)]


def corpus():
    rng = np.random.default_rng(RNG_SEED)
    cases = [
        Case("footprint_256x32x16", (256, 32, 16), soup(rng, 80, (256, 32, 16), 6), seed=1),
        Case("footprint_16x64x512", (16, 64, 512), soup(rng, 80, (16, 64, 512), 8), seed=2),
        Case("x1_wide", (1, 64, 32), soup(rng, 40, (1, 64, 32), 5), seed=3),
        Case("z1_wide", (32, 16, 1), soup(rng, 40, (32, 16, 1), 5), seed=4),
        Case("thin_y1", (32, 1, 32), soup(rng, 30, (32, 1, 32), 6), seed=5),
        Case("thin_y2", (32, 2, 16), soup(rng, 30, (32, 2, 16), 6), seed=6),
        Case("thin_y4", (16, 4, 64), soup(rng, 30, (16, 4, 64), 6), seed=7),
    ]
    flip_soup = soup(rng, 60, (64, 32, 16), 6)
    for f in range(8):
        flips = (bool(f & 1), bool(f & 2), bool(f & 4))
        cases.append(Case("flips_" + "".join("T" if b else "F" for b in flips), (64, 32, 16), flip_soup, flips=flips, seed=8))
    # vertices on the faces, edges and corners of the box: expanded corners below 0 and above dims - 1
    clamp = quad((0, 0, 0), (64, 0, 0), (0, 0, 32)) + quad((0, 16, 0), (64, 0, 0), (0, 0, 32)) + quad((0, 0, 0), (0, 16, 0), (0, 0, 32))
    clamp += [(64, 16, 32), (0, 0, 0), (64, 0, 32), (0, 16, 32), (64, 16, 0), (32, 8, 16), (64, 16, 32), (63.9, 15.9, 31.9), (64, 15.5, 30)]
    cases.append(Case("clamp", (64, 16, 32), clamp, seed=9))
    degenerate = [(5, 5, 5), (5, 5, 5), (20, 30, 40),                     # repeated vertex
                  (1, 2, 3), (2, 4, 6), (3, 6, 9),                        # exactly collinear
                  (10, 10, 10), (40, 40, 40.001), (50, 50, 50),           # slivers
                  (3, 50, 7), (60, 51, 9), (31.5, 50.5, 8.0001),
                  (20, 20, 20), (20.0001, 20, 20), (20, 20.0001, 20)]     # tiny
    cases.append(Case("degenerate_and_slivers", (64, 64, 64), degenerate + NAN_SLIVER + list(soup(rng, 10, (64, 64, 64), 6).reshape(-1, 3)), seed=10))
    cases.append(Case("nan_corner_sliver", (64, 64, 64), NAN_SLIVER, colors=[(10, 200, 30, 255), (250, 5, 90, 255), (128, 64, 32, 255)]))
    # 64 coincident triangles with different vertex colours, and a dense 32^3 stack (one LOD-5 cell averages 32768 voxels)
    co = np.tile(np.array([(3, 10, 4), (40, 12, 9), (9, 50, 44)], dtype=np.float32), (64, 1))
    stack = sum((quad((0, k + 0.5, 0), (32, 0, 0), (0, 0, 32)) for k in range(32)), [])
    cases.append(Case("overlap_and_dense_stack", (64, 64, 64), list(co) + stack, seed=11))
    levels = np.array([0, 255, 127, 128, 1, 254, 64, 191])
    cases.append(Case("colour_edges", (32, 32, 32), soup(rng, 60, (32, 32, 32), 6),
                      colors=np.stack([levels[rng.integers(0, 8, 180)] for _ in range(4)], axis=1), seed=12))
    # one flat triangle just under VOXELIZE_BUFFER_MAX voxels (261726) and one over (262450): the host cuts it in scan order,
    # the device refuses the build
    cases.append(Case("cap_under", (1024, 1, 1024), [(1, 0.5, 1), (724.5, 0.5, 1), (1, 0.5, 724.5)], seed=13))
    cases.append(Case("cap_over", (1024, 1, 1024), [(1, 0.5, 1), (725, 0.5, 1), (1, 0.5, 725)], seed=14))
    # a wall whose columns hold 32768 voxels: the int16 Length of the single run wraps to -32768
    cases.append(Case("tall_wall", (4, 32768, 4), quad((0, 0, 2), (4, 0, 0), (0, 32768, 0)), seed=15))
    cases.append(Case("empty", (16, 8, 32), [(1, 1, 1), (1, 1, 1), (9, 5, 20), (2, 2, 2), (4, 4, 4), (6, 6, 6)]))
    return cases


CORPUS = corpus()
BY_NAME = {c.name: c for c in CORPUS}
THIN = ("thin_y1", "thin_y2", "thin_y4", "x1_wide", "z1_wide")
DEVICE_REFUSES = ("cap_over",)              # CVX_ERR_INVALID_ARGUMENT: a triangle over VOXELIZE_BUFFER_MAX
UPLOAD_REFUSES = ("tall_wall",)             # CVX_ERR_FORMAT: Length -32768


_refs = {}


def reference(case: Case, lods=None) -> voxref.RefWorld:
    key = (case.name, case.lods if lods is None else lods)
    if key not in _refs:
        _refs[key] = voxref.build(case.positions, case.colors, case.max_dimension, case.flips, key[1])
    return _refs[key]


def assert_same_world(got, want, what):
    assert tuple(got.dims) == tuple(want.dims), f"{what}: dims {got.dims} != {want.dims}"
    assert len(got.blobs) == len(want.blobs), f"{what}: {len(got.blobs)} LODs, want {len(want.blobs)}"
    assert list(got.column_counts) == list(want.column_counts), f"{what}: column counts {got.column_counts} != {want.column_counts}"
    assert list(got.voxel_counts) == list(want.voxel_counts), f"{what}: voxel counts {got.voxel_counts} != {want.voxel_counts}"
    for lod, (a, b) in enumerate(zip(got.blobs, want.blobs)):
        assert a.nbytes == b.nbytes, f"{what} LOD {lod}: blob of {a.nbytes} bytes, want {b.nbytes}"
        if not np.array_equal(a, b):
            i = int(np.nonzero(a != b)[0][0])
            raise AssertionError(f"{what} LOD {lod}: {int((a != b).sum())} bytes differ, first at byte {i}")


# ---- CPU -----------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("case", CORPUS, ids=repr)
def test_reference_equals_host_builder(cv, case):
    ref = reference(case)
    host = cv.World.from_mesh(case.positions, case.colors, case.max_dimension, flips=case.flips, lods=case.lods)
    assert_same_world(host, ref, f"{case.name}: host builder")


def test_corpus_reaches_its_edges(cv):
    """The cases exercise what they are named for (so a corpus edit cannot quietly lose an edge)."""
    r = {c.name: reference(c) for c in CORPUS}
    assert r["footprint_256x32x16"].dims == (256, 32, 16) and r["footprint_16x64x512"].dims == (16, 64, 512)
    assert len(r["x1_wide"].blobs) == 1 and len(r["z1_wide"].blobs) == 1 and len(r["thin_y1"].blobs) == 1
    assert len(r["thin_y2"].blobs) == 2 and len(r["thin_y4"].blobs) == 3
    assert r["empty"].voxel_counts == [0] * 4 and r["degenerate_and_slivers"].triangle_voxels[1:3].tolist() == [0, 0]
    under, over = r["cap_under"].triangle_voxels[1], r["cap_over"].triangle_voxels[1]
    assert voxref.VOXELIZE_BUFFER_MAX - 1000 < under <= voxref.VOXELIZE_BUFFER_MAX < over
    assert r["cap_over"].voxel_counts[0] == voxref.VOXELIZE_BUFFER_MAX
    wall = r["tall_wall"]
    hdr = wall.blobs[0].view(np.uint32)[:3 * wall.column_counts[0]].reshape(-1, 3)
    assert wall.dims == (4, 32768, 4) and (hdr[:, 1] & 0xFFFF).max() == 1 and wall.voxel_counts[0] == 4 * 32768
    # the NaN-corner sliver emits every cell of its b-c box with colour 0 (the box of corners b and c)
    nan = r["nan_corner_sliver"]
    x, y, z, argb = nan.voxels[0]
    assert len(x) > 10000 and (argb == 0xFF).all()
    # a LOD-5 cell averages 32^3 voxels of the dense stack
    stack = r["overlap_and_dense_stack"]
    x, y, z, _ = stack.voxels[0]
    assert len(stack.blobs) == 6 and ((x < 32) & (y < 32) & (z < 32)).sum() == 32 ** 3


@pytest.mark.parametrize("name", ["thin_y1", "thin_y2", "thin_y4", "x1_wide"])
def test_lod_loop_stops_early_on_the_host(cv, name):
    case = BY_NAME[name]
    for lods in range(1, 7):
        ref = reference(case, lods)
        host = cv.World.from_mesh(case.positions, case.colors, case.max_dimension, flips=case.flips, lods=lods)
        assert_same_world(host, ref, f"{name} lods={lods}: host builder")
        assert len(ref.blobs) == voxref.lod_levels(ref.dims, lods) <= lods


def test_reference_decodes_to_its_voxels():
    """voxref.blob against tests/rle.py::decode_world, which also checks the layout invariants (guards, full-height runs,
    worldMin / worldMax)."""
    from rle import decode_world
    for name in ("footprint_256x32x16", "flips_TFT", "overlap_and_dense_stack", "clamp"):
        ref = reference(BY_NAME[name])
        for lod, (b, cc) in enumerate(zip(ref.blobs, ref.column_counts)):
            assert np.array_equal(decode_world(b, cc, ref.dims, lod), voxref.grid_of(ref.voxels[lod], ref.dims, lod)), (name, lod)


def test_host_transcode_verdict_on_builder_blobs():
    """The host transcode accepts every builder blob of the corpus as regular, except the wrapped 32768-voxel run."""
    for case in CORPUS:
        ref = reference(case)
        for lod, (b, cc) in enumerate(zip(ref.blobs, ref.column_counts)):
            ok, bad, regular = emu.transcode_verdict(b, cc, ref.dims, lod)
            if case.name in UPLOAD_REFUSES and lod == 0:
                assert not ok and bad == 2, (case.name, lod, ok, bad)   # column (0, 2), the first of the wall
            else:
                assert ok and bad == -1 and regular, (case.name, lod, ok, bad, regular)


# ---- transcode decision fuzz: seeded corruptions of builder blobs ------------------------------------------------------------------

def _solid_runs(cells, off, rc):
    out = []
    for k in range(rc):
        e = int(cells[off + 1 + k])
        ci, ln = e & 0xFFFF, (e >> 16) & 0xFFFF
        out.append((k, ci - 0x10000 if ci >= 0x8000 else ci, ln - 0x10000 if ln >= 0x8000 else ln))
    return out


def mutate(blob, cc, dims, lod, rng):
    """One corrupted copy of a LOD blob: returns (blob, column_count, description). Kinds: element offset past the end or
    negative, run count past the end or merely wrong, ColorsIndex + Length past the colour table (and exactly at its end), negative
    Length, a zero-length early terminator, lengths summing short of or past dimY, column_count > needCols (extra headers)."""
    words = np.ascontiguousarray(blob).view(np.uint32).copy()
    hdr = words[:3 * cc].reshape(cc, 3)
    cells = words[3 * cc:]
    E = len(cells)
    need = (dims[0] >> lod) * (dims[2] >> lod)
    cols = [i for i in range(need) if hdr[i, 1] & 0xFFFF]
    kind = int(rng.integers(0, 10))
    done = []
    for c in sorted(rng.choice(cols, size=min(len(cols), 1 + int(rng.random() < 0.3)), replace=False)):
        c = int(c)
        off, rc = int(hdr[c, 0]), int(hdr[c, 1] & 0xFFFF)
        runs = _solid_runs(cells, off, rc)
        solid = [r for r in runs if r[1] >= 0]
        colour_cells = E - (off + rc + 2)
        if kind == 0:
            hdr[c, 0] = E - rc - 2 + int(rng.integers(1, 40))
        elif kind == 1:
            hdr[c, 0] = (1 << 32) - int(rng.integers(1, 1 << 20)) if rng.random() < 0.7 else 0x80000000
        elif kind == 2:
            hdr[c, 1] = (int(hdr[c, 1]) & 0xFFFF0000) | min(0xFFFF, E - off - 2 + int(rng.integers(1, 40)))
        elif kind == 3:
            hdr[c, 1] = (int(hdr[c, 1]) & 0xFFFF0000) | int(rng.integers(1, max(2, min(0xFFFF, E - off - 2))))
        elif kind in (4, 5) and solid:
            k, ci, ln = solid[int(rng.integers(0, len(solid)))]
            ci = colour_cells - ln + (int(rng.integers(1, 8)) if kind == 4 else 0)   # 5: exactly at the end of the table
            if 0 <= ci <= 0x7FFF:
                cells[off + 1 + k] = (ci & 0xFFFF) | (ln << 16)
        elif kind == 6:
            k = int(rng.integers(0, rc))
            cells[off + 1 + k] = (int(cells[off + 1 + k]) & 0xFFFF) | (((-int(rng.integers(1, 300))) & 0xFFFF) << 16)
        elif kind == 7:
            k = int(rng.integers(0, rc))
            cells[off + 1 + k] = int(cells[off + 1 + k]) & 0xFFFF
        elif kind == 8:
            k = int(rng.integers(0, rc))
            e = int(cells[off + 1 + k])
            ln = max(1, min(0x7FFF, ((e >> 16) & 0xFFFF) + int(rng.choice([-3, -2, -1, 1, 2, 3]))))
            cells[off + 1 + k] = (e & 0xFFFF) | (ln << 16)
        done.append(c)
    if kind == 9:   # more column headers than the LOD addresses; the extra ones hold garbage and are never read
        extra = int(rng.integers(1, 50))
        junk = rng.integers(0, 1 << 32, size=3 * extra, dtype=np.uint64).astype(np.uint32)
        words = np.concatenate([words[:3 * cc], junk, cells])
        return words.view(np.uint8), cc + extra, f"kind 9: {extra} extra headers"
    return words.view(np.uint8), cc, f"kind {kind} on columns {done}"


def fuzz_cases(count=240):
    """(world of reference blobs with one LOD corrupted, corrupted LOD, description), seeded."""
    rng = np.random.default_rng(RNG_SEED + 1)
    bases = [reference(BY_NAME[n]) for n in ("flips_FTF", "footprint_256x32x16", "overlap_and_dense_stack")]
    for i in range(count):
        base = bases[i % len(bases)]
        lod = int(rng.integers(0, min(3, len(base.blobs))))
        b, cc, what = mutate(base.blobs[lod], base.column_counts[lod], base.dims, lod, rng)
        blobs, ccs = list(base.blobs), list(base.column_counts)
        blobs[lod], ccs[lod] = b, cc
        yield voxref.RefWorld(base.dims, blobs=blobs, column_counts=ccs), lod, what


def test_fuzz_reaches_both_verdicts():
    verdicts = [emu.transcode_verdict(w.blobs[lod], w.column_counts[lod], w.dims, lod) for w, lod, _ in fuzz_cases()]
    assert sum(1 for ok, _, _ in verdicts if not ok) >= 60
    assert sum(1 for ok, _, reg in verdicts if ok and not reg) >= 20
    assert sum(1 for ok, _, reg in verdicts if ok and reg) >= 20


# ---- GPU -----------------------------------------------------------------------------------------------------------------------

gpu = pytest.mark.gpu
W, H = 96, 64


@pytest.fixture(scope="module")
def rm(cv):
    r = cv.RenderManager(0)
    r.set_resolution(W, H)
    yield r
    r.destroy()


def probe_rays(dims, rng):
    """A grid of rays down through every column lattice point, along x and along z through the world, from inside it, plus the
    random rays of the ray-query tests (inside, outside, aimed, axis-parallel, cut off, zero and NaN directions)."""
    X, Y, Z = dims
    gx, gz = np.meshgrid(np.linspace(0.25, X - 0.25, min(X, 24)), np.linspace(0.25, Z - 0.25, min(Z, 24)), indexing="ij")
    down = np.stack([gx.ravel(), np.full(gx.size, Y + 3.0), gz.ravel()], axis=1)
    gy, gz2 = np.meshgrid(np.linspace(0.3, Y - 0.3, min(Y, 16)), np.linspace(0.3, Z - 0.3, min(Z, 16)), indexing="ij")
    along_x = np.stack([np.full(gy.size, -2.0), gy.ravel(), gz2.ravel()], axis=1)
    gx2, gy2 = np.meshgrid(np.linspace(0.3, X - 0.3, min(X, 16)), np.linspace(0.3, Y - 0.3, min(Y, 16)), indexing="ij")
    along_z = np.stack([gx2.ravel(), gy2.ravel(), np.full(gx2.size, Z + 2.0)], axis=1)
    inside = rng.uniform(0, 1, (500, 3)) * np.array(dims, dtype=np.float64)
    origins = np.concatenate([down, along_x, along_z, inside])
    dirs = np.concatenate([np.tile([0.1, -1.0, 0.07], (len(down), 1)), np.tile([1.0, 0.01, 0.02], (len(along_x), 1)),
                           np.tile([0.03, -0.02, -1.0], (len(along_z), 1)), rng.normal(size=(500, 3))])
    from cpuvox_b200 import make_rays
    return np.concatenate([make_rays(origins, dirs), random_rays(rng, dims, 2000)])


def multi_lod_setup(cv, dims, lods):
    """A view from outside and above the world with LOD distances short enough that every LOD the world has is drawn (and none
    it lacks)."""
    span = float(max(dims))
    dist = [span * 0.35 * (k + 1) for k in range(lods - 1)] + [1e9] * (6 - (lods - 1))
    eye = np.array([-0.15 * dims[0], dims[1] + 0.25 * span, -0.15 * dims[2]])
    to = np.array(dims, dtype=np.float64) * 0.5 - eye                     # aimed at the centre of the world
    euler = (np.degrees(np.arctan2(-to[1], np.hypot(to[0], to[2]))), np.degrees(np.arctan2(to[0], to[2])), 0.0)
    pose = cv.CameraPose.from_euler(tuple(eye), euler, far_clip=4.0 * span)
    return cv.frame_setup(pose, W, H, np.array(dist, dtype=np.float32), dims[1])


def gpu_frame(rm, setup):
    rm.clear_raybuffers(0)
    rm.draw_setup(setup)
    rm.sync()
    td, lr = rm.read_raybuffers()
    return td, lr, rm.read_frame()


def oracle_frame(world, setup):
    from oracle import oracle as orc
    ow = orc.OracleWorld(world.dims, world.blobs, world.column_counts)
    os_ = orc.copy_setup(setup)
    td, lr, _ = orc.render_raybuffers(ow, os_, W, H)
    return td, lr, orc.blit(os_, W, H, td, lr)


def assert_same_frames(a, b, what):
    for name, x, y in zip(("top/down raybuffer", "left/right raybuffer", "frame"), a, b):
        bad = int((x != y).sum())
        assert bad == 0, f"{what}: {name} differs in {bad} of {x.size} pixels"


def assert_raycast_equals_definition(rm, world, rays, lods, what):
    rw = rco.RayWorld(world)
    for lod in lods:
        want = rco.raycast(rw, rays, lod)
        got = rm.raycast_rays(rays, lod)
        assert same(got, want), f"{what} LOD {lod}: {first_mismatch(rays, got, want)}"


def upload_error(rm, cv, world):
    """None when the upload succeeds, else (code, column, lod) of the refusal."""
    try:
        rm.upload_world(cv.World(world.dims, list(world.blobs), list(world.column_counts), []))
        return None
    except cv.CvxError as e:
        m = re.search(r"column (-?\d+) of LOD (\d+)", str(e))
        return e.code, int(m.group(1)) if m else None, int(m.group(2)) if m else None


@gpu
@pytest.mark.parametrize("case", CORPUS, ids=repr)
def test_device_builder_equals_reference(cv, rm, case):
    ref = reference(case)
    if case.name in DEVICE_REFUSES:
        with pytest.raises(cv.CvxError) as e:
            rm.build_world_from_mesh(case.positions, case.colors, case.max_dimension, flips=case.flips, lods=case.lods)
        assert e.value.code == CVX_ERR_INVALID_ARGUMENT
        return
    dev = rm.build_world_from_mesh(case.positions, case.colors, case.max_dimension, flips=case.flips, lods=case.lods)
    assert_same_world(dev, ref, f"{case.name}: device builder")


@gpu
@pytest.mark.parametrize("case", CORPUS, ids=repr)
def test_resident_build_equals_reference(cv, rm, case):
    """The resident build's tables at every LOD (ray queries against the per-cell definition on the reference blobs), one
    multi-LOD view (against the uploaded reference blobs and the oracle) and the regular flag (against the host transcode)."""
    ref = reference(case)
    build = lambda: rm.build_resident_world_from_mesh(case.positions, case.colors, case.max_dimension, flips=case.flips, lods=case.lods)
    if case.name in DEVICE_REFUSES + UPLOAD_REFUSES:
        with pytest.raises(cv.CvxError) as e:
            build()
        assert e.value.code == (CVX_ERR_INVALID_ARGUMENT if case.name in DEVICE_REFUSES else CVX_ERR_FORMAT)
        with pytest.raises(cv.CvxError) as e:
            rm.draw_setup(multi_lod_setup(cv, ref.dims, 1))
        assert e.value.code == CVX_ERR_NO_WORLD
        if case.name in UPLOAD_REFUSES:
            _, bad, _ = emu.transcode_verdict(ref.blobs[0], ref.column_counts[0], ref.dims, 0)
            assert upload_error(rm, cv, ref) == (CVX_ERR_FORMAT, bad, 0)
        good = BY_NAME["flips_TFF"]
        res = rm.build_resident_world_from_mesh(good.positions, good.colors, good.max_dimension, flips=good.flips)
        assert res.voxel_counts == reference(good).voxel_counts
        return
    res = build()
    assert tuple(res.dims) == ref.dims and res.voxel_counts == ref.voxel_counts
    assert rm.world_is_regular() == emu.EmuWorld(ref).regular
    rays = probe_rays(ref.dims, np.random.default_rng(RNG_SEED + 2))
    assert_raycast_equals_definition(rm, ref, rays, range(len(ref.blobs)), f"{case.name} resident")
    setup = multi_lod_setup(cv, ref.dims, len(ref.blobs))
    resident = gpu_frame(rm, setup)
    rm.upload_world(cv.World(ref.dims, ref.blobs, ref.column_counts, ref.voxel_counts))
    assert_same_frames(resident, gpu_frame(rm, setup), f"{case.name}: resident build vs uploaded reference blobs")
    assert_same_frames(resident, oracle_frame(ref, setup), f"{case.name}: resident build vs oracle")


@gpu
@pytest.mark.parametrize("name", THIN)
def test_lod_loop_stops_early_on_the_device(cv, rm, name):
    case = BY_NAME[name]
    for lods in range(1, 7):
        ref = reference(case, lods)
        dev = rm.build_world_from_mesh(case.positions, case.colors, case.max_dimension, flips=case.flips, lods=lods)
        assert_same_world(dev, ref, f"{name} lods={lods}: device builder")
        res = rm.build_resident_world_from_mesh(case.positions, case.colors, case.max_dimension, flips=case.flips, lods=lods)
        assert res.voxel_counts == ref.voxel_counts, f"{name} lods={lods}: resident voxel counts"
        for lod in range(len(ref.blobs)):
            rm.raycast(np.zeros((1, 3)), np.ones((1, 3)), lod=lod)
        with pytest.raises(cv.CvxError):
            rm.raycast(np.zeros((1, 3)), np.ones((1, 3)), lod=len(ref.blobs))


@gpu
def test_empty_world_draws_sky_and_hits_nothing(cv, rm):
    case = BY_NAME["empty"]
    ref = reference(case)
    res = rm.build_resident_world_from_mesh(case.positions, case.colors, case.max_dimension)
    assert res.voxel_counts == [0] * len(ref.blobs)
    setup = multi_lod_setup(cv, ref.dims, len(ref.blobs))
    frame = gpu_frame(rm, setup)[2]
    assert (frame == cv.SKYBOX_ARGB).all()
    rays = probe_rays(ref.dims, np.random.default_rng(5))
    for lod in range(len(ref.blobs)):
        assert (rm.raycast_rays(rays, lod)["hit"] != 1).all()
    rm.upload_world(cv.World(ref.dims, ref.blobs, ref.column_counts, ref.voxel_counts))
    assert (gpu_frame(rm, setup)[2] == cv.SKYBOX_ARGB).all()


@gpu
def test_transcode_decisions_equal_the_host(cv, rm):
    """The device transcode's verdict on every corrupted blob is compared with world_transcode.h's before anything is drawn; only
    blobs both accept are then ray-cast (the corrupted LOD, against the per-cell definition) and drawn (against the oracle)."""
    rng = np.random.default_rng(RNG_SEED + 3)
    checked = 0
    for world, lod, what in fuzz_cases():
        verdicts = [emu.transcode_verdict(b, cc, world.dims, l) for l, (b, cc) in enumerate(zip(world.blobs, world.column_counts))]
        ok, bad, _ = verdicts[lod]
        err = upload_error(rm, cv, world)
        if not ok:
            assert err == (CVX_ERR_FORMAT, bad, lod), f"{what} at LOD {lod}: host rejects column {bad}, device {err}"
            continue
        assert err is None, f"{what} at LOD {lod}: host accepts, device {err}"
        assert rm.world_is_regular() == all(v[2] for v in verdicts), f"{what} at LOD {lod}: regular flag"
        assert_raycast_equals_definition(rm, world, random_rays(rng, world.dims, 300), [lod], what)
        if checked < 60:
            setup = multi_lod_setup(cv, world.dims, len(world.blobs))
            assert_same_frames(gpu_frame(rm, setup), oracle_frame(world, setup), f"{what} at LOD {lod}: drawn")
        checked += 1
    assert checked >= 40
