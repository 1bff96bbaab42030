"""Ray queries against the resident world (cvx_raycast, cvx_host_screen_ray; DESIGN.md §3.5).

CPU: the per-cell definition (tools/raycast_oracle) against an independent float64 brute force, the kernel's traversal (raycast.h
compiled for the CPU) against the definition bit for bit, the screen ray against the frame setup's projection, and picking against
rendering. GPU: cvx_raycast against the definition bit for bit, ordering and errors."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from conftest import MILL, POSES, comb_world, irregular_world, limited, parse_obj, pose_for, random_world_and_cameras
import raycast_oracle as rco

# ---- fixtures and helpers ---------------------------------------------------------------------------------------------------

def random_rays(rng, dims, n, scale=1.0):
    """Rays starting inside and outside the box, random and axis-parallel directions, max_distance cut-offs, and a few zero and
    NaN directions. scale: world units per LOD-0 unit of the cut-offs."""
    dims = np.array(dims, dtype=np.float64)
    inside = rng.random(n) < 0.5
    o = np.where(inside[:, None], rng.uniform(0, 1, (n, 3)) * dims, rng.uniform(-0.6, 1.6, (n, 3)) * dims)
    d = rng.normal(size=(n, 3))
    par = rng.random(n)
    d[par < 0.15, rng.integers(0, 3)] = 0.0                       # one component zero
    two = (par >= 0.15) & (par < 0.25)
    keep = rng.integers(0, 3, n)
    for i in np.nonzero(two)[0]:
        v = d[i, keep[i]]
        d[i] = 0.0
        d[i, keep[i]] = v if v != 0 else 1.0                      # axis-parallel
    aim = rng.random(n) < 0.3                                      # outside rays aimed at the box so that they enter it
    target = rng.uniform(0, 1, (n, 3)) * dims
    d[aim & ~inside] = (target - o)[aim & ~inside]
    md = np.where(rng.random(n) < 0.6, np.inf, rng.uniform(0, 1.5, n) * dims.max() * scale)
    rays = np.zeros(n, dtype=rco.RAY_DTYPE)
    rays["origin"] = o
    rays["direction"] = d
    rays["max_distance"] = md
    rays["direction"][0] = 0.0                                     # zero length
    if n > 2:
        rays["direction"][1, 1] = np.nan
        rays["origin"][2, 0] = np.inf
    return rays


def decode_cells(blob, cc, dims, lod=0):
    """Dense LOD grid by the run rules of the definition (DESIGN.md §3.5), also for irregular blobs: runs top to bottom from the
    top cell, Length <= 0 ends the column, cells outside the header's [worldMin, worldMax) are air."""
    dx, dy, dz = dims[0] >> lod, dims[1] >> lod, dims[2] >> lod
    words = np.frombuffer(np.ascontiguousarray(blob).tobytes(), dtype=np.uint32)
    hdr = words[:3 * cc].reshape(cc, 3)
    cells = words[3 * cc:]
    grid = np.zeros((dx, dy, dz), dtype=np.uint32)
    for x in range(dx):
        for z in range(dz):
            off, w1, w2 = (int(v) for v in hdr[x * dz + z])
            rc = w1 & 0xFFFF
            top = dy
            for k in range(rc):
                e = int(cells[off + 1 + k])
                ci = (e & 0xFFFF) - ((e & 0x8000) << 1)                  # int16 ColorsIndex
                ln = ((e >> 16) & 0xFFFF) - ((e >> 16 & 0x8000) << 1)    # int16 Length
                if ln <= 0:
                    break
                if ci >= 0:
                    for cy in range(max(top - ln, 0), top):
                        if ((cy + 1) << lod) > (w1 >> 16) and (cy << lod) < (w2 & 0xFFFF):
                            grid[x, cy, z] = cells[off + rc + 2 + ci + (top - 1 - cy)]
                top -= ln
    return grid


def brute_force(grid, ray):
    """Independent float64 3D DDA over a dense grid (LOD 0). Returns (hit, cell, face, color, ambiguous)."""
    o = np.array(ray["origin"], dtype=np.float64)
    dr = np.array(ray["direction"], dtype=np.float64)
    md = float(ray["max_distance"])
    if not (np.all(np.isfinite(o)) and np.all(np.isfinite(dr))) or np.isnan(md) or md == -np.inf or not np.any(dr != 0):
        return -1, None, None, None, False
    d = dr / np.linalg.norm(dr)
    n = np.array(grid.shape)
    tol = lambda t: 1e-4 + 1e-6 * abs(t)  # noqa: E731  (fp32 rounding of crossing distances grows with t)
    near, far = [], []
    for i in range(3):
        if d[i] == 0:
            if not (0 <= o[i] < n[i]):
                return 0, None, None, None, bool(min(abs(o[i]), abs(o[i] - n[i])) < 1e-4)
            continue
        a, b = (0 - o[i]) / d[i], (n[i] - o[i]) / d[i]
        near.append((min(a, b), i))
        far.append(max(a, b))
    t_enter, entry = max(near)
    t_exit = min(far)
    amb = any(abs(t - t_enter) < tol(t_enter) for t, i in near if i != entry)
    if abs(t_enter - t_exit) < tol(t_exit) or abs(t_exit) < 1e-4 or abs(t_enter) < 1e-4 or abs(max(t_enter, 0) - md) < tol(md):
        amb = True
    if t_enter > t_exit or t_exit < 0 or max(t_enter, 0) > md:
        return 0, None, None, None, amb
    t0 = max(t_enter, 0.0)
    p = o + t0 * d
    c = np.clip(np.floor(p), 0, n - 1).astype(np.int64)
    if t_enter > 0:
        c[entry] = 0 if d[entry] > 0 else n[entry] - 1
    for i in range(3):
        if d[i] == 0 or (t_enter > 0 and i == entry):
            continue
        if abs(p[i] - round(p[i])) < 1e-4:
            amb = True
    face = 2 * entry + (0 if d[entry] > 0 else 1) if t_enter > 0 else 6
    step = np.sign(d).astype(np.int64)
    tm = np.array([((c[i] + (step[i] > 0)) - o[i]) / d[i] if step[i] else np.inf for i in range(3)])
    while True:
        if grid[c[0], c[1], c[2]]:
            return 1, tuple(int(v) for v in c), face, int(grid[c[0], c[1], c[2]]), amb
        a = int(np.argmin(tm))
        srt = np.sort(tm)
        if srt[1] - srt[0] < tol(srt[0]):
            amb = True
        if abs(tm[a] - md) < tol(md):
            amb = True
        nxt = c[a] + step[a]
        if tm[a] > md or nxt < 0 or nxt >= n[a]:
            return 0, None, None, None, amb
        c[a] = nxt
        face = 2 * a + (0 if step[a] > 0 else 1)
        tm[a] = ((c[a] + (step[a] > 0)) - o[a]) / d[a]


def fuzz_worlds(cv, count=100):
    rng = np.random.default_rng(2024)
    for _ in range(count):
        world, blob, cc, _, _, _ = random_world_and_cameras(cv, rng, cameras=1)
        yield world, blob, cc, rng


def same(a, b):
    """Bit-for-bit equality of two hit arrays (every field, distance bits included)."""
    return np.ascontiguousarray(a).view(np.uint8).tobytes() == np.ascontiguousarray(b).view(np.uint8).tobytes()


def first_mismatch(rays, a, b):
    bad = np.nonzero(np.ascontiguousarray(a).view(np.uint32).reshape(-1, 8) != np.ascontiguousarray(b).view(np.uint32).reshape(-1, 8))[0]
    if len(bad) == 0:
        return None
    i = int(bad[0])
    return f"{len(np.unique(bad))} rays differ; first {i}: ray {rays[i]} -> {a[i]} vs {b[i]}"


@pytest.fixture(scope="module")
def mill1080(cv, mill_world):
    """Mill 256 at 1920x1080 for the POSES table with every LOD distance beyond the far clip (only LOD 0 is drawn) and the far clip
    beyond the world (the renderer clips by distance in the XZ plane, a ray query by distance along the ray)."""
    from oracle import oracle as orc
    W, H = 1920, 1080
    ow = orc.OracleWorld(mill_world.dims, mill_world.blobs, mill_world.column_counts)
    lods = np.full(6, 1e6, dtype=np.float32)
    out = []
    for spec in POSES:
        pose = limited(cv, pose_for(cv, mill_world, spec, far_scale=8.0))
        setup = cv.frame_setup(pose, W, H, lods, mill_world.dims[1], limit_horizon=False)
        osetup = orc.copy_setup(setup)
        td, lr, _ = orc.render_raybuffers(ow, osetup, W, H)
        out.append((pose, setup, orc.blit(osetup, W, H, td, lr)))
    return W, H, out


def pick_rays(cv, pose, W, H, stride=7):
    ys, xs = np.mgrid[0:H:stride, 0:W:stride]
    o = np.zeros((xs.size, 3), dtype=np.float32)
    d = np.zeros((xs.size, 3), dtype=np.float32)
    for k, (x, y) in enumerate(zip(xs.ravel(), ys.ravel())):
        o[k], d[k] = cv.screen_ray(pose, x + 0.5, y + 0.5, W, H)
    return xs.ravel(), ys.ravel(), cv.make_rays(o, d)


def pick_share(cv, frame, xs, ys, hits):
    """(voxel pixels whose pick hits a voxel of the pixel's colour, voxel pixels, sky pixels whose pick hits a voxel, sky pixels)."""
    px = frame[ys, xs]
    sky = px == cv.SKYBOX_ARGB
    vox = ~sky
    return (int(np.sum((hits["hit"][vox] == 1) & (hits["color"][vox] == px[vox]))), int(np.sum(vox)),
            int(np.sum(hits["hit"][sky] != 0)), int(np.sum(sky)))


# ---- CPU ----------------------------------------------------------------------------------------------------------------------

def test_struct_layouts(cv):
    from cpuvox_b200 import native as N
    assert C.sizeof(N.Ray) == 32 and C.sizeof(N.RayHit) == 32
    assert cv.RAY_DTYPE.itemsize == 32 and cv.RAY_HIT_DTYPE.itemsize == 32
    assert cv.RAY_DTYPE == rco.RAY_DTYPE and cv.RAY_HIT_DTYPE == rco.RAY_HIT_DTYPE


def _check_against_brute_force(grid, world, rays):
    hits = rco.raycast(rco.RayWorld(world), rays)
    amb = 0
    for r, h in zip(rays, hits):
        hit, cell, face, color, ambiguous = brute_force(grid, r)
        if ambiguous:
            amb += 1
            continue
        assert h["hit"] == hit, (r, h, hit, cell, face)
        if hit == 1:
            assert tuple(h["cell"]) == cell and h["face"] == face and h["color"] == color, (r, h, cell, face, color)
    return amb


def test_definition_matches_float64_brute_force(cv):
    rng = np.random.default_rng(1)
    total = amb = 0
    cases = [comb_world(cv), irregular_world(cv)]
    for world, blob, cc in cases:
        rays = random_rays(rng, world.dims, 3000)
        amb += _check_against_brute_force(decode_cells(blob, cc, world.dims), world, rays)
        total += len(rays)
    for world, blob, cc, _ in fuzz_worlds(cv):
        rays = random_rays(rng, world.dims, 200)
        amb += _check_against_brute_force(decode_cells(blob, cc, world.dims), world, rays)
        total += len(rays)
    assert amb < 0.01 * total, (amb, total)


def _emu_equals_definition(world, rays, lods=None):
    from emu import EmuWorld
    ew, rw = EmuWorld(world), rco.RayWorld(world)
    for lod in range(len(world.blobs)) if lods is None else lods:
        ref = rco.raycast(rw, rays, lod)
        assert np.any(ref["hit"] == 1)
        for general in (False, True):
            got = rco.emu_raycast(ew, rays, lod, general)
            assert same(got, ref), (lod, general, first_mismatch(rays, got, ref))


def test_kernel_traversal_equals_definition_small_worlds(cv):
    rng = np.random.default_rng(2)
    for world, _, _ in (comb_world(cv), irregular_world(cv)):
        _emu_equals_definition(world, random_rays(rng, world.dims, 20000))
    for world, _, _, _ in fuzz_worlds(cv):
        _emu_equals_definition(world, random_rays(rng, world.dims, 200))


@pytest.mark.parametrize("name", ["mill_world", "terrain_world", "structure_world"])
def test_kernel_traversal_equals_definition_every_lod(cv, request, name):
    world = request.getfixturevalue(name)
    _emu_equals_definition(world, random_rays(np.random.default_rng(3), world.dims, 20000))


def _quat_rotate(q, v):
    x, y, z, w = (float(a) for a in q)
    u = np.array([x, y, z])
    v = np.asarray(v, dtype=np.float64)
    return 2 * np.dot(u, v) * u + (w * w - np.dot(u, u)) * v + 2 * w * np.cross(u, v)


def test_screen_ray_centre_is_forward(cv):
    dims = (256, 256, 256)
    for spec in POSES:
        pose = pose_for(cv, cv.World(dims, [], []), spec)
        for W, H in ((1920, 1080), (640, 480), (101, 77)):
            o, d = cv.screen_ray(pose, W / 2, H / 2, W, H)
            fwd = _quat_rotate(pose.rotation, (0, 0, 1))
            assert np.allclose(d, fwd, atol=1e-6), (spec[0], d, fwd)
            assert np.allclose(o, np.array(pose.position) + pose.near_clip * fwd, atol=1e-5)
            assert abs(np.linalg.norm(d.astype(np.float64)) - 1) < 1e-6


def test_screen_ray_reprojects_onto_its_pixel(cv):
    dims = (256, 256, 256)
    rng = np.random.default_rng(4)
    W, H = 1920, 1080
    lods = cv.setup_lods(256, W, H)
    for spec in POSES:
        pose = pose_for(cv, cv.World(dims, [], []), spec)
        M = np.array(cv.frame_setup(pose, W, H, lods, 256, limit_horizon=False).camera.world_to_screen[:], dtype=np.float64).reshape(4, 4).T
        for px, py in rng.uniform(0, 1, (50, 2)) * (W, H):
            o, d = cv.screen_ray(pose, px, py, W, H)
            for t in (100.0, 400.0):  # nearer points resolve the fp32 rounding of the origin, not the ray
                p = o.astype(np.float64) + t * d.astype(np.float64)
                clip = M @ np.append(p, 1.0)
                assert abs(clip[0] / clip[3] - px) < 1e-3 and abs(clip[1] / clip[3] - py) < 1e-3, (spec[0], px, py, t, clip)


def test_picking_agrees_with_rendering(cv, mill_world, mill1080):
    """Every 7th pixel of the 1080p oracle frames of mill 256 (POSES, LOD 0 only) picked with the per-cell definition at the pixel
    centre. Measured: 94.75 % of the voxel pixels carry the colour of the voxel the pick hits, and 54 of the 276 871 sky pixels (0.02 %)
    pick a voxel. Both come from the renderer, not the query: the raybuffer traces W + 2H (or 2W + H) rays per screen segment and every
    pixel samples its nearest ray row, so a pixel shows what a ray up to half a row spacing away saw — at silhouettes and across
    one-voxel-thin features (railings, beams) that ray can see a different voxel or the sky."""
    W, H, frames = mill1080
    rw = rco.RayWorld(mill_world)
    total = np.zeros(4, dtype=np.int64)
    for pose, _, frame in frames:
        xs, ys, rays = pick_rays(cv, pose, W, H)
        total += pick_share(cv, frame, xs, ys, rco.raycast(rw, rays))
    agree, voxel, sky_hits, sky = (int(v) for v in total)
    print(f"pick/render agreement {agree}/{voxel} = {agree / voxel:.5f}; sky pixels that pick a voxel {sky_hits}/{sky}")
    assert agree >= 0.92 * voxel, (agree, voxel)
    assert sky_hits <= 0.001 * sky, (sky_hits, sky)


# ---- GPU ----------------------------------------------------------------------------------------------------------------------

gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def rm(cv):
    r = cv.RenderManager(0)
    yield r
    r.destroy()


def _device_raycast(rm, rays, lod):
    import torch
    t_rays = torch.from_numpy(np.ascontiguousarray(rays).view(np.uint8).copy()).cuda()
    t_hits = torch.zeros(len(rays) * 32, dtype=torch.uint8, device="cuda")
    rm.raycast_device(t_rays.data_ptr(), t_hits.data_ptr(), len(rays), lod)
    rm.sync()
    return t_hits.cpu().numpy().view(rco.RAY_HIT_DTYPE)


def _gpu_equals_definition(rm, world, rays):
    rm.upload_world(world)
    rw = rco.RayWorld(world)
    for lod in range(len(world.blobs)):
        ref = rco.raycast(rw, rays, lod)
        for general in (False, True):
            rm.set_general_path(general)
            got = rm.raycast_rays(rays, lod)
            assert same(got, ref), (lod, general, first_mismatch(rays, got, ref))
            got = _device_raycast(rm, rays, lod)
            assert same(got, ref), ("device", lod, general, first_mismatch(rays, got, ref))
    rm.set_general_path(False)


@gpu
def test_gpu_equals_definition_small_worlds(cv, rm):
    rng = np.random.default_rng(2)
    for world, _, _ in (comb_world(cv), irregular_world(cv)):
        _gpu_equals_definition(rm, world, random_rays(rng, world.dims, 20000))
    rm.upload_world(irregular_world(cv)[0])
    assert not rm.world_is_regular()
    for world, _, _, _ in fuzz_worlds(cv):
        _gpu_equals_definition(rm, world, random_rays(rng, world.dims, 200))


@gpu
@pytest.mark.parametrize("name", ["mill_world", "terrain_world", "structure_world"])
def test_gpu_equals_definition_every_lod(cv, rm, request, name):
    world = request.getfixturevalue(name)
    _gpu_equals_definition(rm, world, random_rays(np.random.default_rng(3), world.dims, 20000))


@gpu
def test_gpu_mill1024_resident_pick_grid(cv):
    r = cv.RenderManager(0)
    try:
        P, Cc = parse_obj(MILL)
        host = r.build_world_from_mesh(P, Cc, 1024, flips=(True, False, False))
        r.build_resident_world_from_mesh(P, Cc, 1024, flips=(True, False, False))
        rw = rco.RayWorld(host)
        W, H = 1920, 1080
        for k in range(6):
            pose = limited(cv, cv.benchmark_pose(cv.benchmark_length() * k / 5, host.dims, far_clip=2048.0))
            _, _, rays = pick_rays(cv, pose, W, H, stride=5)
            got = r.raycast_rays(rays)
            ref = rco.raycast(rw, rays)
            assert same(got, ref), (k, first_mismatch(rays, got, ref))
            assert np.mean(got["hit"] == 1) > 0.05
    finally:
        r.destroy()


@gpu
def test_gpu_picking_agrees_with_rendering(cv, mill_world, mill1080):
    W, H, frames = mill1080
    r = cv.RenderManager(0)
    try:
        r.upload_world(mill_world)
        r.set_resolution(W, H)
        rw = rco.RayWorld(mill_world)
        for pose, setup, oframe in frames:
            r.draw_setup(setup)
            r.sync()
            frame = r.read_frame()
            xs, ys, rays = pick_rays(cv, pose, W, H)
            hits = r.raycast_rays(rays)
            assert same(hits, rco.raycast(rw, rays))
            assert np.array_equal(frame, oframe)
            assert pick_share(cv, frame, xs, ys, hits) == pick_share(cv, oframe, xs, ys, rco.raycast(rw, rays))
    finally:
        r.destroy()


@gpu
def test_gpu_ordering_and_errors(cv, terrain_world, structure_world):
    from cpuvox_b200 import native as N
    r = cv.RenderManager(0)
    try:
        # errors
        ray = cv.make_rays([[1.0, 300.0, 1.0]], [[0.1, -1.0, 0.2]])
        hit = np.zeros(1, dtype=cv.RAY_HIT_DTYPE)
        p = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
        assert N.lib.cvx_raycast(r._ctx, p(ray), 1, 0, p(hit), 0) == -5        # CVX_ERR_NO_WORLD
        w4 = cv.World(terrain_world.dims, terrain_world.blobs[:4], terrain_world.column_counts[:4])
        r.upload_world(w4)
        assert N.lib.cvx_raycast(r._ctx, p(ray), 1, 4, p(hit), 0) == -1         # LOD 4 not uploaded
        assert N.lib.cvx_raycast(r._ctx, p(ray), 1, 6, p(hit), 0) == -1
        assert N.lib.cvx_raycast(r._ctx, p(ray), -1, 0, p(hit), 0) == -1
        assert N.lib.cvx_raycast(r._ctx, None, 1, 0, p(hit), 0) == -1
        assert N.lib.cvx_raycast(r._ctx, p(ray), 1, 0, None, 1) == -1
        launches = r.launch_count()
        assert N.lib.cvx_raycast(r._ctx, None, 0, 0, None, 0) == 0 and r.launch_count() == launches
        rw = rco.RayWorld(w4)
        assert same(r.raycast_rays(ray), rco.raycast(rw, ray))
        assert r.raycast_rays(ray)["hit"][0] == 1
        # 5 M rays in one call (scratch growth), then a small call reusing it
        big = random_rays(np.random.default_rng(9), w4.dims, 5_000_000)
        assert same(r.raycast_rays(big, 1), rco.raycast(rw, big, 1))
        assert same(r.raycast_rays(big[:1000], 2), rco.raycast(rw, big[:1000], 2))
        # a raycast issued while two asynchronous batches are outstanding
        W, H = 640, 360
        r.set_resolution(W, H)
        poses = [cv.CameraPose.from_euler((128.0, 200.0 + 5 * i, 128.0), (50.0, 20.0 * i, 0.0), far_clip=512.0) for i in range(8)]
        setups = [r.make_setup(q) for q in poses]
        dst = [cv.alloc_pinned((len(setups), H, W)) for _ in range(2)]
        b0 = r.draw_batch_async(setups[:4], dst[0])
        b1 = r.draw_batch_async(setups[4:], dst[1])
        rays = random_rays(np.random.default_rng(10), w4.dims, 100000)
        got = r.raycast_rays(rays)
        r.batch_wait(b0)
        r.batch_wait(b1)
        assert same(got, rco.raycast(rw, rays))
        for i, s in enumerate(setups):
            r.draw_setup(s)
            r.sync()
            assert np.array_equal(r.read_frame(), dst[i // 4][i % 4]), i
        # a world replacement is seen by the next query (host and device paths)
        r.upload_world(structure_world)
        rs = random_rays(np.random.default_rng(11), structure_world.dims, 100000)
        ref = rco.raycast(rco.RayWorld(structure_world), rs)
        assert same(r.raycast_rays(rs), ref)
        assert same(_device_raycast(r, rs, 0), ref)
        assert same(r.raycast_rays(rays[:1]), rco.raycast(rco.RayWorld(structure_world), rays[:1]))
        # pick: the screen ray through the library
        r.upload_world(terrain_world)
        r.set_resolution(320, 180)
        pose = poses[0]
        h = r.pick(pose, 160.5, 90.5)
        o, d = cv.screen_ray(pose, 160.5, 90.5, 320, 180)
        assert same(np.array([h]), rco.raycast(rco.RayWorld(terrain_world), cv.make_rays(o[None], d[None])))
    finally:
        r.destroy()
