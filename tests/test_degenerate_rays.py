"""The renderer on axis-aligned rays and degenerate poses: a seeded corpus of cameras whose rays have a direction component of
exactly 0, integer and half-integer coordinates, positions on and outside the world faces, pitches of exactly 0 and ±90, and
screens from 1x1 to the 8192-pixel axis limit (CVXD_MAX_AXIS).

The fuzz elsewhere draws from continuous distributions and never lands on these inputs. Here each restatement of Phase 1 is compared
on them: the C++ oracle against the independent Python restatement (oracle/pyref.py), the kernel source through the SIMT emulator
against the oracle, and on the GPU the CUDA kernels against the oracle. The still-axis rule and the LOD bound of DESIGN.md §3.1/§5
and the math.min/math.max NaN rule are what these edges exercise; the corpus asserts that it reaches them."""
from __future__ import annotations

import itertools

import numpy as np
import pytest

import emu
from rle import encode_world

SKY = 0x191919FF
MAGENTA = 0xFF | (255 << 8) | (20 << 16) | (147 << 24)
F32 = np.float32

SMALL_DIMS = (16, 16, 32)
RESOLUTIONS = [(1, 1), (2, 1), (1, 2), (3, 3), (7, 300), (300, 7), (63, 31), (64, 32), (65, 33), (8192, 64), (64, 8192)]
YAWS = (0.0, 90.0, 180.0, 270.0, 45.0)
PITCHES = (90.0, -90.0, 89.999, -89.999, 45.0, -45.0, 1e-3, -1e-3, 0.0)   # pitch 0 is drawn with and without the horizon limit
ROLLS = (0.0, 90.0, 180.0)


# ---- worlds ----------------------------------------------------------------------------------------------------------------------
def _colour(rng, n):
    return rng.integers(1, 2 ** 32 - 1, size=n, dtype=np.uint64).astype(np.uint32) | 0xFF


def _edge_world(cv, solid_edges):
    """16x16x32 heightmap whose first and last columns along x and z are empty, or solid from floor to top (the two outcomes of a
    still-axis ray entering through a face: the reference walks on from the first column, or stops there)."""
    rng = np.random.default_rng(11)
    dx, dy, dz = SMALL_DIMS
    grid = np.zeros(SMALL_DIMS, dtype=np.uint32)
    h = rng.integers(1, dy, size=(dx, dz))
    for x in range(dx):
        for z in range(dz):
            grid[x, :h[x, z], z] = _colour(rng, 1)[0]
    grid[4:6, 10:14, 8:20] = _colour(rng, 1)[0]   # an overhang: columns of several runs
    edge = np.zeros((dx, dz), dtype=bool)
    edge[0, :] = edge[-1, :] = edge[:, 0] = edge[:, -1] = True
    cols = grid.transpose(0, 2, 1)   # (x, z, y) view
    cols[edge] = 0
    if solid_edges:
        cols[edge] = _colour(rng, int(edge.sum()))[:, None]
    blob, cc = encode_world(grid)
    return cv.World(SMALL_DIMS, [blob], [cc], [int((grid != 0).sum())])


@pytest.fixture(scope="module")
def worlds(cv):
    """name -> World. The two multi-LOD worlds are drawn with SetupLods' distances, so rays switch LODs; `fewer_lods` has 2 LODs for
    6 finite distances, so rays reach the last LOD and must stay there."""
    return {
        "edges_empty": _edge_world(cv, False),
        "edges_solid": _edge_world(cv, True),
        "multi_lod": cv.World.synthetic(0, (64, 64, 64), seed=5, lods=6),
        "fewer_lods": cv.World.synthetic(1, (64, 32, 32), seed=9, lods=2),
    }


def _lods(cv, world, W, H):
    if len(world.blobs) == 1:
        return np.full(6, 1e9, dtype=np.float32)
    return cv.setup_lods(world.max_dimension, W, H)


# ---- cameras ---------------------------------------------------------------------------------------------------------------------
def _positions(dims):
    """Integer, half-integer and fractional coordinates; on the faces (0 and dim); outside each of the four sides and the corners;
    above and below the world and at y == dimY."""
    dx, dy, dz = (float(d) for d in dims)
    my = dy / 2
    return [
        (dx / 2, my, dz / 2), (dx / 2 + 0.5, my + 0.5, dz / 2 + 0.5), (dx * 0.3 + 0.17, my - 0.31, dz * 0.6 + 0.29),
        (0.0, my, dz / 2 + 0.5), (dx, my, dz / 2), (dx / 2 + 0.5, my, 0.0), (dx / 2, my, dz),
        (-3.0, my, dz / 2), (-3.0, my, dz / 2 + 0.5), (-2.75, my, dz / 2 + 0.375), (dx + 3.0, my, dz / 2), (dx + 2.5, my, dz / 3 + 0.25),
        (dx / 2, my, -4.0), (dx / 2 + 0.5, my, -3.5), (dx / 3 + 0.3, my, dz + 3.0), (dx / 2, my, dz + 2.5),
        (-3.0, my, -3.0), (dx + 2.5, my, dz + 2.5), (-2.5, my, dz + 3.0), (dx + 3.0, my, -2.5),
        (dx / 2 + 0.5, dy + 4.0, dz / 2 + 0.5), (dx / 2, -3.0, dz / 2), (dx / 2 + 0.5, dy, dz / 2), (-3.0, dy, dz / 2),
    ]


def _eulers():
    """(pitch, yaw, roll, limit_horizon): every yaw x pitch x roll; pitch 0 twice, with and without LimitRotationHorizon."""
    out = []
    for p, y, r in itertools.product(PITCHES, YAWS, ROLLS):
        out.append((p, y, r, True))
        if p == 0.0:
            out.append((p, y, r, False))
    return out


# Still-axis rays entering through a world face: yaw 90 / 270 (x moves, z still) and 0 / 180 (z moves, x still) from outside, at an
# integer, half-integer and fractional still coordinate, looking nearly straight down (the top/down segments then hold the
# axis-aligned ray) and at 45 degrees. Drawn on every small world and small screen.
PINNED = [((-3.0, 8.0, z), (p, yaw, 0.0)) for z in (16.0, 16.5, 16.375) for p in (89.999, 45.0, -89.999) for yaw in (90.0, 270.0)] + \
         [((19.0, 8.0, z), (89.999, yaw, 0.0)) for z in (16.0, 16.25) for yaw in (270.0, 90.0)] + \
         [((x, 8.0, -3.0), (p, yaw, 0.0)) for x in (8.0, 8.5, 7.625) for p in (89.999, 45.0) for yaw in (0.0, 180.0)] + \
         [((8.0, 8.0, 35.0), (89.999, 180.0, 0.0)), ((8.5, 8.0, 35.0), (89.999, 180.0, 0.0))]


PINNED_RESOLUTIONS = ((1, 2), (3, 3), (7, 300), (64, 32))


def corpus(cv, worlds):
    """The seeded, deterministic list of cases: (world name, W, H, CameraPose, limit_horizon)."""
    rng = np.random.default_rng(2024)
    eulers = _eulers()
    cases = []
    for name, world in worlds.items():
        dims = world.dims
        pos = _positions(dims)
        size = float(max(dims))
        for (W, H) in RESOLUTIONS:
            big = max(W, H) >= 8192
            per = 1 if big else (3 if max(W, H) >= 300 else 8)
            if name in ("edges_empty", "edges_solid") and (W, H) in PINNED_RESOLUTIONS:
                for p, e in PINNED:
                    cases.append((name, W, H, cv.CameraPose.from_euler(p, e, far_clip=2.0 * size), False))
            for _ in range(per):
                p = pos[int(rng.integers(len(pos)))]
                pitch, yaw, roll, lim = eulers[int(rng.integers(len(eulers)))]
                far = (1.5, 2.0 * size, 1e6)[int(rng.integers(3))]
                cases.append((name, W, H, cv.CameraPose.from_euler(p, (pitch, yaw, roll), far_clip=far), lim))
        if name in ("edges_empty", "edges_solid"):   # straight up and down on odd screens: the vanishing point on a pixel centre
            for (W, H), pitch, yaw in itertools.product(((1, 1), (3, 3)), (90.0, -90.0), (0.0, 90.0, 45.0)):
                cases.append((name, W, H, cv.CameraPose.from_euler(pos[1], (pitch, yaw, 0.0), far_clip=2.0 * size), False))
    return cases


@pytest.fixture(scope="module")
def cases(cv, worlds):
    return corpus(cv, worlds)


def _setup(cv, worlds, case):
    name, W, H, pose, lim = case
    world = worlds[name]
    return cv.frame_setup(pose, W, H, _lods(cv, world, W, H), world.dims[1], limit_horizon=lim)


def _tag(case):
    name, W, H, pose, lim = case
    return f"{name} {W}x{H} pos={tuple(pose.position)} rot={tuple(pose.rotation)} far={pose.far_clip} limit={lim}"


@pytest.fixture(scope="module")
def oracle_worlds(orc, worlds):
    return {k: orc.OracleWorld(w.dims, w.blobs, w.column_counts) for k, w in worlds.items()}


def _oracle_frame(orc, ow, s, W, H, fill):
    td = np.full((W + 2 * H, H), fill, dtype=np.uint32)
    lr = np.full((2 * W + H, W), fill, dtype=np.uint32)
    os_ = orc.copy_setup(s)
    td, lr, cn = orc.render_raybuffers(ow, os_, W, H, td=td, lr=lr)
    return td, lr, cn, orc.blit(os_, W, H, td, lr)


# ---- the corpus reaches its edges ------------------------------------------------------------------------------------------------
def test_corpus_reaches_its_edges(cv, orc, worlds, oracle_worlds, cases):
    """Minimum counts of the inputs this file exists for, so that a change of the corpus cannot quietly drop them."""
    still_int = still_frac = vp_centre = zero_rays = lod_switched = 0
    for case in cases:
        name, W, H = case[:3]
        s = _setup(cv, worlds, case)
        vp = np.array(s.vanishing_point_screen, dtype=np.float64)
        if np.all(np.isfinite(vp)) and np.all(np.abs(vp - np.floor(vp) - 0.5) <= 1e-6):   # a pixel centre up to the setup's rounding
            vp_centre += 1
        if sum(max(0, s.segments[k].ray_count) for k in range(4)) == 0:
            zero_rays += 1
            continue
        st = orc.ray_setup(oracle_worlds[name], orc.copy_setup(s), W, H)
        dims = worlds[name].dims
        pos = np.floor(st["start"].astype(np.float64))
        outside = (pos[:, 0] < 0) | (pos[:, 1] < 0) | (pos[:, 0] >= dims[0]) | (pos[:, 1] >= dims[2])
        for k in range(2):
            still = outside & (st["dir"][:, k] == 0)
            frac = st["start"][still, k] % 1     # the coordinate that does not move
            still_int += int((frac == 0).sum())
            still_frac += int((frac != 0).sum())
        lod_switched += int((st["lod"] > 0).sum())
    assert still_int >= 20, f"rays starting outside with a zero direction component at an integer still coordinate: {still_int}"
    assert still_frac >= 20, f"... at a fractional still coordinate: {still_frac}"
    assert vp_centre >= 10, f"setups with the vanishing point within 1e-6 of a pixel centre: {vp_centre}"
    assert zero_rays >= 5, f"setups with zero rays: {zero_rays}"
    assert lod_switched >= 40, f"rays that enter the world at a LOD above 0: {lod_switched}"


def test_setup_lod_stays_in_the_world(cv, orc, worlds, oracle_worlds, cases):
    """TraceToFirstColumnJob's LOD loop never leaves the uploaded LODs, whatever the entry distance (a still axis once made it +inf
    and the loop ran to LOD 106)."""
    for case in cases:
        name, W, H = case[:3]
        s = _setup(cv, worlds, case)
        st = orc.ray_setup(oracle_worlds[name], orc.copy_setup(s), W, H)
        if len(st):
            n = len(worlds[name].blobs)
            assert st["lod"].min() >= 0 and st["lod"].max() <= n - 1, (_tag(case), int(st["lod"].max()))
            entered = (st["status"] == 0) & np.isfinite(st["dir"]).all(axis=1)
            assert np.isfinite(st["intersection_distances"][entered]).all(), f"{_tag(case)}: a ray that enters the world has a non-finite entry distance"


# ---- CPU legs --------------------------------------------------------------------------------------------------------------------
def test_oracle_equals_python_restatement(cv, orc, worlds, oracle_worlds, cases):
    """oracle/cpuvox_oracle.cpp == oracle/pyref.py, raybuffers and frame, on the small screens of the corpus."""
    from oracle import pyref
    n = 0
    for case in cases:
        name, W, H = case[:3]
        pose = case[3]
        steep = abs(pyref._quat_rotate(pose.rotation, (0.0, 0.0, 1.0))[1]) > 0.99
        if W * H > 300 and not (W * H <= 2200 and name in ("edges_empty", "edges_solid") and steep):
            continue   # pyref is slow: the small screens, and the still-axis cases seen from nearly straight above
        world = worlds[name]
        s = _setup(cv, worlds, case)
        pw = [pyref.PyWorldLod(world.dims, l, b, c) for l, (b, c) in enumerate(zip(world.blobs, world.column_counts))]
        os_ = orc.copy_setup(s)
        otd, olr, _ = orc.render_raybuffers(oracle_worlds[name], os_, W, H)
        ptd, plr = pyref.render_raybuffers(pw, s, W, H)
        assert np.array_equal(otd, ptd), f"{_tag(case)}: top/down raybuffer differs in {int((otd != ptd).sum())} pixels"
        assert np.array_equal(olr, plr), f"{_tag(case)}: left/right raybuffer differs in {int((olr != plr).sum())} pixels"
        of, pf = orc.blit(os_, W, H, otd, olr), pyref.blit(s, W, H, ptd, plr)
        assert np.array_equal(of, pf), f"{_tag(case)}: frame differs in {int((of != pf).sum())} pixels"
        n += 1
    assert n >= 150


def test_emulated_kernel_equals_oracle(cv, orc, worlds, oracle_worlds, cases):
    """The Phase-1 kernel source through the SIMT emulator == the oracle, raybuffers and counters, on every case below the 8192 axis
    (the GPU legs draw those): the boundary-table kernel everywhere, the general kernel up to 65x33, and on the screens of at most
    9 pixels also at 8 and 16 lanes and with the counters compiled out."""
    ews = {k: emu.EmuWorld(w) for k, w in worlds.items()}
    for case in cases:
        name, W, H = case[:3]
        if max(W, H) >= 8192:
            continue   # the 8192 axis is drawn on the GPU
        s = _setup(cv, worlds, case)
        otd, olr, ocn, _ = _oracle_frame(orc, oracle_worlds[name], s, W, H, MAGENTA)
        tiny, small = W * H <= 9, max(W, H) <= 65
        for variant, group, counters in itertools.product((1, 0) if small else (1,), (32, 16, 8) if tiny else (32,), (True, False) if tiny else (True,)):
            td, lr, cn = emu.render_raybuffers(ews[name], s, W, H, variant=variant, group=group, counters=counters, fill=MAGENTA)
            tag = f"{_tag(case)} kernel={'boundary-table' if variant else 'general'} g{group} counters={counters}"
            assert np.array_equal(td, otd), f"{tag}: top/down raybuffer differs in {int((td != otd).sum())} pixels"
            assert np.array_equal(lr, olr), f"{tag}: left/right raybuffer differs in {int((lr != olr).sum())} pixels"
            assert cn is None or cn == ocn, f"{tag}: counters {cn} != {ocn}"


def _shim_min_max(a, b):
    """Unity.Mathematics math.min / math.max as the reference build pins them: isnan(y) || x < y ? x : y (and > for max)."""
    mn = np.where(np.isnan(b) | (a < b), a, b)
    mx = np.where(np.isnan(b) | (a > b), a, b)
    return mn, mx


def test_min_max_follow_the_reference_rule_on_nan_zero_and_inf():
    """Every pair of {NaN, ±0, ±inf, ±1, 2.5, the smallest denormal}: the oracle's m_min/m_max, the kernel's minf_/maxf_ (emulated) and
    pyref's umin/umax give the very operand the rule picks, bit for bit (a NaN second operand gives the first; a tie, including
    +0 against -0, gives the second)."""
    from oracle import oracle as orc
    from oracle import pyref
    vals = np.array([np.nan, 0.0, -0.0, np.inf, -np.inf, 1.0, -1.0, 2.5], dtype=F32)
    vals = np.append(vals, np.array([1], dtype=np.uint32).view(F32))
    a, b = (x.ravel() for x in np.meshgrid(vals, vals, indexing="ij"))
    want_min, want_max = _shim_min_max(a, b)
    bits = lambda x: np.asarray(x, dtype=F32).view(np.uint32)   # noqa: E731
    for who, (mn, mx) in (("oracle", orc.min_max(a, b)), ("kernel", emu.min_max(a, b)),
                          ("pyref", ([pyref.umin(x, y) for x, y in zip(a, b)], [pyref.umax(x, y) for x, y in zip(a, b)]))):
        for op, got, want in (("min", mn, want_min), ("max", mx, want_max)):
            bad = np.nonzero(bits(got) != bits(want))[0]
            assert len(bad) == 0, f"{who} {op}: " + ", ".join(f"({a[i]!r}, {b[i]!r}) -> {np.asarray(got)[i]!r}, want {want[i]!r}" for i in bad[:6])
    # the cases that decide it: a NaN second operand, and a signed-zero tie
    assert (want_min[np.isnan(a) & (b == 1.0)] == 1.0).all() and (want_min[(a == 1.0) & np.isnan(b)] == 1.0).all()
    assert bits(want_max[(bits(a) == 0) & (bits(b) == 0x80000000)])[0] == 0x80000000


# ---- GPU legs --------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def rm(cv):
    m = cv.RenderManager(0, counters=True)
    yield m
    m.destroy()


def _gpu_frame(rm, s, fill):
    """Renders twice: with the work counters on (every column the reference enters is entered, so the counts are exact)
    and in the product configuration (counters compiled out, columns that provably cannot write are skipped); the pixels of
    both must be identical, and the caller compares them and the counters with the oracle."""
    rm.clear_raybuffers(fill)
    rm.counters()
    rm.draw_setup(s)
    rm.sync()
    td, lr = rm.read_raybuffers()
    cn, frame = rm.counters(), rm.read_frame()
    rm.set_counters(False)
    rm.clear_raybuffers(fill)
    rm.draw_setup(s)
    rm.sync()
    td2, lr2 = rm.read_raybuffers()
    frame2 = rm.read_frame()
    assert np.array_equal(td, td2) and np.array_equal(lr, lr2) and np.array_equal(frame, frame2), "product build differs from counter build"
    if rm.world_is_regular():
        # the same frame through the general kernel (element area, run by run) instead of the boundary-table kernel
        rm.set_general_path(True)
        rm.clear_raybuffers(fill)
        rm.draw_setup(s)
        rm.sync()
        td3, lr3 = rm.read_raybuffers()
        rm.set_general_path(False)
        assert np.array_equal(td, td3) and np.array_equal(lr, lr3), "general kernel differs from the boundary-table kernel"
    rm.set_counters(True)
    return td, lr, cn, frame


def _assert_same(g, o, what):
    for name, a, b in zip(("top/down raybuffer", "left/right raybuffer"), g[:2], o[:2]):
        bad = int((a != b).sum())
        assert bad == 0, f"{what}: {name} differs in {bad} of {a.size} pixels"
    assert g[2] == o[2], f"{what}: counters {g[2]} != {o[2]}"
    bad = int((g[3] != o[3]).sum())
    assert bad == 0, f"{what}: frame differs in {bad} pixels"


def _by_world_and_size(cases):
    out = {}
    for case in cases:
        out.setdefault((case[0], case[1], case[2]), []).append(case)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("group", [0, 8, 16])
def test_cuda_equals_oracle_on_the_corpus(cv, orc, rm, worlds, oracle_worlds, cases, group):
    """CUDA == oracle bit for bit on every case: raybuffers, work counters and frame, counters on and off, boundary-table and general
    kernel; the setup state of every ray equals the oracle's on every field."""
    rm.set_group_size(group)
    try:
        for (name, W, H), group_cases in _by_world_and_size(cases).items():
            rm.upload_world(worlds[name])
            rm.set_resolution(W, H)
            for case in group_cases:
                s = _setup(cv, worlds, case)
                _assert_same(_gpu_frame(rm, s, MAGENTA), _oracle_frame(orc, oracle_worlds[name], s, W, H, MAGENTA), f"{_tag(case)} g{group}")
                if group == 0:
                    g = rm.ray_setup(s)
                    o = orc.ray_setup(oracle_worlds[name], orc.copy_setup(s), W, H)
                    assert len(g) == len(o), _tag(case)
                    for field in o.dtype.names:   # bit for bit, except that any NaN equals any NaN (the payloads are the hardware's)
                        gv, ov = g[field], o[field]
                        same = gv.view(np.uint32) == ov.view(np.uint32)
                        if gv.dtype.kind == "f":
                            same |= np.isnan(gv) & np.isnan(ov)
                        assert same.all(), (_tag(case), field)
    finally:
        rm.set_group_size(0)


@pytest.mark.gpu
def test_cuda_8192_square_on_a_tiny_world(cv, orc, rm):
    """Both axes at the 8192 limit: the longest seen-mask row in both raybuffers, on an 8x8x8 world seen from outside a corner and
    from straight above."""
    rng = np.random.default_rng(3)
    grid = np.zeros((8, 8, 8), dtype=np.uint32)
    m = rng.random(grid.shape) < 0.3
    grid[m] = _colour(rng, int(m.sum()))
    blob, cc = encode_world(grid)
    world = cv.World((8, 8, 8), [blob], [cc], [int(m.sum())])
    ow = orc.OracleWorld(world.dims, world.blobs, world.column_counts)
    rm.upload_world(world)
    W = H = 8192
    rm.set_resolution(W, H)
    lods = np.full(6, 1e9, dtype=np.float32)
    for pos, eul in (((-2.0, 9.0, -2.0), (30.0, 45.0, 0.0)), ((4.0, 12.0, 4.0), (90.0, 90.0, 0.0))):
        s = cv.frame_setup(cv.CameraPose.from_euler(pos, eul, far_clip=32.0), W, H, lods, 8)
        _assert_same(_gpu_frame(rm, s, MAGENTA), _oracle_frame(orc, ow, s, W, H, MAGENTA), f"8192x8192 {pos} {eul}")


@pytest.mark.gpu
@pytest.mark.parametrize("res", [(1, 1), (2, 1), (8192, 64)])
def test_present_and_debug_views_at_edge_sizes(cv, orc, rm, worlds, res):
    """cvx_present in its three formats against NumPy byte shuffles, and the COPY_MAIN1 / COPY_MAIN2 debug views against the oracle,
    on a 1x1 and a 2x1 screen (packed RGB8 byte path) and the 8192-wide one."""
    W, H = res
    world = worlds["edges_solid"]
    rm.upload_world(world)
    rm.set_resolution(W, H)
    s = cv.frame_setup(cv.CameraPose.from_euler((-3.0, 8.0, 16.0), (45.0, 90.0, 0.0), far_clip=64.0), W, H,
                       np.full(6, 1e9, dtype=np.float32), world.dims[1], limit_horizon=False)
    rm.clear_raybuffers(MAGENTA)
    rm.draw_setup(s)
    rm.sync()
    frame = rm.read_frame()
    td, lr = rm.read_raybuffers()
    for which, buf in ((0, td), (1, lr)):
        rm.blit_raybuffer(which)
        rm.sync()
        assert np.array_equal(rm.read_frame(), orc.blit_raybuffer(buf, W, H)), f"debug view {which} at {W}x{H}"
    rm.draw_setup(s)
    rm.sync()
    assert np.array_equal(rm.read_frame(), frame)
    b = frame.view(np.uint8).reshape(H, W, 4)   # bytes a, r, g, b
    rgba = np.stack([b[..., 1], b[..., 2], b[..., 3], b[..., 0]], axis=-1)
    bgra = np.stack([b[..., 3], b[..., 2], b[..., 1], b[..., 0]], axis=-1)
    assert np.array_equal(rm.present(0, top_down=False), rgba)
    assert np.array_equal(rm.present(0, top_down=True), rgba[::-1])
    assert np.array_equal(rm.present(1, top_down=True), bgra[::-1])
    assert np.array_equal(rm.present(1, top_down=False), bgra)
    assert np.array_equal(rm.present(2, top_down=True), rgba[::-1, :, :3])
    assert np.array_equal(rm.present(2, top_down=False), rgba[:, :, :3])
