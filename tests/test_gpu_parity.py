"""Parity tests proper: the CUDA path, called through the C ABI (cpuvox_b200/libcpuvox_b200.so), against the CPU oracle on the
same inputs — bit-exact raybuffers, frame and work counters — and against the committed golden fixtures. Run on a B200:
    python -m pytest tests -m gpu
north_star's tolerance is >= 99.5 % identical pixels with the rest off by <= 1 pixel / 1 LSB at span boundaries; these
tests hold the stricter bar of 100 % identical (tolerance = 0), which the IEEE-fp32, no-FMA kernels meet."""
from __future__ import annotations

import json
import os

import numpy as np
import pytest

from conftest import COMB_POSES, MILL, POSES, ROOT, comb_world, crc, irregular_world, limited, parse_obj, pose_for, setup_for
from rle import encode_world

pytestmark = pytest.mark.gpu

SKY = 0x191919FF
MAGENTA = 0xFF | (255 << 8) | (20 << 16) | (147 << 24)
RESOLUTIONS = [(320, 180), (333, 217), (256, 400)]


@pytest.fixture(scope="module")
def rm(cv):
    m = cv.RenderManager(0, counters=True)
    yield m
    m.destroy()


def _oracle_frame(orc, ow, s, W, H, fill):
    td = np.full((W + 2 * H, H), fill, dtype=np.uint32)
    lr = np.full((2 * W + H, W), fill, dtype=np.uint32)
    os_ = orc.copy_setup(s)
    td, lr, cn = orc.render_raybuffers(ow, os_, W, H, td=td, lr=lr)
    return td, lr, cn, orc.blit(os_, W, H, td, lr)


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


def _translated_reference():
    """oracle/ref.py when the reference's library can be built, else None: the tests that compare with the reference then check
    the stored vectors alone."""
    from oracle import ref
    return ref if ref.build() else None


def _golden(name):
    with open(os.path.join(ROOT, "tests", "golden", name)) as f:
        return json.load(f)


def _assert_same(g, o, what):
    for name, a, b in zip(("top/down raybuffer", "left/right raybuffer"), g[:2], o[:2]):
        bad = int((a != b).sum())
        assert bad == 0, f"{what}: {name} differs in {bad} of {a.size} pixels"
    assert g[2] == o[2], f"{what}: counters {g[2]} != {o[2]}"
    bad = int((g[3] != o[3]).sum())
    assert bad == 0, f"{what}: frame differs in {bad} pixels"


def test_product_library_is_the_one_loaded(cv, rm):
    maps = open("/proc/self/maps").read()
    assert "libcpuvox_b200.so" in maps
    assert rm.launch_count() >= 0


@pytest.mark.parametrize("group", [0, 8, 16])
@pytest.mark.parametrize("world_name", ["terrain_world", "structure_world", "mill_world"])
def test_matches_oracle_all_poses(cv, orc, rm, request, world_name, group):
    """Every pose class x 3 resolutions (16:9, odd sizes, portrait), all three lane-group widths of the Phase-1 kernel."""
    world = request.getfixturevalue(world_name)
    ow = orc.OracleWorld(world.dims, world.blobs, world.column_counts)
    rm.upload_world(world)
    assert rm.world_is_regular(), "builder-made worlds are regular: the boundary-table kernel is the one under test at group 0/32"
    rm.set_group_size(group)
    for (W, H) in RESOLUTIONS:
        rm.set_resolution(W, H)
        for spec in POSES:
            s = setup_for(cv, world, spec, W, H)
            _assert_same(_gpu_frame(rm, s, MAGENTA), _oracle_frame(orc, ow, s, W, H, MAGENTA), f"{world_name} {spec[0]} {W}x{H} g{group}")
    rm.set_group_size(0)


def test_matches_golden_fixtures(cv, rm, terrain_world, structure_world, mill_world):
    """File-based reference (tests/golden/golden_v1.json, made by tests/golden/make_golden.py): no oracle call here."""
    with open(os.path.join(ROOT, "tests", "golden", "golden_v1.json")) as f:
        golden = json.load(f)["worlds"]
    worlds = {"terrain256": terrain_world, "structure512x128x256": structure_world, "mill256": mill_world}
    specs = {p[0]: p for p in POSES}
    for name, g in golden.items():
        w = worlds[name]
        rm.upload_world(w)
        for c in g["cases"]:
            W, H = c["width"], c["height"]
            rm.set_resolution(W, H)
            s = setup_for(cv, w, specs[c["pose"]], W, H)
            td, lr, cn, frame = _gpu_frame(rm, s, 0)
            assert cn == c["counters"], (name, c["pose"], W, H)
            assert (crc(td), crc(lr), crc(frame)) == (c["td_crc"], c["lr_crc"], c["frame_crc"]), (name, c["pose"], W, H)


@pytest.mark.parametrize("world_name", ["terrain_world", "structure_world", "mill_world"])
def test_matches_the_translated_reference(cv, rm, request, world_name):
    """CUDA raybuffers vs oracle/_ref — the reference's own DrawSegmentRayJob.cs / SegmentDDAData.cs / CameraData.cs /
    World.cs / RenderManager.DrawSegments translated to C++ (oracle/ref.py) — tolerance 0: against the CRCs it recorded for these
    very cases (tests/golden/golden_ref_v1.json) and, where its library can be built, against its raybuffers live; then the frame
    against the reference's BlitSegments + shader through the stand-in rasteriser within north_star's tolerance (>= 99.5 %
    identical pixels)."""
    world = request.getfixturevalue(world_name)
    g = _golden("golden_ref_v1.json")["worlds"][{"terrain_world": "terrain256", "structure_world": "structure512x128x256", "mill_world": "mill256"}[world_name]]
    assert [crc(b) for b in world.blobs] == g["blob_crcs"], world_name
    recorded = {(c["pose"], c["width"], c["height"]): (c["td_crc"], c["lr_crc"]) for c in g["cases"]}
    ref = _translated_reference()
    rw = ref.RefWorld(world.dims, world.blobs, world.column_counts) if ref else None
    rm.upload_world(world)
    rm.set_counters(False)
    for (W, H) in RESOLUTIONS:
        rm.set_resolution(W, H)
        for spec in POSES:
            s = setup_for(cv, world, spec, W, H)
            rm.clear_raybuffers(0)
            rm.draw_setup(s)
            rm.sync()
            td, lr = rm.read_raybuffers()
            frame = rm.read_frame()
            assert (crc(td), crc(lr)) == recorded[(spec[0], W, H)], (world_name, spec[0], W, H)
            if rw is None:
                continue
            rtd, rlr = ref.render_raybuffers(rw, ref.copy_setup(s), W, H)
            assert np.array_equal(td, rtd) and np.array_equal(lr, rlr), (world_name, spec[0], W, H)
            rframe = ref.blit(ref.copy_setup(s), W, H, rtd, rlr)
            assert (frame == rframe).mean() >= 0.995, (world_name, spec[0], W, H, (frame == rframe).mean())
    rm.set_counters(True)


def test_matches_golden_vectors_made_by_the_reference(cv, rm, terrain_world, structure_world, mill_world):
    """tests/golden/golden_ref_v1.json: raybuffer CRCs produced by the translated reference's RenderManager.DrawWorld from the
    recorded camera poses (tests/golden/make_golden_ref.py). No oracle, no reference library at run time."""
    with open(os.path.join(ROOT, "tests", "golden", "golden_ref_v1.json")) as f:
        golden = json.load(f)["worlds"]
    worlds = {"terrain256": terrain_world, "structure512x128x256": structure_world, "mill256": mill_world}
    rm.set_counters(False)
    for name, g in golden.items():
        w = worlds[name]
        assert [crc(b) for b in w.blobs] == g["blob_crcs"], name
        rm.upload_world(w)
        for c in g["cases"]:
            W, H = c["width"], c["height"]
            rm.set_resolution(W, H)
            pose = cv.CameraPose(tuple(c["position"]), tuple(c["rotation"]), far_clip=c["far_clip"])
            s = cv.frame_setup(pose, W, H, np.array(c["lod_distances"], dtype=np.float32), w.dims[1], limit_horizon=False)
            assert crc(np.frombuffer(bytes(s), dtype=np.uint8)) == c["setup_crc"], (name, c["pose"], W, H)
            rm.clear_raybuffers(0)
            rm.draw_setup(s)
            rm.sync()
            td, lr = rm.read_raybuffers()
            assert (crc(td), crc(lr)) == (c["td_crc"], c["lr_crc"]), (name, c["pose"], W, H)
    rm.set_counters(True)


def test_mill_1024_matches_the_translated_reference_1080p(cv, rm):
    """BASELINE config 1 at full size against the reference's own code: mill 1024^3, 1920x1080, 6 poses of the benchmark path
    (outside the world, looking up, the dive, the roll, the end pose). Against the raybuffer CRCs of
    tests/golden/golden_mill1024_v1.json (its "generator" says what recorded them, tests/golden/make_golden_mill1024.py) and,
    where the reference's library can be built, against its raybuffers live."""
    world = cv.World.from_obj(MILL, 1024)
    g = _golden("golden_mill1024_v1.json")
    assert [crc(b) for b in world.blobs] == g["blob_crcs"]
    ref = _translated_reference()
    rw = ref.RefWorld(world.dims, world.blobs, world.column_counts) if ref else None
    rm.upload_world(world)
    rm.set_counters(False)
    W, H = 1920, 1080
    rm.set_resolution(W, H)
    poses = cv.benchmark_path(world.dims, 60, far_clip=2.0 * world.max_dimension)
    for i in (0, 12, 24, 36, 48, 59):
        s = rm.make_setup(poses[i])
        rm.clear_raybuffers(0)
        rm.draw_setup(s)
        rm.sync()
        td, lr = rm.read_raybuffers()
        assert (crc(td), crc(lr)) == tuple(g["cases"][str(i)]), i
        if rw is not None:
            rtd, rlr = ref.render_raybuffers(rw, ref.copy_setup(s), W, H)
            assert np.array_equal(td, rtd) and np.array_equal(lr, rlr), i
    rm.set_counters(True)


def test_world_file_written_by_the_reference_uploads_and_renders(cv, orc, rm, tmp_path):
    """f1 on the device: datasets/mill.obj -> the reference's own voxelizer / builder / WorldSaveFile.Serialize (oracle/_ref) ->
    .world file -> cvx_world_file_read -> cvx_world_upload -> frames bit-equal to the directly built world's and to the oracle's;
    and the library's own writer/reader round trip gives the same frames. Where the reference's library cannot be built, the file
    is the library writer's (byte for byte the reference's Serialize: test_world_file_interop_with_the_reference) and the blobs
    read from it must carry the CRCs the reference's own builder recorded for mill256 (tests/golden/golden_ref_v1.json)."""
    ref = _translated_reference()
    path = tmp_path / "mill256_ref.world"
    direct = cv.World.from_obj(MILL, 256)
    if ref is not None:
        P, Cc = parse_obj(MILL)
        ref.build_world_from_mesh(P, Cc, np.arange(P.shape[0]), 256, save_to=path)
    else:
        direct.save(str(path))
    loaded = cv.World.load(str(path))
    assert [crc(b) for b in loaded.blobs] == _golden("golden_ref_v1.json")["worlds"]["mill256"]["blob_crcs"]
    path2 = tmp_path / "mill256_ours.world"
    direct.save(str(path2))
    again = cv.World.load(str(path2))
    ow = orc.OracleWorld(loaded.dims, loaded.blobs, loaded.column_counts)
    W, H = 333, 217
    rm.set_resolution(W, H)
    frames = []
    for w in (loaded, direct, again):
        rm.upload_world(w)
        got = []
        for spec in POSES[:5]:
            s = setup_for(cv, direct, spec, W, H)
            g = _gpu_frame(rm, s, 0)
            if w is loaded:
                _assert_same(g, _oracle_frame(orc, ow, s, W, H, 0), f".world from the reference, {spec[0]}")
            got.append(g[3])
        frames.append(got)
    for a, b, c in zip(*frames):
        assert np.array_equal(a, b) and np.array_equal(a, c)


def test_counters_off_gives_identical_pixels(cv, rm, mill_world):
    rm.upload_world(mill_world)
    rm.set_resolution(333, 217)
    s = setup_for(cv, mill_world, POSES[0], 333, 217)
    a = _gpu_frame(rm, s, 0)
    rm.set_counters(False)
    b = _gpu_frame(rm, s, 0)
    rm.set_counters(True)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and np.array_equal(a[3], b[3])
    assert all(v == 0 for v in b[2].values())


def test_ray_ranges_blit_rows_and_owned_blits_compose(cv, rm, terrain_world):
    """The multi-GPU building blocks: ray ranges and row ranges partition the work without changing a pixel, and owned
    blits over disjoint ray ranges write disjoint pixels whose union is the frame."""
    world = terrain_world
    rm.upload_world(world)
    W, H = 333, 217
    rm.set_resolution(W, H)
    s = setup_for(cv, world, POSES[8], W, H)
    td, lr, cn, frame = _gpu_frame(rm, s, 0)
    total = cn["rays"]
    rm.clear_raybuffers(0)
    rm.counters()
    cuts = [0, total // 3, total // 2 + 5, total]
    for a, b in zip(cuts[:-1], cuts[1:]):
        rm.draw_rays(s, a, b)
    for a, b in ((0, 100), (100, 101), (101, H)):
        rm.blit_rows(s, a, b)
    rm.sync()
    td2, lr2 = rm.read_raybuffers()
    assert np.array_equal(td, td2) and np.array_equal(lr, lr2) and rm.counters() == cn
    assert np.array_equal(rm.read_frame(), frame)
    import torch
    acc = np.zeros((H, W), dtype=np.uint64)
    for a, b in zip(cuts[:-1], cuts[1:]):
        buf = torch.zeros(H * W, dtype=torch.int32, device="cuda:0")
        rm.blit_owned(s, a, b, buf.data_ptr())
        rm.sync()
        part = buf.cpu().numpy().view(np.uint32).reshape(H, W)
        assert ((acc != 0) & (part != 0)).sum() == 0, "owned pixels must be disjoint"
        acc += part
    assert np.array_equal(acc.astype(np.uint32), frame)


def test_frame_ring_shares_compose_on_one_device(cv, rm, terrain_world, mill_world):
    """The ray-sharded path of SURVEY.md §8(e) without a second GPU: a frame ring for N ranks lives in this process, every rank's share
    of a view (cvx_draw_sharded: Phase 1 of its rays, Phase 2 of the pixels they feed — strips of tiles, most of them skipped) is stored
    into the same ring frame, and the consumed frame must equal the single-launch frame bit for bit: interleaved chunks and contiguous
    ranges, 2 / 3 / 8 ranks, widths that end inside a tile and inside a strip of tiles."""
    from conftest import partition_rays_even
    for world, W, H in ((terrain_world, 1000, 600), (mill_world, 1920, 1080), (terrain_world, 333, 217)):
        rm.upload_world(world)
        rm.set_resolution(W, H)
        rm.set_frames_in_flight(1)
        out = cv.alloc_pinned((1, H, W))
        view = 0
        for spec in (POSES[0], POSES[3], POSES[8]):
            s = rm.make_setup(pose_for(cv, world, spec))
            rm.draw_setup(s)
            rm.sync()
            want = rm.read_frame().copy()
            total = sum(max(0, s.segments[k].ray_count) for k in range(4))
            for n, chunk in ((2, 32), (3, 0), (8, 512), (8, 64)):
                rm.ring_create(4, n)
                out[:] = 0
                for r in range(n):
                    if chunk:
                        rm.draw_sharded(s, -1, chunk, view, r)
                    else:
                        b, e = partition_rays_even(total, n, r)
                        rm.draw_sharded(s, b, e, view, r)
                rm.ring_consume(view, out[0])
                rm.sync()
                rm.ring_status()
                assert np.array_equal(out[0], want), (W, H, spec[0], n, chunk)
                rm.ring_close()
    rm.set_frames_in_flight(6)


def test_draw_batch_equals_individual_draws(cv, rm, mill_world):
    world = mill_world
    rm.upload_world(world)
    W, H = 320, 180
    rm.set_resolution(W, H)
    setups = [setup_for(cv, world, spec, W, H) for spec in POSES]
    singles = []
    for s in setups:
        rm.draw_setup(s)
        rm.sync()
        singles.append(rm.read_frame().copy())
    dst = cv.alloc_pinned((len(setups), H, W))
    dst[:] = 0
    rm.draw_batch(setups, dst)
    for i, f in enumerate(singles):
        assert np.array_equal(dst[i], f), i
    # every number of views in flight gives the same frames (views render concurrently on separate streams / buffer sets), and
    # the device-only form leaves the LAST view's frame and raybuffers readable
    for k in (1, 2, 3, 8):
        rm.set_frames_in_flight(k)
        dst[:] = 0
        rm.draw_batch(setups, dst)
        for i, f in enumerate(singles):
            assert np.array_equal(dst[i], f), (k, i)
        rm.draw_batch(setups)
        assert np.array_equal(rm.read_frame(), singles[-1]), k
    # a batch much longer than the views in flight
    many = [setups[(7 * i) % len(setups)] for i in range(37)]
    big = cv.alloc_pinned((len(many), H, W))
    for k in (2, 6):
        rm.set_frames_in_flight(k)
        big[:] = 0
        rm.draw_batch(many, big)
        for i in range(len(many)):
            assert np.array_equal(big[i], singles[(7 * i) % len(setups)]), (k, i)
        assert np.array_equal(rm.read_frame(), singles[(7 * 36) % len(setups)]), k   # the last view also stays readable on the device
        rm.draw_batch(many)
        assert np.array_equal(rm.read_frame(), singles[(7 * 36) % len(setups)]), k
    rm.set_frames_in_flight(4)
    with pytest.raises(cv.CvxError):
        rm.set_frames_in_flight(17)


def test_asynchronous_batches_deliver_the_same_frames(cv, rm, mill_world):
    """cvx_draw_batch_async: three batches outstanding at once (each into its own pinned destination, the later ones rendering while the
    earlier ones' frames are still being copied out; the framebuffer pool and the last view's buffer are shared between them), waited for
    out of order, mixed with synchronous calls: every frame equals the single draw."""
    rm.upload_world(mill_world)
    W, H = 640, 360
    rm.set_resolution(W, H)
    setups = [rm.make_setup(pose_for(cv, mill_world, spec)) for spec in POSES]
    singles = []
    for s in setups:
        rm.draw_setup(s)
        rm.sync()
        singles.append(rm.read_frame().copy())
    orders = [[(3 * i + b) % len(setups) for i in range(41)] for b in range(3)]   # longer than the pool of 32 framebuffers
    dsts = [cv.alloc_pinned((41, H, W)) for _ in range(3)]
    for k in (6, 2):
        rm.set_frames_in_flight(k)
        for d in dsts:
            d[:] = 0
        ids = [rm.draw_batch_async([setups[j] for j in orders[b]], dsts[b]) for b in range(3)]
        assert ids[1] == ids[0] + 1 and ids[2] == ids[0] + 2
        for b in (1, 0, 2):
            rm.batch_wait(ids[b])
            for i, j in enumerate(orders[b]):
                assert np.array_equal(dsts[b][i], singles[j]), (k, b, i)
        assert np.array_equal(rm.read_frame(), singles[orders[2][-1]])       # the last view of the last batch stays readable
        # a synchronous batch right behind an asynchronous one
        dsts[0][:] = 0; dsts[1][:] = 0
        b0 = rm.draw_world_batch_async([pose_for(cv, mill_world, POSES[j]) for j in orders[0]], dsts[0])
        rm.draw_batch([setups[j] for j in orders[1]], dsts[1])
        for i, j in enumerate(orders[1]):
            assert np.array_equal(dsts[1][i], singles[j]), (k, "sync", i)
        rm.batch_wait(b0)
        for i, j in enumerate(orders[0]):
            assert np.array_equal(dsts[0][i], singles[j]), (k, "async world", i)
        # a single draw right behind an asynchronous batch (with 2 views in flight the batch's last view sits in the framebuffer the single
        # draw writes): the draw is ordered behind the batch's copies
        dsts[2][:] = 0
        b2 = rm.draw_batch_async([setups[j] for j in orders[2]], dsts[2])
        rm.draw_setup(setups[5])
        rm.blit_raybuffer(0)
        rm.batch_wait(b2)
        for i, j in enumerate(orders[2]):
            assert np.array_equal(dsts[2][i], singles[j]), (k, "single behind async", i)
        rm.sync()
    with pytest.raises(cv.CvxError):
        rm.batch_wait(10 ** 6)
    with pytest.raises(cv.CvxError):
        rm.draw_batch_async(setups[:1], dsts[0])
    rm.set_frames_in_flight(6)
    for d in dsts:
        cv.native.lib.cvx_free_pinned(d.ctypes.data)


def test_draw_world_batch_equals_setup_batch(cv, rm, mill_world):
    """cvx_draw_world_batch (poses in, host setup inside the library) == cvx_draw_batch of the setups the host computes itself."""
    rm.upload_world(mill_world)
    W, H = 320, 180
    rm.set_resolution(W, H)
    poses = [pose_for(cv, mill_world, POSES[k]) for k in (0, 3, 4, 7, 9)]   # includes the horizon pose (LimitRotationHorizon applies)
    setups = [rm.make_setup(p) for p in poses]
    a = cv.alloc_pinned((len(poses), H, W))
    b = cv.alloc_pinned((len(poses), H, W))
    rm.set_counters(False)
    rm.draw_batch(setups, a)
    rm.draw_world_batch(poses, b)
    rm.set_counters(True)
    assert np.array_equal(a, b)
    assert (a != 0).all()
    for x in (a, b):
        cv.native.lib.cvx_free_pinned(x.ctypes.data)


def test_ray_setup_state_matches_oracle(cv, orc, rm, mill_world):
    """RaySetupJob + DDASetupJob + TraceToFirstColumnJob (DrawSegmentRayJob.cs:12-144), including rays that start outside
    the world (StepToWorldIntersection) and rays skybox-filled before the march."""
    world = mill_world
    ow = orc.OracleWorld(world.dims, world.blobs, world.column_counts)
    rm.upload_world(world)
    W, H = 320, 180
    rm.set_resolution(W, H)
    for spec in POSES:
        s = setup_for(cv, world, spec, W, H)
        g = rm.ray_setup(s)
        o = orc.ray_setup(ow, orc.copy_setup(s), W, H)
        assert len(g) == len(o)
        for field in g.dtype.names:
            assert np.array_equal(g[field].view(np.uint32), o[field].view(np.uint32)), (spec[0], field)


def test_hand_made_worlds(cv, orc, rm):
    """Empty world -> all skybox; a single three-voxel column -> its colours bottom to top (orientation and colour order)."""
    dims = (32, 32, 32)
    lods = np.full(6, 1e9, dtype=np.float32)
    W, H = 320, 180
    rm.set_resolution(W, H)
    blob, cc = encode_world(np.zeros(dims, dtype=np.uint32))
    rm.upload_world(cv.World(dims, [blob], [cc], [0]))
    pose = cv.CameraPose.from_euler((16.5, 10.5, 4.0), (0.0, 0.0, 0.0), far_clip=64.0)
    s = cv.frame_setup(pose, W, H, lods, dims[1])
    td, lr, cn, frame = _gpu_frame(rm, s, 0)
    assert (frame == SKY).all() and cn["px_voxel"] == 0 and cn["runs_visited"] == 0
    grid = np.zeros(dims, dtype=np.uint32)
    c_bot, c_mid, c_top = 0x0000FFFF, 0x00FF00FF, 0xFF0000FF
    grid[16, 9, 16], grid[16, 10, 16], grid[16, 11, 16] = c_bot, c_mid, c_top
    blob, cc = encode_world(grid)
    world = cv.World(dims, [blob], [cc], [3])
    rm.upload_world(world)
    g = _gpu_frame(rm, s, 0)
    col = g[3][:, W // 2]
    seq = [int(c) for i, c in enumerate(col) if c != SKY and (i == 0 or col[i - 1] != c)]
    assert seq == [c_bot, c_mid, c_top]
    ow = orc.OracleWorld(dims, [blob], [cc])
    _assert_same(g, _oracle_frame(orc, ow, s, W, H, 0), "single column")


def test_tall_columns_near_plane_and_irregular_worlds(cv, orc, rm):
    """Columns of 70..128 runs (several round-cache passes), cameras inside geometry (runs straddling the near plane), and a world
    that is not made of full-height valid runs (must be classified irregular and rendered by the general kernel)."""
    lods = np.full(6, 1e9, dtype=np.float32)
    world, blob, cc = comb_world(cv)
    ow = orc.OracleWorld(world.dims, [blob], [cc])
    rm.upload_world(world)
    assert rm.world_is_regular()
    for (W, H) in [(320, 180), (200, 300)]:
        rm.set_resolution(W, H)
        for pos, eul in COMB_POSES:
            s = cv.frame_setup(cv.CameraPose.from_euler(pos, eul, far_clip=200.0), W, H, lods, world.dims[1])
            _assert_same(_gpu_frame(rm, s, MAGENTA), _oracle_frame(orc, ow, s, W, H, MAGENTA), f"comb {pos} {eul} {W}x{H}")
    world, blob, cc = irregular_world(cv)
    ow = orc.OracleWorld(world.dims, [blob], [cc])
    rm.upload_world(world)
    assert not rm.world_is_regular()
    W, H = 256, 192
    rm.set_resolution(W, H)
    for pos, eul in [((16.5, 40.5, 2.5), (10, 0, 0)), ((16.5, 70.5, 16.5), (75, 30, 0)), ((3.5, 20.5, 3.5), (-30, 45, 0))]:
        s = cv.frame_setup(cv.CameraPose.from_euler(pos, eul, far_clip=100.0), W, H, lods, world.dims[1])
        _assert_same(_gpu_frame(rm, s, MAGENTA), _oracle_frame(orc, ow, s, W, H, MAGENTA), f"irregular {pos} {eul}")


def test_debug_views_and_presentation(cv, orc, rm, mill_world, tmp_path):
    """f4: the shader's COPY_MAIN1 / COPY_MAIN2 debug views (RayBufferBlit.shader:48-53) against the oracle's restatement, after
    the magenta clear the reference uses (RenderManager.cs:58-92); cvx_present against numpy byte shuffles; the .bmp writer."""
    rm.upload_world(mill_world)
    for (W, H) in ((320, 180), (333, 217)):
        rm.set_resolution(W, H)
        s = rm.make_setup(pose_for(cv, mill_world, POSES[0]))
        rm.clear_raybuffers(MAGENTA)
        rm.draw_setup(s)
        rm.sync()
        frame = rm.read_frame()
        td, lr = rm.read_raybuffers()
        for which, buf in ((0, td), (1, lr)):
            rm.blit_raybuffer(which)
            rm.sync()
            got = rm.read_frame()
            want = orc.blit_raybuffer(buf, W, H)
            assert np.array_equal(got, want), f"debug view {which} at {W}x{H}"
            assert (got == MAGENTA).any() and (got != MAGENTA).any()   # untouched rows/pixels stay magenta, written ones do not
        rm.draw_setup(s)   # back to the normal frame
        rm.sync()
        assert np.array_equal(rm.read_frame(), frame)
        b = frame.view(np.uint8).reshape(H, W, 4)   # bytes a, r, g, b
        rgba = np.stack([b[..., 1], b[..., 2], b[..., 3], b[..., 0]], axis=-1)
        bgra = np.stack([b[..., 3], b[..., 2], b[..., 1], b[..., 0]], axis=-1)
        assert np.array_equal(rm.present(0, top_down=False), rgba)
        assert np.array_equal(rm.present(0, top_down=True), rgba[::-1])
        assert np.array_equal(rm.present(1, top_down=True), bgra[::-1])
        assert np.array_equal(rm.present(1, top_down=False), bgra)
        assert np.array_equal(rm.present(2, top_down=True), rgba[::-1, :, :3])    # packed RGB8: word path at W % 4 == 0, byte path else
        assert np.array_equal(rm.present(2, top_down=False), rgba[:, :, :3])
    # device destination: a torch buffer stands in for a mapped graphics resource
    import torch
    dst = torch.zeros(H * W, dtype=torch.int32, device="cuda:0")
    rm.present_device(dst.data_ptr(), 0, True)
    rm.sync()
    assert np.array_equal(dst.cpu().numpy().view(np.uint8).reshape(H, W, 4), rgba[::-1])
    with pytest.raises(cv.CvxError):
        rm.present(7)
    with pytest.raises(cv.CvxError):
        rm.blit_raybuffer(2)


def test_present_jpeg_decodes_to_the_frame(cv, rm, mill_world):
    """f4, encode of the device framebuffer: cvx_present_jpeg (frame -> RGB8 on the device -> nvJPEG CUDA encoder) must decode, with an
    independent decoder (Pillow), to the frame within JPEG's loss: PSNR > 38 dB at quality 95 4:4:4, > 30 dB at quality 75 4:2:0, and the
    bitstream must be much smaller than the frame. Odd sizes included (partial MCUs, the byte path of the RGB8 packer)."""
    import io
    from PIL import Image
    rm.upload_world(mill_world)
    for (W, H) in ((1280, 720), (333, 217)):
        rm.set_resolution(W, H)
        rm.draw_setup(rm.make_setup(pose_for(cv, mill_world, POSES[1])))
        rm.sync()
        want = rm.present(2, top_down=True).astype(np.float64)
        for quality, sub, floor_db in ((95, 0, 38.0), (75, 1, 30.0)):
            data = rm.present_jpeg(quality, sub)
            assert data[:2] == b"\xff\xd8" and data[-2:] == b"\xff\xd9"
            assert len(data) < W * H * 3 // 3
            img = Image.open(io.BytesIO(data))
            assert img.size == (W, H) and img.mode == "RGB"
            got = np.asarray(img).astype(np.float64)
            psnr = 10.0 * np.log10(255.0 ** 2 / max(1e-9, ((got - want) ** 2).mean()))
            assert psnr > floor_db, (W, H, quality, sub, psnr)
    with pytest.raises(cv.CvxError):
        rm.present_jpeg(0)
    with pytest.raises(cv.CvxError):
        rm.present_jpeg(90, 5)


def test_gpu_world_builder_matches_host_builder(cv, rm):
    """f2: voxelizer + RLE + LOD mips on the device (cvx_gpu_builder_from_mesh) against the host restatement of
    VoxelizerHelper / WorldBuilder.ToFinalColumn / World.DownSample — every LOD blob byte for byte, voxel counts included."""
    import time
    for maxdim in (128, 256, 1024):
        t0 = time.perf_counter()
        host = cv.World.from_obj(MILL, maxdim)
        t1 = time.perf_counter()
        dev = rm.build_world_from_obj(MILL, maxdim)
        t2 = time.perf_counter()
        assert dev.dims == host.dims and dev.column_counts == host.column_counts and dev.voxel_counts == host.voxel_counts
        assert len(dev.blobs) == len(host.blobs)
        for lod, (a, b) in enumerate(zip(dev.blobs, host.blobs)):
            assert a.nbytes == b.nbytes, f"mill {maxdim} LOD {lod}: blob sizes {a.nbytes} != {b.nbytes}"
            assert np.array_equal(a, b), f"mill {maxdim} LOD {lod}: {int((a != b).sum())} bytes differ"
        print(f"mill {maxdim}^3: host builder {t1 - t0:.3f} s, device builder {t2 - t1:.3f} s (incl. blob download), {host.voxel_counts[0]} voxels")
    # a random triangle soup with random vertex colours, no flip and all three flips. Its triangles lie in the unit cube, so the
    # world is 256^3; non-cubic worlds and the other edges are in test_world_production.py
    rng = np.random.default_rng(17)
    pos = rng.uniform(0.0, 1.0, size=(300 * 3, 3)).astype(np.float32) * np.array([1.0, 0.45, 0.7], dtype=np.float32)
    tri_c = rng.uniform(0.0, 1.0, size=(300, 1, 3)).astype(np.float32)
    pos = (tri_c + 0.08 * (pos.reshape(300, 3, 3) - 0.5)).reshape(-1, 3).astype(np.float32)
    col = rng.integers(0, 256, size=(900, 4), dtype=np.uint8)
    col[:, 3] = 255
    for flips in ((False, False, False), (True, True, True)):
        host = cv.World.from_mesh(pos, col, 200, flips=flips)
        dev = rm.build_world_from_mesh(pos, col, 200, flips=flips)
        assert dev.dims == host.dims and dev.voxel_counts == host.voxel_counts and len(dev.blobs) == len(host.blobs) == 6
        for lod, (a, b) in enumerate(zip(dev.blobs, host.blobs)):
            assert np.array_equal(a, b), f"soup flips {flips} LOD {lod}"
    # mesh -> resident world without leaving the device (cvx_world_build_from_mesh): frames equal those of the uploaded host-built world
    W, H = 640, 360
    rm.set_resolution(W, H)
    rm.upload_world(host)
    pose = cv.CameraPose.from_euler((0.5 * host.dims[0], 0.9 * host.dims[1], 0.5 * host.dims[2]), (50.0, 20.0, 0.0), far_clip=2.0 * host.max_dimension)
    want = _gpu_frame(rm, rm.make_setup(pose), 0)
    res = rm.build_resident_world_from_mesh(pos, col, 200, flips=flips)
    assert res.dims == host.dims and res.voxel_counts == host.voxel_counts and rm.world_is_regular()
    got = _gpu_frame(rm, rm.make_setup(pose), 0)
    _assert_same(got, want, "resident device-built world")
    assert int((got[3] != SKY).sum()) > 1000
    # fewer LODs on request
    dev3 = rm.build_world_from_mesh(pos, col, 200, flips=flips, lods=3)
    assert len(dev3.blobs) == 3
    for a, b in zip(dev3.blobs, host.blobs[:3]):
        assert np.array_equal(a, b)
    with pytest.raises(cv.CvxError):
        rm.build_world_from_mesh(pos[:2], col[:2], 200)


def test_error_paths(cv):
    from cpuvox_b200 import native as N
    m = cv.RenderManager(0)
    try:
        s = N.FrameSetup()
        with pytest.raises(cv.CvxError) as e:
            m.draw_setup(s)
        assert e.value.code == -5  # CVX_ERR_NO_WORLD
        blob, cc = encode_world(np.zeros((8, 8, 8), dtype=np.uint32))
        with pytest.raises(cv.CvxError):
            m.upload_world(cv.World((12, 8, 8), [blob], [cc], [0]))  # x not a power of two
        bad = blob.copy()
        bad.view(np.uint32)[0:3] = (1 << 20, 5, 0)  # column 0 points far outside the element area
        with pytest.raises(cv.CvxError) as e:
            m.upload_world(cv.World((8, 8, 8), [bad], [cc], [0]))
        assert e.value.code == -8  # CVX_ERR_FORMAT
        # a run whose colour range (ColorsIndex + Length) leaves the element area: Phase 1 would gather out of bounds
        g = np.zeros((8, 8, 8), dtype=np.uint32)
        g[3, 2:5, 4] = 0x11223344
        blob2, cc2 = encode_world(g)
        words = blob2.copy().view(np.uint32)
        hdr = words[:3 * cc2].reshape(cc2, 3)
        col = 3 * 8 + 4
        cells = words[3 * cc2:]
        k = int(hdr[col, 0]) + 1
        solid = next(i for i in range(k, k + int(hdr[col, 1] & 0xFFFF)) if (int(cells[i]) & 0xFFFF) < 0x8000)
        cells[solid] = (int(cells[solid]) & 0xFFFF0000) | 0x7F00  # ColorsIndex 32512
        with pytest.raises(cv.CvxError) as e:
            m.upload_world(cv.World((8, 8, 8), [words.view(np.uint8)], [cc2], [3]))
        assert e.value.code == -8  # CVX_ERR_FORMAT
        m.upload_world(cv.World((8, 8, 8), [blob], [cc], [0]))
        with pytest.raises(cv.CvxError) as e:
            m.draw_setup(s)
        assert e.value.code == -6  # CVX_ERR_NO_RESOLUTION
        m.set_resolution(64, 48)
        s.segments[0].ray_count = -3
        s.segments[1].ray_count = 10
        with pytest.raises(cv.CvxError) as e:
            m.draw_setup(s)
        assert e.value.code == -1  # CVX_ERR_INVALID_ARGUMENT: negative ray count
        with pytest.raises(cv.CvxError):
            m.draw_batch([N.FrameSetup(), s])  # refused before anything is enqueued
        m.sync()
        with pytest.raises(cv.CvxError):
            m.set_resolution(0, 100)
        with pytest.raises(cv.CvxError):
            m.set_group_size(7)
    finally:
        m.destroy()


def test_world_with_fewer_lods_than_distances(cv, orc, rm):
    """A 3-LOD world drawn with SetupLods' six default distances and a far clip beyond all of them: the reference would index
    LODs that do not exist (DrawSegmentRayJob.cs:237-243, unchecked); the library never leaves the last uploaded LOD, which equals
    the oracle run with the distances of the missing LODs at infinity."""
    world = cv.World.from_obj(MILL, 256, lods=3)
    assert len(world.blobs) == 3
    ow = orc.OracleWorld(world.dims, world.blobs, world.column_counts)
    rm.upload_world(world)
    W, H = 320, 180
    rm.set_resolution(W, H)
    lods = cv.setup_lods(world.max_dimension, W, H)
    inf_lods = lods.copy()
    inf_lods[2:] = np.inf
    for spec in POSES[:6]:
        pose = pose_for(cv, world, spec, far_scale=8.0)
        s = cv.frame_setup(pose, W, H, lods, world.dims[1])
        so = cv.frame_setup(pose, W, H, inf_lods, world.dims[1])
        _assert_same(_gpu_frame(rm, s, 0), _oracle_frame(orc, ow, so, W, H, 0), f"3-LOD world {spec[0]}")


@pytest.fixture(scope="module")
def mill_1024(cv):
    return cv.World.from_obj(MILL, 1024)


@pytest.mark.parametrize("res,frames", [((1920, 1080), 60), ((3840, 2160), 12)])
def test_benchmark_path_full_size(cv, orc, rm, mill_1024, res, frames):
    """BASELINE config 1 at full size: datasets/mill.obj at 1024^3, the BenchmarkPath.anim camera path, 1080p (all 60 poses)
    and 4K (12 poses) — bit-exact against the oracle, plus the size-independent invariants (every writable pixel written
    exactly once, nothing else touched)."""
    world = mill_1024
    ow = orc.OracleWorld(world.dims, world.blobs, world.column_counts)
    rm.upload_world(world)
    W, H = res
    rm.set_resolution(W, H)
    poses = cv.benchmark_path(world.dims, frames, far_clip=2.0 * world.max_dimension)
    for i, pose in enumerate(poses):
        s = rm.make_setup(pose)
        g = _gpu_frame(rm, s, MAGENTA)
        o = _oracle_frame(orc, ow, s, W, H, MAGENTA)
        _assert_same(g, o, f"mill1024 {W}x{H} pose {i}")
        assert (g[3] != MAGENTA).all() and (g[3] != 0).all()
        written = int((g[0] != MAGENTA).sum() + (g[1] != MAGENTA).sum())
        assert written == g[2]["px_voxel"] + g[2]["px_sky"]


@pytest.fixture(scope="module")
def terrain_2048(cv):
    return cv.World.synthetic(0, (2048, 2048, 2048), seed=1234)


def test_terrain_2048_configs_2_3_full_size(cv, orc, rm, terrain_2048):
    """BASELINE configs 2 and 3 at FULL size: the fBm terrain 2048^3 (seed 1234); config 2 = 1920x1080, camera at the centre, y 1700,
    pitch 60 down (vanishing point on screen, 4 segments); config 3 = 3840x2160, 40 above the ground, pitch 3 and pitch 0
    (LimitRotationHorizon, clamped segments). Raybuffers, counters and frame bit-exact vs the oracle, raybuffers also vs the
    translated reference where its library can be built (oracle/ref.py)."""
    ref = _translated_reference()
    world = terrain_2048
    ow = orc.OracleWorld(world.dims, world.blobs, world.column_counts)
    rw = ref.RefWorld(world.dims, world.blobs, world.column_counts) if ref else None
    rm.upload_world(world)
    hdr = np.asarray(world.blobs[0])[: 12 * world.column_counts[0]].view(np.uint32).reshape(-1, 3)
    ground = int(hdr[1024 * 2048 + 1024, 2] & 0xFFFF)
    cases = [((1920, 1080), cv.CameraPose.from_euler((1024.0, 1700.0, 1024.0), (60.0, 30.0, 0.0), far_clip=4096.0), 4),
             ((3840, 2160), cv.CameraPose.from_euler((1024.5, ground + 40.0, 1024.5), (3.0, 75.0, 0.0), far_clip=4096.0), None),
             ((3840, 2160), cv.CameraPose.from_euler((1024.5, ground + 40.0, 1024.5), (0.0, 165.0, 0.0), far_clip=4096.0), None)]
    for (W, H), pose, segs in cases:
        rm.set_resolution(W, H)
        s = rm.make_setup(pose)
        if segs:
            assert sum(1 for k in range(4) if s.segments[k].ray_count > 0) == segs
        g = _gpu_frame(rm, s, 0)
        _assert_same(g, _oracle_frame(orc, ow, s, W, H, 0), f"terrain 2048^3 {W}x{H}")
        if rw is not None:
            rtd, rlr = ref.render_raybuffers(rw, ref.copy_setup(s), W, H)
            assert np.array_equal(g[0], rtd) and np.array_equal(g[1], rlr), f"terrain 2048^3 {W}x{H} vs the translated reference"


def test_structure_world_config4_full_size(cv, orc, rm):
    """BASELINE config 4 at FULL size: boxes/pipes/slabs 4096x1024x4096 (seed 7, a 4.5 GB LOD-0 blob), 7680x4320, far 8192, two of the
    bench's four views: bit-exact vs the oracle."""
    world = cv.World.synthetic(1, (4096, 1024, 4096), seed=7)
    ow = orc.OracleWorld(world.dims, world.blobs, world.column_counts)
    rm.upload_world(world)
    W, H = 7680, 4320
    rm.set_resolution(W, H)
    for pos, euler in (((2048.5, 700.5, 2048.5), (35.0, 20.0, 0.0)), ((3000.5, 950.5, 1000.5), (70.0, 200.0, 10.0))):
        s = rm.make_setup(cv.CameraPose.from_euler(pos, euler, far_clip=8192.0))
        _assert_same(_gpu_frame(rm, s, 0), _oracle_frame(orc, ow, s, W, H, 0), f"structures 4096x1024x4096 8K {pos}")
    rm.upload_world(cv.World.synthetic(0, (64, 64, 64), seed=1))   # release the 6 GB world before the next tests
    rm.set_resolution(320, 180)


def test_structure_world_8k_and_batched_cameras_configs_4_5(cv, orc, rm):
    """BASELINE config 4 shape at a second, smaller size (X != Z, other camera classes) and config 5 (seeded random cameras at
    1280x720 over the terrain, rendered as one batch) at test size; bench.py --config 4 / 5 are the full-size runs (DESIGN.md §7)."""
    world = cv.World.synthetic(1, (1024, 256, 1024), seed=7)
    ow = orc.OracleWorld(world.dims, world.blobs, world.column_counts)
    rm.upload_world(world)
    W, H = 7680, 4320
    rm.set_resolution(W, H)
    for pos, euler in (((512.5, 180.5, 512.5), (35.0, 20.0, 0.0)), ((100.5, 90.5, 200.5), (8.0, 50.0, 0.0))):
        s = rm.make_setup(cv.CameraPose.from_euler(pos, euler, far_clip=2048.0))
        _assert_same(_gpu_frame(rm, s, 0), _oracle_frame(orc, ow, s, W, H, 0), f"structures 8K {pos}")
    terrain = cv.World.synthetic(0, (1024, 1024, 1024), seed=1234)
    ow = orc.OracleWorld(terrain.dims, terrain.blobs, terrain.column_counts)
    rm.upload_world(terrain)
    W, H = 1280, 720
    rm.set_resolution(W, H)
    rng = np.random.default_rng(99)
    poses = [cv.CameraPose.from_euler((float(rng.uniform(0, 1024)), float(rng.uniform(800, 950)), float(rng.uniform(0, 1024))),
                                      (float(rng.uniform(-30, 80)), float(rng.uniform(0, 360)), 0.0), far_clip=2048.0) for _ in range(12)]
    setups = [rm.make_setup(p) for p in poses]
    dst = cv.alloc_pinned((len(setups), H, W))
    rm.set_counters(False)
    rm.draw_batch(setups, dst)
    rm.set_counters(True)
    for i, s in enumerate(setups):
        o = _oracle_frame(orc, ow, s, W, H, 0)
        assert np.array_equal(dst[i], o[3]), f"batched camera {i}"
    cv.native.lib.cvx_free_pinned(dst.ctypes.data)


def test_fuzz_random_worlds_and_cameras(cv, orc, rm):
    """Seeded fuzz through the C ABI: 300 random small worlds x 4 random cameras (inside geometry, outside the world, steep, rolled,
    random resolution and far clip) — raybuffers, counters and frame bit-exact against the oracle, product and counter builds and
    the general kernel included (_gpu_frame)."""
    from conftest import random_world_and_cameras
    rng = np.random.default_rng(424242)
    lods = np.full(6, 1e9, dtype=np.float32)
    for it in range(300):
        world, blob, cc, W, H, poses = random_world_and_cameras(cv, rng)
        ow = orc.OracleWorld(world.dims, [blob], [cc])
        rm.upload_world(world)
        rm.set_resolution(W, H)
        for k, pose in enumerate(poses):
            s = cv.frame_setup(pose, W, H, lods, world.dims[1])
            _assert_same(_gpu_frame(rm, s, MAGENTA), _oracle_frame(orc, ow, s, W, H, MAGENTA), f"fuzz world {it} {world.dims} {W}x{H} camera {k}")
