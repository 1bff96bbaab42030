"""Pins the hand-written oracle (oracle/cpuvox_oracle.cpp) and the product's host code to THE REFERENCE ITSELF.

`oracle/_ref/libcpuvox_ref.so` is the reference's own C# — World.cs, SegmentDDAData.cs, CameraData.cs, RayBuffer.cs,
RenderManager.cs, DrawSegmentRayJob.cs, WordBuilder.cs, VoxelizerHelper.cs, SimpleMesh.cs, RayBufferBlit.shader — translated
token for token to C++ by oracle/refbuild/cs2cpp.py and compiled with g++ (IEEE fp32, no FMA contraction; see oracle/ref.py
for why no .NET build can run here). These tests run on CPU; tests/test_gpu_parity.py checks the CUDA kernels against the
same library and against tests/golden/golden_ref_v1.json (vectors produced by it).
"""
from __future__ import annotations

import json
import os

import numpy as np
import pytest

from conftest import COMB_POSES, MILL, POSES, ROOT, comb_world, crc, irregular_world, limited, parse_obj, pose_for, random_world_and_cameras, setup_for

RES = [(320, 180), (200, 300)]
ONE_LOD = np.full(6, 1e9, dtype=np.float32)  # worlds with LOD 0 only: never leave it (the reference indexes worldLODs unchecked)


def _both(orc, ref, w):
    return orc.OracleWorld(w.dims, w.blobs, w.column_counts), ref.RefWorld(w.dims, w.blobs, w.column_counts)


def _same_raybuffers(orc, ref, ow, rw, s, W, H, what):
    td, lr, _ = orc.render_raybuffers(ow, orc.copy_setup(s), W, H, threads=2)
    rtd, rlr = ref.render_raybuffers(rw, ref.copy_setup(s), W, H, threads=2)
    assert (td == rtd).all() and (lr == rlr).all(), what
    return td, lr


@pytest.mark.parametrize("world_name", ["terrain_world", "structure_world", "mill_world"])
def test_oracle_raybuffers_equal_the_reference(cv, orc, ref, world_name, request):
    """a6-a17: DrawSegments + the four jobs of DrawSegmentRayJob.cs. Tolerance 0 on both raybuffers."""
    w = request.getfixturevalue(world_name)
    ow, rw = _both(orc, ref, w)
    for (W, H) in RES:
        for spec in POSES:
            _same_raybuffers(orc, ref, ow, rw, setup_for(cv, w, spec, W, H), W, H, (world_name, spec[0], W, H))


def test_oracle_equals_reference_on_tall_columns_and_near_plane(cv, orc, ref):
    """70-128 run columns, cameras inside geometry (ClipHomogeneousCameraSpaceLine carrying u), a far clip inside the world."""
    w, blob, cc = comb_world(cv)
    ow, rw = _both(orc, ref, w)
    for (pos, euler) in COMB_POSES:
        for (W, H) in ((160, 120), (97, 211)):
            for far in (512.0, 40.0):
                pose = cv.CameraPose.from_euler(pos, euler, far_clip=far)
                s = cv.frame_setup(pose, W, H, ONE_LOD, 256)
                _same_raybuffers(orc, ref, ow, rw, s, W, H, (pos, euler, W, H, far))


def test_oracle_equals_reference_on_an_irregular_world(cv, orc, ref):
    """Zero-length element inside a column, a column shorter than the world: the reference's loop semantics (IsValid break)."""
    w, blob, cc = irregular_world(cv)
    ow, rw = _both(orc, ref, w)
    for (pos, euler) in [((16.5, 40.5, 16.5), (50, 30, 0)), ((3.5, 70.5, 3.5), (40, 45, 0)), ((16.5, 10.5, 16.5), (-40, 100, 0))]:
        pose = cv.CameraPose.from_euler(pos, euler, far_clip=128.0)
        s = cv.frame_setup(pose, 128, 96, ONE_LOD, 64)
        _same_raybuffers(orc, ref, ow, rw, s, 128, 96, (pos, euler))


def test_oracle_equals_reference_fuzz(cv, orc, ref):
    """150 random small worlds x 4 random cameras (inside, outside, steep, rolled), random resolution and far clip."""
    rng = np.random.default_rng(2024)
    for i in range(150):
        w, blob, cc, W, H, poses = random_world_and_cameras(cv, rng)
        ow, rw = _both(orc, ref, w)
        for pose in poses:
            s = cv.frame_setup(pose, W, H, ONE_LOD, w.dims[1])
            _same_raybuffers(orc, ref, ow, rw, s, W, H, (i, pose))


def test_dda_walk_equals_the_reference(orc, ref):
    """SegmentDDAData ctor / Step / NextLOD (SegmentDDAData.cs:17-73,135-150): cell sequence and distances, bit for bit."""
    rng = np.random.default_rng(9)
    lods = [20.0, 45.0, 100.0, 220.0, 500.0, 1e9]
    for i in range(300):
        start = rng.uniform(-50.0, 300.0, 2).astype(np.float32)
        ang = rng.uniform(0, 2 * np.pi)
        d = np.array([np.cos(ang), np.sin(ang)], dtype=np.float32)
        if i % 10 == 0:
            d = np.array([[1, 0], [0, -1], [-1, 0], [0, 1]][(i // 10) % 4], dtype=np.float32)  # sign(0) = 0
        c0, d0 = orc.dda_walk(start, d, lods, 800.0, 5000)
        c1, d1 = ref.dda_walk(start, d, lods, 800.0, 5000)
        assert c0.shape == c1.shape and (c0 == c1).all() and (d0.view(np.uint32) == d1.view(np.uint32)).all()


def test_segment_setup_equals_the_reference(cv, orc, ref, terrain_world):
    """a1-a5 through the reference's CalculateVanishingPointWorld / ProjectVanishingPointScreenToWorld /
    GetGenericSegmentParameters / CameraData ctor: the product's cvx_host_frame_setup and the oracle's restatement give the
    same 212 bytes. (UnityEngine's Camera/Transform/Matrix4x4 behaviour underneath is an assumption shared by all three:
    SURVEY.md Appendix A2-A7.)"""
    w = terrain_world
    for (W, H) in [(640, 360), (333, 217), (1920, 1080), (3840, 2160)]:
        lods = cv.setup_lods(w.max_dimension, W, H)
        for spec in POSES:
            pose = limited(cv, pose_for(cv, w, spec))
            r = ref.frame_setup(pose.position, pose.rotation, W, H, lods, w.dims[1], far=pose.far_clip)
            s = cv.frame_setup(pose, W, H, lods, w.dims[1], limit_horizon=False)
            o = orc.frame_setup(pose.position, pose.rotation, W, H, lods, w.dims[1], far=pose.far_clip, limit_horizon=False)
            assert bytes(r) == bytes(s) == bytes(o), (spec[0], W, H)


def test_reference_draw_world_equals_its_parts(cv, ref, mill_world):
    """RenderManager.DrawWorld as a whole (ref.draw_world) == setup + DrawSegments + BlitSegments called separately: checks
    the four guards of RenderManager.cs:127-141 that ref_frame_setup_from_pose restates, and the partial-texture plumbing."""
    w = mill_world
    rw = ref.RefWorld(w.dims, w.blobs, w.column_counts)
    W, H = 256, 144
    lods = cv.setup_lods(w.max_dimension, W, H)
    for spec in POSES:
        pose = limited(cv, pose_for(cv, w, spec))
        td, lr, frame = ref.draw_world(rw, pose.position, pose.rotation, W, H, lods, far=pose.far_clip)
        s = ref.frame_setup(pose.position, pose.rotation, W, H, lods, w.dims[1], far=pose.far_clip)
        td2, lr2 = ref.render_raybuffers(rw, s, W, H)
        rows_td = max(0, s.segments[0].ray_count) + max(0, s.segments[1].ray_count)
        rows_lr = max(0, s.segments[2].ray_count) + max(0, s.segments[3].ray_count)
        # DrawWorld only copies the partial textures it used (RayBuffer.ApplyPartials): compare the rows rays wrote
        assert (td[:rows_td] == td2[:rows_td]).all() and (lr[:rows_lr] == lr2[:rows_lr]).all(), spec[0]
        frame2 = ref.blit(s, W, H, td, lr)
        assert (frame == frame2).all(), spec[0]


def _row_frames(orc, ref, s, W, H):
    """Phase 2 on raybuffers whose pixels hold their own row number: the frame then shows which ray row every pixel took."""
    td = np.repeat(np.arange(W + 2 * H, dtype=np.uint32)[:, None], H, 1).copy()
    lr = (np.repeat(np.arange(2 * W + H, dtype=np.uint32)[:, None], W, 1) + (1 << 20)).copy()
    return orc.blit(orc.copy_setup(s), W, H, td, lr), ref.blit(ref.copy_setup(s), W, H, td, lr)


def test_blit_matches_the_reference_within_tolerance(cv, orc, ref, terrain_world):
    """a18: RenderManager.BlitSegments + RayBufferBlit.shader frag through a D3D-rule rasteriser (vertices snapped to 1/256 px,
    integer edge functions, top-left rule) vs the oracle's per-pixel restatement. A GPU's interpolator bits are not
    reproducible (SURVEY.md §8 a18), so this is the one place with a tolerance, north_star's: the rendered frame is identical
    on >= 99.5 % of the pixels; every pixel takes the same ray row or its neighbour (<= 1 % take the neighbour), or, on a
    segment boundary, the neighbouring segment."""
    ow = orc.OracleWorld(terrain_world.dims, terrain_world.blobs, terrain_world.column_counts)
    for (W, H) in ((320, 180), (250, 333)):
        for spec in POSES:
            s = setup_for(cv, terrain_world, spec, W, H)
            td, lr, _ = orc.render_raybuffers(ow, orc.copy_setup(s), W, H, threads=2)
            fa, fb = orc.blit(orc.copy_setup(s), W, H, td, lr), ref.blit(ref.copy_setup(s), W, H, td, lr)
            assert (fa == fb).mean() >= 0.995, (spec[0], W, H, (fa == fb).mean())
            a, b = _row_frames(orc, ref, s, W, H)
            a = a.astype(np.int64)
            b = b.astype(np.int64)
            same_buffer = (a >> 20) == (b >> 20)
            d = np.abs(a - b)
            assert (d != 0).mean() <= 0.01, (spec[0], W, H, (d != 0).mean())
            assert (d[same_buffer] <= 1).all(), (spec[0], W, H, d[same_buffer].max())
            # pixels that took the other raybuffer: only next to a pixel the oracle also gives to that buffer
            ys, xs = np.nonzero(~same_buffer)
            assert len(ys) <= 0.005 * W * H
            for y, x in zip(ys, xs):
                nb = a[max(0, y - 1):y + 2, max(0, x - 1):x + 2] >> 20
                assert ((b[y, x] >> 20) == nb).any(), (spec[0], x, y)


def test_world_builder_equals_the_reference(cv, ref):
    """f2: SimpleMesh.Remap_Internal + VoxelizerHelper.GetVoxelsInternal + RLEColumnBuilder.ToFinalColumn + World.DownSample
    (the reference's own code) vs the product's host builder: all six LOD blobs byte for byte, datasets/mill.obj at 64/128/256
    and a random triangle soup with many shared voxels (colour averaging)."""
    P, Cc = parse_obj(MILL)
    for md in (64, 128, 256):
        w = cv.World.from_obj(MILL, md)
        dims, blobs, ccs, vox = ref.build_world_from_mesh(P, Cc, np.arange(P.shape[0]), md)
        assert tuple(dims) == tuple(w.dims) and list(ccs) == list(w.column_counts) and list(vox) == list(w.voxel_counts)
        for j in range(6):
            assert np.asarray(w.blobs[j]).tobytes() == blobs[j].tobytes(), (md, j)
    rng = np.random.default_rng(77)
    n = 300
    base = rng.uniform(0, 10, (n, 1, 3))
    P2 = (base + rng.normal(0, 0.8, (n, 3, 3))).astype(np.float32).reshape(-1, 3)
    C2 = rng.integers(0, 256, (n * 3, 4), dtype=np.uint8)
    C2[:, 3] = 255
    for flips in ((False, False, False), (True, False, True)):
        w = cv.World.from_mesh(P2, C2, 64, flips=flips)
        dims, blobs, ccs, vox = ref.build_world_from_mesh(P2, C2, np.arange(n * 3), 64, flips=flips)
        assert tuple(dims) == tuple(w.dims) and list(vox) == list(w.voxel_counts)
        for j in range(6):
            assert np.asarray(w.blobs[j]).tobytes() == blobs[j].tobytes(), (flips, j)


def test_column_count_quirk_is_the_references(cv, ref):
    """World.ColumnCount = dimX*dimZ/((lod+1)^2) (World.cs:17), an over-estimate from lod 2 on, read from the reference's own property."""
    for dims in ((256, 256, 256), (512, 128, 256), (64, 32, 128)):
        for lod in range(6):
            assert ref.lib().ref_world_column_count(dims[0], dims[1], dims[2], lod) == (dims[0] * dims[2]) // ((lod + 1) ** 2)
    w = cv.World.synthetic(0, (64, 64, 64), seed=3)
    assert list(w.column_counts) == [ref.lib().ref_world_column_count(64, 64, 64, j) for j in range(6)]


def test_golden_vectors_made_by_the_reference(cv, orc):
    """tests/golden/golden_ref_v1.json was produced by oracle/_ref (tests/golden/make_golden_ref.py, RenderManager.DrawWorld
    from a pose). The oracle must reproduce every raybuffer CRC from the recorded inputs, and the round-1 golden file (made
    by the oracle) must agree with it case by case. Stored vectors only: runs without the reference library."""
    with open(os.path.join(ROOT, "tests", "golden", "golden_ref_v1.json")) as f:
        g = json.load(f)
    with open(os.path.join(ROOT, "tests", "golden", "golden_v1.json")) as f:
        g1 = json.load(f)
    P, Cc = parse_obj(MILL)
    worlds = {"terrain256": cv.World.synthetic(0, (256, 256, 256), seed=1234),
              "structure512x128x256": cv.World.synthetic(1, (512, 128, 256), seed=7),
              "mill256": cv.World.from_obj(MILL, 256)}
    for name, gw in g["worlds"].items():
        w = worlds[name]
        assert [crc(b) for b in w.blobs] == gw["blob_crcs"], name
        ow = orc.OracleWorld(w.dims, w.blobs, w.column_counts)
        old = {(c["pose"], c["width"], c["height"]): c for c in g1["worlds"][name]["cases"]}
        for c in gw["cases"]:
            W, H = c["width"], c["height"]
            s = orc.frame_setup(c["position"], c["rotation"], W, H, c["lod_distances"], w.dims[1], far=c["far_clip"], limit_horizon=False)
            assert crc(np.frombuffer(bytes(s), dtype=np.uint8)) == c["setup_crc"], (name, c["pose"], W, H)
            td, lr, _ = orc.render_raybuffers(ow, s, W, H, threads=2)
            assert (crc(td), crc(lr)) == (c["td_crc"], c["lr_crc"]), (name, c["pose"], W, H)
            o = old[(c["pose"], W, H)]
            assert (o["td_crc"], o["lr_crc"], o["ray_counts"]) == (c["td_crc"], c["lr_crc"], c["ray_counts"])


def test_mill_benchmark_path_equals_the_reference(cv, orc, ref):
    """BASELINE config 1 at reduced size: mill 512^3 (LOD switches on the path), 640x360, 12 poses of the benchmark path."""
    w = cv.World.from_obj(MILL, 512)
    ow, rw = _both(orc, ref, w)
    W, H = 640, 360
    lods = cv.setup_lods(w.max_dimension, W, H)
    poses = cv.benchmark_path(w.dims, 60, far_clip=2.0 * w.max_dimension)
    for i in range(0, 60, 5):
        s = cv.frame_setup(poses[i], W, H, lods, w.dims[1])
        _same_raybuffers(orc, ref, ow, rw, s, W, H, i)


def test_world_file_interop_with_the_reference(cv, orc, ref, tmp_path):
    """f1: a .world written by the reference's own WorldSaveFile.Serialize (from worlds its own builder made of datasets/mill.obj)
    is read by the library's reader with every blob intact, the library's writer produces the same file byte for byte, and the
    reference's Deserialize of the library-written file renders the same raybuffers."""
    P, Cc = parse_obj(MILL)
    ref_file, our_file = tmp_path / "mill_ref.world", tmp_path / "mill_ours.world"
    dims, blobs, ccs, vox = ref.build_world_from_mesh(P, Cc, np.arange(P.shape[0]), 128, save_to=ref_file)
    w = cv.World.load(str(ref_file))
    assert tuple(w.dims) == tuple(dims) and len(w.blobs) == 6
    for j in range(6):
        assert np.asarray(w.blobs[j]).tobytes() == blobs[j].tobytes(), j
        assert w.column_counts[j] == ccs[j]
    cv.World.from_obj(MILL, 128).save(str(our_file))
    assert open(ref_file, "rb").read() == open(our_file, "rb").read()
    rw = ref.load_world_file(our_file)
    assert rw.dims == tuple(dims) and rw.world_count == 6
    ow = orc.OracleWorld(w.dims, w.blobs, w.column_counts)
    W, H = 320, 180
    for spec in POSES[:5]:
        s = setup_for(cv, w, spec, W, H)
        td, lr, _ = orc.render_raybuffers(ow, orc.copy_setup(s), W, H, threads=2)
        rtd, rlr = ref.render_raybuffers(rw, ref.copy_setup(s), W, H, threads=2)
        assert (td == rtd).all() and (lr == rlr).all(), spec[0]


def test_degenerate_triangle_quirk_of_the_reference(cv, ref):
    """A zero-area triangle makes VoxelizerHelper.GetVoxelsInternal return before it sets writtenVoxelCount (VoxelizerHelper.cs:45-47),
    so WorldBuilder.Import (WordBuilder.cs:71-74) submits the PREVIOUS triangle's voxels of the same worker task once more — which
    changes colour averages and depends on Environment.ProcessorCount (the task partition). The library skips such triangles
    (= the reference whenever a degenerate triangle opens a task, and for meshes without any, like datasets/mill.obj). This test
    pins the understanding: the reference (one task) on a soup with a degenerate triangle == the library on the same soup with that
    triangle replaced by a copy of its predecessor."""
    rng = np.random.default_rng(77)
    n = 300
    base = rng.uniform(0, 10, (n, 1, 3))
    P = (base + rng.normal(0, 0.8, (n, 3, 3))).astype(np.float32).reshape(-1, 3)
    C = rng.integers(0, 256, (n * 3, 4), dtype=np.uint8)
    C[:, 3] = 255
    P[30:33] = P[30]                      # triangle 10 has zero area
    dims, blobs, ccs, vox = ref.build_world_from_mesh(P, C, np.arange(n * 3), 64, flips=(False, False, False))
    skipped = cv.World.from_mesh(P, C, 64)
    assert any(np.asarray(a).tobytes() != b.tobytes() for a, b in zip(skipped.blobs, blobs)), "the quirk changes colours"
    P2, C2 = P.copy(), C.copy()
    P2[30:33], C2[30:33] = P[27:30], C[27:30]   # the predecessor, submitted twice
    # same bounds => same rescale: the degenerate triangle's vertex lies inside its predecessor's neighbourhood only if it does not
    # extend the mesh bounds; build both and compare when the dimensions agree
    dup = cv.World.from_mesh(P2, C2, 64)
    if tuple(dup.dims) == tuple(dims) and np.array_equal(P.min(0), P2.min(0)) and np.array_equal(P.max(0), P2.max(0)):
        for j in range(6):
            assert np.asarray(dup.blobs[j]).tobytes() == blobs[j].tobytes(), j
