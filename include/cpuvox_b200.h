/*
 * cpuvox_b200.h — C ABI of libcpuvox_b200.so, the B200-native raybuffer renderer.
 *
 * This is the drop-in boundary for the one hot path of pipliz/cpuvox: the body of
 * RenderManager.DrawSegments (Assets/Code/RenderManager.cs:258-372), the raybuffer
 * upload/copy (Assets/Code/Rendering/RayBuffer.cs:79-96) and BlitSegments +
 * RayBufferBlit.shader (RenderManager.cs:199-256, Assets/Shaders/RayBufferBlit.shader:47-64).
 * The reference has no FFI seam (Phase 1 runs as in-process Burst jobs); each entry point below
 * cites the reference interface it replaces. A C# host binds these with
 * [DllImport("cpuvox_b200")] — see INTEGRATION.md.
 *
 * Plain C99: fixed-width integers, no bool, no STL, no torch types. Every function returns
 * CVX_OK (0) or a negative cvx_status; nothing throws or exits across the boundary.
 * The library has no CPU fallback: without a CUDA device cvx_create fails with CVX_ERR_NO_DEVICE.
 */
#ifndef CPUVOX_B200_H
#define CPUVOX_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CVX_LOD_LEVELS 6 /* UnityManager.LOD_LEVELS, Assets/Code/UnityManager.cs:42 */

typedef enum cvx_status {
    CVX_OK = 0,
    CVX_ERR_INVALID_ARGUMENT = -1,
    CVX_ERR_NO_DEVICE = -2,
    CVX_ERR_CUDA = -3,
    CVX_ERR_OUT_OF_MEMORY = -4,
    CVX_ERR_NO_WORLD = -5,
    CVX_ERR_NO_RESOLUTION = -6,
    CVX_ERR_IO = -7,
    CVX_ERR_FORMAT = -8,
    CVX_ERR_UNSUPPORTED = -9
} cvx_status;

/* ---- blittable per-frame inputs -------------------------------------------------------- */

/* RenderManager.SegmentData, RenderManager.cs:503-510 (36 bytes, sequential layout). */
typedef struct cvx_segment {
    float min_screen[2];
    float max_screen[2];
    float cam_local_plane_ray_min[2];
    float cam_local_plane_ray_max[2];
    int32_t ray_count;
} cvx_segment;

/* CameraData, Assets/Code/Utils/CameraData.cs:11-36. The matrix is the float4x4
 * WorldToScreenMatrix stored column after column (c0.xyzw, c1.xyzw, c2.xyzw, c3.xyzw). */
typedef struct cvx_camera {
    float world_to_screen[16];
    float position_xz[2];
    float position_y;
    int32_t inverse_element_iteration_direction; /* camera.transform.forward.y >= 0 */
    float far_clip;
    float lod_distances[CVX_LOD_LEVELS];
} cvx_camera;

/* Everything RenderManager.DrawWorld hands to DrawSegments + BlitSegments for one frame
 * (RenderManager.cs:120-167,179-189). */
typedef struct cvx_frame_setup {
    cvx_segment segments[4];
    cvx_camera camera;
    float vanishing_point_screen[2];
} cvx_frame_setup;

/* Work-unit counters, identical for the CPU oracle and the GPU path (SURVEY.md §8(d)). */
typedef struct cvx_counters {
    uint64_t dda_steps;        /* loop iterations reaching World.GetVoxelColumn (DrawSegmentRayJob.cs:245) + NextLOD iterations of :123-128 */
    uint64_t columns_nonempty; /* of those, columns with runCount > 0 */
    uint64_t runs_visited;     /* valid RLEElements dereferenced at :444-447 ("voxel-runs") */
    uint64_t px_voxel;         /* raybuffer pixels written at :531 and :600 */
    uint64_t px_sky;           /* raybuffer pixels written at :705 and :714 */
    uint64_t rays;             /* rays set up (sum of RayCount, or the range drawn) */
} cvx_counters;

typedef struct cvx_config {
    int32_t device;            /* CUDA device ordinal */
    int32_t flags;             /* CVX_FLAG_* */
} cvx_config;

#define CVX_FLAG_COUNTERS 1    /* accumulate cvx_counters on the device (small cost) */

typedef struct cvx_ctx cvx_ctx;

/* ---- lifetime: new RenderManager() / Destroy(), RenderManager.cs:25-51 ------------------ */
int cvx_create(const cvx_config* config, cvx_ctx** out_ctx);
int cvx_destroy(cvx_ctx* ctx);
/* Error text of the last failing call on this context (or of cvx_create when ctx == NULL). */
const char* cvx_last_error(const cvx_ctx* ctx);

/* Optional: run on a caller-owned CUDA stream (cudaStream_t) instead of the context's own. NULL restores the
 * context's own stream; to use the legacy default stream pass cudaStreamLegacy. */
int cvx_set_stream(cvx_ctx* ctx, void* cuda_stream);

/* ---- world hand-off: World / WorldAllocator, Assets/Code/World.cs:8-43,261-313 ------------
 * blob = WorldAllocator.GetStartPointer()/GetByteLength(): column_count 12-byte RLEColumn
 * headers followed by 4-byte RLEElement / ColorARGB32 cells. The caller keeps its blob (host or device memory); the
 * library copies it to its own device allocation and builds its Phase-1 tables from it with a CUDA kernel. */
int cvx_world_upload(cvx_ctx* ctx, int32_t lod, int32_t dim_x, int32_t dim_y, int32_t dim_z,
                     const void* blob, int64_t bytes, int32_t column_count);
int cvx_world_free(cvx_ctx* ctx);

/* ---- RenderManager.SetResolution, RenderManager.cs:94-109 --------------------------------
 * (re)allocates the top/down raybuffer H x (W+2H), the left/right raybuffer W x (2W+H)
 * (RenderManager.cs:35-36) and the W x H framebuffer. */
int cvx_set_resolution(cvx_ctx* ctx, int32_t width, int32_t height);

/* ---- RenderManager.DrawSegments + ApplyPartials + BlitSegments ----------------------------
 * cvx_draw runs Phase 1 for every ray of the four segments and Phase 2 for the whole screen,
 * asynchronously on the context's stream. cvx_draw_rays runs Phase 1 only for the flat ray
 * indices [ray_begin, ray_end) in RaySetupJob order (DrawSegmentRayJob.cs:12-40) and Phase 2
 * only for screen rows [row_begin, row_end): the multi-GPU building blocks. */
int cvx_draw(cvx_ctx* ctx, const cvx_frame_setup* setup);
int cvx_draw_rays(cvx_ctx* ctx, const cvx_frame_setup* setup, int32_t ray_begin, int32_t ray_end);
int cvx_blit_rows(cvx_ctx* ctx, const cvx_frame_setup* setup, int32_t row_begin, int32_t row_end);
/* Multi-GPU Phase 2: write only the screen pixels whose source ray lies in [ray_begin, ray_end) into
 * device_frame (a W*H*4 device buffer, possibly a peer GPU's mapped framebuffer; NULL = own frame).
 * Ranks with disjoint ray ranges write disjoint pixels, so the gather is the store itself. */
int cvx_blit_owned(cvx_ctx* ctx, const cvx_frame_setup* setup, int32_t ray_begin, int32_t ray_end, void* device_frame);
/* Batched views over one world (SURVEY.md §8(e), config 5): n frames, up to CVX_OPT_FRAMES_IN_FLIGHT of them in flight at
 * once; frame i is read back (if dst_frames != NULL) to dst_frames + i*W*H*4 and the call returns when all frames are on the
 * host. With dst_frames == NULL the call only enqueues: the frames stay on the device, ordered before anything queued later on
 * the context's stream. Either way the read functions and device pointers refer to the LAST view afterwards.
 * With dst_frames the frames pass through a pool of up to 32 device framebuffers (allocated on first use, W*H*4 bytes each) that
 * a copy stream drains in view order, so rendering runs ahead of the device->host copies instead of waiting for them. */
int cvx_draw_batch(cvx_ctx* ctx, const cvx_frame_setup* setups, int32_t n_views, void* dst_frames);
/* Asynchronous form (dst_frames required, n_views >= 2): returns as soon as the batch is enqueued and hands out a batch number;
 * cvx_batch_wait(batch) returns when that batch's frames are in dst_frames (cvx_sync waits for everything). A further asynchronous
 * batch may be issued before the previous one has finished — into a different destination — and then renders while the previous
 * batch's frames are still being copied out: the way to stream batches without idling the GPU during the copy backlog at the end of
 * each one. Up to 4 batches may be outstanding. The views of consecutive batches use the same buffer sets in order. */
int cvx_draw_batch_async(cvx_ctx* ctx, const cvx_frame_setup* setups, int32_t n_views, void* dst_frames, int64_t* out_batch);
int cvx_batch_wait(cvx_ctx* ctx, int64_t batch);
int cvx_sync(cvx_ctx* ctx);

/* ---- outputs --------------------------------------------------------------------------------
 * Pixels are ColorARGB32 (bytes a,r,g,b; Assets/Code/Utils/Color24.cs:5-11). The frame is
 * W*H pixels, row 0 = bottom of the screen (Unity screen space, as RenderManager uses it).
 * Raybuffers are flat: row r (one ray) at r*row_len pixels — the RenderTexture contents after
 * RayBuffer.ApplyPartials (RayBuffer.cs:79-89). which: 0 = top/down, 1 = left/right. */
int cvx_read_frame(cvx_ctx* ctx, void* dst_argb, int64_t bytes);
int cvx_read_raybuffer(cvx_ctx* ctx, int32_t which, void* dst_argb, int64_t bytes);
int cvx_get_counters(cvx_ctx* ctx, cvx_counters* out, int32_t reset);
/* Debug: fill both raybuffers with one colour (RenderManager.ClearRayBuffer, RenderManager.cs:58-92 uses magenta). */
int cvx_clear_raybuffers(cvx_ctx* ctx, uint32_t argb);
/* Debug views, the shader's COPY_MAIN1 / COPY_MAIN2 variants (RayBufferBlit.shader:48-53; UnityManager.ERenderMode.RayBufferTopDown /
 * RayBufferLeftRight, UnityManager.cs:129-134,471-483): write the whole raybuffer `which` (0 = top/down, 1 = left/right) of the last
 * view into the framebuffer, stretched over the screen — screen x selects the ray row, screen y the pixel along the row, point
 * sampled. Use with cvx_clear_raybuffers(magenta) before the draw to see which pixels a frame wrote. */
int cvx_blit_raybuffer(cvx_ctx* ctx, int32_t which);
/* Presentation, the step after the path (replaces Unity's camera target, RenderManager.cs:192-193): convert the framebuffer
 * (ColorARGB32, row 0 = bottom) on the device to RGBA8 / BGRA8 (4 bytes per pixel) or packed RGB8 (3 bytes per pixel), rows
 * top-down (top_down != 0: what swap chains, image files and encoders take) or bottom-up, into `dst`: a device buffer of W*H*4
 * (W*H*3 for RGB8) bytes (dst_is_device != 0; e.g. a mapped graphics-interop resource or an encoder surface; ordered on the
 * context's stream) or host memory (the call returns when the copy has landed). */
#define CVX_PRESENT_RGBA8 0
#define CVX_PRESENT_BGRA8 1
#define CVX_PRESENT_RGB8 2
int cvx_present(cvx_ctx* ctx, int32_t format, int32_t top_down, void* dst, int32_t dst_is_device);
/* Presentation as a compressed still: the framebuffer is packed to top-down RGB8 and encoded as a baseline JPEG ON THE DEVICE
 * (nvJPEG's CUDA encoder, a CUDA toolkit library loaded with dlopen at the first call; CVX_ERR_UNSUPPORTED when it is not installed —
 * nothing else in the library depends on it). Only the bitstream crosses to the host: *out_bytes receives its length, and it is
 * copied to `dst` if dst_capacity holds it. dst_capacity == 0 queries the length (the frame is encoded, nothing is copied).
 * quality 1..100; subsampling CVX_JPEG_444 (no chroma subsampling: hard voxel edges stay sharp) or CVX_JPEG_420. */
#define CVX_JPEG_444 0
#define CVX_JPEG_420 1
int cvx_present_jpeg(cvx_ctx* ctx, int32_t quality, int32_t subsampling, void* dst, int64_t dst_capacity, int64_t* out_bytes);
/* Page-locked host memory for asynchronous frame readback (cvx_draw_batch, cvx_read_frame). */
int cvx_alloc_pinned(int64_t bytes, void** out);
int cvx_free_pinned(void* p);
/* Device pointers for interop (display, NCCL gather): valid until the next cvx_set_resolution. */
int cvx_device_frame(cvx_ctx* ctx, void** out_device_ptr, int64_t* out_bytes);
int cvx_device_raybuffer(cvx_ctx* ctx, int32_t which, void** out_device_ptr, int64_t* out_bytes);
/* Render into a caller-owned device framebuffer (W*H*4 bytes) instead of the internal one;
 * NULL restores the internal buffer. */
int cvx_set_external_frame(cvx_ctx* ctx, void* device_ptr);
/* Timing of the last cvx_draw on the device, in milliseconds (CUDA events on the stream). */
int cvx_last_draw_ms(cvx_ctx* ctx, float* out_phase1_ms, float* out_phase2_ms);
/* Number of kernel launches issued by this context since creation. */
int64_t cvx_launch_count(const cvx_ctx* ctx);

/* Tuning / measurement knobs (no reference analogue).
 *   CVX_OPT_GROUP_SIZE  lanes cooperating on one ray in Phase 1: 0 = choose per frame from the ray count, or 8, 16, 32.
 *   CVX_OPT_COUNTERS    1 = accumulate cvx_counters (same as CVX_FLAG_COUNTERS at creation), 0 = off.
 *   CVX_OPT_GENERAL_PATH 1 = always run the general Phase-1 kernel (reads the reference element area run by run); 0 (default) =
 *                       use the boundary-table kernel whenever the uploaded world is regular (see cvx_world_is_regular).
 *   CVX_OPT_FRAMES_IN_FLIGHT 1..16 (default 6): views of one cvx_draw_batch rendered concurrently, each on its own stream with its
 *                       own raybuffers and framebuffer (the reference double-buffers its raybuffers for the same reason,
 *                       RenderManager.cs:14,53-56). Extra buffer sets are allocated on the first batch that needs them. */
#define CVX_OPT_GROUP_SIZE 1
#define CVX_OPT_COUNTERS 2
#define CVX_OPT_GENERAL_PATH 3
#define CVX_OPT_FRAMES_IN_FLIGHT 4
int cvx_set_option(cvx_ctx* ctx, int32_t option, int32_t value);
/* 1 when every uploaded LOD consists of full-height columns of valid runs (what WorldBuilder.ToFinalColumn emits,
 * WordBuilder.cs:232-256): Phase 1 then runs its boundary-table kernel. 0 = the general kernel is used. < 0 = error. */
int cvx_world_is_regular(const cvx_ctx* ctx);
/* Device-side timing of many draws: after cvx_profile_begin every cvx_draw / cvx_draw_batch view records CUDA
 * events around Phase 1 and Phase 2 on the context's stream (up to max_draws views); cvx_profile_end waits for
 * them and returns the summed kernel durations in milliseconds and the number of views timed. */
int cvx_profile_begin(cvx_ctx* ctx, int32_t max_draws);
int cvx_profile_end(cvx_ctx* ctx, double* out_phase1_ms, double* out_phase2_ms, int32_t* out_draws);

/* ---- multi-GPU, one process per GPU (SURVEY.md §8(e)) -------------------------------------------
 * The root rank exports its internal framebuffer as a CUDA IPC handle; every other rank opens it and passes the mapped
 * pointer to cvx_blit_owned, so Phase 2 stores each rank's pixels straight into the root's framebuffer over NVLink —
 * the gather is the kernel's own stores, no staging copy and no collective on the data path. */
#define CVX_IPC_HANDLE_BYTES 64
int cvx_ipc_export_frame(cvx_ctx* ctx, uint8_t out_handle[CVX_IPC_HANDLE_BYTES]);
int cvx_ipc_open(cvx_ctx* ctx, const uint8_t handle[CVX_IPC_HANDLE_BYTES], void** out_device_ptr);
int cvx_ipc_close(cvx_ctx* ctx, void* device_ptr);

/* Frame ring: the pipelined form of the same gather, for a stream of ray-sharded views. The root allocates `slots` framebuffers
 * plus flag words in ONE device allocation and exports it; every other rank maps it. For view v every rank calls cvx_draw_sharded
 * with its flat-ray range: Phase 1 for those rays, Phase 2 for the pixels they feed, stored into ring frame v % slots on the root
 * (NVLink peer stores), then a flag store. All ordering between ranks is on the device — a rank waits for "slot released" before
 * it stores, the root's consumer waits for "all ranks arrived" — so no host barrier and no collective sits between two views
 * (the reference's analogue of the unit of work is RenderManager.cs:358-363: one frame's rays as one parallel job).
 * A wait gives up after 4 s and raises the ring's error flag (cvx_ring_status) instead of hanging the GPU. Set the resolution
 * before creating / opening a ring; cvx_set_resolution and cvx_destroy close it (close the mappings before the root frees). */
int cvx_ring_create(cvx_ctx* ctx, int32_t slots, int32_t world_size, uint8_t out_handle[CVX_IPC_HANDLE_BYTES]);
int cvx_ring_open(cvx_ctx* ctx, const uint8_t handle[CVX_IPC_HANDLE_BYTES], int32_t slots, int32_t world_size);
int cvx_ring_close(cvx_ctx* ctx);
/* ray_begin >= 0: this rank draws the flat rays [ray_begin, ray_end). ray_begin == CVX_SHARD_INTERLEAVED: the rays are dealt to the
 * ranks in chunks of `ray_end` rays (a power of two; chunk c to rank c mod world_size) and this rank draws its chunks — heavy rays come in runs of
 * neighbours, so this balances the ranks without a cost estimate. */
#define CVX_SHARD_INTERLEAVED (-1)
int cvx_draw_sharded(cvx_ctx* ctx, const cvx_frame_setup* setup, int32_t ray_begin, int32_t ray_end, int64_t view_index, int32_t rank);
/* Root: wait for view_index from all ranks, copy it to dst_host (optional, pinned), release the slot; asynchronous (cvx_sync). */
int cvx_ring_consume(cvx_ctx* ctx, int64_t view_index, void* dst_host, void** out_device_frame);
int cvx_ring_status(cvx_ctx* ctx);

/* ---- ray queries against the resident world (no reference analogue: SURVEY.md lists no ray query in the reference) -----------
 * Picking, hit-scan, line of sight and depth probes: what does a ray hit first? The query runs at one uploaded LOD j (cells of
 * 2^j world units); the ray starts at `origin` (world units), `direction` need not be normalised, and `distance` is measured along
 * the normalised direction in world units, up to `max_distance` (+inf allowed). The exact definition, which the device kernel
 * follows bit for bit in IEEE fp32, is DESIGN.md §3.5.
 *   hit       1 = hit, 0 = miss, -1 = invalid ray (zero-length direction, or a NaN / infinite input other than max_distance = +inf)
 *   face      outward normal of the face the ray entered the hit cell through: 0 -X, 1 +X, 2 -Y, 3 +Y, 4 -Z, 5 +Z;
 *             6 = the origin lies inside the solid cell (distance 0)
 *   cell      the hit cell in LOD-j cells; color its ColorARGB32; steps = cells the definition tests (also on a miss)
 * A miss or an invalid ray has every field but `steps` zero. */
typedef struct cvx_ray {
    float origin[3];
    float max_distance;
    float direction[3];
    int32_t reserved;
} cvx_ray; /* 32 bytes */
typedef struct cvx_ray_hit {
    int32_t hit;
    int32_t face;
    int32_t cell[3];
    float distance;
    uint32_t color;
    int32_t steps;
} cvx_ray_hit; /* 32 bytes */
/* on_device == 0: rays / out are host arrays; the call returns when the hits are in `out` (device scratch grows to the largest n
 * and is freed by cvx_world_free / cvx_destroy). on_device != 0: device pointers; the query is ordered on the context's stream
 * after whatever is queued there and the call returns at once. Either way it reads the world uploaded at the time of the call.
 * CVX_ERR_NO_WORLD without a world; CVX_ERR_INVALID_ARGUMENT for a LOD that is not uploaded, n < 0, or NULL arrays with n > 0;
 * n == 0 does nothing. CVX_OPT_GENERAL_PATH 1 makes it read runs from the element area (same results). */
int cvx_raycast(cvx_ctx* ctx, const cvx_ray* rays, int32_t n, int32_t lod, cvx_ray_hit* out, int32_t on_device);

/* Debug: dump the per-ray state after RaySetupJob/DDASetupJob/TraceToFirstColumnJob
 * (DrawSegmentRayJob.cs:12-144) for every flat ray index; 18 x 4 bytes per ray, see cvx_ray_state. */
typedef struct cvx_ray_state {
    int32_t segment;
    int32_t plane_ray_index;
    int32_t status;          /* 0 = continues into RenderJob, 1 = skybox-filled in TraceToFirstColumn */
    int32_t lod;
    int32_t position[2];
    int32_t step[2];
    float start[2];
    float dir[2];
    float t_delta[2];
    float t_max[2];
    float intersection_distances[2];
} cvx_ray_state;
int cvx_debug_ray_setup(cvx_ctx* ctx, const cvx_frame_setup* setup, cvx_ray_state* out, int32_t max_rays);
/* Debug: run Phase 1 once with per-ray cycle counters; CVX_TIMING_REGIONS int64 per flat ray index:
 * 0 setup/other, 1 DDA look-ahead + header fetch, 2 column selection (frustum cull), 3 frustum re-narrowing,
 * 4 run fetch + bounds, 5 span geometry, 6 column resolve + commit-loop control, 7 skybox fill, 8 commit re-test (span_would_write),
 * 9 ReducePixelHorizon, 10 cap pixels, 11 side-span perspective setup, 12 side pixels, 13 written-mask update, 14-15 unused.
 * Returns the frame's ray count. */
#define CVX_TIMING_REGIONS 16
int cvx_debug_ray_timing(cvx_ctx* ctx, const cvx_frame_setup* setup, int64_t* out_cycles, int32_t max_rays);

/* =============================================================================================
 * Host-side helpers (pure CPU, no device): C++ restatement of the managed code around the path,
 * for hosts that have no UnityEngine (tests, bench, headless servers). A Unity host keeps using
 * RenderManager's own code for these and only calls the device entry points above.
 * ============================================================================================= */

/* UnityEngine.Camera + Transform state that RenderManager.DrawWorld reads. */
typedef struct cvx_pose {
    float position[3];
    float rotation[4];     /* quaternion x,y,z,w */
    float fov_y_degrees;   /* SampleScene.unity:178 = 85 */
    float near_clip;       /* SampleScene.unity:176 = 0.05 */
    float far_clip;        /* UnityManager.SetupLods: 2 * world max dimension */
    int32_t pixel_width;
    int32_t pixel_height;
} cvx_pose;

/* Quaternion.Euler(x,y,z) (Z-X-Y order), degrees. */
void cvx_host_quat_euler(float x_deg, float y_deg, float z_deg, float out_quat[4]);
/* UnityManager.LimitRotationHorizon, UnityManager.cs:193-201. */
void cvx_host_limit_rotation_horizon(cvx_pose* pose);
/* UnityManager.SetupLods, UnityManager.cs:417-458 (window size == render resolution). */
void cvx_host_setup_lods(int32_t world_max_dimension, int32_t res_x, int32_t res_y,
                         float fov_y_degrees, float lod_error, float out_lod_distances[CVX_LOD_LEVELS]);
/* RenderManager.DrawWorld up to the DrawSegments call: vanishing point (RenderManager.cs:374-394),
 * GetGenericSegmentParameters x4 (:402-501), CameraData ctor (CameraData.cs:18-36). */
int cvx_host_frame_setup(const cvx_pose* pose, const float lod_distances[CVX_LOD_LEVELS],
                         int32_t world_dim_y, cvx_frame_setup* out);
/* Camera.ScreenPointToRay for pixel (px, py) in Unity screen space (bottom-left origin, the framebuffer's rows) of a camera of
 * pose->pixel_width x pose->pixel_height: the origin on the near plane, the direction normalised (feed it to cvx_raycast). */
void cvx_host_screen_ray(const cvx_pose* pose, float px, float py, float out_origin[3], float out_direction[3]);
/* RenderManager.DrawWorld for a batch of cameras on a host without UnityEngine (RenderManager.cs:111-194; with limit_rotation_horizon != 0
 * also UnityManager.LimitRotationHorizon, UnityManager.cs:181): the library computes each view's frame setup from its pose at the
 * context's resolution (pixel_width / pixel_height of the poses are ignored) and renders the views like cvx_draw_batch. */
int cvx_draw_world_batch(cvx_ctx* ctx, const cvx_pose* poses, int32_t n_views, const float lod_distances[CVX_LOD_LEVELS],
                         int32_t limit_rotation_horizon, void* dst_frames);
/* The same through cvx_draw_batch_async: returns once enqueued, cvx_batch_wait(*out_batch) for the frames. */
int cvx_draw_world_batch_async(cvx_ctx* ctx, const cvx_pose* poses, int32_t n_views, const float lod_distances[CVX_LOD_LEVELS],
                               int32_t limit_rotation_horizon, void* dst_frames, int64_t* out_batch);
/* BenchmarkPath.anim sampled at clip time t in [0, 1.15] (UnityManager.cs:86-87): position is
 * the normalised curve value times the world dimensions; rotation from the Euler curves. */
void cvx_host_benchmark_pose(float clip_time, const int32_t world_dims[3], cvx_pose* inout_pose);
float cvx_host_benchmark_length(void);

/* ---- world production (host, offline): ObjModel/SimpleMesh/VoxelizerHelper/WorldBuilder/
 * World.DownSample restated (Assets/Code/Utils/ObjModel.cs, SimpleMesh.cs:64-106,
 * VoxelizerHelper.cs:28-132, WordBuilder.cs:39-268, World.cs:45-127). */
typedef struct cvx_world_builder cvx_world_builder;
/* vertices: n_vertices x {x,y,z} float + n_vertices x {r,g,b,a} bytes (Color32); triangles are
 * consecutive vertex triples (the .obj importer emits non-indexed meshes). flips: 1 = flip axis. */
int cvx_builder_from_mesh(const float* positions, const uint8_t* colors32, int32_t n_vertices,
                          int32_t max_dimension, const int32_t flips[3], int32_t n_threads,
                          cvx_world_builder** out);
/* The same world production on the device (SURVEY.md §8(f) 2): triangles are voxelized, merged per (column, y), run-length encoded and
 * downsampled into n_lods LODs by CUDA kernels on the context's GPU; the builder then holds blobs identical, byte for byte, to what
 * cvx_builder_from_mesh + cvx_builder_lod produce (read them with cvx_builder_lod, release with cvx_builder_free). A triangle that
 * covers more than 262144 voxels (VOXELIZE_BUFFER_MAX, WordBuilder.cs:37: the reference truncates it in scan order) is refused with
 * CVX_ERR_INVALID_ARGUMENT — use the host builder for such meshes. */
int cvx_gpu_builder_from_mesh(cvx_ctx* ctx, const float* positions, const uint8_t* colors32, int32_t n_vertices,
                              int32_t max_dimension, const int32_t flips[3], int32_t n_lods, cvx_world_builder** out);
/* Mesh -> resident world entirely on the device: builds the LODs like cvx_gpu_builder_from_mesh and installs them as the context's
 * world (replacing any uploaded one) without copying the blobs to the host. out_dims / out_voxel_counts (optional) receive the world
 * dimensions and the per-LOD voxel counts the reference logs (UnityManager.cs:326-331). */
int cvx_world_build_from_mesh(cvx_ctx* ctx, const float* positions, const uint8_t* colors32, int32_t n_vertices,
                              int32_t max_dimension, const int32_t flips[3], int32_t n_lods, int32_t out_dims[3],
                              int64_t out_voxel_counts[CVX_LOD_LEVELS]);
/* Parse a text .obj (v with optional rgb, f with v, v/vt, v/vt/vn or v//vn) into the arrays above. */
int cvx_obj_parse(const char* path, int32_t swap_yz, float** out_positions, uint8_t** out_colors32,
                  int32_t* out_n_vertices);
void cvx_host_free(void* p);
/* Synthetic worlds of BASELINE.json configs 2-5 (SURVEY.md §8(d)); kind 0 = fBm heightmap shell,
 * kind 1 = structured boxes/pipes/slabs. */
int cvx_builder_synthetic(int32_t kind, int32_t dim_x, int32_t dim_y, int32_t dim_z, uint32_t seed,
                          int32_t n_threads, cvx_world_builder** out);
int cvx_builder_dims(const cvx_world_builder* b, int32_t out_dims[3]);
/* Build LOD `lod` (0 = ToLOD0World, j>0 = World.DownSample(j) of LOD 0); the blob stays owned by
 * the builder. voxel_count = the count the reference logs per LOD (UnityManager.cs:326-331). */
int cvx_builder_lod(cvx_world_builder* b, int32_t lod, const void** out_blob, int64_t* out_bytes,
                    int32_t* out_column_count, int64_t* out_voxel_count);
void cvx_builder_free(cvx_world_builder* b);

/* ---- .world files, Assets/Code/WorldSaveFile.cs:8-103 ---------------------------------------- */
int cvx_world_file_write(const char* path, const int32_t dims[3], int32_t world_count,
                         const void* const* blobs, const int64_t* blob_bytes);
/* Reads header + table; blobs are malloc'ed (free each with cvx_host_free). */
int cvx_world_file_read(const char* path, int32_t out_dims[3], int32_t* out_world_count,
                        void** out_blobs /* [CVX_LOD_LEVELS] */, int64_t* out_blob_bytes /* [CVX_LOD_LEVELS] */);

/* Write a ColorARGB32 frame (as returned by cvx_read_frame: row 0 = bottom) as an uncompressed 32-bit .bmp (bottom-up BGRA,
 * so rows are stored in the order they arrive). Host only. */
int cvx_host_write_bmp(const char* path, const void* argb_frame, int32_t width, int32_t height);

#ifdef __cplusplus
}
#endif
#endif /* CPUVOX_B200_H */
