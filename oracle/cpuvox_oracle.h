/*
 * cpuvox_oracle.h — TEST INFRASTRUCTURE ONLY. C ABI of the CPU oracle: a restatement of the
 * reference's raybuffer renderer (pipliz/cpuvox) in plain C++ with IEEE fp32, no FMA contraction.
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this library. The product (libcpuvox_b200.so, cpuvox_b200/) never links or calls it.
 *
 * PARITY UNPINNED: the reference ships no tests, golden vectors or fixtures for this path
 * (SURVEY.md §4, §8(c)) and cannot be compiled here (C# on UnityEngine/Burst; no dotnet/mono in
 * the image). This oracle follows the reference source line by line (citations in the .cpp);
 * it is a port, not the shipping Burst FloatMode.Fast binary.
 *
 * Struct layouts deliberately equal include/cpuvox_b200.h so a test can feed one side's frame
 * setup to the other; the two implementations share no code.
 */
#ifndef CPUVOX_ORACLE_H
#define CPUVOX_ORACLE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define ORC_LOD_LEVELS 6

typedef struct orc_segment {
    float min_screen[2];
    float max_screen[2];
    float cam_local_plane_ray_min[2];
    float cam_local_plane_ray_max[2];
    int32_t ray_count;
} orc_segment;

typedef struct orc_camera {
    float world_to_screen[16]; /* column-major */
    float position_xz[2];
    float position_y;
    int32_t inverse_element_iteration_direction;
    float far_clip;
    float lod_distances[ORC_LOD_LEVELS];
} orc_camera;

typedef struct orc_frame_setup {
    orc_segment segments[4];
    orc_camera camera;
    float vanishing_point_screen[2];
} orc_frame_setup;

typedef struct orc_counters {
    uint64_t dda_steps;
    uint64_t columns_nonempty;
    uint64_t runs_visited;
    uint64_t px_voxel;
    uint64_t px_sky;
    uint64_t rays;
} orc_counters;

typedef struct orc_pose {
    float position[3];
    float rotation[4];
    float fov_y_degrees;
    float near_clip;
    float far_clip;
    int32_t pixel_width;
    int32_t pixel_height;
} orc_pose;

typedef struct orc_ray_state {
    int32_t segment;
    int32_t plane_ray_index;
    int32_t status;
    int32_t lod;
    int32_t position[2];
    int32_t step[2];
    float start[2];
    float dir[2];
    float t_delta[2];
    float t_max[2];
    float intersection_distances[2];
} orc_ray_state;

typedef struct orc_world orc_world;

/* World LODs in the reference blob layout (World.cs:285-293): borrowed pointers, must outlive the world. */
orc_world* orc_world_create(int32_t dim_x, int32_t dim_y, int32_t dim_z);
int orc_world_set_lod(orc_world* w, int32_t lod, const void* blob, int64_t bytes, int32_t column_count);
void orc_world_free(orc_world* w);
/* math.min / math.max of the renderer, elementwise (test hook for the NaN and signed-zero rule) */
void orc_min_max(const float* a, const float* b, int32_t n, float* out_min, float* out_max);

void orc_quat_euler(float x_deg, float y_deg, float z_deg, float out_quat[4]);
void orc_limit_rotation_horizon(orc_pose* pose);
void orc_setup_lods(int32_t world_max_dimension, int32_t res_x, int32_t res_y, float fov_y_degrees,
                    float lod_error, float out[ORC_LOD_LEVELS]);
int orc_frame_setup_from_pose(const orc_pose* pose, const float lod_distances[ORC_LOD_LEVELS],
                              int32_t world_dim_y, orc_frame_setup* out);
void orc_benchmark_pose(float clip_time, const int32_t world_dims[3], orc_pose* inout_pose);

/* Phase 1: all four jobs of DrawSegmentRayJob.cs for flat ray indices [ray_begin, ray_end)
 * (ray_end < 0: all). td/lr are flat raybuffers: H x (W+2H) and W x (2W+H) ColorARGB32 pixels.
 * n_threads <= 0: all hardware threads. counters may be NULL. */
int orc_render_raybuffers(const orc_world* w, const orc_frame_setup* setup, int32_t width, int32_t height,
                          uint32_t* td, uint32_t* lr, int32_t ray_begin, int32_t ray_end,
                          int32_t n_threads, orc_counters* counters);
/* Phase 2: RayBufferBlit.shader default variant, restated per pixel. frame: W*H, row 0 = bottom. */
int orc_blit(const orc_frame_setup* setup, int32_t width, int32_t height, const uint32_t* td,
             const uint32_t* lr, uint32_t* frame, int32_t row_begin, int32_t row_end, int32_t n_threads);
/* Debug views COPY_MAIN1 / COPY_MAIN2 of the blit shader (RayBufferBlit.shader:48-53): raybuffer `buf` (rows x row_len) stretched over the screen. */
int orc_blit_raybuffer(const uint32_t* buf, int32_t rows, int32_t row_len, int32_t width, int32_t height, uint32_t* frame);
/* Per-ray state after the three setup jobs (DrawSegmentRayJob.cs:12-144). */
int orc_ray_setup(const orc_world* w, const orc_frame_setup* setup, int32_t width, int32_t height,
                  orc_ray_state* out, int32_t max_rays);
/* Test hook: DDA cell sequence of one ray (3 ints per step: x, z, lod; 2 floats per step: last, next distance). */
int orc_dda_walk(const float start[2], const float dir[2], const float lod_distances[ORC_LOD_LEVELS], float far_clip,
                 int32_t max_steps, int32_t* out_cells, float* out_dists);
/* Diagnostics: per-ray work counts (see the .cpp), ORC_RAY_STAT_FIELDS uint64 per ray. */
#define ORC_RAY_STAT_FIELDS 10
int orc_ray_stats(const orc_world* w, const orc_frame_setup* setup, int32_t width, int32_t height,
                  uint64_t* out, int32_t max_rays);
int orc_hardware_threads(void);

#ifdef __cplusplus
}
#endif
#endif
