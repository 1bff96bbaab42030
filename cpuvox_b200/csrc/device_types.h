/*
 * device_types.h — plain structs shared by the C-ABI layer (capi.cu) and the kernels (raybuffer_kernels.cu).
 * Everything here is passed to kernels by value (__grid_constant__), so a frame needs no host->device copy
 * besides the launch parameters themselves.
 */
#pragma once
#include <stdint.h>

#define CVXD_LODS 6
#define CVXD_MAX_AXIS 8192          /* longest raybuffer row (max(W,H)) the seen-mask in shared memory supports */
/* Phase 1 runs one warp (one ray at the default group width) per CTA: a CTA of several warps lives as long as its slowest ray and
 * keeps the other warps' slots idle; with 96 registers or fewer per thread 21+ such CTAs are resident per SM (profiles/r01e). */
#ifndef CVXD_THREADS_PER_CTA
#define CVXD_THREADS_PER_CTA 32
#endif
#define CVXD_TIMING_REGIONS 16

/* Device copy of one World LOD (Assets/Code/World.cs:8-43,161-188), transcoded on the host at upload (world_transcode.h):
 *   headers   one 16-byte aligned uint4 per column, fetched by a lane with a single 128-bit load:
 *               x = element offset (in 4-byte cells, relative to `elements`)
 *               y = runCount | worldMin << 16
 *               z = worldMax
 *               w = offset of the column's first boundary record in `bounds`
 *   elements  the reference element area verbatim: [guard][runs...][guard][ColorARGB32...] per column
 *   bounds    runCount + 1 records {world-Y of the boundary above run i, RLEElement i} per non-empty column, top to bottom
 *             (valid when cvxd_world.regular; see world_transcode.h) */
struct cvxd_lod {
    const uint4* headers;
    const uint32_t* elements;
    const uint2* bounds;
    int32_t mul_x;      /* dimZ >> lod, World.cs:31 */
    int32_t lod;
};

struct cvxd_world {
    cvxd_lod lods[CVXD_LODS];
    int32_t dim_x, dim_y, dim_z;
    int32_t lod_count;
    int32_t regular;    /* every uploaded LOD consists of full-height columns of valid runs: `bounds` may be used */
    /* derived on the host so that the kernels read them as constant-bank operands instead of holding them in registers */
    float dim_y_f;      /* (float)dim_y = worldMaxY (DrawSegmentRayJob.cs:213) */
    float inv_dim_y;    /* 1 / dim_y, exact when dim_y is a power of two */
    int32_t y_pow2;     /* dim_y is a power of two: unlerp(0, worldMaxY, y) == y * inv_dim_y exactly */
};

static inline void cvxd_world_set_dims(cvxd_world* w, int dx, int dy, int dz) {
    w->dim_x = dx; w->dim_y = dy; w->dim_z = dz;
    w->dim_y_f = (float)dy; w->inv_dim_y = 1.0f / (float)dy; w->y_pow2 = (dy & (dy - 1)) == 0 ? 1 : 0;
}

/* DrawSegmentRayJob.SegmentContext (Assets/Code/Rendering/DrawSegmentRayJob.cs:718-727) minus the pointers. */
struct cvxd_segment {
    float ray_min[2], ray_max[2];   /* CamLocalPlaneRayMin/Max */
    float min_screen[2], max_screen[2];
    int32_t ray_count;
    int32_t axis_mapped_to_y;
    int32_t ray_index_offset;
    int32_t pix_min, pix_max;       /* originalNextFreePixelMin/Max */
    int32_t buffer;                 /* 0 = top/down, 1 = left/right */
};

struct cvxd_counters {
    unsigned long long dda_steps, columns_nonempty, runs_visited, px_voxel, px_sky, rays;
};

struct cvxd_frame {
    float wts[16];                  /* CameraData.WorldToScreenMatrix, column-major */
    float pos_x, pos_z, pos_y;
    int32_t inverse;                /* InverseElementIterationDirection */
    float far_clip;
    float cam_y_norm;               /* PositionY / worldMaxY (DrawSegmentRayJob.cs:214), set with cvxd_frame_set_world */
    float lod_dist[CVXD_LODS];
    cvxd_segment seg[4];
    float vp_x, vp_y;
    int32_t width, height;
    int32_t total_rays;
    int32_t ray_begin, ray_end;     /* flat ray indices drawn by this launch (RaySetupJob order) */
    int32_t il_chunk, il_ranks, il_rank; /* il_chunk > 0: rays are dealt in chunks of il_chunk (chunk c -> rank c mod il_ranks) and this
                                     launch draws rank il_rank's; ray_begin / ray_end then count the rank's LOCAL rays [0, n) */
    uint32_t* td;                   /* top/down raybuffer: rows of `height` pixels */
    uint32_t* lr;                   /* left/right raybuffer: rows of `width` pixels */
    cvxd_counters* counters;        /* may be null */
    long long* timing;              /* debug: CVXD_TIMING_REGIONS cycle counts per flat ray, or null */
    int32_t general_path;           /* debug/test: force the general (element-area) kernel even for a regular world */
};

struct cvxd_blit {
    cvxd_segment seg[4];
    float vp_x, vp_y;
    int32_t width, height;
    int32_t row_begin, row_end;     /* screen rows written */
    int32_t ray_begin, ray_end;     /* only pixels sourced from these flat rays are written when `owned_only` */
    int32_t owned_only;
    int32_t il_chunk, il_ranks, il_rank; /* il_chunk > 0: ownership is "chunk (flat / il_chunk) belongs to rank il_rank" instead of the range */
    const uint32_t* td;
    const uint32_t* lr;
    uint32_t* frame;
    /* per-segment constants of the row formula (RenderManager.cs:235-242), filled by cvxd_blit_prepare on the host: _RayScale, _RayOffset
     * (two IEEE divisions a tile would otherwise repeat), the first raybuffer row of the segment and the flat index of its first ray */
    float seg_scale[4], seg_offset[4];
    int32_t seg_off01[4], seg_flat_base[4];
};

static inline void cvxd_blit_prepare(cvxd_blit* b) {
    int flat = 0;
    for (int k = 0; k < 4; k++) {
        const int rows = k < 2 ? b->width + 2 * b->height : 2 * b->width + b->height;
        const float rowsF = (float)rows;
        const int off01 = k == 1 ? b->seg[0].ray_count : (k == 3 ? b->seg[2].ray_count : 0);
        b->seg_scale[k] = (float)b->seg[k].ray_count / rowsF;
        b->seg_off01[k] = off01;
        b->seg_offset[k] = (k == 1 || k == 3) ? (float)off01 / rowsF : 0.0f;
        b->seg_flat_base[k] = flat;
        flat += b->seg[k].ray_count > 0 ? b->seg[k].ray_count : 0;
    }
}

/* The reference indexes worldLODs / LODDistances unchecked (DrawSegmentRayJob.cs:123-128,237-243): a ray that passes LODDistances[lod]
 * moves on to LOD lod + 1 whether or not it exists. Here the last uploaded LOD of the contiguous run from LOD 0 is never left: its
 * distance and the ones after it are +inf (identical to the reference whenever the reference is well defined, i.e. every LOD a ray
 * can reach exists and LODDistances[5] lies beyond the far clip, as SetupLods makes it). */
static inline void cvxd_frame_set_world(cvxd_frame* f, const cvxd_world* w) {
    f->cam_y_norm = f->pos_y / w->dim_y_f;
    int last = 0;
    while (last + 1 < CVXD_LODS && w->lods[last + 1].headers) last++;
    for (int i = last; i < CVXD_LODS; i++) f->lod_dist[i] = __builtin_inff();
}

struct cvxd_ray_state { /* mirrors cvx_ray_state */
    int32_t segment, plane_ray_index, status, lod;
    int32_t position[2], step[2];
    float start[2], dir[2], t_delta[2], t_max[2], intersection_distances[2];
};

#ifdef __CUDACC__
cudaError_t cvxd_launch_phase1(const cvxd_world& world, const cvxd_frame& frame, int group_size, cudaStream_t stream);
cudaError_t cvxd_launch_phase2(const cvxd_blit& blit, cudaStream_t stream);
cudaError_t cvxd_launch_ray_setup(const cvxd_world& world, const cvxd_frame& frame, cvxd_ray_state* out, int n, cudaStream_t stream);
cudaError_t cvxd_launch_fill(uint32_t* dst, uint32_t value, int64_t n, cudaStream_t stream);
cudaError_t cvxd_launch_raybuffer_view(const uint32_t* buf, int rows, int row_len, uint32_t* frame, int width, int height, cudaStream_t stream);
cudaError_t cvxd_launch_present(const uint32_t* frame, uint32_t* out, int width, int height, int bgra, int top_down, cudaStream_t stream);
cudaError_t cvxd_launch_present_rgb8(const uint32_t* frame, uint8_t* out, int width, int height, int top_down, cudaStream_t stream);
#endif
