/*
 * raybuffer_kernels.cu — sm_100a kernels of the raybuffer renderer.
 *
 *   phase1_kernel   one WARP per raybuffer row (ray). Replaces RaySetupJob, DDASetupJob, TraceToFirstColumnJob and
 *                   RenderJob/ExecuteRay (Assets/Code/Rendering/DrawSegmentRayJob.cs:12-620) in a single launch.
 *   phase2_kernel   one CTA per 64 x 32 screen tile; replaces BlitSegments + RayBufferBlit.shader
 *                   (Assets/Code/RenderManager.cs:199-256, Assets/Shaders/RayBufferBlit.shader:47-64).
 *
 * Phase 1 design (not a translation of the per-thread C# loop; DESIGN.md §3.1 has the long form):
 *  - The DDA cell sequence of a ray (including the LOD switches, SegmentDDAData.cs:31-73,135-150) does not depend on
 *    world data, so the warp walks it 32 cells ahead: every lane keeps the (uniform) DDA state, lane i captures cell i,
 *    then all 32 column headers are fetched with one 128-bit load per lane. A ballot picks the non-empty columns; only
 *    those enter the order-dependent part.
 *  - Boundary-table kernel (FAST, regular worlds): a ROUND caches the run boundaries of several consecutive columns, one
 *    boundary per lane; each boundary is projected once on the last and once on the next line, the side span of a run is the
 *    pair of its two boundaries' projections, its cap span the last/next pair of one boundary. None of that depends on the
 *    written-pixel state. Per round, ballots record which lanes' spans still hold an unwritten pixel (hot lanes); cached
 *    columns without one are skipped, and the commit loop of an entered column walks its hot lanes in reference order.
 *    The general kernel (!FAST, any world) keeps one run per lane with a segmented prefix sum for the world-Y extents.
 *  - The per-row written-pixel set is a bitmask in shared memory (one word per 32 pixels). Pixels are written lane-parallel
 *    over a span, the mask words of the span are OR-ed by one lane per word, and the "skip already written pixels" scans of
 *    ReducePixelHorizon (:660-697) are bit scans.
 *  - Numerics: IEEE fp32, no FMA contraction (-fmad=false), IEEE division/sqrt, denormals kept (float.Epsilon sentinel
 *    of :220-221 must survive), same operation order as the reference expressions, so rows match the reference's own code
 *    (compiled for the CPU) bit for bit.
 */
#ifdef CVX_EMU /* test-only CPU build of this source under tools/simt_emu (never part of the product library) */
#include "cuda_emu.h"
#else
#include <cuda_runtime.h>
#endif
#include <limits.h>
#include <stdint.h>
#include "device_types.h"

#define FULL_MASK 0xffffffffu
#if defined(CVX_EMU) && defined(CVX_EMU_STATS) /* emulator-only event counts per ray (tools/simt_emu), lane 0 of the group counts */
#define EMU_STAT(i) do { if (gl == 0) emu_stats[(int64_t)flat * 16 + (i)]++; } while (0)
#define EMU_STAT_ADD(i, v) do { if (gl == 0) emu_stats[(int64_t)flat * 16 + (i)] += (unsigned long long)(v); } while (0)
extern unsigned long long* emu_stats;
#else
#define EMU_STAT(i) do { } while (0)
#define EMU_STAT_ADD(i, v) do { } while (0)
#endif
#define SKYBOX_ARGB 0x191919FFu /* ColorARGB32(25,25,25): bytes a=255,r,g,b (DrawSegmentRayJob.cs:702) */

namespace {

struct F3 { float x, y, z; }; // (screen-axis coordinate, z', w) as kept by SetupProjectedPlaneParams (:642-650)

__device__ __forceinline__ float lerpf(float a, float b, float t) { return a + t * (b - a); }
__device__ __forceinline__ float unlerpf(float a, float b, float x) { return (x - a) / (b - a); }
__device__ __forceinline__ F3 lerp3(F3 a, F3 b, float t) { return F3{lerpf(a.x, b.x, t), lerpf(a.y, b.y, t), lerpf(a.z, b.z, t)}; }
__device__ __forceinline__ float signf(float x) { return (float)((x > 0.0f ? 1 : 0) - (x < 0.0f ? 1 : 0)); }
// math.min / math.max as the reference build pins them (Unity.Mathematics): a NaN second operand gives the first, a tie (±0) the second
__device__ __forceinline__ float minf_(float a, float b) { return (b != b || a < b) ? a : b; }
__device__ __forceinline__ float maxf_(float a, float b) { return (b != b || a > b) ? a : b; }
// (int)float as x64 cvttss2si: NaN / out of range -> INT_MIN
__device__ __forceinline__ int f2i(float f) { const int r = __float2int_rz(f); return f < 2147483648.0f ? r : (int)0x80000000; } // cvt saturates low; NaN/high -> INT_MIN
__device__ __forceinline__ float float_epsilon() { return __int_as_float(1); }

// ---- SegmentDDAData (Assets/Code/Utils/SegmentDDAData.cs) -------------------------------------------------
struct Dda {
    int px, pz, sx, sz;
    float start_x, start_z, dir_x, dir_z, tdx, tdz, tmx, tmz, dl, dn; // dl/dn = IntersectionDistances (last, next)
};

__device__ __forceinline__ void dda_init(Dda& d, float sx, float sz, float dx, float dz) { // :17-28
    d.start_x = sx; d.start_z = sz; d.dir_x = dx; d.dir_z = dz;
    float fx = floorf(sx), fz = floorf(sz);
    d.px = f2i(fx); d.pz = f2i(fz);
    d.tdx = 1.0f / maxf_(0.0000001f, fabsf(dx));
    d.tdz = 1.0f / maxf_(0.0000001f, fabsf(dz));
    float gx = signf(dx), gz = signf(dz);
    d.sx = f2i(gx); d.sz = f2i(gz);
    d.tmx = (gx * -(sx - fx) + (gx * 0.5f) + 0.5f) * d.tdx;
    d.tmz = (gz * -(sz - fz) + (gz * 0.5f) + 0.5f) * d.tdz;
    d.dl = maxf_(d.tmx - d.tdx, d.tmz - d.tdz);
    d.dn = minf_(d.tmx, d.tmz);
}

__device__ __forceinline__ void dda_next_lod(Dda& d, int voxelSize) { // :31-73
    const float ninf = __int_as_float(0xff800000), pinf = __int_as_float(0x7f800000);
    int rx = d.px & (voxelSize * 2 - 1), rz = d.pz & (voxelSize * 2 - 1);
    // a still axis entered from outside has tMax = +inf (dda_step_to_world): its last crossing stays -inf, tMax - tDelta would be +inf
    float prevx = d.tmx != pinf ? d.tmx - d.tdx : ninf, prevz = d.tmz != pinf ? d.tmz - d.tdz : ninf;
    if ((d.dir_x >= 0.0f) == (rx < voxelSize)) d.tmx += d.tdx; else prevx -= d.tdx;
    if ((d.dir_z >= 0.0f) == (rz < voxelSize)) d.tmz += d.tdz; else prevz -= d.tdz;
    d.dl = maxf_(prevx, prevz);
    d.dn = minf_(d.tmx, d.tmz);
    d.px -= rx; d.pz -= rz;
    d.tdx *= 2.0f; d.tdz *= 2.0f;
    d.sx *= 2; d.sz *= 2;
}

__device__ bool dda_step_to_world(Dda& d, float dimX, float dimZ) { // StepToWorldIntersection :75-130
    const float ninf = __int_as_float(0xff800000), pinf = __int_as_float(0x7f800000);
    float ix = 1.0f / d.dir_x, iz = 1.0f / d.dir_z;
    float tminx = ninf, tminz = ninf, tmaxx = pinf, tmaxz = pinf;
    if (d.dir_x != 0.0f) {
        float t1 = -d.start_x * ix, t2 = (dimX - d.start_x) * ix;
        tminx = minf_(t1, t2); tmaxx = maxf_(t1, t2);
    }
    if (d.dir_z != 0.0f) {
        float t1 = -d.start_z * iz, t2 = (dimZ - d.start_z) * iz;
        tminz = minf_(t1, t2); tmaxz = maxf_(t1, t2);
    }
    float tmint = maxf_(tminx, tminz), tmaxt = minf_(tmaxx, tmaxz);
    if (tmaxt < tmint || tmint <= 0.0f) return false;
    float lastx, lastz;
    if (tminx < tminz && tminx != ninf) {
        lastz = tminz;
        float off = tmint * d.dir_x;
        float hit = d.start_x + off;
        hit = d.dir_x > 0.0f ? floorf(hit) : ceilf(hit);
        off = hit - d.start_x;
        lastx = off / d.dir_x;
    } else if (d.dir_z != 0.0f) {
        lastx = tminx;
        float off = tmint * d.dir_z;
        float hit = d.start_z + off;
        hit = d.dir_z > 0.0f ? floorf(hit) : ceilf(hit);
        off = hit - d.start_z;
        lastz = off / d.dir_z;
    } else {
        lastx = tminx; lastz = ninf;
    }
    // Still-axis rule (DESIGN.md §5): an axis with dir == 0 never bounds the entry and is never crossed, tLast = -inf and tMax = +inf.
    // The reference divides by the zero component here (a NaN or +inf last distance for a still z, tMax = -inf for a still x).
    d.tmx = d.dir_x != 0.0f ? lastx + d.tdx : pinf;
    d.tmz = d.dir_z != 0.0f ? lastz + d.tdz : pinf;
    d.dl = maxf_(lastx, lastz);
    d.dn = minf_(d.tmx, d.tmz);
    float mid = lerpf(d.dl, d.dn, 0.5f);
    d.px = f2i(floorf(d.start_x + mid * d.dir_x));
    d.pz = f2i(floorf(d.start_z + mid * d.dir_z));
    return true;
}

// ---- CameraData clip helpers (Assets/Code/Utils/CameraData.cs:50-157) --------------------------------------
__device__ __forceinline__ float cross2(float ax, float ay, float bx, float by) { return ax * by - ay * bx; }
// GetWorldBoundsClippingCamSpace (:50-99) is evaluated lane-parallel inside the frustum re-narrowing of phase1_kernel: four lanes, one
// (line, end) pair each; ClipMin (:101-107) = 1 - c0 / (c0 - c1), ClipMax (:109-115) = c1 / (c1 - c0) with
// c0 = cross((1, 1/frustum), pMax.xz), c1 = cross((1, 1/frustum), pMin.xz).
__device__ __forceinline__ bool clip_near(F3& a, F3& b) { // :123-137, near plane z' <= 0 (F3.y)
    if (a.y <= 0.0f) {
        if (b.y <= 0.0f) return false;
        float v = b.y / (b.y - a.y);
        a = lerp3(b, a, v);
    } else if (b.y <= 0.0f) {
        float v = a.y / (a.y - b.y);
        b = lerp3(a, b, v);
    }
    return true;
}
__device__ __forceinline__ bool clip_near_u(F3& a, F3& b, float& uA, float& uB) { // :140-157
    if (a.y <= 0.0f) {
        if (b.y <= 0.0f) return false;
        float v = b.y / (b.y - a.y);
        a = lerp3(b, a, v);
        uA = lerpf(uB, uA, v);
    } else if (b.y <= 0.0f) {
        float v = a.y / (a.y - b.y);
        b = lerp3(a, b, v);
        uB = lerpf(uA, uB, v);
    }
    return true;
}

// mul(WorldToScreenMatrix, (x,y,z,w)) with the float4x4 column order, summed left to right
__device__ __forceinline__ void project(const float* m, float x, float y, float z, float w, float out[4]) {
#pragma unroll
    for (int r = 0; r < 4; r++) out[r] = m[r] * x + m[4 + r] * y + m[8 + r] * z + m[12 + r] * w;
}

// ---- per-ray setup: RaySetupJob :12-40, DDASetupJob :49-77, TraceToFirstColumnJob :87-144 -----------------
struct RaySetup {
    int segment, plane_index, lod, status; // status 0 = continue into ExecuteRay, 1 = skybox the whole row, -1 = no such ray
    int lod_steps;                         // NextLOD iterations of :123-128 (counted as dda_steps)
    Dda dda;
};

__device__ void setup_ray(const cvxd_world& world, const cvxd_frame& f, int flatIndex, RaySetup& rs) {
    int planeIndex = flatIndex, seg = -1;
#pragma unroll
    for (int j = 0; j < 4; j++) {
        int n = f.seg[j].ray_count;
        if (seg >= 0 || n <= 0) continue;
        if (planeIndex >= n) { planeIndex -= n; continue; }
        seg = j;
    }
    rs.segment = seg; rs.plane_index = planeIndex; rs.lod = 0; rs.lod_steps = 0; rs.status = -1;
    if (seg < 0) return;
    const cvxd_segment& sg = f.seg[seg];
    float t = planeIndex / (float)sg.ray_count;
    float dx = lerpf(sg.ray_min[0], sg.ray_max[0], t), dz = lerpf(sg.ray_min[1], sg.ray_max[1], t);
    float inv = 1.0f / sqrtf(dx * dx + dz * dz); // normalize(v) = v * rsqrt(dot(v,v)), rsqrt = 1/sqrt
    dda_init(rs.dda, f.pos_x, f.pos_z, dx * inv, dz * inv);
    rs.status = 0;
    if (rs.dda.px < 0 || rs.dda.pz < 0 || rs.dda.px >= world.dim_x || rs.dda.pz >= world.dim_z) {
        rs.status = 1;
        if (dda_step_to_world(rs.dda, (float)world.dim_x, (float)world.dim_z)) {
            // never past the last LOD of the contiguous run uploaded from LOD 0 (the reference indexes worldLODs unchecked)
            int lastLod = 0;
            while (lastLod + 1 < CVXD_LODS && world.lods[lastLod + 1].headers) lastLod++;
            float lodMax = f.lod_dist[0];
            while (rs.lod < lastLod && rs.dda.dl >= lodMax) {
                dda_next_lod(rs.dda, 1 << rs.lod);
                rs.lod++;
                rs.lod_steps++;
                lodMax = f.lod_dist[rs.lod];
            }
            if (!(minf_(rs.dda.tmx, rs.dda.tmz) >= f.far_clip)) rs.status = 0; // IsBeyondFarClip :152-155
        }
    }
}

// ---- written-pixel bitmask helpers -------------------------------------------------------------------------
// One bit per pixel of the row in shared memory (the README's "bitmask"; the reference keeps a byte per pixel, :208). A second
// level (one bit per fully written word) was measured slower once the screen-hull test was dropped: spans and horizon scans touch one
// or two words, and the extra bookkeeping (a shared atomic per completed word, ~350 SASS instructions) cost 5 % (profiles/r01e).
// bits [a & 31 .. 31] of the word holding a, and bits [0 .. b & 31] of the word holding b
__device__ __forceinline__ uint32_t mask_from(int a) { return FULL_MASK << (a & 31); }
__device__ __forceinline__ uint32_t mask_to(int b) { return FULL_MASK >> (31 - (b & 31)); }

// index of the first word in [wlo, whi] that is not fully written, or whi + 1
__device__ __forceinline__ int next_open_word(const uint32_t* seen, int wlo, int whi) {
    for (int w = wlo; w <= whi; w++) if (~seen[w]) return w;
    return whi + 1;
}
// index of the last word in [wlo, whi] that is not fully written, or wlo - 1
__device__ __forceinline__ int prev_open_word(const uint32_t* seen, int wlo, int whi) {
    for (int w = whi; w >= wlo; w--) if (~seen[w]) return w;
    return wlo - 1;
}
// first index >= start whose bit is clear, at most limit+1  ("while (i <= limit && seen[i]) i++")
__device__ __forceinline__ int scan_up(const uint32_t* seen, int start, int limit) {
    if (start > limit) return start;
    uint32_t x = ~seen[start >> 5] & mask_from(start);
    int w = start >> 5;
    if (!x) {
        w = next_open_word(seen, w + 1, limit >> 5);
        if (w > (limit >> 5)) return limit + 1;
        x = ~seen[w];
    }
    const int j = (w << 5) + __ffs(x) - 1;
    return j <= limit ? j : limit + 1;
}
// last index <= start whose bit is clear, at least limit-1  ("while (i >= limit && seen[i]) i--")
__device__ __forceinline__ int scan_down(const uint32_t* seen, int start, int limit) {
    if (start < limit) return start;
    uint32_t x = ~seen[start >> 5] & mask_to(start);
    int w = start >> 5;
    if (!x) {
        w = prev_open_word(seen, limit >> 5, w - 1);
        if (w < (limit >> 5)) return limit - 1;
        x = ~seen[w];
    }
    const int j = (w << 5) + 31 - __clz(x);
    return j >= limit ? j : limit - 1;
}
// any clear bit in [a, b] (a <= b, both inside the row)
__device__ __forceinline__ bool any_unseen(const uint32_t* seen, int a, int b) {
    const int wa = a >> 5, wb = b >> 5;
    if (wa == wb) return (~seen[wa] & mask_from(a) & mask_to(b)) != 0u;
    if ((~seen[wa] & mask_from(a)) | (~seen[wb] & mask_to(b))) return true;
    return wa + 1 < wb && next_open_word(seen, wa + 1, wb - 1) < wb;
}
// mark [a, b] written: lane `gl` of G handles every G-th word; returns how many of them were new (for the counters)
template <int G>
__device__ __forceinline__ int mark_seen(uint32_t* seen, int a, int b, int gl) {
    int fresh = 0;
    for (int w = (a >> 5) + gl; w <= (b >> 5); w += G) {
        uint32_t m = FULL_MASK;
        if (w == (a >> 5)) m &= mask_from(a);
        if (w == (b >> 5)) m &= mask_to(b);
        const uint32_t old = seen[w], now = old | m;
        fresh += __popc(~old & m);
        seen[w] = now;
    }
    return fresh;
}

struct RowState {
    uint32_t* seen;         // shared-memory bitmask of this row
    uint32_t* row;          // raybuffer row
    int orig_min, orig_max; // originalNextFreePixelMin/Max
    int nf_min, nf_max;     // nextFreePixelMin/Max
    float fb_min, fb_max;   // frustumBoundsMin/Max
};

// A span [bMin, bMax] changes anything (pixels, horizon, frustum) only if it holds a still-unwritten pixel of the
// writable range: nextFreePixelMin/Max are themselves unwritten pixels (the scans of :407-415,678-692 stop on one),
// so a span that reaches an end of the range (the only way ReducePixelHorizon :660-697 moves the horizon) always
// contains one. Everything else passes the overlap test of :505/:581, writes nothing and leaves all state untouched.
__device__ __forceinline__ bool span_would_write(const RowState& rw, int bMin, int bMax) {
    if (!(bMax >= rw.nf_min && bMin <= rw.nf_max)) return false;
    const int a = bMin > rw.nf_min ? bMin : rw.nf_min, b = bMax < rw.nf_max ? bMax : rw.nf_max;
    return a <= b && any_unseen(rw.seen, a, b);
}

// ReducePixelHorizon :660-697 (uniform across the group)
__device__ __forceinline__ void reduce_pixel_horizon(RowState& rw, int& bMin, int& bMax) {
    if (bMin <= rw.nf_min) {
        bMin = rw.nf_min;
        if (bMax >= rw.nf_min) {
            rw.nf_min = scan_up(rw.seen, bMax + 1, rw.orig_max);
            rw.fb_min = rw.nf_min - 0.501f;
        }
    }
    if (bMax >= rw.nf_max) {
        bMax = rw.nf_max;
        if (bMin <= rw.nf_max) {
            rw.nf_max = scan_down(rw.seen, bMin - 1, rw.orig_min);
            rw.fb_max = rw.nf_max + 0.501f;
        }
    }
}

struct Acc { unsigned long long dda_steps, columns_nonempty, runs_visited, px_voxel, px_sky; };

/*
 * phase1_kernel<G, COUNTERS>: one GROUP of G lanes (8, 16 or 32) per raybuffer row, 32/G rows per warp.
 * Neighbouring rows (adjacent rays of one segment) share a warp: they walk nearly the same columns, so the groups of
 * a warp stay mostly convergent while the number of rays in flight per SM grows by 32/G.
 */
#ifndef CVXD_MIN_CTAS_PER_SM /* with 32-thread CTAs: 21 -> ptxas settles on 80 registers (25 resident warps per SM); measured best */
#define CVXD_MIN_CTAS_PER_SM 21
#endif
#if CVXD_MIN_CTAS_PER_SM > 0
#define CVXD_P1_BOUNDS __launch_bounds__(CVXD_THREADS_PER_CTA, CVXD_MIN_CTAS_PER_SM)
#else /* variants built with -maxrregcount */
#define CVXD_P1_BOUNDS
#endif
template <int G, bool COUNTERS, bool TIMING, bool FAST, bool INV>
__global__ void CVXD_P1_BOUNDS
phase1_kernel(const __grid_constant__ cvxd_world world, const __grid_constant__ cvxd_frame f) {
#ifdef CVX_EMU
    uint32_t* seen_all = emu::g_shared;
#else
    extern __shared__ uint32_t seen_all[];
#endif
    constexpr int GROUPS_PER_CTA = CVXD_THREADS_PER_CTA / G;
    constexpr uint32_t GBITS = G == 32 ? FULL_MASK : ((1u << (G & 31)) - 1u);
    const int lane = threadIdx.x & 31;
    const int gl = lane & (G - 1);          // lane inside the group
    const int gshift = lane & ~(G - 1);     // first lane of the group inside the warp
    const uint32_t gmask = GBITS << gshift;
    const int group = threadIdx.x / G;
    int flat = f.ray_begin + blockIdx.x * GROUPS_PER_CTA + group;
    if (flat >= f.ray_end) return;
    if (f.il_chunk > 0) {  // interleaved sharding: local ray j of this rank is ray j % chunk of the rank's (j / chunk)-th chunk
        flat = ((flat / f.il_chunk) * f.il_ranks + f.il_rank) * f.il_chunk + (flat & (f.il_chunk - 1));
        if (flat >= f.total_rays) return;
    }
#define GBALLOT(p) ((__ballot_sync(gmask, (p)) >> gshift) & GBITS)
#define GSHFL(v, src) __shfl_sync(gmask, (v), (src), G)

    // TIMING builds (cvx_debug_ray_timing): cycles per code region of this ray, STAMP(r) closes the current region
    long long tAcc[CVXD_TIMING_REGIONS] = {0};
    long long tPrev = TIMING ? clock64() : 0;
    int tCur = 0;
#define STAMP(r) do { if (TIMING) { const long long t_ = clock64(); tAcc[tCur] += t_ - tPrev; tPrev = t_; tCur = (r); } } while (0)

    RaySetup rs;
    setup_ray(world, f, flat, rs);
    if (rs.status < 0) return;
    const cvxd_segment& sg = f.seg[rs.segment];
    const int rowLen = sg.buffer == 0 ? f.height : f.width;
    uint32_t* row = (sg.buffer == 0 ? f.td : f.lr) + (int64_t)(rs.plane_index + sg.ray_index_offset) * rowLen;
    const int seenWords = ((f.width > f.height ? f.width : f.height) + 31) >> 5;

    Acc acc = {0, 0, 0, 0, 0}; // per lane; summed with atomics at the end (COUNTERS only)
    if (COUNTERS && gl == 0) acc.dda_steps = (unsigned long long)rs.lod_steps;
    RowState rw;
    rw.seen = seen_all + group * (seenWords + 9 * G);
    int* scratch = (int*)(rw.seen + seenWords); // G ints: lane of a round -> batch cell of its column
    uint32_t* cache = (uint32_t*)(scratch + G); // 8 x G words: commit-only fields of the round cache
    rw.row = row;
    rw.orig_min = sg.pix_min; rw.orig_max = sg.pix_max;
    rw.nf_min = rw.orig_min; rw.nf_max = rw.orig_max;
    rw.fb_min = rw.nf_min - 0.501f; rw.fb_max = rw.nf_max + 0.501f;

    if (rs.status == 1) { // WriteSkyboxFull :710-716
        for (int y = rw.orig_min + gl; y <= rw.orig_max; y += G) row[y] = SKYBOX_ARGB;
        if (COUNTERS && gl == 0 && rw.orig_max >= rw.orig_min) acc.px_sky += rw.orig_max - rw.orig_min + 1;
    } else {
        for (int w = gl; w < seenWords; w += G) rw.seen[w] = 0u; // stackalloc, zero-initialised (:208)
        __syncwarp(gmask);

        Dda ray = rs.dda;
        int lod = rs.lod;
        int voxelScale = 1 << lod;
        const float farClip = f.far_clip;
        float lodMax = f.lod_dist[lod];
        #define worldMaxY (world.dim_y_f) /* a constant-bank operand, not a register */
        const float camY = f.pos_y;
        #define cameraPosYNormalized (f.cam_y_norm)
        constexpr int ITER = INV ? -1 : 1; // RenderJob.Execute :174-178 (INV = InverseElementIterationDirection, one kernel instance per direction)
        const float EPS = float_epsilon();
        float frustumDirMaxWorld = EPS, frustumDirMinWorld = EPS;

        // SetupProjectedPlaneParams :622-651
        F3 planeBottom, planeTop, planeDir;
        {
            float top[4], bot[4], dir[4];
            project(f.wts, ray.start_x, worldMaxY, ray.start_z, 1.0f, top);
            project(f.wts, ray.start_x, 0.0f, ray.start_z, 1.0f, bot);
            project(f.wts, ray.dir_x, 0.0f, ray.dir_z, 0.0f, dir);
            const int a = sg.axis_mapped_to_y ? 1 : 0;
            planeBottom = F3{bot[a], bot[2], bot[3]};
            planeTop = F3{top[a], top[2], top[3]};
            planeDir = F3{dir[a], dir[2], dir[3]};
        }
        const int maskX = world.dim_x - 1, maskZ = world.dim_z - 1;
        // unlerp(0, worldMaxY, y) = (y - 0) / (worldMaxY - 0): for a power-of-two height the quotient is exactly y * 2^-k

        bool terminated = false; // ray ended inside the loop: skybox the rest and stop
        bool reachedEnd = false; // far clip or world exit
        while (!terminated && !reachedEnd) {
            STAMP(1);
            EMU_STAT(0); // batches
            // ---- look ahead: the next G cells of the DDA at once, lane k of the group gets cell k -------------------------
            // Step() (SegmentDDAData.cs:135-150) crosses the x boundary when tMax.x < tMax.y, else the z boundary, and then adds
            // tDelta to that tMax: the crossing times are the merge of the two sequences X[a] = tMax.x + a additions of tDelta.x and
            // Z[b] likewise (ties go to z). The two chains are accumulated serially (same float additions as the reference), lane j
            // keeps X[j] and Z[j]; lane k then finds by a merge-path binary search how many of its first k steps were x steps —
            // a_k = the largest a with X[a-1] < Z[k-a] — which gives its cell, its last/next distances and its header address.
            // :237-243, tested once per visited cell: here for cell 0, for later cells by cutting the batch. This needs no LOD bound:
            // lod_dist of the last uploaded LOD is +inf (cvxd_frame_set_world), and dl is never +inf here, since every dl is a finite
            // crossing distance, a still axis contributes -inf (dda_step_to_world, dda_next_lod) and a NaN compares false.
            if (ray.dl >= lodMax) {
                dda_next_lod(ray, voxelScale);
                lod++; voxelScale *= 2;
                lodMax = f.lod_dist[lod];
            }
            float myX = ray.tmx, myZ = ray.tmz, xEnd, zEnd;
            {
                float x = ray.tmx, z = ray.tmz;
#pragma unroll
                for (int j = 1; j < G; j++) {
                    x += ray.tdx; z += ray.tdz;
                    if (gl == j) { myX = x; myZ = z; }
                }
                xEnd = x + ray.tdx; zEnd = z + ray.tdz; // X[G], Z[G]
            }
            int aK = 0;
            {
                int lo = 0, hi = gl;
#pragma unroll
                for (int it = 0; it < (G == 32 ? 5 : (G == 16 ? 4 : 3)); it++) {
                    const int mid = (lo + hi + 1) >> 1;
                    const float xv = GSHFL(myX, mid > 0 ? mid - 1 : 0), zv = GSHFL(myZ, gl - mid >= 0 ? gl - mid : 0);
                    if (lo < hi) { if (xv < zv) lo = mid; else hi = mid - 1; }
                }
                aK = lo;
            }
            const int bK = gl - aK;
            const float xa = GSHFL(myX, aK), zb = GSHFL(myZ, bK); // tMax of my cell
            const bool xStep = xa < zb;                          // which boundary Step() crosses leaving my cell
            const float myDn = xStep ? xa : zb;                  // crossed distance = next intersection of my cell
            float myDl = __shfl_up_sync(gmask, myDn, 1, G);      // the previous cell's crossing is my last intersection
            if (gl == 0) myDl = ray.dl;
            const int cellX = ray.px + aK * ray.sx, cellZ = ray.pz + bK * ray.sz;
            const bool oob = ((cellX & maskX) != cellX) || ((cellZ & maskZ) != cellZ);   // World.cs:135-138
            // first event in walk order: LOD switch before cell k (k >= 1), world exit at cell k, far clip after cell k (:613-615)
            const uint32_t swMask = GBALLOT(gl >= 1 && myDl >= lodMax), oobMask = GBALLOT(oob), farMask = GBALLOT(myDn >= farClip);
            const int kS = swMask ? __ffs(swMask) - 1 : G, kO = oobMask ? __ffs(oobMask) - 1 : G, kF = farMask ? __ffs(farMask) - 1 : G;
            int n, endKind = 0; // 1 = next cell is outside the world, 2 = far clip crossed after the last cell
            if (kS <= kO && kS <= kF) n = kS;                    // cut: the next batch starts with the LOD switch (or n == G: plain end of batch)
            else if (kO <= kF) { n = kO; endKind = 1; }
            else { n = kF + 1; endKind = 2; }
            const int myIdx = (cellX >> lod) * world.lods[lod].mul_x + (cellZ >> lod); // GetIndexKnownInBounds World.cs:145-149
            const int myLod = lod;                               // one LOD per batch
            if (endKind == 0 && n > 0) {                         // advance the ray to the cell after the batch
                const int aN = GSHFL(aK + (xStep ? 1 : 0), n - 1), bN = n - aN;
                const float tx = GSHFL(myX, aN < G ? aN : 0), tz = GSHFL(myZ, bN < G ? bN : 0);
                ray.tmx = aN < G ? tx : xEnd; ray.tmz = bN < G ? tz : zEnd;
                ray.px += aN * ray.sx; ray.pz += bN * ray.sz;
                ray.dl = GSHFL(myDn, n - 1);
                ray.dn = minf_(ray.tmx, ray.tmz);
            }
            uint4 hdr = make_uint4(0, 0, 0, 0);
            if (gl < n) hdr = __ldg(world.lods[myLod].headers + myIdx);
            const bool myNonEmpty = (hdr.y & 0xffffu) != 0u;
            const float myWorldMin = (float)(hdr.y >> 16), myWorldMax = (float)(hdr.z & 0xffffu);
            uint32_t remaining = GBALLOT(myNonEmpty);
            int cellsDone = n + (endKind == 1 ? 1 : 0); // the out-of-world probe counts as a step

            // Round cache: span geometry of several consecutive columns of this batch, one run per lane (see form_round below).
            uint32_t roundCols = 0u;      // batch cells whose runs are cached in the lanes
            uint32_t roundInvalid = 0u;   // lanes holding an invalid element (Length == 0), which ends its column (:445-447)
            int myBase = 0;               // batch lane c: first round lane of column c
            // per-lane cached run: element fields, world-Y bounds, side span and cap span (none of it depends on the written-pixel state)
            // (what only the commit of a span needs — colour indices, unrounded bounds, 1/w and u/w of both ends — is parked in
            // shared memory, cache[field * G + lane], and read back by the whole group at the committing lane's index)
            int r_ci = 0, r_sMin = 0, r_sMax = 0, r_cMin = 0, r_cMax = 0, r_capKind = 0;
            bool r_sideClip = false, r_capClip = false;
            float r_eMin = 0.0f, r_eMax = 0.0f;
            // FAST rounds: one BOUNDARY per lane (see world_transcode.h); the lane also owns the run between its boundary and the
            // next lane's. Kept for the commit: the run's length, its cap colour and the boundary's point on the last line.
            int r_len = 0; uint32_t r_capColor = 0u; float bFx = 0.0f, bFy = 0.0f, bFz = 0.0f;
            // Lanes of the round whose side / cap span held an unwritten pixel of the writable range when the round was formed. Written
            // pixels only grow and the writable range only shrinks, so these stay SUPERSETS of the spans that can still write: a
            // cached column none of whose lanes is set is inert (skipped like a culled one, see the hull comment below), and the
            // commit loop looks at the set lanes only.
            uint32_t roundHotS = 0u, roundHotC = 0u;
            bool r_solid = false;         // this lane holds a valid, non-air run
            const int myRunCount = (int)(hdr.y & 0xffffu);

            while (remaining) {
                STAMP(2);
                EMU_STAT(1); // select iterations
                // ---- next column that is not culled by the narrowed frustum (:261-281), found for all columns at once ----
                int c;
                float worldBoundsMin = 0.0f, worldBoundsMax = worldMaxY;
                if (frustumDirMaxWorld != EPS) {
                    const float distTop = frustumDirMaxWorld > 0.0f ? myDn : myDl;
                    const float distBot = frustumDirMinWorld < 0.0f ? myDn : myDl;
                    const float newMax = camY + frustumDirMaxWorld * distTop;
                    const float newMin = camY + frustumDirMinWorld * distBot;
                    const bool outOfWorld = newMin > worldMaxY || newMax < 0.0f;      // frustum left the world: ray ends
                    const bool culled = myWorldMin > newMax || myWorldMax < newMin;   // column outside the writable world bounds
                    // cannot write, hence no side effects: exactly known for a column in the round cache (product builds; counter builds
                    // enter every column the reference enters, to count its runs)
                    bool inert = false;
                    if (!COUNTERS && !culled && myNonEmpty && ((roundCols >> gl) & 1u))
                        inert = !((roundHotS | roundHotC) & ((myRunCount >= 32 ? FULL_MASK : ((1u << myRunCount) - 1u)) << myBase));
                    const uint32_t cand = GBALLOT(myNonEmpty && (outOfWorld || !(culled || inert))) & remaining;
                    if (!cand) {
                        if (COUNTERS && gl == 0) acc.columns_nonempty += __popc(remaining);
                        remaining = 0u;
                        break;
                    }
                    c = __ffs(cand) - 1;
                    const uint32_t upto = remaining & ((2u << c) - 1u);
                    if (COUNTERS && gl == 0) acc.columns_nonempty += __popc(upto);
                    remaining &= ~upto;
                    if (GSHFL((int)outOfWorld, c)) { terminated = true; cellsDone = c + 1; break; }
                    worldBoundsMin = GSHFL(newMin, c); worldBoundsMax = GSHFL(newMax, c);
                } else {
                    c = __ffs(remaining) - 1;
                    remaining &= remaining - 1;
                    if (COUNTERS && gl == 0) acc.columns_nonempty++;
                }
                const float distLast = GSHFL(myDl, c);
                const float distNext = GSHFL(myDn, c);
                const int cLod = GSHFL(myLod, c);
                const uint32_t hOff = GSHFL(hdr.x, c);
                const int runCount = GSHFL(myRunCount, c);
                const int cScale = 1 << cLod;

                if (distLast > 2.0f && frustumDirMaxWorld == EPS) { // re-narrow the frustum :295-422
                    STAMP(3);
                    EMU_STAT(2); // renarrows
                    // The four clip parameters (last/next line x min/max end) and their projections are independent:
                    // lane L&3 of the group computes one of them (same operations as CameraData.cs:50-121), then they are shared.
                    const int L = gl & 3;
                    const float dLine = (L & 2) ? distNext : distLast; // :289-293 for this lane's line
                    const F3 pMin = F3{planeBottom.x + planeDir.x * dLine, planeBottom.y + planeDir.y * dLine, planeBottom.z + planeDir.z * dLine};
                    const F3 pMax = F3{planeTop.x + planeDir.x * dLine, planeTop.y + planeDir.y * dLine, planeTop.z + planeDir.z * dLine};
                    const bool A = pMin.x > pMin.z * rw.fb_max, B = pMax.x > pMax.z * rw.fb_max;
                    const bool C = pMin.x < pMin.z * rw.fb_min, D = pMax.x < pMax.z * rw.fb_min;
                    const bool clipped = (A && B) || (!A && !B && C && D);
                    // ClipMin / ClipMax (CameraData.cs:101-115) against whichever frustum bound this lane's end crosses, if any
                    const bool isMax = L & 1;
                    const bool crossHi = isMax ? B : A, crossLo = isMax ? D : C;
                    float myLerp = isMax ? 1.0f : 0.0f;
                    if (crossHi || crossLo) {
                        const float fi = 1.0f / (crossHi ? rw.fb_max : rw.fb_min);
                        const float c0 = cross2(1.0f, fi, pMax.x, pMax.z), c1 = cross2(1.0f, fi, pMin.x, pMin.z);
                        const float num = isMax ? c1 : c0, den = isMax ? c1 - c0 : c0 - c1; // one division: c1/(c1-c0) or c0/(c0-c1)
                        const float q = num / den;
                        myLerp = isMax ? q : 1.0f - q;
                    }
                    const F3 pc = lerp3(pMin, pMax, myLerp);
                    const float myProj = pc.x / pc.z;
                    const float lastMinL = GSHFL(myLerp, 0), lastMaxL = GSHFL(myLerp, 1), nextMinL = GSHFL(myLerp, 2), nextMaxL = GSHFL(myLerp, 3);
                    float mnL = GSHFL(myProj, 0), mxL = GSHFL(myProj, 1), mnN = GSHFL(myProj, 2), mxN = GSHFL(myProj, 3);
                    const bool clippedLast = GSHFL((int)clipped, 0) != 0, clippedNext = GSHFL((int)clipped, 2) != 0;
                    float clippedMin, clippedMax, distForMin, distForMax; // which line's distance each frustum direction is taken at
                    if (clippedLast) {
                        if (clippedNext) { terminated = true; cellsDone = c + 1; break; }
                        worldBoundsMin = lerpf(0.0f, worldMaxY, nextMinL); distForMin = distNext;
                        worldBoundsMax = lerpf(0.0f, worldMaxY, nextMaxL); distForMax = distNext;
                        clippedMin = mnN; clippedMax = mxN;
                        if (clippedMax < clippedMin) { float t = clippedMin; clippedMin = clippedMax; clippedMax = t; }
                    } else if (clippedNext) {
                        worldBoundsMin = lerpf(0.0f, worldMaxY, lastMinL); distForMin = distLast;
                        worldBoundsMax = lerpf(0.0f, worldMaxY, lastMaxL); distForMax = distLast;
                        clippedMin = mnL; clippedMax = mxL;
                        if (clippedMax < clippedMin) { float t = clippedMin; clippedMin = clippedMax; clippedMax = t; }
                    } else {
                        const bool minFromLast = lastMinL < nextMinL, maxFromLast = lastMaxL > nextMaxL;
                        worldBoundsMin = lerpf(0.0f, worldMaxY, minFromLast ? lastMinL : nextMinL); distForMin = minFromLast ? distLast : distNext;
                        worldBoundsMax = lerpf(0.0f, worldMaxY, maxFromLast ? lastMaxL : nextMaxL); distForMax = maxFromLast ? distLast : distNext;
                        if (mxN < mnN) { float t = mxN; mxN = mnN; mnN = t; }
                        if (mxL < mnL) { float t = mxL; mxL = mnL; mnL = t; }
                        clippedMin = minf_(mnL, mnN);
                        clippedMax = maxf_(mxL, mxN);
                    }
                    frustumDirMaxWorld = (worldBoundsMax - camY) / distForMax; // :329-330,348-349,359-370
                    frustumDirMinWorld = (worldBoundsMin - camY) / distForMin;
                    worldBoundsMin = floorf(worldBoundsMin);
                    worldBoundsMax = ceilf(worldBoundsMax);
                    const int writableMin = f2i(floorf(clippedMin));
                    const int writableMax = f2i(ceilf(clippedMax));
                    if (writableMax < rw.nf_min || writableMin > rw.nf_max) { terminated = true; cellsDone = c + 1; break; }
                    if (writableMin > rw.nf_min) rw.nf_min = scan_up(rw.seen, writableMin, rw.orig_max);
                    if (writableMax < rw.nf_max) rw.nf_max = scan_down(rw.seen, writableMax, rw.orig_min);
                    if (rw.nf_min > rw.nf_max) { terminated = true; cellsDone = c + 1; break; }
                }

                const uint32_t* colColors = world.lods[cLod].elements + hOff + runCount + 2; // ColorPointer World.cs:185-188

                // ---- runs of this column (:424-611). A column of at most G runs is resolved from the round cache in one pass; a
                // taller one goes through the same code G runs at a time (k0 = first run of the pass, yDone = world-Y extent of the
                // runs before it, in LOD voxels times the LOD scale).
                const bool tall = FAST ? runCount >= G : runCount > G; // FAST: runCount + 1 boundaries must fit the G lanes
                int k0 = 0, yDone = 0;
                bool colStop = false;
                do {
                    STAMP(4);
                    EMU_STAT(3); // column passes
                    const int runsHere = tall ? (FAST ? (runCount - k0 < G - 1 ? runCount - k0 : G - 1) : (runCount - k0 < G ? runCount - k0 : G)) : runCount;
                    if (tall || !((roundCols >> c) & 1u)) {
                        // ---- form a round: this column (pass) plus, if it is not a tall one, the following columns that are likely
                        // to be entered, as long as their runs fit in the G lanes. One run per lane: fetch, world-Y bounds (segmented
                        // prefix sum), and the projected side/cap spans — the float-heavy part — once for all of them.
                        EMU_STAT(4); // rounds formed
                        const uint32_t follow = !tall ? remaining : 0u;
                        const uint32_t consider = (1u << c) | follow;
                        // lanes a column needs: one per run, or (FAST) one per boundary = runs + 1; a pass of a tall column takes G
                        // boundaries, the last of which opens the next pass
                        const int v = gl == c ? runsHere + (FAST ? 1 : 0) : (((consider >> gl) & 1u) ? myRunCount + (FAST ? 1 : 0) : 0);
                        int incl = v;
#pragma unroll
                        for (int o = 1; o < G; o <<= 1) { int t = __shfl_up_sync(gmask, incl, o, G); if (gl >= o) incl += t; }
                        const bool inRound = ((consider >> gl) & 1u) && incl <= G;
                        roundCols = GBALLOT(inRound);
                        myBase = incl - v;
                        if (inRound) scratch[myBase] = gl;           // first lane of each cached column -> its batch cell
                        const uint32_t startMask = __reduce_or_sync(gmask, inRound ? (1u << myBase) : 0u);
                        const int totalRuns = GSHFL(incl, 31 - __clz(roundCols));
                        EMU_STAT_ADD(9, totalRuns);            // lanes used by the rounds
                        EMU_STAT_ADD(10, __popc(roundCols));   // columns cached by the rounds
                        EMU_STAT_ADD(11, __popc(consider));    // columns that were candidates for the round
                        __syncwarp(gmask);
                        const int myStart = 31 - __clz(startMask & ((2u << gl) - 1u)); // lane 0 always starts a column
                        const bool hasRun = gl < totalRuns;
                        const int myCol = hasRun ? scratch[myStart] : c;
                        const int k = gl - myStart + (myCol == c ? k0 : 0);           // run index inside its column
                        __syncwarp(gmask);
                        const float cDl = GSHFL(myDl, myCol), cDn = GSHFL(myDn, myCol);
                        const uint32_t colOff = GSHFL(hdr.x, myCol);
                        const int colRuns = GSHFL(myRunCount, myCol);
                        const uint32_t* colElems = world.lods[cLod].elements + colOff; // one LOD per batch
                        if (FAST) {
                            // ---- one boundary per lane: record k of the column (from the top, or from the bottom when iterating
                            // upwards) = {world-Y of the boundary, RLEElement below it}. The run of lane i lies between the boundaries
                            // of lanes i and i + 1 (:449-455 without the running sums), and each boundary is projected ONCE on the
                            // last line (an end of two side spans, :478-502) and once on the next line (an end of one cap span, :554-578).
                            const uint32_t colB = GSHFL(hdr.w, myCol);
                            uint2 rec = make_uint2(0u, 0u);
                            if (hasRun) rec = __ldg(world.lods[cLod].bounds + colB + (ITER > 0 ? k : colRuns - k));
                            const int yB = (int)rec.x;
                            const int nextY = __shfl_down_sync(gmask, yB, 1, G);
                            const uint32_t nextEl = __shfl_down_sync(gmask, rec.y, 1, G);
                            const bool laneRun = hasRun && k < colRuns && gl + 1 < totalRuns; // a boundary lane followed by the run's other boundary
                            const uint32_t el = laneRun ? (ITER > 0 ? rec.y : nextEl) : 0x0000ffffu; // others: air of length 0, never solid
                            r_ci = (int)(short)(el & 0xffffu); r_len = (int)(short)(el >> 16);           // RLEElement World.cs:245-259
                            if (ITER > 0) { r_eMax = (float)yB; r_eMin = (float)nextY; } else { r_eMin = (float)yB; r_eMax = (float)nextY; }

                            STAMP(5);
                            const F3 lMinLast = F3{planeBottom.x + planeDir.x * cDl, planeBottom.y + planeDir.y * cDl, planeBottom.z + planeDir.z * cDl}; // :289-293
                            const F3 lMinNext = F3{planeBottom.x + planeDir.x * cDn, planeBottom.y + planeDir.y * cDn, planeBottom.z + planeDir.z * cDn};
                            const F3 lMaxLast = F3{planeTop.x + planeDir.x * cDl, planeTop.y + planeDir.y * cDl, planeTop.z + planeDir.z * cDl};
                            const F3 lMaxNext = F3{planeTop.x + planeDir.x * cDn, planeTop.y + planeDir.y * cDn, planeTop.z + planeDir.z * cDn};
                            const float portion = world.y_pow2 ? (float)yB * world.inv_dim_y : unlerpf(0.0f, worldMaxY, (float)yB); // :478-479
                            const F3 Fp = lerp3(lMinLast, lMaxLast, portion), Np = lerp3(lMinNext, lMaxNext, portion);
                            bFx = Fp.x; bFy = Fp.y; bFz = Fp.z;
                            const bool fFront = !(Fp.y <= 0.0f), nFront = !(Np.y <= 0.0f); // in front of the near plane (CameraData.cs:126,143)
                            // which run's cap ends on this boundary: the run below it when it is seen from above (:549), the run above it
                            // when seen from below (:556); a run takes the first of the two that applies
                            const int bKind = portion < cameraPosYNormalized ? 1 : (portion > cameraPosYNormalized ? 2 : 0);
                            const float fpx = Fp.x / Fp.z;
                            const int fr = f2i(rintf(fpx));
                            int bcMin = 0, bcMax = 0;
                            if (bKind && fFront && nFront) { // :571-578
                                const int nr = f2i(rintf(Np.x / Np.z));
                                bcMin = nr; bcMax = fr;
                                if (bcMin > bcMax) { bcMin = fr; bcMax = nr; }
                            }
                            const int flags = (fFront ? 1 : 0) | (nFront ? 2 : 0) | (bKind << 2);
                            const float nextFpx = __shfl_down_sync(gmask, fpx, 1, G);
                            const int nextFlags = __shfl_down_sync(gmask, flags, 1, G);
                            const int nextCMin = __shfl_down_sync(gmask, bcMin, 1, G), nextCMax = __shfl_down_sync(gmask, bcMax, 1, G);
                            const bool nextFront = nextFlags & 1;
                            const int topKind = ITER > 0 ? bKind : (nextFlags >> 2), botKind = ITER > 0 ? (nextFlags >> 2) : bKind;
                            r_capKind = topKind == 1 ? 1 : (botKind == 2 ? 2 : 0); // :549,556
                            const bool capOwn = (r_capKind == 1) == (ITER > 0);      // the cap's boundary is this lane's (else the next lane's)
                            const bool capNFront = capOwn ? nFront : ((nextFlags & 2) != 0);
                            r_sideClip = false; r_capClip = false;
                            const bool solidRun = laneRun && r_ci >= 0;
                            r_solid = solidRun;
                            bool needExact = false;
                            if (solidRun) {
                                if (fFront && nextFront) {
                                    // both ends in front of the near plane: ClipHomogeneousCameraSpaceLine changes nothing
                                    const float fb = ITER > 0 ? nextFpx : fpx, ft = ITER > 0 ? fpx : nextFpx; // bottom / top end
                                    const int nextFr = f2i(rintf(nextFpx));
                                    const int rb = ITER > 0 ? nextFr : fr, rt = ITER > 0 ? fr : nextFr;
                                    if (fb > ft) { r_sMin = rt; r_sMax = rb; } else { r_sMin = rb; r_sMax = rt; } // :496-502
                                    r_sideClip = true;
                                    if (r_capKind) {
                                        if (capNFront) { r_cMin = capOwn ? bcMin : nextCMin; r_cMax = capOwn ? bcMax : nextCMax; r_capClip = true; }
                                        else needExact = true;
                                    }
                                } else if (!fFront && !nextFront) {
                                    // both ends behind: no side span; the cap's last-line end is behind too, so the cap exists only if its
                                    // next-line end is in front (and then it is clipped)
                                    if (r_capKind && capNFront) needExact = true;
                                } else needExact = true;
                                if (r_capKind) r_capColor = __ldg(colElems + colRuns + 2 + (r_capKind == 1 ? r_ci : r_ci + r_len - 1)); // :553,560
                            }
                            if (GBALLOT(needExact)) {
                                EMU_STAT(8); // rounds with a run straddling the near plane
                                // ---- a run straddles the near plane: the reference's per-run clipping (rare; columns next to the camera)
                                const F3 nF = F3{__shfl_down_sync(gmask, Fp.x, 1, G), __shfl_down_sync(gmask, Fp.y, 1, G), __shfl_down_sync(gmask, Fp.z, 1, G)};
                                const F3 nN = F3{__shfl_down_sync(gmask, Np.x, 1, G), __shfl_down_sync(gmask, Np.y, 1, G), __shfl_down_sync(gmask, Np.z, 1, G)};
                                if (needExact) {
                                    F3 frontBottom = ITER > 0 ? nF : Fp, frontTop = ITER > 0 ? Fp : nF;
                                    float uA = (float)r_len, uB = 0.0f;
                                    r_sideClip = false; r_capClip = false;
                                    if (clip_near_u(frontBottom, frontTop, uA, uB)) { // :489-502 (clips frontBottom/Top in place)
                                        float bfx = frontBottom.x / frontBottom.z, bfy = frontTop.x / frontTop.z;
                                        if (bfx > bfy) { float t = bfx; bfx = bfy; bfy = t; }
                                        r_sMin = f2i(rintf(bfx)); r_sMax = f2i(rintf(bfy));
                                        r_sideClip = true;
                                    }
                                    if (r_capKind) { // :554-578
                                        F3 secA = capOwn ? Np : nN, secB = r_capKind == 1 ? frontTop : frontBottom;
                                        if (clip_near(secA, secB)) {
                                            r_cMin = f2i(rintf(secA.x / secA.z)); r_cMax = f2i(rintf(secB.x / secB.z));
                                            if (r_cMin > r_cMax) { int t = r_cMin; r_cMin = r_cMax; r_cMax = t; }
                                            r_capClip = true;
                                        }
                                    }
                                }
                            }
                        } else {
                            uint32_t el = 0u;
                            if (hasRun) el = __ldg(colElems + (ITER > 0 ? 1 + k : colRuns - k));
                            r_ci = (int)(short)(el & 0xffffu); r_len = (int)(short)(el >> 16); // RLEElement World.cs:245-259
                            roundInvalid = GBALLOT(hasRun && r_len == 0);  // an invalid element (Length == 0) ends its column (:445-447)
                            // lanes of my column from its start up to me, and whether an invalid element precedes me there
                            const uint32_t mineUpToMe = ((2u << gl) - 1u) & ~((1u << myStart) - 1u);
                            const bool valid = hasRun && !(roundInvalid & mineUpToMe);
                            r_solid = valid && r_ci >= 0;
                            const int span = valid ? r_len * cScale : 0;
                            int sum = span;
    #pragma unroll
                            for (int o = 1; o < G; o <<= 1) { int t = __shfl_up_sync(gmask, sum, o, G); if (gl >= o) sum += t; }
                            const int before = GSHFL(sum, myStart > 0 ? myStart - 1 : 0);
                            const int inclCol = sum - (myStart > 0 ? before : 0) + (myCol == c ? yDone : 0); // my column's runs up to and including me
                            if (tall) yDone = GSHFL(inclCol, runsHere - 1);                // extent after this pass (the round holds only this column)
                            if (ITER > 0) { r_eMax = (float)(world.dim_y - (inclCol - span)); r_eMin = (float)(world.dim_y - inclCol); } // :449-455
                            else          { r_eMin = (float)(inclCol - span); r_eMax = (float)inclCol; }

                            STAMP(5);
                            const F3 lMinLast = F3{planeBottom.x + planeDir.x * cDl, planeBottom.y + planeDir.y * cDl, planeBottom.z + planeDir.z * cDl}; // :289-293
                            const F3 lMinNext = F3{planeBottom.x + planeDir.x * cDn, planeBottom.y + planeDir.y * cDn, planeBottom.z + planeDir.z * cDn};
                            const F3 lMaxLast = F3{planeTop.x + planeDir.x * cDl, planeTop.y + planeDir.y * cDl, planeTop.z + planeDir.z * cDl};
                            const F3 lMaxNext = F3{planeTop.x + planeDir.x * cDn, planeTop.y + planeDir.y * cDn, planeTop.z + planeDir.z * cDn};
                            r_sideClip = false; r_capClip = false; r_capKind = 0;
                            {
                                float bfx = 0.0f, bfy = 0.0f, uvAx = 0.0f, uvAy = 0.0f, uvBx = 0.0f, uvBy = 0.0f;
                                int capIdx = 0;
                                const float portionBottom = unlerpf(0.0f, worldMaxY, r_eMin); // :478-481
                                const float portionTop = unlerpf(0.0f, worldMaxY, r_eMax);
                                F3 frontBottom = lerp3(lMinLast, lMaxLast, portionBottom);
                                F3 frontTop = lerp3(lMinLast, lMaxLast, portionTop);
                                // which cap, if any, depends on the camera height only (:549,556); its flat colour (:553,560) is fetched
                                // now, while the divisions below run, and parked in the cache
                                if (portionTop < cameraPosYNormalized) { r_capKind = 1; capIdx = r_ci; }
                                else if (portionBottom > cameraPosYNormalized) { r_capKind = 2; capIdx = r_ci + r_len - 1; }
                                uint32_t capColor = 0u;
                                if (r_capKind && valid && r_ci >= 0) capColor = __ldg(colElems + colRuns + 2 + capIdx);
                                float uA = (float)r_len, uB = 0.0f;
                                if (clip_near_u(frontBottom, frontTop, uA, uB)) { // :489-502 (clips frontBottom/Top in place)
                                    uvAx = 1.0f / frontBottom.z; uvAy = uA / frontBottom.z;
                                    uvBx = 1.0f / frontTop.z;    uvBy = uB / frontTop.z;
                                    bfx = frontBottom.x / frontBottom.z; bfy = frontTop.x / frontTop.z;
                                    if (bfx > bfy) {
                                        float t = bfx; bfx = bfy; bfy = t;
                                        t = uvAx; uvAx = uvBx; uvBx = t;
                                        t = uvAy; uvAy = uvBy; uvBy = t;
                                    }
                                    r_sMin = f2i(rintf(bfx)); r_sMax = f2i(rintf(bfy));
                                    r_sideClip = true;
                                }
                                if (r_capKind) { // :554-578
                                    const float portion = r_capKind == 1 ? portionTop : portionBottom;
                                    F3 secA = lerp3(lMinNext, lMaxNext, portion), secB = r_capKind == 1 ? frontTop : frontBottom;
                                    if (clip_near(secA, secB)) {
                                        r_cMin = f2i(rintf(secA.x / secA.z)); r_cMax = f2i(rintf(secB.x / secB.z));
                                        if (r_cMin > r_cMax) { int t = r_cMin; r_cMin = r_cMax; r_cMax = t; }
                                        r_capClip = true;
                                    }
                                }
                                cache[0 * G + gl] = __float_as_uint(bfx);  cache[1 * G + gl] = __float_as_uint(bfy);
                                cache[2 * G + gl] = __float_as_uint(uvAx); cache[3 * G + gl] = __float_as_uint(uvAy);
                                cache[4 * G + gl] = __float_as_uint(uvBx); cache[5 * G + gl] = __float_as_uint(uvBy);
                                cache[6 * G + gl] = (uint32_t)r_len;       cache[7 * G + gl] = capColor;
                                __syncwarp(gmask);
                            }
                        }
                        STAMP(6);
                        roundHotS = GBALLOT(r_solid && r_sideClip && span_would_write(rw, r_sMin, r_sMax));
                        roundHotC = GBALLOT(r_solid && r_capClip && span_would_write(rw, r_cMin, r_cMax));
                        STAMP(4);
                    }

                    // ---- resolve this column (pass) against the current frustum / written-pixel state (:441-611) -----------
                    const int base = GSHFL(myBase, c);
                    const uint32_t colMask = (runsHere >= 32 ? FULL_MASK : ((1u << runsHere) - 1u)) << base;
                    const bool inCol = (colMask >> gl) & 1u;
                    const uint32_t invalidHere = roundInvalid & colMask;
                    const int endValid = invalidHere ? __ffs(invalidHere) - 1 : base + runsHere; // first lane past the valid runs
                    const bool solid = inCol && gl < endValid && r_ci >= 0; // valid and !IsAir
                    const bool above = r_eMin > worldBoundsMax, below = r_eMax < worldBoundsMin;
                    const bool isBreak = solid && (ITER > 0 ? (!above && below) : above); // :461-475 (above is tested first)
                    const uint32_t breakMask = GBALLOT(isBreak);
                    const int endVisit = breakMask ? __ffs(breakMask) : endValid;           // the breaking run itself was dereferenced
                    if (invalidHere | breakMask) colStop = true;
                    const bool active = solid && gl < endVisit && !above && !below;
                    const bool sideOk = active && r_sideClip;
                    const bool capOk = active && r_capClip &&
                                       (r_capKind == 1 ? !(r_eMax > worldBoundsMax) : !(r_eMin < worldBoundsMin)); // :549-565

                    STAMP(6);
                    // ---- commit, in reference order (side of run j, cap of run j, side of run j+1, ...), only the spans that still
                    // hold an unwritten pixel; everything ordered before the committed span is a no-op now and stays one (written
                    // pixels only grow, the writable range only shrinks), so it is retired with it.
                    uint32_t candS = GBALLOT(sideOk) & roundHotS, candC = GBALLOT(capOk) & roundHotC;
                    int visitedHere = endVisit - base;
                    while (candS | candC) {
                        const int jS = candS ? __ffs(candS) - 1 : 64, jC = candC ? __ffs(candC) - 1 : 64;
                        const bool isCap = jC < jS;
                        const int j = isCap ? jC : jS;
                        if (isCap) candC &= candC - 1u; else candS &= candS - 1u;
                        int bMin = GSHFL(isCap ? r_cMin : r_sMin, j), bMax = GSHFL(isCap ? r_cMax : r_sMax, j);
                        EMU_STAT(5); // commit candidates examined
                        STAMP(8);
                        if (!span_would_write(rw, bMin, bMax)) { STAMP(6); continue; } // written over / cut off since the round was formed
                        EMU_STAT(6); // spans committed (each writes at least one pixel)
                        if (isCap) EMU_STAT(7);
                        STAMP(9);
                        reduce_pixel_horizon(rw, bMin, bMax); // :507-517 / :583-593
                        STAMP(10);
                        if (isCap) {
                            const uint32_t color = FAST ? GSHFL(r_capColor, j) : cache[7 * G + j];
                            for (int y = bMin + gl; y <= bMax; y += G) // :595-602
                                if (!((rw.seen[y >> 5] >> (y & 31)) & 1u)) row[y] = color;
                        } else {
                            STAMP(11);
                            float jbfx, jbfy, jAx, jAy, jBx, jBy;
                            int jLen;
                            const int jCi = GSHFL(r_ci, j);
                            if (FAST) {
                                // the perspective-correct u of :490-491,525-530 is needed only now, for the one span that writes, and
                                // only if the run is longer than one voxel (clamp(floor(u), 0, Length - 1) is 0 otherwise): rebuild the
                                // span's ends from the boundary points of lanes j and j + 1 exactly as :478-502 does
                                jLen = GSHFL(r_len, j);
                                jbfx = jbfy = jAx = jAy = jBx = jBy = 0.0f;
                                if (jLen > 1) {
                                    const F3 pj = F3{GSHFL(bFx, j), GSHFL(bFy, j), GSHFL(bFz, j)}, pn = F3{GSHFL(bFx, j + 1), GSHFL(bFy, j + 1), GSHFL(bFz, j + 1)};
                                    F3 frontBottom = ITER > 0 ? pn : pj, frontTop = ITER > 0 ? pj : pn;
                                    float uA = (float)jLen, uB = 0.0f;
                                    clip_near_u(frontBottom, frontTop, uA, uB);
                                    jAx = 1.0f / frontBottom.z; jAy = uA / frontBottom.z;
                                    jBx = 1.0f / frontTop.z;    jBy = uB / frontTop.z;
                                    jbfx = frontBottom.x / frontBottom.z; jbfy = frontTop.x / frontTop.z;
                                    if (jbfx > jbfy) {
                                        float t = jbfx; jbfx = jbfy; jbfy = t;
                                        t = jAx; jAx = jBx; jBx = t;
                                        t = jAy; jAy = jBy; jBy = t;
                                    }
                                }
                            } else {
                                jbfx = __uint_as_float(cache[0 * G + j]); jbfy = __uint_as_float(cache[1 * G + j]);
                                jAx = __uint_as_float(cache[2 * G + j]); jAy = __uint_as_float(cache[3 * G + j]);
                                jBx = __uint_as_float(cache[4 * G + j]); jBy = __uint_as_float(cache[5 * G + j]);
                                jLen = (int)cache[6 * G + j];
                            }
                            STAMP(12);
                            for (int y = bMin + gl; y <= bMax; y += G) { // :519-533
                                if (!((rw.seen[y >> 5] >> (y & 31)) & 1u)) {
                                    int idx = jCi;
                                    if (!FAST || jLen > 1) {
                                        float l = unlerpf(jbfx, jbfy, (float)y);
                                        float wx = lerpf(jAx, jBx, l), wy = lerpf(jAy, jBy, l);
                                        float u = wy / wx;
                                        idx = max(0, min(jLen - 1, f2i(floorf(u)))) + jCi;
                                    }
                                    row[y] = __ldg(colColors + idx);
                                }
                            }
                        }
                        STAMP(13);
                        __syncwarp(gmask);
                        { const int fresh = mark_seen<G>(rw.seen, bMin, bMax, gl); if (COUNTERS) acc.px_voxel += fresh; }
                        __syncwarp(gmask);
                        STAMP(6);
                        frustumDirMaxWorld = EPS; // a pixel was written (:522,598)
                        if (rw.nf_min > rw.nf_max) { terminated = true; visitedHere = j + 1 - base; break; } // :535-539,604-608
                    }
                    if (COUNTERS && gl == 0) acc.runs_visited += visitedHere;
                    if (tall) { k0 += FAST ? G - 1 : G; roundCols = 0u; } // the cache held one pass of this column only
                } while (tall && k0 < runCount && !colStop && !terminated);
                STAMP(4);
                if (terminated) { cellsDone = c + 1; break; }
            }
            if (COUNTERS && gl == 0) acc.dda_steps += cellsDone;
            if (endKind != 0) reachedEnd = true;
        }
        STAMP(7);
        // WriteSkybox :699-708 — :248,268,323,401,419,537,606,619 all end here
        __syncwarp(gmask);
        for (int y = rw.orig_min + gl; y <= rw.orig_max; y += G)
            if (!((rw.seen[y >> 5] >> (y & 31)) & 1u)) row[y] = SKYBOX_ARGB;
        if (COUNTERS) {
            for (int w = (rw.orig_min >> 5) + gl; w <= (rw.orig_max >> 5); w += G) {
                uint32_t m = FULL_MASK;
                if (w == (rw.orig_min >> 5)) m &= mask_from(rw.orig_min);
                if (w == (rw.orig_max >> 5)) m &= mask_to(rw.orig_max);
                acc.px_sky += __popc(~rw.seen[w] & m);
            }
        }
    }

    STAMP(0);
    if (TIMING && f.timing && gl == 0)
        for (int i = 0; i < CVXD_TIMING_REGIONS; i++) f.timing[(int64_t)flat * CVXD_TIMING_REGIONS + i] = tAcc[i];
#undef STAMP
    if (COUNTERS && f.counters) {
        if (acc.dda_steps) atomicAdd(&f.counters->dda_steps, acc.dda_steps);
        if (acc.columns_nonempty) atomicAdd(&f.counters->columns_nonempty, acc.columns_nonempty);
        if (acc.runs_visited) atomicAdd(&f.counters->runs_visited, acc.runs_visited);
        if (acc.px_voxel) atomicAdd(&f.counters->px_voxel, acc.px_voxel);
        if (acc.px_sky) atomicAdd(&f.counters->px_sky, acc.px_sky);
        if (gl == 0) atomicAdd(&f.counters->rays, 1ull);
    }
#undef GBALLOT
#undef GSHFL
#undef worldMaxY
#undef cameraPosYNormalized
}

// ---- Phase 2 -----------------------------------------------------------------------------------------------
// Per pixel centre (x+0.5, y+0.5), bottom-left origin. Triangle k = (VP, MaxScreen_k, MinScreen_k) carries
// uv = (0,0),(1,0),(0,1) (RenderManager.cs:215-222), so uv.x / uv.y are the affine weights b / c of Max / Min.
// The pixel takes the first segment with b >= 0 and c >= 0 (else the one with the largest min(b,c)); the ray row is
// floor((offset_k + b/(b+c) * scale_k) * bufferRows) (shader :55-56, RenderManager.cs:235-242) clamped to the
// segment's rows, the column is y (top/down) or x (left/right) (shader :58-62), point sampled.
//
// phase2_kernel is a tile mover: one CTA per 64 x 32 screen tile, 8 pixels per thread.
//  - Which segment a pixel belongs to is a sign test; almost every tile lies inside ONE segment (only the tiles the two diagonals
//    through the vanishing point cross do not). Each warp decides that from the tile's four corner pixels with a safety margin
//    (far above fp32 rounding), and then every pixel needs the two weights of that segment and ONE IEEE division, b / (b + c).
//  - A warp instruction covers an 8 x 4 pixel block with the 8 along the raybuffer's contiguous axis (x for the left/right
//    buffer, y for the top/down buffer): the ray row changes by about one row per pixel in both screen directions near the
//    diagonals, so a 32 x 1 strip touches up to 32 rows (32 sectors) where the block touches ~12.
//  - Top/down tiles are therefore read with lanes along y, staged in shared memory (pitch 36: conflict free both ways) and
//    written to the frame with lanes along x (full 128-byte rows); left/right tiles are written directly.
//  - Tiles crossed by a segment boundary take the general per-pixel path (every segment tested, as the restated formula reads).
// Same arithmetic in all paths (IEEE fp32, no FMA contraction): the frame is bit-identical whichever path a pixel takes.
struct P2Pixel { uint32_t color; bool owned; };

// per-segment constants of the row formula (RenderManager.cs:235-242), computed once per thread
struct P2Seg {
    float e1x, e1y, e2x, e2y, det;  // VP -> MaxScreen (weight b), VP -> MinScreen (weight c), their cross product
    float scale, offset, rowsF;     // _RayScale[k], _RayOffset[k], rows of the segment's raybuffer
    int off01, rc, flatBase;        // first raybuffer row of the segment, its ray count, flat index of its first ray
};
__device__ __forceinline__ P2Seg p2_seg(const cvxd_blit& p, int k) {
    P2Seg g;
    g.e1x = p.seg[k].max_screen[0] - p.vp_x; g.e1y = p.seg[k].max_screen[1] - p.vp_y;
    g.e2x = p.seg[k].min_screen[0] - p.vp_x; g.e2y = p.seg[k].min_screen[1] - p.vp_y;
    g.det = g.e1x * g.e2y - g.e1y * g.e2x;
    const int rows = k < 2 ? p.width + 2 * p.height : 2 * p.width + p.height;
    g.rc = p.seg[k].ray_count;
    g.rowsF = (float)rows;
    g.scale = p.seg_scale[k];        // (float)rc / rowsF and (float)off01 / rowsF, divided once on the host (cvxd_blit_prepare)
    g.off01 = p.seg_off01[k];
    g.offset = p.seg_offset[k];
    g.flatBase = p.seg_flat_base[k];
    return g;
}

// The shader's x = uv.x / (uv.x + uv.y) (RayBufferBlit.shader:55): uv.x, uv.y are the affine weights nb/det, nc/det of MaxScreen and
// MinScreen; their common factor 1/det cancels, so the weights stay unnormalised (signs as for det > 0) and a pixel costs one division.
// raybuffer row of a pixel with weights (nb, nc) in segment g, and whether this launch owns it (sharded mode)
template <bool OWNED>
__device__ __forceinline__ int p2_row(const cvxd_blit& p, const P2Seg& g, float nb, float nc, bool& owned) {
    const float t = nb / (nb + nc);
    const float v = g.offset + t * g.scale;
    int row = f2i(floorf(v * g.rowsF));
    row = max(g.off01, min(g.off01 + g.rc - 1, row));
    owned = true;
    if (OWNED) {
        const int flat = g.flatBase + row - g.off01;
        // interleaved: chunk (a power of two) c = flat / chunk belongs to rank c mod ranks
        owned = p.il_chunk > 0 ? (int)((uint32_t)(flat >> (31 - __clz(p.il_chunk))) % (uint32_t)p.il_ranks) == p.il_rank : (flat >= p.ray_begin && flat < p.ray_end);
    }
    return row;
}
template <bool OWNED>
__device__ __forceinline__ P2Pixel p2_fetch(const cvxd_blit& p, const P2Seg& g, bool td, float nb, float nc, int x, int y) {
    P2Pixel r; r.color = 0u;
    const int row = p2_row<OWNED>(p, g, nb, nc, r.owned);
    if (r.owned) r.color = td ? __ldg(p.td + (int64_t)row * p.height + y) : __ldg(p.lr + (int64_t)row * p.width + x);
    return r;
}

// general path: the first active segment whose weights are both >= 0, else (rounding on an outer edge) the nearest one
template <bool OWNED>
__device__ __forceinline__ P2Pixel p2_pixel_general(const cvxd_blit& p, int x, int y) {
    const float px = (float)x + 0.5f, py = (float)y + 0.5f;
    const float dx = px - p.vp_x, dy = py - p.vp_y;
    int best = -1; float bestB = 0.0f, bestC = 0.0f, bestScore = __int_as_float(0xff800000);
    bool found = false;
#pragma unroll
    for (int k = 0; k < 4; k++) {
        if (p.seg[k].ray_count <= 0 || found) continue;
        const float e1x = p.seg[k].max_screen[0] - p.vp_x, e1y = p.seg[k].max_screen[1] - p.vp_y;
        const float e2x = p.seg[k].min_screen[0] - p.vp_x, e2y = p.seg[k].min_screen[1] - p.vp_y;
        const float det = e1x * e2y - e1y * e2x;
        float nb = dx * e2y - dy * e2x, nc = e1x * dy - e1y * dx;
        if (det < 0.0f) { nb = -nb; nc = -nc; }
        if (nb >= 0.0f && nc >= 0.0f) { best = k; bestB = nb; bestC = nc; found = true; }
        else {
            const float score = minf_(nb, nc) / fabsf(det);
            if (score > bestScore) { bestScore = score; best = k; bestB = nb; bestC = nc; }
        }
    }
    if (best < 0) { P2Pixel r; r.color = 0u; r.owned = true; return r; }
    const P2Seg g = p2_seg(p, best);
    return p2_fetch<OWNED>(p, g, best < 2, bestB, bestC, x, y);
}

// a pixel known to lie inside segment g (both weights >= 0 there, and in no earlier segment): the same weights and row as above
template <bool OWNED>
__device__ __forceinline__ int p2_row_in(const cvxd_blit& p, const P2Seg& g, int x, int y, bool& owned) {
    const float px = (float)x + 0.5f, py = (float)y + 0.5f;
    const float dx = px - p.vp_x, dy = py - p.vp_y;
    float nb = dx * g.e2y - dy * g.e2x, nc = g.e1x * dy - g.e1y * dx;
    if (g.det < 0.0f) { nb = -nb; nc = -nc; }
    return p2_row<OWNED>(p, g, nb, nc, owned);
}

#ifndef P2_TW /* tile width in pixels: 32 or 64 (8 pixels per thread); the height is 32 */
#define P2_TW 64
#endif
#ifndef P2_MINB
#define P2_MINB 6
#endif
#define P2_TH 32
#define P2_PITCH (P2_TW + 4) /* = 4 mod 32: the staged top/down tile is bank-conflict free both ways */
#ifndef CVX_EMU /* the emulator build covers Phase 1 only */
template <bool OWNED>
__global__ void __launch_bounds__(256, P2_MINB)
phase2_kernel(const __grid_constant__ cvxd_blit p) {
    constexpr int NX = P2_TW / 8;    // left/right path: 8-pixel groups along x per thread
    constexpr int NH = P2_TW / 32;   // top/down path: 32-column halves of the tile
    __shared__ uint32_t tile[P2_TH * P2_PITCH];
    __shared__ uint32_t ownBits[P2_TH * NH];
    __shared__ int uniShared;
    __shared__ P2Seg segShared;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * P2_TW, y0 = p.row_begin + blockIdx.y * P2_TH;
    const int xLast = min(x0 + P2_TW, p.width) - 1, yLast = min(y0 + P2_TH, p.row_end) - 1;

    // ---- the segment that holds the whole tile, if one does: lanes 0..3 of warp 0 test one corner pixel each against every
    // segment; the verdict and that segment's constants go to the other warps through shared memory
    if (warp == 0) {
        // 16 lanes: lane = 4 * segment + corner tests one corner pixel against one segment; a segment holds the tile if its four lanes agree
        int u = -1;
        {
            const int k = (lane >> 2) & 3;
            const float px = (float)((lane & 1) ? xLast : x0) + 0.5f, py = (float)((lane & 2) ? yLast : y0) + 0.5f;
            const float dx = px - p.vp_x, dy = py - p.vp_y;
            bool in = false;
            if (lane < 16 && p.seg[k].ray_count > 0) {
                const float e1x = p.seg[k].max_screen[0] - p.vp_x, e1y = p.seg[k].max_screen[1] - p.vp_y;
                const float e2x = p.seg[k].min_screen[0] - p.vp_x, e2y = p.seg[k].min_screen[1] - p.vp_y;
                const float det = e1x * e2y - e1y * e2x;
                const float tb0 = dx * e2y, tb1 = dy * e2x, tc0 = e1x * dy, tc1 = e1y * dx;
                const float sgn = det > 0.0f ? 1.0f : -1.0f;
                // margin: 1e-5 of the products' magnitude, ~40x the rounding error of the difference; a linear function that
                // clears it at the four corners is positive — also as computed — at every pixel of the tile
                const float nb = (tb0 - tb1) * sgn, nc = (tc0 - tc1) * sgn;
                in = fabsf(det) > 1e-20f && fabsf(det) < 1e30f && nb > 1e-5f * (fabsf(tb0) + fabsf(tb1)) && nc > 1e-5f * (fabsf(tc0) + fabsf(tc1));
            }
            const uint32_t m = __ballot_sync(FULL_MASK, in);
#pragma unroll
            for (int j = 3; j >= 0; j--) if (((m >> (4 * j)) & 0xfu) == 0xfu) u = j;   // the first segment that holds all four corners
        }
        P2Seg g;
        if (u >= 0) g = p2_seg(p, u);
        if (OWNED && u >= 0) {
            // sharded mode: the ray row is monotone along any line inside one segment, so the tile's rows lie between the rows of its
            // four corner pixels; if none of them (nor anything between) belongs to this launch the whole tile is someone else's
            bool owned;
            const int cx = (lane & 1) ? xLast : x0, cy = (lane & 2) ? yLast : y0;
            const int row = p2_row_in<false>(p, g, cx, cy, owned);
            int lo = row, hi = row;
#pragma unroll
            for (int o = 1; o < 4; o <<= 1) {
                lo = min(lo, __shfl_xor_sync(FULL_MASK, lo, o));
                hi = max(hi, __shfl_xor_sync(FULL_MASK, hi, o));
            }
            const int f0 = g.flatBase + lo - g.off01 - 1, f1 = g.flatBase + hi - g.off01 + 1;   // +-1: rounding at the corners
            bool mine;
            if (p.il_chunk > 0) {
                const int sh = 31 - __clz(p.il_chunk);
                const int c0 = max(f0, 0) >> sh, c1 = max(f1, 0) >> sh;
                // chunks c0..c1: one of them is this rank's iff the span covers a multiple of ranks or wraps onto il_rank
                mine = (c1 - c0 + 1 >= p.il_ranks) || ((p.il_rank - c0 % p.il_ranks + p.il_ranks) % p.il_ranks <= c1 - c0);
            } else mine = f1 >= p.ray_begin && f0 < p.ray_end;
            if (!mine) u = -2;
        }
        if (lane == 0) {
            uniShared = u;
            if (u >= 0) segShared = g;
        }
    }
    if (OWNED && threadIdx.x < P2_TH * NH) ownBits[threadIdx.x] = 0u;
    __syncthreads();
    const int uni = uniShared;
    if (uni == -2) return;   // sharded mode: no pixel of this tile is fed by this launch's rays

    if (uni >= 2) {
        // ---- left/right segment: lanes 8 along x, 4 along y; read and write directly. The rows first, then the gathers back
        // to back, then the stores (pixels beyond the screen edge: clamped, not stored)
        const P2Seg g = segShared;
        const int y = y0 + (lane >> 3) + 4 * warp;
        int xs[NX]; const uint32_t* src[NX]; bool ok[NX]; uint32_t col[NX];
        const int yc = min(y, yLast);
#pragma unroll
        for (int j = 0; j < NX; j++) {
            const int x = x0 + (lane & 7) + 8 * j;
            xs[j] = min(x, xLast);
            bool owned;
            const int row = p2_row_in<OWNED>(p, g, xs[j], yc, owned);
            ok[j] = owned && x <= xLast && y <= yLast;
            src[j] = p.lr + (int64_t)row * p.width + xs[j];
        }
#pragma unroll
        for (int j = 0; j < NX; j++) col[j] = (!OWNED || ok[j]) ? __ldg(src[j]) : 0u;
#pragma unroll
        for (int j = 0; j < NX; j++) if (ok[j]) p.frame[(int64_t)y * p.width + xs[j]] = col[j];
        return;
    }
    if (uni >= 0) {
        // ---- top/down segment: lanes 8 along y (the raybuffer's contiguous axis), 4 along x; staged for the row-major write
        const P2Seg g = segShared;
        const uint32_t* src[4 * NH]; bool ok[4 * NH]; uint32_t col[4 * NH];
#pragma unroll
        for (int h = 0; h < NH; h++) {
            const int x = x0 + (lane >> 3) + 4 * warp + 32 * h, xc = min(x, xLast);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int y = y0 + (lane & 7) + 8 * j, yc = min(y, yLast);
                bool owned;
                const int row = p2_row_in<OWNED>(p, g, xc, yc, owned);
                ok[h * 4 + j] = owned && x <= xLast && y <= yLast;
                src[h * 4 + j] = p.td + (int64_t)row * p.height + yc;
            }
        }
#pragma unroll
        for (int i = 0; i < 4 * NH; i++) col[i] = (!OWNED || ok[i]) ? __ldg(src[i]) : 0u;
#pragma unroll
        for (int h = 0; h < NH; h++) {
            const int lx = (lane >> 3) + 4 * warp + 32 * h;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int ly = (lane & 7) + 8 * j;
                tile[ly * P2_PITCH + lx] = col[h * 4 + j];
                if (OWNED && ok[h * 4 + j]) atomicOr(&ownBits[ly * NH + h], 1u << (lx & 31));
            }
        }
    } else {
        // ---- a segment boundary crosses the tile (or no segment is active): general per-pixel path, lanes along x
#pragma unroll
        for (int h = 0; h < NH; h++)
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int ly = warp + 8 * j, x = x0 + lane + 32 * h, y = y0 + ly;
                if (x <= xLast && y <= yLast) {
                    const P2Pixel r = p2_pixel_general<OWNED>(p, x, y);
                    if (r.owned) p.frame[(int64_t)y * p.width + x] = r.color;
                }
            }
        return;
    }
    __syncthreads();
#pragma unroll
    for (int h = 0; h < NH; h++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int ly = warp + 8 * j, x = x0 + lane + 32 * h, y = y0 + ly;
            if (x <= xLast && y <= yLast && (!OWNED || ((ownBits[ly * NH + h] >> lane) & 1u))) p.frame[(int64_t)y * p.width + x] = tile[ly * P2_PITCH + lane + 32 * h];
        }
}

#endif /* !CVX_EMU */

// ---- debug views: the shader's COPY_MAIN1 / COPY_MAIN2 variants (RayBufferBlit.shader:48-53) -----------------------
// uv = SV_POSITION.xy / _ScreenParams.xy with the pixel centre measured from the TOP (D3D, SURVEY.md A12); the fragment
// samples tex2D(buffer, float2(1 - uv.y, uv.x)), point filtered (RayBuffer.cs:32): texture x runs along a ray row
// (rowLen texels), texture y over the rows. So screen x selects the ray row and screen y the pixel along it.
__global__ void __launch_bounds__(256)
raybuffer_view_kernel(const uint32_t* __restrict__ buf, int rows, int rowLen, uint32_t* __restrict__ frame, int width, int height) {
    const int x = blockIdx.x * 32 + (threadIdx.x & 31);
    const int y = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (x >= width || y >= height) return;
    const float vx = (float)x + 0.5f, vy = (float)height - ((float)y + 0.5f); // SV_POSITION, y from the top
    const float uvx = vx / (float)width, uvy = vy / (float)height;
    const float tu = 1.0f - uvy, tv = uvx;
    int col = f2i(floorf(tu * (float)rowLen)), row = f2i(floorf(tv * (float)rows));
    col = max(0, min(rowLen - 1, col)); row = max(0, min(rows - 1, row)); // clamp addressing
    frame[(int64_t)y * width + x] = __ldg(buf + (int64_t)row * rowLen + col);
}

// ---- presentation: ColorARGB32 frame (bytes a,r,g,b; row 0 = bottom) -> RGBA8 or BGRA8, optionally top-down ------------
// One 128-bit load and store per thread (4 pixels); width is a multiple of 4 on this path, other widths take the scalar tail.
__global__ void __launch_bounds__(256)
present_kernel(const uint32_t* __restrict__ frame, uint32_t* __restrict__ out, int width, int height, int bgra, int topDown) {
    const int quadsPerRow = (width + 3) >> 2;
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= (int64_t)quadsPerRow * height) return;
    const int y = (int)(q / quadsPerRow), x = (int)(q - (int64_t)y * quadsPerRow) * 4;
    const uint32_t* src = frame + (int64_t)y * width + x;
    uint32_t* dst = out + (int64_t)(topDown ? height - 1 - y : y) * width + x;
    // [a,r,g,b] -> [r,g,b,a] is a byte rotation, -> [b,g,r,a] a byte reversal
    const uint32_t sel = bgra ? 0x0123u : 0x0321u;
    if (x + 3 < width && (width & 3) == 0) {
        uint4 v = *reinterpret_cast<const uint4*>(src);
        v.x = __byte_perm(v.x, 0u, sel); v.y = __byte_perm(v.y, 0u, sel); v.z = __byte_perm(v.z, 0u, sel); v.w = __byte_perm(v.w, 0u, sel);
        *reinterpret_cast<uint4*>(dst) = v;
    } else {
        for (int i = 0; i < 4 && x + i < width; i++) dst[i] = __byte_perm(src[i], 0u, sel);
    }
}

// ColorARGB32 frame -> packed R,G,B bytes (3 per pixel: the input of still/video encoders and of image files), optionally top-down.
// A thread takes 4 pixels (one 128-bit load) and writes 12 bytes as three words when the row pitch allows, else byte by byte.
__global__ void __launch_bounds__(256)
present_rgb8_kernel(const uint32_t* __restrict__ frame, uint8_t* __restrict__ out, int width, int height, int topDown) {
    const int quadsPerRow = (width + 3) >> 2;
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= (int64_t)quadsPerRow * height) return;
    const int y = (int)(q / quadsPerRow), x = (int)(q - (int64_t)y * quadsPerRow) * 4;
    const uint32_t* src = frame + (int64_t)y * width + x;
    uint8_t* dst = out + ((int64_t)(topDown ? height - 1 - y : y) * width + x) * 3;
    if ((width & 3) == 0) { // rows of 3 * width bytes start on a word boundary, and so does every quad
        const uint4 v = *reinterpret_cast<const uint4*>(src);
        uint32_t* d = reinterpret_cast<uint32_t*>(dst);
        d[0] = __byte_perm(v.x, v.y, 0x5321u); // r0 g0 b0 r1   (a pixel's bytes in memory: a, r, g, b)
        d[1] = __byte_perm(v.y, v.z, 0x6532u); // g1 b1 r2 g2
        d[2] = __byte_perm(v.z, v.w, 0x7653u); // b2 r3 g3 b3
    } else {
        for (int i = 0; i < 4 && x + i < width; i++) {
            const uint32_t p = src[i];
            dst[3 * i] = (uint8_t)(p >> 8); dst[3 * i + 1] = (uint8_t)(p >> 16); dst[3 * i + 2] = (uint8_t)(p >> 24);
        }
    }
}

__global__ void ray_setup_kernel(const __grid_constant__ cvxd_world world, const __grid_constant__ cvxd_frame f, cvxd_ray_state* out, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    RaySetup rs;
    setup_ray(world, f, i, rs);
    cvxd_ray_state o;
    o.segment = rs.segment; o.plane_ray_index = rs.plane_index; o.status = rs.status; o.lod = rs.lod;
    o.position[0] = rs.dda.px; o.position[1] = rs.dda.pz; o.step[0] = rs.dda.sx; o.step[1] = rs.dda.sz;
    o.start[0] = rs.dda.start_x; o.start[1] = rs.dda.start_z; o.dir[0] = rs.dda.dir_x; o.dir[1] = rs.dda.dir_z;
    o.t_delta[0] = rs.dda.tdx; o.t_delta[1] = rs.dda.tdz; o.t_max[0] = rs.dda.tmx; o.t_max[1] = rs.dda.tmz;
    o.intersection_distances[0] = rs.dda.dl; o.intersection_distances[1] = rs.dda.dn;
    out[i] = o;
}

__global__ void fill_kernel(uint32_t* dst, uint32_t value, int64_t n) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) dst[i] = value;
}

} // namespace

#ifndef CVX_EMU
template <int G>
static cudaError_t launch_phase1_g(const cvxd_world& world, const cvxd_frame& frame, int n, cudaStream_t stream) {
    constexpr int groupsPerCta = CVXD_THREADS_PER_CTA / G;
    const int blocks = (n + groupsPerCta - 1) / groupsPerCta;
    const int seenWords = ((frame.width > frame.height ? frame.width : frame.height) + 31) >> 5;
    const size_t smem = (size_t)groupsPerCta * (seenWords + 9 * G) * sizeof(uint32_t);
    // FAST: the boundary-table kernel, for regular worlds (world_transcode.h)
    const bool fast = world.regular && !frame.general_path;
#define CVXD_P1(C, T, F) do { \
        if (frame.inverse) phase1_kernel<G, C, T, F, true><<<blocks, CVXD_THREADS_PER_CTA, smem, stream>>>(world, frame); \
        else               phase1_kernel<G, C, T, F, false><<<blocks, CVXD_THREADS_PER_CTA, smem, stream>>>(world, frame); } while (0)
    if (frame.timing) {
        if constexpr (G != 32) return cudaErrorInvalidValue; // the timing build exists for the default group width only
        else { if (fast) CVXD_P1(false, true, true); else CVXD_P1(false, true, false); }
    }
    else if (frame.counters) { if (fast) CVXD_P1(true, false, true); else CVXD_P1(true, false, false); }
    else { if (fast) CVXD_P1(false, false, true); else CVXD_P1(false, false, false); }
#undef CVXD_P1
    return cudaGetLastError();
}

// group_size: lanes per ray (8, 16, 32) or 0 = automatic. Measured on B200 (mill 1024^3, 1080p and 4K, 1920..12000 rays
// per frame): the frame time is set by its slowest ray, and a full warp per ray has the shortest per-ray chain, so
// automatic = 32; narrower groups only pay off when far more rays than resident warps are in flight.
cudaError_t cvxd_launch_phase1(const cvxd_world& world, const cvxd_frame& frame, int group_size, cudaStream_t stream) {
    const int n = frame.ray_end - frame.ray_begin;
    if (n <= 0) return cudaSuccess;
    int g = group_size;
    if (g != 8 && g != 16 && g != 32) g = 32;
    if (g == 32) return launch_phase1_g<32>(world, frame, n, stream);
    if (g == 16) return launch_phase1_g<16>(world, frame, n, stream);
    return launch_phase1_g<8>(world, frame, n, stream);
}

cudaError_t cvxd_launch_phase2(const cvxd_blit& blit, cudaStream_t stream) {
    int rows = blit.row_end - blit.row_begin;
    if (rows <= 0 || blit.width <= 0) return cudaSuccess;
    dim3 grid((blit.width + P2_TW - 1) / P2_TW, (rows + P2_TH - 1) / P2_TH);
    if (blit.owned_only) phase2_kernel<true><<<grid, 256, 0, stream>>>(blit);
    else phase2_kernel<false><<<grid, 256, 0, stream>>>(blit);
    return cudaGetLastError();
}

cudaError_t cvxd_launch_ray_setup(const cvxd_world& world, const cvxd_frame& frame, cvxd_ray_state* out, int n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    ray_setup_kernel<<<(n + 127) / 128, 128, 0, stream>>>(world, frame, out, n);
    return cudaGetLastError();
}

cudaError_t cvxd_launch_fill(uint32_t* dst, uint32_t value, int64_t n, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    fill_kernel<<<148 * 8, 256, 0, stream>>>(dst, value, n);
    return cudaGetLastError();
}
cudaError_t cvxd_launch_raybuffer_view(const uint32_t* buf, int rows, int row_len, uint32_t* frame, int width, int height, cudaStream_t stream) {
    if (width <= 0 || height <= 0) return cudaSuccess;
    dim3 grid((width + 31) / 32, (height + 7) / 8);
    raybuffer_view_kernel<<<grid, 256, 0, stream>>>(buf, rows, row_len, frame, width, height);
    return cudaGetLastError();
}

cudaError_t cvxd_launch_present(const uint32_t* frame, uint32_t* out, int width, int height, int bgra, int top_down, cudaStream_t stream) {
    if (width <= 0 || height <= 0) return cudaSuccess;
    const int64_t quads = (int64_t)((width + 3) >> 2) * height;
    present_kernel<<<(unsigned)((quads + 255) / 256), 256, 0, stream>>>(frame, out, width, height, bgra, top_down);
    return cudaGetLastError();
}
cudaError_t cvxd_launch_present_rgb8(const uint32_t* frame, uint8_t* out, int width, int height, int top_down, cudaStream_t stream) {
    if (width <= 0 || height <= 0) return cudaSuccess;
    const int64_t quads = (int64_t)((width + 3) >> 2) * height;
    present_rgb8_kernel<<<(unsigned)((quads + 255) / 256), 256, 0, stream>>>(frame, out, width, height, top_down);
    return cudaGetLastError();
}
#endif /* !CVX_EMU */
