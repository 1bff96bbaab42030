/*
 * capi.cu — the C ABI of libcpuvox_b200.so (include/cpuvox_b200.h): context, world upload, resolution, draw, readback.
 * Replaces the body of RenderManager.DrawSegments (Assets/Code/RenderManager.cs:258-372), RayBuffer upload/copy
 * (Assets/Code/Rendering/RayBuffer.cs:79-96) and BlitSegments (RenderManager.cs:199-256). No CPU fallback: every
 * entry point that renders needs a CUDA device, and fails with an error code (never an exception) otherwise.
 */
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/cpuvox_b200.h"
#include "device_types.h"
#include "host_frame.h"
#include "jpeg_encoder.h"
#include "nvtx_ranges.h"
#include "raycast.h"
#include "world_builder.h"

static_assert(sizeof(cvx_ray_state) == sizeof(cvxd_ray_state), "ray state layout");
static_assert(sizeof(cvx_counters) == sizeof(cvxd_counters), "counter layout");
static_assert(CVX_LOD_LEVELS == CVXD_LODS, "lod levels");
static_assert(sizeof(cvx_ray) == sizeof(cvxd_ray) && sizeof(cvx_ray) == 32, "ray layout");
static_assert(sizeof(cvx_ray_hit) == sizeof(cvxd_ray_hit) && sizeof(cvx_ray_hit) == 32, "ray hit layout");

#define CVX_MAX_SLOTS 16
#define CVX_DEFAULT_SLOTS 6
#define CVX_POOL_FRAMES 32 /* cvx_draw_batch with a host destination: framebuffers between Phase 2 and the device->host copies */

extern "C" int cvx_ring_close(cvx_ctx* ctx);

// cvx_draw_batch keeps several views in flight: view i renders on slot i % slotCount, each slot with its own raybuffers and
// framebuffer. Slot 0 renders on the context's stream (slot_stream; its own `stream` stays null) and gets its buffers from
// cvx_set_resolution; the others have a stream of their own and get their buffers on first use.
struct cvx_slot {
    cudaStream_t stream = nullptr;
    uint32_t* td = nullptr;
    uint32_t* lr = nullptr;
    uint32_t* frame = nullptr;
    cudaEvent_t done = nullptr;     // slots 1..: joins the slot's views into the context's stream
};

// device memory of one uploaded LOD (what ctx->world.lods[i] points into)
struct cvx_lod_memory {
    void* blob = nullptr;           // the uploaded blob: column headers, then the element area the kernels read
    void* headers = nullptr;        // the Phase-1 tables built from it (world_builder_gpu.cu)
    void* bounds = nullptr;
    bool regular = false;
};

struct cvx_ctx {
    int device = 0;
    int flags = 0;
    cudaStream_t stream = nullptr;      // compute
    cudaStream_t copyStream = nullptr;  // device->host copies of pooled batch frames (cvx_draw_batch with dst_frames) and cvx_ring_consume
    bool ownStream = true;
    cvxd_world world;
    cvx_lod_memory lod[CVX_LOD_LEVELS];
    int width = 0, height = 0;
    cvx_slot slots[CVX_MAX_SLOTS];
    int slotCount = CVX_DEFAULT_SLOTS;  // CVX_OPT_FRAMES_IN_FLIGHT
    int slotsReady = 0;                 // slots holding buffers for the current resolution
    int lastSlot = 0;                   // slot of the most recent view (what the read functions return)
    cudaEvent_t evBatchStart = nullptr;
    // cvx_draw_batch with dst_frames: Phase 2 writes into a pool of framebuffers that a copy stream drains, so a slot starts its next
    // view without waiting for its frame's device->host copy (poolReady[p]: frame p rendered; poolFree[p]: frame p copied out)
    uint32_t* pool[CVX_POOL_FRAMES] = {nullptr};
    cudaEvent_t poolReady[CVX_POOL_FRAMES] = {nullptr}, poolFree[CVX_POOL_FRAMES] = {nullptr};
    int poolCount = 0;                  // pool frames allocated for the current resolution
    bool poolUsed[CVX_POOL_FRAMES] = {false};
    // asynchronous batches (cvx_draw_batch_async): batchDone[b % 4] is recorded on the copy stream behind batch b's last copy
    cudaEvent_t batchDone[4] = {nullptr, nullptr, nullptr, nullptr};
    int64_t batchSeq = 0, batchSettled = 0;   // batches issued / batches the context's stream has been ordered behind
    uint32_t* externalFrame = nullptr;
    uint32_t* presentStage = nullptr;   // cvx_present with a host destination / cvx_present_jpeg: converted frame (W*H*4 bytes)
    cvxjpeg::Encoder* jpeg = nullptr;   // created by the first cvx_present_jpeg
    std::vector<uint8_t> jpegOut;
    cvxd_counters* counters = nullptr;
    cudaEvent_t evStart = nullptr, evMid = nullptr, evEnd = nullptr;
    cudaEvent_t evFrameDone = nullptr, evCopyDone = nullptr;  // a pooled batch: its last view rendered / its copies done
    bool timed = false;
    int64_t launches = 0;
    std::vector<cudaEvent_t> profEvents; // 3 per profiled view: start, mid, end
    int profCapacity = 0, profCount = 0;
    // frame ring (multi-GPU, rays sharded): `ringSlots` framebuffers + flag words in one allocation that lives on the root rank;
    // the other ranks hold an IPC mapping of it. Flag words: arrive[slot][rank] and released[slot] (see cvx_ring_create).
    uint8_t* ring = nullptr;
    bool ringOwner = false;
    int ringSlots = 0, ringWorld = 0;
    size_t ringFrameBytes = 0;
    int groupSize = 0;                  // lanes per ray in phase 1: 0 = auto, 8, 16, 32
    int generalPath = 0;                // 1 = never use the boundary-table kernel
    void* rayScratch = nullptr;         // cvx_raycast with host arrays: rays then hits, grown to the largest call
    size_t rayScratchBytes = 0;
    std::string error;
};

namespace {

std::string g_createError;

int fail(cvx_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->error = buf; else g_createError = buf;
    return code;
}

#define CU(ctx, call)                                                                                     \
    do {                                                                                                  \
        cudaError_t e_ = (call);                                                                          \
        if (e_ != cudaSuccess) return fail(ctx, cvx_code(e_), "%s failed: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

bool pow2(int n) { return n > 0 && (n & (n - 1)) == 0; }

// Raybuffer `which` (0 = top/down, 1 = left/right; RenderManager.cs:35-36): W + 2H rows of H pixels, or 2W + H rows of W pixels
int raybuffer_rows(const cvx_ctx* ctx, int which) { return which == 0 ? ctx->width + 2 * ctx->height : 2 * ctx->width + ctx->height; }
int raybuffer_row_length(const cvx_ctx* ctx, int which) { return which == 0 ? ctx->height : ctx->width; }
int64_t raybuffer_pixels(const cvx_ctx* ctx, int which) { return (int64_t)raybuffer_rows(ctx, which) * raybuffer_row_length(ctx, which); }
uint32_t* raybuffer(const cvx_slot& sl, int which) { return which == 0 ? sl.td : sl.lr; }

cudaStream_t slot_stream(const cvx_ctx* ctx, int s) { return s == 0 ? ctx->stream : ctx->slots[s].stream; }

int validate_setup(cvx_ctx* ctx, const cvx_frame_setup* s) {
    int tdRays = (s->segments[0].ray_count > 0 ? s->segments[0].ray_count : 0) + (s->segments[1].ray_count > 0 ? s->segments[1].ray_count : 0);
    int lrRays = (s->segments[2].ray_count > 0 ? s->segments[2].ray_count : 0) + (s->segments[3].ray_count > 0 ? s->segments[3].ray_count : 0);
    if (tdRays > raybuffer_rows(ctx, 0) || lrRays > raybuffer_rows(ctx, 1))
        return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "segment ray counts (%d top/down, %d left/right) exceed the raybuffers (%d, %d rows)", tdRays, lrRays, raybuffer_rows(ctx, 0), raybuffer_rows(ctx, 1));
    // RenderManager.cs:482-483 clamps RayCount at 0; a negative count would give a negative row offset (host_frame.h: ray_index_offset)
    for (int k = 0; k < 4; k++)
        if (s->segments[k].ray_count < 0) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "segment %d has a negative ray count (%d)", k, s->segments[k].ray_count);
    return CVX_OK;
}

// the frame of `s`, drawn into slot `slot`'s raybuffers
void make_frame(cvx_ctx* ctx, const cvx_frame_setup* s, int slot, cvxd_frame& f) {
    cvxh::frame_from_setup(s, ctx->width, ctx->height, f);
    cvxd_frame_set_world(&f, &ctx->world); // also sets the distances of the last uploaded LOD and beyond to +inf
    f.td = ctx->slots[slot].td; f.lr = ctx->slots[slot].lr;
    f.counters = (ctx->flags & CVX_FLAG_COUNTERS) ? ctx->counters : nullptr;
    f.general_path = ctx->generalPath;
}

// Phase 2 of frame `f` into `target`: every row, from the raybuffers and rays of `f`
void make_blit(const cvxd_frame& f, uint32_t* target, cvxd_blit& b) {
    memset(&b, 0, sizeof b);
    memcpy(b.seg, f.seg, sizeof b.seg);
    b.vp_x = f.vp_x; b.vp_y = f.vp_y;
    b.width = f.width; b.height = f.height;
    b.row_begin = 0; b.row_end = f.height;
    b.ray_begin = f.ray_begin; b.ray_end = f.ray_end; b.owned_only = 0;
    b.il_chunk = f.il_chunk; b.il_ranks = f.il_ranks; b.il_rank = f.il_rank;
    b.td = f.td; b.lr = f.lr;
    b.frame = target;
    cvxd_blit_prepare(&b);
}

// [begin, end) within [0, n): an end below 0 or past n means n
void clamp_range(int& begin, int& end, int n) {
    if (end < 0 || end > n) end = n;
    if (begin < 0) begin = 0;
}

int check_ready(cvx_ctx* ctx, const void* setup) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (!setup) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "frame setup is NULL");
    if (ctx->world.lod_count <= 0 || !ctx->world.lods[0].headers) return fail(ctx, CVX_ERR_NO_WORLD, "no world uploaded (LOD 0 missing)");
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "cvx_set_resolution has not been called");
    return CVX_OK;
}

// What the entry points that draw one setup start with: the context is ready and `f` is the frame of `setup` on slot `slot`,
// checked against the raybuffers if `validate`, drawing the rays [ray_begin, ray_end) clamped to its rays
int begin_frame(cvx_ctx* ctx, const cvx_frame_setup* setup, int slot, bool validate, int ray_begin, int ray_end, cvxd_frame& f) {
    int r = check_ready(ctx, setup);
    if (r) return r;
    make_frame(ctx, setup, slot, f);
    if (validate && (r = validate_setup(ctx, setup))) return r;
    clamp_range(ray_begin, ray_end, f.total_rays);
    f.ray_begin = ray_begin; f.ray_end = ray_end;
    return CVX_OK;
}

// Event k of a view on `stream` (0: before Phase 1, 1: between the phases, 2: after Phase 2): cvx_last_draw_ms's events if `timed`,
// and the view's cvx_profile_begin events while there is room for them
cudaError_t mark_phase(cvx_ctx* ctx, int k, cudaStream_t stream, bool timed) {
    cudaError_t e = cudaSuccess;
    if (timed) e = cudaEventRecord(k == 0 ? ctx->evStart : k == 1 ? ctx->evMid : ctx->evEnd, stream);
    if (e == cudaSuccess && timed && k == 2) ctx->timed = true;
    const bool prof = ctx->profCount < ctx->profCapacity;
    if (e == cudaSuccess && prof) e = cudaEventRecord(ctx->profEvents[3 * (size_t)ctx->profCount + k], stream);
    if (e == cudaSuccess && prof && k == 2) ctx->profCount++;
    return e;
}

uint32_t* current_target(cvx_ctx* ctx) { return ctx->externalFrame ? ctx->externalFrame : ctx->slots[ctx->lastSlot].frame; }

// An asynchronous batch leaves its device->host copies unjoined (that is its point); its last view's frame lives in a slot's own
// framebuffer until copied. Whatever else is about to WRITE a slot framebuffer first orders the context's stream behind those copies.
cudaError_t settle_async(cvx_ctx* ctx) {
    if (ctx->batchSettled == ctx->batchSeq) return cudaSuccess;
    ctx->batchSettled = ctx->batchSeq;
    return cudaStreamWaitEvent(ctx->stream, ctx->batchDone[(ctx->batchSeq - 1) % 4], 0);
}


// ---- frame ring: device-side flow control between ranks (no host barrier, no collective on the data path) ------------------
#define CVX_RING_MAX_RANKS 64
#define CVX_RING_TIMEOUT_NS 4000000000ll /* a peer that never signals must not hang the GPU: give up after 4 s and flag an error */
struct ring_flags {
    uint32_t arrive[CVX_RING_MAX_RANKS];  // arrive[r] = view index + 1 of the last view rank r finished storing into this slot
    uint32_t released;                    // view index + 1 of the last view the root has consumed from this slot
    uint32_t error;                       // set by a wait that timed out
    uint32_t pad[62];
};
__device__ __forceinline__ uint32_t ring_load(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// thread i waits until flags[i] >= value
__global__ void ring_wait_kernel(const uint32_t* flags, int n, uint32_t value, uint32_t* error) {
    const int i = threadIdx.x;
    if (i >= n) return;
    long long t0;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t0));
    while ((int32_t)(ring_load(flags + i) - value) < 0) {
        if (ring_load(error)) break;              // another wait of this ring has already given up: do not queue up more timeouts
        __nanosleep(256);
        long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        if (t - t0 > CVX_RING_TIMEOUT_NS) { atomicExch(error, 1u); break; }
    }
    __threadfence_system();
}
// everything this stream stored before (this rank's pixels of the view, through the peer mapping) is visible before the flag
__global__ void ring_signal_kernel(uint32_t* flag, uint32_t value) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" :: "l"(flag), "r"(value) : "memory");
}
uint32_t* ring_frame(cvx_ctx* ctx, int slot) { return (uint32_t*)(ctx->ring + (size_t)slot * ctx->ringFrameBytes); }
ring_flags* ring_flag_block(cvx_ctx* ctx, int slot) { return (ring_flags*)(ctx->ring + (size_t)ctx->ringSlots * ctx->ringFrameBytes) + slot; }

void free_slot(cvx_slot& sl) {
    if (sl.stream) cudaStreamSynchronize(sl.stream);
    cudaFree(sl.td); cudaFree(sl.lr); cudaFree(sl.frame);
    sl.td = sl.lr = sl.frame = nullptr;
}

// zero-initialised raybuffers and framebuffer of the current resolution for slot s; nothing stays allocated if this fails
cudaError_t alloc_slot(cvx_ctx* ctx, int s) {
    cvx_slot& sl = ctx->slots[s];
    const cudaStream_t stream = slot_stream(ctx, s);
    const size_t tdBytes = (size_t)raybuffer_pixels(ctx, 0) * 4, lrBytes = (size_t)raybuffer_pixels(ctx, 1) * 4;
    const size_t fbBytes = (size_t)ctx->width * ctx->height * 4;
    cudaError_t e = cudaMalloc(&sl.td, tdBytes);
    if (e == cudaSuccess) e = cudaMalloc(&sl.lr, lrBytes);
    if (e == cudaSuccess) e = cudaMalloc(&sl.frame, fbBytes);
    if (e == cudaSuccess) e = cudaMemsetAsync(sl.td, 0, tdBytes, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(sl.lr, 0, lrBytes, stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(sl.frame, 0, fbBytes, stream);
    if (e != cudaSuccess) free_slot(sl);
    return e;
}

// `want` pool framebuffers of the current resolution (events are created once per context)
int ensure_pool(cvx_ctx* ctx, int want) {
    if (want > CVX_POOL_FRAMES) want = CVX_POOL_FRAMES;
    const size_t fbBytes = (size_t)ctx->width * ctx->height * 4;
    while (ctx->poolCount < want) {
        const int i = ctx->poolCount;
        cudaError_t e = cudaSuccess;
        if (!ctx->poolReady[i]) e = cudaEventCreateWithFlags(&ctx->poolReady[i], cudaEventDisableTiming);
        if (e == cudaSuccess && !ctx->poolFree[i]) e = cudaEventCreateWithFlags(&ctx->poolFree[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaMalloc(&ctx->pool[i], fbBytes);
        if (e != cudaSuccess) { ctx->pool[i] = nullptr; return fail(ctx, cvx_code(e), "frame pool allocation failed: %s", cudaGetErrorString(e)); }
        ctx->poolCount++;
    }
    return CVX_OK;
}

// slots 1 .. want-1 get a stream, an event and their buffers (slot 0 has its buffers from cvx_set_resolution)
int ensure_slots(cvx_ctx* ctx, int want) {
    if (want > ctx->slotCount) want = ctx->slotCount;
    while (ctx->slotsReady < want) {
        cvx_slot& sl = ctx->slots[ctx->slotsReady];
        cudaError_t e = cudaSuccess;
        if (!sl.stream) e = cudaStreamCreateWithFlags(&sl.stream, cudaStreamNonBlocking);
        if (e == cudaSuccess && !sl.done) e = cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming);
        if (e == cudaSuccess) e = alloc_slot(ctx, ctx->slotsReady);
        if (e != cudaSuccess) return fail(ctx, cvx_code(e), "frame slot allocation failed: %s", cudaGetErrorString(e));
        ctx->slotsReady++;
    }
    return CVX_OK;
}

// everything sized by the resolution: the slots' buffers, the frame pool and the present staging frame
void free_resolution(cvx_ctx* ctx) {
    if (ctx->copyStream) cudaStreamSynchronize(ctx->copyStream);
    for (cvx_slot& sl : ctx->slots) free_slot(sl);
    ctx->slotsReady = 0;
    ctx->lastSlot = 0;
    for (int i = 0; i < CVX_POOL_FRAMES; i++) { cudaFree(ctx->pool[i]); ctx->pool[i] = nullptr; ctx->poolUsed[i] = false; }
    ctx->poolCount = 0;
    cudaFree(ctx->presentStage); ctx->presentStage = nullptr;
    ctx->width = ctx->height = 0;
}

void free_world(cvx_ctx* ctx) {
    for (cvx_lod_memory& m : ctx->lod) {
        cudaFree(m.headers); cudaFree(m.blob); cudaFree(m.bounds);
        m = cvx_lod_memory();
    }
    memset(&ctx->world, 0, sizeof ctx->world);
}

void free_ray_scratch(cvx_ctx* ctx) {
    cudaFree(ctx->rayScratch);
    ctx->rayScratch = nullptr;
    ctx->rayScratchBytes = 0;
}

// Takes ownership of `dblob` (a whole LOD blob in device memory: column_count 12-byte headers + element area), builds the Phase-1
// tables from it on the device (world_builder_gpu.cu: the same tables world_transcode.h builds on the host for the emulator; it
// also validates what the kernels index with) and makes it LOD `lod` of the context's world.
int install_lod(cvx_ctx* ctx, int lod, int dim_x, int dim_y, int dim_z, void* dblob, int64_t bytes, int column_count) {
    const int64_t needCols = (int64_t)(dim_x >> lod) * (dim_z >> lod);
    const int64_t headerBytes = 12 * (int64_t)column_count;
    const int64_t elementCells = (bytes - headerBytes) / 4;
    void* headers = nullptr; void* bounds = nullptr; int regular = 0; long long bad = -1;
    std::string err;
    int r = cvxd_transcode_lod_device(ctx->stream, dblob, needCols, column_count, elementCells, lod, dim_y, &headers, &bounds, &regular, &bad, &ctx->launches, err);
    if (r) {
        cudaFree(dblob);
        if (r == CVX_ERR_FORMAT) return fail(ctx, CVX_ERR_FORMAT, "column %lld of LOD %d points outside the element area (element offset, run count or a run's colour range)", bad, lod);
        return fail(ctx, r, "world upload failed: %s", err.c_str());
    }
    cudaStreamSynchronize(ctx->stream);
    cvx_lod_memory& m = ctx->lod[lod];
    cudaFree(m.headers); cudaFree(m.blob); cudaFree(m.bounds);
    m.blob = dblob; m.headers = headers; m.bounds = bounds; m.regular = regular != 0;
    cvxd_world_set_dims(&ctx->world, dim_x, dim_y, dim_z);
    cvxd_lod& l = ctx->world.lods[lod];
    l.headers = (const uint4*)headers;
    l.elements = (const uint32_t*)((const uint8_t*)dblob + headerBytes); // the reference element area, verbatim
    l.bounds = (const uint2*)bounds;
    l.mul_x = dim_z >> lod;
    l.lod = lod;
    ctx->world.regular = 1;
    for (const cvx_lod_memory& mi : ctx->lod) if (mi.headers && !mi.regular) ctx->world.regular = 0;
    if (lod + 1 > ctx->world.lod_count) ctx->world.lod_count = lod + 1;
    return CVX_OK;
}

} // namespace

extern "C" {

int cvx_create(const cvx_config* config, cvx_ctx** out_ctx) {
    if (!out_ctx) return fail(nullptr, CVX_ERR_INVALID_ARGUMENT, "out_ctx is NULL");
    *out_ctx = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count <= 0)
        return fail(nullptr, CVX_ERR_NO_DEVICE, "no CUDA device (%s); libcpuvox_b200 has no CPU fallback", e != cudaSuccess ? cudaGetErrorString(e) : "count = 0");
    int dev = config ? config->device : 0;
    if (dev < 0 || dev >= count) return fail(nullptr, CVX_ERR_INVALID_ARGUMENT, "device %d out of range (%d devices)", dev, count);
    cvx_ctx* ctx = new (std::nothrow) cvx_ctx();
    if (!ctx) return fail(nullptr, CVX_ERR_OUT_OF_MEMORY, "out of host memory");
    ctx->device = dev;
    ctx->flags = config ? config->flags : 0;
    memset(&ctx->world, 0, sizeof ctx->world);
    // without a context to hold it, a failure's message goes where cvx_last_error(NULL) finds it; the partial context is torn down
    auto init = [ctx, dev]() -> int {
        CU(nullptr, cudaSetDevice(dev));
        CU(nullptr, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        CU(nullptr, cudaStreamCreateWithFlags(&ctx->copyStream, cudaStreamNonBlocking));
        CU(nullptr, cudaEventCreate(&ctx->evStart));
        CU(nullptr, cudaEventCreate(&ctx->evMid));
        CU(nullptr, cudaEventCreate(&ctx->evEnd));
        CU(nullptr, cudaEventCreateWithFlags(&ctx->evBatchStart, cudaEventDisableTiming));
        CU(nullptr, cudaEventCreateWithFlags(&ctx->evFrameDone, cudaEventDisableTiming));
        CU(nullptr, cudaEventCreateWithFlags(&ctx->evCopyDone, cudaEventDisableTiming));
        CU(nullptr, cudaMalloc(&ctx->counters, sizeof(cvxd_counters)));
        CU(nullptr, cudaMemset(ctx->counters, 0, sizeof(cvxd_counters)));
        return CVX_OK;
    };
    if (int r = init()) { cvx_destroy(ctx); return r; }
    *out_ctx = ctx;
    return CVX_OK;
}

int cvx_destroy(cvx_ctx* ctx) {
    if (!ctx) return CVX_OK;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->copyStream) cudaStreamSynchronize(ctx->copyStream);
    cvx_ring_close(ctx);
    free_resolution(ctx);
    free_world(ctx);
    free_ray_scratch(ctx);
    for (cudaEvent_t e : ctx->profEvents) cudaEventDestroy(e);
    cvxjpeg::destroy(ctx->jpeg);
    cudaFree(ctx->counters);
    for (cudaEvent_t e : {ctx->evStart, ctx->evMid, ctx->evEnd, ctx->evBatchStart, ctx->evFrameDone, ctx->evCopyDone})
        if (e) cudaEventDestroy(e);
    for (cvx_slot& sl : ctx->slots) {
        if (sl.done) cudaEventDestroy(sl.done);
        if (sl.stream) cudaStreamDestroy(sl.stream);
    }
    for (int i = 0; i < 4; i++) if (ctx->batchDone[i]) cudaEventDestroy(ctx->batchDone[i]);
    for (int i = 0; i < CVX_POOL_FRAMES; i++) {
        if (ctx->poolReady[i]) cudaEventDestroy(ctx->poolReady[i]);
        if (ctx->poolFree[i]) cudaEventDestroy(ctx->poolFree[i]);
    }
    if (ctx->ownStream && ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->copyStream) cudaStreamDestroy(ctx->copyStream);
    delete ctx;
    return CVX_OK;
}

const char* cvx_last_error(const cvx_ctx* ctx) { return ctx ? ctx->error.c_str() : g_createError.c_str(); }

int cvx_set_stream(cvx_ctx* ctx, void* cuda_stream) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->ownStream) cudaStreamDestroy(ctx->stream);
    if (cuda_stream) { ctx->stream = (cudaStream_t)cuda_stream; ctx->ownStream = false; }
    else { CU(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)); ctx->ownStream = true; }
    return CVX_OK;
}

int cvx_world_upload(cvx_ctx* ctx, int32_t lod, int32_t dim_x, int32_t dim_y, int32_t dim_z, const void* blob, int64_t bytes, int32_t column_count) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (lod < 0 || lod >= CVX_LOD_LEVELS || !blob) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "bad lod %d or NULL blob", lod);
    if (!pow2(dim_x) || !pow2(dim_z) || dim_y < 1 || dim_y > 32768) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "world dimensions %dx%dx%d: x/z must be powers of two, y <= 32768", dim_x, dim_y, dim_z);
    const int64_t needCols = (int64_t)(dim_x >> lod) * (dim_z >> lod);
    if (needCols < 1 || column_count < needCols) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "column_count %d too small for LOD %d (%lld columns addressed)", column_count, lod, (long long)needCols);
    const int64_t headerBytes = 12 * (int64_t)column_count;
    if (bytes < headerBytes || ((bytes - headerBytes) & 3)) return fail(ctx, CVX_ERR_FORMAT, "blob of %lld bytes cannot hold %d column headers", (long long)bytes, column_count);
    if (ctx->world.lod_count > 0 && (ctx->world.dim_x != dim_x || ctx->world.dim_y != dim_y || ctx->world.dim_z != dim_z))
        return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "LOD %d dimensions differ from the already uploaded world; call cvx_world_free first", lod);
    // the raw blob goes to the device as it is (host or device source: unified addressing) and is transcoded there
    CU(ctx, cudaSetDevice(ctx->device));
    void* dblob = nullptr;
    cudaError_t e = cudaMalloc(&dblob, (size_t)(bytes > 0 ? bytes : 4));
    if (e == cudaSuccess) e = cudaMemcpyAsync(dblob, blob, (size_t)bytes, cudaMemcpyDefault, ctx->stream);
    if (e != cudaSuccess) { cudaFree(dblob); return fail(ctx, cvx_code(e), "world upload failed: %s", cudaGetErrorString(e)); }
    return install_lod(ctx, lod, dim_x, dim_y, dim_z, dblob, bytes, column_count);
}

int cvx_world_free(cvx_ctx* ctx) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    free_world(ctx);
    free_ray_scratch(ctx);
    return CVX_OK;
}

int cvx_set_resolution(cvx_ctx* ctx, int32_t width, int32_t height) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (width < 1 || height < 1 || width > CVXD_MAX_AXIS || height > CVXD_MAX_AXIS)
        return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "resolution %dx%d out of range (1..%d)", width, height, CVXD_MAX_AXIS);
    if (width == ctx->width && height == ctx->height) return CVX_OK;
    CVX_RANGE("Resize textures");            // RenderManager.cs:97
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->copyStream));
    cvx_ring_close(ctx);  // its frames have the old size
    free_resolution(ctx);
    ctx->width = width; ctx->height = height;
    cudaError_t e = alloc_slot(ctx, 0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        free_resolution(ctx);
        return fail(ctx, cvx_code(e), "raybuffer allocation failed: %s", cudaGetErrorString(e));
    }
    ctx->slotsReady = 1;
    return CVX_OK;
}

int cvx_draw_rays(cvx_ctx* ctx, const cvx_frame_setup* setup, int32_t ray_begin, int32_t ray_end) {
    cvxd_frame f;
    int r = begin_frame(ctx, setup, 0, true, ray_begin, ray_end, f);
    if (r) return r;
    ctx->lastSlot = 0;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaEventRecord(ctx->evStart, ctx->stream));
    CU(ctx, cvxd_launch_phase1(ctx->world, f, ctx->groupSize, ctx->stream));
    if (f.ray_end > f.ray_begin) ctx->launches++;
    CU(ctx, cudaEventRecord(ctx->evMid, ctx->stream));
    CU(ctx, cudaEventRecord(ctx->evEnd, ctx->stream));
    ctx->timed = true;
    return CVX_OK;
}

int cvx_blit_rows(cvx_ctx* ctx, const cvx_frame_setup* setup, int32_t row_begin, int32_t row_end) {
    cvxd_frame f;
    int r = begin_frame(ctx, setup, 0, false, 0, -1, f);
    if (r) return r;
    cvxd_blit b;
    make_blit(f, current_target(ctx), b);
    clamp_range(row_begin, row_end, ctx->height);
    b.row_begin = row_begin; b.row_end = row_end;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, settle_async(ctx));
    CU(ctx, cvxd_launch_phase2(b, ctx->stream));
    if (row_end > row_begin) ctx->launches++;
    return CVX_OK;
}

int cvx_blit_owned(cvx_ctx* ctx, const cvx_frame_setup* setup, int32_t ray_begin, int32_t ray_end, void* device_frame) {
    cvxd_frame f;
    int r = begin_frame(ctx, setup, 0, false, ray_begin, ray_end, f);
    if (r) return r;
    cvxd_blit b;
    make_blit(f, device_frame ? (uint32_t*)device_frame : current_target(ctx), b);
    b.owned_only = 1;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, settle_async(ctx));
    CU(ctx, cvxd_launch_phase2(b, ctx->stream));
    ctx->launches++;
    return CVX_OK;
}

static int draw_into(cvx_ctx* ctx, const cvx_frame_setup* setup, int slot, uint32_t* target, bool timed) {
    cvxd_frame f;
    int r;
    {
        CVX_RANGE("Segment setup overhead"); // RenderManager.cs:277: the SegmentContext fill
        r = begin_frame(ctx, setup, slot, true, 0, -1, f);
    }
    if (r) return r;
    cvxd_blit b;
    make_blit(f, target, b);
    cudaStream_t stream = slot_stream(ctx, slot);
    CU(ctx, mark_phase(ctx, 0, stream, timed));
    {
        CVX_RANGE("Draw planes");            // RenderManager.cs:154
        CU(ctx, cvxd_launch_phase1(ctx->world, f, ctx->groupSize, stream));
    }
    if (f.total_rays > 0) ctx->launches++;
    CU(ctx, mark_phase(ctx, 1, stream, timed));
    {
        CVX_RANGE("Blit raybuffer");         // RenderManager.cs:178
        CU(ctx, cvxd_launch_phase2(b, stream));
    }
    ctx->launches++;
    CU(ctx, mark_phase(ctx, 2, stream, timed));
    ctx->lastSlot = slot;
    return CVX_OK;
}

int cvx_draw(cvx_ctx* ctx, const cvx_frame_setup* setup) {
    int r = check_ready(ctx, setup);
    if (r) return r;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, settle_async(ctx));
    ctx->lastSlot = 0;
    return draw_into(ctx, setup, 0, current_target(ctx), true);
}

// out_batch == NULL: cvx_draw_batch (with dst_frames the call returns when the frames are on the host); else cvx_draw_batch_async
static int draw_batch_impl(cvx_ctx* ctx, const cvx_frame_setup* setups, int32_t n_views, void* dst_frames, int64_t* out_batch) {
    int r = check_ready(ctx, setups);
    if (r) return r;
    if (n_views < 0) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "n_views < 0");
    const bool async = out_batch != nullptr;
    if (async && (!dst_frames || n_views < 2 || ctx->externalFrame)) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "an asynchronous batch needs a host destination, at least two views and no external frame");
    if (n_views == 0) return CVX_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t fbBytes = (size_t)ctx->width * ctx->height * 4;
    // View i renders on slot i % K: Phase 1 and Phase 2 are stream-ordered inside the slot and the K slots overlap each other — the
    // long tail of one view's few heavy rays runs beside the bulk of the next views. With dst_frames, Phase 2 writes into a pool of
    // framebuffers which the copy stream drains in view order: the slot goes on to its next view at once, and the device->host
    // copies (0.6 ms per 4K frame, most of the copy engine's time at the rate the kernels deliver) never hold a slot back. The last
    // view renders into its slot's own framebuffer, so the read functions and device pointers refer to it after the call.
    // A caller-owned external frame forces one slot (one target buffer).
    const int K = ctx->externalFrame ? 1 : (ctx->slotCount < n_views ? ctx->slotCount : n_views);
    for (int i = 0; i < n_views; i++)  // every view is checked before the first one is enqueued
        if ((r = validate_setup(ctx, setups + i))) return r;
    if ((r = ensure_slots(ctx, K))) return r;
    const bool pooled = dst_frames && !ctx->externalFrame && n_views > 1;
    const int M = CVX_POOL_FRAMES < n_views - 1 ? CVX_POOL_FRAMES : n_views - 1;
    if (pooled && (r = ensure_pool(ctx, M))) return r;
    if (!pooled) CU(ctx, settle_async(ctx));   // this batch writes the slots' own framebuffers
    CU(ctx, cudaEventRecord(ctx->evBatchStart, ctx->stream)); // the slots start after everything queued on the context's stream
    for (int s = 1; s < K; s++) CU(ctx, cudaStreamWaitEvent(slot_stream(ctx, s), ctx->evBatchStart, 0));
    cudaError_t ce = cudaSuccess;
    for (int i = 0; i < n_views && !r && ce == cudaSuccess; i++) {
        const int slot = i % K;
        cudaStream_t st = slot_stream(ctx, slot);
        if (pooled) {
            const bool last = i == n_views - 1;
            const int pf = i % M;
            uint32_t* target = last ? ctx->slots[slot].frame : ctx->pool[pf];
            // the previous user of the buffer (view i - M, or a view of an earlier asynchronous batch) has been copied out; the last view's
            // own framebuffer may still be read by the previous asynchronous batch's final copy
            if (!last && ctx->poolUsed[pf]) ce = cudaStreamWaitEvent(st, ctx->poolFree[pf], 0);
            if (last && ctx->batchSeq > 0) ce = cudaStreamWaitEvent(st, ctx->batchDone[(ctx->batchSeq - 1) % 4], 0);
            if (ce == cudaSuccess) r = draw_into(ctx, setups + i, slot, target, false);
            if (r || ce != cudaSuccess) break;
            cudaEvent_t ready = last ? ctx->evFrameDone : ctx->poolReady[pf];
            ce = cudaEventRecord(ready, st);
            if (ce == cudaSuccess) ce = cudaStreamWaitEvent(ctx->copyStream, ready, 0);
            // the copy is asynchronous only if dst_frames is page-locked (cvx_alloc_pinned / cudaHostRegister)
            if (ce == cudaSuccess) ce = cudaMemcpyAsync((uint8_t*)dst_frames + (size_t)i * fbBytes, target, fbBytes, cudaMemcpyDeviceToHost, ctx->copyStream);
            if (ce == cudaSuccess && !last) { ce = cudaEventRecord(ctx->poolFree[pf], ctx->copyStream); ctx->poolUsed[pf] = true; }
            continue;
        }
        uint32_t* target = ctx->externalFrame ? ctx->externalFrame : ctx->slots[slot].frame;
        r = draw_into(ctx, setups + i, slot, target, false);
        if (!r && dst_frames) ce = cudaMemcpyAsync((uint8_t*)dst_frames + (size_t)i * fbBytes, target, fbBytes, cudaMemcpyDeviceToHost, st);
    }
    if (pooled && async) {   // the copies of this batch are followed by its completion event; nothing waits for them here
        if (!ctx->batchDone[ctx->batchSeq % 4]) {
            cudaError_t e0 = cudaEventCreateWithFlags(&ctx->batchDone[ctx->batchSeq % 4], cudaEventDisableTiming);
            if (ce == cudaSuccess) ce = e0;
        }
        if (ce == cudaSuccess) ce = cudaEventRecord(ctx->batchDone[ctx->batchSeq % 4], ctx->copyStream);
    } else if (pooled) {     // the context's stream also waits for the copies
        cudaError_t e1 = cudaEventRecord(ctx->evCopyDone, ctx->copyStream);
        if (e1 == cudaSuccess) e1 = cudaStreamWaitEvent(ctx->stream, ctx->evCopyDone, 0);
        if (ce == cudaSuccess) ce = e1;
    }
    // join — also after a failure in the middle of the batch, so that the slots' work stays ordered before whatever the caller
    // queues next on the context's stream (events, reads, the next batch)
    for (int s = 1; s < K; s++) {
        cudaError_t e1 = cudaEventRecord(ctx->slots[s].done, ctx->slots[s].stream);
        if (e1 == cudaSuccess) e1 = cudaStreamWaitEvent(ctx->stream, ctx->slots[s].done, 0);
        if (ce == cudaSuccess) ce = e1;
    }
    if (r) return r;
    CU(ctx, ce);
    if (async) { *out_batch = ctx->batchSeq++; return CVX_OK; }
    if (dst_frames) CU(ctx, cudaStreamSynchronize(ctx->stream)); // frames are on the host when the call returns
    return CVX_OK;
}

int cvx_draw_batch(cvx_ctx* ctx, const cvx_frame_setup* setups, int32_t n_views, void* dst_frames) {
    return draw_batch_impl(ctx, setups, n_views, dst_frames, nullptr);
}

// The kernels of consecutive asynchronous batches follow each other on the same buffer sets while the copy stream is still delivering
// the earlier batch's frames: the copy backlog at the end of a batch (the views of a batch can finish several times faster than one
// copy engine drains them) overlaps the next batch's rendering instead of idling the GPU.
int cvx_draw_batch_async(cvx_ctx* ctx, const cvx_frame_setup* setups, int32_t n_views, void* dst_frames, int64_t* out_batch) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (!out_batch) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "out_batch is NULL");
    return draw_batch_impl(ctx, setups, n_views, dst_frames, out_batch);
}

int cvx_batch_wait(cvx_ctx* ctx, int64_t batch) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (batch < 0 || batch >= ctx->batchSeq) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "no such batch (%lld)", (long long)batch);
    CU(ctx, cudaSetDevice(ctx->device));
    // the events of older batches have been re-recorded behind newer ones on the same in-order copy stream: waiting for those covers them
    CU(ctx, cudaEventSynchronize(ctx->batchDone[batch % 4]));
    return CVX_OK;
}

// RenderManager.DrawWorld for headless hosts (RenderManager.cs:111-194 with UnityManager.LateUpdate's LimitRotationHorizon, UnityManager.cs:181):
// the per-frame host part (vanishing point, segments, CameraData) is computed here from each pose, then the views go through
// cvx_draw_batch. One call per batch: no per-view crossing of the FFI boundary.
static int world_batch_impl(cvx_ctx* ctx, const cvx_pose* poses, int32_t n_views, const float lod_distances[CVX_LOD_LEVELS],
                            int32_t limit_rotation_horizon, void* dst_frames, int64_t* out_batch) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (!poses || n_views < 1 || !lod_distances) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "bad pose batch");
    if (ctx->world.lod_count <= 0) return fail(ctx, CVX_ERR_NO_WORLD, "no world uploaded");
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    std::vector<cvx_frame_setup> setups((size_t)n_views);
    for (int i = 0; i < n_views; i++) {
        cvx_pose p = poses[i];
        p.pixel_width = ctx->width; p.pixel_height = ctx->height;   // fakeCamera.pixelRect = (0, 0, resX, resY), UnityManager.cs:180
        if (limit_rotation_horizon) cvx_host_limit_rotation_horizon(&p);
        int r = cvx_host_frame_setup(&p, lod_distances, ctx->world.dim_y, &setups[(size_t)i]);
        if (r) return fail(ctx, r, "frame setup of view %d failed", i);
    }
    return draw_batch_impl(ctx, setups.data(), n_views, dst_frames, out_batch);   // kernel parameters are copied at launch: setups may go
}

int cvx_draw_world_batch(cvx_ctx* ctx, const cvx_pose* poses, int32_t n_views, const float lod_distances[CVX_LOD_LEVELS],
                         int32_t limit_rotation_horizon, void* dst_frames) {
    return world_batch_impl(ctx, poses, n_views, lod_distances, limit_rotation_horizon, dst_frames, nullptr);
}

int cvx_draw_world_batch_async(cvx_ctx* ctx, const cvx_pose* poses, int32_t n_views, const float lod_distances[CVX_LOD_LEVELS],
                               int32_t limit_rotation_horizon, void* dst_frames, int64_t* out_batch) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (!out_batch) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "out_batch is NULL");
    return world_batch_impl(ctx, poses, n_views, lod_distances, limit_rotation_horizon, dst_frames, out_batch);
}

int cvx_sync(cvx_ctx* ctx) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->copyStream));
    if (ctx->ring)  // sharded views run on the slot streams without a join into the context's stream
        for (const cvx_slot& sl : ctx->slots) if (sl.stream) CU(ctx, cudaStreamSynchronize(sl.stream));
    return CVX_OK;
}

// Debug views: RayBufferBlit.shader COPY_MAIN1 / COPY_MAIN2 (:48-53), selected by UnityManager.ERenderMode.RayBufferTopDown /
// RayBufferLeftRight (UnityManager.cs:129-134,471-483): the whole raybuffer of the last view stretched over the screen.
int cvx_blit_raybuffer(cvx_ctx* ctx, int32_t which) {
    if (!ctx || which < 0 || which > 1) return ctx ? fail(ctx, CVX_ERR_INVALID_ARGUMENT, "which must be 0 (top/down) or 1 (left/right)") : CVX_ERR_INVALID_ARGUMENT;
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    const int W = ctx->width, H = ctx->height;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, settle_async(ctx));
    const uint32_t* buf = raybuffer(ctx->slots[ctx->lastSlot], which);
    CU(ctx, cvxd_launch_raybuffer_view(buf, raybuffer_rows(ctx, which), raybuffer_row_length(ctx, which), current_target(ctx), W, H, ctx->stream));
    ctx->launches++;
    return CVX_OK;
}

// Presentation (SURVEY.md §8(f) 4): the step after the path. The reference ends in Unity's camera target; here the device frame is
// converted to what a graphics API / video encoder takes (RGBA8 or BGRA8, top-down or bottom-up rows) on the device, and either
// stays there (dst_is_device: a mapped graphics resource, an encoder input surface, a peer buffer) or is copied to the host.
int cvx_present(cvx_ctx* ctx, int32_t format, int32_t top_down, void* dst, int32_t dst_is_device) {
    if (!ctx || !dst) return ctx ? fail(ctx, CVX_ERR_INVALID_ARGUMENT, "dst is NULL") : CVX_ERR_INVALID_ARGUMENT;
    if (format != CVX_PRESENT_RGBA8 && format != CVX_PRESENT_BGRA8 && format != CVX_PRESENT_RGB8) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "unknown present format %d", format);
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    const int W = ctx->width, H = ctx->height;
    const size_t fbBytes = (size_t)W * H * 4, outBytes = (size_t)W * H * (format == CVX_PRESENT_RGB8 ? 3 : 4);
    CU(ctx, cudaSetDevice(ctx->device));
    uint32_t* out = (uint32_t*)dst;
    if (!dst_is_device) {
        if (!ctx->presentStage) {
            cudaError_t e = cudaMalloc(&ctx->presentStage, fbBytes);
            if (e != cudaSuccess) return fail(ctx, cvx_code(e), "present staging allocation failed: %s", cudaGetErrorString(e));
        }
        out = ctx->presentStage;
    }
    if (format == CVX_PRESENT_RGB8) CU(ctx, cvxd_launch_present_rgb8(current_target(ctx), (uint8_t*)out, W, H, top_down != 0, ctx->stream));
    else CU(ctx, cvxd_launch_present(current_target(ctx), out, W, H, format == CVX_PRESENT_BGRA8, top_down != 0, ctx->stream));
    ctx->launches++;
    if (!dst_is_device) {
        CU(ctx, cudaMemcpyAsync(dst, out, outBytes, cudaMemcpyDeviceToHost, ctx->stream));
        CU(ctx, cudaStreamSynchronize(ctx->stream));
    }
    return CVX_OK;
}

// Presentation as a compressed still: the frame is packed to top-down R,G,B bytes by present_rgb8_kernel and encoded on the device by
// nvJPEG's CUDA encoder (jpeg_encoder.cpp; the toolkit library is loaded on first use); only the bitstream crosses to the host.
int cvx_present_jpeg(cvx_ctx* ctx, int32_t quality, int32_t subsampling, void* dst, int64_t dst_capacity, int64_t* out_bytes) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (!out_bytes) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "out_bytes is NULL");
    *out_bytes = 0;
    if (quality < 1 || quality > 100) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "JPEG quality %d: expected 1..100", quality);
    if (subsampling != CVX_JPEG_444 && subsampling != CVX_JPEG_420) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "unknown chroma subsampling %d", subsampling);
    if (dst_capacity < 0 || (dst_capacity > 0 && !dst)) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "bad destination buffer");
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    const int W = ctx->width, H = ctx->height;
    CU(ctx, cudaSetDevice(ctx->device));
    if (!ctx->jpeg) {
        std::string err;
        ctx->jpeg = cvxjpeg::create(err);
        if (!ctx->jpeg) return fail(ctx, CVX_ERR_UNSUPPORTED, "%s", err.c_str());
    }
    if (!ctx->presentStage) {
        cudaError_t e = cudaMalloc(&ctx->presentStage, (size_t)W * H * 4);
        if (e != cudaSuccess) return fail(ctx, cvx_code(e), "present staging allocation failed: %s", cudaGetErrorString(e));
    }
    CU(ctx, cvxd_launch_present_rgb8(current_target(ctx), (uint8_t*)ctx->presentStage, W, H, 1, ctx->stream));
    ctx->launches++;
    std::string err;
    if (!cvxjpeg::encode(ctx->jpeg, (const uint8_t*)ctx->presentStage, W, H, quality, subsampling, ctx->stream, ctx->jpegOut, err))
        return fail(ctx, CVX_ERR_CUDA, "%s", err.c_str());
    *out_bytes = (int64_t)ctx->jpegOut.size();
    if (dst_capacity == 0) return CVX_OK; // size query: the caller allocates and calls again
    if ((int64_t)ctx->jpegOut.size() > dst_capacity)
        return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "JPEG bitstream is %lld bytes, the destination holds %lld", (long long)ctx->jpegOut.size(), (long long)dst_capacity);
    memcpy(dst, ctx->jpegOut.data(), ctx->jpegOut.size());
    return CVX_OK;
}

// World production on the device (world_builder_gpu.cu): same inputs and the same blobs, byte for byte, as cvx_builder_from_mesh +
// cvx_builder_lod(0 .. n_lods-1), i.e. WorldBuilder.Import -> ToLOD0World -> World.DownSample (UnityManager.cs:297-331).
int cvx_gpu_builder_from_mesh(cvx_ctx* ctx, const float* positions, const uint8_t* colors32, int32_t n_vertices, int32_t max_dimension,
                              const int32_t flips[3], int32_t n_lods, cvx_world_builder** out) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (!positions || !colors32 || n_vertices < 3 || max_dimension < 1 || n_lods < 1 || n_lods > CVX_LOD_LEVELS || !out)
        return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "bad mesh arguments");
    *out = nullptr;
    std::vector<float> xyz;
    int dims[3];
    int r = cvxh_remap_mesh(positions, n_vertices, max_dimension, flips, xyz, dims);
    if (r) return fail(ctx, r, "mesh cannot be remapped to max dimension %d", max_dimension);
    cvx_world_builder* b = new (std::nothrow) cvx_world_builder();
    if (!b) return fail(ctx, CVX_ERR_OUT_OF_MEMORY, "out of host memory");
    b->dims[0] = dims[0]; b->dims[1] = dims[1]; b->dims[2] = dims[2];
    b->deviceBuilt = true;
    std::string err;
    r = cvxd_build_world_gpu(ctx->device, ctx->stream, xyz.data(), colors32, n_vertices, n_lods, b, nullptr, &ctx->launches, err);
    if (r) { cvx_builder_free(b); return fail(ctx, r, "device world build failed: %s", err.c_str()); }
    *out = b;
    return CVX_OK;
}

// Mesh -> resident world without leaving the device: the LOD blobs produced by the device builder are transcoded in place and become
// the context's world (as if cvx_world_free + cvx_world_upload had been called with them). Nothing is copied to the host.
int cvx_world_build_from_mesh(cvx_ctx* ctx, const float* positions, const uint8_t* colors32, int32_t n_vertices, int32_t max_dimension,
                              const int32_t flips[3], int32_t n_lods, int32_t out_dims[3], int64_t out_voxel_counts[CVX_LOD_LEVELS]) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (!positions || !colors32 || n_vertices < 3 || max_dimension < 1 || n_lods < 1 || n_lods > CVX_LOD_LEVELS)
        return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "bad mesh arguments");
    std::vector<float> xyz;
    int dims[3];
    int r = cvxh_remap_mesh(positions, n_vertices, max_dimension, flips, xyz, dims);
    if (r) return fail(ctx, r, "mesh cannot be remapped to max dimension %d", max_dimension);
    if (!pow2(dims[0]) || !pow2(dims[2])) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "world dimensions %dx%dx%d: x/z must be powers of two", dims[0], dims[1], dims[2]);
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    free_world(ctx);
    cvx_world_builder b;
    b.dims[0] = dims[0]; b.dims[1] = dims[1]; b.dims[2] = dims[2];
    b.deviceBuilt = true;
    cvxd_lod_sink sink = [&](int lod, void* dblob, int64_t bytes, int columnCount) {
        return install_lod(ctx, lod, dims[0], dims[1], dims[2], dblob, bytes, columnCount);
    };
    std::string err;
    r = cvxd_build_world_gpu(ctx->device, ctx->stream, xyz.data(), colors32, n_vertices, n_lods, &b, &sink, &ctx->launches, err);
    if (r) { free_world(ctx); return ctx->error.empty() || r != CVX_ERR_FORMAT ? fail(ctx, r, "device world build failed: %s", err.c_str()) : r; }
    if (out_dims) { out_dims[0] = dims[0]; out_dims[1] = dims[1]; out_dims[2] = dims[2]; }
    if (out_voxel_counts) for (int i = 0; i < CVX_LOD_LEVELS; i++) out_voxel_counts[i] = i < n_lods ? b.lods[i].voxelCount : 0;
    return CVX_OK;
}

// Ray queries (raycast.h, raycast_kernels.cu): the kernel reads the world tables the context holds at the time of the call, on the
// context's stream, so it follows any draw or batch join queued there and a later world replacement (which synchronises that stream
// before freeing the old tables) cannot pull them from under it.
int cvx_raycast(cvx_ctx* ctx, const cvx_ray* rays, int32_t n, int32_t lod, cvx_ray_hit* out, int32_t on_device) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (ctx->world.lod_count <= 0) return fail(ctx, CVX_ERR_NO_WORLD, "no world uploaded");
    if (lod < 0 || lod >= CVX_LOD_LEVELS || !ctx->world.lods[lod].headers) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "LOD %d is not uploaded", lod);
    if (n < 0) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "n = %d < 0", n);
    if (n > 0 && (!rays || !out)) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "rays or hits is NULL");
    if (n == 0) return CVX_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    const bool bounds = ctx->lod[lod].regular && !ctx->generalPath;
    if (on_device) {
        CU(ctx, cvxd_launch_raycast(ctx->world, lod, (const cvxd_ray*)rays, (cvxd_ray_hit*)out, n, bounds, ctx->stream));
        ctx->launches++;
        return CVX_OK;
    }
    const size_t rayBytes = (size_t)n * sizeof(cvx_ray), need = rayBytes + (size_t)n * sizeof(cvx_ray_hit);
    if (need > ctx->rayScratchBytes) {
        CU(ctx, cudaStreamSynchronize(ctx->stream));
        free_ray_scratch(ctx);
        cudaError_t e = cudaMalloc(&ctx->rayScratch, need);
        if (e != cudaSuccess) { ctx->rayScratch = nullptr; return fail(ctx, cvx_code(e), "ray scratch allocation failed: %s", cudaGetErrorString(e)); }
        ctx->rayScratchBytes = need;
    }
    cvxd_ray* dRays = (cvxd_ray*)ctx->rayScratch;
    cvxd_ray_hit* dHits = (cvxd_ray_hit*)((uint8_t*)ctx->rayScratch + rayBytes);
    CU(ctx, cudaMemcpyAsync(dRays, rays, rayBytes, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cvxd_launch_raycast(ctx->world, lod, dRays, dHits, n, bounds, ctx->stream));
    ctx->launches++;
    CU(ctx, cudaMemcpyAsync(out, dHits, (size_t)n * sizeof(cvx_ray_hit), cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return CVX_OK;
}

int cvx_read_frame(cvx_ctx* ctx, void* dst_argb, int64_t bytes) {
    if (!ctx || !dst_argb) return CVX_ERR_INVALID_ARGUMENT;
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    const int64_t need = (int64_t)ctx->width * ctx->height * 4;
    if (bytes < need) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "destination holds %lld bytes, frame needs %lld", (long long)bytes, (long long)need);
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(dst_argb, current_target(ctx), (size_t)need, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return CVX_OK;
}

int cvx_read_raybuffer(cvx_ctx* ctx, int32_t which, void* dst_argb, int64_t bytes) {
    if (!ctx || !dst_argb || which < 0 || which > 1) return CVX_ERR_INVALID_ARGUMENT;
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    const int64_t full = raybuffer_pixels(ctx, which) * 4;
    const int64_t n = bytes < full ? bytes : full;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(dst_argb, raybuffer(ctx->slots[ctx->lastSlot], which), (size_t)n, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return CVX_OK;
}

int cvx_clear_raybuffers(cvx_ctx* ctx, uint32_t argb) { // RenderManager.ClearRayBuffer (debug), RenderManager.cs:58-92
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cvxd_launch_fill(ctx->slots[0].td, argb, raybuffer_pixels(ctx, 0), ctx->stream));
    CU(ctx, cvxd_launch_fill(ctx->slots[0].lr, argb, raybuffer_pixels(ctx, 1), ctx->stream));
    ctx->launches += 2;
    return CVX_OK;
}

int cvx_get_counters(cvx_ctx* ctx, cvx_counters* out, int32_t reset) {
    if (!ctx || !out) return CVX_ERR_INVALID_ARGUMENT;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(out, ctx->counters, sizeof *out, cudaMemcpyDeviceToHost, ctx->stream));
    if (reset) CU(ctx, cudaMemsetAsync(ctx->counters, 0, sizeof(cvxd_counters), ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return CVX_OK;
}

int cvx_device_frame(cvx_ctx* ctx, void** out_device_ptr, int64_t* out_bytes) {
    if (!ctx || !out_device_ptr) return CVX_ERR_INVALID_ARGUMENT;
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    *out_device_ptr = current_target(ctx);
    if (out_bytes) *out_bytes = (int64_t)ctx->width * ctx->height * 4;
    return CVX_OK;
}

int cvx_device_raybuffer(cvx_ctx* ctx, int32_t which, void** out_device_ptr, int64_t* out_bytes) {
    if (!ctx || !out_device_ptr || which < 0 || which > 1) return CVX_ERR_INVALID_ARGUMENT;
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    *out_device_ptr = raybuffer(ctx->slots[ctx->lastSlot], which);
    if (out_bytes) *out_bytes = raybuffer_pixels(ctx, which) * 4;
    return CVX_OK;
}

int cvx_set_external_frame(cvx_ctx* ctx, void* device_ptr) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    ctx->externalFrame = (uint32_t*)device_ptr;
    return CVX_OK;
}

int cvx_last_draw_ms(cvx_ctx* ctx, float* out_phase1_ms, float* out_phase2_ms) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (!ctx->timed) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "no timed draw yet");
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaEventSynchronize(ctx->evEnd));
    float a = 0, b = 0;
    CU(ctx, cudaEventElapsedTime(&a, ctx->evStart, ctx->evMid));
    CU(ctx, cudaEventElapsedTime(&b, ctx->evMid, ctx->evEnd));
    if (out_phase1_ms) *out_phase1_ms = a;
    if (out_phase2_ms) *out_phase2_ms = b;
    return CVX_OK;
}

int64_t cvx_launch_count(const cvx_ctx* ctx) { return ctx ? ctx->launches : 0; }

int cvx_world_is_regular(const cvx_ctx* ctx) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    return ctx->world.lod_count > 0 && ctx->world.regular ? 1 : 0;
}

int cvx_set_option(cvx_ctx* ctx, int32_t option, int32_t value) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    switch (option) {
    case CVX_OPT_GROUP_SIZE:
        if (value != 0 && value != 8 && value != 16 && value != 32) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "group size %d: expected 0, 8, 16 or 32", value);
        ctx->groupSize = value;
        return CVX_OK;
    case CVX_OPT_COUNTERS:
        ctx->flags = value ? (ctx->flags | CVX_FLAG_COUNTERS) : (ctx->flags & ~CVX_FLAG_COUNTERS);
        return CVX_OK;
    case CVX_OPT_FRAMES_IN_FLIGHT:
        if (value < 1 || value > CVX_MAX_SLOTS) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "frames in flight %d: expected 1..%d", value, CVX_MAX_SLOTS);
        ctx->slotCount = value;
        return CVX_OK;
    case CVX_OPT_GENERAL_PATH:
        ctx->generalPath = value ? 1 : 0;
        return CVX_OK;
    default:
        return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "unknown option %d", option);
    }
}

static void free_profile(cvx_ctx* ctx) {
    for (cudaEvent_t e : ctx->profEvents) cudaEventDestroy(e);
    ctx->profEvents.clear();
    ctx->profCapacity = ctx->profCount = 0;
}

int cvx_profile_begin(cvx_ctx* ctx, int32_t max_draws) {
    if (!ctx || max_draws < 1 || max_draws > (1 << 20)) return CVX_ERR_INVALID_ARGUMENT;
    CU(ctx, cudaSetDevice(ctx->device));
    free_profile(ctx);
    ctx->profEvents.reserve(3 * (size_t)max_draws);
    for (int i = 0; i < 3 * max_draws; i++) {
        cudaEvent_t e;
        CU(ctx, cudaEventCreate(&e));
        ctx->profEvents.push_back(e);
    }
    ctx->profCapacity = max_draws;
    return CVX_OK;
}

int cvx_profile_end(cvx_ctx* ctx, double* out_phase1_ms, double* out_phase2_ms, int32_t* out_draws) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    double p1 = 0.0, p2 = 0.0;
    for (int i = 0; i < ctx->profCount; i++) {
        float a = 0.0f, b = 0.0f;
        CU(ctx, cudaEventElapsedTime(&a, ctx->profEvents[3 * (size_t)i], ctx->profEvents[3 * (size_t)i + 1]));
        CU(ctx, cudaEventElapsedTime(&b, ctx->profEvents[3 * (size_t)i + 1], ctx->profEvents[3 * (size_t)i + 2]));
        p1 += a; p2 += b;
    }
    if (out_phase1_ms) *out_phase1_ms = p1;
    if (out_phase2_ms) *out_phase2_ms = p2;
    if (out_draws) *out_draws = ctx->profCount;
    free_profile(ctx);
    return CVX_OK;
}

int cvx_debug_ray_setup(cvx_ctx* ctx, const cvx_frame_setup* setup, cvx_ray_state* out, int32_t max_rays) {
    cvxd_frame f;
    int r = begin_frame(ctx, setup, 0, false, 0, -1, f);
    if (r) return r;
    if (!out || max_rays < 0) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "bad output buffer");
    int n = f.total_rays < max_rays ? f.total_rays : max_rays;
    if (n == 0) return f.total_rays;
    CU(ctx, cudaSetDevice(ctx->device));
    cvxd_ray_state* d = nullptr;
    CU(ctx, cudaMalloc(&d, sizeof(cvxd_ray_state) * (size_t)n));
    cudaError_t e = cvxd_launch_ray_setup(ctx->world, f, d, n, ctx->stream);
    ctx->launches++;
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d, sizeof(cvxd_ray_state) * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess) return fail(ctx, CVX_ERR_CUDA, "ray setup dump failed: %s", cudaGetErrorString(e));
    return f.total_rays;
}

int cvx_debug_ray_timing(cvx_ctx* ctx, const cvx_frame_setup* setup, int64_t* out_cycles, int32_t max_rays) {
    cvxd_frame f;
    int r = begin_frame(ctx, setup, 0, false, 0, -1, f);
    if (r) return r;
    if (!out_cycles || max_rays < 0) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "bad output buffer");
    if ((r = validate_setup(ctx, setup))) return r;
    const int n = f.total_rays < max_rays ? f.total_rays : max_rays;
    if (n == 0) return f.total_rays;
    CU(ctx, cudaSetDevice(ctx->device));
    long long* d = nullptr;
    const size_t bytes = sizeof(long long) * CVXD_TIMING_REGIONS * (size_t)f.total_rays;
    CU(ctx, cudaMalloc(&d, bytes));
    f.timing = d; f.counters = nullptr;
    cudaError_t e = cudaMemsetAsync(d, 0, bytes, ctx->stream);
    if (e == cudaSuccess) { e = cvxd_launch_phase1(ctx->world, f, 32, ctx->stream); ctx->launches++; }
    if (e == cudaSuccess) e = cudaMemcpyAsync(out_cycles, d, sizeof(long long) * CVXD_TIMING_REGIONS * (size_t)n, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d);
    if (e != cudaSuccess) return fail(ctx, CVX_ERR_CUDA, "ray timing failed: %s", cudaGetErrorString(e));
    return f.total_rays;
}

static_assert(CVX_IPC_HANDLE_BYTES == sizeof(cudaIpcMemHandle_t), "ipc handle size");

int cvx_ipc_export_frame(cvx_ctx* ctx, uint8_t out_handle[CVX_IPC_HANDLE_BYTES]) {
    if (!ctx || !out_handle) return CVX_ERR_INVALID_ARGUMENT;
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    CU(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    CU(ctx, cudaIpcGetMemHandle(&h, ctx->slots[0].frame));
    memcpy(out_handle, &h, sizeof h);
    return CVX_OK;
}

int cvx_ipc_open(cvx_ctx* ctx, const uint8_t handle[CVX_IPC_HANDLE_BYTES], void** out_device_ptr) {
    if (!ctx || !handle || !out_device_ptr) return CVX_ERR_INVALID_ARGUMENT;
    CU(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    CU(ctx, cudaIpcOpenMemHandle(out_device_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return CVX_OK;
}

int cvx_ipc_close(cvx_ctx* ctx, void* device_ptr) {
    if (!ctx || !device_ptr) return CVX_ERR_INVALID_ARGUMENT;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    CU(ctx, cudaIpcCloseMemHandle(device_ptr));
    return CVX_OK;
}

// ---- frame ring -----------------------------------------------------------------------------------------------------------------
static size_t ring_bytes(size_t frameBytes, int slots) { return (size_t)slots * frameBytes + (size_t)slots * sizeof(ring_flags); }

int cvx_ring_close(cvx_ctx* ctx) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (!ctx->ring) return CVX_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->copyStream);
    for (const cvx_slot& sl : ctx->slots) if (sl.stream) cudaStreamSynchronize(sl.stream);
    if (ctx->ringOwner) cudaFree(ctx->ring); else cudaIpcCloseMemHandle(ctx->ring);
    ctx->ring = nullptr; ctx->ringSlots = 0; ctx->ringWorld = 0; ctx->ringOwner = false;
    return CVX_OK;
}

int cvx_ring_create(cvx_ctx* ctx, int32_t slots, int32_t world_size, uint8_t out_handle[CVX_IPC_HANDLE_BYTES]) {
    if (!ctx || !out_handle) return CVX_ERR_INVALID_ARGUMENT;
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    if (slots < 1 || slots > 64 || world_size < 1 || world_size > CVX_RING_MAX_RANKS) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "ring of %d slots for %d ranks", slots, world_size);
    cvx_ring_close(ctx);
    CU(ctx, cudaSetDevice(ctx->device));
    const size_t fb = (size_t)ctx->width * ctx->height * 4;
    void* mem = nullptr;
    CU(ctx, cudaMalloc(&mem, ring_bytes(fb, slots)));
    cudaError_t e = cudaMemsetAsync(mem, 0, ring_bytes(fb, slots), ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, mem);
    if (e != cudaSuccess) { cudaFree(mem); return fail(ctx, CVX_ERR_CUDA, "frame ring: %s", cudaGetErrorString(e)); }
    memcpy(out_handle, &h, sizeof h);
    ctx->ring = (uint8_t*)mem; ctx->ringOwner = true; ctx->ringSlots = slots; ctx->ringWorld = world_size; ctx->ringFrameBytes = fb;
    return CVX_OK;
}

int cvx_ring_open(cvx_ctx* ctx, const uint8_t handle[CVX_IPC_HANDLE_BYTES], int32_t slots, int32_t world_size) {
    if (!ctx || !handle) return CVX_ERR_INVALID_ARGUMENT;
    if (ctx->width <= 0) return fail(ctx, CVX_ERR_NO_RESOLUTION, "no resolution set");
    if (slots < 1 || slots > 64 || world_size < 1 || world_size > CVX_RING_MAX_RANKS) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "ring of %d slots for %d ranks", slots, world_size);
    cvx_ring_close(ctx);
    CU(ctx, cudaSetDevice(ctx->device));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof h);
    void* mem = nullptr;
    CU(ctx, cudaIpcOpenMemHandle(&mem, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->ring = (uint8_t*)mem; ctx->ringOwner = false; ctx->ringSlots = slots; ctx->ringWorld = world_size;
    ctx->ringFrameBytes = (size_t)ctx->width * ctx->height * 4;
    return CVX_OK;
}

// One rank's share of view `view_index`: waits (on the device) until the root has released the ring slot, runs Phase 1 for the rays
// [ray_begin, ray_end), Phase 2 for the pixels those rays feed — stored straight into the ring frame on the root (NVLink peer stores
// when this is not the root) — and signals arrive[slot][rank]. Views rotate over the context's frame slots like cvx_draw_batch.
int cvx_draw_sharded(cvx_ctx* ctx, const cvx_frame_setup* setup, int32_t ray_begin, int32_t ray_end, int64_t view_index, int32_t rank) {
    int r = check_ready(ctx, setup);
    if (r) return r;
    if (!ctx->ring) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "no frame ring (cvx_ring_create / cvx_ring_open)");
    if (rank < 0 || rank >= ctx->ringWorld || view_index < 0) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "rank %d / view %lld outside the ring", rank, (long long)view_index);
    if ((r = validate_setup(ctx, setup))) return r;
    CU(ctx, cudaSetDevice(ctx->device));
    const int K = ctx->slotCount;
    if ((r = ensure_slots(ctx, K))) return r;
    const int slot = (int)(view_index % K), rslot = (int)(view_index % ctx->ringSlots);
    cudaStream_t stream = slot_stream(ctx, slot);
    cvxd_frame f;
    make_frame(ctx, setup, slot, f);
    if (ray_begin == CVX_SHARD_INTERLEAVED) {
        // rays dealt in chunks of `ray_end` rays, chunk c to rank c mod world: heavy rays come in runs of neighbouring rays, so every
        // rank gets its share of them without any cost estimate; the launch covers the rank's local rays [0, n)
        const int chunk = ray_end;
        if (chunk < 1 || (chunk & (chunk - 1))) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "interleaved sharding needs a power-of-two chunk size (got %d)", chunk);
        const int world = ctx->ringWorld;
        const int fullRounds = f.total_rays / (chunk * world), rest = f.total_rays % (chunk * world);
        int n = fullRounds * chunk;
        const int mine = rest - rank * chunk;
        n += mine <= 0 ? 0 : (mine < chunk ? mine : chunk);
        f.il_chunk = chunk; f.il_ranks = world; f.il_rank = rank;
        ray_begin = 0; ray_end = n;
    } else {
        clamp_range(ray_begin, ray_end, f.total_rays);
    }
    f.ray_begin = ray_begin; f.ray_end = ray_end;
    ring_flags* fl = ring_flag_block(ctx, rslot);
    CU(ctx, mark_phase(ctx, 0, stream, false));   // cvx_profile_begin: events around this share's Phase 1 and Phase 2
    CU(ctx, cvxd_launch_phase1(ctx->world, f, ctx->groupSize, stream));   // Phase 1 writes this rank's own raybuffers: no need to wait for the ring
    if (ray_end > ray_begin) ctx->launches++;
    if (view_index >= ctx->ringSlots) {  // the ring frame still holds view_index - slots until the root releases it
        ring_wait_kernel<<<1, 32, 0, stream>>>(&fl->released, 1, (uint32_t)(view_index - ctx->ringSlots + 1), &ring_flag_block(ctx, 0)->error);
        ctx->launches++;
    }
    cvxd_blit b;
    make_blit(f, ring_frame(ctx, rslot), b);
    b.owned_only = 1;
    CU(ctx, mark_phase(ctx, 1, stream, false));
    CU(ctx, cvxd_launch_phase2(b, stream));
    CU(ctx, mark_phase(ctx, 2, stream, false));
    ring_signal_kernel<<<1, 1, 0, stream>>>(&fl->arrive[rank], (uint32_t)(view_index + 1));
    ctx->launches += 2;
    CU(ctx, cudaGetLastError());
    ctx->lastSlot = slot;
    return CVX_OK;
}

// Root only: waits (device side, on the copy stream) until every rank has stored its pixels of `view_index`, copies the frame to
// dst_host if given (pinned memory for an asynchronous copy), and releases the ring slot for view_index + slots.
// out_device_frame (optional) receives the frame's device address (valid until the slot is reused).
int cvx_ring_consume(cvx_ctx* ctx, int64_t view_index, void* dst_host, void** out_device_frame) {
    if (!ctx) return CVX_ERR_INVALID_ARGUMENT;
    if (!ctx->ring || !ctx->ringOwner) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "cvx_ring_consume is for the rank that created the ring");
    if (view_index < 0) return fail(ctx, CVX_ERR_INVALID_ARGUMENT, "view index < 0");
    CU(ctx, cudaSetDevice(ctx->device));
    const int rslot = (int)(view_index % ctx->ringSlots);
    ring_flags* fl = ring_flag_block(ctx, rslot);
    ring_wait_kernel<<<1, CVX_RING_MAX_RANKS, 0, ctx->copyStream>>>(fl->arrive, ctx->ringWorld, (uint32_t)(view_index + 1), &ring_flag_block(ctx, 0)->error);
    if (dst_host) CU(ctx, cudaMemcpyAsync(dst_host, ring_frame(ctx, rslot), ctx->ringFrameBytes, cudaMemcpyDeviceToHost, ctx->copyStream));
    ring_signal_kernel<<<1, 1, 0, ctx->copyStream>>>(&fl->released, (uint32_t)(view_index + 1));
    ctx->launches += 2;
    CU(ctx, cudaGetLastError());
    if (out_device_frame) *out_device_frame = ring_frame(ctx, rslot);
    return CVX_OK;
}

// 0 = no wait of this context's ring has timed out so far (call after cvx_sync; root only sees every slot's flag block)
int cvx_ring_status(cvx_ctx* ctx) {
    if (!ctx || !ctx->ring) return CVX_ERR_INVALID_ARGUMENT;
    CU(ctx, cudaSetDevice(ctx->device));
    uint32_t bad = 0;   // one error word for the whole ring (slot 0's): the first wait that times out raises it, later waits return at once
    CU(ctx, cudaMemcpy(&bad, &ring_flag_block(ctx, 0)->error, 4, cudaMemcpyDeviceToHost));
    return bad ? fail(ctx, CVX_ERR_CUDA, "a frame-ring wait timed out (a rank did not deliver its share of a view)") : CVX_OK;
}

int cvx_alloc_pinned(int64_t bytes, void** out) {
    if (!out || bytes <= 0) return CVX_ERR_INVALID_ARGUMENT;
    cudaError_t e = cudaHostAlloc(out, (size_t)bytes, cudaHostAllocDefault);
    return e == cudaSuccess ? CVX_OK : cvx_code(e);
}

int cvx_free_pinned(void* p) { return cudaFreeHost(p) == cudaSuccess ? CVX_OK : CVX_ERR_CUDA; }

} // extern "C"
