// emu_phase1.cpp — TEST-ONLY: compiles cpuvox_b200/csrc/raybuffer_kernels.cu for the CPU through the SIMT emulator
// (cuda_emu.h) and exposes Phase 1 to the tests, so kernel logic can be compared with the oracle without a GPU.
// Not linked into libcpuvox_b200.so and never used by the product path.
#define CVX_EMU 1
#include "cuda_emu.h"

#include <atomic>
#include <thread>
#include <vector>

#ifdef CVX_EMU_STATS
unsigned long long* emu_stats = nullptr;
#endif
#include "../../cpuvox_b200/csrc/raybuffer_kernels.cu"
#include "../../cpuvox_b200/csrc/host_frame.h"
#include "../../cpuvox_b200/csrc/world_transcode.h"
#include "../../cpuvox_b200/csrc/raycast.h"

struct emu_world {
    cvxh_lod_tables tables[CVXD_LODS];
    std::vector<uint32_t> elements[CVXD_LODS];
    cvxd_world w;
};

namespace {

struct LaunchArgs { const cvxd_world* world; const cvxd_frame* frame; int variant, group; bool counters; };

template <int G, bool INV>
void body_gi(const LaunchArgs* a) {
    if (a->variant == 0) {
        if (a->counters) phase1_kernel<G, true, false, false, INV>(*a->world, *a->frame);
        else phase1_kernel<G, false, false, false, INV>(*a->world, *a->frame);
    } else {
        if (a->counters) phase1_kernel<G, true, false, true, INV>(*a->world, *a->frame);
        else phase1_kernel<G, false, false, true, INV>(*a->world, *a->frame);
    }
}

template <int G>
void body_g(void* p) {
    const LaunchArgs* a = (const LaunchArgs*)p;
    if (a->frame->inverse) body_gi<G, true>(a); else body_gi<G, false>(a);
}

} // namespace

extern "C" {

emu_world* emu_world_create(int lods, const int32_t dims[3], const void* const* blobs, const int64_t* bytes, const int32_t* column_counts) {
    emu_world* w = new emu_world();
    memset(&w->w, 0, sizeof w->w);
    cvxd_world_set_dims(&w->w, dims[0], dims[1], dims[2]);
    w->w.lod_count = lods;
    w->w.regular = 1;
    for (int l = 0; l < lods; l++) {
        const int64_t needCols = (int64_t)(dims[0] >> l) * (dims[2] >> l);
        const int64_t headerBytes = 12 * (int64_t)column_counts[l];
        const int64_t cells = (bytes[l] - headerBytes) / 4;
        if (!cvxh_transcode_lod(blobs[l], needCols, column_counts[l], cells, l, dims[1], w->tables[l])) { delete w; return nullptr; }
        w->elements[l].assign((const uint32_t*)((const uint8_t*)blobs[l] + headerBytes), (const uint32_t*)((const uint8_t*)blobs[l] + headerBytes) + cells);
        cvxd_lod& d = w->w.lods[l];
        d.headers = (const uint4*)w->tables[l].headers.data();
        d.elements = w->elements[l].data();
        d.bounds = (const uint2*)w->tables[l].bounds.data();
        d.mul_x = dims[2] >> l;
        d.lod = l;
        if (!w->tables[l].regular) w->w.regular = 0;
    }
    return w;
}

// The host transcode's verdict on one LOD blob, as cvx_world_upload would be given it: returns 1 when it accepts the blob, 0 when it
// rejects it (*bad_column = the first column pointing outside the element area); *regular = the LOD's boundary-table flag.
int emu_transcode_verdict(const void* blob, int64_t bytes, int32_t column_count, int lod, const int32_t dims[3], int64_t* bad_column, int* regular) {
    const int64_t needCols = (int64_t)(dims[0] >> lod) * (dims[2] >> lod);
    const int64_t cells = (bytes - 12 * (int64_t)column_count) / 4;
    cvxh_lod_tables t;
    const bool ok = cvxh_transcode_lod(blob, needCols, column_count, cells, lod, dims[1], t);
    *bad_column = t.bad_column;
    *regular = t.regular ? 1 : 0;
    return ok ? 1 : 0;
}

// The kernel's minf_ / maxf_, elementwise (test hook for the NaN and signed-zero rule).
void emu_min_max(const float* a, const float* b, int n, float* out_min, float* out_max) {
    for (int i = 0; i < n; i++) { out_min[i] = minf_(a[i], b[i]); out_max[i] = maxf_(a[i], b[i]); }
}

#ifdef CVX_EMU_STATS
void emu_set_stats(unsigned long long* p) { emu_stats = p; } // 16 counters per flat ray
#endif
void emu_world_destroy(emu_world* w) { delete w; }
int emu_world_regular(const emu_world* w) { return w->w.regular; }

// Renders rays [ray_begin, ray_end) of the frame into td / lr (host memory, same layout as the device raybuffers).
int emu_phase1(const emu_world* w, const cvx_frame_setup* setup, int W, int H, uint32_t* td, uint32_t* lr, cvxd_counters* counters,
               int variant, int group, int threads, int ray_begin, int ray_end) {
    cvxd_frame f;
    cvxh::frame_from_setup(setup, W, H, f);
    cvxd_frame_set_world(&f, &w->w);
    f.td = td; f.lr = lr; f.counters = counters;
    if (ray_end < 0 || ray_end > f.total_rays) ray_end = f.total_rays;
    if (ray_begin < 0) ray_begin = 0;
    f.ray_begin = ray_begin; f.ray_end = ray_end;
    const int n = ray_end - ray_begin;
    if (n <= 0) return 0;
    if (group != 8 && group != 16 && group != 32) group = 32;
    const int groupsPerCta = CVXD_THREADS_PER_CTA / group;
    const int blocks = (n + groupsPerCta - 1) / groupsPerCta;
    const size_t smemWords = phase1_smem_bytes(group, W, H) / sizeof(uint32_t) + 64;
    LaunchArgs args{&w->w, &f, variant, group, counters != nullptr};
    std::atomic<int> next{0};
    if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
    if (threads > blocks) threads = blocks;
    auto worker = [&]() {
        std::vector<uint32_t> smem(smemWords);
        for (;;) {
            const int b = next.fetch_add(1);
            if (b >= blocks) break;
            emu::g_shared = smem.data();
            for (int warp = 0; warp < CVXD_THREADS_PER_CTA / 32; warp++) {
                emu_dim3 tids[32];
                for (int i = 0; i < 32; i++) tids[i] = emu_dim3{warp * 32 + i, 0, 0};
                void (*body)(void*) = group == 32 ? body_g<32> : (group == 16 ? body_g<16> : body_g<8>);
                emu::run_warp(body, &args, tids, emu_dim3{b, 0, 0}, emu_dim3{CVXD_THREADS_PER_CTA, 1, 1}, emu_dim3{blocks, 1, 1}, 32);
            }
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; t++) pool.emplace_back(worker);
    worker();
    for (auto& t : pool) t.join();
    return n;
}

// cvx_raycast's traversal (raycast.h) for rays [0, n) at LOD lod: one call per ray, as one device thread runs it. general != 0 reads
// runs from the element area even for a regular LOD (CVX_OPT_GENERAL_PATH).
int emu_raycast(const emu_world* w, int lod, const cvxd_ray* rays, int n, cvxd_ray_hit* hits, int general, int threads) {
    if (lod < 0 || lod >= w->w.lod_count || n < 0) return -1;
    const bool bounds = w->tables[lod].regular && !general;
    std::atomic<int> next{0};
    if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
    auto worker = [&]() {
        for (;;) {
            const int b = next.fetch_add(1024);
            if (b >= n) break;
            for (int i = b; i < n && i < b + 1024; i++) cvxr_cast(w->w, lod, rays[i], bounds, hits[i]);
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; t++) pool.emplace_back(worker);
    worker();
    for (auto& t : pool) t.join();
    return 0;
}

} // extern "C"
