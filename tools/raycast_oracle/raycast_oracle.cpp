// raycast_oracle.cpp — TEST INFRASTRUCTURE ONLY: the definition of cvx_raycast (DESIGN.md §3.5), written as the literal per-cell
// walk over the LOD blob in the reference layout (12-byte RLEColumn headers, then the element area; World.cs:161-209,285-313),
// with no skipping. Every cell the walk enters is looked up through GetVoxelColumn-style decoding of its column. The product
// kernel (cpuvox_b200/csrc/raycast.h) must equal this bit for bit, including `distance` bits and `steps`. Shares no code with it.
// Built with -ffp-contract=off: IEEE fp32 in the order written.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <atomic>
#include <thread>
#include <vector>

namespace {

struct Ray { float origin[3]; float max_distance; float direction[3]; int32_t reserved; };
struct Hit { int32_t hit; int32_t face; int32_t cell[3]; float distance; uint32_t color; int32_t steps; };
struct Box { float center[3]; float max_distance; float direction[3]; int32_t reserved0; float half_extent[3]; int32_t reserved1; };
static_assert(sizeof(Ray) == 32 && sizeof(Hit) == 32 && sizeof(Box) == 48, "layouts");

struct Lod { const uint8_t* blob; int64_t bytes; int32_t column_count; };

struct World {
    int32_t dims[3];
    Lod lods[6];
};

bool finite(float v) { return std::isfinite(v); }

// World.GetVoxelColumn restated for one cell: walk the column's runs top to bottom from cell ny. Returns true and the colour
// when cell cy is solid. Cells whose world-Y range misses the header's [worldMin, worldMax) are air.
bool solid(const World& w, int lod, int cx, int cy, int cz, uint32_t* colour) {
    const Lod& L = w.lods[lod];
    const int nz = w.dims[2] >> lod, ny = w.dims[1] >> lod;
    const int64_t col = (int64_t)cx * nz + cz;
    uint32_t h[3];
    memcpy(h, L.blob + 12 * col, 12);
    const int runCount = (int)(h[1] & 0xffffu);
    if (runCount == 0) return false;
    const int64_t worldMin = h[1] >> 16, worldMax = h[2] & 0xffffu;
    const int64_t y0 = (int64_t)cy << lod, y1 = (int64_t)(cy + 1) << lod;
    if (y1 <= worldMin || y0 >= worldMax) return false;
    const uint32_t* cells = (const uint32_t*)(L.blob + 12 * (int64_t)L.column_count);
    const uint32_t* runs = cells + h[0] + 1;
    const uint32_t* colours = cells + h[0] + runCount + 2;
    int top = ny;
    for (int k = 0; k < runCount; k++) {
        uint32_t e = runs[k];
        const int16_t colorsIndex = (int16_t)(e & 0xffffu), length = (int16_t)(e >> 16);
        if (length <= 0) return false;               // the column ends here
        if (cy >= top - length && cy < top) {
            if (colorsIndex < 0) return false;
            *colour = colours[colorsIndex + (top - 1 - cy)];
            return true;
        }
        top -= length;
    }
    return false;
}

float tmax_of(int cell, int step, int lod, float o, float inv) {
    if (step == 0) return INFINITY;
    return ((float)((cell + (step > 0 ? 1 : 0)) << lod) - o) * inv;
}

// step 1 of §3.5 and §3.6: false when the squared length is 0 or not finite
bool normalise(const float dir[3], float d[3], float inv[3], int step[3]) {
    const float len2 = dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2];
    if (!(len2 > 0.0f) || !finite(len2)) return false;
    const float invLen = 1.0f / sqrtf(len2);
    for (int i = 0; i < 3; i++) {
        d[i] = dir[i] * invLen;
        inv[i] = 0.0f;
        step[i] = 0;
        if (d[i] != 0.0f) {
            const float v = 1.0f / d[i];
            if (finite(v)) { inv[i] = v; step[i] = d[i] > 0.0f ? 1 : -1; }
            else d[i] = 0.0f;
        }
    }
    return true;
}

void cast(const World& w, int lod, const Ray& r, Hit& out) {
    memset(&out, 0, sizeof out);
    out.hit = -1;
    // 1. normalise
    for (int i = 0; i < 3; i++)
        if (!finite(r.origin[i]) || !finite(r.direction[i])) return;
    if (std::isnan(r.max_distance) || r.max_distance == -INFINITY) return;
    float d[3], inv[3];
    int step[3];
    if (!normalise(r.direction, d, inv, step)) return;
    out.hit = 0;
    const float* o = r.origin;
    const float maxd = r.max_distance;
    const int n[3] = {w.dims[0] >> lod, w.dims[1] >> lod, w.dims[2] >> lod};
    // 2. enter the box of the LOD's cells, [0, n_i << lod] per axis (short of dim_y when 2^lod does not divide it)
    float tEnter = -INFINITY, tExit = INFINITY;
    int entry = -1;
    const int order[3] = {0, 2, 1};
    for (int q = 0; q < 3; q++) {
        const int i = order[q];
        const float dim = (float)(n[i] << lod);
        if (step[i] == 0) {
            if (!(o[i] >= 0.0f && o[i] < dim)) return;
            continue;
        }
        const float a = (0.0f - o[i]) * inv[i], b = (dim - o[i]) * inv[i];
        const float nearT = step[i] > 0 ? a : b, farT = step[i] > 0 ? b : a;
        if (nearT > tEnter) { tEnter = nearT; entry = i; }
        if (farT < tExit) tExit = farT;
    }
    const float t0 = tEnter > 0.0f ? tEnter : 0.0f;
    if (tEnter > tExit || tExit < 0.0f || !(t0 <= maxd) || t0 == INFINITY) return;
    // 3. start cell, 4. boundary distances
    const float invS = 1.0f / (float)(1 << lod);
    int c[3];
    float tm[3];
    for (int i = 0; i < 3; i++) {
        if (tEnter > 0.0f && i == entry) c[i] = step[i] > 0 ? 0 : n[i] - 1;
        else {
            const float f = floorf((o[i] + t0 * d[i]) * invS);
            c[i] = f < 0.0f ? 0 : (f > (float)(n[i] - 1) ? n[i] - 1 : (int)f);
        }
        tm[i] = tmax_of(c[i], step[i], lod, o[i], inv[i]);
    }
    int face = tEnter > 0.0f ? 2 * entry + (step[entry] > 0 ? 0 : 1) : 6;
    float t = t0;
    // 5. walk
    for (int steps = 1;; steps++) {
        uint32_t colour = 0;
        if (solid(w, lod, c[0], c[1], c[2], &colour)) {
            out.hit = 1; out.face = face; out.distance = t; out.color = colour; out.steps = steps;
            out.cell[0] = c[0]; out.cell[1] = c[1]; out.cell[2] = c[2];
            return;
        }
        int a;
        if (tm[0] <= tm[1] && tm[0] <= tm[2]) a = 0;
        else if (tm[2] <= tm[1]) a = 2;
        else a = 1;
        const int next = c[a] + step[a];
        if (tm[a] > maxd || tm[a] == INFINITY || next < 0 || next >= n[a]) { out.steps = steps; return; }
        c[a] = next;
        t = tm[a];
        face = 2 * a + (step[a] > 0 ? 0 : 1);
        tm[a] = tmax_of(c[a], step[a], lod, o[a], inv[a]);
    }
}

// cvx_sweep (DESIGN.md §3.6) evaluated cell by cell over the swept box's bounding box: on each axis the cells whose own window
// meets [0, max_distance] (a cell outside that set cannot be a candidate: T >= enter_i, T' <= exit_i). steps stays 0.
struct Window { int k; float enter, exit; };

void sweep(const World& w, int lod, const Box& b, Hit& out) {
    memset(&out, 0, sizeof out);
    out.hit = -1;
    // 1. invalid inputs, normalise
    for (int i = 0; i < 3; i++)
        if (!finite(b.center[i]) || !finite(b.direction[i]) || !finite(b.half_extent[i]) || !(b.half_extent[i] > 0.0f)) return;
    const float maxd = b.max_distance;
    if (std::isnan(maxd) || maxd == -INFINITY) return;
    float d[3], inv[3];
    int step[3];
    if (!normalise(b.direction, d, inv, step)) return;
    out.hit = 0;
    const int n[3] = {w.dims[0] >> lod, w.dims[1] >> lod, w.dims[2] >> lod};
    // 2. per-axis windows
    std::vector<Window> win[3];
    for (int i = 0; i < 3; i++) {
        const float c = b.center[i], h = b.half_extent[i];
        for (int k = 0; k < n[i]; k++) {
            const float lo = (float)(k << lod) - h, hi = (float)((k + 1) << lod) + h;
            float enter, exit;
            if (step[i] == 0) {
                if (!(lo < c && c < hi)) continue;
                enter = -INFINITY;
                exit = INFINITY;
            } else {
                const float a = (lo - c) * inv[i], bb = (hi - c) * inv[i];
                enter = step[i] > 0 ? a : bb;
                exit = step[i] > 0 ? bb : a;
            }
            if (enter < exit && exit > 0.0f && enter <= maxd) win[i].push_back(Window{k, enter, exit});
        }
    }
    // 3. candidates, 4. the smallest key (t*, overlapping first, cx, cz, cy)
    bool found = false, bestOv = false;
    float bestT = 0.0f;
    int best[3] = {0, 0, 0}, bestFace = 0;
    uint32_t bestColour = 0;
    for (const Window& X : win[0])
        for (const Window& Z : win[2]) {
            // the XZ part alone already rules the column out (max and min only grow and shrink with the y window)
            const float txz = Z.enter > X.enter ? Z.enter : X.enter, uxz = Z.exit < X.exit ? Z.exit : X.exit;
            if (!(txz < uxz) || !(txz <= maxd)) continue;
            for (const Window& Y : win[1]) {
                float T = X.enter;
                int axis = 0;
                if (Z.enter > T) { T = Z.enter; axis = 2; }
                if (Y.enter > T) { T = Y.enter; axis = 1; }
                float Tp = X.exit;
                if (Z.exit < Tp) Tp = Z.exit;
                if (Y.exit < Tp) Tp = Y.exit;
                const float ts = T > 0.0f ? T : 0.0f;
                if (!(T < Tp && Tp > 0.0f && ts <= maxd && finite(ts))) continue;
                const bool ov = T < 0.0f;
                const int cell[3] = {X.k, Y.k, Z.k};
                bool better = !found;
                if (found) {
                    if (ts != bestT) better = ts < bestT;
                    else if (ov != bestOv) better = ov;
                    else if (cell[0] != best[0]) better = cell[0] < best[0];
                    else if (cell[2] != best[2]) better = cell[2] < best[2];
                    else better = cell[1] < best[1];
                }
                if (!better) continue;
                uint32_t colour = 0;
                if (!solid(w, lod, cell[0], cell[1], cell[2], &colour)) continue;
                found = true; bestT = ts; bestOv = ov; bestColour = colour;
                best[0] = cell[0]; best[1] = cell[1]; best[2] = cell[2];
                bestFace = ov ? 6 : 2 * axis + (step[axis] > 0 ? 0 : 1);
            }
        }
    if (!found) return;
    out.hit = 1; out.face = bestFace; out.distance = bestT; out.color = bestColour;
    out.cell[0] = best[0]; out.cell[1] = best[1]; out.cell[2] = best[2];
}

// body(i) for i in [0, n) on `threads` host threads (<= 0: all hardware threads), `chunk` queries at a time
template <class F>
void parallel(int n, int threads, int chunk, F body) {
    if (threads <= 0) threads = (int)std::thread::hardware_concurrency();
    if (threads < 1) threads = 1;
    std::atomic<int> next{0};
    auto worker = [&]() {
        for (;;) {
            const int b = next.fetch_add(chunk);
            if (b >= n) break;
            const int e = b + chunk < n ? b + chunk : n;
            for (int i = b; i < e; i++) body(i);
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < threads; t++) pool.emplace_back(worker);
    worker();
    for (auto& t : pool) t.join();
}

} // namespace

extern "C" {

void* rco_world_create(int32_t dim_x, int32_t dim_y, int32_t dim_z) {
    World* w = new World();
    memset(w, 0, sizeof *w);
    w->dims[0] = dim_x; w->dims[1] = dim_y; w->dims[2] = dim_z;
    return w;
}

// borrowed blob: must outlive the world
int rco_world_set_lod(void* world, int32_t lod, const void* blob, int64_t bytes, int32_t column_count) {
    if (!world || lod < 0 || lod >= 6 || !blob) return -1;
    World* w = (World*)world;
    w->lods[lod] = Lod{(const uint8_t*)blob, bytes, column_count};
    return 0;
}

void rco_world_free(void* world) { delete (World*)world; }

// n rays at LOD lod on `threads` host threads (<= 0: all hardware threads)
int rco_raycast(const void* world, int32_t lod, const void* rays, int32_t n, void* hits, int32_t threads) {
    const World* w = (const World*)world;
    if (!w || lod < 0 || lod >= 6 || !w->lods[lod].blob || n < 0) return -1;
    const Ray* in = (const Ray*)rays;
    Hit* out = (Hit*)hits;
    parallel(n, threads, 1024, [&](int i) { cast(*w, lod, in[i], out[i]); });
    return 0;
}

// n boxes at LOD lod on `threads` host threads (<= 0: all hardware threads)
int rco_sweep(const void* world, int32_t lod, const void* boxes, int32_t n, void* hits, int32_t threads) {
    const World* w = (const World*)world;
    if (!w || lod < 0 || lod >= 6 || !w->lods[lod].blob || n < 0) return -1;
    const Box* in = (const Box*)boxes;
    Hit* out = (Hit*)hits;
    parallel(n, threads, 64, [&](int i) { sweep(*w, lod, in[i], out[i]); });
    return 0;
}

} // extern "C"
