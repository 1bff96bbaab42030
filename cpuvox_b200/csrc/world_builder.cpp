/*
 * world_builder.cpp — host-side (offline, CPU) world production for libcpuvox_b200: the step before the
 * hot path. Produces byte-compatible World blobs (Assets/Code/World.cs:161-188,245-259,285-313) that
 * cvx_world_upload consumes, from a triangle mesh or from the seeded synthetic generators of
 * BASELINE.json configs 2-5.
 *
 * Follows: ObjModel.Import (Assets/Code/Utils/ObjModel.cs:36-196), SimpleMesh.Remap_Internal
 * (Assets/Code/Utils/SimpleMesh.cs:64-106), VoxelizerHelper.GetVoxelsInternal (Assets/Code/VoxelizerHelper.cs:28-132),
 * WorldBuilder.Import/ToLOD0World/RLEColumnBuilder.ToFinalColumn (Assets/Code/WordBuilder.cs:39-130,181-268),
 * World.DownSample/DownSampleColumn/DownSamplePartial (Assets/Code/World.cs:45-127), RLEColumn ctor (:190-234),
 * WorldAllocator capacity growth (:295-373), WorldSaveFile (Assets/Code/WorldSaveFile.cs:8-103).
 *
 * Re-designed, not translated: the reference appends voxels into per-column List<Voxel> under locks, sorts
 * and dedupes; here voxels are binned by column and resolved with a per-Y accumulator (sum/count per channel),
 * which yields the same column (the dedupe average (first + sum others)/count is order independent) with a
 * deterministic element layout (columns allocated in index order, independent of thread count).
 */
#include "../../include/cpuvox_b200.h"
#include "world_builder.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

namespace {

using Blob = cvx_lod_blob;

struct ColHeader { // World.RLEColumn, 12 bytes
    int32_t offset;
    uint16_t runCount, worldMin, worldMax, pad;
};
struct Run { int16_t colorsIndex, length; }; // World.RLEElement
static_assert(sizeof(ColHeader) == 12 && sizeof(Run) == 4, "layout");

template <class F>
void run_parallel(int64_t n, int n_threads, F fn) {
    if (n_threads <= 0) n_threads = (int)std::thread::hardware_concurrency();
    if (n_threads < 1) n_threads = 1;
    if (n_threads == 1 || n <= 1) { for (int64_t i = 0; i < n; i++) fn(i, 0); return; }
    std::atomic<int64_t> next(0);
    std::vector<std::thread> th;
    for (int t = 0; t < n_threads; t++)
        th.emplace_back([&, t]() { for (;;) { int64_t i = next.fetch_add(1); if (i >= n) break; fn(i, t); } });
    for (auto& x : th) x.join();
}

// Per-Y accumulator standing in for RLEColumnBuilder's List<Voxel> + sort + dedupe (WordBuilder.cs:183-228).
struct YAccumulator {
    std::vector<uint32_t> r, g, b, n;
    std::vector<uint8_t> a;
    std::vector<int> touched;
    void reset(int height) {
        if ((int)n.size() < height) { r.assign(height, 0); g.assign(height, 0); b.assign(height, 0); n.assign(height, 0); a.assign(height, 0); }
        for (int y : touched) { r[y] = g[y] = b[y] = n[y] = 0; }
        touched.clear();
    }
    inline void add(int y, uint32_t argb) { // bytes a,r,g,b
        if (n[y] == 0) { touched.push_back(y); a[y] = (uint8_t)(argb & 0xff); }
        r[y] += (argb >> 8) & 0xff; g[y] += (argb >> 16) & 0xff; b[y] += (argb >> 24) & 0xff;
        n[y]++;
    }
};

// One chunk of consecutive columns resolved into headers (offsets local to the chunk) + elements.
struct Chunk {
    std::vector<ColHeader> headers;
    std::vector<uint32_t> elements;
    int64_t voxels = 0;
};

// RLEColumnBuilder.ToFinalColumn (WordBuilder.cs:181-268) + RLEColumn ctor (World.cs:190-234) on an accumulator.
void finalize_column(YAccumulator& acc, int voxelScale, int topY, Chunk& out, ColHeader& hdr, std::vector<Run>& runs, std::vector<uint32_t>& colors) {
    memset(&hdr, 0, sizeof hdr);
    if (acc.touched.empty()) return;
    std::sort(acc.touched.begin(), acc.touched.end(), [](int p, int q) { return p > q; }); // descending Y
    runs.clear(); colors.clear();
    const int count = (int)acc.touched.size();
    for (int i = 0; i < count; i++) {
        int y = acc.touched[i];
        uint32_t w = acc.n[y];
        uint32_t cr = (acc.r[y] / w) & 0xff, cg = (acc.g[y] / w) & 0xff, cb = (acc.b[y] / w) & 0xff;
        colors.push_back((uint32_t)acc.a[y] | (cr << 8) | (cg << 16) | (cb << 24));
    }
    out.voxels += count;
    int top = topY;
    for (int i = 0; i < count;) {
        int voxelY = acc.touched[i];
        int airFromTop = top - voxelY;
        if (airFromTop > 0) { runs.push_back(Run{(int16_t)-1, (int16_t)airFromTop}); top -= airFromTop; }
        int runLength = 1;
        for (int j = i + 1; j < count; j++) { if (top - (j - i) == acc.touched[j]) runLength++; else break; }
        runs.push_back(Run{(int16_t)i, (int16_t)runLength});
        top -= runLength;
        i += runLength;
    }
    if (top >= 0) runs.push_back(Run{(int16_t)-1, (int16_t)(top + 1)});

    const int runCount = (int)runs.size();
    hdr.offset = (int32_t)out.elements.size();
    hdr.runCount = (uint16_t)runCount;
    out.elements.push_back(0); // guard (0,0)
    for (const Run& r : runs) { uint32_t v; memcpy(&v, &r, 4); out.elements.push_back(v); }
    out.elements.push_back(0); // guard
    for (uint32_t c : colors) out.elements.push_back(c);
    int wmin = INT32_MAX, wmax = INT32_MIN, bmin = 0, bmax = 0;
    for (int i = runCount - 1; i >= 0; i--) {
        bmin = bmax; bmax = bmin + runs[i].length;
        if (runs[i].colorsIndex < 0) continue;
        wmin = std::min(wmin, bmin); wmax = std::max(wmax, bmax);
    }
    hdr.worldMin = (uint16_t)(wmin * voxelScale);
    hdr.worldMax = (uint16_t)(wmax * voxelScale);
}

const int CHUNK_COLUMNS = 4096;

// Assemble chunks (in column order) into a blob with the reference's allocator capacity rule (World.cs:295-373):
// capacity starts at columnCount*4 elements and doubles until it fits; byte length = 12*columnCount + 4*capacity.
void assemble_blob(Blob& blob, int columnCount, int64_t slots, const std::vector<Chunk>& chunks,
                   const std::vector<int64_t>& chunkFirstSlot, const std::vector<std::vector<int64_t>>* slotMap) {
    int64_t total = 0;
    for (auto& c : chunks) total += (int64_t)c.elements.size();
    int64_t capacity = (int64_t)columnCount * 4;
    while (capacity < total) capacity = capacity > INT32_MAX / 2 ? INT32_MAX : capacity * 2;
    blob.columnCount = columnCount;
    blob.bytes.assign((size_t)(12 * (int64_t)columnCount + 4 * capacity), 0);
    ColHeader* headers = (ColHeader*)blob.bytes.data();
    uint32_t* elements = (uint32_t*)(blob.bytes.data() + 12 * (int64_t)columnCount);
    int64_t base = 0;
    blob.voxelCount = 0;
    for (size_t ci = 0; ci < chunks.size(); ci++) {
        const Chunk& c = chunks[ci];
        for (size_t i = 0; i < c.headers.size(); i++) {
            ColHeader h = c.headers[i];
            if (h.runCount > 0) h.offset += (int32_t)base;
            int64_t slot = slotMap ? (*slotMap)[ci][i] : chunkFirstSlot[ci] + (int64_t)i;
            if (slot < slots) headers[slot] = h;
        }
        if (!c.elements.empty()) memcpy(elements + base, c.elements.data(), c.elements.size() * 4);
        base += (int64_t)c.elements.size();
        blob.voxelCount += c.voxels;
    }
    blob.built = true;
}


inline uint8_t to_byte(float c) { // Color -> Color32: round(clamp01(c)*255), half-to-even (SURVEY A10); NaN -> 0
    float v = c > 0.0f ? (c < 1.0f ? c : 1.0f) : 0.0f;
    return (uint8_t)rintf(v * 255.0f);
}
inline int next_pow2(int n) { int p = 1; while (p < n) p <<= 1; return n <= 0 ? 0 : p; } // Mathf.NextPowerOfTwo (A11)
inline int clampi(int x, int a, int b) { return std::max(a, std::min(b, x)); }
inline int f2i(float f) { if (!(f >= -2147483648.0f && f < 2147483648.0f)) return INT32_MIN; return (int)f; }

struct V3 { float x, y, z; };
inline V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
inline V3 operator*(V3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
inline float dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline V3 cross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline V3 normalize(V3 a) { float r = 1.0f / sqrtf(dot(a, a)); return a * r; }

// VoxelizerHelper.GetVoxelsInternal (VoxelizerHelper.cs:28-132) for one triangle.
void voxelize_triangle(const V3 pa, const V3 pb, const V3 pc, const uint8_t* c0, const uint8_t* c1, const uint8_t* c2,
                       const int maxDim[3], std::vector<MeshVoxel>& out) {
    V3 a = pa, b = pb, c = pc;
    V3 nc = cross(b - a, c - a);
    float l2 = dot(nc, nc);
    if (l2 == 0.0f) return;
    V3 n = nc * (1.0f / sqrtf(l2));
    V3 mid = (a + b + c) * 1.0f; mid = {mid.x / 3.0f, mid.y / 3.0f, mid.z / 3.0f};
    a = a + normalize(a - mid) * 0.5f;
    b = b + normalize(b - mid) * 0.5f;
    c = c + normalize(c - mid) * 0.5f;
    // math.min / math.max ignore a NaN operand, as fminf / fmaxf do: a corner on the centroid (normalize(0) = NaN) drops out of
    // the box, which then spans the other two corners (DESIGN.md §3.4)
    V3 mn = {fminf(a.x, fminf(b.x, c.x)), fminf(a.y, fminf(b.y, c.y)), fminf(a.z, fminf(b.z, c.z))};
    V3 mx = {fmaxf(a.x, fmaxf(b.x, c.x)), fmaxf(a.y, fmaxf(b.y, c.y)), fmaxf(a.z, fmaxf(b.z, c.z))};
    int lo[3] = {clampi(f2i(floorf(mn.x)), 0, maxDim[0]), clampi(f2i(floorf(mn.y)), 0, maxDim[1]), clampi(f2i(floorf(mn.z)), 0, maxDim[2])};
    int hi[3] = {clampi(f2i(ceilf(mx.x)), 0, maxDim[0]), clampi(f2i(ceilf(mx.y)), 0, maxDim[1]), clampi(f2i(ceilf(mx.z)), 0, maxDim[2])};
    float col0[3] = {c0[0] / 255.0f, c0[1] / 255.0f, c0[2] / 255.0f};
    float col1[3] = {c1[0] / 255.0f, c1[1] / 255.0f, c1[2] / 255.0f};
    float col2[3] = {c2[0] / 255.0f, c2[1] / 255.0f, c2[2] / 255.0f};
    const size_t cap = 1024 * 256; // VOXELIZE_BUFFER_MAX (WordBuilder.cs:37)
    size_t written = 0;
    V3 p0 = b - a, p1 = c - a;
    for (int x = lo[0]; x <= hi[0]; x++)
        for (int z = lo[2]; z <= hi[2]; z++)
            for (int y = lo[1]; y <= hi[1]; y++) {
                V3 voxel = {(float)x + 0.5f, (float)y + 0.5f, (float)z + 0.5f};
                float d = dot(voxel - a, n);
                if (fabsf(d) > 0.5f) continue;
                V3 p = voxel - n * d;
                V3 p2 = p - a;
                float d00 = dot(p0, p0), d01 = dot(p0, p1), d11 = dot(p1, p1), d20 = dot(p2, p0), d21 = dot(p2, p1);
                float denom = 1.0f / (d00 * d11 - d01 * d01);
                float by = (d11 * d20 - d01 * d21) * denom;
                float bz = (d00 * d21 - d01 * d20) * denom;
                float bx = 1.0f - by - bz;
                if (bx < 0 || by < 0 || bz < 0 || bx > 1 || by > 1 || bz > 1) continue;
                float cr = col0[0] * bx + col1[0] * by + col2[0] * bz;
                float cg = col0[1] * bx + col1[1] * by + col2[1] * bz;
                float cb = col0[2] * bx + col1[2] * by + col2[2] * bz;
                uint32_t argb = 255u | ((uint32_t)to_byte(cr) << 8) | ((uint32_t)to_byte(cg) << 16) | ((uint32_t)to_byte(cb) << 24);
                out.push_back(MeshVoxel{x * (maxDim[2] + 1) + z, (int16_t)y, argb});
                if (++written == cap) return;
            }
}

inline uint32_t hash32(uint32_t x) { x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16; return x; }
inline float hash01(uint32_t x) { return (hash32(x) >> 8) * (1.0f / 16777216.0f); }

} // namespace

namespace {

// ---- synthetic kind 0: fBm value-noise heightmap shell (SURVEY.md §8(d) config 2) -------------------
float value_noise(uint32_t seed, float x, float z) {
    int xi = (int)floorf(x), zi = (int)floorf(z);
    float fx = x - xi, fz = z - zi;
    auto g = [&](int a, int b) { return hash01(seed ^ hash32((uint32_t)a * 0x9e3779b1u + hash32((uint32_t)b + 0x85ebca6bu))); };
    float sx = fx * fx * (3 - 2 * fx), sz = fz * fz * (3 - 2 * fz);
    float v00 = g(xi, zi), v10 = g(xi + 1, zi), v01 = g(xi, zi + 1), v11 = g(xi + 1, zi + 1);
    float a = v00 + sx * (v10 - v00), b = v01 + sx * (v11 - v01);
    return a + sz * (b - a);
}
void build_heightmap(cvx_world_builder* b) {
    const int X = b->dims[0], Y = b->dims[1], Z = b->dims[2];
    b->height.assign((size_t)X * Z, 0);
    const float lo = Y * (64.0f / 2048.0f), hi = Y * (1536.0f / 2048.0f);
    run_parallel(X, b->nThreads, [&](int64_t x, int) {
        for (int z = 0; z < Z; z++) {
            float amp = 1.0f, freq = 4.0f / (float)std::max(X, Z), sum = 0, norm = 0;
            for (int o = 0; o < 6; o++) {
                sum += amp * value_noise(b->seed + 101u * o, x * freq, z * freq);
                norm += amp; amp *= 0.5f; freq *= 2.0f;
            }
            float v = sum / norm;                     // ~[0,1], concentrated near 0.5
            v = (v - 0.5f) * 1.9f + 0.5f;             // widen
            v = v < 0 ? 0 : (v > 1 ? 1 : v);
            int h = (int)(lo + v * (hi - lo));
            b->height[(size_t)x * Z + z] = (uint16_t)clampi(h, 1, Y - 1);
        }
    });
}
inline uint32_t terrain_color(uint32_t seed, int x, int y, int z, int dimY) {
    float t = (float)y / (float)dimY;
    float r, g, bl;
    if (t < 0.18f) { r = 194; g = 178; bl = 128; }       // sand
    else if (t < 0.42f) { r = 70; g = 140; bl = 60; }    // grass
    else if (t < 0.6f) { r = 100; g = 95; bl = 85; }     // rock
    else { r = 235; g = 235; bl = 240; }                 // snow
    int j = (int)(hash32(seed ^ (uint32_t)(x * 73856093) ^ (uint32_t)(y * 19349663) ^ (uint32_t)(z * 83492791)) & 31) - 16;
    auto c = [&](float v) { return (uint32_t)clampi((int)v + j, 0, 255); };
    return 255u | (c(r) << 8) | (c(g) << 16) | (c(bl) << 24);
}

// ---- synthetic kind 1: boxes / pipes / slabs (config 4) ------------------------------------------------
void build_structures(cvx_world_builder* b) {
    const int X = b->dims[0], Y = b->dims[1], Z = b->dims[2];
    uint32_t s = b->seed * 2654435761u + 12345u;
    auto rnd = [&]() { s = hash32(s + 0x9e3779b9u); return s; };
    auto rrange = [&](int lo, int hi) { return lo + (int)(rnd() % (uint32_t)(hi - lo + 1)); };
    // floor slabs: 3 levels covering large areas
    int nSlabs = std::max(4, (X / 512) * (Z / 512));
    for (int i = 0; i < nSlabs; i++) {
        int w = rrange(X / 8, X / 3), d = rrange(Z / 8, Z / 3);
        int x0 = rrange(0, X - w - 1), z0 = rrange(0, Z - d - 1), y0 = rrange(2, Y / 2);
        b->boxes.push_back({x0, x0 + w, y0, y0 + 1, z0, z0 + d, 255u | (120u << 8) | (120u << 16) | (125u << 24), 0});
    }
    // hollow boxes (buildings / tanks)
    int nBoxes = (int)((int64_t)X * Z / 6000);
    for (int i = 0; i < nBoxes; i++) {
        int w = rrange(12, 96), d = rrange(12, 96), h = rrange(16, std::min(Y - 8, 420));
        int x0 = rrange(0, X - w - 1), z0 = rrange(0, Z - d - 1), y0 = rrange(0, std::max(1, Y - h - 4));
        uint32_t col = 255u | ((uint32_t)rrange(60, 230) << 8) | ((uint32_t)rrange(60, 230) << 16) | ((uint32_t)rrange(60, 230) << 24);
        b->boxes.push_back({x0, x0 + w, y0, y0 + h, z0, z0 + d, col, 1});
    }
    // pipes: long thin axis-aligned hollow tubes (square cross-section shell)
    int nPipes = (int)((int64_t)X * Z / 9000);
    for (int i = 0; i < nPipes; i++) {
        int len = rrange(100, std::min(X, Z) / 2), rad = rrange(2, 9), y0 = rrange(4, Y - 2 * rad - 4);
        uint32_t col = 255u | ((uint32_t)rrange(120, 255) << 8) | ((uint32_t)rrange(80, 200) << 16) | ((uint32_t)rrange(40, 120) << 24);
        if (rnd() & 1) { int x0 = rrange(0, X - len - 1), z0 = rrange(0, Z - 2 * rad - 1); b->boxes.push_back({x0, x0 + len, y0, y0 + 2 * rad, z0, z0 + 2 * rad, col, 1}); }
        else { int z0 = rrange(0, Z - len - 1), x0 = rrange(0, X - 2 * rad - 1); b->boxes.push_back({x0, x0 + 2 * rad, y0, y0 + 2 * rad, z0, z0 + len, col, 1}); }
    }
    b->binShift = 6;
    b->binsX = (X >> b->binShift) + 1; b->binsZ = (Z >> b->binShift) + 1;
    b->boxBins.assign((size_t)b->binsX * b->binsZ, {});
    for (int i = 0; i < (int)b->boxes.size(); i++) {
        auto& q = b->boxes[i];
        for (int bx = q.x0 >> b->binShift; bx <= q.x1 >> b->binShift; bx++)
            for (int bz = q.z0 >> b->binShift; bz <= q.z1 >> b->binShift; bz++)
                b->boxBins[(size_t)bx * b->binsZ + bz].push_back(i);
    }
}

// Emit the voxels of LOD-0 column (x,z) into the accumulator.
void emit_column(const cvx_world_builder* b, int x, int z, YAccumulator& acc) {
    const int Y = b->dims[1], Z = b->dims[2];
    if (b->synthKind == 0) {
        const int X = b->dims[0];
        auto H = [&](int xx, int zz) { return (int)b->height[(size_t)clampi(xx, 0, X - 1) * Z + clampi(zz, 0, Z - 1)]; };
        int h = H(x, z);
        int lo = std::min(std::min(H(x - 1, z), H(x + 1, z)), std::min(H(x, z - 1), H(x, z + 1)));
        lo = std::max(0, std::min(lo, h) - 1);
        for (int y = lo; y <= h; y++) acc.add(y, terrain_color(b->seed, x, y, z, Y));
    } else if (b->synthKind == 1) {
        // ground plane: 2 voxels thick
        for (int y = 0; y < 2; y++) acc.add(y, terrain_color(b->seed, x, y * 40, z, 256));
        const auto& bin = b->boxBins[(size_t)(x >> b->binShift) * b->binsZ + (z >> b->binShift)];
        for (int bi : bin) {
            const auto& q = b->boxes[bi];
            if (x < q.x0 || x > q.x1 || z < q.z0 || z > q.z1) continue;
            int j = (int)(hash32(b->seed ^ (uint32_t)(x * 73856093) ^ (uint32_t)(z * 83492791) ^ (uint32_t)bi) & 15) - 8;
            auto shade = [&](uint32_t c, int yy) {
                int k = j + ((yy >> 2) & 1) * 6;
                uint32_t r = (uint32_t)clampi((int)((c >> 8) & 255) + k, 0, 255), g = (uint32_t)clampi((int)((c >> 16) & 255) + k, 0, 255), bl = (uint32_t)clampi((int)((c >> 24) & 255) + k, 0, 255);
                return 255u | (r << 8) | (g << 16) | (bl << 24);
            };
            bool wall = (q.kind == 0) || x == q.x0 || x == q.x1 || z == q.z0 || z == q.z1;
            if (wall) { for (int y = q.y0; y <= std::min(q.y1, Y - 1); y++) if (acc.n[y] == 0) acc.add(y, shade(q.color, y)); }
            else {
                if (acc.n[q.y0] == 0) acc.add(q.y0, shade(q.color, q.y0));
                int yt = std::min(q.y1, Y - 1);
                if (acc.n[yt] == 0) acc.add(yt, shade(q.color, yt));
            }
        }
    } else {
        int64_t idx = (int64_t)x * Z + z;
        for (int64_t i = b->colStart[idx]; i < b->colStart[idx + 1]; i++) acc.add(b->voxels[i].y, b->voxels[i].argb);
    }
}

// World.DownSamplePartial (World.cs:101-127): decode a LOD-0 column of the blob into the accumulator at Y >> nextLod.
void emit_downsampled(const Blob& lod0, int dimY, int dimZ, int x, int z, int nextLod, YAccumulator& acc) {
    const ColHeader* headers = (const ColHeader*)lod0.bytes.data();
    const uint32_t* elements = (const uint32_t*)(lod0.bytes.data() + 12 * (int64_t)lod0.columnCount);
    const ColHeader& h = headers[(int64_t)x * dimZ + z];
    if (h.runCount == 0) return;
    const uint32_t* base = elements + h.offset;
    const uint32_t* colors = base + h.runCount + 2;
    int top = dimY; // elementBounds = dimensions.y >> lod (lod 0)
    for (int run = 0; run < h.runCount; run++) {
        Run e; memcpy(&e, base + 1 + run, 4);
        // the 16 bits of Length as the count finalize_column wrote: a run of 32768 voxels (a full column of a 32768-high world)
        // is stored as int16 -32768
        const int length = (uint16_t)e.length;
        int bottom = top - length;
        if (e.colorsIndex >= 0)
            for (int i = 0; i < length; i++) acc.add((bottom + i) >> nextLod, colors[e.colorsIndex + length - i - 1]);
        top = bottom;
    }
}

int build_lod(cvx_world_builder* b, int lod) {
    Blob& blob = b->lods[lod];
    if (blob.built) return CVX_OK;
    if (b->deviceBuilt) return CVX_ERR_INVALID_ARGUMENT; // a device-built world holds exactly the LODs it was asked for
    if (lod > 0 && !b->lods[0].built) { int r = build_lod(b, 0); if (r) return r; }
    const int X = b->dims[0], Y = b->dims[1], Z = b->dims[2];
    const int cx = X >> lod, cz = Z >> lod;
    const int64_t nCols = (int64_t)cx * cz;
    const int columnCount = (int)(((int64_t)X * Z) / ((int64_t)(lod + 1) * (lod + 1))); // World.ColumnCount quirk (World.cs:17)
    const int64_t nChunks = (nCols + CHUNK_COLUMNS - 1) / CHUNK_COLUMNS;
    std::vector<Chunk> chunks((size_t)nChunks);
    std::vector<int64_t> firstSlot((size_t)nChunks);
    const int voxelScale = 1 << lod, topY = (Y >> lod) - 1, step = 1 << lod;
    int nt = b->nThreads <= 0 ? (int)std::thread::hardware_concurrency() : b->nThreads;
    if (nt < 1) nt = 1;
    std::vector<YAccumulator> accs((size_t)nt);
    run_parallel(nChunks, nt, [&](int64_t ci, int t) {
        YAccumulator& acc = accs[t];
        Chunk& ch = chunks[ci];
        std::vector<Run> runs; std::vector<uint32_t> colors;
        int64_t c0 = ci * CHUNK_COLUMNS, c1 = std::min(nCols, c0 + CHUNK_COLUMNS);
        firstSlot[ci] = c0;
        ch.headers.resize((size_t)(c1 - c0));
        for (int64_t c = c0; c < c1; c++) {
            int lx = (int)(c / cz), lz = (int)(c % cz);
            acc.reset(Y >> lod);
            if (lod == 0) emit_column(b, lx, lz, acc);
            else
                for (int ix = 0; ix < step; ix++)
                    for (int iz = 0; iz < step; iz++) emit_downsampled(b->lods[0], Y, Z, lx * step + ix, lz * step + iz, lod, acc);
            finalize_column(acc, voxelScale, topY, ch, ch.headers[(size_t)(c - c0)], runs, colors);
        }
    });
    assemble_blob(blob, columnCount, columnCount, chunks, firstSlot, nullptr);
    return CVX_OK;
}

} // namespace

int cvxh_remap_mesh(const float* positions, int32_t n_vertices, int32_t max_dimension, const int32_t flips[3],
                    std::vector<float>& out_xyz, int dims[3]) {
    if (!positions || n_vertices < 3 || max_dimension < 1) return CVX_ERR_INVALID_ARGUMENT;
    std::vector<V3> v((size_t)n_vertices);
    for (int i = 0; i < n_vertices; i++) v[i] = {positions[3 * i], positions[3 * i + 1], positions[3 * i + 2]};
    // SimpleMesh.Remap_Internal, SimpleMesh.cs:64-106
    V3 mn = v[0], mx = v[0];
    for (int i = 1; i < n_vertices; i++) {
        mn = {std::min(v[i].x, mn.x), std::min(v[i].y, mn.y), std::min(v[i].z, mn.z)};
        mx = {std::max(v[i].x, mx.x), std::max(v[i].y, mx.y), std::max(v[i].z, mx.z)};
    }
    V3 size = mx - mn;
    float scale = (float)max_dimension / std::max(size.x, std::max(size.y, size.z));
    dims[0] = next_pow2((int)(size.x * scale)); dims[1] = next_pow2((int)(size.y * scale)); dims[2] = next_pow2((int)(size.z * scale));
    for (auto& p : v) p = (p - mn) * scale;
    if (flips && flips[0]) for (auto& p : v) p.x = (float)dims[0] - p.x;
    if (flips && flips[1]) for (auto& p : v) p.y = (float)dims[1] - p.y;
    if (flips && flips[2]) for (auto& p : v) p.z = (float)dims[2] - p.z;
    if (dims[0] < 1 || dims[1] < 1 || dims[2] < 1 || dims[1] > 32768) return CVX_ERR_INVALID_ARGUMENT;
    out_xyz.resize(3 * (size_t)n_vertices);
    for (int i = 0; i < n_vertices; i++) { out_xyz[3 * (size_t)i] = v[i].x; out_xyz[3 * (size_t)i + 1] = v[i].y; out_xyz[3 * (size_t)i + 2] = v[i].z; }
    return CVX_OK;
}

extern "C" {

void cvx_host_free(void* p) { free(p); }

int cvx_obj_parse(const char* path, int32_t swap_yz, float** out_positions, uint8_t** out_colors32, int32_t* out_n_vertices) {
    if (!path || !out_positions || !out_colors32 || !out_n_vertices) return CVX_ERR_INVALID_ARGUMENT;
    FILE* f = fopen(path, "r");
    if (!f) return CVX_ERR_IO;
    std::vector<float> lutPos; std::vector<uint8_t> lutCol;
    std::vector<float> pos; std::vector<uint8_t> col;
    char line[4096];
    while (fgets(line, sizeof line, f)) {
        size_t n = strlen(line);
        while (n && (line[n - 1] == '\n' || line[n - 1] == '\r')) line[--n] = 0;
        if (n == 0) continue;
        if (line[0] == 'v' && line[1] == ' ') { // ParsePositionLine, ObjModel.cs:60-80
            float v[6]; int got = 0; char* p = line + 2;
            while (got < 6) { while (*p == ' ') p++; if (!*p) break; char* e; v[got] = strtof(p, &e); if (e == p) break; got++; p = e; }
            if (got < 3) { fclose(f); return CVX_ERR_FORMAT; }
            float x = v[0], y = v[1], z = v[2];
            if (swap_yz) std::swap(y, z);
            lutPos.push_back(x); lutPos.push_back(y); lutPos.push_back(z);
            if (got >= 6) { lutCol.push_back(to_byte(v[3])); lutCol.push_back(to_byte(v[4])); lutCol.push_back(to_byte(v[5])); lutCol.push_back(255); }
            else { lutCol.push_back(255); lutCol.push_back(255); lutCol.push_back(255); lutCol.push_back(255); }
        } else if (line[0] == 'f' && line[1] == ' ') { // ParseFaceLine :87-133 — first three corners only
            char* p = line + 2;
            for (int i = 0; i < 3; i++) {
                while (*p == ' ') p++;
                long idx = strtol(p, &p, 10) - 1; // ParseFaceIndex :173-196
                while (*p && *p != ' ') p++;      // skip /vt/vn
                if (idx < 0 || (size_t)idx * 3 + 2 >= lutPos.size()) { fclose(f); return CVX_ERR_FORMAT; }
                for (int k = 0; k < 3; k++) pos.push_back(lutPos[(size_t)idx * 3 + k]);
                for (int k = 0; k < 4; k++) col.push_back(lutCol[(size_t)idx * 4 + k]);
            }
        }
    }
    fclose(f);
    int nv = (int)(pos.size() / 3);
    *out_positions = (float*)malloc(std::max<size_t>(1, pos.size() * sizeof(float)));
    *out_colors32 = (uint8_t*)malloc(std::max<size_t>(1, col.size()));
    memcpy(*out_positions, pos.data(), pos.size() * sizeof(float));
    memcpy(*out_colors32, col.data(), col.size());
    *out_n_vertices = nv;
    return CVX_OK;
}

int cvx_builder_from_mesh(const float* positions, const uint8_t* colors32, int32_t n_vertices, int32_t max_dimension,
                          const int32_t flips[3], int32_t n_threads, cvx_world_builder** out) {
    if (!positions || !colors32 || n_vertices < 3 || max_dimension < 1 || !out) return CVX_ERR_INVALID_ARGUMENT;
    std::vector<float> xyz;
    int dims[3];
    int rr = cvxh_remap_mesh(positions, n_vertices, max_dimension, flips, xyz, dims);
    if (rr) return rr;
    std::vector<V3> v((size_t)n_vertices);
    for (int i = 0; i < n_vertices; i++) v[i] = {xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2]};

    cvx_world_builder* b = new cvx_world_builder();
    b->dims[0] = dims[0]; b->dims[1] = dims[1]; b->dims[2] = dims[2];
    b->nThreads = n_threads;
    // WorldBuilder.Import, WordBuilder.cs:39-97 (triangle-parallel); per-thread voxel lists, then a counting sort by column
    int nt = n_threads <= 0 ? (int)std::thread::hardware_concurrency() : n_threads;
    if (nt < 1) nt = 1;
    const int maxDim[3] = {dims[0] - 1, dims[1] - 1, dims[2] - 1};
    std::vector<std::vector<MeshVoxel>> lists((size_t)nt);
    run_parallel(n_vertices / 3, nt, [&](int64_t tri, int t) {
        voxelize_triangle(v[3 * tri], v[3 * tri + 1], v[3 * tri + 2], colors32 + 12 * tri, colors32 + 12 * tri + 4, colors32 + 12 * tri + 8, maxDim, lists[t]);
    });
    const int64_t nCols = (int64_t)dims[0] * dims[2];
    b->colStart.assign((size_t)nCols + 1, 0);
    for (auto& l : lists) for (auto& mv : l) b->colStart[(size_t)mv.xz + 1]++;
    for (int64_t i = 0; i < nCols; i++) b->colStart[i + 1] += b->colStart[i];
    b->voxels.resize((size_t)b->colStart[nCols]);
    std::vector<int64_t> cursor(b->colStart.begin(), b->colStart.end() - 1);
    for (auto& l : lists) { for (auto& mv : l) b->voxels[(size_t)cursor[mv.xz]++] = mv; std::vector<MeshVoxel>().swap(l); }
    *out = b;
    return CVX_OK;
}

int cvx_builder_synthetic(int32_t kind, int32_t dim_x, int32_t dim_y, int32_t dim_z, uint32_t seed, int32_t n_threads, cvx_world_builder** out) {
    auto pow2 = [](int n) { return n > 0 && (n & (n - 1)) == 0; };
    if (!out || kind < 0 || kind > 1 || !pow2(dim_x) || !pow2(dim_y) || !pow2(dim_z) || dim_y > 32768) return CVX_ERR_INVALID_ARGUMENT;
    cvx_world_builder* b = new cvx_world_builder();
    b->dims[0] = dim_x; b->dims[1] = dim_y; b->dims[2] = dim_z;
    b->nThreads = n_threads; b->synthKind = kind; b->seed = seed;
    if (kind == 0) build_heightmap(b); else build_structures(b);
    *out = b;
    return CVX_OK;
}

int cvx_builder_dims(const cvx_world_builder* b, int32_t out_dims[3]) {
    if (!b || !out_dims) return CVX_ERR_INVALID_ARGUMENT;
    out_dims[0] = b->dims[0]; out_dims[1] = b->dims[1]; out_dims[2] = b->dims[2];
    return CVX_OK;
}

int cvx_builder_lod(cvx_world_builder* b, int32_t lod, const void** out_blob, int64_t* out_bytes, int32_t* out_column_count, int64_t* out_voxel_count) {
    if (!b || lod < 0 || lod >= CVX_LOD_LEVELS) return CVX_ERR_INVALID_ARGUMENT;
    if ((b->dims[0] >> lod) < 1 || (b->dims[2] >> lod) < 1 || (b->dims[1] >> lod) < 1) return CVX_ERR_INVALID_ARGUMENT;
    int r = build_lod(b, lod);
    if (r) return r;
    if (out_blob) *out_blob = b->lods[lod].bytes.data();
    if (out_bytes) *out_bytes = (int64_t)b->lods[lod].bytes.size();
    if (out_column_count) *out_column_count = b->lods[lod].columnCount;
    if (out_voxel_count) *out_voxel_count = b->lods[lod].voxelCount;
    return CVX_OK;
}

void cvx_builder_free(cvx_world_builder* b) { delete b; }

// WorldSaveFile.Serialize, WorldSaveFile.cs:8-55: 24-byte header, (offset,length) int64 pairs, raw blobs.
int cvx_world_file_write(const char* path, const int32_t dims[3], int32_t world_count, const void* const* blobs, const int64_t* blob_bytes) {
    if (!path || !dims || world_count < 1 || world_count > CVX_LOD_LEVELS || !blobs || !blob_bytes) return CVX_ERR_INVALID_ARGUMENT;
    FILE* f = fopen(path, "wb");
    if (!f) return CVX_ERR_IO;
    int64_t empty = 0;
    int32_t hdr[4] = {dims[0], dims[1], dims[2], world_count};
    bool ok = fwrite(&empty, 8, 1, f) == 1 && fwrite(hdr, 4, 4, f) == 4;
    int64_t off = 24 + 16 * (int64_t)world_count;
    for (int i = 0; i < world_count && ok; i++) { int64_t pair[2] = {off, blob_bytes[i]}; ok = fwrite(pair, 8, 2, f) == 2; off += blob_bytes[i]; }
    for (int i = 0; i < world_count && ok; i++) ok = blob_bytes[i] == 0 || fwrite(blobs[i], 1, (size_t)blob_bytes[i], f) == (size_t)blob_bytes[i];
    fclose(f);
    return ok ? CVX_OK : CVX_ERR_IO;
}

// WorldSaveFile.Deserialize, WorldSaveFile.cs:57-94
int cvx_world_file_read(const char* path, int32_t out_dims[3], int32_t* out_world_count, void** out_blobs, int64_t* out_blob_bytes) {
    if (!path || !out_dims || !out_world_count || !out_blobs || !out_blob_bytes) return CVX_ERR_INVALID_ARGUMENT;
    FILE* f = fopen(path, "rb");
    if (!f) return CVX_ERR_IO;
    int64_t empty; int32_t hdr[4];
    if (fread(&empty, 8, 1, f) != 1 || fread(hdr, 4, 4, f) != 4) { fclose(f); return CVX_ERR_FORMAT; }
    if (hdr[3] < 1 || hdr[3] > CVX_LOD_LEVELS || hdr[0] < 1 || hdr[1] < 1 || hdr[2] < 1) { fclose(f); return CVX_ERR_FORMAT; }
    int64_t table[2 * CVX_LOD_LEVELS];
    if (fread(table, 16, (size_t)hdr[3], f) != (size_t)hdr[3]) { fclose(f); return CVX_ERR_FORMAT; }
    for (int i = 0; i < CVX_LOD_LEVELS; i++) { out_blobs[i] = nullptr; out_blob_bytes[i] = 0; }
    // an error in the middle of the file hands nothing out: the blobs read so far are freed again
    auto bail = [&](int code) {
        for (int i = 0; i < CVX_LOD_LEVELS; i++) { free(out_blobs[i]); out_blobs[i] = nullptr; out_blob_bytes[i] = 0; }
        fclose(f);
        return code;
    };
    for (int i = 0; i < hdr[3]; i++) {
        int64_t off = table[2 * i], len = table[2 * i + 1];
        if (off < 0 || len < 0 || fseek(f, (long)off, SEEK_SET) != 0) return bail(CVX_ERR_FORMAT);
        void* p = malloc((size_t)std::max<int64_t>(1, len));
        if (!p) return bail(CVX_ERR_OUT_OF_MEMORY);
        if (fread(p, 1, (size_t)len, f) != (size_t)len) { free(p); return bail(CVX_ERR_FORMAT); }
        out_blobs[i] = p; out_blob_bytes[i] = len;
    }
    fclose(f);
    out_dims[0] = hdr[0]; out_dims[1] = hdr[1]; out_dims[2] = hdr[2];
    *out_world_count = hdr[3];
    return CVX_OK;
}

// Presentation helper: a ColorARGB32 frame (bytes a,r,g,b; row 0 = bottom) as an uncompressed 32-bit BMP. BMP rows are stored
// bottom-up and its pixels are B,G,R,A bytes, so every pixel is the byte reversal of ours and rows keep their order.
int cvx_host_write_bmp(const char* path, const void* argb_frame, int32_t width, int32_t height) {
    if (!path || !argb_frame || width < 1 || height < 1) return CVX_ERR_INVALID_ARGUMENT;
    FILE* f = fopen(path, "wb");
    if (!f) return CVX_ERR_IO;
    const uint32_t pixelBytes = (uint32_t)width * (uint32_t)height * 4u;
    uint8_t hdr[54] = {0};
    auto put32 = [&](int at, uint32_t v) { hdr[at] = (uint8_t)v; hdr[at + 1] = (uint8_t)(v >> 8); hdr[at + 2] = (uint8_t)(v >> 16); hdr[at + 3] = (uint8_t)(v >> 24); };
    hdr[0] = 'B'; hdr[1] = 'M';
    put32(2, 54u + pixelBytes); put32(10, 54u);
    put32(14, 40u); put32(18, (uint32_t)width); put32(22, (uint32_t)height);
    hdr[26] = 1; hdr[28] = 32;             // planes, bits per pixel; compression 0 = BI_RGB
    put32(34, pixelBytes); put32(38, 2835u); put32(42, 2835u);
    bool ok = fwrite(hdr, 1, 54, f) == 54;
    std::vector<uint32_t> line((size_t)width);
    const uint32_t* src = (const uint32_t*)argb_frame;
    for (int y = 0; y < height && ok; y++) {
        for (int x = 0; x < width; x++) line[(size_t)x] = __builtin_bswap32(src[(size_t)y * width + x]);
        ok = fwrite(line.data(), 4, (size_t)width, f) == (size_t)width;
    }
    fclose(f);
    return ok ? CVX_OK : CVX_ERR_IO;
}

} // extern "C"
