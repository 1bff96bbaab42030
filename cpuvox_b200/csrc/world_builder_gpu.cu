/*
 * world_builder_gpu.cu — world production on the device (SURVEY.md §8(f) rank 2): the step BEFORE the hot path.
 *
 *   triangles --voxelize--> (column, y, colour) records --sort + merge--> unique voxels --RLE per column--> LOD-0 blob
 *                                                              unique LOD-0 voxels --re-key (>> j), sort + merge, RLE--> LOD-j blob
 *
 * Replaces, for hosts that want it, WorldBuilder.Import + VoxelizerHelper.GetVoxelsInternal (Assets/Code/WordBuilder.cs:39-97,
 * Assets/Code/VoxelizerHelper.cs:28-132), RLEColumnBuilder.ToFinalColumn + the RLEColumn ctor (WordBuilder.cs:181-268,
 * Assets/Code/World.cs:190-234) and World.DownSample (World.cs:45-127). The result is the SAME bytes the host builder
 * (world_builder.cpp) produces: the reference's WorldAllocator blob (World.cs:285-313) with columns allocated in index order.
 *
 * Not a translation: the reference appends voxels to per-column lists under a lock, sorts each list and dedupes it, and
 * downsamples by decoding 2^j x 2^j columns. Here every stage is a flat data-parallel pass over records keyed
 * (column << 16 | y): a radix sort brings equal keys together, a segmented merge averages them (sum / count per channel — the
 * reference's (first + sum of the others) / count, order independent), and one thread per column turns its slice of the
 * sorted unique voxels into runs. LOD j re-keys the unique LOD-0 voxels with (x >> j, z >> j, y >> j) and runs the same passes.
 * Sort and scan are CUB device primitives (library code); the voxelizer, merge and RLE kernels are ours.
 * Arithmetic: IEEE fp32, no FMA contraction (-fmad=false), the reference's expression order — voxel sets and colours are
 * bit-identical to the host builder's (tests/test_gpu_parity.py::test_gpu_world_builder_matches_host_builder).
 */
#include <cuda_runtime.h>
#include <cub/cub.cuh>

#include <algorithm>
#include <climits>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

#include "world_builder.h"

namespace {

#define VOXELIZE_BUFFER_MAX (1024 * 256) /* WordBuilder.cs:37 */

struct V3 { float x, y, z; };
__device__ __forceinline__ V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
__device__ __forceinline__ V3 operator*(V3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
__device__ __forceinline__ float dot3(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ V3 cross3(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
__device__ __forceinline__ V3 normalize3(V3 a) { float r = 1.0f / sqrtf(dot3(a, a)); return a * r; }
__device__ __forceinline__ int clampi(int x, int a, int b) { return max(a, min(b, x)); }
__device__ __forceinline__ int f2i_x64(float f) { if (!(f >= -2147483648.0f && f < 2147483648.0f)) return INT_MIN; return (int)f; } // cvttss2si
__device__ __forceinline__ uint32_t to_byte(float c) { // Color -> Color32: round(clamp01(c) * 255), half to even; NaN -> 0
    float v = c > 0.0f ? (c < 1.0f ? c : 1.0f) : 0.0f;
    return (uint32_t)rintf(v * 255.0f) & 0xffu;
}

// Per-triangle constants of VoxelizerHelper.GetVoxelsInternal (:28-66): expanded corners, normal, AABB, vertex colours.
struct Tri {
    V3 a, n, p0, p1;
    int lo[3], hi[3];
    float col0[3], col1[3], col2[3];
    float d00, d01, d11, denom;
    bool degenerate;
};

__device__ void tri_setup(const float* __restrict__ xyz, const uint8_t* __restrict__ colors, int64_t tri, int mx, int my, int mz, Tri& t) {
    const float* p = xyz + 9 * tri;
    V3 a = {p[0], p[1], p[2]}, b = {p[3], p[4], p[5]}, c = {p[6], p[7], p[8]};
    V3 nc = cross3(b - a, c - a);
    float l2 = dot3(nc, nc);
    t.degenerate = l2 == 0.0f;
    if (t.degenerate) return;
    t.n = nc * (1.0f / sqrtf(l2));
    V3 mid = (a + b + c) * 1.0f; mid = {mid.x / 3.0f, mid.y / 3.0f, mid.z / 3.0f};
    a = a + normalize3(a - mid) * 0.5f;   // corners pushed outwards by half a voxel (:44-46)
    b = b + normalize3(b - mid) * 0.5f;
    c = c + normalize3(c - mid) * 0.5f;
    // fminf / fmaxf ignore a NaN corner (math.min / math.max of the reference; DESIGN.md §3.4)
    V3 mn = {fminf(a.x, fminf(b.x, c.x)), fminf(a.y, fminf(b.y, c.y)), fminf(a.z, fminf(b.z, c.z))};
    V3 mxv = {fmaxf(a.x, fmaxf(b.x, c.x)), fmaxf(a.y, fmaxf(b.y, c.y)), fmaxf(a.z, fmaxf(b.z, c.z))};
    t.lo[0] = clampi(f2i_x64(floorf(mn.x)), 0, mx); t.lo[1] = clampi(f2i_x64(floorf(mn.y)), 0, my); t.lo[2] = clampi(f2i_x64(floorf(mn.z)), 0, mz);
    t.hi[0] = clampi(f2i_x64(ceilf(mxv.x)), 0, mx); t.hi[1] = clampi(f2i_x64(ceilf(mxv.y)), 0, my); t.hi[2] = clampi(f2i_x64(ceilf(mxv.z)), 0, mz);
    const uint8_t* q = colors + 12 * tri;
    for (int k = 0; k < 3; k++) { t.col0[k] = q[k] / 255.0f; t.col1[k] = q[4 + k] / 255.0f; t.col2[k] = q[8 + k] / 255.0f; }
    t.a = a; t.p0 = b - a; t.p1 = c - a;
    t.d00 = dot3(t.p0, t.p0); t.d01 = dot3(t.p0, t.p1); t.d11 = dot3(t.p1, t.p1);
    t.denom = 1.0f / (t.d00 * t.d11 - t.d01 * t.d01);
}

// The per-voxel test and colour of :68-131. Returns false when the voxel is not part of the triangle.
__device__ __forceinline__ bool voxel_test(const Tri& t, int x, int y, int z, uint32_t& argb) {
    V3 voxel = {(float)x + 0.5f, (float)y + 0.5f, (float)z + 0.5f};
    float d = dot3(voxel - t.a, t.n);
    if (fabsf(d) > 0.5f) return false;
    V3 p = voxel - t.n * d;
    V3 p2 = p - t.a;
    float d20 = dot3(p2, t.p0), d21 = dot3(p2, t.p1);
    float by = (t.d11 * d20 - t.d01 * d21) * t.denom;
    float bz = (t.d00 * d21 - t.d01 * d20) * t.denom;
    float bx = 1.0f - by - bz;
    if (bx < 0 || by < 0 || bz < 0 || bx > 1 || by > 1 || bz > 1) return false;
    float cr = t.col0[0] * bx + t.col1[0] * by + t.col2[0] * bz;
    float cg = t.col0[1] * bx + t.col1[1] * by + t.col2[1] * bz;
    float cb = t.col0[2] * bx + t.col1[2] * by + t.col2[2] * bz;
    argb = 255u | (to_byte(cr) << 8) | (to_byte(cg) << 16) | (to_byte(cb) << 24);
    return true;
}

// One CTA per triangle, threads stride over the cells of its bounding box (y fastest, like the reference's loops).
// EMIT == false: count the voxels of each triangle. EMIT == true: write them at offsets[tri] + (atomic cursor); the order
// inside a triangle is irrelevant, the records are sorted by key next.
template <bool EMIT>
__global__ void __launch_bounds__(256)
voxelize_kernel(const float* __restrict__ xyz, const uint8_t* __restrict__ colors, int64_t nTris, int dimX, int dimY, int dimZ,
                unsigned long long* __restrict__ counts, const unsigned long long* __restrict__ offsets,
                unsigned long long* __restrict__ keys, uint32_t* __restrict__ vals) {
    const int64_t tri = blockIdx.x;
    if (tri >= nTris) return;
    __shared__ Tri t;
    __shared__ unsigned long long cursor;
    if (threadIdx.x == 0) { tri_setup(xyz, colors, tri, dimX - 1, dimY - 1, dimZ - 1, t); cursor = 0ull; }
    __syncthreads();
    if (t.degenerate) { if (!EMIT && threadIdx.x == 0) counts[tri] = 0ull; return; }
    const int ny = t.hi[1] - t.lo[1] + 1, nz = t.hi[2] - t.lo[2] + 1, nx = t.hi[0] - t.lo[0] + 1;
    const int64_t cells = (int64_t)nx * nz * ny;
    unsigned long long mine = 0ull;
    for (int64_t i = threadIdx.x; i < cells; i += blockDim.x) {
        const int y = t.lo[1] + (int)(i % ny);
        const int64_t r = i / ny;
        const int z = t.lo[2] + (int)(r % nz), x = t.lo[0] + (int)(r / nz);
        uint32_t argb;
        if (!voxel_test(t, x, y, z, argb)) continue;
        if (EMIT) {
            const unsigned long long slot = offsets[tri] + atomicAdd(&cursor, 1ull);
            keys[slot] = ((unsigned long long)((int64_t)x * dimZ + z) << 16) | (unsigned long long)y;
            vals[slot] = argb;
        } else mine++;
    }
    if (!EMIT) {
        // block sum of `mine`
        __shared__ unsigned long long warpSums[8];
        for (int o = 16; o > 0; o >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, o);
        if ((threadIdx.x & 31) == 0) warpSums[threadIdx.x >> 5] = mine;
        __syncthreads();
        if (threadIdx.x == 0) { unsigned long long s = 0; for (int w = 0; w < 8; w++) s += warpSums[w]; counts[tri] = s; }
    }
}

// heads[i] = 1 where a new key starts in the sorted record list
__global__ void mark_heads_kernel(const unsigned long long* __restrict__ keys, int64_t n, uint32_t* __restrict__ heads) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) heads[i] = (i == 0 || keys[i] != keys[i - 1]) ? 1u : 0u;
}

// One thread per head: average the records of its key (RLEColumnBuilder dedupe, WordBuilder.cs:203-228: per channel
// (first + sum of the others) / count, alpha of the first — every producer here writes alpha 255).
__global__ void merge_kernel(const unsigned long long* __restrict__ keys, const uint32_t* __restrict__ vals, const uint32_t* __restrict__ rank,
                             int64_t n, unsigned long long* __restrict__ ukeys, uint32_t* __restrict__ ucolors) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long k = keys[i];
    if (i > 0 && keys[i - 1] == k) return;
    uint32_t r = 0, g = 0, b = 0, cnt = 0, a = vals[i] & 0xffu;
    for (int64_t j = i; j < n && keys[j] == k; j++) { const uint32_t v = vals[j]; r += (v >> 8) & 0xffu; g += (v >> 16) & 0xffu; b += v >> 24; cnt++; }
    const int64_t u = (int64_t)rank[i] - 1; // inclusive scan of heads
    ukeys[u] = k;
    ucolors[u] = a | (((r / cnt) & 0xffu) << 8) | (((g / cnt) & 0xffu) << 16) | (((b / cnt) & 0xffu) << 24);
}

// LOD j key of a unique LOD-0 voxel: column (x >> j, z >> j) of the (dimZ >> j)-wide grid, y >> j (World.cs:101-127)
__global__ void rekey_kernel(const unsigned long long* __restrict__ keys0, int64_t n, int dimZ, int lod, unsigned long long* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned long long k = keys0[i];
    const int64_t col = (int64_t)(k >> 16);
    const int y = (int)(k & 0xffffu), x = (int)(col / dimZ), z = (int)(col % dimZ);
    out[i] = ((unsigned long long)((int64_t)(x >> lod) * (dimZ >> lod) + (z >> lod)) << 16) | (unsigned long long)(y >> lod);
}

__device__ __forceinline__ int64_t lower_bound_key(const unsigned long long* __restrict__ keys, int64_t n, unsigned long long v) {
    int64_t lo = 0, hi = n;
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (keys[mid] < v) lo = mid + 1; else hi = mid; }
    return lo;
}

// One thread per column. SIZES: element cells the column needs (0 = empty column). !SIZES: write header + elements.
// ToFinalColumn (WordBuilder.cs:232-268) on the column's slice of the sorted unique voxels, read from the top voxel down:
// [guard][runs, top -> bottom][guard][colours, top first]; run = {ColorsIndex (of its top voxel) | Length << 16}, air = -1.
template <bool SIZES>
__global__ void rle_kernel(const unsigned long long* __restrict__ ukeys, const uint32_t* __restrict__ ucolors, int64_t nVox, int64_t nCols,
                           int topY, int voxelScale, unsigned long long* __restrict__ sizes, const unsigned long long* __restrict__ offsets,
                           uint32_t* __restrict__ headers /* 3 words per column */, uint32_t* __restrict__ elements) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= nCols) return;
    const int64_t begin = lower_bound_key(ukeys, nVox, (unsigned long long)c << 16);
    const int64_t end = lower_bound_key(ukeys, nVox, (unsigned long long)(c + 1) << 16);
    const int count = (int)(end - begin);
    if (count == 0) { if (SIZES) sizes[c] = 0ull; return; }
    // voxel i (0 = top) is record end - 1 - i
    int runCount = 0;
    uint32_t* out = nullptr;
    if (!SIZES) { out = elements + offsets[c]; *out++ = 0u; }
    int top = topY;
    for (int i = 0; i < count;) {
        const int voxelY = (int)(ukeys[end - 1 - i] & 0xffffu);
        const int airFromTop = top - voxelY;
        if (airFromTop > 0) { if (!SIZES) *out++ = 0xffffu | ((uint32_t)(airFromTop & 0xffff) << 16); runCount++; top -= airFromTop; }
        int runLength = 1;
        for (int j = i + 1; j < count; j++) { if (top - (j - i) == (int)(ukeys[end - 1 - j] & 0xffffu)) runLength++; else break; }
        if (!SIZES) *out++ = (uint32_t)(i & 0xffff) | ((uint32_t)(runLength & 0xffff) << 16);
        runCount++;
        top -= runLength;
        i += runLength;
    }
    if (top >= 0) { if (!SIZES) *out++ = 0xffffu | ((uint32_t)((top + 1) & 0xffff) << 16); runCount++; }
    if (SIZES) { sizes[c] = (unsigned long long)(2 + runCount + count); return; }
    *out++ = 0u;
    for (int i = 0; i < count; i++) *out++ = ucolors[end - 1 - i];
    const int yMin = (int)(ukeys[begin] & 0xffffu), yMax = (int)(ukeys[end - 1] & 0xffffu);
    headers[3 * c + 0] = (uint32_t)offsets[c];
    headers[3 * c + 1] = (uint32_t)(runCount & 0xffff) | ((uint32_t)((yMin * voxelScale) & 0xffff) << 16); // worldMin (World.cs:211-226)
    headers[3 * c + 2] = (uint32_t)(((yMax + 1) * voxelScale) & 0xffff);                                  // worldMax
}

struct DeviceBuffers {
    std::vector<void*> all;
    ~DeviceBuffers() { for (void* p : all) cudaFree(p); }
    template <class T> cudaError_t alloc(T** p, size_t n) {
        *p = nullptr;
        cudaError_t e = cudaMalloc((void**)p, std::max<size_t>(n, 1) * sizeof(T));
        if (e == cudaSuccess) all.push_back(*p);
        return e;
    }
    void release(void* p) { for (auto& q : all) if (q == p) { cudaFree(p); q = nullptr; } }
};

#define CK(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) { err = std::string(#expr) + ": " + cudaGetErrorString(e_); return cvx_code(e_); } } while (0)

inline int bits_for(unsigned long long maxKey) { int b = 1; while (b < 64 && (maxKey >> b) != 0ull) b++; return b; }

// records (keys, vals) -> sorted, merged unique voxels (ukeys, ucolors); returns their number in nUnique
int sort_and_merge(DeviceBuffers& mem, unsigned long long* keys, uint32_t* vals, int64_t n, int keyBits, cudaStream_t stream,
                   unsigned long long** ukeys, uint32_t** ucolors, int64_t& nUnique, std::string& err) {
    nUnique = 0; *ukeys = nullptr; *ucolors = nullptr;
    if (n == 0) { CK(mem.alloc(ukeys, 1)); CK(mem.alloc(ucolors, 1)); return CVX_OK; }
    if (n > INT32_MAX) { err = "more than 2^31 voxel records"; return CVX_ERR_INVALID_ARGUMENT; }
    unsigned long long* keys2; uint32_t* vals2; uint32_t* heads; uint32_t* rank;
    CK(mem.alloc(&keys2, (size_t)n)); CK(mem.alloc(&vals2, (size_t)n));
    cub::DoubleBuffer<unsigned long long> dk(keys, keys2);
    cub::DoubleBuffer<uint32_t> dv(vals, vals2);
    size_t tmpBytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, tmpBytes, dk, dv, (int)n, 0, keyBits, stream));
    uint8_t* tmp; CK(mem.alloc(&tmp, tmpBytes));
    CK(cub::DeviceRadixSort::SortPairs(tmp, tmpBytes, dk, dv, (int)n, 0, keyBits, stream));
    mem.release(tmp);
    CK(mem.alloc(&heads, (size_t)n)); CK(mem.alloc(&rank, (size_t)n));
    const unsigned blocks = (unsigned)((n + 255) / 256);
    mark_heads_kernel<<<blocks, 256, 0, stream>>>(dk.Current(), n, heads);
    CK(cudaGetLastError());
    tmpBytes = 0;
    CK(cub::DeviceScan::InclusiveSum(nullptr, tmpBytes, heads, rank, (int)n, stream));
    CK(mem.alloc(&tmp, tmpBytes));
    CK(cub::DeviceScan::InclusiveSum(tmp, tmpBytes, heads, rank, (int)n, stream));
    uint32_t last = 0;
    CK(cudaMemcpyAsync(&last, rank + (n - 1), 4, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    nUnique = (int64_t)last;
    CK(mem.alloc(ukeys, (size_t)nUnique)); CK(mem.alloc(ucolors, (size_t)nUnique));
    merge_kernel<<<blocks, 256, 0, stream>>>(dk.Current(), dv.Current(), rank, n, *ukeys, *ucolors);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(stream));
    mem.release(tmp); mem.release(heads); mem.release(rank); mem.release(keys2); mem.release(vals2);
    return CVX_OK;
}

// sorted unique voxels of one LOD -> blob in the reference layout, copied into `blob`
int encode_lod(DeviceBuffers& mem, const unsigned long long* ukeys, const uint32_t* ucolors, int64_t nVox, int dimX, int dimY, int dimZ, int lod,
               cudaStream_t stream, cvx_lod_blob& blob, const cvxd_lod_sink* sink, std::string& err) {
    const int64_t nCols = (int64_t)(dimX >> lod) * (dimZ >> lod);
    const int columnCount = (int)(((int64_t)dimX * dimZ) / ((int64_t)(lod + 1) * (lod + 1))); // World.ColumnCount (World.cs:17)
    unsigned long long *sizes, *offsets;
    CK(mem.alloc(&sizes, (size_t)nCols + 1)); CK(mem.alloc(&offsets, (size_t)nCols + 1));
    CK(cudaMemsetAsync(sizes + nCols, 0, 8, stream));
    const unsigned blocks = (unsigned)((nCols + 127) / 128);
    const int topY = (dimY >> lod) - 1, voxelScale = 1 << lod;
    rle_kernel<true><<<blocks, 128, 0, stream>>>(ukeys, ucolors, nVox, nCols, topY, voxelScale, sizes, nullptr, nullptr, nullptr);
    CK(cudaGetLastError());
    size_t tmpBytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes, sizes, offsets, (int)(nCols + 1), stream));
    uint8_t* tmp; CK(mem.alloc(&tmp, tmpBytes));
    CK(cub::DeviceScan::ExclusiveSum(tmp, tmpBytes, sizes, offsets, (int)(nCols + 1), stream));
    unsigned long long total = 0;
    CK(cudaMemcpyAsync(&total, offsets + nCols, 8, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    if (total > (unsigned long long)INT32_MAX) { err = "element area exceeds the reference's int32 offsets"; return CVX_ERR_INVALID_ARGUMENT; }
    int64_t capacity = (int64_t)columnCount * 4;      // WorldAllocator: starts at columnCount * 4 elements, doubles until it fits (World.cs:295-373)
    while (capacity < (int64_t)total) capacity = capacity > INT32_MAX / 2 ? INT32_MAX : capacity * 2;
    const size_t bytes = (size_t)(12 * (int64_t)columnCount + 4 * capacity);
    uint8_t* dblob; CK(mem.alloc(&dblob, bytes));
    CK(cudaMemsetAsync(dblob, 0, bytes, stream));
    rle_kernel<false><<<blocks, 128, 0, stream>>>(ukeys, ucolors, nVox, nCols, topY, voxelScale, nullptr, offsets,
                                                    (uint32_t*)dblob, (uint32_t*)(dblob + 12 * (int64_t)columnCount));
    CK(cudaGetLastError());
    blob.columnCount = columnCount; blob.voxelCount = nVox;
    mem.release(tmp); mem.release(sizes); mem.release(offsets);
    if (sink && *sink) {
        // hand the device blob over (the sink takes ownership: the world stays resident, nothing goes through the host)
        CK(cudaStreamSynchronize(stream));
        for (auto& q : mem.all) if (q == dblob) q = nullptr;
        int r = (*sink)(lod, dblob, (int64_t)bytes, columnCount);
        if (r) { err = "installing the device-built LOD failed"; return r; }
        return CVX_OK;
    }
    blob.bytes.resize(bytes);
    CK(cudaMemcpyAsync(blob.bytes.data(), dblob, bytes, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    blob.built = true;
    mem.release(dblob);
    return CVX_OK;
}

// ---- device-side transcode of one LOD blob into the Phase-1 layout (same tables as world_transcode.h builds on the host) -----------
// blob words: 3 per column header {elementOffset, runCount | worldMin << 16, worldMax | pad << 16}, then the element area.
__global__ void transcode_count_kernel(const uint32_t* __restrict__ words, int64_t needCols, int64_t columnCount, int64_t elementCells,
                                       unsigned long long* __restrict__ counts, long long* __restrict__ bad) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= needCols) return;
    const uint32_t w0 = words[3 * i], rc = words[3 * i + 1] & 0xffffu;
    unsigned long long n = 0ull;
    if (rc) {
        const int32_t off = (int32_t)w0;
        if (off < 0 || (int64_t)off + rc + 2 > elementCells) atomicMin(bad, (long long)i); // offsets + run counts must stay inside the element area
        else {
            n = rc + 1ull;
            // the colour table follows the runs (World.cs:185-188): every solid run's ColorsIndex .. ColorsIndex + Length - 1 is gathered
            // from it by Phase 1 (side colours, first/last colour of the caps), so it must stay inside the element area as well
            const int64_t colourCells = elementCells - ((int64_t)off + rc + 2);
            const uint32_t* el = words + 3 * columnCount + off + 1;
            for (uint32_t k = 0; k < rc; k++) {
                const uint32_t e = el[k];
                const int ci = (int)(short)(e & 0xffffu), len = (int)(short)(e >> 16);
                if (len == 0) break;                       // an invalid element ends the column (DrawSegmentRayJob.cs:445-447)
                if (ci >= 0 && (len < 0 || (int64_t)ci + len > colourCells)) { atomicMin(bad, (long long)i); break; }
            }
        }
    }
    counts[i] = n;
}

__global__ void transcode_write_kernel(const uint32_t* __restrict__ words, const uint32_t* __restrict__ elements, int64_t needCols, int lod, int dimY,
                                       const unsigned long long* __restrict__ offsets, uint4* __restrict__ headers, uint2* __restrict__ bounds,
                                       int* __restrict__ irregular) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= needCols) return;
    const uint32_t w0 = words[3 * i], w1 = words[3 * i + 1], w2 = words[3 * i + 2];
    const uint32_t rc = w1 & 0xffffu;
    uint4 h = make_uint4(w0, w1, w2 & 0xffffu, 0u);
    if (rc) {
        const unsigned long long o = offsets[i];
        h.w = (uint32_t)o;
        const int scale = 1 << lod;
        long long y = dimY;
        bool ok = true;
        for (uint32_t k = 0; k < rc; k++) {
            const uint32_t el = elements[(int64_t)(int32_t)w0 + 1 + k];
            const int len = (int)(short)(el >> 16);
            bounds[o + k] = make_uint2((uint32_t)(y < 0 ? 0 : y), el);
            if (len <= 0) ok = false;
            y -= (long long)len * scale;
            if (y < 0) ok = false;
        }
        bounds[o + rc] = make_uint2((uint32_t)(y < 0 ? 0 : y), 0u);
        if (y != 0) ok = false;
        if (!ok) *irregular = 1;
    }
    headers[i] = h;
}

} // namespace

// blob_dev: the whole LOD blob in device memory. Allocates *out_headers (needCols uint4) and *out_bounds; the element area stays
// where it is (blob_dev + 12 * column_count). Returns CVX_ERR_FORMAT with *bad_column set when a column points outside the blob.
int cvxd_transcode_lod_device(cudaStream_t stream, const void* blob_dev, int64_t need_cols, int64_t column_count, int64_t element_cells, int lod, int dim_y,
                              void** out_headers, void** out_bounds, int* out_regular, long long* bad_column, int64_t* launches, std::string& err) {
    *out_headers = nullptr; *out_bounds = nullptr; *out_regular = 0; *bad_column = -1;
    DeviceBuffers mem;
    const uint32_t* words = (const uint32_t*)blob_dev;
    const uint32_t* elements = words + 3 * column_count;
    unsigned long long *counts, *offsets; long long* bad; int* irregular;
    CK(mem.alloc(&counts, (size_t)need_cols + 1)); CK(mem.alloc(&offsets, (size_t)need_cols + 1));
    CK(mem.alloc(&bad, 1)); CK(mem.alloc(&irregular, 1));
    const long long none = LLONG_MAX;
    CK(cudaMemcpyAsync(bad, &none, 8, cudaMemcpyHostToDevice, stream));
    CK(cudaMemsetAsync(irregular, 0, 4, stream));
    CK(cudaMemsetAsync(counts + need_cols, 0, 8, stream));
    const unsigned blocks = (unsigned)((need_cols + 255) / 256);
    transcode_count_kernel<<<blocks, 256, 0, stream>>>(words, need_cols, column_count, element_cells, counts, bad);
    CK(cudaGetLastError());
    size_t tmpBytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes, counts, offsets, (int)(need_cols + 1), stream));
    uint8_t* tmp; CK(mem.alloc(&tmp, tmpBytes));
    CK(cub::DeviceScan::ExclusiveSum(tmp, tmpBytes, counts, offsets, (int)(need_cols + 1), stream));
    long long hostBad = none; unsigned long long total = 0;
    CK(cudaMemcpyAsync(&hostBad, bad, 8, cudaMemcpyDeviceToHost, stream));
    CK(cudaMemcpyAsync(&total, offsets + need_cols, 8, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    if (hostBad != none) { *bad_column = hostBad; err = "column points outside the element area (element offset, run count or a run's colour range)"; return CVX_ERR_FORMAT; }
    void* headers = nullptr; void* bounds = nullptr;
    CK(cudaMalloc(&headers, (size_t)(16 * need_cols)));
    cudaError_t e = cudaMalloc(&bounds, total ? (size_t)total * 8 : 8);
    if (e != cudaSuccess) { cudaFree(headers); err = cudaGetErrorString(e); return cvx_code(e); }
    transcode_write_kernel<<<blocks, 256, 0, stream>>>(words, elements, need_cols, lod, dim_y, offsets, (uint4*)headers, (uint2*)bounds, irregular);
    int hostIrregular = 1;
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(&hostIrregular, irregular, 4, cudaMemcpyDeviceToHost, stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) { cudaFree(headers); cudaFree(bounds); err = cudaGetErrorString(e); return CVX_ERR_CUDA; }
    if (launches) *launches += 2;
    *out_headers = headers; *out_bounds = bounds;
    // `bounds` offsets are 32-bit in the header and y is 16-bit in the kernels' records (world_transcode.h)
    *out_regular = (!hostIrregular && dim_y <= 65535 && total < 0xffffffffull) ? 1 : 0;
    return CVX_OK;
}

namespace {

} // namespace

// xyz: n_vertices x {x,y,z} already remapped (cvxh_remap_mesh); colors32: n_vertices x {r,g,b,a}. Fills b->lods[0 .. n_lods).
// kernel_ms (optional): device time of the whole build. launches: kernels launched (ours + CUB's are not counted separately).
int cvxd_build_world_gpu(int device, cudaStream_t stream, const float* xyz, const uint8_t* colors32, int32_t n_vertices, int32_t n_lods,
                         cvx_world_builder* b, const cvxd_lod_sink* sink, int64_t* launches, std::string& err) {
    const int X = b->dims[0], Y = b->dims[1], Z = b->dims[2];
    const int64_t nTris = n_vertices / 3;
    if (Y > 65536 || (int64_t)X * Z > ((int64_t)1 << 40)) { err = "dimensions exceed the 16 + 40 bit record key"; return CVX_ERR_INVALID_ARGUMENT; }
    CK(cudaSetDevice(device));
    DeviceBuffers mem;
    float* dxyz; uint8_t* dcol; unsigned long long *counts, *offsets;
    CK(mem.alloc(&dxyz, 9 * (size_t)nTris)); CK(mem.alloc(&dcol, 12 * (size_t)nTris));
    CK(mem.alloc(&counts, (size_t)nTris + 1)); CK(mem.alloc(&offsets, (size_t)nTris + 1));
    CK(cudaMemcpyAsync(dxyz, xyz, 9 * (size_t)nTris * sizeof(float), cudaMemcpyHostToDevice, stream));
    CK(cudaMemcpyAsync(dcol, colors32, 12 * (size_t)nTris, cudaMemcpyHostToDevice, stream));
    CK(cudaMemsetAsync(counts + nTris, 0, 8, stream));
    voxelize_kernel<false><<<(unsigned)nTris, 256, 0, stream>>>(dxyz, dcol, nTris, X, Y, Z, counts, nullptr, nullptr, nullptr);
    CK(cudaGetLastError());
    size_t tmpBytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, tmpBytes, counts, offsets, (int)(nTris + 1), stream));
    uint8_t* tmp; CK(mem.alloc(&tmp, tmpBytes));
    CK(cub::DeviceScan::ExclusiveSum(tmp, tmpBytes, counts, offsets, (int)(nTris + 1), stream));
    std::vector<unsigned long long> hostCounts((size_t)nTris + 1);
    unsigned long long total = 0;
    CK(cudaMemcpyAsync(hostCounts.data(), counts, (size_t)nTris * 8, cudaMemcpyDeviceToHost, stream));
    CK(cudaMemcpyAsync(&total, offsets + nTris, 8, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    for (int64_t t = 0; t < nTris; t++)
        if (hostCounts[(size_t)t] > VOXELIZE_BUFFER_MAX) {
            // the reference stops a triangle after VOXELIZE_BUFFER_MAX voxels in scan order (WordBuilder.cs:37,60-66); reproducing
            // that order-dependent cut is left to the host builder
            err = "triangle " + std::to_string(t) + " covers more than VOXELIZE_BUFFER_MAX voxels: use cvx_builder_from_mesh";
            return CVX_ERR_INVALID_ARGUMENT;
        }
    unsigned long long* keys; uint32_t* vals;
    CK(mem.alloc(&keys, (size_t)total)); CK(mem.alloc(&vals, (size_t)total));
    voxelize_kernel<true><<<(unsigned)nTris, 256, 0, stream>>>(dxyz, dcol, nTris, X, Y, Z, nullptr, offsets, keys, vals);
    CK(cudaGetLastError());
    if (launches) *launches += 2;
    mem.release(tmp);

    unsigned long long* ukeys0; uint32_t* ucolors0; int64_t n0 = 0;
    int r = sort_and_merge(mem, keys, vals, (int64_t)total, 16 + bits_for((unsigned long long)((int64_t)X * Z - 1)), stream, &ukeys0, &ucolors0, n0, err);
    if (r) return r;
    mem.release(keys); mem.release(vals);
    if (launches) *launches += 2;
    r = encode_lod(mem, ukeys0, ucolors0, n0, X, Y, Z, 0, stream, b->lods[0], sink, err);
    if (r) return r;
    if (launches) *launches += 2;
    for (int lod = 1; lod < n_lods; lod++) {
        if ((X >> lod) < 1 || (Y >> lod) < 1 || (Z >> lod) < 1) break;
        unsigned long long* kj; uint32_t* vj;
        CK(mem.alloc(&kj, (size_t)n0)); CK(mem.alloc(&vj, (size_t)n0));
        if (n0 > 0) {
            rekey_kernel<<<(unsigned)((n0 + 255) / 256), 256, 0, stream>>>(ukeys0, n0, Z, lod, kj);
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(vj, ucolors0, (size_t)n0 * 4, cudaMemcpyDeviceToDevice, stream));
        }
        unsigned long long* uk; uint32_t* uc; int64_t nj = 0;
        r = sort_and_merge(mem, kj, vj, n0, 16 + bits_for((unsigned long long)((int64_t)(X >> lod) * (Z >> lod))), stream, &uk, &uc, nj, err);
        if (r) return r;
        r = encode_lod(mem, uk, uc, nj, X, Y, Z, lod, stream, b->lods[lod], sink, err);
        if (r) return r;
        mem.release(kj); mem.release(vj); mem.release(uk); mem.release(uc);
        if (launches) *launches += 5;
    }
    return CVX_OK;
}
