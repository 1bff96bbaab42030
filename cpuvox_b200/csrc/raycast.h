/*
 * raycast.h — ray queries against the resident world (cvx_raycast): one ray through the tables of one uploaded LOD.
 * No reference analogue: SURVEY.md lists no ray query in the reference (picking, hit-scan and depth probes are host needs
 * that come with a resident world, like the multi-GPU entry points).
 *
 * Plain __device__ code without CUDA-only dependencies: raycast_kernels.cu runs it one thread per ray, and the SIMT emulator
 * (tools/simt_emu) compiles the same source for the CPU so that the tests compare it with a per-cell walk without a GPU.
 *
 * The definition (DESIGN.md §3.5) is a cell-by-cell walk at LOD j (cells of s = 2^j world units, fp32, no FMA contraction):
 * normalise, slab-test the box [0,dim], pick the start cell, then step the axis with the smallest closed-form boundary distance
 * tmax_i = ((float)((cell_i + (step_i > 0)) << j) - o_i) * inv_i (ties: x, then z, then y). This file returns the same hit,
 * distance, face, colour and step count without stepping air cell by cell inside a column: tmax_y is monotone along the ray,
 * so the y cells visited in column (cx, cz) are one interval that ends at the first cell whose tmax_y is not below
 * min(tmax_x, tmax_z) (or that passes max_distance, or the last cell); the interval comes from a position estimate fixed up
 * against the closed form, and its first solid cell in travel order from the column's run list.
 */
#pragma once
#include "device_types.h"

/* mirror cvx_ray / cvx_ray_hit (include/cpuvox_b200.h) */
struct cvxd_ray { float origin[3]; float max_distance; float direction[3]; int32_t reserved; };
struct cvxd_ray_hit { int32_t hit; int32_t face; int32_t cell[3]; float distance; uint32_t color; int32_t steps; };

#define CVXR_THREADS_PER_CTA 128

__device__ __forceinline__ bool cvxr_finite(float v) { return v - v == 0.0f; } // false for NaN and +-inf

// closed-form boundary distance of `cell` along one axis (+inf for an axis the ray does not move along)
__device__ __forceinline__ float cvxr_tmax(int cell, int step, int lod, float o, float inv) {
    return step == 0 ? __builtin_inff() : ((float)((cell + (step > 0 ? 1 : 0)) << lod) - o) * inv;
}

// First solid cell of [lo, hi) (LOD cells, lo < hi) in travel order (up: lowest, else highest), -1 if none; *colour_at receives
// the element-area index of its colour. Runs are read from the reference element area: [guard][runs...][guard][colours...],
// top to bottom from cell ny; a run with Length <= 0 ends the column.
__device__ __forceinline__ int cvxr_first_solid_elements(const cvxd_lod& L, uint4 h, int ny, int lo, int hi, bool up, uint32_t* colour_at) {
    const int rc = (int)(h.y & 0xffffu);
    const uint32_t* runs = L.elements + h.x + 1;
    const uint32_t colours = h.x + (uint32_t)rc + 2u;
    int top = ny, found = -1;
    for (int k = 0; k < rc && top > lo; k++) {
        const uint32_t e = __ldg(runs + k);
        const int len = (int)(int16_t)(e >> 16), ci = (int)(int16_t)(e & 0xffffu);
        if (len <= 0) break;
        const int bot = top - len;
        if (ci >= 0 && bot < hi) {
            const int a = bot > lo ? bot : lo, b = top < hi ? top : hi;
            if (a < b) {
                found = up ? a : b - 1;
                *colour_at = colours + (uint32_t)(ci + (top - 1 - found));
                if (!up) break;            // travelling down: the highest intersecting run wins
            }
        }
        top = bot;
    }
    return found;
}

// The same from the boundary records of a regular LOD (runs cover [0, ny) exactly, record k = {world-Y of the top of run k,
// element k}): a binary search finds the run holding the first cell in travel order, then at most a few runs are read.
__device__ __forceinline__ int cvxr_first_solid_bounds(const cvxd_lod& L, uint4 h, int lod, int lo, int hi, bool up, uint32_t* colour_at) {
    const int rc = (int)(h.y & 0xffffu);
    const uint2* rec = L.bounds + h.w;
    const int start = up ? lo : hi - 1;
    int a = 0, b = rc - 1;                 // the run k with top_{k+1} <= start < top_k: last k with top_k > start
    while (a < b) {
        const int mid = (a + b + 1) >> 1;
        if ((int)(__ldg(&rec[mid].x) >> lod) > start) a = mid; else b = mid - 1;
    }
    const uint32_t colours = h.x + (uint32_t)rc + 2u;
    for (int k = a; k >= 0 && k < rc; k += up ? -1 : 1) {
        const uint2 r = __ldg(&rec[k]);
        const int top = (int)(r.x >> lod), bot = (int)(__ldg(&rec[k + 1].x) >> lod);
        if (up ? bot >= hi : top <= lo) break;
        const int ci = (int)(int16_t)(r.y & 0xffffu);
        if (ci >= 0) {
            const int c = up ? (bot > lo ? bot : lo) : (top < hi ? top : hi) - 1;
            *colour_at = colours + (uint32_t)(ci + (top - 1 - c));
            return c;
        }
    }
    return -1;
}

// Step 1 of DESIGN.md §3.5 (shared by §3.6): normalise `dir` into d, with inv_i = 1/d_i and step_i = sign(d_i) per axis; an axis
// whose component is 0 or too small to invert does not move (d_i = inv_i = 0, step_i = 0). False when the squared length is 0 or
// not finite (the query is invalid).
__device__ __forceinline__ bool cvxr_normalise(const float dir[3], float d[3], float inv[3], int step[3]) {
    const float len2 = dir[0] * dir[0] + dir[1] * dir[1] + dir[2] * dir[2];
    if (!(len2 > 0.0f) || !cvxr_finite(len2)) return false;
    const float invLen = 1.0f / sqrtf(len2);
    for (int i = 0; i < 3; i++) {
        d[i] = dir[i] * invLen;
        inv[i] = 0.0f; step[i] = 0;
        if (d[i] != 0.0f) {
            const float v = 1.0f / d[i];
            if (cvxr_finite(v)) { inv[i] = v; step[i] = d[i] > 0.0f ? 1 : -1; }
            else d[i] = 0.0f;
        }
    }
    return true;
}

// One ray at LOD `lod` (uploaded). use_bounds: read runs from the boundary records (the LOD is regular) instead of the element area.
__device__ __forceinline__ void cvxr_cast(const cvxd_world& w, int lod, const cvxd_ray& r, bool use_bounds, cvxd_ray_hit& out) {
    out.hit = -1; out.face = 0; out.cell[0] = out.cell[1] = out.cell[2] = 0; out.distance = 0.0f; out.color = 0; out.steps = 0;
    const float inf = __builtin_inff();
    float o[3] = {r.origin[0], r.origin[1], r.origin[2]};
    const float maxd = r.max_distance;
    if (!cvxr_finite(o[0]) || !cvxr_finite(o[1]) || !cvxr_finite(o[2]) || !cvxr_finite(r.direction[0]) || !cvxr_finite(r.direction[1]) ||
        !cvxr_finite(r.direction[2]) || !(maxd == inf || cvxr_finite(maxd)))
        return;
    float d[3], inv[3];
    int step[3];
    if (!cvxr_normalise(r.direction, d, inv, step)) return;
    out.hit = 0;
    const int n[3] = {w.dim_x >> lod, w.dim_y >> lod, w.dim_z >> lod};
    // the box of the LOD's cells: n << lod is the world size along x and z, and short of dim_y by dim_y mod 2^lod
    const float dimf[3] = {(float)(n[0] << lod), (float)(n[1] << lod), (float)(n[2] << lod)};
    // box entry: slab test, axes in the order x, z, y (ties of the entry distance go to the earlier axis)
    float tEnter = -inf, tExit = inf;
    int entry = -1;
    for (int q = 0; q < 3; q++) {
        const int i = q == 0 ? 0 : (q == 1 ? 2 : 1);
        if (step[i] == 0) {
            if (!(o[i] >= 0.0f && o[i] < dimf[i])) return;
            continue;
        }
        const float a = (0.0f - o[i]) * inv[i], b = (dimf[i] - o[i]) * inv[i];
        const float nearT = step[i] > 0 ? a : b, farT = step[i] > 0 ? b : a;
        if (nearT > tEnter) { tEnter = nearT; entry = i; }
        if (farT < tExit) tExit = farT;
    }
    const float t0 = tEnter > 0.0f ? tEnter : 0.0f;
    if (tEnter > tExit || tExit < 0.0f || !(t0 <= maxd) || t0 == inf) return;
    const float invS = 1.0f / (float)(1 << lod);
    int c[3];
    float tm[3];
    for (int i = 0; i < 3; i++) {
        if (tEnter > 0.0f && i == entry) c[i] = step[i] > 0 ? 0 : n[i] - 1;
        else {
            const float f = floorf((o[i] + t0 * d[i]) * invS);
            c[i] = f < 0.0f ? 0 : (f > (float)(n[i] - 1) ? n[i] - 1 : (int)f);
        }
        tm[i] = cvxr_tmax(c[i], step[i], lod, o[i], inv[i]);
    }
    int face = tEnter > 0.0f ? 2 * entry + (step[entry] > 0 ? 0 : 1) : 6;
    float t = t0;
    int steps = 0;
    const cvxd_lod& L = w.lods[lod];
    const int s = 1 << lod;
    const int lastY = step[1] > 0 ? n[1] - 1 : 0;
    for (;;) {
        // column (c[0], c[2]) entered at cell c[1]: the y cells visited form [c[1] .. cEnd] in travel order
        const float m = tm[0] < tm[2] ? tm[0] : tm[2];
        int cEnd = c[1];
        if (step[1] != 0 && tm[1] < m && !(tm[1] > maxd) && c[1] != lastY) {
            // y continues from cell cy while tmax_y(cy) < m and tmax_y(cy) <= maxd: estimate where that stops, then fix it up
            const int sy = step[1];
            const float tl = m < maxd ? m : maxd;
            const float f = floorf((o[1] + tl * d[1]) * invS);
            int e;
            if (sy > 0) e = f <= (float)c[1] ? c[1] : (f >= (float)lastY ? lastY : (int)f);
            else e = f >= (float)c[1] ? c[1] : (f <= 0.0f ? 0 : (int)f);
            auto stops = [&](int cy) { const float ty = cvxr_tmax(cy, sy, lod, o[1], inv[1]); return !(ty < m) || ty > maxd; };
            while (e != c[1] && stops(e - sy)) e -= sy;
            while (e != lastY && !stops(e)) e += sy;
            cEnd = e;
        }
        const int lo = c[1] < cEnd ? c[1] : cEnd, hi = (c[1] < cEnd ? cEnd : c[1]) + 1;
        const uint4 h = __ldg(L.headers + (size_t)c[0] * (size_t)L.mul_x + (size_t)c[2]);
        if (h.y & 0xffffu) {
            // a cell whose world-Y range misses the header's [worldMin, worldMax) is air: solid cells lie in [yMin, yMax)
            const int yMin = (int)((h.y >> 16) >> lod), yMax = (int)((h.z + (uint32_t)s - 1u) >> lod);
            const int a = lo > yMin ? lo : yMin, b = hi < yMax ? hi : yMax;
            if (a < b) {
                uint32_t colourAt = 0;
                const bool up = step[1] >= 0;
                const int ch = use_bounds ? cvxr_first_solid_bounds(L, h, lod, a, b, up, &colourAt)
                                          : cvxr_first_solid_elements(L, h, n[1], a, b, up, &colourAt);
                if (ch >= 0) {
                    const int k = ch > c[1] ? ch - c[1] : c[1] - ch;
                    out.hit = 1;
                    out.steps = steps + k + 1;
                    out.distance = k == 0 ? t : cvxr_tmax(ch - step[1], step[1], lod, o[1], inv[1]);
                    out.face = k == 0 ? face : (step[1] > 0 ? 2 : 3);
                    out.cell[0] = c[0]; out.cell[1] = ch; out.cell[2] = c[2];
                    out.color = __ldg(L.elements + colourAt);
                    return;
                }
            }
        }
        steps += hi - lo;
        if (cEnd != c[1]) { c[1] = cEnd; tm[1] = cvxr_tmax(cEnd, step[1], lod, o[1], inv[1]); }
        if (tm[1] < m) { out.steps = steps; return; }   // the y step is next, and it passes max_distance or leaves the grid
        // x or z (written out per axis so that the per-axis state stays in registers)
        const bool xAxis = tm[0] <= tm[1] && tm[0] <= tm[2];
        const float ta = xAxis ? tm[0] : tm[2];
        const int sa = xAxis ? step[0] : step[2];
        const int nc = (xAxis ? c[0] : c[2]) + sa;
        if (ta > maxd || ta == inf || nc < 0 || nc >= (xAxis ? n[0] : n[2])) { out.steps = steps; return; }
        t = ta;
        face = (xAxis ? 0 : 4) + (sa > 0 ? 0 : 1);
        if (xAxis) { c[0] = nc; tm[0] = cvxr_tmax(nc, sa, lod, o[0], inv[0]); }
        else { c[2] = nc; tm[2] = cvxr_tmax(nc, sa, lod, o[2], inv[2]); }
    }
}

/*
 * Swept boxes (cvx_sweep, DESIGN.md §3.6): how far an axis-aligned box moves along a direction before it touches a solid cell.
 * Per axis, cell k's window is the open interval (enter, exit) of times at which the open box overlaps the cell's slab, with
 * lo = (float)(k << j) - h and hi = (float)((k+1) << j) + h; a cell is a candidate when the three windows meet after 0 and enter by
 * max_distance, and the solid candidate with the smallest key (t*, overlapping first, cx, cz, cy) is the result.
 *
 * Along the direction of travel of a moving axis both enter(k) and exit(k) are non-decreasing (every operation rounds
 * monotonically), so every condition but "enter < exit of one cell" selects a prefix or a suffix of an axis's cells: the walk below
 * visits the slabs of the XZ major axis in travel order, in each the interval of minor cells, and in each column the interval of
 * y cells, each interval found from a position estimate fixed up against the exact expressions. The cost grows with the box's XZ
 * footprint in cells (one header per column it sweeps) and with its length of travel; there is no size cap.
 */
struct cvxd_box { float center[3]; float max_distance; float direction[3]; int32_t reserved0; float half_extent[3]; int32_t reserved1; };

// one axis of a sweep: centre, half extent, normalised direction component, its inverse and sign (step 0: still)
struct cvxr_axis { float c, h, d, inv; int step; };

// cell k's window on one axis (§3.6 step 2); a still axis has (-inf, +inf) where lo < c < hi and an empty window elsewhere
__device__ __forceinline__ void cvxr_window(const cvxr_axis& a, int k, int lod, float& enter, float& exit) {
    const float inf = __builtin_inff();
    const float lo = (float)(k << lod) - a.h, hi = (float)((k + 1) << lod) + a.h;
    if (a.step == 0) {
        const bool in = lo < a.c && a.c < hi;
        enter = in ? -inf : inf; exit = in ? inf : -inf;
        return;
    }
    const float p = (lo - a.c) * a.inv, q = (hi - a.c) * a.inv;
    enter = a.step > 0 ? p : q; exit = a.step > 0 ? q : p;
}
__device__ __forceinline__ float cvxr_enter(const cvxr_axis& a, int k, int lod) { float e, x; cvxr_window(a, k, lod, e, x); return e; }
__device__ __forceinline__ float cvxr_exit(const cvxr_axis& a, int k, int lod) { float e, x; cvxr_window(a, k, lod, e, x); return x; }

// First k of [lo, hi] at which `pred` holds, for a predicate that is false then true over [lo, hi); e (a floor) is an estimate.
template <class P>
__device__ __forceinline__ int cvxr_first_true(int lo, int hi, float e, P pred) {
    int k = e >= (float)lo ? (e <= (float)hi ? (int)e : hi) : lo;     // NaN: lo
    while (k > lo && pred(k - 1)) k--;
    while (k < hi && !pred(k)) k++;
    return k;
}

// The cells [*A, *B) of [lo, hi) whose window has exit > m1, enter < u and enter <= lim (every cell of the still-axis window).
__device__ __forceinline__ void cvxr_window_cells(const cvxr_axis& a, int lod, float invS, int lo, int hi, float m1, float u, float lim,
                                                  int* A, int* B) {
    if (a.step == 0) {
        *A = cvxr_first_true(lo, hi, floorf((a.c - a.h) * invS), [&](int k) { return a.c < (float)((k + 1) << lod) + a.h; });
        *B = cvxr_first_true(*A, hi, floorf((a.c + a.h) * invS) + 1.0f, [&](int k) { return !((float)(k << lod) - a.h < a.c); });
        return;
    }
    // in travel order `early` holds for a prefix and `late` for a suffix; the estimates are the box's extent in cells at m1 and tu
    auto early = [&](int k) { const float e = cvxr_enter(a, k, lod); return e < u && e <= lim; };
    auto late = [&](int k) { return cvxr_exit(a, k, lod) > m1; };
    const float tu = u < lim ? u : lim;
    if (a.step > 0) {
        *A = cvxr_first_true(lo, hi, floorf((a.c - a.h + m1 * a.d) * invS), late);
        *B = cvxr_first_true(*A, hi, floorf((a.c + a.h + tu * a.d) * invS) + 1.0f, [&](int k) { return !early(k); });
    } else {
        *A = cvxr_first_true(lo, hi, floorf((a.c - a.h + tu * a.d) * invS), early);
        *B = cvxr_first_true(*A, hi, floorf((a.c + a.h + m1 * a.d) * invS) + 1.0f, [&](int k) { return !late(k); });
    }
}

// One box at LOD `lod` (uploaded); use_bounds as in cvxr_cast. out.steps = column headers read.
__device__ __forceinline__ void cvxr_sweep(const cvxd_world& w, int lod, const cvxd_box& b, bool use_bounds, cvxd_ray_hit& out) {
    out.hit = -1; out.face = 0; out.cell[0] = out.cell[1] = out.cell[2] = 0; out.distance = 0.0f; out.color = 0; out.steps = 0;
    const float inf = __builtin_inff();
    const float maxd = b.max_distance;
    for (int i = 0; i < 3; i++)
        if (!cvxr_finite(b.center[i]) || !cvxr_finite(b.direction[i]) || !cvxr_finite(b.half_extent[i]) || !(b.half_extent[i] > 0.0f)) return;
    if (!(maxd == inf || cvxr_finite(maxd))) return;
    float d[3], inv[3];
    int step[3];
    if (!cvxr_normalise(b.direction, d, inv, step)) return;
    out.hit = 0;
    if (!(maxd >= 0.0f)) return;                                     // every candidate has t* >= 0
    const cvxr_axis ax = {b.center[0], b.half_extent[0], d[0], inv[0], step[0]};
    const cvxr_axis az = {b.center[2], b.half_extent[2], d[2], inv[2], step[2]};
    const cvxr_axis ay = {b.center[1], b.half_extent[1], d[1], inv[1], step[1]};
    const bool xMajor = fabsf(d[0]) >= fabsf(d[2]);
    const cvxr_axis aM = xMajor ? ax : az, am = xMajor ? az : ax;
    const int nx = w.dim_x >> lod, ny = w.dim_y >> lod, nz = w.dim_z >> lod;
    const int nM = xMajor ? nx : nz, nm = xMajor ? nz : nx;
    const float invS = 1.0f / (float)(1 << lod);
    const int s = 1 << lod;
    const cvxd_lod& L = w.lods[lod];

    bool found = false, bOv = false;
    float bt = inf;                                                  // best t*
    int bx = 0, by = 0, bz = 0, bFace = 0;
    uint32_t bColourAt = 0;
    float lim = maxd;                                                // min(max_distance, best t*): a cell entered later cannot win
    int steps = 0;

    int MA, MB;
    cvxr_window_cells(aM, lod, invS, 0, nM, 0.0f, inf, lim, &MA, &MB);
    const int sM = aM.step < 0 ? -1 : 1, sm = am.step < 0 ? -1 : 1;
    for (int kM = sM > 0 ? MA : MB - 1; kM >= MA && kM < MB; kM += sM) {
        float eM, xM;
        cvxr_window(aM, kM, lod, eM, xM);
        if (eM > lim) break;
        if (!(eM < xM)) continue;
        int mA, mB;
        cvxr_window_cells(am, lod, invS, 0, nm, eM > 0.0f ? eM : 0.0f, xM, lim, &mA, &mB);
        for (int km = sm > 0 ? mA : mB - 1; km >= mA && km < mB; km += sm) {
            float em, xm;
            cvxr_window(am, km, lod, em, xm);
            if (em > lim) break;
            if (!(em < xm)) continue;
            // column (cx, cz): T and T' of its XZ windows, entry axis x before z on ties
            const int cx = xMajor ? kM : km, cz = xMajor ? km : kM;
            const float ex = xMajor ? eM : em, ez = xMajor ? em : eM;
            const float txz = ez > ex ? ez : ex, uxz = xm < xM ? xm : xM;
            const int faceXZ = ez > ex ? 4 + (az.step > 0 ? 0 : 1) : (ax.step > 0 ? 0 : 1);
            const uint4 h = __ldg(L.headers + (size_t)cx * (size_t)L.mul_x + (size_t)cz);
            steps++;
            if (!(h.y & 0xffffu)) continue;
            // y candidates: exit_y > max(T_xz, 0), enter_y < T'_xz, enter_y <= lim, inside the header's [worldMin, worldMax)
            const int yMin = (int)((h.y >> 16) >> lod), yMax = (int)((h.z + (uint32_t)s - 1u) >> lod);
            const int ylo = yMin > 0 ? yMin : 0, yhi = yMax < ny ? yMax : ny;
            if (ylo >= yhi) continue;
            int A, B;
            cvxr_window_cells(ay, lod, invS, ylo, yhi, txz > 0.0f ? txz : 0.0f, uxz, lim, &A, &B);
            if (A >= B) continue;
            // first solid cell of [lo, hi) in travel order whose own y window is not empty
            uint32_t colourAt = 0;
            auto search = [&](int lo, int hi, bool up) {
                for (;;) {
                    const int c = lo >= hi ? -1
                                           : (use_bounds ? cvxr_first_solid_bounds(L, h, lod, lo, hi, up, &colourAt)
                                                         : cvxr_first_solid_elements(L, h, ny, lo, hi, up, &colourAt));
                    if (c < 0) return -1;
                    float e, x;
                    cvxr_window(ay, c, lod, e, x);
                    if (e < x) return c;
                    if (up) lo = c + 1; else hi = c;
                }
            };
            auto tOf = [&](int k) { const float e = cvxr_enter(ay, k, lod); return e > txz ? e : txz; };
            int f = search(A, B, ay.step >= 0);
            if (f < 0) continue;
            float T = tOf(f);
            if (ay.step < 0) {
                // T is non-decreasing in travel order, so the cells below f that share its (t*, overlapping) form [g, f]; the lowest
                // solid one wins
                const float ts = T > 0.0f ? T : 0.0f;
                const bool ov = T < 0.0f;
                const int g = cvxr_first_true(A, f, floorf((ay.c - ay.h + ts * ay.d) * invS), [&](int k) {
                    const float t = tOf(k);
                    return (t > 0.0f ? t : 0.0f) == ts && (t < 0.0f) == ov;
                });
                if (g < f) { f = search(g, f + 1, true); T = tOf(f); }
            }
            const float ts = T > 0.0f ? T : 0.0f;
            const bool ov = T < 0.0f;
            const bool better = !found || (ts != bt ? ts < bt
                                         : ov != bOv ? ov
                                         : cx != bx ? cx < bx
                                         : cz != bz ? cz < bz : f < by);
            if (better) {
                found = true; bt = ts; bOv = ov; bx = cx; by = f; bz = cz; bColourAt = colourAt;
                bFace = ov ? 6 : (cvxr_enter(ay, f, lod) > txz ? (ay.step > 0 ? 2 : 3) : faceXZ);
                lim = bt < maxd ? bt : maxd;
            }
        }
    }
    out.steps = steps;
    if (!found) return;
    out.hit = 1; out.face = bFace; out.distance = bt;
    out.cell[0] = bx; out.cell[1] = by; out.cell[2] = bz;
    out.color = __ldg(L.elements + bColourAt);
}

#ifdef __CUDACC__
cudaError_t cvxd_launch_raycast(const cvxd_world& world, int lod, const cvxd_ray* rays, cvxd_ray_hit* hits, int n, bool use_bounds,
                                cudaStream_t stream);
cudaError_t cvxd_launch_sweep(const cvxd_world& world, int lod, const cvxd_box* boxes, cvxd_ray_hit* hits, int n, bool use_bounds,
                              cudaStream_t stream);
#endif
