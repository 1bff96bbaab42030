/*
 * raycast_kernels.cu — cvx_raycast and cvx_sweep on the device: one thread per ray or box in 128-thread CTAs, queries in the caller's
 * order (a pick grid keeps neighbouring rays, which walk neighbouring columns, in one warp). The traversals themselves are raycast.h.
 */
#include <cuda_runtime.h>

#include "raycast.h"

namespace {

template <bool BOUNDS>
__global__ void __launch_bounds__(CVXR_THREADS_PER_CTA) raycast_kernel(const __grid_constant__ cvxd_world world, int lod,
                                                                       const cvxd_ray* __restrict__ rays, cvxd_ray_hit* __restrict__ hits, int n) {
    const int i = blockIdx.x * CVXR_THREADS_PER_CTA + threadIdx.x;
    if (i >= n) return;
    const cvxd_ray r = rays[i];
    cvxd_ray_hit h;
    cvxr_cast(world, lod, r, BOUNDS, h);
    hits[i] = h;
}

// at least 4 CTAs per SM: without the minimum ptxas keeps this kernel at 64 registers and spills; with it, up to 128 and none
template <bool BOUNDS>
__global__ void __launch_bounds__(CVXR_THREADS_PER_CTA, 4) sweep_kernel(const __grid_constant__ cvxd_world world, int lod,
                                                                     const cvxd_box* __restrict__ boxes, cvxd_ray_hit* __restrict__ hits, int n) {
    const int i = blockIdx.x * CVXR_THREADS_PER_CTA + threadIdx.x;
    if (i >= n) return;
    const cvxd_box b = boxes[i];
    cvxd_ray_hit h;
    cvxr_sweep(world, lod, b, BOUNDS, h);
    hits[i] = h;
}

} // namespace

cudaError_t cvxd_launch_raycast(const cvxd_world& world, int lod, const cvxd_ray* rays, cvxd_ray_hit* hits, int n, bool use_bounds,
                                cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((n + CVXR_THREADS_PER_CTA - 1) / CVXR_THREADS_PER_CTA);
    if (use_bounds) raycast_kernel<true><<<blocks, CVXR_THREADS_PER_CTA, 0, stream>>>(world, lod, rays, hits, n);
    else raycast_kernel<false><<<blocks, CVXR_THREADS_PER_CTA, 0, stream>>>(world, lod, rays, hits, n);
    return cudaGetLastError();
}

cudaError_t cvxd_launch_sweep(const cvxd_world& world, int lod, const cvxd_box* boxes, cvxd_ray_hit* hits, int n, bool use_bounds,
                              cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((n + CVXR_THREADS_PER_CTA - 1) / CVXR_THREADS_PER_CTA);
    if (use_bounds) sweep_kernel<true><<<blocks, CVXR_THREADS_PER_CTA, 0, stream>>>(world, lod, boxes, hits, n);
    else sweep_kernel<false><<<blocks, CVXR_THREADS_PER_CTA, 0, stream>>>(world, lod, boxes, hits, n);
    return cudaGetLastError();
}
