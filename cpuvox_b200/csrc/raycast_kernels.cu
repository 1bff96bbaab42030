/*
 * raycast_kernels.cu — cvx_raycast on the device: one thread per ray in 128-thread CTAs, rays in the caller's order (a pick grid
 * keeps neighbouring rays, which walk neighbouring columns, in one warp). The traversal itself is raycast.h.
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

} // namespace

cudaError_t cvxd_launch_raycast(const cvxd_world& world, int lod, const cvxd_ray* rays, cvxd_ray_hit* hits, int n, bool use_bounds,
                                cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const unsigned blocks = (unsigned)((n + CVXR_THREADS_PER_CTA - 1) / CVXR_THREADS_PER_CTA);
    if (use_bounds) raycast_kernel<true><<<blocks, CVXR_THREADS_PER_CTA, 0, stream>>>(world, lod, rays, hits, n);
    else raycast_kernel<false><<<blocks, CVXR_THREADS_PER_CTA, 0, stream>>>(world, lod, rays, hits, n);
    return cudaGetLastError();
}
