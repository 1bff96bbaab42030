/*
 * world_builder.h — state shared by the host world builder (world_builder.cpp) and the device one (world_builder_gpu.cu):
 * a builder owns the LOD blobs in the reference's WorldAllocator layout (World.cs:285-313), whoever produced them.
 */
#pragma once
#include <stdint.h>
#include <vector>
#include "../../include/cpuvox_b200.h"

struct cvx_lod_blob {
    std::vector<uint8_t> bytes;
    int columnCount = 0;
    int64_t voxelCount = 0;
    bool built = false;
};


struct MeshVoxel { int32_t xz; int16_t y; uint32_t argb; };

struct cvx_world_builder {
    int dims[3] = {0, 0, 0};
    int nThreads = 0;
    bool deviceBuilt = false; // LODs were produced by cvx_gpu_builder_from_mesh: nothing left to build on the host
    cvx_lod_blob lods[CVX_LOD_LEVELS];
    // mesh path: voxels binned by column (CSR)
    std::vector<int64_t> colStart;
    std::vector<MeshVoxel> voxels;
    // synthetic path: kind + seed; columns generated on the fly
    int synthKind = -1;
    uint32_t seed = 0;
    std::vector<uint16_t> height; // kind 0: heightmap
    struct Box { int x0, x1, y0, y1, z0, z1; uint32_t color; int kind; }; // kind 1 objects
    std::vector<Box> boxes;
    std::vector<std::vector<int>> boxBins; int binShift = 6, binsX = 0, binsZ = 0;
};


/* SimpleMesh.Remap_Internal (SimpleMesh.cs:64-106) on the host: rescale to [0, max_dimension], power-of-two dimensions, axis
 * flips. out_xyz = n_vertices x {x,y,z}. Shared by both builders so they voxelize bit-identical vertices. */
int cvxh_remap_mesh(const float* positions, int32_t n_vertices, int32_t max_dimension, const int32_t flips[3],
                    std::vector<float>& out_xyz, int out_dims[3]);

#ifdef __CUDACC__
#include <functional>
#include <string>
/* The CVX_ERR_* code a failed CUDA call reports: running out of device memory is told apart from every other failure. */
inline int cvx_code(cudaError_t e) { return e == cudaErrorMemoryAllocation ? CVX_ERR_OUT_OF_MEMORY : CVX_ERR_CUDA; }
/* Receives each finished LOD blob while it is still in device memory and takes ownership of the allocation (cudaFree it). */
typedef std::function<int(int lod, void* device_blob, int64_t bytes, int column_count)> cvxd_lod_sink;
/* world_builder_gpu.cu: voxelize + RLE + LOD mips on the device (b->dims set by the caller). Without a sink the blobs are copied into
 * b->lods[0 .. n_lods); with one they are handed over on the device and b only records column and voxel counts. */
int cvxd_build_world_gpu(int device, cudaStream_t stream, const float* xyz, const uint8_t* colors32, int32_t n_vertices, int32_t n_lods,
                         cvx_world_builder* b, const cvxd_lod_sink* sink, int64_t* launches, std::string& err);
/* world_builder_gpu.cu: the Phase-1 tables of one LOD (uint4 headers + boundary records, see world_transcode.h) from a blob in device memory. */
int cvxd_transcode_lod_device(cudaStream_t stream, const void* blob_dev, int64_t need_cols, int64_t column_count, int64_t element_cells, int lod, int dim_y,
                              void** out_headers, void** out_bounds, int* out_regular, long long* bad_column, int64_t* launches, std::string& err);
#endif
