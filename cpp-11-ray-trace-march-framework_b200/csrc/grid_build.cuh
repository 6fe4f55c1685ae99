// Device-side uniform grid construction (K3 count, K4 scan, K5 fill + per-cell sort).
#pragma once

#include <cstdint>
#include <string>
#include <cuda_runtime.h>

#include "../../include/cuda_trace.h"
#include "device_array.cuh"

namespace rtm
{

struct GridBuildResult
{
    cuda_trace_grid_desc desc;
    DeviceArray<uint32_t> d_cell_start; // num_cells + 1
    DeviceArray<uint32_t> d_tri_index;  // num_refs (at least 1 allocated)
};

// Builds the reference's grid (grid.cpp:12-154) for the mesh in device memory (d_vtx: V x 6 floats,
// d_tri: T x 6 words).  All device work goes to `stream`; the call synchronises the stream a few
// times (it needs the grid dimensions and the reference count on the host to size allocations).
// On failure returns a non-zero cuda_trace_status and sets err.  *launches is incremented per kernel.
int build_grid_device(const float *d_vtx, uint32_t num_vtx, const uint32_t *d_tri, uint32_t num_tri,
                      uint32_t grid_res, cudaStream_t stream, GridBuildResult *out, std::string& err,
                      uint64_t *launches);

// Enqueues the vertex-index check of T x 6-word triangle records in device memory: *d_first_bad, which the caller sets
// to 0xFFFFFFFF first, becomes the lowest triangle with an index >= num_vtx and is left alone when there is none
void launch_check_triangle_indices(const uint32_t *d_tri, uint32_t num_tri, uint32_t num_vtx, uint32_t *d_first_bad,
                                   cudaStream_t stream);

// Exclusive prefix sum over n uint32 words (in place allowed); synchronises `stream` when n spans several tiles
int exclusive_scan_u32(const uint32_t *d_in, uint32_t *d_out, uint64_t n, cudaStream_t stream, std::string& err,
                       uint64_t *launches);

} // namespace rtm
