// K3/K4/K5: the reference's uniform-grid construction (grid.cpp:12-154) rebuilt for the GPU as
// count -> exclusive scan -> fill -> per-cell sort, producing the compact CSR layout
// (cell_start[cells+1] + ascending triangle indices) the reference's own TODO asks for
// (grid.h:35-36).  Membership is decided by the same fp64 separating-axis test
// (aabb_tri_internal.h:112-186) on the same fp32-derived cell boxes, so the arrays come out
// identical to the flattened reference grid (tests/test_gpu_grid.py checks array equality).
//
// Compiled with -fmad=false: the SAT's fp64 products/sums and the fp32 cell boxes must round
// like the reference's (no FMA on its x86-64 baseline).
#include "grid_build.cuh"

#include <cfloat>
#include <utility>
#include <vector>

namespace rtm
{

namespace
{

#define GB_CK(call)                                                                              \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
        {                                                                                        \
            err = std::string(#call) + ": " + cudaGetErrorString(e_);                            \
            return CUDA_TRACE_ERR_CUDA;                                                          \
        }                                                                                        \
    } while (0)

struct GridParamsDev
{
    uint32_t dim[3];
    float aabb_min[3];
    float aabb_max[3];
    float cell_wdh;
    float inv_cell_wdh;
};

// std::min / std::max as ComponentMin / ComponentMax use them (lin_alg.h:157-170)
__device__ __forceinline__ float std_min(float a, float b) { return (b < a) ? b : a; }
__device__ __forceinline__ float std_max(float a, float b) { return (a < b) ? b : a; }

// ---- mesh AABB (mesh.cpp:72-94): only vertices referenced by triangles; note the max is seeded
// with numeric_limits<float>::min() (= FLT_MIN > 0), which this reproduces.  min/max are exact
// and order independent, so a parallel reduction gives the reference's bits.
__global__ void mesh_aabb_partial_kernel(const float *__restrict__ vtx, const uint32_t *__restrict__ tri,
                                         uint32_t num_tri, float *__restrict__ partial /* blocks x 6 */)
{
    float mn[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, mx[3] = { FLT_MIN, FLT_MIN, FLT_MIN };
    for (uint32_t ti = blockIdx.x * blockDim.x + threadIdx.x; ti < num_tri; ti += gridDim.x * blockDim.x)
        for (int c = 0; c < 3; c++)
        {
            const float *p = vtx + (size_t) tri[(size_t) ti * 6 + c] * 6;
            for (int k = 0; k < 3; k++)
            {
                mn[k] = std_min(mn[k], p[k]);
                mx[k] = std_max(mx[k], p[k]);
            }
        }
    __shared__ float s[6][256];
    for (int k = 0; k < 3; k++)
    {
        s[k][threadIdx.x] = mn[k];
        s[3 + k][threadIdx.x] = mx[k];
    }
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1)
    {
        if ((int) threadIdx.x < w)
            for (int k = 0; k < 3; k++)
            {
                s[k][threadIdx.x] = std_min(s[k][threadIdx.x], s[k][threadIdx.x + w]);
                s[3 + k][threadIdx.x] = std_max(s[3 + k][threadIdx.x], s[3 + k][threadIdx.x + w]);
            }
        __syncthreads();
    }
    if (threadIdx.x < 6)
        partial[blockIdx.x * 6 + threadIdx.x] = s[threadIdx.x][0];
}

// ---- grid.cpp:29-38: grow the box by 1e-4, cell width from the longest axis, dimensions
__global__ void grid_params_kernel(const float *__restrict__ partial, uint32_t blocks, uint32_t grid_res,
                                   GridParamsDev *__restrict__ out)
{
    float mn[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, mx[3] = { FLT_MIN, FLT_MIN, FLT_MIN };
    for (uint32_t b = 0; b < blocks; b++)
        for (int k = 0; k < 3; k++)
        {
            mn[k] = std_min(mn[k], partial[b * 6 + k]);
            mx[k] = std_max(mx[k], partial[b * 6 + 3 + k]);
        }
    float ext[3];
    for (int k = 0; k < 3; k++)
    {
        out->aabb_min[k] = mn[k] - 0.0001f;
        out->aabb_max[k] = mx[k] + 0.0001f;
        ext[k] = out->aabb_max[k] - out->aabb_min[k];
    }
    const float largest = std_max(std_max(ext[0], ext[1]), ext[2]);
    out->cell_wdh = largest / (float) grid_res;
    out->inv_cell_wdh = 1.0f / out->cell_wdh;
    for (int k = 0; k < 3; k++)
        out->dim[k] = __float2uint_rz(ceilf(ext[k] / out->cell_wdh));
}

// ---- aabb_tri_internal.h:42-62
__device__ __forceinline__ bool plane_box_overlap(const double normal[3], double d, const double maxbox[3])
{
    double vmin[3], vmax[3];
#pragma unroll
    for (int q = 0; q < 3; q++)
    {
        if (normal[q] > 0.0) { vmin[q] = -maxbox[q]; vmax[q] = maxbox[q]; }
        else                 { vmin[q] = maxbox[q];  vmax[q] = -maxbox[q]; }
    }
    if (normal[0] * vmin[0] + normal[1] * vmin[1] + normal[2] * vmin[2] + d > 0.0) return false;
    if (normal[0] * vmax[0] + normal[1] * vmax[1] + normal[2] * vmax[2] + d >= 0.0) return true;
    return false;
}

// One edge (ex,ey,ez) against the three box axes; (a*, b*) are the two vertices the reference's
// AXISTEST_* macro for that (edge, axis) projects (aabb_tri_internal.h:65-110)
#define RTM_AXIS_X(va, vb)                                                                       \
    {                                                                                            \
        const double pa = ez * va[1] - ey * va[2], pb = ez * vb[1] - ey * vb[2];                 \
        const double rad = fez * h[1] + fey * h[2];                                              \
        if ((pa < pb ? pa : pb) > rad || (pa < pb ? pb : pa) < -rad) return false;               \
    }
#define RTM_AXIS_Y(va, vb)                                                                       \
    {                                                                                            \
        const double pa = -ez * va[0] + ex * va[2], pb = -ez * vb[0] + ex * vb[2];               \
        const double rad = fez * h[0] + fex * h[2];                                              \
        if ((pa < pb ? pa : pb) > rad || (pa < pb ? pb : pa) < -rad) return false;               \
    }
#define RTM_AXIS_Z(va, vb)                                                                       \
    {                                                                                            \
        const double pa = ey * va[0] - ex * va[1], pb = ey * vb[0] - ex * vb[1];                 \
        const double rad = fey * h[0] + fex * h[1];                                              \
        if ((pa < pb ? pa : pb) > rad || (pa < pb ? pb : pa) < -rad) return false;               \
    }

// aabb.h:15-32 + aabb_tri_internal.h:112-186: centre/half in fp32 then widened, SAT in fp64
__device__ bool tri_box_overlap(const float p0[3], const float p1[3], const float p2[3], const float cmin[3],
                                const float cmax[3])
{
    double h[3], v0[3], v1[3], v2[3];
#pragma unroll
    for (int k = 0; k < 3; k++)
    {
        const double c = (double) ((cmin[k] + cmax[k]) * 0.5f);
        h[k] = (double) ((cmax[k] - cmin[k]) * 0.5f);
        v0[k] = (double) p0[k] - c;
        v1[k] = (double) p1[k] - c;
        v2[k] = (double) p2[k] - c;
    }
    double ex, ey, ez, fex, fey, fez;
    // edge 0 = v1 - v0: X01, Y02, Z12
    ex = v1[0] - v0[0]; ey = v1[1] - v0[1]; ez = v1[2] - v0[2];
    const double e0x = ex, e0y = ey, e0z = ez;
    fex = fabs(ex); fey = fabs(ey); fez = fabs(ez);
    RTM_AXIS_X(v0, v2) RTM_AXIS_Y(v0, v2) RTM_AXIS_Z(v1, v2)
    // edge 1 = v2 - v1: X01, Y02, Z0
    ex = v2[0] - v1[0]; ey = v2[1] - v1[1]; ez = v2[2] - v1[2];
    const double e1x = ex, e1y = ey, e1z = ez;
    fex = fabs(ex); fey = fabs(ey); fez = fabs(ez);
    RTM_AXIS_X(v0, v2) RTM_AXIS_Y(v0, v2) RTM_AXIS_Z(v0, v1)
    // edge 2 = v0 - v2: X2, Y1, Z12
    ex = v0[0] - v2[0]; ey = v0[1] - v2[1]; ez = v0[2] - v2[2];
    fex = fabs(ex); fey = fabs(ey); fez = fabs(ez);
    RTM_AXIS_X(v0, v1) RTM_AXIS_Y(v0, v1) RTM_AXIS_Z(v1, v2)
    // the three box axes (:154-166)
#pragma unroll
    for (int k = 0; k < 3; k++)
    {
        double mn = v0[k], mx = v0[k];
        if (v1[k] < mn) mn = v1[k];
        if (v1[k] > mx) mx = v1[k];
        if (v2[k] < mn) mn = v2[k];
        if (v2[k] > mx) mx = v2[k];
        if (mn > h[k] || mx < -h[k]) return false;
    }
    // the triangle's plane (:172-175): normal = e0 x e1, d = -normal . v0
    double normal[3];
    normal[0] = e0y * e1z - e0z * e1y;
    normal[1] = e0z * e1x - e0x * e1z;
    normal[2] = e0x * e1y - e0y * e1x;
    const double d = -(normal[0] * v0[0] + normal[1] * v0[1] + normal[2] * v0[2]);
    return plane_box_overlap(normal, d, h);
}

struct TriRange
{
    float p0[3], p1[3], p2[3];
    uint32_t start[3], n[3]; // candidate cell range (grid.cpp:70-92), clamped to the grid
};

// triangle.h:116-131 (max seeded with FLT_MIN > 0) and grid.cpp:70-92 (division, not * inv)
__device__ __forceinline__ void tri_range(const float *__restrict__ vtx, const uint32_t *__restrict__ tri,
                                          uint32_t ti, const GridParamsDev& g, TriRange& r)
{
    const uint32_t *tr = tri + (size_t) ti * 6;
    const float *a = vtx + (size_t) tr[0] * 6, *b = vtx + (size_t) tr[1] * 6, *c = vtx + (size_t) tr[2] * 6;
#pragma unroll
    for (int k = 0; k < 3; k++)
    {
        r.p0[k] = a[k]; r.p1[k] = b[k]; r.p2[k] = c[k];
        float mn = FLT_MAX, mx = FLT_MIN;
        mn = std_min(mn, a[k]); mx = std_max(mx, a[k]);
        mn = std_min(mn, b[k]); mx = std_max(mx, b[k]);
        mn = std_min(mn, c[k]); mx = std_max(mx, c[k]);
        const uint32_t s = __float2uint_rz((mn - g.aabb_min[k]) / g.cell_wdh);
        uint32_t e = __float2uint_rz((mx - g.aabb_min[k]) / g.cell_wdh);
        // The reference seeds the maximum with FLT_MIN (> 0), so for a triangle whose coordinates
        // on this axis are all negative its candidate range runs on to the cell containing 0 --
        // thousands of cells the exact test then rejects one by one.  Membership is decided by
        // that test alone (it contains the per-axis interval test, aabb_tri_internal.h:154-166),
        // so the range may be cut at the triangle's TRUE maximum plus one guard cell without
        // changing a single list; the wider range only costs time (26 s -> well under a second
        // for the 50 M-triangle soup at 256^3).
        const float true_mx = std_max(std_max(a[k], b[k]), c[k]);
        const uint32_t e_true = __float2uint_rz((true_mx - g.aabb_min[k]) / g.cell_wdh) + 1u;
        if (e > e_true) e = e_true;
        // the reference does not clamp `end` (it relies on the 1e-4 growth, grid.cpp:18-30);
        // clamping cannot change the result because cells outside the grid do not exist
        if (e > g.dim[k] - 1) e = g.dim[k] - 1;
        r.start[k] = s;
        r.n[k] = (s <= e) ? (e - s + 1) : 0;
    }
}

__device__ __forceinline__ bool candidate_overlaps(const TriRange& r, const GridParamsDev& g, uint32_t x,
                                                   uint32_t y, uint32_t z)
{
    // grid.cpp:98-106 cell box in world space, fp32
    const float cmin[3] = { g.aabb_min[0] + (float) x * g.cell_wdh, g.aabb_min[1] + (float) y * g.cell_wdh,
                            g.aabb_min[2] + (float) z * g.cell_wdh };
    const float cmax[3] = { g.aabb_min[0] + (float) (x + 1) * g.cell_wdh,
                            g.aabb_min[1] + (float) (y + 1) * g.cell_wdh,
                            g.aabb_min[2] + (float) (z + 1) * g.cell_wdh };
    return tri_box_overlap(r.p0, r.p1, r.p2, cmin, cmax);
}

__device__ __forceinline__ void emit(uint32_t cell, uint32_t ti, bool fill, uint32_t *__restrict__ counts_or_cursor,
                                     uint32_t *__restrict__ tri_index)
{
    const uint32_t slot = atomicAdd(&counts_or_cursor[cell], 1u);
    if (fill)
        tri_index[slot] = ti;
}

constexpr uint32_t kBigTriCandidates = 96; // triangles with more candidate cells get a whole CTA

// K3 / K5, small triangles: one thread per triangle.  fill == false: counts[cell]++;
// fill == true: tri_index[cursor[cell]++] = ti.  Big triangles are queued for the CTA kernel.
__global__ void grid_bin_small_kernel(const float *__restrict__ vtx, const uint32_t *__restrict__ tri,
                                      uint32_t num_tri, const GridParamsDev *__restrict__ gp, bool fill,
                                      uint32_t *__restrict__ counts_or_cursor, uint32_t *__restrict__ tri_index,
                                      uint32_t *__restrict__ big_list, uint32_t *__restrict__ big_count)
{
    const uint32_t ti = blockIdx.x * blockDim.x + threadIdx.x;
    if (ti >= num_tri)
        return;
    const GridParamsDev g = *gp;
    TriRange r;
    tri_range(vtx, tri, ti, g, r);
    const uint64_t cand = (uint64_t) r.n[0] * r.n[1] * r.n[2];
    if (cand > kBigTriCandidates)
    {
        if (!fill) // the list built by the count pass is reused by the fill pass
            big_list[atomicAdd(big_count, 1u)] = ti;
        return;
    }
    const uint32_t sx = g.dim[0], sxz = g.dim[0] * g.dim[2];
    for (uint32_t x = r.start[0]; x < r.start[0] + r.n[0]; x++)
        for (uint32_t y = r.start[1]; y < r.start[1] + r.n[1]; y++)
            for (uint32_t z = r.start[2]; z < r.start[2] + r.n[2]; z++)
                if (candidate_overlaps(r, g, x, y, z))
                    emit(x + z * sx + y * sxz, ti, fill, counts_or_cursor, tri_index);
}

// K3 / K5, big triangles (e.g. a ground plane spanning thousands of cells): one CTA each
__global__ void grid_bin_big_kernel(const float *__restrict__ vtx, const uint32_t *__restrict__ tri,
                                    const GridParamsDev *__restrict__ gp, bool fill,
                                    uint32_t *__restrict__ counts_or_cursor, uint32_t *__restrict__ tri_index,
                                    const uint32_t *__restrict__ big_list)
{
    const uint32_t ti = big_list[blockIdx.x];
    const GridParamsDev g = *gp;
    TriRange r;
    tri_range(vtx, tri, ti, g, r);
    const uint64_t cand = (uint64_t) r.n[0] * r.n[1] * r.n[2];
    const uint32_t sx = g.dim[0], sxz = g.dim[0] * g.dim[2];
    for (uint64_t c = threadIdx.x; c < cand; c += blockDim.x)
    {
        const uint32_t z = r.start[2] + (uint32_t) (c % r.n[2]);
        const uint32_t y = r.start[1] + (uint32_t) ((c / r.n[2]) % r.n[1]);
        const uint32_t x = r.start[0] + (uint32_t) (c / ((uint64_t) r.n[2] * r.n[1]));
        if (candidate_overlaps(r, g, x, y, z))
            emit(x + z * sx + y * sxz, ti, fill, counts_or_cursor, tri_index);
    }
}

// ---- K4: exclusive scan over uint32 (three-phase, recursive on the block sums) ------------
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

__global__ void scan_tile_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, uint64_t n,
                                 uint32_t *__restrict__ tile_sums)
{
    __shared__ uint32_t s_warp[kScanThreads / 32];
    const uint64_t base = (uint64_t) blockIdx.x * kScanTile + (uint64_t) threadIdx.x * kScanItems;
    uint32_t v[kScanItems], sum = 0;
#pragma unroll
    for (int i = 0; i < kScanItems; i++)
    {
        v[i] = (base + i < n) ? in[base + i] : 0u;
        sum += v[i];
    }
    // inclusive scan of the per-thread sums
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t inc = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1)
    {
        const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
        if (lane >= (uint32_t) o) inc += t;
    }
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    if (warp == 0)
    {
        uint32_t w = (lane < kScanThreads / 32) ? s_warp[lane] : 0u;
#pragma unroll
        for (int o = 1; o < kScanThreads / 32; o <<= 1)
        {
            const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, w, o);
            if (lane >= (uint32_t) o) w += t;
        }
        if (lane < kScanThreads / 32) s_warp[lane] = w;
    }
    __syncthreads();
    uint32_t excl = inc - sum + (warp ? s_warp[warp - 1] : 0u);
#pragma unroll
    for (int i = 0; i < kScanItems; i++)
    {
        if (base + i < n) out[base + i] = excl;
        excl += v[i];
    }
    if (threadIdx.x == kScanThreads - 1 && tile_sums)
        tile_sums[blockIdx.x] = s_warp[kScanThreads / 32 - 1];
}

__global__ void scan_add_kernel(uint32_t *__restrict__ data, uint64_t n, const uint32_t *__restrict__ tile_offsets)
{
    const uint64_t i = (uint64_t) blockIdx.x * kScanTile + threadIdx.x;
    const uint32_t add = tile_offsets[blockIdx.x];
#pragma unroll
    for (int k = 0; k < kScanItems; k++)
    {
        const uint64_t j = i + (uint64_t) k * kScanThreads;
        if (j < n) data[j] += add;
    }
}

__global__ void sum_u32_kernel(const uint32_t *__restrict__ in, uint64_t n, unsigned long long *__restrict__ total)
{
    unsigned long long s = 0;
    for (uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t) gridDim.x * blockDim.x)
        s += in[i];
    for (int o = 16; o > 0; o >>= 1)
        s += __shfl_down_sync(0xFFFFFFFFu, s, o);
    if ((threadIdx.x & 31) == 0 && s)
        atomicAdd(total, s);
}

// ---- the index check of a mesh given in device memory (the host path checks on the host): the lowest triangle with
// a vertex index >= num_vtx goes to *first_bad (preset to 0xFFFFFFFF) through atomicMin
__global__ void check_triangle_indices_kernel(const uint32_t *__restrict__ tri, uint32_t num_tri, uint32_t num_vtx,
                                              uint32_t *__restrict__ first_bad)
{
    for (uint64_t ti = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x; ti < num_tri;
         ti += (uint64_t) gridDim.x * blockDim.x)
    {
        const uint32_t *t = tri + ti * 6;
        if ((t[0] >= num_vtx) | (t[1] >= num_vtx) | (t[2] >= num_vtx))
            atomicMin(first_bad, (uint32_t) ti);
    }
}

} // namespace

void launch_check_triangle_indices(const uint32_t *d_tri, uint32_t num_tri, uint32_t num_vtx, uint32_t *d_first_bad,
                                   cudaStream_t stream)
{
    const unsigned blocks = (unsigned) std::min<uint64_t>(1024, ((uint64_t) num_tri + 255) / 256);
    check_triangle_indices_kernel<<<std::max(blocks, 1u), 256, 0, stream>>>(d_tri, num_tri, num_vtx, d_first_bad);
}

int exclusive_scan_u32(const uint32_t *d_in, uint32_t *d_out, uint64_t n, cudaStream_t stream, std::string& err,
                       uint64_t *launches)
{
    if (n == 0)
        return 0;
    const uint64_t tiles = (n + kScanTile - 1) / kScanTile;
    DeviceArray<uint32_t> d_sums;
    if (tiles > 1)
        GB_CK(d_sums.alloc(tiles));
    scan_tile_kernel<<<(unsigned) tiles, kScanThreads, 0, stream>>>(d_in, d_out, n, d_sums.get());
    (*launches)++;
    if (tiles > 1)
    {
        StreamDrain drain(stream);
        const int rc = exclusive_scan_u32(d_sums.get(), d_sums.get(), tiles, stream, err, launches);
        if (rc)
            return rc;
        scan_add_kernel<<<(unsigned) tiles, kScanThreads, 0, stream>>>(d_out, n, d_sums.get());
        (*launches)++;
        GB_CK(drain.sync());
    }
    GB_CK(cudaGetLastError());
    return 0;
}

namespace
{

// ---- K5b: the reference pushes triangle indices in ascending order (grid.cpp:65,122) and the
// traversal's strict "cur_t < t" keeps the FIRST of equal-t hits (grid.cpp:259), so list order is
// part of the result: sort every cell's list ascending after the atomic fill.
constexpr uint32_t kSmallList = 24;

__global__ void sort_small_cells_kernel(const uint32_t *__restrict__ cell_start, uint64_t num_cells,
                                        uint32_t *__restrict__ tri_index, uint32_t *__restrict__ long_cells,
                                        uint32_t *__restrict__ long_count)
{
    const uint64_t c = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= num_cells)
        return;
    const uint32_t beg = cell_start[c], end = cell_start[c + 1], len = end - beg;
    if (len < 2)
        return;
    if (len > kSmallList)
    {
        long_cells[atomicAdd(long_count, 1u)] = (uint32_t) c;
        return;
    }
    for (uint32_t i = beg + 1; i < end; i++) // insertion sort
    {
        const uint32_t key = tri_index[i];
        uint32_t j = i;
        while (j > beg && tri_index[j - 1] > key)
        {
            tri_index[j] = tri_index[j - 1];
            j--;
        }
        tri_index[j] = key;
    }
}

// One CTA per long cell.  Lists that fit the shared-memory budget: bitonic sort; longer ones:
// rank sort through a scratch copy (indices within a cell are unique, so ranks are a permutation)
__global__ void sort_long_cells_kernel(const uint32_t *__restrict__ cell_start, const uint32_t *__restrict__ long_cells,
                                       uint32_t *__restrict__ tri_index, uint32_t *__restrict__ scratch,
                                       uint32_t smem_capacity)
{
    extern __shared__ uint32_t s_keys[];
    const uint32_t c = long_cells[blockIdx.x];
    const uint32_t beg = cell_start[c], len = cell_start[c + 1] - beg;
    if (len <= smem_capacity)
    {
        uint32_t n = 1;
        while (n < len) n <<= 1;
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x)
            s_keys[i] = i < len ? tri_index[beg + i] : 0xFFFFFFFFu;
        __syncthreads();
        for (uint32_t k = 2; k <= n; k <<= 1)
            for (uint32_t j = k >> 1; j > 0; j >>= 1)
            {
                for (uint32_t i = threadIdx.x; i < n; i += blockDim.x)
                {
                    const uint32_t l = i ^ j;
                    if (l > i)
                    {
                        const uint32_t a = s_keys[i], b = s_keys[l];
                        const bool up = (i & k) == 0;
                        if ((a > b) == up)
                        {
                            s_keys[i] = b;
                            s_keys[l] = a;
                        }
                    }
                }
                __syncthreads();
            }
        for (uint32_t i = threadIdx.x; i < len; i += blockDim.x)
            tri_index[beg + i] = s_keys[i];
    }
    else
    {
        for (uint32_t i = threadIdx.x; i < len; i += blockDim.x)
            scratch[beg + i] = tri_index[beg + i];
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < len; i += blockDim.x)
        {
            const uint32_t key = scratch[beg + i];
            uint32_t rank = 0;
            for (uint32_t j = 0; j < len; j++)
                rank += scratch[beg + j] < key ? 1u : 0u;
            tri_index[beg + rank] = key;
        }
    }
}

} // namespace

int build_grid_device(const float *d_vtx, uint32_t num_vtx, const uint32_t *d_tri, uint32_t num_tri,
                      uint32_t grid_res, cudaStream_t stream, GridBuildResult *out, std::string& err,
                      uint64_t *launches)
{
    // grid.cpp:15-16 asserts
    if (num_vtx == 0 || num_tri == 0 || grid_res == 0)
    {
        err = "build_grid: empty mesh or grid_res == 0";
        return CUDA_TRACE_ERR_ARG;
    }
    DeviceArray<float> d_partial;
    DeviceArray<GridParamsDev> d_gp;
    DeviceArray<unsigned long long> d_total;
    DeviceArray<uint32_t> d_counts, d_big_list, d_big_count, d_cursor, d_tri_index, d_scratch;
    StreamDrain drain(stream);

    // mesh box -> grid parameters
    const uint32_t aabb_blocks = (uint32_t) std::min<uint64_t>(1024, (num_tri + 255) / 256);
    GB_CK(d_partial.alloc(6 * aabb_blocks));
    GB_CK(d_gp.alloc(1));
    mesh_aabb_partial_kernel<<<aabb_blocks, 256, 0, stream>>>(d_vtx, d_tri, num_tri, d_partial.get());
    grid_params_kernel<<<1, 1, 0, stream>>>(d_partial.get(), aabb_blocks, grid_res, d_gp.get());
    *launches += 2;
    GridParamsDev gp;
    GB_CK(cudaMemcpyAsync(&gp, d_gp.get(), sizeof(gp), cudaMemcpyDeviceToHost, stream));
    GB_CK(cudaStreamSynchronize(stream));

    const uint64_t num_cells = (uint64_t) gp.dim[0] * gp.dim[1] * gp.dim[2];
    if (num_cells == 0 || num_cells >= (1ull << 31))
    {
        err = "build_grid: grid has " + std::to_string(num_cells) + " cells (supported: 1 .. 2^31-1)";
        return CUDA_TRACE_ERR_ARG;
    }

    // K3 count
    GB_CK(d_counts.alloc(num_cells + 1));
    GB_CK(d_big_list.alloc(num_tri));
    GB_CK(d_big_count.alloc(1));
    GB_CK(cudaMemsetAsync(d_counts.get(), 0, (num_cells + 1) * sizeof(uint32_t), stream));
    GB_CK(cudaMemsetAsync(d_big_count.get(), 0, sizeof(uint32_t), stream));
    const unsigned tri_blocks = (num_tri + 127) / 128;
    grid_bin_small_kernel<<<tri_blocks, 128, 0, stream>>>(d_vtx, d_tri, num_tri, d_gp.get(), false, d_counts.get(), nullptr,
                                                          d_big_list.get(), d_big_count.get());
    (*launches)++;
    uint32_t big_count = 0;
    GB_CK(cudaMemcpyAsync(&big_count, d_big_count.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    GB_CK(cudaStreamSynchronize(stream));
    if (big_count)
    {
        grid_bin_big_kernel<<<big_count, 256, 0, stream>>>(d_vtx, d_tri, d_gp.get(), false, d_counts.get(), nullptr,
                                                           d_big_list.get());
        (*launches)++;
    }

    // total references (64-bit, to refuse grids whose CSR offsets would not fit uint32)
    unsigned long long total = 0;
    GB_CK(d_total.alloc(1));
    GB_CK(cudaMemsetAsync(d_total.get(), 0, sizeof(unsigned long long), stream));
    sum_u32_kernel<<<1024, 256, 0, stream>>>(d_counts.get(), num_cells, d_total.get());
    (*launches)++;
    GB_CK(cudaMemcpyAsync(&total, d_total.get(), sizeof(total), cudaMemcpyDeviceToHost, stream));
    GB_CK(cudaStreamSynchronize(stream));
    if (total >= (1ull << 32))
    {
        err = "build_grid: " + std::to_string(total) + " cell references do not fit 32-bit offsets";
        return CUDA_TRACE_ERR_ARG;
    }

    // K4 scan (in place: counts -> exclusive offsets; entry num_cells becomes the total)
    int rc = exclusive_scan_u32(d_counts.get(), d_counts.get(), num_cells + 1, stream, err, launches);
    if (rc)
        return rc;
    uint32_t *d_cell_start = d_counts.get();

    // K5 fill through a cursor copy
    GB_CK(d_cursor.alloc(num_cells));
    GB_CK(d_tri_index.alloc(std::max<uint64_t>(total, 1)));
    GB_CK(cudaMemcpyAsync(d_cursor.get(), d_cell_start, num_cells * sizeof(uint32_t), cudaMemcpyDeviceToDevice, stream));
    grid_bin_small_kernel<<<tri_blocks, 128, 0, stream>>>(d_vtx, d_tri, num_tri, d_gp.get(), true, d_cursor.get(),
                                                          d_tri_index.get(), d_big_list.get(), d_big_count.get());
    (*launches)++;
    if (big_count)
    {
        grid_bin_big_kernel<<<big_count, 256, 0, stream>>>(d_vtx, d_tri, d_gp.get(), true, d_cursor.get(), d_tri_index.get(),
                                                           d_big_list.get());
        (*launches)++;
    }

    // K5b per-cell sort (d_cursor is dead now: reuse it as the long-cell list)
    uint32_t *d_long_cells = d_cursor.get(), *d_long_count = d_big_count.get();
    GB_CK(cudaMemsetAsync(d_long_count, 0, sizeof(uint32_t), stream));
    sort_small_cells_kernel<<<(unsigned) ((num_cells + 255) / 256), 256, 0, stream>>>(d_cell_start, num_cells,
                                                                                      d_tri_index.get(), d_long_cells,
                                                                                      d_long_count);
    (*launches)++;
    uint32_t long_count = 0;
    GB_CK(cudaMemcpyAsync(&long_count, d_long_count, sizeof(uint32_t), cudaMemcpyDeviceToHost, stream));
    GB_CK(cudaStreamSynchronize(stream));
    if (long_count)
    {
        const uint32_t smem_cap = 32768; // keys; 128 KB of shared memory
        GB_CK(d_scratch.alloc(std::max<uint64_t>(total, 1)));
        GB_CK(cudaFuncSetAttribute(sort_long_cells_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   (int) (smem_cap * sizeof(uint32_t))));
        sort_long_cells_kernel<<<long_count, 512, smem_cap * sizeof(uint32_t), stream>>>(d_cell_start, d_long_cells,
                                                                                        d_tri_index.get(),
                                                                                        d_scratch.get(), smem_cap);
        (*launches)++;
    }
    GB_CK(drain.sync());
    GB_CK(cudaGetLastError());

    for (int k = 0; k < 3; k++)
    {
        out->desc.dim[k] = gp.dim[k];
        out->desc.aabb_min[k] = gp.aabb_min[k];
        out->desc.aabb_max[k] = gp.aabb_max[k];
    }
    out->desc.cell_wdh = gp.cell_wdh;
    out->desc.inv_cell_wdh = gp.inv_cell_wdh;
    out->desc.num_cells = num_cells;
    out->desc.num_refs = total;
    out->d_cell_start = std::move(d_counts);
    out->d_tri_index = std::move(d_tri_index);
    return 0;
}

} // namespace rtm
