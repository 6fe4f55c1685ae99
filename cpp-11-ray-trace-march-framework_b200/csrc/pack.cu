// K6: scene packing -- Mesh AoS (reference mesh.h:12-24) -> the device layout of rt_device.cuh.
// Removes the double indirection the reference pays per triangle test (grid.cpp:245-253:
// cell list -> m_triangles[idx] -> 3 x m_vertices[v].p) and per hit (renderer.cpp:109-115).
// Compiled with -fmad=false: e1/e2 and the variant-B constants must carry the reference's bits.
#include "trace_kernels.cuh"

#include <math_constants.h>

namespace rtm
{

namespace
{

__global__ void pack_cell_tris_kernel(const float *__restrict__ vtx, const uint32_t *__restrict__ tri,
                                      const uint32_t *__restrict__ tri_index, uint64_t num_refs,
                                      float4 *__restrict__ cell_tris, float4 *__restrict__ cell_tris_b)
{
    const uint64_t k = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= num_refs)
        return;
    const uint32_t ti = tri_index[k];
    const uint32_t *tr = tri + (size_t) ti * 6;
    const float *p0 = vtx + (size_t) tr[0] * 6, *p1 = vtx + (size_t) tr[1] * 6, *p2 = vtx + (size_t) tr[2] * 6;
    const float v0x = p0[0], v0y = p0[1], v0z = p0[2];
    // triangle.h:39-40 (SUB edge1 = vert1 - vert0, edge2 = vert2 - vert0)
    const float e1x = p1[0] - v0x, e1y = p1[1] - v0y, e1z = p1[2] - v0z;
    const float e2x = p2[0] - v0x, e2y = p2[1] - v0y, e2z = p2[2] - v0z;
    cell_tris[3 * k + 0] = make_float4(v0x, v0y, v0z, __uint_as_float(ti));
    cell_tris[3 * k + 1] = make_float4(e1x, e1y, e1z, 0.0f);
    cell_tris[3 * k + 2] = make_float4(e2x, e2y, e2z, 0.0f);
    // variant B constants: face normal n = Mesh::Triangle::n, d = Dot(n, v0) (triangle.h:205),
    // ComputeBarycentric's e0 = v2 - v0 (= e2 here), e1 = v1 - v0 (triangle.h:140-149)
    const float nx = __uint_as_float(tr[3]), ny = __uint_as_float(tr[4]), nz = __uint_as_float(tr[5]);
    const float d00 = dot_ref(e2x, e2y, e2z, e2x, e2y, e2z);
    const float d01 = dot_ref(e2x, e2y, e2z, e1x, e1y, e1z);
    const float d11 = dot_ref(e1x, e1y, e1z, e1x, e1y, e1z);
    cell_tris_b[2 * k + 0] = make_float4(nx, ny, nz, dot_ref(nx, ny, nz, v0x, v0y, v0z));
    cell_tris_b[2 * k + 1] = make_float4(d00, d01, d11, 1.0f / (d00 * d11 - d01 * d01));
}

__global__ void pack_normals_kernel(const float *__restrict__ vtx, const uint32_t *__restrict__ tri,
                                    uint32_t num_tri, float4 *__restrict__ tri_normals)
{
    const uint32_t ti = blockIdx.x * blockDim.x + threadIdx.x;
    if (ti >= num_tri)
        return;
    const uint32_t *tr = tri + (size_t) ti * 6;
#pragma unroll
    for (int c = 0; c < 3; c++)
    {
        const float *n = vtx + (size_t) tr[c] * 6 + 3;
        tri_normals[3 * (size_t) ti + c] = make_float4(n[0], n[1], n[2], 0.0f);
    }
}

__global__ void cell_occupancy_kernel(const uint32_t *__restrict__ cell_start, uint64_t num_cells,
                                      uint32_t *__restrict__ cell_occ)
{
    const uint64_t w = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t first = w * 32;
    if (first >= num_cells)
        return;
    uint32_t bits = 0;
    const uint32_t n = (uint32_t) min((uint64_t) 32, num_cells - first);
    uint32_t prev = cell_start[first];
    for (uint32_t i = 0; i < n; i++)
    {
        const uint32_t next = cell_start[first + i + 1];
        if (next != prev)
            bits |= 1u << i;
        prev = next;
    }
    cell_occ[w] = bits;
}

// Padded grid (see rt_device.cuh): padded cell q = X + Z*pdx + Y*pdx*pdz with X in [0, dx+2) etc.
// Interior cells keep their relative order, so the padded CSR offset of q is the unpadded offset
// of the first interior cell at or after q.
__device__ __forceinline__ uint32_t interior_cells_before(uint32_t X, uint32_t Y, uint32_t Z, uint32_t dx,
                                                          uint32_t dy, uint32_t dz)
{
    const uint32_t ys = min(Y > 0 ? Y - 1 : 0u, dy);
    uint32_t r = ys * dx * dz;
    if (Y >= 1 && Y <= dy)
    {
        const uint32_t zs = min(Z > 0 ? Z - 1 : 0u, dz);
        r += zs * dx;
        if (Z >= 1 && Z <= dz)
            r += min(X > 0 ? X - 1 : 0u, dx);
    }
    return r;
}

__global__ void pad_cell_start_kernel(const uint32_t *__restrict__ cell_start, uint32_t dx, uint32_t dy, uint32_t dz,
                                      uint32_t *__restrict__ pcell_start)
{
    const uint32_t pdx = dx + 2, pdy = dy + 2, pdz = dz + 2;
    const uint64_t pcells = (uint64_t) pdx * pdy * pdz;
    const uint64_t q = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (q > pcells)
        return;
    if (q == pcells)
    {
        pcell_start[q] = cell_start[(uint64_t) dx * dy * dz];
        return;
    }
    const uint32_t X = (uint32_t) (q % pdx), Z = (uint32_t) ((q / pdx) % pdz), Y = (uint32_t) (q / ((uint64_t) pdx * pdz));
    pcell_start[q] = cell_start[interior_cells_before(X, Y, Z, dx, dy, dz)];
}

__global__ void pad_cell_occ_kernel(const uint32_t *__restrict__ pcell_start, uint32_t dx, uint32_t dy, uint32_t dz,
                                    uint32_t *__restrict__ pcell_occ)
{
    const uint32_t pdx = dx + 2, pdy = dy + 2, pdz = dz + 2;
    const uint64_t pcells = (uint64_t) pdx * pdy * pdz;
    const uint64_t w = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t first = w * 32;
    if (first >= pcells)
        return;
    uint32_t bits = 0;
    const uint32_t n = (uint32_t) min((uint64_t) 32, pcells - first);
    for (uint32_t i = 0; i < n; i++)
    {
        const uint64_t q = first + i;
        const uint32_t X = (uint32_t) (q % pdx), Z = (uint32_t) ((q / pdx) % pdz), Y = (uint32_t) (q / ((uint64_t) pdx * pdz));
        const bool border = X == 0 || X == pdx - 1 || Y == 0 || Y == pdy - 1 || Z == 0 || Z == pdz - 1;
        if (border || pcell_start[q] != pcell_start[q + 1])
            bits |= 1u << i;
    }
    pcell_occ[w] = bits;
}

// ---- distance map over the padded grid (second level of the empty-space walk, warp_trace.cuh kOccGlobalDist):
// dist[q] = min(255, city-block distance in cells from padded cell q to the nearest cell whose occupancy bit is
// set -- a non-empty cell or a border cell), one byte per cell.  (Two bits per cell, min(3, distance) -- a quarter of
// the footprint, L2-resident at 512^3 -- was measured on the 50 M-triangle soup: 84.6 against 83.6 ms with K1, and
// slower with K7 as well: the extra look-ups and the unpacking cost more than the cache misses saved.)  A DDA step moves to a face neighbour, so a ray standing on a cell of
// distance v meets only empty cells during its next v - 1 steps, whatever its direction: those steps need no
// look-up at all.  The city-block transform is separable: one forward / backward sweep per axis is exact.
__global__ void dist_sweep_x_kernel(const uint32_t *__restrict__ pcell_occ, uint32_t pdx, uint64_t lines, uint8_t *__restrict__ dist)
{
    const uint64_t line = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (line >= lines)
        return;
    const uint64_t q0 = line * pdx;
    uint32_t d = 255;
    for (uint32_t x = 0; x < pdx; x++)
    {
        const uint64_t q = q0 + x;
        const bool set = (pcell_occ[q >> 5] >> (q & 31)) & 1u;
        d = set ? 0u : min(d + 1u, 255u);
        dist[q] = (uint8_t) d;
    }
    for (uint32_t x = pdx; x-- > 0;)
    {
        const uint64_t q = q0 + x;
        d = min((uint32_t) dist[q], min(d + 1u, 255u));
        dist[q] = (uint8_t) d;
    }
}

// sweep along an axis whose cell stride is `stride`; thread t handles the line starting at
// (t % inner) + (t / inner) * outer_stride (neighbouring threads = neighbouring x: coalesced)
__global__ void dist_sweep_kernel(uint8_t *__restrict__ dist, uint32_t n, uint64_t stride, uint32_t inner, uint64_t outer_stride,
                                  uint64_t lines)
{
    const uint64_t t = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= lines)
        return;
    const uint64_t q0 = (t % inner) + (t / inner) * outer_stride;
    uint32_t d = 255;
    for (uint32_t i = 0; i < n; i++)
    {
        const uint64_t q = q0 + i * stride;
        d = min((uint32_t) dist[q], min(d + 1u, 255u));
        dist[q] = (uint8_t) d;
    }
    for (uint32_t i = n; i-- > 0;)
    {
        const uint64_t q = q0 + i * stride;
        d = min((uint32_t) dist[q], min(d + 1u, 255u));
        dist[q] = (uint8_t) d;
    }
}

__global__ void narrow_offsets_kernel(const uint64_t *__restrict__ in, uint64_t n, uint32_t *__restrict__ out)
{
    const uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        out[i] = (uint32_t) in[i];
}

__global__ void widen_offsets_kernel(const uint32_t *__restrict__ in, uint64_t n, uint64_t *__restrict__ out)
{
    const uint64_t i = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n)
        out[i] = in[i];
}

inline unsigned blocks_for(uint64_t n, unsigned threads) { return (unsigned) ((n + threads - 1) / threads); }

} // namespace

// ---- pair records (rt_device.cuh): two triangles of a cell interleaved component by component, for the
// packed-fp32 Moeller-Trumbore of K1 (warp_trace.cuh)
namespace
{

__global__ void pair_count_kernel(const uint32_t *__restrict__ pcell_start, uint64_t pcells, uint32_t *__restrict__ counts)
{
    const uint64_t q = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (q > pcells)
        return;
    counts[q] = q < pcells ? (pcell_start[q + 1] - pcell_start[q] + 1u) / 2u : 0u;
}

// The b half of an odd list's last pair: a triangle no ray can hit.  With v0 = (-1e18, 0, 0), e1 = x, e2 = y the
// determinant is -dir.z and u = tvec . pvec / det ~ 1e18 for every |det| >= 1e-8 (rejected by the u test,
// triangle.h:83-85); a smaller |det| is rejected by the determinant test itself (triangle.h:77-78).  Valid for
// scenes whose coordinates stay below ~1e9, which the launcher checks.
__device__ __forceinline__ void dummy_triangle(float4& a, float4& b, float4& c)
{
    a = make_float4(-1.0e18f, 0.0f, 0.0f, __uint_as_float(0xFFFFFFFFu));
    b = make_float4(1.0f, 0.0f, 0.0f, 0.0f);
    c = make_float4(0.0f, 1.0f, 0.0f, 0.0f);
}

// one thread per padded cell (lists are short: the count over 2 of the cell's references)
__global__ void pack_pairs_kernel(const uint32_t *__restrict__ pcell_start, const uint32_t *__restrict__ ppair_start,
                                  uint64_t pcells, const float4 *__restrict__ cell_tris, float4 *__restrict__ pair_recs)
{
    const uint64_t q = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= pcells)
        return;
    const uint32_t beg = pcell_start[q], end = pcell_start[q + 1];
    uint64_t out = ppair_start[q];
    for (uint32_t k = beg; k < end; k += 2, out++)
    {
        const float4 a0 = cell_tris[3 * (uint64_t) k + 0], a1 = cell_tris[3 * (uint64_t) k + 1], a2 = cell_tris[3 * (uint64_t) k + 2];
        float4 b0, b1, b2;
        if (k + 1 < end)
        {
            b0 = cell_tris[3 * (uint64_t) k + 3]; b1 = cell_tris[3 * (uint64_t) k + 4]; b2 = cell_tris[3 * (uint64_t) k + 5];
        }
        else
            dummy_triangle(b0, b1, b2);
        float4 *r = pair_recs + 5 * out;
        r[0] = make_float4(a0.x, b0.x, a0.y, b0.y);
        r[1] = make_float4(a0.z, b0.z, a1.x, b1.x);
        r[2] = make_float4(a1.y, b1.y, a1.z, b1.z);
        r[3] = make_float4(a2.x, b2.x, a2.y, b2.y);
        r[4] = make_float4(a2.z, b2.z, a0.w, b0.w);
    }
}

// Primary rays share their origin, so everything in the Moeller-Trumbore test (triangle.h:15-107) that does not
// involve the direction is the same for every ray of a frame: tvec = orig - v0, qvec = tvec x e1, e2 . qvec.
// Computed here once per camera position with the very expressions of the per-ray test (same operand order, no
// contraction), so the per-ray results stay bit-identical.  One thread per pair record.
__global__ void origin_relative_pairs_kernel(const float4 *__restrict__ pair_recs, uint64_t num_pairs, float ox, float oy,
                                             float oz, float4 *__restrict__ rel)
{
    const uint64_t k = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= num_pairs)
        return;
    const float4 *r = pair_recs + 5 * k;
    const float4 f0 = r[0], f1 = r[1], f2 = r[2], f3 = r[3], f4 = r[4];
    float tv[2][3], q[2][3], e2q[2];
    const float v0[2][3] = { { f0.x, f0.z, f1.x }, { f0.y, f0.w, f1.y } };
    const float e1[2][3] = { { f1.z, f2.x, f2.z }, { f1.w, f2.y, f2.w } };
    const float e2[2][3] = { { f3.x, f3.z, f4.x }, { f3.y, f3.w, f4.y } };
#pragma unroll
    for (int h = 0; h < 2; h++)
    {
        const float tx = ox - v0[h][0], ty = oy - v0[h][1], tz = oz - v0[h][2];
        const float qx = ty * e1[h][2] - tz * e1[h][1];
        const float qy = tz * e1[h][0] - tx * e1[h][2];
        const float qz = tx * e1[h][1] - ty * e1[h][0];
        tv[h][0] = tx; tv[h][1] = ty; tv[h][2] = tz;
        q[h][0] = qx; q[h][1] = qy; q[h][2] = qz;
        e2q[h] = e2[h][0] * qx + e2[h][1] * qy + e2[h][2] * qz;
    }
    float4 *o = rel + 7 * k;
    o[0] = make_float4(tv[0][0], tv[1][0], tv[0][1], tv[1][1]);
    o[1] = make_float4(tv[0][2], tv[1][2], f1.z, f1.w);
    o[2] = f2;
    o[3] = f3;
    o[4] = f4;
    o[5] = make_float4(q[0][0], q[1][0], q[0][1], q[1][1]);
    o[6] = make_float4(q[0][2], q[1][2], e2q[0], e2q[1]);
}

// ---- screen boxes (K1's screen cull, warp_trace.cuh test_pair_list; DESIGN.md section 3, "Screen cull"): for one camera,
// the box in generate_ray's image plane (x = ndc_x * fov_xs, y = ndc_y * fov_xs / aspect) outside which no ray can be
// accepted by either triangle of a pair.  float64 throughout, without contraction (-fmad=false), operation for
// operation as tools/screen_cull.py restates it; the final narrowing rounds outwards.
constexpr double kCullEps = 5.9604644775390625e-8; // 2^-24
constexpr double kCullTau = 0.015625;              // a vertex counts as in front if its depth > 2^-6 |camera-space vector|
constexpr double kCullRound = 16.0, kCullDir = 16.0, kCullSafety = 4.0, kCullKappaMax = 1.0e4;

struct CullCamera
{
    double inv[9], k;
    bool ok;
};

__device__ CullCamera cull_camera(const CameraDev& cam)
{
    CullCamera c;
    const double m00 = cam.m[0][0], m01 = cam.m[0][1], m02 = cam.m[0][2], m10 = cam.m[1][0], m11 = cam.m[1][1],
                 m12 = cam.m[1][2], m20 = cam.m[2][0], m21 = cam.m[2][1], m22 = cam.m[2][2];
    const double c00 = m11 * m22 - m12 * m21, c01 = m12 * m20 - m10 * m22, c02 = m10 * m21 - m11 * m20;
    const double det = m00 * c00 + m01 * c01 + m02 * c02;
    c.inv[0] = c00 / det; c.inv[1] = (m02 * m21 - m01 * m22) / det; c.inv[2] = (m01 * m12 - m02 * m11) / det;
    c.inv[3] = c01 / det; c.inv[4] = (m00 * m22 - m02 * m20) / det; c.inv[5] = (m02 * m10 - m00 * m12) / det;
    c.inv[6] = c02 / det; c.inv[7] = (m01 * m20 - m00 * m21) / det; c.inv[8] = (m00 * m11 - m01 * m10) / det;
    const double m[9] = { m00, m01, m02, m10, m11, m12, m20, m21, m22 };
    double fro = 0.0, fro_inv = 0.0;
    for (int i = 0; i < 9; i++)
        fro = fro + m[i] * m[i];
    for (int i = 0; i < 9; i++)
        fro_inv = fro_inv + c.inv[i] * c.inv[i];
    fro = sqrt(fro);
    fro_inv = sqrt(fro_inv);
    const double fx = cam.fov_xs, fy = fx / (double) cam.aspect;
    const double l_img = sqrt(1.0 + 4.0 * (fx * fx) + 4.0 * (fy * fy));
    c.k = kCullEps * fro * l_img / fabs(det);
    c.ok = isfinite(c.k) && det != 0.0 && isfinite(fro_inv) && fro * fro_inv <= kCullKappaMax;
    return c;
}

__device__ __forceinline__ double norm3(double x, double y, double z) { return sqrt(x * x + y * y + z * z); }

// box {xmin, xmax, ymin, ymax} of one triangle (v0, e1, e2 as the records hold them): the projected triangle with each
// edge line pushed outwards by kCullSafety x the bound on that edge's error; +-inf = never cull; empty for the dummy
__device__ void triangle_screen_box(float v0x, float v0y, float v0z, float e1x, float e1y, float e1z, float e2x, float e2y,
                                    float e2z, uint32_t idx, const CameraDev& cam, const CullCamera& cc, double box[4])
{
    if (idx == 0xFFFFFFFFu)
    {
        box[0] = box[2] = CUDART_INF;
        box[1] = box[3] = -CUDART_INF;
        return;
    }
    const double o[3] = { cam.origin[0], cam.origin[1], cam.origin[2] };
    const double p[3][3] = { { v0x, v0y, v0z },
                             { (double) v0x + (double) e1x, (double) v0y + (double) e1y, (double) v0z + (double) e1z },
                             { (double) v0x + (double) e2x, (double) v0y + (double) e2y, (double) v0z + (double) e2z } };
    double V[3][3], cx[3], cy[3], w[3];
    bool good = cc.ok;
    for (int q = 0; q < 3; q++)
    {
        const double vx = p[q][0] - o[0], vy = p[q][1] - o[1], vz = p[q][2] - o[2];
        const double x = vx * cc.inv[0] + vy * cc.inv[3] + vz * cc.inv[6];
        const double y = vx * cc.inv[1] + vy * cc.inv[4] + vz * cc.inv[7];
        const double z = vx * cc.inv[2] + vy * cc.inv[5] + vz * cc.inv[8];
        V[q][0] = vx; V[q][1] = vy; V[q][2] = vz;
        cx[q] = x / -z;
        cy[q] = y / -z;
        w[q] = -z;
        good = good && w[q] > kCullTau * norm3(x, y, z);
    }
    const double R = fmax(fmax(norm3(V[0][0], V[0][1], V[0][2]), norm3(V[1][0], V[1][1], V[1][2])), norm3(V[2][0], V[2][1], V[2][2]));
    const double l1 = norm3(e1x, e1y, e1z), l2 = norm3(e2x, e2y, e2z);
    // rounding error of the test's three edge functions: v's numerator (edge 0-1), the u + v <= 1 test (edge 1-2),
    // u's numerator (edge 2-0)
    const double base[3] = { kCullRound * (R * l1), kCullRound * (R * (l1 + l2) + l1 * l2), kCullRound * (R * l2) };
    const double a2s = (cx[1] - cx[0]) * (cy[2] - cy[0]) - (cy[1] - cy[0]) * (cx[2] - cx[0]);
    const double sgn = a2s < 0.0 ? -1.0 : 1.0;
    double nx[3], ny[3], off[3], perim_slack = 0.0;
    for (int q = 0; q < 3; q++)
    {
        const int i = q, j = q == 2 ? 0 : q + 1;
        const double dx = cx[j] - cx[i], dy = cy[j] - cy[i];
        const double lij = sqrt(dx * dx + dy * dy);
        const double crx = V[i][1] * V[j][2] - V[i][2] * V[j][1];
        const double cry = V[i][2] * V[j][0] - V[i][0] * V[j][2];
        const double crz = V[i][0] * V[j][1] - V[i][1] * V[j][0];
        const double dij = kCullSafety * (cc.k * (base[q] + kCullDir * norm3(crx, cry, crz)) / (w[i] * w[j] * lij));
        nx[q] = sgn * dy / lij; // outward unit normal
        ny[q] = -sgn * dx / lij;
        off[q] = dij;
        perim_slack = perim_slack + lij * dij;
    }
    // vertex q lies on edges q - 1 and q: its pushed-out position solves n . s = slack for both lines
    double px[3], py[3];
    for (int q = 0; q < 3; q++)
    {
        const int a = (q + 2) % 3, b = q;
        const double det2 = nx[a] * ny[b] - ny[a] * nx[b];
        px[q] = cx[q] + (off[a] * ny[b] - off[b] * ny[a]) / det2;
        py[q] = cy[q] + (nx[a] * off[b] - nx[b] * off[a]) / det2;
        good = good && isfinite(px[q]) && isfinite(py[q]);
    }
    box[0] = fmin(fmin(px[0], px[1]), px[2]);
    box[1] = fmax(fmax(px[0], px[1]), px[2]);
    box[2] = fmin(fmin(py[0], py[1]), py[2]);
    box[3] = fmax(fmax(py[0], py[1]), py[2]);
    good = good && perim_slack < fabs(a2s);
    for (int q = 0; q < 4; q++)
        good = good && isfinite(box[q]);
    if (!good)
    {
        box[0] = box[2] = -CUDART_INF;
        box[1] = box[3] = CUDART_INF;
    }
}

// one thread per pair record
__global__ void screen_boxes_kernel(const float4 *__restrict__ pair_recs, uint64_t num_pairs, const __grid_constant__ CameraDev cam,
                                    float small_side, float4 *__restrict__ sbox, unsigned int *__restrict__ small_boxes)
{
    const uint64_t k = (uint64_t) blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= num_pairs)
        return;
    const CullCamera cc = cull_camera(cam);
    const float4 *r = pair_recs + 5 * k;
    const float4 f0 = r[0], f1 = r[1], f2 = r[2], f3 = r[3], f4 = r[4];
    double a[4], b[4];
    triangle_screen_box(f0.x, f0.z, f1.x, f1.z, f2.x, f2.z, f3.x, f3.z, f4.x, __float_as_uint(f4.z), cam, cc, a);
    triangle_screen_box(f0.y, f0.w, f1.y, f1.w, f2.y, f2.w, f3.y, f3.w, f4.y, __float_as_uint(f4.w), cam, cc, b);
    const float4 out = make_float4(__double2float_rd(fmin(a[0], b[0])), __double2float_ru(fmax(a[1], b[1])),
                                   __double2float_rd(fmin(a[2], b[2])), __double2float_ru(fmax(a[3], b[3])));
    sbox[k] = out;
    if (fmaxf(out.y - out.x, out.w - out.z) <= small_side)
        atomicAdd(small_boxes, 1u);
}

} // namespace

void launch_screen_boxes(const float4 *pair_recs, uint64_t num_pairs, const CameraDev& cam, float4 *sbox,
                         unsigned int *small_boxes, cudaStream_t stream)
{
    cudaMemsetAsync(small_boxes, 0, sizeof(unsigned int), stream);
    // kScreenCullSmallPixels pixels: the image spans 2 fov_xs over width_f pixels
    const float small_side = kScreenCullSmallPixels * (2.0f * cam.fov_xs / cam.width_f);
    if (num_pairs)
        screen_boxes_kernel<<<blocks_for(num_pairs, 128), 128, 0, stream>>>(pair_recs, num_pairs, cam, small_side, sbox, small_boxes);
}

void launch_origin_relative_pairs(const float4 *pair_recs, uint64_t num_pairs, const float origin[3], float4 *rel,
                                  cudaStream_t stream)
{
    if (num_pairs)
        origin_relative_pairs_kernel<<<blocks_for(num_pairs, 256), 256, 0, stream>>>(pair_recs, num_pairs, origin[0], origin[1],
                                                                                     origin[2], rel);
}

void launch_pair_counts(const uint32_t *pcell_start, uint64_t pcells, uint32_t *counts, cudaStream_t stream)
{
    pair_count_kernel<<<blocks_for(pcells + 1, 256), 256, 0, stream>>>(pcell_start, pcells, counts);
}

void launch_pack_pairs(const uint32_t *pcell_start, const uint32_t *ppair_start, uint64_t pcells, const float4 *cell_tris,
                       float4 *pair_recs, cudaStream_t stream)
{
    pack_pairs_kernel<<<blocks_for(pcells, 256), 256, 0, stream>>>(pcell_start, ppair_start, pcells, cell_tris, pair_recs);
}

void launch_pack_cell_tris(const float *vtx, const uint32_t *tri, const uint32_t *tri_index, uint64_t num_refs,
                           float4 *cell_tris, float4 *cell_tris_b, cudaStream_t stream)
{
    if (num_refs)
        pack_cell_tris_kernel<<<blocks_for(num_refs, 256), 256, 0, stream>>>(vtx, tri, tri_index, num_refs,
                                                                             cell_tris, cell_tris_b);
}

void launch_pack_normals(const float *vtx, const uint32_t *tri, uint32_t num_tri, float4 *tri_normals,
                         cudaStream_t stream)
{
    if (num_tri)
        pack_normals_kernel<<<blocks_for(num_tri, 256), 256, 0, stream>>>(vtx, tri, num_tri, tri_normals);
}

void launch_cell_occupancy(const uint32_t *cell_start, uint64_t num_cells, uint32_t *cell_occ, cudaStream_t stream)
{
    const uint64_t words = (num_cells + 31) / 32;
    if (words)
        cell_occupancy_kernel<<<blocks_for(words, 256), 256, 0, stream>>>(cell_start, num_cells, cell_occ);
}

void launch_pad_grid(const uint32_t *cell_start, const uint32_t dim[3], uint32_t *pcell_start, uint32_t *pcell_occ,
                     cudaStream_t stream)
{
    const uint64_t pcells = (uint64_t) (dim[0] + 2) * (dim[1] + 2) * (dim[2] + 2);
    pad_cell_start_kernel<<<blocks_for(pcells + 1, 256), 256, 0, stream>>>(cell_start, dim[0], dim[1], dim[2], pcell_start);
    pad_cell_occ_kernel<<<blocks_for((pcells + 31) / 32, 256), 256, 0, stream>>>(pcell_start, dim[0], dim[1], dim[2], pcell_occ);
}

void launch_distance_map(const uint32_t *pcell_occ, const uint32_t dim[3], uint8_t *pcell_dist, cudaStream_t stream)
{
    const uint32_t pdx = dim[0] + 2, pdy = dim[1] + 2, pdz = dim[2] + 2;
    const uint64_t plane = (uint64_t) pdx * pdz;
    // x: one thread per (z, y) line; z: one per (x, y), lines start at x + y * plane; y: one per (x, z), start x + z * pdx
    dist_sweep_x_kernel<<<blocks_for((uint64_t) pdz * pdy, 128), 128, 0, stream>>>(pcell_occ, pdx, (uint64_t) pdz * pdy, pcell_dist);
    dist_sweep_kernel<<<blocks_for((uint64_t) pdx * pdy, 128), 128, 0, stream>>>(pcell_dist, pdz, pdx, pdx, plane, (uint64_t) pdx * pdy);
    dist_sweep_kernel<<<blocks_for(plane, 128), 128, 0, stream>>>(pcell_dist, pdy, plane, (uint32_t) plane, 0, plane);
}

void launch_narrow_offsets(const uint64_t *off64, uint64_t n, uint32_t *off32, cudaStream_t stream)
{
    if (n)
        narrow_offsets_kernel<<<blocks_for(n, 256), 256, 0, stream>>>(off64, n, off32);
}

void launch_widen_offsets(const uint32_t *off32, uint64_t n, uint64_t *off64, cudaStream_t stream)
{
    if (n)
        widen_offsets_kernel<<<blocks_for(n, 256), 256, 0, stream>>>(off32, n, off64);
}

} // namespace rtm
