// Ray queries on caller-supplied rays that live on the device (cuda_trace_query_rays): the closest hit up to t_max,
// or only whether there is one (occlusion).
//
// The traversal is K1's warp-cooperative walk (warp_trace.cuh) with 32 consecutive rays per warp: the occupancy map
// staged in shared memory or the distance map, lock-step phases with warp votes, and the packed-fp32 pair test on the
// absolute pair records for Moeller-Trumbore.  The bound and the any-hit exit are template parameters, so the
// unbounded closest-hit instantiation does exactly K1's work per ray.  Persistent CTAs stage the map once and take
// 32-ray groups by a static grid stride: no work counter, so queries on different streams share nothing writable.
// Only immutable scene arrays are read (not pair_recs_rel, which frames rewrite per camera).
//
// Compiled with -fmad=false (see rt_device.cuh).
#include "trace_kernels.cuh"
#include "warp_trace.cuh"

namespace rtm
{

namespace
{

constexpr int kQueryThreads = 1024;
constexpr size_t kOptInDynamicSmem = 48 * 1024;

template <int VARIANT, bool OCCLUSION, bool BOUNDED, int OCC_MODE>
__global__ void __launch_bounds__(kQueryThreads) ray_query_kernel(const __grid_constant__ RayQueryParams p)
{
    extern __shared__ uint32_t s_occ[];
    if (OCC_MODE == kOccSmemBits)
        for (uint32_t i = threadIdx.x; i < p.occ_smem_words; i += blockDim.x)
            s_occ[i] = __ldg(&p.grid.pcell_occ[i]);
    if (OCC_MODE == kOccSmemBytes)
        for (uint32_t i = threadIdx.x; i < p.occ_smem_words; i += blockDim.x)
        {
            const uint32_t nib = (__ldg(&p.grid.pcell_occ[i >> 3]) >> ((i & 7u) * 4u)) & 0xFu;
            s_occ[i] = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
        }
    if (OCC_MODE == kOccSmemBits || OCC_MODE == kOccSmemBytes)
        __syncthreads();

    PackedUnits pku;
    pku.one = p.pk_one;
    pku.minus_one = p.pk_minus_one;
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp = ((uint64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t stride = ((uint64_t) gridDim.x * blockDim.x) >> 5;
    for (uint64_t base = warp * 32; base < p.n; base += stride * 32) // warp-uniform
    {
        const uint64_t i = base + lane;
        const bool in_batch = i < p.n;
        float3 o = make_float3(0.0f, 0.0f, 0.0f), d = make_float3(0.0f, 0.0f, 1.0f);
        float t_max = p.t_max_all;
        if (in_batch)
        {
            o = make_float3(__ldg(p.origins + 3 * i), __ldg(p.origins + 3 * i + 1), __ldg(p.origins + 3 * i + 2));
            d = make_float3(__ldg(p.dirs + 3 * i), __ldg(p.dirs + 3 * i + 1), __ldg(p.dirs + 3 * i + 2));
            if (p.t_max)
                t_max = __ldg(p.t_max + i);
        }
        // t_max <= 0 or NaN: nothing can be accepted (t >= 0 is required), a miss without walking
        const bool valid = in_batch && (!BOUNDED || t_max > 0.0f);
        // the range-check-free divisions of the DDA set-up hold for |dir| <= 1 per component (as for camera rays)
        const bool unit = fabsf(d.x) <= 1.0f && fabsf(d.y) <= 1.0f && fabsf(d.z) <= 1.0f;
        const bool fast = p.fast_math && __all_sync(kFullMask, unit || !valid);
        Hit hit;
        hit.t = hit.u = hit.v = 0.0f;
        hit.tri = 0xFFFFFFFFu;
        const bool is_hit = warp_grid_intersect<VARIANT, false, OCC_MODE, true, BOUNDED, OCCLUSION>(
            p.grid, s_occ, o, d, valid, hit, nullptr, pku, fast, t_max);
        if (!in_batch)
            continue;
        if (OCCLUSION)
        {
            p.occluded[i] = is_hit ? 1 : 0;
        }
        else
        {
            p.tri[i] = is_hit ? hit.tri : 0xFFFFFFFFu;
            if (p.t) p.t[i] = is_hit ? hit.t : 0.0f;
            if (p.u) p.u[i] = is_hit ? hit.u : 0.0f;
            if (p.v) p.v[i] = is_hit ? hit.v : 0.0f;
        }
    }
}

template <int VARIANT, bool OCCLUSION, bool BOUNDED, int OCC_MODE>
void launch_instance(const RayQueryParams& p, int grid_blocks, cudaStream_t stream)
{
    const size_t smem = sizeof(uint32_t) * p.occ_smem_words;
    if (smem > kOptInDynamicSmem)
    {
        // once per device and size, not on every launch
        static size_t opted_in[64] = {};
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev < 0 || dev >= 64 || opted_in[dev] < smem)
        {
            cudaFuncSetAttribute(ray_query_kernel<VARIANT, OCCLUSION, BOUNDED, OCC_MODE>,
                                 cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
            if (dev >= 0 && dev < 64)
                opted_in[dev] = smem;
        }
    }
    ray_query_kernel<VARIANT, OCCLUSION, BOUNDED, OCC_MODE><<<grid_blocks, kQueryThreads, smem, stream>>>(p);
}

template <int VARIANT, bool OCCLUSION, bool BOUNDED>
void launch_mode(const RayQueryParams& p, int grid_blocks, cudaStream_t stream)
{
    if (p.occ_mode == kOccSmemBytes)
        launch_instance<VARIANT, OCCLUSION, BOUNDED, kOccSmemBytes>(p, grid_blocks, stream);
    else if (p.occ_mode == kOccSmemBits)
        launch_instance<VARIANT, OCCLUSION, BOUNDED, kOccSmemBits>(p, grid_blocks, stream);
    else if (p.occ_mode == kOccGlobalDist)
        launch_instance<VARIANT, OCCLUSION, BOUNDED, kOccGlobalDist>(p, grid_blocks, stream);
    else
        launch_instance<VARIANT, OCCLUSION, BOUNDED, kOccGlobalBits>(p, grid_blocks, stream);
}

template <int VARIANT>
void launch_kind(const RayQueryParams& p, bool occlusion, bool bounded, int grid_blocks, cudaStream_t stream)
{
    // occlusion is always the bounded walk: with t_max = +inf it is the same walk (the crossing test is strict)
    if (occlusion)
        launch_mode<VARIANT, true, true>(p, grid_blocks, stream);
    else if (bounded)
        launch_mode<VARIANT, false, true>(p, grid_blocks, stream);
    else
        launch_mode<VARIANT, false, false>(p, grid_blocks, stream);
}

} // namespace

int ray_query_threads() { return kQueryThreads; }

void launch_ray_query(const RayQueryParams& p, uint32_t variant, bool occlusion, bool bounded, int grid_blocks,
                      cudaStream_t stream)
{
    if (p.n == 0 || grid_blocks <= 0)
        return;
    if (variant == kVariantBary)
        launch_kind<kVariantBary>(p, occlusion, bounded, grid_blocks, stream);
    else
        launch_kind<kVariantMT>(p, occlusion, bounded, grid_blocks, stream);
}

} // namespace rtm
