// K1 trace_tiles, K2 build_sample_table and the ray-batch kernel (sm_100a).
//
// K1 supersedes Renderer::RenderTile (reference renderer.cpp:43-136) together with the worker
// pool that calls it (framebuffer.cpp:59-92): persistent warps pull 8x4-pixel strips of the
// requested tiles from an atomic counter; the 32 lanes of a warp take the strip's rays in
// (pixel, sample) order with the SAMPLE index fastest, so a warp works on 32/spp neighbouring
// pixels at a time and its rays walk (nearly) the same cells.  Ray generation, grid entry,
// 3D-DDA, ray/triangle tests, shading, the in-order sample average, gamma and BGRA8 packing are
// all in this one kernel; the only global write is one uint32 per pixel.
//
// Compiled with -fmad=false (see rt_device.cuh).
#include "trace_kernels.cuh"
#include "warp_trace.cuh"

#include <map>
#include <mutex>

namespace rtm
{

namespace
{

constexpr unsigned kFull = 0xFFFFFFFFu;
// the 48 KB a kernel gets without opting in cover static + dynamic shared memory; K1 has ~21 KB of static
constexpr size_t kOptInDynamicSmem = 24 * 1024;

// One sample per lane; ALL lanes of the warp call this together (valid == false: no ray)
template <int VARIANT, bool KEEP_HITS, bool COUNT, int OCC_MODE, bool RCP_GUARD, bool CULL>
__device__ __forceinline__ float3 trace_sample(const TraceParams& p, const void *s_occ, bool valid,
                                               uint32_t px, uint32_t py, uint32_t s, const float2 *smp, Counters *cnt)
{
    constexpr bool FROM_HITS = VARIANT == kVariantFromHits;
    constexpr bool ALT = VARIANT >= kVariantMTAlt && !FROM_HITS;
    constexpr int TRI_VARIANT = ALT ? VARIANT - kVariantMTAlt : VARIANT;
    Hit hit;
    hit.t = hit.u = hit.v = 0.0f;
    hit.tri = 0xFFFFFFFFu;
    bool is_hit = false;
    if constexpr (FROM_HITS)
    {
        // the traversal was done by K7 trace_pool (pool_trace.cu): take the sample's hit record as it left it
        if (valid)
        {
            const size_t k = ((size_t) py * p.width + px) * p.spp + s;
            hit.tri = p.hit_tri[k];
            hit.u = p.hit_u[k];
            hit.v = p.hit_v[k];
            is_hit = hit.tri != 0xFFFFFFFFu;
        }
    }
    else
    {
        float3 o, d;
        float2 img;
        const float2 off = smp[valid ? s : 0];
        generate_ray<ALT>(p.cam, px, py, off.x, off.y, o, d, CULL ? &img : nullptr);
        if (COUNT && valid) cnt->rays++;
        PackedUnits pku;
        pku.one = p.pk_one;
        pku.minus_one = p.pk_minus_one;
        if constexpr (CULL)
            is_hit = warp_grid_intersect<TRI_VARIANT, COUNT, OCC_MODE, RCP_GUARD, false, false, CULL>(
                p.grid, s_occ, o, d, valid, hit, cnt, pku, p.cam.fast_math != 0, FLT_MAX, p.pair_sbox, img);
        else
            is_hit = warp_grid_intersect<TRI_VARIANT, COUNT, OCC_MODE, RCP_GUARD>(p.grid, s_occ, o, d, valid, hit, cnt, pku, p.cam.fast_math != 0);
        if (COUNT && is_hit) cnt->hits++;
        if (KEEP_HITS && valid)
        {
            const size_t k = ((size_t) py * p.width + px) * p.spp + s;
            p.hit_tri[k] = is_hit ? hit.tri : 0xFFFFFFFFu;
            if (p.hit_t) p.hit_t[k] = is_hit ? hit.t : 0.0f;
            if (p.hit_u) p.hit_u[k] = is_hit ? hit.u : 0.0f;
            if (p.hit_v) p.hit_v[k] = is_hit ? hit.v : 0.0f;
        }
    }
    float3 rgb = make_float3(0.0f, 0.0f, 0.0f);
    if (valid)
        rgb = shade_sample<ALT>(p.grid, is_hit, hit, py, p.cam.height_f, p.shade_mode);
    return rgb;
}

// Two-level completion count of a row band (called by lane 0 after a warp barrier).  Level 1, per GPU and in
// its own memory: pieces of strips finished, a release at GPU scope -- cheap, once per few strips (no acquire
// here: that would invalidate the SM's L1 and cost 6 % of the frame).  Level 2: the warp whose increment
// completes this GPU's share of the band turns it into an acquire with a fence and bumps the band's counter
// behind the (possibly remote) framebuffer, once per band and GPU, with a release at system scope: the counter's
// reader is a copy engine or another GPU, neither inside this GPU's .gpu scope.  Every pixel store of the band on
// this GPU happens-before that release (warp barrier -> level-1 release -> level-1 read + acquire fence by the
// completing warp -> its release; causality order is cumulative), so whoever waits on the band counter sees the
// pixels.  A system-scope release per strip batch instead costs +35 % kernel time on the GPUs that store over NVLink.
__device__ __forceinline__ void release_add(const TraceParams& p, uint32_t band, uint32_t count)
{
    uint32_t before;
    asm volatile("atom.release.gpu.global.add.u32 %0, [%1], %2;" : "=r"(before) : "l"(p.band_local + band), "r"(count) : "memory");
    if (before + count == p.band_share[band])
    {
        asm volatile("fence.acq_rel.sys;" ::: "memory");
        asm volatile("red.release.sys.global.add.u32 [%0], %1;" :: "l"(p.band_done + band), "r"(1u) : "memory");
    }
}

template <int VARIANT, bool KEEP_HITS, bool COUNT, int OCC_MODE, bool RCP_GUARD, bool BANDS, bool CULL>
__global__ void __launch_bounds__(kTraceMaxThreads) trace_tiles_kernel(const __grid_constant__ TraceParams p)
{
    // shared memory: [sample table (renderer.cpp:49-60), spp x float2]
    //                [padded occupancy map: p.occ_smem_words 32-bit words of bits (mode 1) or of
    //                 bytes, four cells per word (mode 2)]
    extern __shared__ float2 s_mem[];
    float2 *s_smp = s_mem;
    uint32_t *s_occ = reinterpret_cast<uint32_t *>(s_mem + p.spp);
    if (OCC_MODE == kOccSmemBits)
        for (uint32_t i = threadIdx.x; i < p.occ_smem_words; i += blockDim.x)
            s_occ[i] = __ldg(&p.grid.pcell_occ[i]);
    if (OCC_MODE == kOccSmemBytes)
        for (uint32_t i = threadIdx.x; i < p.occ_smem_words; i += blockDim.x)
        {
            // expand 4 occupancy bits into 4 bytes (cells 4i .. 4i+3)
            const uint32_t nib = (__ldg(&p.grid.pcell_occ[i >> 3]) >> ((i & 7u) * 4u)) & 0xFu;
            s_occ[i] = (nib & 1u) | ((nib & 2u) << 7) | ((nib & 4u) << 14) | ((nib & 8u) << 21);
        }
    for (uint32_t i = threadIdx.x; i < p.spp; i += blockDim.x)
        s_smp[i] = p.smp[i];
    __syncthreads();

    const uint32_t lane = threadIdx.x & 31u;
    const float spp_f = (float) p.spp;
    Counters cnt = { 0, 0, 0, 0 };
    __shared__ float4 s_rgb[kTraceMaxThreads]; // one colour sample per lane (the in-order sum below)
    PackedUnits pku;
    pku.one = p.pk_one;
    pku.minus_one = p.pk_minus_one;

    const uint32_t slots = p.strip_w * p.strip_h;
    // finished pieces not yet published (see the band publication below): lane b holds those of row band b
    // (kMaxBands == 32), slot 0 of s_pend_total their warp-uniform sum.  In shared memory, touched once per
    // strip: as registers they would be live across the whole traversal, which is at its 64-register cap
    __shared__ uint32_t s_pend[BANDS ? kTraceMaxThreads : 1], s_pend_total[BANDS ? kTraceMaxThreads / 32 : 1];
    if (BANDS)
    {
        s_pend[threadIdx.x] = 0;
        if (lane == 0)
            s_pend_total[threadIdx.x >> 5] = 0;
        __syncwarp();
    }
    const uint32_t n_visits = p.fetch_order ? __ldg(p.visit_total) : p.shard_strips;
    const uint32_t part_slots = slots / p.split_parts;
    for (;;)
    {
        // dynamic strip scheduler: one atomic per strip per warp
        // A cancelled frame still walks its strip list -- without tracing -- so that the per-band
        // completion counts the read-back waits on are reached (framebuffer.h:32 m_threads_stop)
        uint32_t visit = 0;
        bool cancel_seen = false;
        if (lane == 0)
        {
            cancel_seen = *(volatile const uint32_t *) p.cancel == p.frame_seq;
            visit = atomicAdd(p.strip_counter, 1u);
            if (cancel_seen) // tell the host (mapped memory; only ever on a cancelled frame)
                *(volatile uint32_t *) p.cancel_seen = p.frame_seq;
        }
        visit = __shfl_sync(kFull, visit, 0);
        // a VOTE result is warp-uniform by construction, which lets the compiler keep the traversal
        // below free of divergence checks around its own votes
        const bool cancelled = __any_sync(kFull, cancel_seen);
        if (__any_sync(kFull, visit >= n_visits) || (cancelled && !(BANDS && p.band_done)))
            break;
        // `fetch` = index of the strip within this shard, taken through the cost order of the
        // previous frame when there is one (schedule.cu)
        // (broadcast through a shuffle: a loaded value is not provably warp-uniform, and everything
        // derived from it -- strip, rectangle, loop bounds -- would make the compiler guard the
        // traversal's votes with divergence checks: +3 instructions per triangle test)
        const uint32_t entry = __shfl_sync(kFull, p.fetch_order ? __ldg(&p.fetch_order[visit]) : visit, 0);
        // an entry of the cost order names a whole strip or, for a strip that was expensive in the previous
        // frame, one of its split_parts pieces (whole rounds of whole pixels -- results do not depend on it)
        const uint32_t piece = p.fetch_order ? entry >> 28 : 0u;
        const uint32_t fetch = p.fetch_order ? entry & kVisitStripMask : entry;
        const long long t_begin = p.visit_cycles ? clock64() : 0;
        const uint32_t slot_begin = piece ? (piece - 1u) * part_slots : 0u;
        const uint32_t slot_end = piece ? slot_begin + part_slots : slots;
        const uint32_t units = piece ? 1u : p.split_parts; // band counters count pieces
        // the n-th strip of this shard: strips are dealt out in chunks of p.shard_chunk consecutive
        // ids (neighbouring strips stay on one GPU / in one CTA: their rays share triangle records
        // in L1), round-robin over the shards, the owner rotating from round to round so that
        // regular cost patterns do not all land on the same shard
        const uint32_t my_chunk = fetch / p.shard_chunk, in_chunk = fetch - my_chunk * p.shard_chunk;
        const uint64_t chunk_id = (uint64_t) my_chunk * p.shard_world +
                                  (p.shard_rank + p.shard_world - my_chunk % p.shard_world) % p.shard_world;
        const uint64_t strip64 = chunk_id * p.shard_chunk + in_chunk;
        if (__any_sync(kFull, strip64 >= p.total_strips)) // (votes keep these branches provably warp-uniform)
            continue;
        const uint32_t strip = (uint32_t) strip64;

        // which tile? (upper bound over the per-tile strip prefix)
        uint32_t lo = 0, hi = p.n_tiles;
        while (hi - lo > 1)
        {
            const uint32_t mid = (lo + hi) >> 1;
            if (__ldg(&p.tile_strip_prefix[mid]) <= strip) lo = mid; else hi = mid;
        }
        const uint4 rect = __ldg(&p.tile_rects[lo]);
        const uint32_t local = strip - __ldg(&p.tile_strip_prefix[lo]);
        const uint32_t strips_x = (rect.z - rect.x + p.strip_w - 1) / p.strip_w;
        const uint32_t bx0 = rect.x + (local % strips_x) * p.strip_w;
        const uint32_t by0 = rect.y + (local / strips_x) * p.strip_h;
        const uint32_t bw = min(p.strip_w, rect.z - bx0);
        const uint32_t bh = min(p.strip_h, rect.w - by0);

        if (cancelled)
        {
            // nothing rendered, but the strip counts as finished for the read-back
        }
        else if (p.spp <= 32)
        {
            // 32 / spp whole pixels per round; lane = (pixel in round) * spp + sample.  The 32
            // pixel slots of the 8x4 strip are visited in 2x2-quad (Morton) order, so the pixels
            // of one round form a compact block (spp 16: 2x1, spp 4: 4x2, spp 1: 8x4) whose rays
            // walk nearly the same cells.
            const uint32_t ppr = 32u / p.spp;
            const uint32_t pl = lane / p.spp, s = lane - pl * p.spp;
            // (uniform loop bounds + a vote to skip the rounds outside this piece: bounds derived from the
            // visit entry would count as possibly divergent and bring the vote guards back)
            for (uint32_t pbase = 0; pbase < slots; pbase += ppr)
            {
                const uint32_t slot = pbase + pl;
                const uint32_t ox = (slot & 1u) | ((slot >> 1) & 2u) | ((slot >> 2) & 4u);
                const uint32_t oy = ((slot >> 1) & 1u) | ((slot >> 2) & 2u);
                const bool active = pl < ppr && slot >= slot_begin && slot < slot_end && ox < bw && oy < bh;
                if (!__any_sync(kFull, active))
                    continue;
                const uint32_t px = bx0 + ox, py = by0 + oy;
                const float3 rgb = trace_sample<VARIANT, KEEP_HITS, COUNT, OCC_MODE, RCP_GUARD, CULL>(p, s_occ, active, px, py, s, s_smp, &cnt);
                // col += sample, smp = 0..N-1 in order (renderer.cpp:87-122).  The samples of a pixel sit in
                // consecutive lanes; they go through shared memory -- one 16-byte store per lane, one broadcast
                // load per term -- and every lane of the pixel adds them up in sample order (red and green as one
                // packed add): a third of the instructions of a shuffle per channel and term.
                s_rgb[threadIdx.x] = make_float4(rgb.x, rgb.y, rgb.z, 0.0f);
                __syncwarp();
                f32x2 acc_rg = pk2(0.0f, 0.0f);
                float acc_b = 0.0f;
                // (lanes beyond the round's last pixel read that pixel's slots: inside their warp's 32)
                const float4 *mine = s_rgb + (threadIdx.x & ~31u) + min(pl, ppr - 1u) * p.spp;
                for (uint32_t k = 0; k < p.spp; k++)
                {
                    const float4 v = mine[k];
                    acc_rg = add2(pk2(v.x, v.y), acc_rg, pku);
                    acc_b += v.z;
                }
                __syncwarp();
                float3 acc;
                unpk2(acc_rg, acc.x, acc.y);
                acc.z = acc_b;
                if (active && s == 0)
                    p.framebuffer[(size_t) py * p.width + px] = resolve_pixel(acc, spp_f, p.gamma != 0);
            }
        }
        else
        {
            // one pixel at a time, 32 samples per round.  (No `continue` in this loop: with one the
            // compiler treats the whole strip loop as possibly divergent and guards every vote.)
            for (uint32_t slot = 0; slot < slots; slot++)
            {
                const uint32_t ox = (slot & 1u) | ((slot >> 1) & 2u) | ((slot >> 2) & 4u);
                const uint32_t oy = ((slot >> 1) & 1u) | ((slot >> 2) & 2u);
                // clipped strips: the pixel lies outside the tile; split strips: outside this piece
                const bool inside = slot >= slot_begin && slot < slot_end && ox < bw && oy < bh;
                const uint32_t px = bx0 + ox, py = by0 + oy;
                float3 acc = make_float3(0.0f, 0.0f, 0.0f);
                for (uint32_t sb = 0; sb < p.spp; sb += 32)
                {
                    const uint32_t s = sb + lane;
                    const float3 rgb = trace_sample<VARIANT, KEEP_HITS, COUNT, OCC_MODE, RCP_GUARD, CULL>(p, s_occ, inside && s < p.spp, px, py, s, s_smp, &cnt);
                    const uint32_t n = min(32u, p.spp - sb);
                    for (uint32_t k = 0; k < n; k++)
                    {
                        acc.x += __shfl_sync(kFull, rgb.x, (int) k);
                        acc.y += __shfl_sync(kFull, rgb.y, (int) k);
                        acc.z += __shfl_sync(kFull, rgb.z, (int) k);
                    }
                }
                if (inside && lane == 0)
                    p.framebuffer[(size_t) py * p.width + px] = resolve_pixel(acc, spp_f, p.gamma != 0);
            }
        }
        // this visit's cost; schedule.cu sums the pieces per strip for the next frame's visiting order.  Every lane
        // stores the same word (one transaction): a lane-0 branch, or an atomic in inline PTX, would make the
        // compiler guard the traversal's votes again
        if (p.visit_cycles)
            p.visit_cycles[visit] = (uint32_t) min(__shfl_sync(kFull, clock64() - t_begin, 0), 0x0FFFFFFFll);
        // (compiled out of the BANDS == false instantiation: the warp barrier in here makes the compiler
        // guard every vote of the traversal with a divergence check, +3 instructions per triangle test)
        if (BANDS && p.band_done)
        {
            // Publish "these strips' pixels are stored" per row band.  The publication is a release: a warp
            // barrier orders every lane's pixel stores before the release-increments, whose fence is the
            // expensive part -- so finished pieces are collected per warp, lane b keeping the count of band b
            // (consecutive strips of one warp are thousands of strip ids apart and rarely share a band), and
            // published a few strips at a time (band_flush_units): one fence, then one increment per band touched.
            // The host's copy stream waits on these counters and ships each row band to the host while later
            // bands are still being traced.
            const uint32_t b0 = by0 / p.band_rows, b1 = (by0 + bh - 1) / p.band_rows;
            // (a strip straddling two bands counts in both)
            const uint32_t my_pend = s_pend[threadIdx.x] + (lane == b0 ? units : 0u) + ((b1 != b0 && lane == b1) ? units : 0u);
            const uint32_t pend_total = s_pend_total[threadIdx.x >> 5] + units;
            const bool flush = pend_total >= p.band_flush_units;
            __syncwarp(); // unconditional, at the top level of the strip loop (a barrier under a
                          // data-dependent branch would make the compiler guard every vote in the loop)
            if (flush && my_pend)
                release_add(p, lane, my_pend);
            s_pend[threadIdx.x] = flush ? 0u : my_pend;
            if (lane == 0)
                s_pend_total[threadIdx.x >> 5] = flush ? 0u : pend_total;
            __syncwarp();
        }
    }
    if (BANDS && p.band_done)
    {
        __syncwarp();
        if (s_pend[threadIdx.x])
            release_add(p, lane, s_pend[threadIdx.x]);
    }

    if (COUNT)
    {
        atomicAdd(&p.counters->rays, cnt.rays);
        atomicAdd(&p.counters->cells, cnt.cells);
        atomicAdd(&p.counters->tri_tests, cnt.tri_tests);
        atomicAdd(&p.counters->hits, cnt.hits);
    }
}

template <int VARIANT, bool MAILBOX>
__global__ void __launch_bounds__(128) intersect_rays_kernel(const __grid_constant__ RayBatchParams p)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n)
        return;
    const float3 o = make_float3(p.origins[3 * (size_t) i], p.origins[3 * (size_t) i + 1], p.origins[3 * (size_t) i + 2]);
    const float3 d = make_float3(p.dirs[3 * (size_t) i], p.dirs[3 * (size_t) i + 1], p.dirs[3 * (size_t) i + 2]);
    Hit hit;
    hit.t = hit.u = hit.v = 0.0f;
    hit.tri = 0xFFFFFFFFu;
    const bool is_hit = grid_intersect<VARIANT, false, MAILBOX>(p.grid, o, d, hit, nullptr, p.mailbox_stats);
    p.tri[i] = is_hit ? hit.tri : 0xFFFFFFFFu;
    p.t[i] = is_hit ? hit.t : 0.0f;
    p.u[i] = is_hit ? hit.u : 0.0f;
    p.v[i] = is_hit ? hit.v : 0.0f;
}

// renderer.cpp:157-197: closest hit over ALL triangles in index order (strict "cur_t < t": first wins ties)
__global__ void __launch_bounds__(128) brute_force_kernel(const float *__restrict__ vtx, const uint32_t *__restrict__ tri,
                                                          uint32_t num_tri, const __grid_constant__ RayBatchParams p)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n)
        return;
    const float3 o = make_float3(p.origins[3 * (size_t) i], p.origins[3 * (size_t) i + 1], p.origins[3 * (size_t) i + 2]);
    const float3 d = make_float3(p.dirs[3 * (size_t) i], p.dirs[3 * (size_t) i + 1], p.dirs[3 * (size_t) i + 2]);
    float best_t = FLT_MAX, best_u = 0.0f, best_v = 0.0f;
    uint32_t best = 0xFFFFFFFFu;
    for (uint32_t k = 0; k < num_tri; k++)
    {
        const uint32_t *tr = tri + (size_t) k * 6;
        const float *p0 = vtx + (size_t) tr[0] * 6, *p1 = vtx + (size_t) tr[1] * 6, *p2 = vtx + (size_t) tr[2] * 6;
        const float4 a = make_float4(p0[0], p0[1], p0[2], 0.0f);
        const float4 b = make_float4(p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2], 0.0f);
        const float4 c = make_float4(p2[0] - p0[0], p2[1] - p0[1], p2[2] - p0[2], 0.0f);
        float ct, cu, cv;
        if (ray_tri_mt(o, d, a, b, c, ct, cu, cv) && ct < best_t)
        {
            best_t = ct; best_u = cu; best_v = cv; best = k;
        }
    }
    const bool hit = best_t != FLT_MAX; // renderer.cpp:196
    p.tri[i] = hit ? best : 0xFFFFFFFFu;
    p.t[i] = hit ? best_t : 0.0f;
    p.u[i] = hit ? best_u : 0.0f;
    p.v[i] = hit ? best_v : 0.0f;
}

// triangle.h:172-181: squared distance from p to the segment a-b
__device__ __forceinline__ float seg_dist_sq(const float a[3], const float b[3], const float p[3])
{
    const float abx = b[0] - a[0], aby = b[1] - a[1], abz = b[2] - a[2];
    const float len_sq = dot_ref(abx, aby, abz, abx, aby, abz);
    float t = dot_ref(p[0] - a[0], p[1] - a[1], p[2] - a[2], abx, aby, abz) / len_sq;
    t = t < 0.0f ? 0.0f : (t > 1.0f ? 1.0f : t); // Clamp (lin_alg.h:205-212)
    const float qx = p[0] - (a[0] + abx * t), qy = p[1] - (a[1] + aby * t), qz = p[2] - (a[2] + abz * t);
    return dot_ref(qx, qy, qz, qx, qy, qz);
}

// triangle.h:183-198 DistancePointTri = ComputeBarycentric (:133-156) then plane distance or nearest edge
__device__ float point_tri_distance(const float p[3], const float v0[3], const float v1[3], const float v2[3])
{
    const float e0x = v2[0] - v0[0], e0y = v2[1] - v0[1], e0z = v2[2] - v0[2];
    const float e1x = v1[0] - v0[0], e1y = v1[1] - v0[1], e1z = v1[2] - v0[2];
    const float e2x = p[0] - v0[0], e2y = p[1] - v0[1], e2z = p[2] - v0[2];
    const float d00 = dot_ref(e0x, e0y, e0z, e0x, e0y, e0z), d01 = dot_ref(e0x, e0y, e0z, e1x, e1y, e1z);
    const float d02 = dot_ref(e0x, e0y, e0z, e2x, e2y, e2z), d11 = dot_ref(e1x, e1y, e1z, e1x, e1y, e1z);
    const float d12 = dot_ref(e1x, e1y, e1z, e2x, e2y, e2z);
    const float inv_denom = 1.0f / (d00 * d11 - d01 * d01);
    const float u = (d00 * d12 - d01 * d02) * inv_denom, v = (d11 * d02 - d01 * d12) * inv_denom;
    if ((u >= 0.0f) && (v >= 0.0f) && (u + v < 1.0f))
    {
        const float w = 1.0f - u - v; // BarycentricInterpolate(u, v, v0, v1, v2) (triangle.h:158-161)
        const float qx = p[0] - (v1[0] * u + v2[0] * v + v0[0] * w);
        const float qy = p[1] - (v1[1] * u + v2[1] * v + v0[1] * w);
        const float qz = p[2] - (v1[2] * u + v2[2] * v + v0[2] * w);
        return sqrtf(dot_ref(qx, qy, qz, qx, qy, qz));
    }
    const float a = seg_dist_sq(v0, v1, p), b = seg_dist_sq(v0, v2, p), c = seg_dist_sq(v1, v2, p);
    const float bc = (c < b) ? c : b; // std::min(b, c)
    return sqrtf((bc < a) ? bc : a);  // std::min(a, min(b, c))
}

// renderer.cpp:24-41 (RayMarch) over renderer.cpp:138-155 (DistanceBruteForce)
__global__ void __launch_bounds__(128) ray_march_kernel(const float *__restrict__ vtx, const uint32_t *__restrict__ tri,
                                                        uint32_t num_tri, uint32_t n, const float *__restrict__ origins,
                                                        const float *__restrict__ dirs, uint32_t *__restrict__ hit_out,
                                                        float *__restrict__ t_out)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n)
        return;
    const float o[3] = { origins[3 * (size_t) i], origins[3 * (size_t) i + 1], origins[3 * (size_t) i + 2] };
    const float d[3] = { dirs[3 * (size_t) i], dirs[3 * (size_t) i + 1], dirs[3 * (size_t) i + 2] };
    float t = 0.0f;
    uint32_t hit = 0;
    for (uint32_t step = 0; step < 128u; step++)
    {
        const float pos[3] = { o[0] + d[0] * t, o[1] + d[1] * t, o[2] + d[2] * t };
        float dist = FLT_MAX;
        for (uint32_t k = 0; k < num_tri; k++)
        {
            const uint32_t *tr = tri + (size_t) k * 6;
            const float dk = point_tri_distance(pos, vtx + (size_t) tr[0] * 6, vtx + (size_t) tr[1] * 6, vtx + (size_t) tr[2] * 6);
            dist = (dk < dist) ? dk : dist; // std::min(dist, dk)
        }
        t += dist;
        if (dist < 0.001f)
        {
            hit = 1;
            break;
        }
    }
    hit_out[i] = hit;
    t_out[i] = t;
}

// K2: renderer.cpp:49-60 -> smp[s] = (Hammersley(s,0,N) - 0.5f, Hammersley(s,1,N) - 0.5f) with
// sampling.h:113-120 / sampling.cpp:194-210 in fp64 (dim 0: double(n)/double(N); dim 1: radical
// inverse base 2), rounded to fp32 by the store.  No FMA: -fmad=false covers fp64 too.
__global__ void sample_table_kernel(float2 *smp, uint32_t spp)
{
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= spp)
        return;
    const double inv_base = 1.0 / 2.0;
    double inv_base_i = inv_base, val = 0.0;
    for (uint32_t n = s; n > 0; n /= 2)
    {
        const uint32_t digit = n % 2;
        val += digit * inv_base_i;
        inv_base_i *= inv_base;
    }
    const double x = (double) s / (double) spp;
    smp[s] = make_float2((float) (x - 0.5), (float) (val - 0.5));
}

// The instance set of trace_tiles_kernel.  The plain kernel (no hit records, no counters, not an alternate) exists with
// and without the rcp range guard (scenes larger than 1e14 units) and with and without the row-band completion
// counters; every other kernel carries both
template <int VARIANT, bool KEEP_HITS, bool COUNT, int OCC_MODE, bool CULL>
TraceTilesKernel instance_by_flags(bool rcp_guard, bool bands)
{
    if constexpr (!KEEP_HITS && !COUNT && VARIANT < kVariantMTAlt)
    {
        if (!rcp_guard && !bands) return trace_tiles_kernel<VARIANT, false, false, OCC_MODE, false, false, CULL>;
        if (!rcp_guard)           return trace_tiles_kernel<VARIANT, false, false, OCC_MODE, false, true, CULL>;
        if (!bands)               return trace_tiles_kernel<VARIANT, false, false, OCC_MODE, true, false, CULL>;
    }
    return trace_tiles_kernel<VARIANT, KEEP_HITS, COUNT, OCC_MODE, true, true, CULL>;
}

template <int VARIANT, bool KEEP_HITS, bool COUNT, bool CULL>
TraceTilesKernel instance_by_occ(int occ_mode, bool rcp_guard, bool bands)
{
    switch (occ_mode)
    {
        case kOccSmemBits: return instance_by_flags<VARIANT, KEEP_HITS, COUNT, kOccSmemBits, CULL>(rcp_guard, bands);
        case kOccSmemBytes: return instance_by_flags<VARIANT, KEEP_HITS, COUNT, kOccSmemBytes, CULL>(rcp_guard, bands);
        case kOccGlobalDist: return instance_by_flags<VARIANT, KEEP_HITS, COUNT, kOccGlobalDist, CULL>(rcp_guard, bands);
        default: return instance_by_flags<VARIANT, KEEP_HITS, COUNT, kOccGlobalBits, CULL>(rcp_guard, bands);
    }
}

// the screen cull exists for kVariantMTRel only: the boxes belong to the origin-relative records
template <int VARIANT, bool KEEP_HITS, bool COUNT>
TraceTilesKernel instance_by_cull(int occ_mode, bool rcp_guard, bool bands, bool cull)
{
    if constexpr (VARIANT == kVariantMTRel)
        if (cull)
            return instance_by_occ<VARIANT, KEEP_HITS, COUNT, true>(occ_mode, rcp_guard, bands);
    return instance_by_occ<VARIANT, KEEP_HITS, COUNT, false>(occ_mode, rcp_guard, bands);
}

// the work counters exist for variants 0 and 1 only, the hit records for every variant that traverses
template <int VARIANT>
TraceTilesKernel instance_by_records(bool keep_hits, bool count, int occ_mode, bool rcp_guard, bool bands, bool cull)
{
    constexpr bool kCounts = VARIANT == kVariantMT || VARIANT == kVariantBary, kHits = VARIANT != kVariantFromHits;
    if constexpr (kCounts)
        if (count)
            return keep_hits ? instance_by_cull<VARIANT, true, true>(occ_mode, rcp_guard, bands, cull)
                             : instance_by_cull<VARIANT, false, true>(occ_mode, rcp_guard, bands, cull);
    if constexpr (kHits)
        if (keep_hits)
            return instance_by_cull<VARIANT, true, false>(occ_mode, rcp_guard, bands, cull);
    return instance_by_cull<VARIANT, false, false>(occ_mode, rcp_guard, bands, cull);
}

// opt in to large dynamic shared memory once per device, kernel and size, not on every launch
void opt_in_smem(TraceTilesKernel k, size_t smem)
{
    if (smem <= kOptInDynamicSmem)
        return;
    static std::mutex mtx;
    static std::map<std::pair<TraceTilesKernel, int>, size_t> opted_in;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mtx);
    size_t& done = opted_in[{ k, dev }];
    if (done < smem && cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem) == cudaSuccess)
        done = smem;
}

} // namespace

TraceTilesKernel trace_tiles_instance(uint32_t variant, bool keep_hits, bool count, int occ_mode, bool rcp_guard, bool bands,
                                      bool cull)
{
    switch (variant)
    {
        case kVariantMT: return instance_by_records<kVariantMT>(keep_hits, count, occ_mode, rcp_guard, bands, cull);
        case kVariantBary: return instance_by_records<kVariantBary>(keep_hits, count, occ_mode, rcp_guard, bands, cull);
        case kVariantMTRel: // the counting kernels walk the plain records
            return count ? instance_by_records<kVariantMT>(keep_hits, count, occ_mode, rcp_guard, bands, cull)
                         : instance_by_records<kVariantMTRel>(keep_hits, count, occ_mode, rcp_guard, bands, cull);
        case kVariantMTAlt: return instance_by_records<kVariantMTAlt>(keep_hits, count, occ_mode, rcp_guard, bands, cull);
        case kVariantBaryAlt: return instance_by_records<kVariantBaryAlt>(keep_hits, count, occ_mode, rcp_guard, bands, cull);
        case kVariantFromHits: return instance_by_records<kVariantFromHits>(keep_hits, count, occ_mode, rcp_guard, bands, cull);
        default: return nullptr;
    }
}

size_t trace_tiles_smem_bytes(uint32_t spp, uint32_t occ_smem_words)
{
    return sizeof(float2) * spp + sizeof(uint32_t) * occ_smem_words;
}

void launch_trace_tiles(TraceTilesKernel k, const TraceParams& p, int grid_blocks, int threads, cudaStream_t stream)
{
    const size_t smem = trace_tiles_smem_bytes(p.spp, p.occ_smem_words);
    opt_in_smem(k, smem);
    k<<<grid_blocks, threads, smem, stream>>>(p);
}

int trace_tiles_max_blocks_per_sm(TraceTilesKernel k, int threads, size_t smem_bytes)
{
    int n = 0;
    opt_in_smem(k, smem_bytes);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, k, threads, smem_bytes);
    return n;
}

void launch_intersect_rays(const RayBatchParams& p, uint32_t variant, cudaStream_t stream)
{
    const uint32_t blocks = (p.n + 127) / 128;
    if (blocks == 0)
        return;
    if (variant)
        intersect_rays_kernel<1, true><<<blocks, 128, 0, stream>>>(p);
    else
        intersect_rays_kernel<0, true><<<blocks, 128, 0, stream>>>(p);
}

void launch_brute_force(const float *vtx, const uint32_t *tri, uint32_t num_tri, const RayBatchParams& p, cudaStream_t stream)
{
    if (p.n)
        brute_force_kernel<<<(p.n + 127) / 128, 128, 0, stream>>>(vtx, tri, num_tri, p);
}

void launch_ray_march(const float *vtx, const uint32_t *tri, uint32_t num_tri, uint32_t n, const float *origins,
                      const float *dirs, uint32_t *hit, float *t, cudaStream_t stream)
{
    if (n)
        ray_march_kernel<<<(n + 127) / 128, 128, 0, stream>>>(vtx, tri, num_tri, n, origins, dirs, hit, t);
}

void launch_sample_table(float2 *smp, uint32_t spp, cudaStream_t stream)
{
    sample_table_kernel<<<(spp + 127) / 128, 128, 0, stream>>>(smp, spp);
}

} // namespace rtm
