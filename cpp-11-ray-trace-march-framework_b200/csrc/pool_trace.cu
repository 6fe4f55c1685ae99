// K7 trace_pool: the traversal of K1 for INCOHERENT rays -- grids too large for a shared-memory occupancy map
// (the 50 M-triangle soup at 512^3), where the 32 rays of a warp part ways after a few cells.
//
// K1 keeps a warp's 32 rays in lock step between its two phases: lanes that have reached an occupied cell wait
// for the last walker (measured on the soup: 10.9 of 32 lanes walking, 18 of 32 threads per instruction overall).
// Here a warp owns a POOL of 96 rays in shared memory and picks, round by round, rays that all need the same kind of
// work -- the active lanes are compacted by ballot / population count across the divergent DDA walks:
//
//   test    32 rays standing on occupied cells test their cells' pair records (test_pair_list of K1, unchanged)
//           -> hit, or back to walking
//   refill  32 new rays (the next round of the warp's current strip): ray generation, grid entry, DDA set-up
//   walk    up to 64 rays standing in empty space, two per lane, step through the distance map (warp_trace.cuh,
//           kOccGlobalDist), one cell per ray and iteration, until they reach an occupied cell (-> test), leave the
//           grid (-> miss) or the round's step budget is used up
// in this order of preference: by the time a warp walks it holds more than 32 walkers, so most lanes carry two and one
// ray's look-up is in flight while the other one steps.
//
// Per-ray arithmetic is exactly K1's (same functions / the same included set-up), so every ray visits the same
// cells and tests the same triangles in the same order: results are bit-identical.  Finished rays leave only their
// hit record (triangle, t, u, v per sample); K1 instantiated with kVariantFromHits then shades, sums the samples
// in order, resolves and publishes the row bands exactly as for its own hits.
//
// Compiled with -fmad=false (see rt_device.cuh).
#include "trace_kernels.cuh"
#include "warp_trace.cuh"

namespace rtm
{

namespace
{

constexpr unsigned kFull = 0xFFFFFFFFu;
constexpr uint32_t kSlotFree = 0, kSlotWalk = 1, kSlotTest = 2;
constexpr uint32_t kOwn = kPoolSlots / 32; // slots whose status a lane keeps track of: lane, lane + 32, ...
constexpr uint32_t kMetaStepsMask = 0xFFu, kMetaNegX = 0x100u, kMetaNegY = 0x200u, kMetaNegZ = 0x400u;

// One warp's pool, structure of arrays over the slots
struct PoolWarp
{
    float n[3][kPoolSlots];   // next crossing per axis (grid.cpp:199-214)
    float dl[3][kPoolSlots];  // increment per cell
    float d[3][kPoolSlots];   // ray direction
    int pc[kPoolSlots];       // padded cell index
    uint32_t meta[kPoolSlots]; // bits 0-7: steps up to and including the next cell to look at (0: standing on a cell
                               // not looked at yet); bits 8-10: the x / y / z stride is negative
    uint32_t ray[kPoolSlots]; // index of the sample's hit record: (py * width + px) * spp + s
    uint32_t status[kPoolSlots];
    uint32_t list[64];        // the slots picked for this round, compacted (walk rounds take up to 64, two per lane)
};
static_assert(sizeof(PoolWarp) == kPoolWarpBytes, "trace_kernels.cuh: kPoolWarpBytes");

// Compaction: the owners of the slots whose bit is set in mask[] write the slot numbers, in order, to list[0 .. 64)
__device__ __forceinline__ void pick_slots(PoolWarp& pw, uint32_t lane, const unsigned mask[kOwn])
{
    const unsigned lt = (1u << lane) - 1u;
    uint32_t before = 0;
#pragma unroll
    for (uint32_t j = 0; j < kOwn; j++)
    {
        const uint32_t r = before + __popc(mask[j] & lt);
        if (((mask[j] >> lane) & 1u) && r < 64u)
            pw.list[r] = lane + 32u * j;
        before += __popc(mask[j]);
    }
    __syncwarp();
}

__device__ __forceinline__ void store_miss(const TraceParams& p, uint32_t k)
{
    p.hit_tri[k] = 0xFFFFFFFFu;
    p.hit_t[k] = 0.0f;
    p.hit_u[k] = 0.0f;
    p.hit_v[k] = 0.0f;
}

// One ray of a walk round in registers
struct Walker
{
    float n0, n1, n2, dl0, dl1, dl2;
    int pc, c0, c1, c2;
    uint32_t steps; // DDA steps up to and including the next cell to look at; 0: arrived (or no ray)
    uint32_t meta, slot;
    bool mine;
};

// all 32 lanes together (the x stride goes through a shuffle, the others through an opaque move: held in registers
// instead of being re-derived from the sign bits in every step, like in K1)
__device__ __forceinline__ void walker_load(const PoolWarp& pw, uint32_t slot, bool mine, uint32_t lane, int stride_y, int stride_z,
                                            const uint8_t *__restrict__ dist, Walker& w)
{
    w.slot = slot;
    w.mine = mine;
    w.n0 = pw.n[0][slot]; w.n1 = pw.n[1][slot]; w.n2 = pw.n[2][slot];
    w.dl0 = pw.dl[0][slot]; w.dl1 = pw.dl[1][slot]; w.dl2 = pw.dl[2][slot];
    w.pc = pw.pc[slot];
    w.meta = pw.meta[slot];
    w.c0 = __shfl_sync(kFull, (w.meta & kMetaNegX) ? -1 : 1, (int) lane);
    w.c1 = (w.meta & kMetaNegY) ? -stride_y : stride_y;
    w.c2 = (w.meta & kMetaNegZ) ? -stride_z : stride_z;
    asm volatile("" : "+r"(w.c1), "+r"(w.c2));
    w.steps = mine ? (w.meta & kMetaStepsMask) : 0u;
    if (mine && w.steps == 0) // standing on a cell not looked at yet
        w.steps = cell_distance(dist, w.pc);
}

// one DDA step of a ray that still has steps to go; after the last blind one, look at the cell reached (0 = occupied
// or padding: arrived).  (The same step with every instruction predicated on steps != 0 instead of the branch -- 48
// instead of 52 instructions per iteration of two rays -- and L1 prefetches of the pair records ahead of the test
// rounds were measured: 71.1 against 70.4 ms on the soup at 768^3.  Not kept.)
__device__ __forceinline__ void walker_step(Walker& w, const uint8_t *__restrict__ dist)
{
    if (w.steps != 0)
    {
        dda_step(w.n0, w.n1, w.n2, w.dl0, w.dl1, w.dl2, w.pc, w.c0, w.c1, w.c2);
        if (--w.steps == 0)
            w.steps = cell_distance(dist, w.pc);
    }
}

__device__ __forceinline__ void walker_store(const TraceParams& p, PoolWarp& pw, const uint32_t *__restrict__ pstart, const Walker& w)
{
    if (!w.mine)
        return;
    uint32_t status = kSlotWalk;
    if (w.steps == 0)
    {
        // an occupied cell, or the padding: the ray has left the grid (grid.cpp:275-276)
        if (__ldg(&pstart[w.pc]) == __ldg(&pstart[w.pc + 1]))
        {
            store_miss(p, pw.ray[w.slot]);
            status = kSlotFree;
        }
        else
            status = kSlotTest;
    }
    pw.n[0][w.slot] = w.n0; pw.n[1][w.slot] = w.n1; pw.n[2][w.slot] = w.n2;
    pw.pc[w.slot] = w.pc;
    pw.meta[w.slot] = (w.meta & ~kMetaStepsMask) | w.steps;
    pw.status[w.slot] = status;
}

template <bool RCP_GUARD>
__global__ void __launch_bounds__(kTraceMaxThreads) trace_pool_kernel(const __grid_constant__ TraceParams p)
{
    // shared memory: [sample table, spp x float2, padded to 16 bytes] [one PoolWarp per warp]
    extern __shared__ float2 s_mem[];
    float2 *s_smp = s_mem;
    PoolWarp *pools = reinterpret_cast<PoolWarp *>(s_mem + ((p.spp + 1u) & ~1u));
    for (uint32_t i = threadIdx.x; i < p.spp; i += blockDim.x)
        s_smp[i] = p.smp[i];
    __syncthreads();

    const uint32_t lane = threadIdx.x & 31u;
    PoolWarp& pw = pools[threadIdx.x >> 5];
    for (uint32_t j = 0; j < kOwn; j++)
        pw.status[lane + 32u * j] = kSlotFree;
    __syncwarp();

    PackedUnits pku;
    pku.one = p.pk_one;
    pku.minus_one = p.pk_minus_one;
    const GridDev& g = p.grid;
    const bool fast_math = p.cam.fast_math != 0;
    const int stride_y = ((int) g.dim[0] + 2) * ((int) g.dim[2] + 2), stride_z = (int) g.dim[0] + 2;
    const uint32_t *__restrict__ pstart = g.ppair_start;
    const uint8_t *__restrict__ dist = g.pcell_dist;
    const float4 *__restrict__ recs = g.pair_recs;
    const float3 o = make_float3(p.cam.origin[0], p.cam.origin[1], p.cam.origin[2]); // primary rays share their origin

    // the warp's current strip (warp-uniform): pixel slots [pbase, slots) are still to be handed out
    const uint32_t slots = p.strip_w * p.strip_h, ppr = 32u / p.spp;
    const uint32_t pl = lane / p.spp, s = lane - pl * p.spp;
    uint32_t pbase = slots, bx0 = 0, by0 = 0, bw = 0, bh = 0;
    bool more = true;

    for (;;)
    {
        unsigned walkers[kOwn], testers[kOwn], vacant[kOwn];
        uint32_t n_walk = 0, n_test = 0;
#pragma unroll
        for (uint32_t j = 0; j < kOwn; j++)
        {
            const uint32_t st = pw.status[lane + 32u * j];
            walkers[j] = __ballot_sync(kFull, st == kSlotWalk);
            testers[j] = __ballot_sync(kFull, st == kSlotTest);
            vacant[j] = ~(walkers[j] | testers[j]);
            n_walk += __popc(walkers[j]);
            n_test += __popc(testers[j]);
        }
        const uint32_t n_free = (uint32_t) kPoolSlots - n_walk - n_test;
        // What the lanes can do together: a full round of tests; else take in 32 new rays; else walk -- by then more
        // than 32 rays stand in empty space, enough for two per lane (one's look-up is in flight while the other
        // steps); else (the pool is draining) whichever kind there is more of
        enum { kRefill, kWalk, kTest } action;
        if (n_test >= 32u) action = kTest;
        else if (more && n_free >= 32u) action = kRefill;
        else if (n_walk >= 32u) action = kWalk;
        else if (n_walk + n_test == 0u) break;
        else action = n_test >= n_walk ? kTest : kWalk;

        if (action == kRefill)
        {
            if (pbase >= slots)
            {
                // next strip of this shard: the scheduler and the strip -> pixel mapping of K1 (trace_kernels.cu)
                uint32_t visit = 0;
                bool cancel_seen = false;
                if (lane == 0)
                {
                    cancel_seen = *(volatile const uint32_t *) p.cancel == p.frame_seq;
                    visit = atomicAdd(p.strip_counter + kPoolCounterWord, 1u);
                    if (cancel_seen)
                        *(volatile uint32_t *) p.cancel_seen = p.frame_seq;
                }
                visit = __shfl_sync(kFull, visit, 0);
                if (__any_sync(kFull, cancel_seen) || visit >= p.shard_strips)
                {
                    more = false; // a cancelled frame drains what is in flight and stops
                    continue;
                }
                const uint32_t my_chunk = visit / p.shard_chunk, in_chunk = visit - my_chunk * p.shard_chunk;
                const uint64_t chunk_id = (uint64_t) my_chunk * p.shard_world +
                                          (p.shard_rank + p.shard_world - my_chunk % p.shard_world) % p.shard_world;
                const uint64_t strip64 = chunk_id * p.shard_chunk + in_chunk;
                if (strip64 >= p.total_strips)
                    continue;
                const uint32_t strip = (uint32_t) strip64;
                uint32_t lo = 0, hi = p.n_tiles;
                while (hi - lo > 1)
                {
                    const uint32_t mid = (lo + hi) >> 1;
                    if (__ldg(&p.tile_strip_prefix[mid]) <= strip) lo = mid; else hi = mid;
                }
                const uint4 rect = __ldg(&p.tile_rects[lo]);
                const uint32_t local = strip - __ldg(&p.tile_strip_prefix[lo]);
                const uint32_t strips_x = (rect.z - rect.x + p.strip_w - 1) / p.strip_w;
                bx0 = rect.x + (local % strips_x) * p.strip_w;
                by0 = rect.y + (local / strips_x) * p.strip_h;
                bw = min(p.strip_w, rect.z - bx0);
                bh = min(p.strip_h, rect.w - by0);
                pbase = 0;
            }
            // one round of the strip: 32 / spp pixels in 2x2-quad order, lane = (pixel in round) * spp + sample
            const uint32_t slot = pbase + pl;
            pbase += ppr;
            const uint32_t ox = (slot & 1u) | ((slot >> 1) & 2u) | ((slot >> 2) & 4u);
            const uint32_t oy = ((slot >> 1) & 1u) | ((slot >> 2) & 2u);
            const bool valid = pl < ppr && slot < slots && ox < bw && oy < bh;
            if (!__any_sync(kFull, valid))
                continue;
            const uint32_t px = bx0 + ox, py = by0 + oy;
            const float2 off = s_smp[valid ? s : 0];
            float3 d, o_ray;
            generate_ray<false>(p.cam, px, py, off.x, off.y, o_ray, d);
            const uint32_t k = (py * p.width + px) * p.spp + s; // (< 2^32: checked by the launcher)
            bool active;
            float enter_t, n0, n1, n2, dl0, dl1, dl2;
            int c0, c1, c2, pc;
#include "dda_setup.inc"
            if (valid && !active)
                store_miss(p, k); // the ray misses the grid's box (grid.cpp:182-184)
            // the i-th ray of this round takes the i-th free slot
            pick_slots(pw, lane, vacant);
            const unsigned need = __ballot_sync(kFull, active);
            if (active)
            {
                const uint32_t slot_id = pw.list[__popc(need & ((1u << lane) - 1u))];
                pw.n[0][slot_id] = n0; pw.n[1][slot_id] = n1; pw.n[2][slot_id] = n2;
                pw.dl[0][slot_id] = dl0; pw.dl[1][slot_id] = dl1; pw.dl[2][slot_id] = dl2;
                pw.d[0][slot_id] = d.x; pw.d[1][slot_id] = d.y; pw.d[2][slot_id] = d.z;
                pw.pc[slot_id] = pc;
                pw.meta[slot_id] = (c0 < 0 ? kMetaNegX : 0u) | (c1 < 0 ? kMetaNegY : 0u) | (c2 < 0 ? kMetaNegZ : 0u);
                pw.ray[slot_id] = k;
                pw.status[slot_id] = kSlotWalk;
            }
            __syncwarp();
        }
        else if (action == kWalk)
        {
            // Phase A of K1 on the distance map (warp_trace.cuh): v = distance of the cell the ray stands on -> the
            // next v - 1 steps need no look-up; every step still does its own next_t += delta.  One step per ray and
            // iteration, so that no lane waits for another one's run of blind steps; TWO rays per lane where the
            // pool has them, so that one ray's look-up is in flight while the other one steps.  A ray that has
            // arrived idles until the round's budget is used up or every ray has arrived
            pick_slots(pw, lane, walkers);
            const uint32_t n_round = min(n_walk, 64u);
            Walker wa, wb;
            walker_load(pw, pw.list[lane < n_round ? lane : 0u], lane < n_round, lane, stride_y, stride_z, dist, wa);
            walker_load(pw, pw.list[lane + 32u < n_round ? lane + 32u : 0u], lane + 32u < n_round, lane, stride_y, stride_z, dist, wb);
#pragma unroll 1
            for (uint32_t it = 0; it < p.pool_walk_steps; it++)
            {
                if (!__any_sync(kFull, (wa.steps | wb.steps) != 0))
                    break;
                walker_step(wa, dist);
                walker_step(wb, dist);
            }
            walker_store(p, pw, pstart, wa);
            walker_store(p, pw, pstart, wb);
            __syncwarp();
        }
        else
        {
            pick_slots(pw, lane, testers);
            const bool mine = lane < min(n_test, 32u);
            const uint32_t slot_id = pw.list[mine ? lane : 0u];
            const float3 d = make_float3(pw.d[0][slot_id], pw.d[1][slot_id], pw.d[2][slot_id]);
            const float n0 = pw.n[0][slot_id], n1 = pw.n[1][slot_id], n2 = pw.n[2][slot_id];
            const int pc = pw.pc[slot_id];
            const uint32_t beg = mine ? __ldg(&pstart[pc]) : 0u, len = mine ? __ldg(&pstart[pc + 1]) - beg : 0u;
            const uint32_t max_len = __reduce_max_sync(kFull, len);
            // next_crossing_t[step_axis] (grid.cpp:236-239,260) -- the step axis rule of dda_step
            const bool a2 = (n2 <= n0) && (n2 <= n1);
            const bool a1 = !a2 && (n1 <= n0);
            float bound = a2 ? n2 : (a1 ? n1 : n0);
            float best_t = FLT_MAX;
            Hit hit;
            hit.t = hit.u = hit.v = 0.0f;
            hit.tri = 0xFFFFFFFFu;
            test_pair_list<false, RCP_GUARD>(recs, beg, len, len ? len - 1u : 0u, max_len, o, d, pku, bound, best_t, hit);
            if (mine)
            {
                if (best_t != FLT_MAX) // grid.cpp:270-271: the walk ends at the first cell with a hit
                {
                    const uint32_t k = pw.ray[slot_id];
                    p.hit_tri[k] = hit.tri;
                    p.hit_t[k] = hit.t;
                    p.hit_u[k] = hit.u;
                    p.hit_v[k] = hit.v;
                    pw.status[slot_id] = kSlotFree;
                }
                else
                {
                    pw.meta[slot_id] = (pw.meta[slot_id] & ~kMetaStepsMask) | 1u; // step, then look
                    pw.status[slot_id] = kSlotWalk;
                }
            }
            __syncwarp();
        }
    }
}

} // namespace

size_t trace_pool_smem_bytes(uint32_t spp, int threads)
{
    return sizeof(float2) * ((spp + 1u) & ~1u) + (size_t) kPoolWarpBytes * (threads / 32);
}

void launch_trace_pool(const TraceParams& p, int grid_blocks, int threads, cudaStream_t stream)
{
    const size_t smem = trace_pool_smem_bytes(p.spp, threads);
    static size_t opted_in[64][2] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    const int gi = p.rcp_guard ? 1 : 0;
    if (dev < 0 || dev >= 64 || opted_in[dev][gi] < smem)
    {
        if (gi)
            cudaFuncSetAttribute(trace_pool_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
        else
            cudaFuncSetAttribute(trace_pool_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
        if (dev >= 0 && dev < 64)
            opted_in[dev][gi] = smem;
    }
    if (gi)
        trace_pool_kernel<true><<<grid_blocks, threads, smem, stream>>>(p);
    else
        trace_pool_kernel<false><<<grid_blocks, threads, smem, stream>>>(p);
}

} // namespace rtm
