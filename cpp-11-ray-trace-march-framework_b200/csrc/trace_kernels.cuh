// Kernel launch interface between api.cu and the .cu files holding the kernels.
#pragma once

#include "rt_device.cuh"

namespace rtm
{

// A strip -- the unit of the dynamic scheduler -- is a strip_w x strip_h pixel block of a tile,
// one of 2x1, 2x2, 4x2, 4x4, 8x4 (its pixel slots are visited in 2x2-quad Morton order).  The
// host picks the size so that a strip carries about 128 rays (32 for frames below 16 M rays):
// small enough that the most expensive strip is a short tail -- measured +8 % (killeroo 4K) to
// +36 % (1080p, 4 spp) over 8x4 strips -- large enough that the atomic per strip is noise.
inline void strip_size_for_spp(uint32_t spp, uint64_t frame_rays, uint32_t& w, uint32_t& h)
{
    const uint64_t target = frame_rays >= (16ull << 20) ? 128 : 32;
    uint32_t pixels = 32;
    while (pixels > 2 && (uint64_t) pixels * spp > target)
        pixels /= 2;
    w = pixels >= 32 ? 8 : (pixels >= 8 ? 4 : 2);
    h = pixels >= 16 ? 4 : (pixels >= 4 ? 2 : 1);
}
// A strip the previous frame found expensive is handed out in `parts` pieces (whole rounds of 32 rays, whole
// pixels) so that no single warp holds the end of the frame: 4, 2 or 1 pieces (schedule.cu)
inline uint32_t strip_split_parts(uint32_t strip_w, uint32_t strip_h, uint32_t spp)
{
    const uint32_t slots = strip_w * strip_h, ppr = spp <= 32 ? 32u / spp : 1u; // pixels per round
    return slots % (4 * ppr) == 0 ? 4u : (slots % (2 * ppr) == 0 ? 2u : 1u);
}
constexpr uint32_t kVisitStripMask = 0x0FFFFFFFu; // visit entry = strip in shard | (part + 1) << 28, 0 in the top bits = whole strip
constexpr int kMaxBands = 32;          // row bands of the overlapped framebuffer read-back (api.cu)
constexpr int kTraceMaxThreads = 1024; // launch bound (caps the kernel at 64 registers); actual CTA size is chosen per launch

// Where the padded occupancy map lives (chosen per scene / frame by the launcher):
//   0  bits in global memory, read through L1            (any grid size)
//   1  bits staged in shared memory                      (<= ~1.6 M padded cells)
//   2  one BYTE per cell in shared memory                (<= ~220 K padded cells, i.e. the res-64
//      grids of configs C2-C4): the test is a single LDS.U8 without shift / mask arithmetic
//   3  distance map in global memory, read through L1   (grids too large for 1 / 2): one byte per cell holding the
//      city-block distance to the nearest occupied cell -- a ray steps that many cells between look-ups
// (The distance map staged in shared memory, one byte per cell on the LDS.U8 of mode 2, was measured on the res-64
// grids: 17.2 against 10.4 ms on killeroo 4K/16 -- lanes wait for each other's runs of blind steps.  Not kept.)
// (The DDA step on packed fp32 -- (next crossing, partial cell index as an exact float) pairs advanced by one
// predicated FADD2 per axis instead of FADD + IADD, 7 instead of 10 instructions on paper -- was written for mode 2:
// ptxas 12.9 does not predicate FADD2, it computes all three sums and selects, 19 instructions per step.  Not kept.)
enum { kOccGlobalBits = 0, kOccSmemBits = 1, kOccSmemBytes = 2, kOccGlobalDist = 3 };

// Kernel-side intersection variants: 0 / 1 are the ABI's (Moeller-Trumbore, plane + barycentric); 2 is
// Moeller-Trumbore on origin-relative records (GridDev::pair_recs_rel) -- the launcher's choice for primary rays
// 3 / 4 are 0 / 1 with the reference's alternates compiled in (orthographic camera, face-normal and depth shading:
// CameraDev::ortho, TraceParams::shade_mode) -- separate instantiations so that the live path does not carry them
// 5 does not traverse at all: the hit records were written by K7 trace_pool (pool_trace.cu); K1 shades, sums, resolves
enum { kVariantMT = 0, kVariantBary = 1, kVariantMTRel = 2, kVariantMTAlt = 3, kVariantBaryAlt = 4, kVariantFromHits = 5 };

// K7 trace_pool (pool_trace.cu): rays per warp pool, bytes of one warp's pool in shared memory, and the word of the
// strip-counter line its scheduler counts in (word 0 is K1's, which runs behind it on the same stream)
constexpr int kPoolSlots = 96;
constexpr int kPoolWarpBytes = (9 + 4) * kPoolSlots * 4 + 64 * 4;
constexpr int kPoolCounterWord = 16;

struct TraceParams
{
    GridDev grid;
    CameraDev cam;
    uint32_t width, height, spp;
    uint32_t gamma;
    uint32_t shade_mode;               // 0 interpolated vertex normal (live), 1 face normal, 2 depth (rt_device.cuh)
    const float2 *smp;                 // sample table, spp entries (K2)
    uint32_t occ_mode;                 // kOccGlobalBits / kOccSmemBits / kOccSmemBytes / kOccGlobalDist (warp_trace.cuh)
    uint32_t occ_smem_words;           // 32-bit words of the occupancy map staged in shared memory
    uint32_t rcp_guard;                // 1: the scene extent allows |det| > 1e30, keep rcp_exact's range check
    const uint4 *tile_rects;           // n_tiles x {x0,y0,x1,y1}
    const uint32_t *tile_strip_prefix; // n_tiles + 1: first strip id of each tile
    uint32_t n_tiles;
    uint32_t strip_w, strip_h;         // see strip_size_for_spp
    uint32_t shard_strips;             // strips this launch may fetch (upper bound; out-of-range ids are skipped)
    uint32_t total_strips;
    uint32_t shard_rank, shard_world;  // this launch renders the strips of shard `rank` out of `world`
    uint32_t shard_chunk;              // consecutive strips per deal (see trace_tiles_kernel)
    const uint32_t *fetch_order;       // cost-ordered visit list of this shard (schedule.cu) or null = strips in image order
    const uint32_t *visit_total;       // device word: entries in fetch_order
    uint32_t split_parts;              // pieces an expensive strip is visited in (strip_split_parts); band counters count pieces
    uint32_t pool_walk_steps;          // K7: DDA steps per ray in one walk round
    uint32_t *visit_cycles;            // out: cycles spent per visit (feeds the next frame's order, schedule.cu) or null
    uint32_t *strip_counter;           // dynamic strip scheduler (zeroed before launch)
    const uint32_t *cancel;            // == frame_seq => stop tracing (the word names the frame to cancel, api.cu)
    uint32_t frame_seq;
    uint32_t *cancel_seen;             // host-mapped word: a warp that saw the request stores frame_seq there
    uint32_t *framebuffer;             // width * height, row 0 = y 0 (may be a peer / IPC pointer)
    uint32_t *band_done;               // per row band: GPUs whose share of the band is finished (monotone across frames;
                                       // lives behind the framebuffer, so peers / other ranks reach it through the
                                       // same mapping) or null
    uint32_t *band_local;              // per row band: pieces of strips THIS GPU has finished in this frame (local memory)
    uint32_t band_share[kMaxBands];    // ... and how many that makes when its share of the band is complete
    uint32_t band_rows;                // rows per band
    uint32_t band_flush_units;         // a warp publishes its finished pieces once it holds this many
    uint32_t *hit_tri;                 // optional per-sample records (KEEP_HITS)
    float *hit_t, *hit_u, *hit_v;
    Counters *counters;                // optional (COUNT)
    // (1.0f, 1.0f) and (-1.0f, -1.0f) as register pairs: the multiplier of the packed sums and differences in
    // warp_trace.cuh.  Passed as data so that ptxas cannot fold them into a contracted FFMA2.
    unsigned long long pk_one, pk_minus_one;
    const float4 *pair_sbox;           // kVariantMTRel: screen box of every pair record for this camera (pack.cu) or
                                       // null = no screen cull
};

struct RayBatchParams
{
    GridDev grid;
    uint32_t n;
    const float *origins, *dirs;
    uint32_t *tri;
    float *t, *u, *v;
    unsigned long long *mailbox_stats; // mailbox mode: [0] tests asked for, [1] answered from the mailbox (or null)
};

// cuda_trace_query_rays (ray_query.cu): every pointer is device memory; tri / occluded by kind, t / u / v optional
struct RayQueryParams
{
    GridDev grid;
    uint64_t n;
    const float *origins, *dirs; // n x 3
    const float *t_max;          // n, or null: t_max_all for every ray
    float t_max_all;
    uint32_t *tri;               // closest hit
    float *t, *u, *v;
    uint8_t *occluded;           // occlusion
    uint32_t occ_mode;           // as TraceParams
    uint32_t occ_smem_words;
    uint32_t fast_math;          // the range-check-free DDA set-up may be used (rays with |dir| <= 1, voted per warp)
    unsigned long long pk_one, pk_minus_one;
};

// K1 (trace_kernels.cu): the kernel instance for a frame's intersection variant, per-sample hit records (KEEP_HITS),
// work counters (COUNT), occupancy map home, rcp range guard (TraceParams::rcp_guard), band publication
// (TraceParams::band_done set) and screen cull (TraceParams::pair_sbox set).  Only the plain kernel exists without the
// guard or without band publication (the others test rcp_guard and band_done at run time); the work counters exist for
// variants 0 and 1 (2 counts as 0), the cull for variant 2.  Null for an unknown variant.
using TraceTilesKernel = void (*)(TraceParams);
TraceTilesKernel trace_tiles_instance(uint32_t variant, bool keep_hits, bool count, int occ_mode, bool rcp_guard, bool bands,
                                      bool cull);
void launch_trace_tiles(TraceTilesKernel k, const TraceParams& p, int grid_blocks, int threads, cudaStream_t stream);
int trace_tiles_max_blocks_per_sm(TraceTilesKernel k, int threads, size_t smem_bytes);
size_t trace_tiles_smem_bytes(uint32_t spp, uint32_t occ_smem_words);
// K7: traverses the strips of this launch's shard with pooled rays and leaves (tri, t, u, v) per sample in p.hit_*
// (all four required); follow it with K1 in variant kVariantFromHits on the same stream
void launch_trace_pool(const TraceParams& p, int grid_blocks, int threads, cudaStream_t stream);
size_t trace_pool_smem_bytes(uint32_t spp, int threads);
// the scalar one-thread-per-ray walk, kept for the mailboxing mode of cuda_trace_intersect_rays (the plain mode runs
// launch_ray_query)
void launch_intersect_rays(const RayBatchParams& p, uint32_t variant, cudaStream_t stream);
// bounded: the t_max rules apply (t_max given per ray or finite); occlusion queries always run bounded
void launch_ray_query(const RayQueryParams& p, uint32_t variant, bool occlusion, bool bounded, int grid_blocks,
                      cudaStream_t stream);
int ray_query_threads(); // CTA size of launch_ray_query
void launch_sample_table(float2 *smp, uint32_t spp, cudaStream_t stream);
void launch_ray_march(const float *vtx, const uint32_t *tri, uint32_t num_tri, uint32_t n, const float *origins,
                      const float *dirs, uint32_t *hit, float *t, cudaStream_t stream);
void launch_brute_force(const float *vtx, const uint32_t *tri, uint32_t num_tri, const RayBatchParams& p, cudaStream_t stream);

// cost-ordered scheduling (schedule.cu): 5 kernels; scratch = 2 * ceil(n / 1024) + 2 words; order holds up to
// strip_order_capacity(n, parts) visit entries, *visit_total how many were written.  visit_cycles = what K1
// recorded for this frame's visits (made through `order` when order_was_used, else strip by strip);
// strip_cycles[n] receives the per-strip sums.
void launch_build_strip_order(const uint32_t *visit_cycles, bool order_was_used, uint32_t *strip_cycles, uint32_t n,
                              uint32_t parts, unsigned long long *sum, uint32_t *scratch, uint32_t *visit_total,
                              uint32_t *order, cudaStream_t stream);
size_t strip_order_scratch_words(uint32_t n);
size_t strip_order_capacity(uint32_t n, uint32_t parts);

// scene packing (pack.cu)
void launch_pair_counts(const uint32_t *pcell_start, uint64_t pcells, uint32_t *counts, cudaStream_t stream); // counts[pcells + 1]
void launch_pack_pairs(const uint32_t *pcell_start, const uint32_t *ppair_start, uint64_t pcells, const float4 *cell_tris,
                       float4 *pair_recs, cudaStream_t stream);
void launch_origin_relative_pairs(const float4 *pair_recs, uint64_t num_pairs, const float origin[3], float4 *rel,
                                  cudaStream_t stream);
// screen box of every pair record for camera `cam` (pack.cu); *small_boxes (zeroed here) counts the pairs whose box is at
// most kScreenCullSmallPixels pixels on its longer side
void launch_screen_boxes(const float4 *pair_recs, uint64_t num_pairs, const CameraDev& cam, float4 *sbox,
                         unsigned int *small_boxes, cudaStream_t stream);
constexpr float kScreenCullSmallPixels = 32.0f;
void launch_pack_cell_tris(const float *vtx, const uint32_t *tri, const uint32_t *tri_index, uint64_t num_refs,
                           float4 *cell_tris, float4 *cell_tris_b, cudaStream_t stream);
void launch_pack_normals(const float *vtx, const uint32_t *tri, uint32_t num_tri, float4 *tri_normals,
                         cudaStream_t stream);
void launch_cell_occupancy(const uint32_t *cell_start, uint64_t num_cells, uint32_t *cell_occ, cudaStream_t stream);
void launch_pad_grid(const uint32_t *cell_start, const uint32_t dim[3], uint32_t *pcell_start, uint32_t *pcell_occ,
                     cudaStream_t stream); // 2 kernels
void launch_distance_map(const uint32_t *pcell_occ, const uint32_t dim[3], uint8_t *pcell_dist, cudaStream_t stream); // 3 kernels
void launch_narrow_offsets(const uint64_t *off64, uint64_t n, uint32_t *off32, cudaStream_t stream);
void launch_widen_offsets(const uint32_t *off32, uint64_t n, uint64_t *off64, cudaStream_t stream);

} // namespace rtm
