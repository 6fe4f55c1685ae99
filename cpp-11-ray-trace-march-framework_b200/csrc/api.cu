// C ABI of the tile tracer (include/cuda_trace.h): contexts, scene upload, frame launches.
//
// This is the "thin launch layer" that replaces the reference's worker-thread tile pool
// (framebuffer.cpp:16-92): a frame is one persistent-kernel launch per device instead of
// hardware_concurrency() threads popping tiles from a mutex-protected queue.
#include "../../include/cuda_trace.h"

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstdint>
#include <array>
#include <chrono>
#include <cstring>
#include <mutex>
#include <string>
#include <tuple>
#include <vector>

#include "device_array.cuh"
#include "grid_build.cuh"
#include "qmc.cuh"
#include "trace_kernels.cuh"

using namespace rtm;

namespace
{

std::string g_init_error;

// A scene's arrays on one device and what describes their contents; replaced whole, by a new scene or by nothing
struct SceneArrays
{
    DeviceArray<float> d_vtx;
    DeviceArray<uint32_t> d_tri, d_cell_start, d_cell_occ, d_tri_index;
    DeviceArray<uint32_t> d_pcell_start, d_pcell_occ; // padded grid (rt_device.cuh)
    DeviceArray<uint8_t> d_pcell_dist;                // its distance map (large grids only)
    DeviceArray<float4> d_cell_tris, d_cell_tris_b, d_tri_normals;
    DeviceArray<uint32_t> d_ppair_start; // padded CSR of the pair records (rt_device.cuh)
    DeviceArray<float4> d_pair_recs;     // two triangles per record, interleaved: the packed-fp32 test of K1
    DeviceArray<float4> d_pair_recs_rel; // ... relative to rel_origin (primary rays; built on demand, pack.cu)
    float rel_origin[3] = { 0.0f, 0.0f, 0.0f };
    bool rel_valid = false;
    // screen boxes of the pair records (K1's screen cull, pack.cu) for the camera sbox_cam, and the per-scene gate
    // taken from them: cull only when enough pairs project small (sbox_cull)
    DeviceArray<float4> d_pair_sbox;
    DeviceArray<unsigned int> d_sbox_small;
    CameraDev sbox_cam;
    uint32_t sbox_small = 0; // boxes of at most kScreenCullSmallPixels pixels for sbox_cam (the gate's count)
    bool sbox_valid = false, sbox_cull = false;
};

struct DeviceState
{
    int ordinal = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t side_stream = nullptr; // cancel flag writes while the main stream is busy
    cudaStream_t copy_stream = nullptr; // overlapped framebuffer read-back (device 0 only)
    // the next frame's visiting order is built behind the trace kernel on its own stream, so that waiting for the
    // frame (cuda_trace_sync) does not wait for it; the next frame's launch does (ev_order)
    cudaStream_t order_stream = nullptr;
    cudaEvent_t ev_traced = nullptr, ev_order = nullptr;
    bool order_pending = false;
    cudaEvent_t ev_copy = nullptr;
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;

    SceneArrays scene;
    // K7 trace_pool: per-sample hit records (tri, t, u, v) of this device's strips, read back by K1 <kVariantFromHits>
    DeviceArray<uint32_t> d_pool_tri;
    DeviceArray<float> d_pool_t, d_pool_u, d_pool_v;
    int resolve_blocks_per_sm = 0, resolve_threads = 0;

    // frame
    DeviceArray<float2> d_smp;
    uint32_t smp_valid_spp = 0;
    DeviceArray<uint4> d_tile_rects;
    DeviceArray<uint32_t> d_tile_prefix;
    DeviceArray<uint32_t> d_strip_counter; // {strip counter, pad to 128 B, this GPU's band piece counts}: one memset per frame
    uint32_t *d_cancel = nullptr;          // behind them and never cleared: the sequence number of the frame to cancel
    PinnedArray<uint32_t, cudaHostAllocMapped | cudaHostAllocPortable> h_cancel_seen; // the kernel stores its frame number here when it saw the request
    uint32_t *d_cancel_seen = nullptr;     // device view of h_cancel_seen
    uint32_t launched_seq = 0;             // sequence number of the frame in flight on this device
    uint64_t layout_serial = 0;            // FramePlan the device copies d_tile_rects / d_tile_prefix hold
    std::tuple<TraceTilesKernel, int, size_t> occupancy_key{}; // K1 instance, CTA size, dynamic smem `blocks_per_sm` is for
    int blocks_per_sm = 0;
    DeviceArray<Counters> d_counters;
    // cost-ordered scheduling (schedule.cu): cycles per strip of the last frame -> order of the next
    DeviceArray<uint32_t> d_strip_cycles, d_fetch_order, d_order_scratch, d_visit_total, d_visit_cycles;
    DeviceArray<unsigned long long> d_cost_sum;
    bool order_valid = false;
    std::vector<uint64_t> order_signature; // plan serial + shard the recorded strip costs belong to
    uint32_t order_strips = 0;             // strips of this shard the recorded costs cover
    bool frame_pending = false;
    bool order_followup = false, order_followup_used = false; // this frame recorded strip costs (through the previous order)
};

} // namespace

namespace
{

// Tuning switches, read ONCE in cuda_trace_init (experiments and tests; every default is the measured best)
struct Tuning
{
    int strip_pixels = 0;  // RTM_STRIP_PIXELS = 2 | 4 | 8 | 16 | 32 pixels per strip (0: by sample count)
    int split_parts = 0;   // RTM_SPLIT_PARTS = 1 | 2 pieces per expensive strip (0: by strip size)
    int occ_mode = -1;     // RTM_OCC_MODE = 0 | 1 | 2 | 3 home of the occupancy map (-1: by grid size)
    int pool = -1;         // RTM_POOL = 0 | 1 pooled-ray traversal K7 for the frames it supports (-1: grids with a distance map)
    int pool_steps = 24;   // RTM_POOL_STEPS = DDA steps per ray in one walk round of K7
    int threads = 0;       // RTM_THREADS = CTA size (0: by frame size)
    int band_flush = 0;    // RTM_BAND_FLUSH = 1..8 strips a warp holds before publishing (0: by frame size)
    int shard_chunk = 0;   // RTM_SHARD_CHUNK = strips per deal when sharding (0: 32)
};

// What a frame's tile list turns into.  Kept between calls: a viewer renders the same layout every frame.
struct FramePlan
{
    uint64_t serial = 0; // changes whenever the plan is rebuilt (devices compare serials, not tile lists)
    uint32_t width = 0, height = 0, spp = 0;
    std::vector<cuda_trace_tile_rect> tiles;
    uint32_t strip_w = 0, strip_h = 0, split_parts = 1;
    std::vector<uint4> rects;
    std::vector<uint32_t> prefix; // first strip id of each tile, + total
    uint64_t total = 0;           // strips
    bool covers_frame = false;    // the tiles partition the whole frame (no gap, no overlap)
};

} // namespace

struct cuda_trace_ctx
{
    std::vector<DeviceState> dev;
    std::string err;
    std::recursive_mutex api_mtx; // entry points that use the streams / the error slot are serialised (not cancel)
    Tuning tune;
    FramePlan plan;
    std::atomic<uint32_t> frame_seq{0}, cancel_seq{0}; // cancel names the frame it is meant for
    std::mutex seq_mtx;           // orders cuda_trace_cancel against the moment a frame gets its number
    bool setting_up = false;      // a tiles call is past its argument checks but has no number yet (seq_mtx)
    bool cancel_pending = false;  // ... and was cancelled in that window: its frame starts cancelled (seq_mtx)
    bool band_dirty = false;      // a launch failed half way: re-read the band counters before the next overlapped frame

    bool have_scene = false;
    cuda_trace_grid_desc desc;
    uint32_t num_vtx = 0, num_tri = 0;
    uint32_t num_pairs = 0; // pair records (two cell references each, rt_device.cuh)

    uint32_t shard_rank = 0, shard_world = 1;
    uint32_t shard_chunk = 32; // consecutive strips dealt to one shard at a time (one CTA's worth of warps)
    bool counting = false;
    bool qmc_ready = false; // prime table uploaded to constant memory (qmc.cu)
    bool occ_in_smem = true;
    bool rel_records = true;    // RTM_REL_RECORDS=0: always the plain records, 2: origin-relative at any frame size (experiments)
    bool rel_records_forced = false;
    int screen_cull = -1;       // RTM_SCREEN_CULL: -1 automatic (the per-scene gate), 0 off, 1 on wherever rel records are used
    bool fast_math = true;      // RTM_FAST_MATH=0: always the range-checked intrinsics (experiments)
    int cost_order_forced = -1; // schedule.cu: -1 automatic, 0 / 1 forced by RTM_COST_ORDER (experiments)
    std::atomic<uint64_t> launches{0};

    // framebuffer (device 0: fb_own, or an imported IPC mapping of another process' framebuffer)
    uint32_t *d_fb = nullptr;
    DeviceArray<uint32_t> fb_own;
    bool fb_imported = false;
    uint32_t fb_w = 0, fb_h = 0;

    // Overlapped read-back: the framebuffer allocation carries kMaxBands completion counters
    // behind the pixels (so IPC peers reach them through the same mapping).  K1 bumps a band's
    // counter once per GPU that has finished its share of the band; band_expected is the running total
    // rank 0 waits for.
    uint32_t band_rows = 1, n_bands = 1;
    uint32_t band_expected[kMaxBands] = {};
    std::vector<uint64_t> band_inc_sig;
    uint32_t band_inc[kMaxBands] = {};
    std::vector<std::array<uint32_t, kMaxBands>> band_share; // per participating GPU: its pieces of strips per band
    bool copy_pending = false;
    // cuda_trace_tiles_into: tiles grouped by the row band that completes them, one event per group
    std::vector<cudaEvent_t> tile_events;
    std::vector<std::vector<uint32_t>> tile_groups;
    PinnedArray<uint32_t, cudaHostAllocPortable> staging; // W x H image small frames pass through on their way into tile buffers
    bool overlap_d2h = true;      // RTM_OVERLAP_D2H=0 disables
    bool shard_signals = false;   // cuda_trace_set_shard_signals: other ranks bump the counters too
    int (*wait_value32)(cudaStream_t, unsigned long long, unsigned int, unsigned int) = nullptr;

    // per-sample hit records of the last KEEP_HITS frame (device 0)
    unsigned long long mailbox_stats[2] = { 0, 0 }; // last mailbox run of cuda_trace_intersect_rays
    DeviceArray<uint32_t> d_hit_tri;
    DeviceArray<float> d_hit_t, d_hit_u, d_hit_v;
    uint64_t hit_count = 0;

    // last frame
    cuda_trace_frame frame;
    std::vector<cuda_trace_tile_rect> tiles;
    bool frame_valid = false;
    float last_kernel_ms = 0.0f;
    // host-clock marks of the last cuda_trace_tiles call, ms since its entry (cuda_trace_last_call_timing)
    std::chrono::steady_clock::time_point t_enter;
    double t_submitted_ms = 0.0, t_traced_ms = 0.0, t_copied_ms = 0.0, t_return_ms = 0.0;
    double t_prepared_ms = 0.0, t_launching_ms = 0.0, t_launched_ms = 0.0; // submission in detail: host set-up done, first device's kernel about to be / has been launched
    bool marks_armed = false;
    PinnedArray<uint32_t> pinned_cancel_src;

    // cuda_trace_query_rays: per stream the context has been given, an event behind its last query (device 0).
    // Replacing the scene or destroying the context waits for them before the scene arrays are freed.
    std::vector<std::pair<cudaStream_t, cudaEvent_t>> query_events;

    // cuda_trace_upload_scene_device (device 0): the allocation-range look-up (driver API), an event the context's
    // stream waits on for the caller's stream, and the word the index check reports its first bad triangle in
    int (*mem_range)(unsigned long long *, size_t *, unsigned long long) = nullptr;
    cudaEvent_t ev_mesh_input = nullptr;
    DeviceArray<uint32_t> d_first_bad;
};

namespace
{

int fail(cuda_trace_ctx *ctx, int code, const std::string& msg)
{
    if (ctx)
        ctx->err = msg;
    else
        g_init_error = msg;
    return code;
}

#define CK(call)                                                                                 \
    do {                                                                                         \
        cudaError_t e_ = (call);                                                                 \
        if (e_ != cudaSuccess)                                                                   \
            return fail(ctx, CUDA_TRACE_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
    } while (0)

// Queries still running on their callers' streams read the scene arrays: wait for them before those are freed
void wait_for_queries(cuda_trace_ctx *ctx)
{
    if (ctx->dev.empty())
        return;
    cudaSetDevice(ctx->dev[0].ordinal);
    for (auto& se : ctx->query_events)
        cudaEventSynchronize(se.second);
}

GridDev grid_dev(const cuda_trace_ctx *ctx, const DeviceState& d)
{
    const SceneArrays& s = d.scene;
    GridDev g;
    for (int k = 0; k < 3; k++)
    {
        g.dim[k] = ctx->desc.dim[k];
        g.aabb_min[k] = ctx->desc.aabb_min[k];
        g.aabb_max[k] = ctx->desc.aabb_max[k];
    }
    g.cell_wdh = ctx->desc.cell_wdh;
    g.inv_cell_wdh = ctx->desc.inv_cell_wdh;
    g.cell_start = s.d_cell_start.get();
    g.cell_occ = s.d_cell_occ.get();
    g.pcell_start = s.d_pcell_start.get();
    g.pcell_occ = s.d_pcell_occ.get();
    g.pcell_dist = s.d_pcell_dist.get();
    g.cell_tris = s.d_cell_tris.get();
    g.cell_tris_b = s.d_cell_tris_b.get();
    g.ppair_start = s.d_ppair_start.get();
    g.pair_recs = s.d_pair_recs.get();
    g.pair_recs_rel = s.d_pair_recs_rel.get();
    g.tri_normals = s.d_tri_normals.get();
    g.tri = s.d_tri.get();
    return g;
}

// shared memory the staged occupancy map may take (next to the sample table) when the launcher chooses by itself
constexpr uint64_t kOccSmemBudget = 160 * 1024;
inline uint64_t occupancy_bits_bytes(uint64_t pcells) { return (pcells + 31) / 32 * 4; }

// After d_vtx / d_tri / d_cell_start / d_tri_index are in place on device d: derived layout
int finish_scene_on_device(cuda_trace_ctx *ctx, DeviceState& d)
{
    SceneArrays& s = d.scene;
    const uint64_t cells = ctx->desc.num_cells, refs = ctx->desc.num_refs;
    const uint64_t pcells = (uint64_t) (ctx->desc.dim[0] + 2) * (ctx->desc.dim[1] + 2) * (ctx->desc.dim[2] + 2);
    if (pcells >= (1ull << 31))
        return fail(ctx, CUDA_TRACE_ERR_ARG, "grid too large: padded cell count must stay below 2^31");
    if (refs * 3 >= (1ull << 32))
        return fail(ctx, CUDA_TRACE_ERR_ARG, "grid too large: 3 x cell references must stay below 2^32");
    CK(s.d_cell_occ.alloc((cells + 31) / 32));
    CK(s.d_pcell_start.alloc(pcells + 1));
    CK(s.d_pcell_occ.alloc((pcells + 31) / 32));
    CK(s.d_cell_tris.alloc(std::max<uint64_t>(refs, 1) * 3));
    CK(s.d_cell_tris_b.alloc(std::max<uint64_t>(refs, 1) * 2));
    CK(s.d_tri_normals.alloc((size_t) ctx->num_tri * 3));
    launch_cell_occupancy(s.d_cell_start.get(), cells, s.d_cell_occ.get(), d.stream);
    launch_pad_grid(s.d_cell_start.get(), ctx->desc.dim, s.d_pcell_start.get(), s.d_pcell_occ.get(), d.stream);
    ctx->launches += 2;
    // grids whose occupancy bits do not fit in shared memory (choose_cta) get the distance map as a second level
    if (occupancy_bits_bytes(pcells) > kOccSmemBudget || ctx->tune.occ_mode == kOccGlobalDist || ctx->tune.pool == 1)
    {
        CK(s.d_pcell_dist.alloc(pcells));
        launch_distance_map(s.d_pcell_occ.get(), ctx->desc.dim, s.d_pcell_dist.get(), d.stream);
        ctx->launches += 3;
    }
    launch_pack_cell_tris(s.d_vtx.get(), s.d_tri.get(), s.d_tri_index.get(), refs, s.d_cell_tris.get(), s.d_cell_tris_b.get(), d.stream);
    launch_pack_normals(s.d_vtx.get(), s.d_tri.get(), ctx->num_tri, s.d_tri_normals.get(), d.stream);
    ctx->launches += 2 + (refs ? 1 : 0);
    CK(cudaGetLastError());
    // pair records: count per padded cell -> exclusive scan -> pack
    CK(s.d_ppair_start.alloc(pcells + 1));
    launch_pair_counts(s.d_pcell_start.get(), pcells, s.d_ppair_start.get(), d.stream);
    ctx->launches++;
    {
        std::string err;
        uint64_t launches = 0;
        const int rc = exclusive_scan_u32(s.d_ppair_start.get(), s.d_ppair_start.get(), pcells + 1, d.stream, err, &launches);
        ctx->launches += launches;
        if (rc)
            return fail(ctx, rc, err);
    }
    uint32_t pairs = 0;
    CK(cudaMemcpyAsync(&pairs, s.d_ppair_start.get() + pcells, sizeof(uint32_t), cudaMemcpyDeviceToHost, d.stream));
    CK(cudaStreamSynchronize(d.stream));
    if ((uint64_t) pairs * 7 >= (1ull << 32))
        return fail(ctx, CUDA_TRACE_ERR_ARG, "grid too large: 7 x pair records must stay below 2^32");
    if (&d == &ctx->dev[0])
        ctx->num_pairs = pairs;
    else if (ctx->num_pairs != pairs)
        return fail(ctx, CUDA_TRACE_ERR_CUDA, "pair records differ between devices");
    CK(s.d_pair_recs.alloc(std::max<uint64_t>(pairs, 1) * 5));
    if (pairs)
    {
        launch_pack_pairs(s.d_pcell_start.get(), s.d_ppair_start.get(), pcells, s.d_cell_tris.get(), s.d_pair_recs.get(), d.stream);
        ctx->launches++;
    }
    else
        CK(cudaMemsetAsync(s.d_pair_recs.get(), 0, 5 * sizeof(float4), d.stream));
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(d.stream));
    return 0;
}

int upload_mesh(cuda_trace_ctx *ctx, DeviceState& d, const float *vertices, uint32_t num_vertices,
                const uint32_t *triangles, uint32_t num_triangles)
{
    CK(cudaSetDevice(d.ordinal));
    CK(d.scene.d_vtx.alloc((size_t) num_vertices * 6));
    CK(d.scene.d_tri.alloc((size_t) num_triangles * 6));
    CK(cudaMemcpyAsync(d.scene.d_vtx.get(), vertices, (size_t) num_vertices * 24, cudaMemcpyHostToDevice, d.stream));
    CK(cudaMemcpyAsync(d.scene.d_tri.get(), triangles, (size_t) num_triangles * 24, cudaMemcpyHostToDevice, d.stream));
    return 0;
}

int check_mesh_args(cuda_trace_ctx *ctx, const float *vertices, uint32_t num_vertices, const uint32_t *triangles,
                    uint32_t num_triangles)
{
    if (!ctx)
        return CUDA_TRACE_ERR_ARG;
    if (!vertices || !triangles || num_vertices == 0 || num_triangles == 0)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "upload_scene: empty mesh (the reference asserts, grid.cpp:15)");
    for (uint32_t i = 0; i < num_triangles; i++)
        for (int c = 0; c < 3; c++)
            if (triangles[(size_t) i * 6 + c] >= num_vertices)
                return fail(ctx, CUDA_TRACE_ERR_ARG, "upload_scene: vertex index out of bounds");
    return 0;
}

// The grid of the mesh staged on device d, the context's i-th.  Every device builds its own copy of the grid (the build
// is deterministic and cheaper than shipping the cell-major records over NVLink would be to code; ~ms)
int build_grid(cuda_trace_ctx *ctx, DeviceState& d, size_t i, uint32_t grid_res)
{
    GridBuildResult res;
    uint64_t launches = 0;
    std::string err;
    const int rc = build_grid_device(d.scene.d_vtx.get(), ctx->num_vtx, d.scene.d_tri.get(), ctx->num_tri, grid_res, d.stream, &res, err, &launches);
    ctx->launches += launches;
    if (rc)
        return fail(ctx, rc, err);
    d.scene.d_cell_start = std::move(res.d_cell_start);
    d.scene.d_tri_index = std::move(res.d_tri_index);
    if (i == 0)
        ctx->desc = res.desc;
    else if (std::memcmp(&ctx->desc, &res.desc, sizeof(res.desc)) != 0)
        return fail(ctx, CUDA_TRACE_ERR_CUDA, "grid build differs between devices");
    return 0;
}

// The per-device part of a scene upload, shared by the entry points: device by device, free the old scene, let
// `stage(d, i)` put the mesh into d.scene.d_vtx / d_tri and the grid into d_cell_start / d_tri_index (and ctx->desc),
// and derive the rest.  Devices are built in order and finish_scene_on_device ends in a synchronisation of the device's
// stream, so device 0's arrays are complete before device 1 stages.  An upload that fails leaves no scene.
template <class Stage>
int build_scene(cuda_trace_ctx *ctx, uint32_t num_vertices, uint32_t num_triangles, Stage stage)
{
    int rc = 0;
    ctx->have_scene = false;
    ctx->num_vtx = num_vertices;
    ctx->num_tri = num_triangles;
    for (size_t i = 0; i < ctx->dev.size(); i++)
    {
        DeviceState& d = ctx->dev[i];
        d.scene = SceneArrays();
        if ((rc = stage(d, i)) || (rc = finish_scene_on_device(ctx, d)))
        {
            for (DeviceState& e : ctx->dev) // released once the work enqueued on them is done
            {
                cudaStreamSynchronize(e.stream);
                e.scene = SceneArrays();
            }
            return rc;
        }
    }
    ctx->have_scene = true;
    return 0;
}

// cuda_trace_upload_scene_device's checks of one caller array (`count` 24-byte records), all on the host and before
// anything is enqueued: 4-byte aligned, device or managed memory of device 0, and inside one allocation
int check_device_array(cuda_trace_ctx *ctx, const void *p, uint32_t count, const char *name)
{
    const int dev0 = ctx->dev[0].ordinal;
    if ((uintptr_t) p & 3)
        return fail(ctx, CUDA_TRACE_ERR_ARG, std::string("upload_scene_device: ") + name + " is not 4-byte aligned");
    cudaPointerAttributes a;
    const cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess)
        cudaGetLastError(); // not sticky: clear it so that the next call does not report it
    if (e != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != dev0)
        return fail(ctx, CUDA_TRACE_ERR_ARG, std::string("upload_scene_device: ") + name +
                                                 " is not device memory of the context's device " + std::to_string(dev0));
    if (!ctx->mem_range)
        return fail(ctx, CUDA_TRACE_ERR_CUDA, "upload_scene_device: the driver has no cuMemGetAddressRange");
    unsigned long long base = 0;
    size_t size = 0;
    const int r = ctx->mem_range(&base, &size, (unsigned long long) (uintptr_t) p);
    if (r != 0)
        return fail(ctx, CUDA_TRACE_ERR_ARG, std::string("upload_scene_device: cuMemGetAddressRange found no "
                                                         "allocation for ") + name + " (error " + std::to_string(r) + ")");
    const uint64_t offset = (uint64_t) (uintptr_t) p - base, bytes = (uint64_t) count * 24;
    if (offset + bytes > size)
        return fail(ctx, CUDA_TRACE_ERR_ARG, std::string("upload_scene_device: ") + std::to_string(count) + " " + name +
                                                 " records (" + std::to_string(bytes) + " bytes) run past the end of "
                                                 "their allocation (" + std::to_string(size - offset) + " bytes left)");
    return 0;
}

size_t fb_pixel_bytes(uint32_t w, uint32_t h) { return ((size_t) w * h * sizeof(uint32_t) + 255) & ~(size_t) 255; }
size_t fb_alloc_bytes(uint32_t w, uint32_t h) { return fb_pixel_bytes(w, h) + kMaxBands * sizeof(uint32_t); }

int ensure_framebuffer(cuda_trace_ctx *ctx, uint32_t w, uint32_t h)
{
    if (ctx->d_fb && ctx->fb_w == w && ctx->fb_h == h)
        return 0;
    if (ctx->fb_imported)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "frame size differs from the imported framebuffer");
    CK(cudaSetDevice(ctx->dev[0].ordinal));
    ctx->d_fb = nullptr;
    CK(ctx->fb_own.alloc(fb_alloc_bytes(w, h) / sizeof(uint32_t)));
    ctx->d_fb = ctx->fb_own.get();
    CK(cudaMemsetAsync(ctx->d_fb, 0, fb_alloc_bytes(w, h), ctx->dev[0].stream));
    CK(cudaStreamSynchronize(ctx->dev[0].stream)); // the zeroed band counters are in place before any stream waits on them
    ctx->fb_w = w;
    ctx->fb_h = h;
    std::memset(ctx->band_expected, 0, sizeof(ctx->band_expected));
    return 0;
}

uint32_t *band_counters(cuda_trace_ctx *ctx)
{
    return reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(ctx->d_fb) + fb_pixel_bytes(ctx->fb_w, ctx->fb_h));
}

// Strips per row band for this frame layout (a strip that straddles a band boundary counts in
// both, exactly as the kernel bumps both)
double ms_since(std::chrono::steady_clock::time_point t0)
{
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

// Row bands of the overlapped read-back: ~1 MB of pixels per band (a DMA that size runs at full PCIe rate; the
// last band's copy is the exposed tail), at most kMaxBands; a small frame is one band.  (Finer bands were measured
// on the 1 MB frame of C1: 8 bands of 128 KB take 54 us to drain against 25 us for the single copy -- every
// device-to-host copy costs ~7 us on its own.)  A band is never lower than a strip.
void band_layout(uint32_t width, uint32_t height, uint32_t strip_h, uint32_t& band_rows, uint32_t& n_bands)
{
    const uint64_t frame_bytes = (uint64_t) width * height * sizeof(uint32_t);
    const uint32_t want_bands = (uint32_t) std::min<uint64_t>(kMaxBands, std::max<uint64_t>(1, frame_bytes >> 20));
    band_rows = std::max<uint32_t>(strip_h, (height + want_bands - 1) / want_bands);
    n_bands = (height + band_rows - 1) / band_rows;
}

// Pieces of strips per row band for every participating GPU (`world` of them; strips dealt in chunks of
// `chunk`, owner rotating from round to round -- the same arithmetic as in trace_tiles_kernel), and how many GPUs
// have a share in each band.  A strip that straddles a band boundary counts in both, exactly as the kernel
// bumps both.
void band_shares(const std::vector<uint4>& rects, const std::vector<uint32_t>& prefix, uint32_t strip_w, uint32_t strip_h,
                 uint32_t band_rows, uint32_t parts, uint32_t chunk, uint32_t world,
                 std::vector<std::array<uint32_t, kMaxBands>>& share, uint32_t *gpus_in_band)
{
    share.assign(world, std::array<uint32_t, kMaxBands>());
    for (size_t k = 0; k < rects.size(); k++)
    {
        const uint4& r = rects[k];
        const uint32_t nx = (r.z - r.x + strip_w - 1) / strip_w;
        uint64_t row_first = prefix[k];
        for (uint32_t y = r.y; y < r.w; y += strip_h, row_first += nx)
        {
            const uint32_t b0 = y / band_rows, b1 = (std::min(y + strip_h, r.w) - 1) / band_rows;
            for (uint64_t s = row_first; s < row_first + nx;)
            {
                const uint64_t c = s / chunk, seg_end = std::min<uint64_t>(row_first + nx, (c + 1) * chunk);
                const uint32_t owner = (uint32_t) ((c % world + c / world) % world);
                const uint32_t n = (uint32_t) (seg_end - s) * parts;
                share[owner][b0] += n;
                if (b1 != b0)
                    share[owner][b1] += n;
                s = seg_end;
            }
        }
    }
    for (int b = 0; b < kMaxBands; b++)
    {
        gpus_in_band[b] = 0;
        for (uint32_t q = 0; q < world; q++)
            gpus_in_band[b] += share[q][b] ? 1u : 0u;
    }
}

} // namespace

extern "C"
{

int cuda_trace_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess)
        return 0;
    return n;
}

int cuda_trace_init_devices(const int *device_ordinals, int n, cuda_trace_ctx **out)
{
    cuda_trace_ctx *ctx = nullptr;
    if (!out || n < 1 || !device_ordinals)
        return fail(nullptr, CUDA_TRACE_ERR_ARG, "cuda_trace_init: bad arguments");
    *out = nullptr;
    int have = 0;
    cudaError_t e = cudaGetDeviceCount(&have);
    if (e != cudaSuccess || have < 1)
        return fail(nullptr, CUDA_TRACE_ERR_NO_DEVICE,
                    std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    for (int i = 0; i < n; i++)
        if (device_ordinals[i] < 0 || device_ordinals[i] >= have)
            return fail(nullptr, CUDA_TRACE_ERR_NO_DEVICE, "requested device ordinal " +
                        std::to_string(device_ordinals[i]) + " but only " + std::to_string(have) + " present");

    ctx = new cuda_trace_ctx();
    std::memset(&ctx->desc, 0, sizeof(ctx->desc));
    std::memset(&ctx->frame, 0, sizeof(ctx->frame));
    ctx->dev.resize(n);
    auto bail = [&](const std::string& msg, int code) {
        g_init_error = msg;
        cuda_trace_destroy(ctx);
        return code;
    };
    for (int i = 0; i < n; i++)
    {
        DeviceState& d = ctx->dev[i];
        d.ordinal = device_ordinals[i];
        cudaDeviceProp prop;
        if ((e = cudaSetDevice(d.ordinal)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, d.ordinal)) != cudaSuccess)
            return bail(std::string("cudaSetDevice/GetDeviceProperties: ") + cudaGetErrorString(e), CUDA_TRACE_ERR_CUDA);
        if (prop.major < 10)
            return bail("device " + std::to_string(d.ordinal) + " (" + prop.name + ") is sm_" +
                        std::to_string(prop.major * 10 + prop.minor) + "; this library is built for sm_100a only",
                        CUDA_TRACE_ERR_NO_DEVICE);
        d.sm_count = prop.multiProcessorCount;
        if ((e = cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaStreamCreateWithFlags(&d.side_stream, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaStreamCreateWithFlags(&d.copy_stream, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaStreamCreateWithFlags(&d.order_stream, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&d.ev_traced, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&d.ev_order, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&d.ev_copy, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaEventCreate(&d.ev_begin)) != cudaSuccess || (e = cudaEventCreate(&d.ev_end)) != cudaSuccess ||
            (e = d.d_strip_counter.alloc(32 + kMaxBands + 32)) != cudaSuccess || // {strip counter, pad to 128 B | band piece counts | cancel word}
            (e = d.h_cancel_seen.alloc(1)) != cudaSuccess ||
            (e = cudaHostGetDevicePointer((void **) &d.d_cancel_seen, d.h_cancel_seen.get(), 0)) != cudaSuccess ||
            (e = d.d_counters.alloc(1)) != cudaSuccess ||
            (e = cudaMemset(d.d_strip_counter.get(), 0, (32 + kMaxBands + 32) * sizeof(uint32_t))) != cudaSuccess ||
            (e = cudaMemset(d.d_counters.get(), 0, sizeof(Counters))) != cudaSuccess)
            return bail(std::string("device set-up: ") + cudaGetErrorString(e), CUDA_TRACE_ERR_CUDA);
        d.d_cancel = d.d_strip_counter.get() + 32 + kMaxBands; // outside the per-frame memset
        *d.h_cancel_seen.get() = 0;
        if (i > 0)
        {
            // strips rendered on device i are stored straight into device 0's framebuffer
            int can = 0;
            cudaDeviceCanAccessPeer(&can, d.ordinal, ctx->dev[0].ordinal);
            if (!can)
                return bail("device " + std::to_string(d.ordinal) + " cannot access device " +
                            std::to_string(ctx->dev[0].ordinal) + " as a peer", CUDA_TRACE_ERR_NO_DEVICE);
            e = cudaDeviceEnablePeerAccess(ctx->dev[0].ordinal, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled)
                cudaGetLastError();
            else if (e != cudaSuccess)
                return bail(std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e), CUDA_TRACE_ERR_CUDA);
        }
    }
    if ((e = ctx->pinned_cancel_src.alloc(1)) != cudaSuccess)
        return bail(std::string("cudaHostAlloc: ") + cudaGetErrorString(e), CUDA_TRACE_ERR_CUDA);
    *ctx->pinned_cancel_src.get() = 0;
    {
        // stream-ordered "wait until *addr >= value" (driver API), used by the overlapped read-back
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuStreamWaitValue32", &fn, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            ctx->wait_value32 = reinterpret_cast<int (*)(cudaStream_t, unsigned long long, unsigned int, unsigned int)>(fn);
        else
            cudaGetLastError();
        // the allocation a device pointer lies in (driver API), for the range check of cuda_trace_upload_scene_device
        fn = nullptr;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            ctx->mem_range = reinterpret_cast<int (*)(unsigned long long *, size_t *, unsigned long long)>(fn);
        else
            cudaGetLastError();
        if (const char *e = std::getenv("RTM_OVERLAP_D2H"))
            ctx->overlap_d2h = std::atoi(e) != 0;
    }
    // Tuning switches are read here, once per context (experiments and tests; every default is the measured best)
    if (const char *e = std::getenv("RTM_REL_RECORDS"))
    {
        ctx->rel_records = std::atoi(e) != 0;
        ctx->rel_records_forced = std::atoi(e) == 2;
    }
    if (const char *e = std::getenv("RTM_SCREEN_CULL"))
        ctx->screen_cull = std::atoi(e) < 0 ? -1 : (std::atoi(e) != 0 ? 1 : 0);
    if (const char *e = std::getenv("RTM_COST_ORDER"))
        ctx->cost_order_forced = std::atoi(e) != 0 ? 1 : 0;
    if (const char *e = std::getenv("RTM_FAST_MATH"))
        ctx->fast_math = std::atoi(e) != 0;
    if (const char *e = std::getenv("RTM_STRIP_PIXELS"))
    {
        const int px = std::atoi(e);
        if (px == 2 || px == 4 || px == 8 || px == 16 || px == 32)
            ctx->tune.strip_pixels = px;
    }
    if (const char *e = std::getenv("RTM_SPLIT_PARTS"))
        ctx->tune.split_parts = (std::atoi(e) == 1 || std::atoi(e) == 2) ? std::atoi(e) : 0;
    if (const char *e = std::getenv("RTM_OCC_MODE"))
        ctx->tune.occ_mode = (std::atoi(e) >= 0 && std::atoi(e) <= 3) ? std::atoi(e) : -1;
    if (const char *e = std::getenv("RTM_POOL"))
        ctx->tune.pool = std::atoi(e) != 0 ? 1 : 0;
    if (const char *e = std::getenv("RTM_POOL_STEPS"))
        ctx->tune.pool_steps = std::min(4096, std::max(1, std::atoi(e)));
    if (const char *e = std::getenv("RTM_THREADS"))
    {
        const int t = std::atoi(e);
        if (t >= 32 && t <= 1024 && t % 32 == 0)
            ctx->tune.threads = t;
    }
    if (const char *e = std::getenv("RTM_BAND_FLUSH"))
        ctx->tune.band_flush = std::min(64, std::max(1, std::atoi(e)));
    if (const char *e = std::getenv("RTM_SHARD_CHUNK"))
        ctx->shard_chunk = (uint32_t) std::max(1, std::atoi(e));
    *out = ctx;
    return 0;
}

int cuda_trace_init(int n_gpus, cuda_trace_ctx **out)
{
    if (n_gpus < 1 || n_gpus > 64)
        return fail(nullptr, CUDA_TRACE_ERR_ARG, "cuda_trace_init: n_gpus must be 1..64");
    int ids[64];
    for (int i = 0; i < n_gpus; i++)
        ids[i] = i;
    return cuda_trace_init_devices(ids, n_gpus, out);
}

void cuda_trace_destroy(cuda_trace_ctx *ctx)
{
    if (!ctx)
        return;
    for (DeviceState& d : ctx->dev)
    {
        cudaSetDevice(d.ordinal);
        if (d.stream) cudaStreamSynchronize(d.stream);
        if (d.copy_stream && !ctx->shard_signals) cudaStreamSynchronize(d.copy_stream);
        if (d.order_stream) cudaStreamSynchronize(d.order_stream);
    }
    wait_for_queries(ctx);
    for (auto& se : ctx->query_events)
        cudaEventDestroy(se.second);
    if (!ctx->dev.empty())
    {
        cudaSetDevice(ctx->dev[0].ordinal);
        if (ctx->fb_imported && ctx->d_fb)
            cudaIpcCloseMemHandle(ctx->d_fb);
        if (ctx->ev_mesh_input) cudaEventDestroy(ctx->ev_mesh_input);
    }
    for (DeviceState& d : ctx->dev)
    {
        cudaSetDevice(d.ordinal);
        if (d.ev_begin) cudaEventDestroy(d.ev_begin);
        if (d.ev_end) cudaEventDestroy(d.ev_end);
        if (d.stream) cudaStreamDestroy(d.stream);
        if (d.side_stream) cudaStreamDestroy(d.side_stream);
        if (d.copy_stream) cudaStreamDestroy(d.copy_stream);
        if (d.order_stream) cudaStreamDestroy(d.order_stream);
        if (d.ev_traced) cudaEventDestroy(d.ev_traced);
        if (d.ev_order) cudaEventDestroy(d.ev_order);
        if (d.ev_copy) cudaEventDestroy(d.ev_copy);
    }
    for (cudaEvent_t ev : ctx->tile_events)
        cudaEventDestroy(ev);
    delete ctx; // and with it every array it owns
}

const char *cuda_trace_last_error(const cuda_trace_ctx *ctx) { return ctx ? ctx->err.c_str() : g_init_error.c_str(); }

uint64_t cuda_trace_kernel_launches(const cuda_trace_ctx *ctx) { return ctx ? ctx->launches.load() : 0; }

int cuda_trace_set_shard(cuda_trace_ctx *ctx, uint32_t rank, uint32_t world)
{
    if (!ctx)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (world == 0 || rank >= world)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "set_shard: need rank < world");
    ctx->shard_rank = rank;
    ctx->shard_world = world;
    return 0;
}

int cuda_trace_set_shard_signals(cuda_trace_ctx *ctx, int enable)
{
    if (!ctx)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    ctx->shard_signals = enable != 0;
    return 0;
}

// ------------------------------------------------------------------------------------- scene
int cuda_trace_upload_scene(cuda_trace_ctx *ctx, const float *vertices, uint32_t num_vertices,
                            const uint32_t *triangles, uint32_t num_triangles, uint32_t grid_res)
{
    int rc = check_mesh_args(ctx, vertices, num_vertices, triangles, num_triangles);
    if (rc)
        return rc;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (grid_res == 0)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "upload_scene: grid_res must be > 0 (grid.cpp:16)");
    if ((rc = cuda_trace_sync(ctx)))
        return rc;
    wait_for_queries(ctx);
    return build_scene(ctx, num_vertices, num_triangles, [&](DeviceState& d, size_t i) {
        const int rc = upload_mesh(ctx, d, vertices, num_vertices, triangles, num_triangles);
        return rc ? rc : build_grid(ctx, d, i, grid_res);
    });
}

int cuda_trace_upload_scene_device(cuda_trace_ctx *ctx, const float *vertices, uint32_t num_vertices,
                                   const uint32_t *triangles, uint32_t num_triangles, uint32_t grid_res, void *stream)
{
    if (!ctx)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (!vertices || !triangles || num_vertices == 0 || num_triangles == 0)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "upload_scene_device: empty mesh (the reference asserts, grid.cpp:15)");
    if (grid_res == 0)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "upload_scene_device: grid_res must be > 0 (grid.cpp:16)");
    DeviceState& d0 = ctx->dev[0];
    CK(cudaSetDevice(d0.ordinal));
    int rc = 0;
    if ((rc = check_device_array(ctx, vertices, num_vertices, "vertices")) ||
        (rc = check_device_array(ctx, triangles, num_triangles, "triangles")))
        return rc;
    if ((rc = cuda_trace_sync(ctx)))
        return rc;
    wait_for_queries(ctx);
    // The caller's arrays are complete once the work already enqueued on its stream is: the context's stream waits
    // for that, then checks the vertex indices on the device.  The old scene is freed only after they passed.
    CK(cudaSetDevice(d0.ordinal));
    if (!ctx->ev_mesh_input)
        CK(cudaEventCreateWithFlags(&ctx->ev_mesh_input, cudaEventDisableTiming));
    CK(ctx->d_first_bad.grow(1));
    CK(cudaEventRecord(ctx->ev_mesh_input, stream ? (cudaStream_t) stream : d0.stream));
    CK(cudaStreamWaitEvent(d0.stream, ctx->ev_mesh_input, 0));
    CK(cudaMemsetAsync(ctx->d_first_bad.get(), 0xFF, sizeof(uint32_t), d0.stream));
    launch_check_triangle_indices(triangles, num_triangles, num_vertices, ctx->d_first_bad.get(), d0.stream);
    ctx->launches++;
    CK(cudaGetLastError());
    uint32_t first_bad = 0;
    CK(cudaMemcpyAsync(&first_bad, ctx->d_first_bad.get(), sizeof(uint32_t), cudaMemcpyDeviceToHost, d0.stream));
    CK(cudaStreamSynchronize(d0.stream));
    if (first_bad != 0xFFFFFFFFu)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "upload_scene_device: vertex index out of bounds in triangle " +
                                                 std::to_string(first_bad) + " (num_vertices " +
                                                 std::to_string(num_vertices) + ")");
    const size_t vtx_bytes = (size_t) num_vertices * 24, tri_bytes = (size_t) num_triangles * 24;
    return build_scene(ctx, num_vertices, num_triangles, [&](DeviceState& d, size_t i) {
        SceneArrays& s = d.scene;
        CK(cudaSetDevice(d.ordinal));
        CK(s.d_vtx.alloc((size_t) num_vertices * 6));
        CK(s.d_tri.alloc((size_t) num_triangles * 6));
        if (i == 0)
        {
            // ordered after the caller's stream by the event wait above
            CK(cudaMemcpyAsync(s.d_vtx.get(), vertices, vtx_bytes, cudaMemcpyDeviceToDevice, d.stream));
            CK(cudaMemcpyAsync(s.d_tri.get(), triangles, tri_bytes, cudaMemcpyDeviceToDevice, d.stream));
        }
        else
        {
            // device 0's copy is complete: its build synchronised its stream (build_scene)
            CK(cudaMemcpyPeerAsync(s.d_vtx.get(), d.ordinal, d0.scene.d_vtx.get(), d0.ordinal, vtx_bytes, d.stream));
            CK(cudaMemcpyPeerAsync(s.d_tri.get(), d.ordinal, d0.scene.d_tri.get(), d0.ordinal, tri_bytes, d.stream));
        }
        return build_grid(ctx, d, i, grid_res);
    });
}

uint32_t cuda_trace_suggest_grid_res(uint32_t num_triangles)
{
    // ~3 cells per triangle while the occupancy map of the grid fits in shared memory (K1); grids beyond that are
    // traversed by K7 (pooled rays, distance map), whose optimum on the soup sweep lies at ~9 cells per triangle
    // (768^3 for 50.1 M triangles: 70.4 ms against 74.0 at 640^3 and 86.5 at 512^3)
    double r = std::cbrt(3.0 * (double) num_triangles);
    if (r > 108.0)
        r = std::cbrt(9.0 * (double) num_triangles);
    return (uint32_t) std::min(896.0, std::max(16.0, std::floor(r + 0.5)));
}

int cuda_trace_upload_scene_with_grid(cuda_trace_ctx *ctx, const float *vertices, uint32_t num_vertices,
                                      const uint32_t *triangles, uint32_t num_triangles,
                                      const cuda_trace_grid_desc *desc, const uint64_t *cell_offset,
                                      const uint32_t *tri_index)
{
    int rc = check_mesh_args(ctx, vertices, num_vertices, triangles, num_triangles);
    if (rc)
        return rc;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (!desc || !cell_offset || (!tri_index && desc->num_refs))
        return fail(ctx, CUDA_TRACE_ERR_ARG, "upload_scene_with_grid: null grid arrays");
    const uint64_t cells = (uint64_t) desc->dim[0] * desc->dim[1] * desc->dim[2];
    if (cells == 0 || cells != desc->num_cells || cells >= (1ull << 31) || desc->num_refs >= (1ull << 32) ||
        cell_offset[0] != 0 || cell_offset[cells] != desc->num_refs)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "upload_scene_with_grid: inconsistent grid description");
    for (uint64_t c = 0; c < cells; c++)
        if (cell_offset[c] > cell_offset[c + 1])
            return fail(ctx, CUDA_TRACE_ERR_ARG, "upload_scene_with_grid: cell_offset not monotone");
    for (uint64_t k = 0; k < desc->num_refs; k++)
        if (tri_index[k] >= num_triangles)
            return fail(ctx, CUDA_TRACE_ERR_ARG, "upload_scene_with_grid: triangle index out of bounds");
    if ((rc = cuda_trace_sync(ctx)))
        return rc;
    wait_for_queries(ctx);
    ctx->desc = *desc;
    return build_scene(ctx, num_vertices, num_triangles, [&](DeviceState& d, size_t) {
        const int rc = upload_mesh(ctx, d, vertices, num_vertices, triangles, num_triangles);
        if (rc)
            return rc;
        DeviceArray<uint64_t> d_off64;
        StreamDrain drain(d.stream);
        CK(d_off64.alloc(cells + 1));
        CK(d.scene.d_cell_start.alloc(cells + 1));
        CK(d.scene.d_tri_index.alloc(std::max<uint64_t>(desc->num_refs, 1)));
        CK(cudaMemcpyAsync(d_off64.get(), cell_offset, (cells + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, d.stream));
        if (desc->num_refs)
            CK(cudaMemcpyAsync(d.scene.d_tri_index.get(), tri_index, desc->num_refs * sizeof(uint32_t), cudaMemcpyHostToDevice,
                               d.stream));
        launch_narrow_offsets(d_off64.get(), cells + 1, d.scene.d_cell_start.get(), d.stream);
        ctx->launches++;
        CK(drain.sync());
        return 0;
    });
}

int cuda_trace_download_grid(cuda_trace_ctx *ctx, cuda_trace_grid_desc *desc, uint64_t *cell_offset,
                             uint32_t *tri_index)
{
    if (!ctx || !desc)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (!ctx->have_scene)
        return fail(ctx, CUDA_TRACE_ERR_NO_SCENE, "download_grid: no scene uploaded");
    *desc = ctx->desc;
    DeviceState& d = ctx->dev[0];
    CK(cudaSetDevice(d.ordinal));
    if (cell_offset)
    {
        DeviceArray<uint64_t> d_off64;
        StreamDrain drain(d.stream);
        CK(d_off64.alloc(ctx->desc.num_cells + 1));
        launch_widen_offsets(d.scene.d_cell_start.get(), ctx->desc.num_cells + 1, d_off64.get(), d.stream);
        ctx->launches++;
        CK(cudaMemcpyAsync(cell_offset, d_off64.get(), (ctx->desc.num_cells + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost,
                           d.stream));
        CK(drain.sync());
    }
    if (tri_index && ctx->desc.num_refs)
    {
        CK(cudaMemcpyAsync(tri_index, d.scene.d_tri_index.get(), ctx->desc.num_refs * sizeof(uint32_t), cudaMemcpyDeviceToHost,
                           d.stream));
        CK(cudaStreamSynchronize(d.stream));
    }
    return 0;
}

int cuda_trace_download_distance_map(cuda_trace_ctx *ctx, uint8_t *out, uint64_t *num_bytes)
{
    if (!ctx || !num_bytes)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (!ctx->have_scene)
        return fail(ctx, CUDA_TRACE_ERR_NO_SCENE, "download_distance_map: no scene uploaded");
    DeviceState& d = ctx->dev[0];
    const uint64_t pcells = (uint64_t) (ctx->desc.dim[0] + 2) * (ctx->desc.dim[1] + 2) * (ctx->desc.dim[2] + 2);
    *num_bytes = d.scene.d_pcell_dist.get() ? pcells : 0;
    if (out && d.scene.d_pcell_dist.get())
    {
        CK(cudaSetDevice(d.ordinal));
        CK(cudaMemcpyAsync(out, d.scene.d_pcell_dist.get(), pcells, cudaMemcpyDeviceToHost, d.stream));
        CK(cudaStreamSynchronize(d.stream));
    }
    return 0;
}

int cuda_trace_download_screen_boxes(cuda_trace_ctx *ctx, float *boxes, uint64_t capacity, uint64_t *num_pairs,
                                     uint32_t *small, int *cull_on)
{
    if (!ctx || !num_pairs || !small || !cull_on || (capacity && !boxes))
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    *num_pairs = 0;
    *small = 0;
    *cull_on = 0;
    if (!ctx->have_scene || ctx->dev.empty() || !ctx->dev[0].scene.sbox_valid)
        return 0;
    // read only: the boxes, their camera and the gate stay as the last frame left them
    DeviceState& d = ctx->dev[0];
    *num_pairs = ctx->num_pairs;
    *small = d.scene.sbox_small;
    *cull_on = d.scene.sbox_cull ? 1 : 0;
    const uint64_t n = std::min<uint64_t>(*num_pairs, capacity / 4);
    if (n)
    {
        CK(cudaSetDevice(d.ordinal));
        CK(cudaMemcpyAsync(boxes, d.scene.d_pair_sbox.get(), n * sizeof(float4), cudaMemcpyDeviceToHost, d.stream));
        CK(cudaStreamSynchronize(d.stream));
    }
    return 0;
}

// ----------------------------------------------------------------------------------- tracing
int cuda_trace_prepare_framebuffer(cuda_trace_ctx *ctx, uint32_t width, uint32_t height)
{
    if (!ctx || width == 0 || height == 0)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    int rc = ensure_framebuffer(ctx, width, height);
    if (rc)
        return rc;
    CK(cudaStreamSynchronize(ctx->dev[0].stream));
    return 0;
}

int cuda_trace_export_framebuffer(cuda_trace_ctx *ctx, void *handle64)
{
    if (!ctx || !handle64)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (!ctx->d_fb || ctx->fb_imported)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "export_framebuffer: call cuda_trace_prepare_framebuffer first");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    CK(cudaSetDevice(ctx->dev[0].ordinal));
    CK(cudaIpcGetMemHandle(&h, ctx->d_fb));
    std::memcpy(handle64, &h, 64);
    return 0;
}

int cuda_trace_import_framebuffer(cuda_trace_ctx *ctx, const void *handle64, uint32_t width, uint32_t height)
{
    if (!ctx || !handle64 || width == 0 || height == 0)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    int rc = cuda_trace_sync(ctx);
    if (rc)
        return rc;
    CK(cudaSetDevice(ctx->dev[0].ordinal));
    if (ctx->fb_imported && ctx->d_fb)
        CK(cudaIpcCloseMemHandle(ctx->d_fb));
    ctx->d_fb = nullptr;
    ctx->fb_own.release();
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle64, 64);
    void *p = nullptr;
    CK(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->d_fb = (uint32_t *) p;
    ctx->fb_imported = true;
    ctx->fb_w = width;
    ctx->fb_h = height;
    return 0;
}

void *cuda_trace_framebuffer_device_ptr(cuda_trace_ctx *ctx) { return ctx ? ctx->d_fb : nullptr; }
void *cuda_trace_stream(cuda_trace_ctx *ctx) { return (ctx && !ctx->dev.empty()) ? (void *) ctx->dev[0].stream : nullptr; }

int cuda_trace_set_counting(cuda_trace_ctx *ctx, int enable)
{
    if (!ctx)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    ctx->counting = enable != 0;
    return 0;
}

} // extern "C"

// ------------------------------------------------------------------------------------------------- one frame
// cuda_trace_tiles in five steps, each its own function:
//   check_frame_args      everything that can be refused is refused BEFORE any state changes
//   update_plan           tile list -> strips (cached while the layout repeats)
//   plan_band_counts      completion targets of the overlapped read-back for this layout (cached)
//   launch_on_device      per-GPU buffers, kernel parameters, launch configuration, launch, cost-order follow-up
//   enqueue_band_copies   copy stream: wait for a row band, ship it to the host buffer
namespace
{

constexpr uint32_t kMaxSpp = 4096; // sample table in shared memory: 32 KB next to the occupancy map

struct FrameKind
{
    bool keep_hits, ortho, alternates, count_inst;
    uint32_t shade_mode;
};

int check_frame_args(cuda_trace_ctx *ctx, const cuda_trace_frame *f, const cuda_trace_tile_rect *tiles, uint32_t n_tiles,
                     FrameKind& kind)
{
    if (!ctx->have_scene)
        return fail(ctx, CUDA_TRACE_ERR_NO_SCENE, "trace_tiles: upload a scene first");
    if (f->width == 0 || f->height == 0 || f->spp == 0 || f->variant > 1)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "trace_tiles: bad frame description");
    if (f->spp > kMaxSpp)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "trace_tiles: at most " + std::to_string(kMaxSpp) + " samples per pixel");
    if ((uint64_t) f->width * f->height >= (1ull << 32))
        return fail(ctx, CUDA_TRACE_ERR_ARG, "trace_tiles: frame too large");
    for (uint32_t i = 0; i < n_tiles; i++)
    {
        const cuda_trace_tile_rect& t = tiles[i];
        if (t.x0 > t.x1 || t.y0 > t.y1 || t.x1 > f->width || t.y1 > f->height)
            return fail(ctx, CUDA_TRACE_ERR_ARG, "trace_tiles: tile " + std::to_string(i) + " outside the frame");
    }
    if (ctx->fb_imported && (ctx->fb_w != f->width || ctx->fb_h != f->height))
        return fail(ctx, CUDA_TRACE_ERR_ARG, "frame size differs from the imported framebuffer");
    kind.keep_hits = (f->flags & CUDA_TRACE_FLAG_KEEP_HITS) != 0;
    kind.ortho = (f->flags & CUDA_TRACE_FLAG_ORTHO) != 0;
    kind.shade_mode = (f->flags & CUDA_TRACE_FLAG_SHADE_FACE_NORMAL) ? 1u : ((f->flags & CUDA_TRACE_FLAG_SHADE_DEPTH) ? 2u : 0u);
    kind.alternates = kind.ortho || kind.shade_mode != 0;
    // The packed-pair test pads odd lists with a triangle at x = -1e18 that no ray can hit as long as scene and
    // camera stay within +-1e9 (pack.cu).  Anything larger takes the scalar test of the counting instantiation.
    bool big_coords = false;
    for (int k = 0; k < 3; k++)
        big_coords = big_coords || !(std::fabs(ctx->desc.aabb_min[k]) < 1.0e9f) || !(std::fabs(ctx->desc.aabb_max[k]) < 1.0e9f) ||
                     !(std::fabs(f->cam_mat[12 + k]) < 1.0e9f);
    if (kind.ortho)
        big_coords = big_coords || !(std::fabs(f->fov_xs) < 1.0e9f) || !(std::fabs(f->fov_xs / f->aspect) < 1.0e9f);
    if (kind.alternates && big_coords)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "trace_tiles: the orthographic camera / shading alternates need scene and "
                                             "camera coordinates within +-1e9");
    if (kind.alternates && ctx->counting)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "trace_tiles: the work counters are not available with the orthographic "
                                             "camera / shading alternates");
    kind.count_inst = ctx->counting || big_coords; // kernel instantiation with the scalar test (+ work counters)
    return 0;
}

// Tile list -> strips (strip_w x strip_h pixel blocks, clipped to the tile).  No device work, no context state
// other than ctx->plan; returns an error only for layouts with too many strips.
int update_plan(cuda_trace_ctx *ctx, const cuda_trace_frame *f, const cuda_trace_tile_rect *tiles, uint32_t n_tiles)
{
    FramePlan& pl = ctx->plan;
    if (pl.serial && pl.width == f->width && pl.height == f->height && pl.spp == f->spp && pl.tiles.size() == n_tiles &&
        (n_tiles == 0 || std::memcmp(pl.tiles.data(), tiles, sizeof(cuda_trace_tile_rect) * n_tiles) == 0))
        return 0;
    FramePlan np;
    np.width = f->width; np.height = f->height; np.spp = f->spp;
    np.tiles.assign(tiles, tiles + n_tiles);
    strip_size_for_spp(f->spp, (uint64_t) f->width * f->height * f->spp, np.strip_w, np.strip_h);
    if (const int px = ctx->tune.strip_pixels)
    {
        np.strip_w = px >= 32 ? 8 : (px >= 8 ? 4 : 2);
        np.strip_h = px >= 16 ? 4 : (px >= 4 ? 2 : 1);
    }
    np.split_parts = strip_split_parts(np.strip_w, np.strip_h, f->spp);
    if (ctx->tune.split_parts == 1 || (ctx->tune.split_parts == 2 && np.split_parts >= 2))
        np.split_parts = (uint32_t) ctx->tune.split_parts;
    np.rects.resize(n_tiles);
    np.prefix.assign(n_tiles + 1, 0);
    uint64_t total = 0, area = 0;
    for (uint32_t i = 0; i < n_tiles; i++)
    {
        const cuda_trace_tile_rect& t = tiles[i];
        np.rects[i] = make_uint4(t.x0, t.y0, t.x1, t.y1);
        np.prefix[i] = (uint32_t) total;
        total += (uint64_t) ((t.x1 - t.x0 + np.strip_w - 1) / np.strip_w) * ((t.y1 - t.y0 + np.strip_h - 1) / np.strip_h);
        area += (uint64_t) (t.x1 - t.x0) * (t.y1 - t.y0);
        if (total >= (1ull << 32))
            return fail(ctx, CUDA_TRACE_ERR_ARG, "trace_tiles: too many strips");
    }
    np.prefix[n_tiles] = (uint32_t) total;
    np.total = total;
    // "the tiles cover the frame" exactly: areas add up to the frame AND no two tiles overlap
    bool disjoint = area == (uint64_t) f->width * f->height;
    for (uint32_t i = 0; disjoint && i < n_tiles; i++)
        for (uint32_t k = i + 1; k < n_tiles; k++)
        {
            const cuda_trace_tile_rect &a = tiles[i], &b = tiles[k];
            if (a.x0 < b.x1 && b.x0 < a.x1 && a.y0 < b.y1 && b.y0 < a.y1 && a.x0 < a.x1 && a.y0 < a.y1 && b.x0 < b.x1 && b.y0 < b.y1)
            {
                disjoint = false;
                break;
            }
        }
    np.covers_frame = disjoint;
    np.serial = pl.serial + 1;
    pl = std::move(np);
    return 0;
}

// Completion targets of the overlapped read-back (cached per layout): ctx->band_inc[b] = what a frame adds to the
// counter of band b, ctx->band_share[q][b] = pieces GPU q contributes
void plan_band_counts(cuda_trace_ctx *ctx)
{
    const FramePlan& pl = ctx->plan;
    band_layout(pl.width, pl.height, pl.strip_h, ctx->band_rows, ctx->n_bands);
    const uint32_t participants = ctx->shard_world * (uint32_t) ctx->dev.size();
    // Two levels: every GPU counts its pieces per band in its own memory (release at GPU scope: cheap) and the warp
    // that completes the GPU's share bumps the band counter once, at system scope -- the reader is a copy engine or
    // another GPU.  So a frame adds to a band's counter the number of GPUs with a share in it.
    const std::vector<uint64_t> sig = { pl.serial, participants, ctx->shard_chunk };
    if (sig == ctx->band_inc_sig)
        return;
    band_shares(pl.rects, pl.prefix, pl.strip_w, pl.strip_h, ctx->band_rows, pl.split_parts, ctx->shard_chunk, participants,
                ctx->band_share, ctx->band_inc);
    ctx->band_inc_sig = sig;
}

// After a launch failed half way the band counters on the device and the totals kept here may disagree: wait for
// whatever is in flight and re-read them (the counters are monotone and never reset)
int resync_band_counters(cuda_trace_ctx *ctx)
{
    for (DeviceState& d : ctx->dev)
    {
        CK(cudaSetDevice(d.ordinal));
        CK(cudaStreamSynchronize(d.stream));
    }
    if (ctx->d_fb)
    {
        CK(cudaSetDevice(ctx->dev[0].ordinal));
        CK(cudaMemcpy(ctx->band_expected, band_counters(ctx), sizeof(ctx->band_expected), cudaMemcpyDeviceToHost));
    }
    ctx->band_dirty = false;
    return 0;
}

int ensure_hit_buffers(cuda_trace_ctx *ctx, const cuda_trace_frame *f)
{
    const uint64_t need = (uint64_t) f->width * f->height * f->spp;
    CK(cudaSetDevice(ctx->dev[0].ordinal));
    CK(ctx->d_hit_tri.grow(need));
    CK(ctx->d_hit_t.grow(need));
    CK(ctx->d_hit_u.grow(need));
    CK(ctx->d_hit_v.grow(need));
    ctx->hit_count = need;
    // samples outside the requested tiles read as "miss"
    CK(cudaMemsetAsync(ctx->d_hit_tri.get(), 0xFF, need * 4, ctx->dev[0].stream));
    CK(cudaMemsetAsync(ctx->d_hit_t.get(), 0, need * 4, ctx->dev[0].stream));
    CK(cudaMemsetAsync(ctx->d_hit_u.get(), 0, need * 4, ctx->dev[0].stream));
    CK(cudaMemsetAsync(ctx->d_hit_v.get(), 0, need * 4, ctx->dev[0].stream));
    CK(cudaStreamSynchronize(ctx->dev[0].stream));
    return 0;
}

void fill_camera(const cuda_trace_ctx *ctx, const cuda_trace_frame *f, const FrameKind& kind, TraceParams& p)
{
    for (int r = 0; r < 3; r++)
    {
        for (int c = 0; c < 3; c++)
            p.cam.m[r][c] = f->cam_mat[r * 4 + c];
        // perspective: origin = Transf4x4(Vec3f(0)) (camera.h:43, lin_alg.h:518-535), all four terms kept
        // (a -0 translation comes out as +0); orthographic: the raw row, used per ray
        const float zero = 0.0f, m3 = f->cam_mat[12 + r];
        p.cam.origin[r] = kind.ortho ? m3 : zero * f->cam_mat[0 + r] + zero * f->cam_mat[4 + r] + zero * f->cam_mat[8 + r] + m3;
    }
    p.cam.ortho = kind.ortho ? 1u : 0u;
    {
        // camera.h:28-31: const float width = width_or_hfov, height = float(width) / aspect; half = x / 2.0
        const float ow = f->fov_xs, oh = ow / f->aspect;
        p.cam.ortho_half_w = (float) ((double) ow / 2.0);
        p.cam.ortho_half_h = (float) ((double) oh / 2.0);
    }
    p.shade_mode = kind.shade_mode;
    p.cam.fov_xs = f->fov_xs;
    p.cam.aspect = f->aspect;
    p.cam.width_f = (float) f->width;
    p.cam.height_f = (float) f->height;
    // frame constants of the range-check-free divisions (rt_device.cuh): valid while every operand and
    // quotient of generate_ray and of the DDA set-up is an ordinary normal number
    p.cam.inv_width = 1.0f / p.cam.width_f;
    p.cam.inv_height = 1.0f / p.cam.height_f;
    p.cam.inv_aspect = 1.0f / f->aspect;
    const auto ordinary = [](float x) { return std::fabs(x) >= 0x1p-20f && std::fabs(x) <= 0x1p20f; };
    p.cam.fast_math = (ctx->fast_math && ordinary(f->fov_xs) && ordinary(f->aspect) && ordinary(ctx->desc.cell_wdh) &&
                       f->width <= (1u << 20) && f->height <= (1u << 20)) ? 1u : 0u;
    p.width = f->width;
    p.height = f->height;
    p.spp = f->spp;
    p.gamma = (f->flags & CUDA_TRACE_FLAG_GAMMA) ? 1u : 0u;
    const float one[2] = { 1.0f, 1.0f }, minus_one[2] = { -1.0f, -1.0f };
    std::memcpy(&p.pk_one, one, sizeof(p.pk_one));
    std::memcpy(&p.pk_minus_one, minus_one, sizeof(p.pk_minus_one));
}

// Where the padded occupancy map is read from (warp_trace.cuh), for frames and ray queries alike: when staging is
// worth it (smem_ok), one byte per cell in shared memory when that leaves room (<= 160 KB next to `other_smem` bytes
// the kernel also needs), else bits in shared memory; otherwise the distance map through L1 where the scene has one,
// else bits through L1.  RTM_OCC_MODE overrides the choice where the forced home exists and fits.
void choose_occupancy_home(const cuda_trace_ctx *ctx, const DeviceState& d, bool smem_ok, size_t other_smem,
                           uint32_t& occ_mode, uint32_t& occ_smem_words)
{
    const uint64_t pcells = (uint64_t) (ctx->desc.dim[0] + 2) * (ctx->desc.dim[1] + 2) * (ctx->desc.dim[2] + 2);
    const uint64_t bit_words = (pcells + 31) / 32, byte_words = (pcells + 3) / 4;
    occ_mode = kOccGlobalBits;
    occ_smem_words = 0;
    if (smem_ok)
    {
        if (byte_words * 4 + other_smem <= 160 * 1024)
        {
            occ_mode = kOccSmemBytes;
            occ_smem_words = (uint32_t) byte_words;
        }
        else if (bit_words * 4 + other_smem <= 160 * 1024)
        {
            occ_mode = kOccSmemBits;
            occ_smem_words = (uint32_t) bit_words;
        }
    }
    if (occ_mode == kOccGlobalBits && d.scene.d_pcell_dist.get() && ctx->tune.occ_mode < 0)
        occ_mode = kOccGlobalDist; // too large for shared memory: distance map through L1
    const int m = ctx->tune.occ_mode;
    if (m == kOccGlobalBits) { occ_mode = kOccGlobalBits; occ_smem_words = 0; }
    if (m == kOccGlobalDist && d.scene.d_pcell_dist.get()) { occ_mode = kOccGlobalDist; occ_smem_words = 0; }
    if (m == kOccSmemBits && bit_words * 4 + other_smem <= 200 * 1024) { occ_mode = kOccSmemBits; occ_smem_words = (uint32_t) bit_words; }
    if (m == kOccSmemBytes && byte_words * 4 + other_smem <= 200 * 1024) { occ_mode = kOccSmemBytes; occ_smem_words = (uint32_t) byte_words; }
}

// Occupancy map: choose_occupancy_home, staged only for frames of >= 4 M rays (tiny frames skip the per-CTA staging).
// CTA size: one 1024-thread CTA per SM measured best on every config (32 warps share one staged occupancy map and
// pull neighbouring strips, which keeps the triangle records of that screen region in L1); small frames use
// smaller CTAs so that every SM gets work.
int choose_cta(const cuda_trace_ctx *ctx, const DeviceState& d, const cuda_trace_frame *f, uint64_t strips_here, TraceParams& p)
{
    int threads = 1024;
    const uint64_t rays = (uint64_t) f->width * f->height * f->spp;
    const size_t smp_bytes = sizeof(float2) * f->spp;
    while (threads > 64 && strips_here < (uint64_t) d.sm_count * (threads / 32))
        threads /= 2;
    choose_occupancy_home(ctx, d, ctx->occ_in_smem && rays >= (4u << 20) && threads == 1024, smp_bytes, p.occ_mode,
                          p.occ_smem_words);
    if (ctx->tune.threads)
        threads = ctx->tune.threads;
    // |det| <= |e1| |e2| |d| <= 3 extent^2: below 1e14 the reciprocal's fast path is always valid
    float extent = 0.0f;
    for (int k = 0; k < 3; k++)
        extent = std::max(extent, ctx->desc.aabb_max[k] - ctx->desc.aabb_min[k]);
    p.rcp_guard = (extent < 1.0e14f) ? 0u : 1u;
    return threads;
}

// Cost order from the previous frame (schedule.cu), valid only if that frame had the same layout and shard.
// Worth its ~1 % instrumentation cost when the frame is sharded or small (the tail of expensive strips is then a
// large part of the launch); RTM_COST_ORDER=0/1 forces it
int prepare_cost_order(cuda_trace_ctx *ctx, DeviceState& d, const cuda_trace_frame *f, TraceParams& p, bool use_pool)
{
    const FramePlan& pl = ctx->plan;
    const uint32_t shard_strips = p.shard_strips;
    p.fetch_order = nullptr;
    p.visit_cycles = nullptr;
    p.visit_total = nullptr;
    const bool want_order = (ctx->cost_order_forced >= 0 ? ctx->cost_order_forced != 0
                            : (p.shard_world > 1 || (uint64_t) f->width * f->height * f->spp < (64ull << 20))) &&
                            shard_strips <= kVisitStripMask && !use_pool; // (K7 balances by pooling, not by order)
    if (!want_order || shard_strips == 0)
    {
        d.order_valid = false;
        return 0;
    }
    if (d.order_pending)
    {
        CK(cudaStreamWaitEvent(d.stream, d.ev_order, 0)); // the order this frame follows / the buffers it reuses
        d.order_pending = false;
    }
    if (d.d_strip_cycles.size() < shard_strips)
    {
        // the order build behind the last frame may still use the buffers.  d_strip_cycles grows last, so that after
        // a failure half way it is still short and the next frame grows what is missing
        CK(cudaStreamSynchronize(d.order_stream));
        d.order_valid = false;
        CK(d.d_fetch_order.grow(strip_order_capacity(shard_strips, 4)));
        CK(d.d_visit_cycles.grow(strip_order_capacity(shard_strips, 4)));
        CK(d.d_order_scratch.grow(strip_order_scratch_words(shard_strips)));
        CK(d.d_cost_sum.grow(1));
        CK(d.d_visit_total.grow(1));
        CK(d.d_strip_cycles.grow(shard_strips));
    }
    const std::vector<uint64_t> sig = { pl.serial, p.shard_rank, p.shard_world, p.shard_chunk, shard_strips };
    if (d.order_valid && sig == d.order_signature)
        p.fetch_order = d.d_fetch_order.get();
    p.visit_total = d.d_visit_total.get();
    d.order_signature = sig;
    d.order_strips = shard_strips;
    p.visit_cycles = d.d_visit_cycles.get();
    CK(cudaMemsetAsync(d.d_visit_cycles.get(), 0, sizeof(uint32_t) * strip_order_capacity(shard_strips, pl.split_parts), d.stream));
    return 0;
}

// Everything device `i` of the context does for this frame
int launch_on_device(cuda_trace_ctx *ctx, uint32_t i, const cuda_trace_frame *f, const FrameKind& kind, bool use_bands, uint32_t seq)
{
    DeviceState& d = ctx->dev[i];
    const FramePlan& pl = ctx->plan;
    const uint32_t n_dev = (uint32_t) ctx->dev.size(), n_tiles = (uint32_t) pl.rects.size();
    CK(cudaSetDevice(d.ordinal));
    bool new_smp = false, new_tiles = false;
    CK(d.d_smp.grow(f->spp, &new_smp));
    if (new_smp || d.smp_valid_spp != f->spp)
    {
        launch_sample_table(d.d_smp.get(), f->spp, d.stream); // K2
        ctx->launches++;
        d.smp_valid_spp = f->spp;
    }
    CK(d.d_tile_rects.grow(std::max<uint32_t>(n_tiles + 1, 128), &new_tiles));
    CK(d.d_tile_prefix.grow(std::max<uint32_t>(n_tiles + 1, 128), &new_tiles));
    // the tile list usually repeats from frame to frame: upload it only when it changed (the plan owns the host
    // arrays, so the asynchronous copies need no synchronisation before returning)
    if (new_tiles || d.layout_serial != pl.serial)
    {
        d.layout_serial = 0;
        if (n_tiles)
            CK(cudaMemcpyAsync(d.d_tile_rects.get(), pl.rects.data(), sizeof(uint4) * n_tiles, cudaMemcpyHostToDevice, d.stream));
        CK(cudaMemcpyAsync(d.d_tile_prefix.get(), pl.prefix.data(), sizeof(uint32_t) * (n_tiles + 1), cudaMemcpyHostToDevice, d.stream));
        CK(cudaStreamSynchronize(d.stream)); // pageable source: consumed before the plan can be replaced
        d.layout_serial = pl.serial;
    }
    // strip counter + this GPU's per-band piece counts (the cancel word behind them is never cleared)
    CK(cudaMemsetAsync(d.d_strip_counter.get(), 0, (32 + kMaxBands) * sizeof(uint32_t), d.stream));
    if (ctx->counting)
        CK(cudaMemsetAsync(d.d_counters.get(), 0, sizeof(Counters), d.stream));

    TraceParams p;
    p.grid = grid_dev(ctx, d);
    p.pair_sbox = nullptr;
    fill_camera(ctx, f, kind, p);
    p.smp = d.d_smp.get();
    p.tile_rects = d.d_tile_rects.get();
    p.tile_strip_prefix = d.d_tile_prefix.get();
    p.n_tiles = n_tiles;
    p.strip_w = pl.strip_w;
    p.strip_h = pl.strip_h;
    p.split_parts = pl.split_parts;
    p.total_strips = (uint32_t) pl.total;
    // strips are interleaved first over the processes (shard), then over this context's devices
    p.shard_world = ctx->shard_world * n_dev;
    p.shard_rank = ctx->shard_rank * n_dev + i;
    p.shard_chunk = ctx->shard_chunk;
    p.strip_counter = d.d_strip_counter.get();
    p.cancel = d.d_cancel;
    p.cancel_seen = d.d_cancel_seen;
    p.frame_seq = seq;
    p.framebuffer = ctx->d_fb;
    p.band_done = use_bands ? band_counters(ctx) : nullptr;
    p.band_rows = ctx->band_rows;
    p.band_local = use_bands ? d.d_strip_counter.get() + 32 : nullptr; // own cache line
    std::memset(p.band_share, 0, sizeof(p.band_share));
    if (use_bands)
        std::memcpy(p.band_share, ctx->band_share[p.shard_rank].data(), sizeof(p.band_share));
    p.pool_walk_steps = 0;
    p.hit_tri = kind.keep_hits ? ctx->d_hit_tri.get() : nullptr;
    p.hit_t = kind.keep_hits ? ctx->d_hit_t.get() : nullptr;
    p.hit_u = kind.keep_hits ? ctx->d_hit_u.get() : nullptr;
    p.hit_v = kind.keep_hits ? ctx->d_hit_v.get() : nullptr;
    p.counters = d.d_counters.get();

    const uint64_t strips_here = (pl.total + p.shard_world - 1) / p.shard_world;
    const int threads = choose_cta(ctx, d, f, strips_here, p);
    {
        const uint64_t chunks_total = (pl.total + p.shard_chunk - 1) / p.shard_chunk;
        const uint64_t my_chunks = (chunks_total + p.shard_world - 1) / p.shard_world;
        p.shard_strips = (uint32_t) (my_chunks * p.shard_chunk); // (< 2^32: checked by the caller)
    }
    // K7 trace_pool (pool_trace.cu) does the traversal when rays are incoherent: grids with a distance map, i.e. too
    // large for a shared-memory occupancy map.  Primary rays of the perspective camera, Moeller-Trumbore, no work
    // counters; RTM_POOL=0/1 forces it off / on wherever it is supported
    // By default only where walking dominates -- fewer than one pair record per three padded cells: on the soup sweep
    // K7 wins at 640^3 and finer (0.25 pairs per cell and less) and loses at 512^3 and coarser (0.42 and more), where
    // most of the time goes into long triangle lists, which coherent lanes (K1) test with broadcast loads
    const uint64_t pcells_here = (uint64_t) (ctx->desc.dim[0] + 2) * (ctx->desc.dim[1] + 2) * (ctx->desc.dim[2] + 2);
    const bool pool_pays = ctx->tune.pool == 1 || (uint64_t) ctx->num_pairs * 3 < pcells_here;
    const bool use_pool = d.scene.d_pcell_dist.get() && ctx->tune.pool != 0 && pool_pays && !kind.alternates && !kind.count_inst &&
                          f->variant == kVariantMT && f->spp <= 32 && ctx->num_pairs > 0 &&
                          (uint64_t) f->width * f->height * f->spp < (1ull << 32);
    int rc = prepare_cost_order(ctx, d, f, p, use_pool);
    if (rc)
        return rc;

    // Moeller-Trumbore on origin-relative records when the per-camera pre-pass is negligible (a few M cell
    // references: < 0.1 ms) -- not for the instrumented (counting) kernels; RTM_REL_RECORDS=0 switches it off;
    // nor for small frames: measured +5..9 % on 33 M rays and more (4K and 1080p at 16 spp), -1 % on the 8 M rays
    // of 1080p / 4 spp, -10 % on 512^2 / 1 spp, which is launch- and cold-miss-bound (the records are 112 B, not 80)
    const bool rel_fits = ctx->desc.num_refs <= (4ull << 20) &&
                          ((uint64_t) f->width * f->height * f->spp >= (16ull << 20) || ctx->rel_records_forced);
    const uint32_t kvariant = kind.alternates ? (uint32_t) kVariantMTAlt + f->variant
                              : (f->variant == kVariantMT && !kind.count_inst && ctx->rel_records && rel_fits)
                                  ? (uint32_t) kVariantMTRel : f->variant;
    if (i == 0)
        ctx->t_launching_ms = ms_since(ctx->t_enter);
    CK(cudaEventRecord(d.ev_begin, d.stream));
    if (kvariant == kVariantMTRel && pl.total)
    {
        SceneArrays& s = d.scene;
        // records relative to this frame's camera position: rebuilt (inside the timed region) when it moved
        CK(s.d_pair_recs_rel.grow(std::max<uint64_t>(ctx->num_pairs, 1) * 7));
        if (!s.rel_valid || std::memcmp(s.rel_origin, p.cam.origin, sizeof(s.rel_origin)) != 0)
        {
            launch_origin_relative_pairs(s.d_pair_recs.get(), std::max<uint64_t>(ctx->num_pairs, 1), p.cam.origin, s.d_pair_recs_rel.get(), d.stream);
            ctx->launches++;
            std::memcpy(s.rel_origin, p.cam.origin, sizeof(s.rel_origin));
            s.rel_valid = true;
        }
        p.grid.pair_recs_rel = s.d_pair_recs_rel.get();
        if (ctx->screen_cull != 0)
        {
            // screen boxes for this frame's camera, rebuilt (inside the timed region) when any camera constant the
            // boxes depend on changed.  The cull pays where a fair share of the pairs projects small -- killeroo4k: 30 %
            // of its boxes are <= 32 pixels, 69 % of its pair iterations are skipped; the room of C4: none are, 6 % would
            // be skipped, and every kept iteration costs a box load and a vote -- so the boxes are counted once per
            // camera (a read-back, only then) and the cull is on when at least a fifth are small
            CK(s.d_pair_sbox.grow(std::max<uint64_t>(ctx->num_pairs, 1)));
            CK(s.d_sbox_small.grow(1));
            const CameraDev& c = p.cam;
            const bool same = s.sbox_valid && std::memcmp(s.sbox_cam.m, c.m, sizeof(c.m)) == 0 &&
                              std::memcmp(s.sbox_cam.origin, c.origin, sizeof(c.origin)) == 0 &&
                              std::memcmp(&s.sbox_cam.fov_xs, &c.fov_xs, sizeof(float)) == 0 &&
                              std::memcmp(&s.sbox_cam.aspect, &c.aspect, sizeof(float)) == 0 &&
                              std::memcmp(&s.sbox_cam.width_f, &c.width_f, sizeof(float)) == 0;
            if (!same)
            {
                launch_screen_boxes(s.d_pair_recs.get(), ctx->num_pairs, c, s.d_pair_sbox.get(), s.d_sbox_small.get(), d.stream);
                ctx->launches++;
                unsigned int small = 0;
                CK(cudaMemcpyAsync(&small, s.d_sbox_small.get(), sizeof(small), cudaMemcpyDeviceToHost, d.stream));
                CK(cudaStreamSynchronize(d.stream));
                s.sbox_cam = c;
                s.sbox_small = small;
                s.sbox_cull = (uint64_t) small * 5 >= ctx->num_pairs;
                s.sbox_valid = true;
            }
            if (ctx->screen_cull == 1 || s.sbox_cull)
                p.pair_sbox = s.d_pair_sbox.get();
        }
    }
    // K1's instance for this frame, now that the records and the cull are decided, and the grid its occupancy allows
    const TraceTilesKernel kernel = trace_tiles_instance(kvariant, kind.keep_hits, kind.count_inst, (int) p.occ_mode,
                                                         p.rcp_guard != 0, p.band_done != nullptr, p.pair_sbox != nullptr);
    const size_t smem_bytes = trace_tiles_smem_bytes(f->spp, p.occ_smem_words);
    const std::tuple<TraceTilesKernel, int, size_t> okey(kernel, threads, smem_bytes);
    if (okey != d.occupancy_key)
    {
        d.blocks_per_sm = std::max(1, trace_tiles_max_blocks_per_sm(kernel, threads, smem_bytes));
        d.occupancy_key = okey;
    }
    const uint64_t want = (strips_here + (threads / 32) - 1) / (threads / 32);
    const int blocks = (int) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) d.sm_count * d.blocks_per_sm, want));
    {
        // How many finished strips a warp collects before it publishes them to the band counters: the fence
        // costs ~1 us, but a held-back strip delays its band's read-back -- at most 1/16 of a warp's share
        // of the frame (8 strips for a whole 4K frame on one GPU, every strip for an eighth of it)
        const uint64_t warps = (uint64_t) blocks * (threads / 32);
        uint64_t hold = std::min<uint64_t>(8, std::max<uint64_t>(1, strips_here / std::max<uint64_t>(1, warps * 16)));
        if (ctx->tune.band_flush)
            hold = (uint64_t) ctx->tune.band_flush;
        p.band_flush_units = (uint32_t) hold * pl.split_parts;
    }
    if (pl.total && use_pool)
    {
        // hit records: the caller's (KEEP_HITS, device 0) or this device's own
        TraceParams pp = p;
        pp.pool_walk_steps = (uint32_t) ctx->tune.pool_steps;
        if (!kind.keep_hits)
        {
            const uint64_t need = (uint64_t) f->width * f->height * f->spp;
            CK(d.d_pool_tri.grow(need));
            CK(d.d_pool_t.grow(need));
            CK(d.d_pool_u.grow(need));
            CK(d.d_pool_v.grow(need));
            pp.hit_tri = d.d_pool_tri.get(); pp.hit_t = d.d_pool_t.get(); pp.hit_u = d.d_pool_u.get(); pp.hit_v = d.d_pool_v.get();
        }
        // K7: one CTA per SM at 1024 threads (64 registers), more of the smaller CTAs of small frames
        const int pool_blocks = (int) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) d.sm_count * std::max(1, 1024 / threads), want));
        launch_trace_pool(pp, pool_blocks, threads, d.stream);
        // K1 behind it: shading, in-order sample sum, resolve, band publication -- from the hit records
        pp.occ_mode = kOccGlobalBits;
        pp.occ_smem_words = 0;
        const TraceTilesKernel resolve = trace_tiles_instance(kVariantFromHits, false, false, kOccGlobalBits, pp.rcp_guard != 0,
                                                              pp.band_done != nullptr, false);
        if (d.resolve_threads != threads)
        {
            d.resolve_blocks_per_sm = std::max(1, trace_tiles_max_blocks_per_sm(resolve, threads, trace_tiles_smem_bytes(f->spp, 0)));
            d.resolve_threads = threads;
        }
        const int resolve_blocks = (int) std::max<uint64_t>(1, std::min<uint64_t>((uint64_t) d.sm_count * d.resolve_blocks_per_sm, want));
        launch_trace_tiles(resolve, pp, resolve_blocks, threads, d.stream);
        ctx->launches += 2;
    }
    else if (pl.total)
    {
        launch_trace_tiles(kernel, p, blocks, threads, d.stream);
        ctx->launches++;
    }
    if (i == 0)
        ctx->t_launched_ms = ms_since(ctx->t_enter);
    CK(cudaEventRecord(d.ev_end, d.stream));
    d.launched_seq = seq;
    d.frame_pending = true;
    d.order_followup = p.visit_cycles && pl.total;
    d.order_followup_used = p.fetch_order != nullptr;
    CK(cudaGetLastError());
    return 0;
}

// this frame's strip costs -> next frame's visiting order (own stream, behind the trace kernel; enqueued after the
// band copies so that it does not delay them)
int enqueue_order_followup(cuda_trace_ctx *ctx, DeviceState& d)
{
    if (!d.order_followup)
        return 0;
    d.order_followup = false;
    CK(cudaSetDevice(d.ordinal));
    CK(cudaEventRecord(d.ev_traced, d.stream));
    CK(cudaStreamWaitEvent(d.order_stream, d.ev_traced, 0));
    launch_build_strip_order(d.d_visit_cycles.get(), d.order_followup_used, d.d_strip_cycles.get(), d.order_strips, ctx->plan.split_parts,
                             d.d_cost_sum.get(), d.d_order_scratch.get(), d.d_visit_total.get(), d.d_fetch_order.get(), d.order_stream);
    CK(cudaEventRecord(d.ev_order, d.order_stream));
    d.order_pending = true;
    ctx->launches += 5;
    d.order_valid = true;
    CK(cudaGetLastError());
    return 0;
}

// Where a frame goes on the host: one W x H image (row 0 = y 0) or one buffer per tile (row-major within the tile)
struct HostDest
{
    uint32_t *frame = nullptr;
    uint32_t *const *tile = nullptr;
    uint32_t *staging = nullptr; // with `tile`: whole bands go here first (small frames), the caller scatters
};

// Copy stream of device 0, per-tile destination: tiles are grouped by the row band that completes them; per group
// wait for the bands up to that one, copy each tile (2-D) into its own buffer, record the group's event.
// `staging` (small frames: a 2-D copy costs ~7 us whatever its size, 108 of them would be most of the call): the
// bands are copied whole into one page-locked image instead and the caller scatters the tiles on the host.
int enqueue_tile_copies(cuda_trace_ctx *ctx, const cuda_trace_frame *f, uint32_t *const *tile_bgra, uint32_t *staging,
                        const uint32_t *expected)
{
    DeviceState& d0 = ctx->dev[0];
    const FramePlan& pl = ctx->plan;
    CK(cudaSetDevice(d0.ordinal));
    uint32_t *counters = band_counters(ctx);
    std::vector<std::vector<uint32_t>> by_band(ctx->n_bands);
    for (uint32_t i = 0; i < pl.rects.size(); i++)
    {
        const uint4& r = pl.rects[i];
        const bool empty = r.x == r.z || r.y == r.w;
        by_band[empty ? 0u : std::min(ctx->n_bands - 1, (r.w - 1) / ctx->band_rows)].push_back(i);
    }
    ctx->tile_groups.clear();
    uint32_t waited = 0; // bands [0, waited) have been waited for on the copy stream (and, staging: copied)
    for (uint32_t b = 0; b < ctx->n_bands; b++)
    {
        if (by_band[b].empty())
            continue;
        for (; waited <= b; waited++)
        {
            if (ctx->wait_value32(d0.copy_stream, (unsigned long long) (uintptr_t) (counters + waited), expected[waited],
                                  0u /* CU_STREAM_WAIT_VALUE_GEQ */) != 0)
                return fail(ctx, CUDA_TRACE_ERR_CUDA, "cuStreamWaitValue32 failed");
            if (staging)
            {
                const uint32_t y0 = waited * ctx->band_rows, y1 = std::min(f->height, y0 + ctx->band_rows);
                CK(cudaMemcpyAsync(staging + (size_t) y0 * f->width, ctx->d_fb + (size_t) y0 * f->width,
                                   (size_t) (y1 - y0) * f->width * sizeof(uint32_t), cudaMemcpyDeviceToHost, d0.copy_stream));
            }
        }
        if (!staging)
            for (uint32_t i : by_band[b])
            {
                const uint4& r = pl.rects[i];
                if (r.x == r.z || r.y == r.w)
                    continue;
                const size_t tw = r.z - r.x;
                CK(cudaMemcpy2DAsync(tile_bgra[i], tw * 4, ctx->d_fb + (size_t) r.y * f->width + r.x, (size_t) f->width * 4, tw * 4,
                                     r.w - r.y, cudaMemcpyDeviceToHost, d0.copy_stream));
            }
        const size_t g = ctx->tile_groups.size();
        if (ctx->tile_events.size() <= g)
        {
            cudaEvent_t ev;
            CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
            ctx->tile_events.push_back(ev);
        }
        CK(cudaEventRecord(ctx->tile_events[g], d0.copy_stream));
        ctx->tile_groups.push_back(std::move(by_band[b]));
    }
    ctx->copy_pending = true;
    return 0;
}

// Copy stream of device 0: wait for each row band's completion count, ship the band to the host buffer
int enqueue_band_copies(cuda_trace_ctx *ctx, const cuda_trace_frame *f, uint32_t *host_bgra, const uint32_t *expected)
{
    DeviceState& d0 = ctx->dev[0];
    CK(cudaSetDevice(d0.ordinal));
    uint32_t *counters = band_counters(ctx);
    for (uint32_t b = 0; b < ctx->n_bands; b++)
    {
        const uint32_t y0 = b * ctx->band_rows, y1 = std::min(f->height, y0 + ctx->band_rows);
        if (ctx->wait_value32(d0.copy_stream, (unsigned long long) (uintptr_t) (counters + b), expected[b],
                              0u /* CU_STREAM_WAIT_VALUE_GEQ */) != 0)
            return fail(ctx, CUDA_TRACE_ERR_CUDA, "cuStreamWaitValue32 failed");
        CK(cudaMemcpyAsync(host_bgra + (size_t) y0 * f->width, ctx->d_fb + (size_t) y0 * f->width,
                           (size_t) (y1 - y0) * f->width * sizeof(uint32_t), cudaMemcpyDeviceToHost, d0.copy_stream));
    }
    ctx->copy_pending = true;
    return 0;
}

} // namespace

static int tiles_async_impl(cuda_trace_ctx *ctx, const cuda_trace_frame *f, const cuda_trace_tile_rect *tiles,
                            uint32_t n_tiles, const HostDest& dst)
{
    if (!ctx || !f || (!tiles && n_tiles))
        return CUDA_TRACE_ERR_ARG;
    uint32_t *const host_bgra = dst.frame;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    FrameKind kind;
    int rc = check_frame_args(ctx, f, tiles, n_tiles, kind);
    if (rc)
        return rc;
    // from here until the frame has its number a cancel request is kept for it (cuda_trace_cancel)
    struct SettingUp
    {
        cuda_trace_ctx *ctx;
        explicit SettingUp(cuda_trace_ctx *c) : ctx(c)
        {
            std::lock_guard<std::mutex> lock(ctx->seq_mtx);
            ctx->setting_up = true;
            ctx->cancel_pending = false;
        }
        ~SettingUp()
        {
            std::lock_guard<std::mutex> lock(ctx->seq_mtx);
            ctx->setting_up = false;
        }
    } setting_up(ctx);
    rc = cuda_trace_sync(ctx); // one frame in flight per context
    if (rc && rc != CUDA_TRACE_ERR_CANCELLED)
        return rc;
    if ((rc = update_plan(ctx, f, tiles, n_tiles)))
        return rc;
    const FramePlan& pl = ctx->plan;
    const uint32_t n_dev = (uint32_t) ctx->dev.size();
    {
        const uint64_t world = (uint64_t) ctx->shard_world * n_dev;
        const uint64_t chunks_total = (pl.total + ctx->shard_chunk - 1) / ctx->shard_chunk;
        if ((chunks_total + world - 1) / world * ctx->shard_chunk >= (1ull << 32))
            return fail(ctx, CUDA_TRACE_ERR_ARG, "trace_tiles: too many strips");
    }
    if (ctx->band_dirty && (rc = resync_band_counters(ctx)))
        return rc;
    if ((rc = ensure_framebuffer(ctx, f->width, f->height)))
        return rc;
    if (kind.keep_hits)
    {
        if ((rc = ensure_hit_buffers(ctx, f)))
            return rc;
    }
    else
        ctx->hit_count = 0;
    if (n_dev > 1)
        CK(cudaStreamSynchronize(ctx->dev[0].stream)); // framebuffer (re)allocation visible to peers

    ctx->frame = *f;
    ctx->tiles.assign(tiles, tiles + n_tiles);
    ctx->frame_valid = true;

    // Overlapped read-back: row bands whose strips are all finished are copied to the host while the rest of the
    // frame is still being traced.  Needs the whole frame covered by the tile list (exactly: a partition) and, when
    // the frame is sharded over processes, every rank signalling (set_shard_signals).
    const bool bands_usable = ctx->overlap_d2h && ctx->wait_value32 && !ctx->fb_imported && pl.total > 0 &&
                              (ctx->shard_world == 1 || ctx->shard_signals);
    const bool can_overlap = (host_bgra && bands_usable && pl.covers_frame) || (dst.tile && bands_usable);
    const bool use_bands = ctx->shard_signals || can_overlap;
    ctx->tile_groups.clear();
    if (use_bands)
        plan_band_counts(ctx);

    // From here on the device counters move: should anything fail before every device's kernel is enqueued, the
    // totals are re-read from the device at the next call instead of being trusted
    uint32_t seq;
    bool start_cancelled;
    {
        std::lock_guard<std::mutex> lock(ctx->seq_mtx);
        seq = ++ctx->frame_seq;
        ctx->setting_up = false;
        start_cancelled = ctx->cancel_pending;
        ctx->cancel_pending = false;
        if (start_cancelled)
        {
            ctx->cancel_seq.store(seq);
            *(volatile uint32_t *) ctx->pinned_cancel_src.get() = seq;
        }
    }
    if (start_cancelled) // requested while this call was being set up: the kernels find the word already there
        for (DeviceState& d : ctx->dev)
        {
            CK(cudaSetDevice(d.ordinal));
            CK(cudaMemcpyAsync(d.d_cancel, ctx->pinned_cancel_src.get(), sizeof(uint32_t), cudaMemcpyHostToDevice, d.stream));
        }
    ctx->band_dirty = use_bands;
    ctx->t_prepared_ms = ms_since(ctx->t_enter);
    uint32_t expected[kMaxBands];
    for (int b = 0; b < kMaxBands; b++)
        expected[b] = ctx->band_expected[b] + (use_bands && (uint32_t) b < ctx->n_bands ? ctx->band_inc[b] : 0u); // monotone across frames (wrap-safe compare)
    // The copy stream is armed (a wait on each band counter + the band's copy) right behind the only kernel of a
    // one-GPU context, while that kernel starts.  With several devices in one process it is armed only after EVERY
    // device's kernel is enqueued: a device's set-up allocates, loads modules and synchronises its stream, any of which
    // may wait for all work queued in the process -- including a copy stream that waits for counters only that device's
    // kernel will bump.  (Armed between device 0 and device 1, a two-device context hung in its first frame.)
    for (uint32_t i = 0; i < n_dev; i++)
    {
        if ((rc = launch_on_device(ctx, i, f, kind, use_bands, seq)))
            return rc;
        if (i + 1 == n_dev && can_overlap &&
            (rc = dst.tile ? enqueue_tile_copies(ctx, f, dst.tile, dst.staging, expected) : enqueue_band_copies(ctx, f, host_bgra, expected)))
            return rc;
    }
    std::memcpy(ctx->band_expected, expected, sizeof(expected));
    ctx->band_dirty = false;
    for (DeviceState& d : ctx->dev)
        if ((rc = enqueue_order_followup(ctx, d)))
            return rc;
    return 0;
}

extern "C"
{

int cuda_trace_tiles_async(cuda_trace_ctx *ctx, const cuda_trace_frame *f, const cuda_trace_tile_rect *tiles,
                           uint32_t n_tiles)
{
    return tiles_async_impl(ctx, f, tiles, n_tiles, HostDest());
}

int cuda_trace_sync(cuda_trace_ctx *ctx)
{
    if (!ctx)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    bool any = false, cancelled = false;
    float ms_max = 0.0f;
    for (DeviceState& d : ctx->dev)
    {
        CK(cudaSetDevice(d.ordinal));
        CK(cudaStreamSynchronize(d.stream));
        if (ctx->marks_armed)
            ctx->t_traced_ms = ms_since(ctx->t_enter);
        if (d.frame_pending)
        {
            float ms = 0.0f;
            CK(cudaEventElapsedTime(&ms, d.ev_begin, d.ev_end));
            ms_max = std::max(ms_max, ms);
            cancelled = cancelled || *(volatile uint32_t *) d.h_cancel_seen.get() == d.launched_seq; // stored by the kernel itself
            d.frame_pending = false;
            any = true;
        }
    }
    if (ctx->copy_pending)
    {
        CK(cudaSetDevice(ctx->dev[0].ordinal));
        CK(cudaStreamSynchronize(ctx->dev[0].copy_stream));
        if (ctx->marks_armed)
            ctx->t_copied_ms = ms_since(ctx->t_enter);
        ctx->copy_pending = false;
    }
    if (any)
        ctx->last_kernel_ms = ms_max;
    if (cancelled)
        return fail(ctx, CUDA_TRACE_ERR_CANCELLED, "frame cancelled");
    return 0;
}

// Not serialised with the other entry points: it is meant to be called while cuda_trace_tiles / cuda_trace_sync
// block in another thread.  The cancel word names the frame it is meant for (its sequence number), is never
// cleared, and the kernel compares it with its own number: a request that lands late cannot stop a later frame, and
// one that arrives while the frame is still being set up on the host is not lost.
int cuda_trace_cancel(cuda_trace_ctx *ctx)
{
    if (!ctx)
        return CUDA_TRACE_ERR_ARG;
    uint32_t seq;
    {
        std::lock_guard<std::mutex> lock(ctx->seq_mtx);
        if (ctx->setting_up)
        {
            ctx->cancel_pending = true; // the frame being set up starts cancelled
            return 0;
        }
        seq = ctx->frame_seq.load();
        if (seq == 0)
            return 0; // nothing was ever launched
        ctx->cancel_seq.store(seq);
        *(volatile uint32_t *) ctx->pinned_cancel_src.get() = seq;
    }
    for (DeviceState& d : ctx->dev)
    {
        if (cudaSetDevice(d.ordinal) != cudaSuccess)
            return CUDA_TRACE_ERR_CUDA;
        if (cudaMemcpyAsync(d.d_cancel, ctx->pinned_cancel_src.get(), sizeof(uint32_t), cudaMemcpyHostToDevice,
                            d.side_stream) != cudaSuccess)
            return CUDA_TRACE_ERR_CUDA;
    }
    return 0;
}

int cuda_trace_read_framebuffer(cuda_trace_ctx *ctx, uint32_t *host_bgra)
{
    if (!ctx || !host_bgra)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (!ctx->d_fb || !ctx->frame_valid)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "read_framebuffer: no frame rendered");
    DeviceState& d0 = ctx->dev[0];
    CK(cudaSetDevice(d0.ordinal));
    const uint32_t w = ctx->fb_w, h = ctx->fb_h;
    const size_t bytes = (size_t) w * h * sizeof(uint32_t);

    // the tile list partitions the whole frame? then one copy, else one 2-D copy per tile
    if (ctx->plan.covers_frame && ctx->plan.width == w && ctx->plan.height == h)
        CK(cudaMemcpyAsync(host_bgra, ctx->d_fb, bytes, cudaMemcpyDeviceToHost, d0.stream));
    else
        for (const auto& t : ctx->tiles)
        {
            if (t.x1 == t.x0 || t.y1 == t.y0)
                continue;
            const size_t o = (size_t) t.y0 * w + t.x0;
            CK(cudaMemcpy2DAsync(host_bgra + o, (size_t) w * 4, ctx->d_fb + o, (size_t) w * 4,
                                 (size_t) (t.x1 - t.x0) * 4, t.y1 - t.y0, cudaMemcpyDeviceToHost, d0.stream));
        }
    CK(cudaStreamSynchronize(d0.stream));
    return 0;
}

int cuda_trace_tiles(cuda_trace_ctx *ctx, const cuda_trace_frame *frame, const cuda_trace_tile_rect *tiles,
                     uint32_t n_tiles, uint32_t *host_bgra)
{
    if (!ctx)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    ctx->t_enter = std::chrono::steady_clock::now();
    HostDest dst;
    dst.frame = host_bgra;
    int rc = tiles_async_impl(ctx, frame, tiles, n_tiles, dst);
    if (rc)
        return rc;
    ctx->t_submitted_ms = ms_since(ctx->t_enter);
    const bool overlapped = ctx->copy_pending; // the bands are already on their way to host_bgra
    ctx->marks_armed = true;
    rc = cuda_trace_sync(ctx);
    ctx->marks_armed = false;
    if (rc)
        return rc;
    if (host_bgra && !overlapped)
        rc = cuda_trace_read_framebuffer(ctx, host_bgra);
    ctx->t_return_ms = ms_since(ctx->t_enter);
    return rc;
}

int cuda_trace_tiles_into(cuda_trace_ctx *ctx, const cuda_trace_frame *frame, const cuda_trace_tile_rect *tiles,
                          uint32_t n_tiles, uint32_t *const *tile_bgra, cuda_trace_tiles_done_fn done, void *user)
{
    if (!ctx || (n_tiles && !tile_bgra))
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    for (uint32_t i = 0; i < n_tiles; i++)
        if (!tile_bgra[i])
            return fail(ctx, CUDA_TRACE_ERR_ARG, "tiles_into: null tile buffer");
    ctx->t_enter = std::chrono::steady_clock::now();
    HostDest dst;
    dst.tile = tile_bgra;
    // frames of up to 4 MB go through one page-locked image (a few large copies) and are scattered into the tile
    // buffers here, group by group; larger ones are copied tile by tile straight from the device (measured on the
    // class route: 512 x 512 0.52 ms tile by tile -> 0.18 ms through the image; 1080p 1.15 ms either way)
    if (frame && frame->width && frame->height && (uint64_t) frame->width * frame->height <= (1u << 20))
    {
        CK(ctx->staging.grow((size_t) frame->width * frame->height));
        dst.staging = ctx->staging.get();
    }
    int rc = tiles_async_impl(ctx, frame, tiles, n_tiles, dst);
    if (rc)
        return rc;
    ctx->t_submitted_ms = ms_since(ctx->t_enter);
    const bool progressive = ctx->copy_pending;
    if (progressive)
    {
        // tiles become available in groups, top of the frame first, while the rest is still being traced
        CK(cudaSetDevice(ctx->dev[0].ordinal));
        for (size_t g = 0; g < ctx->tile_groups.size(); g++)
        {
            CK(cudaEventSynchronize(ctx->tile_events[g]));
            // (once a cancel has been requested for this frame its remaining bands complete without being traced:
            // those tiles are not reported -- the call returns CUDA_TRACE_ERR_CANCELLED below)
            if (ctx->tile_groups[g].empty() || ctx->cancel_seq.load() == ctx->dev[0].launched_seq)
                continue;
            if (dst.staging)
                for (uint32_t i : ctx->tile_groups[g])
                {
                    const cuda_trace_tile_rect& t = tiles[i];
                    const size_t tw = t.x1 - t.x0;
                    for (uint32_t y = t.y0; y < t.y1 && tw; y++)
                        std::memcpy(tile_bgra[i] + (size_t) (y - t.y0) * tw, dst.staging + (size_t) y * frame->width + t.x0, tw * 4);
                }
            if (done)
                done(ctx->tile_groups[g].data(), (uint32_t) ctx->tile_groups[g].size(), user);
        }
    }
    ctx->marks_armed = true;
    rc = cuda_trace_sync(ctx);
    ctx->marks_armed = false;
    if (rc)
        return rc;
    if (!progressive)
    {
        // no band machinery for this context (imported framebuffer, unsignalled shard, ...): copy after the frame
        DeviceState& d0 = ctx->dev[0];
        CK(cudaSetDevice(d0.ordinal));
        std::vector<uint32_t> all;
        for (uint32_t i = 0; i < n_tiles; i++)
        {
            const cuda_trace_tile_rect& t = tiles[i];
            all.push_back(i);
            if (t.x1 == t.x0 || t.y1 == t.y0)
                continue;
            const size_t tw = t.x1 - t.x0;
            CK(cudaMemcpy2DAsync(tile_bgra[i], tw * 4, ctx->d_fb + (size_t) t.y0 * frame->width + t.x0, (size_t) frame->width * 4,
                                 tw * 4, t.y1 - t.y0, cudaMemcpyDeviceToHost, d0.stream));
        }
        CK(cudaStreamSynchronize(d0.stream));
        if (done && n_tiles)
            done(all.data(), n_tiles, user);
    }
    ctx->t_return_ms = ms_since(ctx->t_enter);
    return 0;
}

int cuda_trace_last_call_timing(cuda_trace_ctx *ctx, double ms[7])
{
    if (!ctx || !ms)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    ms[0] = ctx->t_submitted_ms; ms[1] = ctx->t_traced_ms; ms[2] = ctx->t_copied_ms; ms[3] = ctx->t_return_ms;
    ms[4] = ctx->t_prepared_ms; ms[5] = ctx->t_launching_ms; ms[6] = ctx->t_launched_ms;
    return 0;
}

int cuda_trace_last_kernel_ms(cuda_trace_ctx *ctx, float *ms)
{
    if (!ctx || !ms)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    int rc = cuda_trace_sync(ctx);
    if (rc)
        return rc;
    *ms = ctx->last_kernel_ms;
    return 0;
}

int cuda_trace_download_hits(cuda_trace_ctx *ctx, uint32_t *tri_idx, float *t, float *u, float *v)
{
    if (!ctx)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    int rc = cuda_trace_sync(ctx);
    if (rc)
        return rc;
    if (ctx->hit_count == 0)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "download_hits: last frame was not rendered with CUDA_TRACE_FLAG_KEEP_HITS");
    CK(cudaSetDevice(ctx->dev[0].ordinal));
    const size_t bytes = ctx->hit_count * 4;
    if (tri_idx) CK(cudaMemcpy(tri_idx, ctx->d_hit_tri.get(), bytes, cudaMemcpyDeviceToHost));
    if (t) CK(cudaMemcpy(t, ctx->d_hit_t.get(), bytes, cudaMemcpyDeviceToHost));
    if (u) CK(cudaMemcpy(u, ctx->d_hit_u.get(), bytes, cudaMemcpyDeviceToHost));
    if (v) CK(cudaMemcpy(v, ctx->d_hit_v.get(), bytes, cudaMemcpyDeviceToHost));
    return 0;
}

// Enqueue a checked query batch (all pointers device memory of d) on stream s
static void launch_query(cuda_trace_ctx *ctx, const DeviceState& d, const cuda_trace_ray_batch& b, cudaStream_t s)
{
    const bool occlusion = b.kind == CUDA_TRACE_QUERY_OCCLUSION;
    RayQueryParams p;
    p.grid = grid_dev(ctx, d);
    p.grid.pair_recs_rel = nullptr; // rewritten by frames per camera: never read by queries
    p.n = b.n;
    p.origins = b.origins;
    p.dirs = b.dirs;
    p.t_max = b.t_max;
    p.t_max_all = b.t_max_all;
    p.tri = occlusion ? nullptr : b.tri_idx;
    p.t = occlusion ? nullptr : b.t;
    p.u = occlusion ? nullptr : b.u;
    p.v = occlusion ? nullptr : b.v;
    p.occluded = occlusion ? b.occluded : nullptr;
    // no sample table: the shared-memory budget is the map alone
    choose_occupancy_home(ctx, d, ctx->occ_in_smem, 0, p.occ_mode, p.occ_smem_words);
    const auto ordinary = [](float x) { return std::fabs(x) >= 0x1p-20f && std::fabs(x) <= 0x1p20f; };
    p.fast_math = (ctx->fast_math && ordinary(ctx->desc.cell_wdh)) ? 1u : 0u;
    const float one[2] = { 1.0f, 1.0f }, minus_one[2] = { -1.0f, -1.0f };
    std::memcpy(&p.pk_one, one, sizeof(p.pk_one));
    std::memcpy(&p.pk_minus_one, minus_one, sizeof(p.pk_minus_one));
    // t_max == +inf for all rays is Grid::Intersect itself: the unbounded instantiation (K1's work per ray)
    const bool bounded = b.t_max != nullptr || !(b.t_max_all == INFINITY);
    // persistent CTAs, one per SM (the map is staged once per CTA), fewer for small batches
    const int threads = ray_query_threads();
    const uint64_t ctas = (b.n + threads - 1) / threads;
    const int blocks = (int) std::min<uint64_t>(ctas, (uint64_t) d.sm_count);
    launch_ray_query(p, b.variant, occlusion, bounded, blocks, s);
}

static int intersect_rays_impl(cuda_trace_ctx *ctx, uint32_t n, const float *origins, const float *dirs, uint32_t variant,
                               bool brute_force, uint32_t *tri_idx, float *t, float *u, float *v)
{
    const bool mailbox = (variant & CUDA_TRACE_VARIANT_MAILBOX) != 0;
    variant &= ~CUDA_TRACE_VARIANT_MAILBOX;
    if (!ctx || (n && (!origins || !dirs || !tri_idx || !t || !u || !v)) || variant > 1 || (mailbox && brute_force))
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (!ctx->have_scene)
        return fail(ctx, CUDA_TRACE_ERR_NO_SCENE, "intersect_rays: upload a scene first");
    if (n == 0)
        return 0;
    DeviceState& d = ctx->dev[0];
    CK(cudaSetDevice(d.ordinal));
    DeviceArray<float> d_o, d_d, d_t, d_u, d_v;
    DeviceArray<uint32_t> d_i;
    DeviceArray<unsigned long long> d_stats;
    StreamDrain drain(d.stream);
    CK(d_o.alloc((size_t) n * 3));
    CK(d_d.alloc((size_t) n * 3));
    CK(d_t.alloc(n));
    CK(d_u.alloc(n));
    CK(d_v.alloc(n));
    CK(d_i.alloc(n));
    CK(cudaMemcpyAsync(d_o.get(), origins, (size_t) n * 12, cudaMemcpyHostToDevice, d.stream));
    CK(cudaMemcpyAsync(d_d.get(), dirs, (size_t) n * 12, cudaMemcpyHostToDevice, d.stream));
    RayBatchParams p;
    p.grid = grid_dev(ctx, d);
    p.n = n; p.origins = d_o.get(); p.dirs = d_d.get(); p.tri = d_i.get(); p.t = d_t.get(); p.u = d_u.get(); p.v = d_v.get();
    p.mailbox_stats = nullptr;
    if (mailbox)
    {
        CK(d_stats.alloc(2));
        CK(cudaMemsetAsync(d_stats.get(), 0, 2 * sizeof(unsigned long long), d.stream));
        p.mailbox_stats = d_stats.get();
    }
    if (brute_force)
        launch_brute_force(d.scene.d_vtx.get(), d.scene.d_tri.get(), ctx->num_tri, p, d.stream);
    else if (mailbox)
        launch_intersect_rays(p, variant, d.stream);
    else
    {
        // the warp-cooperative query kernel: the same bits, faster on every workload (profiles/r03_ray_query.txt)
        cuda_trace_ray_batch q = {};
        q.n = n; q.kind = CUDA_TRACE_QUERY_CLOSEST; q.variant = variant; q.t_max_all = INFINITY;
        q.origins = p.origins; q.dirs = p.dirs; q.tri_idx = p.tri; q.t = p.t; q.u = p.u; q.v = p.v;
        launch_query(ctx, d, q, d.stream);
    }
    ctx->launches++;
    CK(cudaGetLastError());
    if (mailbox)
    {
        CK(cudaMemcpyAsync(ctx->mailbox_stats, d_stats.get(), sizeof(ctx->mailbox_stats), cudaMemcpyDeviceToHost, d.stream));
        CK(cudaStreamSynchronize(d.stream));
    }
    CK(cudaMemcpyAsync(tri_idx, p.tri, (size_t) n * 4, cudaMemcpyDeviceToHost, d.stream));
    CK(cudaMemcpyAsync(t, p.t, (size_t) n * 4, cudaMemcpyDeviceToHost, d.stream));
    CK(cudaMemcpyAsync(u, p.u, (size_t) n * 4, cudaMemcpyDeviceToHost, d.stream));
    CK(cudaMemcpyAsync(v, p.v, (size_t) n * 4, cudaMemcpyDeviceToHost, d.stream));
    CK(drain.sync());
    return 0;
}

int cuda_trace_intersect_rays(cuda_trace_ctx *ctx, uint32_t n, const float *origins, const float *dirs,
                              uint32_t variant, uint32_t *tri_idx, float *t, float *u, float *v)
{
    return intersect_rays_impl(ctx, n, origins, dirs, variant, false, tri_idx, t, u, v);
}

int cuda_trace_mailbox_stats(cuda_trace_ctx *ctx, uint64_t *tests, uint64_t *reused)
{
    if (!ctx || !tests || !reused)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    *tests = ctx->mailbox_stats[0];
    *reused = ctx->mailbox_stats[1];
    return 0;
}

int cuda_trace_intersect_rays_brute_force(cuda_trace_ctx *ctx, uint32_t n, const float *origins, const float *dirs,
                                          uint32_t *tri_idx, float *t, float *u, float *v)
{
    return intersect_rays_impl(ctx, n, origins, dirs, 0, true, tri_idx, t, u, v);
}

int cuda_trace_query_rays(cuda_trace_ctx *ctx, const cuda_trace_ray_batch *b, void *stream)
{
    if (!ctx)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (!b)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "query_rays: batch is NULL");
    if (b->kind != CUDA_TRACE_QUERY_CLOSEST && b->kind != CUDA_TRACE_QUERY_OCCLUSION)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "query_rays: kind must be CUDA_TRACE_QUERY_CLOSEST or _OCCLUSION");
    if (b->variant & CUDA_TRACE_VARIANT_MAILBOX)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "query_rays: mailboxing is a mode of cuda_trace_intersect_rays only");
    if (b->variant != CUDA_TRACE_VARIANT_MT && b->variant != CUDA_TRACE_VARIANT_BARY)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "query_rays: variant must be CUDA_TRACE_VARIANT_MT or _BARY");
    const bool occlusion = b->kind == CUDA_TRACE_QUERY_OCCLUSION;
    if (b->n && (!b->origins || !b->dirs))
        return fail(ctx, CUDA_TRACE_ERR_ARG, "query_rays: origins and dirs are required");
    if (b->n && (occlusion ? !b->occluded : !b->tri_idx))
        return fail(ctx, CUDA_TRACE_ERR_ARG, occlusion ? "query_rays: an occlusion query needs `occluded`"
                                                       : "query_rays: a closest-hit query needs `tri_idx`");
    if (!ctx->have_scene)
        return fail(ctx, CUDA_TRACE_ERR_NO_SCENE, "query_rays: upload a scene first");
    if (b->n == 0)
        return 0;
    DeviceState& d = ctx->dev[0];
    CK(cudaSetDevice(d.ordinal));
    // every buffer must be device (or managed) memory of device 0: nothing is staged through the host
    const void *ptrs[8] = { b->origins, b->dirs, b->t_max };
    const char *names[8] = { "origins", "dirs", "t_max" };
    int n_ptrs = 3;
    if (occlusion)
    {
        ptrs[n_ptrs] = b->occluded; names[n_ptrs++] = "occluded";
    }
    else
    {
        ptrs[n_ptrs] = b->tri_idx; names[n_ptrs++] = "tri_idx";
        ptrs[n_ptrs] = b->t; names[n_ptrs++] = "t";
        ptrs[n_ptrs] = b->u; names[n_ptrs++] = "u";
        ptrs[n_ptrs] = b->v; names[n_ptrs++] = "v";
    }
    for (int k = 0; k < n_ptrs; k++)
    {
        if (!ptrs[k])
            continue; // optional and absent
        cudaPointerAttributes a;
        const cudaError_t e = cudaPointerGetAttributes(&a, ptrs[k]);
        if (e != cudaSuccess)
            cudaGetLastError(); // not sticky: clear it so that the next call does not report it
        if (e != cudaSuccess || (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) ||
            a.device != d.ordinal)
            return fail(ctx, CUDA_TRACE_ERR_ARG, std::string("query_rays: ") + names[k] +
                                                     " is not device memory of the context's device " +
                                                     std::to_string(d.ordinal));
    }
    cudaStream_t s = stream ? (cudaStream_t) stream : d.stream;
    launch_query(ctx, d, *b, s);
    ctx->launches++;
    CK(cudaGetLastError());
    // remember the stream so that freeing the scene waits for this query
    cudaEvent_t ev = nullptr;
    for (auto& se : ctx->query_events)
        if (se.first == s)
            ev = se.second;
    if (!ev)
    {
        CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        ctx->query_events.emplace_back(s, ev);
    }
    CK(cudaEventRecord(ev, s));
    return 0;
}

int cuda_trace_ray_march(cuda_trace_ctx *ctx, uint32_t n, const float *origins, const float *dirs, uint32_t *hit, float *t)
{
    if (!ctx || (n && (!origins || !dirs || !hit || !t)))
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (!ctx->have_scene)
        return fail(ctx, CUDA_TRACE_ERR_NO_SCENE, "ray_march: upload a scene first");
    if (n == 0)
        return 0;
    DeviceState& d = ctx->dev[0];
    CK(cudaSetDevice(d.ordinal));
    DeviceArray<float> d_o, d_d, d_t;
    DeviceArray<uint32_t> d_h;
    StreamDrain drain(d.stream);
    CK(d_o.alloc((size_t) n * 3)); CK(d_d.alloc((size_t) n * 3));
    CK(d_t.alloc(n)); CK(d_h.alloc(n));
    CK(cudaMemcpyAsync(d_o.get(), origins, (size_t) n * 12, cudaMemcpyHostToDevice, d.stream));
    CK(cudaMemcpyAsync(d_d.get(), dirs, (size_t) n * 12, cudaMemcpyHostToDevice, d.stream));
    launch_ray_march(d.scene.d_vtx.get(), d.scene.d_tri.get(), ctx->num_tri, n, d_o.get(), d_d.get(), d_h.get(), d_t.get(), d.stream);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(hit, d_h.get(), (size_t) n * 4, cudaMemcpyDeviceToHost, d.stream));
    CK(cudaMemcpyAsync(t, d_t.get(), (size_t) n * 4, cudaMemcpyDeviceToHost, d.stream));
    CK(drain.sync());
    return 0;
}

int cuda_trace_sample_table(cuda_trace_ctx *ctx, uint32_t spp, float *xy)
{
    if (!ctx || !xy || spp == 0)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    DeviceState& d = ctx->dev[0];
    CK(cudaSetDevice(d.ordinal));
    DeviceArray<float2> d_smp;
    StreamDrain drain(d.stream);
    CK(d_smp.alloc(spp));
    launch_sample_table(d_smp.get(), spp, d.stream);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(xy, d_smp.get(), sizeof(float2) * spp, cudaMemcpyDeviceToHost, d.stream));
    CK(drain.sync());
    return 0;
}

void *cuda_trace_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess)
    {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}

void cuda_trace_host_free(void *p)
{
    if (p)
        cudaFreeHost(p);
}

int cuda_trace_qmc_sequence(cuda_trace_ctx *ctx, uint32_t kind, uint32_t scramble, const uint32_t *perm,
                            uint32_t perm_primes, uint32_t n_begin, uint32_t count, uint32_t dim_begin,
                            uint32_t dim_count, uint32_t num_smp, uint32_t bits, double *out)
{
    if (!ctx || (!out && count && dim_count) || kind > 6 || scramble > 4)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    const bool table_kind = kind <= 3;
    if (table_kind && ((uint64_t) dim_begin + dim_count > (uint64_t) kQmcPrimes))
        return fail(ctx, CUDA_TRACE_ERR_ARG, "qmc_sequence: dimension beyond the 1000-prime table");
    if ((kind == 1 || kind == 3) && num_smp == 0)
        return fail(ctx, CUDA_TRACE_ERR_ARG, "qmc_sequence: Hammersley needs num_smp > 0");
    const bool caller_table = kind <= 1 && (scramble == kQmcScrambleBraatenWeller || scramble == kQmcScrambleCustom);
    if (caller_table && (!perm || perm_primes == 0 || perm_primes > (uint32_t) kQmcPrimes))
        return fail(ctx, CUDA_TRACE_ERR_ARG, "qmc_sequence: this scramble needs the caller's permutation tables");
    if ((uint64_t) count * dim_count == 0)
        return 0;
    DeviceState& d = ctx->dev[0];
    CK(cudaSetDevice(d.ordinal));
    if (!ctx->qmc_ready)
    {
        CK(qmc_upload_primes());
        ctx->qmc_ready = true;
    }

    // permutation tables: offsets = running sum of the primes
    const std::vector<uint32_t> primes = qmc_primes();
    std::vector<uint32_t> table, offset;
    uint32_t n_primes = 0;
    if (kind <= 1 && scramble != kQmcScrambleNone)
    {
        n_primes = caller_table ? perm_primes : 128u; // FAURE_TBL_SIZE = REVERSE_TBL_SIZE = 128 (sampling.h:52,67)
        offset.resize(n_primes + 1, 0);
        for (uint32_t i = 0; i < n_primes; i++)
            offset[i + 1] = offset[i] + primes[i];
        if (caller_table)
        {
            table.assign(perm, perm + offset[n_primes]);
            for (uint32_t i = 0; i < n_primes; i++)
                for (uint32_t k = offset[i]; k < offset[i + 1]; k++)
                    if (table[k] >= primes[i]) // each table permutes the digits 0 .. prime-1
                        return fail(ctx, CUDA_TRACE_ERR_ARG, "qmc_sequence: permutation entry out of range");
        }
        else if (scramble == kQmcScrambleFaure)
            for (uint32_t i = 0; i < n_primes; i++)
            {
                const std::vector<uint32_t> f = qmc_faure_permutation(primes[i]);
                table.insert(table.end(), f.begin(), f.end());
            }
        else
            table.assign(1, 0u); // reverse is a formula, the table is not read
    }
    DeviceArray<uint32_t> d_table, d_offset;
    DeviceArray<double> d_out;
    StreamDrain drain(d.stream);
    const size_t total = (size_t) count * dim_count;
    if (!table.empty())
    {
        CK(d_table.alloc(table.size()));
        CK(d_offset.alloc(offset.size()));
        CK(cudaMemcpyAsync(d_table.get(), table.data(), table.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, d.stream));
        CK(cudaMemcpyAsync(d_offset.get(), offset.data(), offset.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, d.stream));
    }
    CK(d_out.alloc(total));
    launch_qmc_sequence(kind, scramble, n_begin, count, dim_begin, dim_count, num_smp, bits, d_table.get(), d_offset.get(),
                        n_primes, d_out.get(), d.stream);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d_out.get(), total * sizeof(double), cudaMemcpyDeviceToHost, d.stream));
    CK(drain.sync());
    return 0;
}

int cuda_trace_qmc_cranley_patterson(cuda_trace_ctx *ctx, const double *x, double e, uint32_t count, double *out)
{
    if (!ctx || (count && (!x || !out)))
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    if (count == 0)
        return 0;
    DeviceState& d = ctx->dev[0];
    CK(cudaSetDevice(d.ordinal));
    DeviceArray<double> d_x, d_o;
    StreamDrain drain(d.stream);
    CK(d_x.alloc(count));
    CK(d_o.alloc(count));
    CK(cudaMemcpyAsync(d_x.get(), x, count * sizeof(double), cudaMemcpyHostToDevice, d.stream));
    launch_cranley_patterson(d_x.get(), e, count, d_o.get(), d.stream);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d_o.get(), count * sizeof(double), cudaMemcpyDeviceToHost, d.stream));
    CK(drain.sync());
    return 0;
}

int cuda_trace_get_counters(cuda_trace_ctx *ctx, cuda_trace_counters *out)
{
    if (!ctx || !out)
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    int rc = cuda_trace_sync(ctx);
    if (rc)
        return rc;
    std::memset(out, 0, sizeof(*out));
    for (DeviceState& d : ctx->dev)
    {
        Counters c;
        CK(cudaSetDevice(d.ordinal));
        CK(cudaMemcpy(&c, d.d_counters.get(), sizeof(c), cudaMemcpyDeviceToHost));
        out->rays += c.rays; out->cells += c.cells; out->tri_tests += c.tri_tests; out->hits += c.hits;
    }
    return 0;
}

int cuda_trace_band_shares(uint32_t width, uint32_t height, uint32_t spp, const cuda_trace_tile_rect *tiles, uint32_t n_tiles,
                           uint32_t world, uint32_t chunk, uint32_t *shares, uint32_t *gpus_in_band, uint32_t *band_rows,
                           uint32_t *n_bands, uint32_t *pieces_per_strip)
{
    if (!tiles || !n_tiles || !world || !chunk || !shares || !gpus_in_band || !band_rows || !n_bands || !pieces_per_strip ||
        !width || !height || !spp)
        return CUDA_TRACE_ERR_ARG;
    uint32_t strip_w, strip_h;
    strip_size_for_spp(spp, (uint64_t) width * height * spp, strip_w, strip_h);
    *pieces_per_strip = strip_split_parts(strip_w, strip_h, spp);
    std::vector<uint4> rects(n_tiles);
    std::vector<uint32_t> prefix(n_tiles + 1, 0);
    uint64_t total = 0;
    for (uint32_t i = 0; i < n_tiles; i++)
    {
        const cuda_trace_tile_rect& t = tiles[i];
        if (t.x0 > t.x1 || t.y0 > t.y1 || t.x1 > width || t.y1 > height)
            return CUDA_TRACE_ERR_ARG;
        rects[i] = make_uint4(t.x0, t.y0, t.x1, t.y1);
        prefix[i] = (uint32_t) total;
        total += (uint64_t) ((t.x1 - t.x0 + strip_w - 1) / strip_w) * ((t.y1 - t.y0 + strip_h - 1) / strip_h);
    }
    prefix[n_tiles] = (uint32_t) total;
    band_layout(width, height, strip_h, *band_rows, *n_bands);
    std::vector<std::array<uint32_t, kMaxBands>> share;
    band_shares(rects, prefix, strip_w, strip_h, *band_rows, *pieces_per_strip, chunk, world, share, gpus_in_band);
    for (uint32_t q = 0; q < world; q++)
        std::memcpy(shares + (size_t) q * kMaxBands, share[q].data(), sizeof(uint32_t) * kMaxBands);
    return 0;
}

int cuda_trace_download_strip_cycles(cuda_trace_ctx *ctx, uint32_t *cycles, uint64_t capacity, uint64_t *count)
{
    if (!ctx || !count || (capacity && !cycles))
        return CUDA_TRACE_ERR_ARG;
    std::lock_guard<std::recursive_mutex> guard(ctx->api_mtx);
    int rc = cuda_trace_sync(ctx);
    if (rc)
        return rc;
    DeviceState& d = ctx->dev[0];
    CK(cudaSetDevice(d.ordinal));
    CK(cudaStreamSynchronize(d.order_stream));
    *count = d.order_valid ? d.order_strips : 0;
    const uint64_t n = std::min<uint64_t>(*count, capacity);
    if (n)
    {
        CK(cudaSetDevice(d.ordinal));
        CK(cudaMemcpy(cycles, d.d_strip_cycles.get(), n * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    }
    return 0;
}

} // extern "C"
