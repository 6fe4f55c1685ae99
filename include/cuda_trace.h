/* cuda_trace.h -- C ABI of the B200 (sm_100a) tile tracer.
 *
 * This is the drop-in boundary for the reference's per-tile tracing hot path: everything that
 * `Framebuffer::WorkerThread` -> `virtual RenderTile(Tile&)` -> `Renderer::RenderTile`
 * (reference framebuffer.cpp:59-92, framebuffer.h:72-73, renderer.cpp:43-136) does on host
 * threads is done by these calls on the GPU(s).  Plain C: opaque context, plain pointers and
 * sizes, no C++/torch types, no exceptions.  Every function returns 0 on success and a non-zero
 * cuda_trace_status otherwise; cuda_trace_last_error() then describes the failure.  There is no
 * CPU fallback: without a usable CUDA device cuda_trace_init() fails.
 *
 * Ownership: the caller owns every host buffer it passes; the context owns all device memory.
 * One context must not be used from two threads at once; distinct contexts are independent.
 *
 * Which reference interface each entry point replaces is stated at its declaration.
 */
#ifndef CUDA_TRACE_H
#define CUDA_TRACE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cuda_trace_ctx cuda_trace_ctx;

typedef enum cuda_trace_status
{
    CUDA_TRACE_OK = 0,
    CUDA_TRACE_ERR_ARG = 1,       /* bad argument / call order                   */
    CUDA_TRACE_ERR_CUDA = 2,      /* a CUDA runtime call failed                  */
    CUDA_TRACE_ERR_NO_DEVICE = 3, /* no (or too few) CUDA devices                */
    CUDA_TRACE_ERR_NO_SCENE = 4,  /* trace call before a scene + grid were set   */
    CUDA_TRACE_ERR_CANCELLED = 5  /* cuda_trace_cancel() interrupted the frame   */
} cuda_trace_status;

#define CUDA_TRACE_MISS 0xFFFFFFFFu

/* Ray/triangle test (reference triangle.h) */
#define CUDA_TRACE_VARIANT_MT   0u /* IntersectRayTri, non-culling branch (triangle.h:15-107): the live one */
#define CUDA_TRACE_VARIANT_BARY 1u /* IntersectRayTriBarycentric (triangle.h:210-226)                      */
/* cuda_trace_intersect_rays only, OR-ed onto the variant: "mailboxing", the reference author's TODO at grid.cpp:172 --
 * a ray remembers the outcome of its last 4 ray/triangle tests by triangle index and reuses it when the triangle
 * turns up again in a later cell.  Same results bit for bit (the acceptance window is still evaluated per cell). */
#define CUDA_TRACE_VARIANT_MAILBOX 0x100u

#define CUDA_TRACE_FLAG_GAMMA     1u /* renderer.cpp:125-131 (#define GAMMA_CORRECTION); on in the reference */
#define CUDA_TRACE_FLAG_KEEP_HITS 2u /* also record per-sample tri_idx,t,u,v (cuda_trace_download_hits)      */
/* The alternates the reference keeps next to its live lines (SURVEY 8f N4); none is set by a reference caller */
#define CUDA_TRACE_FLAG_ORTHO             4u  /* GenerateRay's orthographic branch (camera.h:25-36): the frame's
                                               * fov_xs field then carries the WIDTH of the viewing volume      */
#define CUDA_TRACE_FLAG_SHADE_FACE_NORMAL 8u  /* "Vec3f n = tri.n;"      (renderer.cpp:116, commented out)      */
#define CUDA_TRACE_FLAG_SHADE_DEPTH       16u /* "col += Vec3f(t / 3);"  (renderer.cpp:118, commented out)      */

/* Per-frame inputs of Renderer::RenderTile (renderer.cpp:63-72,91-99): frame size (Framebuffer::
 * m_width/m_height), sample count (Renderer::m_sample_count), Scene::GetCameraParameters().
 * fov_xs and aspect are the two constants GenerateRay derives (camera.h:24,41-42); they are
 * computed ON THE HOST by the caller's toolchain (fov_xs = float(tan(double(DegToRad(fov)/2))))
 * so that the device never evaluates a transcendental whose rounding could differ. */
typedef struct cuda_trace_frame
{
    uint32_t width;
    uint32_t height;
    uint32_t spp;
    uint32_t variant; /* CUDA_TRACE_VARIANT_* */
    uint32_t flags;   /* CUDA_TRACE_FLAG_*    */
    float    fov_xs;
    float    aspect;
    float    cam_mat[16]; /* Matrix44f::m_mat in memory order (lin_alg.h:689) */
} cuda_trace_frame;

/* Framebuffer::Tile::GetPosition (framebuffer.h:41-42): [x0,x1) x [y0,y1) in frame pixels */
typedef struct cuda_trace_tile_rect
{
    uint32_t x0, y0, x1, y1;
} cuda_trace_tile_rect;

/* Grid description for cuda_trace_upload_grid / cuda_trace_download_grid = the protected state of
 * the reference's Grid (grid.h:28-39) flattened to CSR in its own cell order
 * (GridIdx = x + z*dim[0] + y*dim[0]*dim[2], grid.h:41-42). */
typedef struct cuda_trace_grid_desc
{
    uint32_t dim[3];
    float    aabb_min[3];
    float    aabb_max[3];
    float    cell_wdh;
    float    inv_cell_wdh;
    uint64_t num_cells; /* dim[0]*dim[1]*dim[2] */
    uint64_t num_refs;  /* cell_offset[num_cells] */
} cuda_trace_grid_desc;

/* Work counters of the last frame (optional instrumentation, see cuda_trace_set_counting) */
typedef struct cuda_trace_counters
{
    uint64_t rays, cells, tri_tests, hits;
} cuda_trace_counters;

/* ---- lifetime -------------------------------------------------------------------------------
 * Replaces Framebuffer::Framebuffer() choosing hardware_concurrency() worker threads
 * (framebuffer.cpp:9-13): here the "workers" are n_gpus devices (ordinals 0..n_gpus-1, or the
 * explicit list).  With n > 1 the scene is replicated and strips are interleaved over the
 * devices; finished pixels are written into device 0's framebuffer over NVLink peer access. */
int  cuda_trace_init(int n_gpus, cuda_trace_ctx **out);
int  cuda_trace_init_devices(const int *device_ordinals, int n, cuda_trace_ctx **out);
void cuda_trace_destroy(cuda_trace_ctx *ctx);
const char *cuda_trace_last_error(const cuda_trace_ctx *ctx); /* ctx may be NULL: last init error */
int  cuda_trace_device_count(void);

/* One-process-per-GPU operation (torchrun): this context renders only its share of every frame's
 * strips -- chunks of 32 consecutive strips dealt round-robin over the world, the owner rotating
 * from round to round.  Default rank 0 / world 1. */
int cuda_trace_set_shard(cuda_trace_ctx *ctx, uint32_t rank, uint32_t world);

/* Sharded frames with an overlapped gather: when enabled on EVERY rank, each rank's kernel counts its
 * finished strips per row band in counters that live behind rank 0's framebuffer (reached through
 * the imported mapping), and rank 0's cuda_trace_tiles() copies each band to the host as soon as
 * all ranks' strips of that band are in -- no barrier between tracing and read-back.  The ranks
 * must still not start frame i+1 before rank 0's call for frame i has returned. */
int cuda_trace_set_shard_signals(cuda_trace_ctx *ctx, int enable);

/* ---- scene ----------------------------------------------------------------------------------
 * Replaces Scene::Scene -> Grid::Grid(mesh, grid_res) (scene.cpp:6-10, grid.cpp:12-154) and the
 * double indirection Grid::Intersect / RenderTile do per triangle (grid.cpp:245-253,
 * renderer.cpp:109-115): vertices = Mesh::m_vertices (V x {p.xyz, n.xyz}, mesh.h:20-24),
 * triangles = Mesh::m_triangles (T x {v0,v1,v2, n.xyz}, mesh.h:12-18), both 24-byte records,
 * passed exactly as they lie in the reference's vectors.  Builds, on every device of the
 * context, the uniform grid (CSR cell offsets + ascending triangle indices), the cell-major
 * float4 triangle records and the per-triangle vertex-normal records. */
int cuda_trace_upload_scene(cuda_trace_ctx *ctx, const float *vertices, uint32_t num_vertices,
                            const uint32_t *triangles, uint32_t num_triangles, uint32_t grid_res);

/* Grid density heuristic for cuda_trace_upload_scene (the reference hard-codes 64 cells on the longest
 * axis, scene.cpp:7): about three cells per triangle, res = cbrt(3 T), while the grid's occupancy map fits in
 * shared memory (res <= 108); about nine, res = cbrt(9 T) <= 896, for the larger grids, which the pooled-ray
 * traversal walks through a distance map.  The density sweep on the 50 M-triangle soup
 * (profiles/r02_c5_grid_density_sweep.txt) has its optimum at 768, where this gives 767; results stay
 * bit-exact for ANY resolution (same algorithm). */
uint32_t cuda_trace_suggest_grid_res(uint32_t num_triangles);

/* Same, but with a grid supplied by the caller instead of built on the device (parity harness:
 * inject the reference's own grid).  cell_offset has desc->num_cells + 1 entries. */
int cuda_trace_upload_scene_with_grid(cuda_trace_ctx *ctx, const float *vertices, uint32_t num_vertices,
                                      const uint32_t *triangles, uint32_t num_triangles,
                                      const cuda_trace_grid_desc *desc, const uint64_t *cell_offset,
                                      const uint32_t *tri_index);

/* Read back the grid the device holds (desc first; arrays may be NULL to query sizes only) */
int cuda_trace_download_grid(cuda_trace_ctx *ctx, cuda_trace_grid_desc *desc, uint64_t *cell_offset,
                             uint32_t *tri_index);

/* Second level of the empty-space walk on large grids (no counterpart in the reference; its author's TODO of a
 * "two-level" grid, grid.h:35-36): one byte per cell of the grid PADDED by one cell on every side, padded cell
 * (X, Y, Z) at X + Z*(dim[0]+2) + Y*(dim[0]+2)*(dim[2]+2), holding min(255, city-block distance in cells to the
 * nearest non-empty cell or padding cell).  The 3D-DDA takes that many steps between look-ups; the cells visited
 * and the arithmetic per step are unchanged, so results stay bit-exact.  Built with the scene whenever the
 * occupancy bitmap of the grid does not fit in shared memory.  out == NULL: query only.  *num_bytes receives
 * the map's size, 0 when this scene has none. */
int cuda_trace_download_distance_map(cuda_trace_ctx *ctx, uint8_t *out, uint64_t *num_bytes);

/* Diagnostics: the screen boxes of device 0 for the camera of the last frame that built them (K1's screen cull,
 * DESIGN.md section 3): 4 floats {xmin, xmax, ymin, ymax} per pair record, in pair-record order; at most
 * capacity / 4 boxes are written.  boxes == NULL: query only.  *num_pairs = pair records (0 when no boxes are
 * built: no scene, or no frame since the upload used the origin-relative records); *small = boxes counted small
 * for that camera; *cull_on = whether the automatic gate turned the cull on (RTM_SCREEN_CULL=1 culls regardless).
 * Read only: it changes neither the boxes nor when they are rebuilt. */
int cuda_trace_download_screen_boxes(cuda_trace_ctx *ctx, float *boxes, uint64_t capacity, uint64_t *num_pairs,
                                     uint32_t *small, int *cull_on);

/* ---- tracing --------------------------------------------------------------------------------
 * cuda_trace_tiles replaces Framebuffer::CreateWorkerThreads + WorkerThread + RenderTile for the
 * given tiles (framebuffer.cpp:16-27,59-92; renderer.cpp:43-136): it renders every pixel of every
 * rect and returns after the pixels are in host_bgra (width*height uint32, row 0 = y 0, pixel
 * value as ToBGRA8 packs it, lin_alg.h:125-132; pixels outside the rects are left untouched).
 * host_bgra may be NULL (render into the device framebuffer only).
 * cuda_trace_tiles_async only enqueues the frame; cuda_trace_sync waits for it, and
 * cuda_trace_read_framebuffer copies the device framebuffer out. */
int cuda_trace_tiles(cuda_trace_ctx *ctx, const cuda_trace_frame *frame, const cuda_trace_tile_rect *tiles,
                     uint32_t n_tiles, uint32_t *host_bgra);
int cuda_trace_tiles_async(cuda_trace_ctx *ctx, const cuda_trace_frame *frame,
                           const cuda_trace_tile_rect *tiles, uint32_t n_tiles);
int cuda_trace_sync(cuda_trace_ctx *ctx);
int cuda_trace_read_framebuffer(cuda_trace_ctx *ctx, uint32_t *host_bgra);

/* The same frame, but every tile lands in its OWN host buffer -- row-major within the tile, index x + y * tile_width:
 * Framebuffer::Tile::m_bgra (framebuffer.h:64, written at renderer.cpp:133) -- and the caller learns of tiles as
 * they complete: done(indices, count, user) is called ON THE CALLING THREAD, top of the frame first, once the pixels
 * of tiles[indices[0 .. count)] are in host memory, while the rest of the frame is still being traced.  That is the
 * moment the reference's worker releases the tile mutex (framebuffer.cpp:72-77), so a drop-in Framebuffer can let
 * SaveToBMP / Draw see a frame in progress (framebuffer.cpp:163,203).  tile_bgra[i] should be page-locked
 * (cuda_trace_host_alloc); `done` may be NULL.  Returns when the whole frame is on the host. */
typedef void (*cuda_trace_tiles_done_fn)(const uint32_t *tile_indices, uint32_t count, void *user);
int cuda_trace_tiles_into(cuda_trace_ctx *ctx, const cuda_trace_frame *frame, const cuda_trace_tile_rect *tiles,
                          uint32_t n_tiles, uint32_t *const *tile_bgra, cuda_trace_tiles_done_fn done, void *user);

/* Framebuffer::m_threads_stop (framebuffer.h:32): ask the running frame to stop early.  Safe to
 * call from another thread while cuda_trace_tiles / cuda_trace_sync block. */
int cuda_trace_cancel(cuda_trace_ctx *ctx);

/* Milliseconds the trace kernel of the last completed frame took (CUDA events on its stream,
 * max over the context's devices) */
int cuda_trace_last_kernel_ms(cuda_trace_ctx *ctx, float *ms);

/* Per-sample hit records of the last frame rendered with CUDA_TRACE_FLAG_KEEP_HITS, indexed
 * (y*width + x)*spp + smp: what Grid::Intersect returned for that sample (grid.cpp:159-281);
 * tri_idx = CUDA_TRACE_MISS (t=u=v=0) on a miss.  Any output pointer may be NULL. */
int cuda_trace_download_hits(cuda_trace_ctx *ctx, uint32_t *tri_idx, float *t, float *u, float *v);

/* Grid::Intersect (grid.h:16-23, grid.cpp:159-281) for a batch of arbitrary rays: origins / dirs
 * are n x 3 floats.  tri_idx = CUDA_TRACE_MISS on a miss. */
int cuda_trace_intersect_rays(cuda_trace_ctx *ctx, uint32_t n, const float *origins, const float *dirs,
                              uint32_t variant, uint32_t *tri_idx, float *t, float *u, float *v);

/* ---- ray queries on rays that already live on the GPU -------------------------------------------
 * No counterpart in the reference: Grid::Intersect (grid.cpp:159-281) for a batch of caller rays in device memory,
 * bounded by t_max, plus a yes/no occlusion answer (shadow rays, ambient occlusion, picking, rays built on the GPU).
 *
 * Closest hit, bounded: the reference walk with two changes --
 *   1. a triangle is accepted in a cell only if  hit && t < best && t < next_crossing_t[step_axis] && t < t_max;
 *   2. the walk ends as a miss at the first cell the ray enters through a crossing greater than t_max (the first
 *      cell's entry is the box entry, 0 for an origin inside the box).
 * Only occupied cells are affected by rule 2, so every occupancy-map mode gives the same bits.  Consequences:
 *   - t_max = +INFINITY gives exactly Grid::Intersect (and cuda_trace_intersect_rays); the crossing test is strict,
 *     so an infinite crossing (delta overflowing on an unnormalised direction) does not end the walk;
 *   - t_max <= 0 or NaN gives a miss;
 *   - the result equals "the unbounded hit, kept if t < t_max" except for one floating-point corner of the grid
 *     build: a triangle the grid registers only in cells entered after t_max can still be hit at t < t_max, and
 *     the bounded walk, which stops before those cells, reports a miss.
 * Occlusion: occluded[i] = 1 exactly when the bounded closest-hit query with the same t_max hits.  Acceptance does
 * not depend on earlier hits before the first one, so the first accepted triangle decides (any-hit exit).
 *
 * Variants: CUDA_TRACE_VARIANT_MT or CUDA_TRACE_VARIANT_BARY; CUDA_TRACE_VARIANT_MAILBOX is refused (ERR_ARG). */
#define CUDA_TRACE_QUERY_CLOSEST   0u
#define CUDA_TRACE_QUERY_OCCLUSION 1u
typedef struct cuda_trace_ray_batch
{
    uint32_t n, kind, variant;       /* rays, CUDA_TRACE_QUERY_*, CUDA_TRACE_VARIANT_MT / _BARY                  */
    float    t_max_all;              /* used when t_max == NULL; INFINITY = unbounded                            */
    const float *origins, *dirs;     /* DEVICE memory, n x 3 float, contiguous                                   */
    const float *t_max;              /* DEVICE, n, or NULL                                                       */
    uint32_t *tri_idx;               /* CLOSEST: DEVICE, n, required; CUDA_TRACE_MISS on a miss                  */
    float *t, *u, *v;                /* CLOSEST: DEVICE, n, each may be NULL (0 on a miss)                       */
    uint8_t *occluded;               /* OCCLUSION: DEVICE, n, required (0 / 1)                                   */
} cuda_trace_ray_batch;
/* Enqueues the query on `stream` (a cudaStream_t of the context's device 0; NULL = cuda_trace_stream(ctx)) and
 * returns: no host synchronisation, no allocation.  Every pointer must be device or managed memory of device 0
 * (checked with cudaPointerGetAttributes); otherwise, and for a bad kind / variant, the MAILBOX bit, a missing
 * required output or n > 0 with NULL inputs, CUDA_TRACE_ERR_ARG is returned and nothing is enqueued.  No scene:
 * CUDA_TRACE_ERR_NO_SCENE.  Queries read only immutable scene arrays, so they may overlap a frame; replacing the
 * scene or destroying the context first waits for the queries already enqueued. */
int cuda_trace_query_rays(cuda_trace_ctx *ctx, const cuda_trace_ray_batch *b, void *stream);

/* After a CUDA_TRACE_VARIANT_MAILBOX call: ray/triangle tests the walk asked for, and how many of them the
 * mailbox answered */
int cuda_trace_mailbox_stats(cuda_trace_ctx *ctx, uint64_t *tests, uint64_t *reused);

/* Renderer::IntersectBruteForce (renderer.cpp:157-197): the same ray/triangle test against EVERY triangle,
 * no grid -- the reference author's own cross-check of Grid::Intersect, kept as an on-device self-check.
 * It differs from the grid result only where the grid's "hit must lie in the current cell" rule or an
 * exact-t tie decides (SURVEY.md section 8c).  O(n * T): meant for small scenes / few rays. */
int cuda_trace_intersect_rays_brute_force(cuda_trace_ctx *ctx, uint32_t n, const float *origins, const float *dirs,
                                          uint32_t *tri_idx, float *t, float *u, float *v);

/* Renderer::RayMarch (renderer.cpp:24-41): sphere tracing -- up to 128 steps of t += DistanceBruteForce(pos)
 * (renderer.cpp:138-155, DistancePointTri triangle.h:163-198) until the distance drops below 0.001.
 * The "march" of the project's name; commented out of the reference's pixel loop, kept as a ray query.
 * hit[i] = 1 / 0, t[i] = the parameter reached.  O(n * 128 * T): small scenes / few rays. */
int cuda_trace_ray_march(cuda_trace_ctx *ctx, uint32_t n, const float *origins, const float *dirs, uint32_t *hit,
                         float *t);

/* The renderer.cpp:49-60 sample table as the device computes it: xy = spp x {x, y} */
int cuda_trace_sample_table(cuda_trace_ctx *ctx, uint32_t spp, float *xy);

/* ---- QMC sample tables on the device (the reference's sampling module, sampling.cpp:55-290) ------
 * out[i * dim_count + j] = sequence(n_begin + i, dim_begin + j), fp64 like the reference.
 *   kind:     0 HaltonSequence, 1 HammersleySequence(num_smp), 2 HaltonZarembaSequence,
 *             3 HammersleyZarembaSequence(num_smp), 4 RadicalInverseBase2(n, bits),
 *             5 SobolRadicalInverseBase2(n, bits), 6 LarcherPillichshammerRadicalInverseBase2(n, bits)
 *   scramble (kinds 0, 1; sampling.h:37-95): 0 ScrambleNone, 2 ScrambleFaure (first 128 primes, generated
 *             here), 3 ScrambleReverse (128 primes), 1 / 4 digit permutations supplied by the caller in
 *             `perm` = the tables of the first `perm_primes` primes back to back (2 + 3 + 5 + ... entries):
 *             1 for the Braaten-Weller table (16 primes; assets/sampling/braaten_weller_16.u32), 4 for any
 *             other, e.g. the reference's ScrambleRandomized table, which is whatever the host's
 *             std::random_shuffle produced (sampling.cpp:174-192) and must therefore be uploaded.
 *   dim_begin + dim_count <= 1000 (PRIME_TBL_SIZE).  perm may be NULL for scramble 0, 2, 3. */
int cuda_trace_qmc_sequence(cuda_trace_ctx *ctx, uint32_t kind, uint32_t scramble, const uint32_t *perm,
                            uint32_t perm_primes, uint32_t n_begin, uint32_t count, uint32_t dim_begin,
                            uint32_t dim_count, uint32_t num_smp, uint32_t bits, double *out);
/* CranleyPattersonRotation(x[i], e) (sampling.cpp:283-290) */
int cuda_trace_qmc_cranley_patterson(cuda_trace_ctx *ctx, const double *x, double e, uint32_t count, double *out);

/* Optional instrumentation: count rays / visited cells / triangle tests / hits of the next frames
 * (slower kernel variant).  cuda_trace_get_counters returns those of the last frame. */
int cuda_trace_set_counting(cuda_trace_ctx *ctx, int enable);
int cuda_trace_get_counters(cuda_trace_ctx *ctx, cuda_trace_counters *out);

/* Host-clock marks of the last cuda_trace_tiles call, in ms since its entry: [0] work submitted, [1] trace stream
 * drained, [2] read-back copies drained (overlapped mode), [3] return, [4] host set-up done, [5] / [6] before /
 * after the launch of the first device's trace kernel.  Diagnostics for the end-to-end figure. */
int cuda_trace_last_call_timing(cuda_trace_ctx *ctx, double ms[7]);

/* Host arithmetic only (no device): the per-GPU completion targets of the overlapped read-back for a frame
 * layout -- shares[q * 32 + b] = pieces of strips GPU q of `world` finishes in row band b (strips dealt in chunks
 * of `chunk`), gpus_in_band[b] = GPUs with a share in band b, plus the band height / count and the pieces a strip
 * counts as.  What cuda_trace_tiles programs into the kernel and waits for; exported for CPU tests of the
 * multi-GPU bookkeeping. */
int cuda_trace_band_shares(uint32_t width, uint32_t height, uint32_t spp, const cuda_trace_tile_rect *tiles, uint32_t n_tiles,
                           uint32_t world, uint32_t chunk, uint32_t *shares, uint32_t *gpus_in_band, uint32_t *band_rows,
                           uint32_t *n_bands, uint32_t *pieces_per_strip);

/* Scheduler diagnostics: SM cycles each strip of the last frame took on device 0, in this shard's strip order
 * (the input of the cost-ordered scheduling, csrc/schedule.cu).  *count = strips recorded (0 when the last frame
 * ran without cost recording -- see RTM_COST_ORDER); at most `capacity` values are written. */
int cuda_trace_download_strip_cycles(cuda_trace_ctx *ctx, uint32_t *cycles, uint64_t capacity, uint64_t *count);

/* Page-locked host memory for the framebuffer passed to cuda_trace_tiles / read_framebuffer: the
 * device-to-host copy is then a single DMA at full PCIe rate.  Any other host memory works too
 * (the driver stages it), only slower.  Free with cuda_trace_host_free. */
void *cuda_trace_host_alloc(size_t bytes);
void  cuda_trace_host_free(void *p);

/* How many kernels this library has launched since cuda_trace_init (all devices) */
uint64_t cuda_trace_kernel_launches(const cuda_trace_ctx *ctx);

/* ---- multi-process gather (one process per GPU) --------------------------------------------
 * Rank 0 exports its device framebuffer as a 64-byte CUDA IPC handle; the other ranks import it
 * and their trace kernels then store finished pixels straight into rank 0's memory over NVLink.
 * cuda_trace_prepare_framebuffer (re)allocates the device framebuffer for width x height. */
int cuda_trace_prepare_framebuffer(cuda_trace_ctx *ctx, uint32_t width, uint32_t height);
int cuda_trace_export_framebuffer(cuda_trace_ctx *ctx, void *handle64);
int cuda_trace_import_framebuffer(cuda_trace_ctx *ctx, const void *handle64, uint32_t width, uint32_t height);

/* Raw device pointer of the framebuffer the kernels write to (for zero-copy consumers, e.g. a
 * torch tensor view or CUDA-GL interop) and the CUDA stream handle (cudaStream_t) used on
 * device 0 */
void *cuda_trace_framebuffer_device_ptr(cuda_trace_ctx *ctx);
void *cuda_trace_stream(cuda_trace_ctx *ctx);

#ifdef __cplusplus
}
#endif

#endif /* CUDA_TRACE_H */
