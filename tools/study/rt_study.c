/* STUDY code (tools/ only -- not the oracle, not the product): instrumented replays of the reference's grid walk
 * used to decide what to build next.  Kept apart from oracle/rt_oracle.c so that the oracle restates the reference
 * and nothing else; this file has its own copy of the walk (grid.cpp:159-281) on top of the oracle's primitives
 * (rto_ray_tri, rto_ray_aabb, ... from oracle/librt_oracle.so) and adds:
 *
 *   rts_ray_walk_profile   the triangle-list length of every cell a ray visits, in order (tools/warp_walk_model.py)
 *   rts_ray_walk_cells     the indices of the occupied cells a ray visits, in order (the screen-cull model of
 *                          tools/warp_walk_model.py)
 *   rts_mailbox_walk       the walk WITH the mailbox of the product's optional mode (CUDA_TRACE_VARIANT_MAILBOX,
 *                          csrc/rt_device.cuh): 4 entries, round-robin over the tests actually computed -- returns the
 *                          hit and counts tests asked for / answered from the mailbox (tests/test_mailbox_model_cpu.py
 *                          checks that results equal the plain walk and that the counts equal what the GPU reported)
 *   rts_bounded_walk       the walk bounded by t_max of the product's ray queries (cuda_trace_query_rays, include/
 *   rts_query_rays         cuda_trace.h): rto_grid_intersect with its rules 1 and 2; a batch entry for the tests
 *                          (tests/test_ray_query_cpu.py, tests/test_gpu_ray_query.py).  The oracle's own walk stays
 *                          the reference's and nothing else, so this one lives here
 *   rts_study_ray          mailbox study  -- how often a ray re-tests a triangle it has tested within its last
 *                                            2 / 8 / 64 tests (the author's "mailboxing" TODO, grid.cpp:172)
 *                          pre-test study -- a conservative sphere reject in front of Moeller-Trumbore: the ray
 *                                            line's squared distance from v0 against 1.01 max(|e1|^2, |e2|^2) +
 *                                            32 ulp |tvec|^2; counts skips, violations (a skipped test that hits:
 *                                            must stay 0) and kept tests that fail anyway
 *
 * Build: gcc -O2 -std=c99 -ffp-contract=off -fPIC -shared -I../../oracle -o librt_study.so rt_study.c \
 *            -L../../oracle -lrt_oracle -Wl,-rpath,'$ORIGIN/../../oracle'     (tools/study/build.sh)
 */
#include <float.h>
#include <stdint.h>
#include <stddef.h>
#include "rt_oracle.h"

typedef struct rts_counters
{
    uint64_t tests;          /* ray/triangle tests replayed                                                   */
    uint64_t rep2, rep8, rep64; /* tests whose triangle is among the ray's last 2 / 8 / 64 tested ids         */
    uint64_t pre_reject;     /* tests the pre-test would skip                                                 */
    uint64_t pre_violation;  /* ... of which the exact test reports a hit (must stay 0)                       */
    uint64_t pre_keep_fail;  /* tests the pre-test keeps and the exact test then rejects                      */
} rts_counters;

static int to_voxel(const rto_grid *g, const float *p, int axis)
{
    const int v = (int) ((p[axis] - g->aabb_min[axis]) * g->inv_cell_wdh);
    const int hi = (int) g->dim[axis] - 1;
    return v < 0 ? 0 : (v > hi ? hi : v);
}
static float to_pos(const rto_grid *g, int vox, int axis) { return g->aabb_min[axis] + vox * g->cell_wdh; }

/* the walk of grid.cpp:159-281 (Moeller-Trumbore) with both recorders; either output may be NULL */
static int walk(const rto_scene *sc, const float *origin, const float *dir, uint16_t *lens, uint32_t *ids, uint32_t cap,
                uint32_t *n_cells, rts_counters *cnt)
{
    const rto_grid *g = &sc->grid;
    float enter_t, leave_t, gi[3];
    *n_cells = 0;
    if (rto_point_in_aabb(origin, g->aabb_min, g->aabb_max))
    {
        enter_t = 0.0f;
        gi[0] = origin[0]; gi[1] = origin[1]; gi[2] = origin[2];
    }
    else if (rto_ray_aabb(origin, dir, g->aabb_min, g->aabb_max, &enter_t, &leave_t))
        for (int a = 0; a < 3; a++)
            gi[a] = origin[a] + dir[a] * enter_t;
    else
        return 0;
    float next_t[3], delta_t[3] = { 0.0f, 0.0f, 0.0f };
    int step[3] = { 1, 1, 1 }, out[3], pos[3];
    for (int a = 0; a < 3; a++)
    {
        out[a] = (int) g->dim[a];
        pos[a] = to_voxel(g, gi, a);
        if (dir[a] == 0.0f)
            next_t[a] = FLT_MAX;
        else if (dir[a] > 0.0f)
        {
            next_t[a] = enter_t + (to_pos(g, pos[a] + 1, a) - gi[a]) / dir[a];
            delta_t[a] = g->cell_wdh / dir[a];
        }
        else
        {
            next_t[a] = enter_t + (to_pos(g, pos[a], a) - gi[a]) / dir[a];
            delta_t[a] = -g->cell_wdh / dir[a];
            step[a] = -1;
            out[a] = -1;
        }
    }
    float best = FLT_MAX;
    uint32_t mbox[64], mbox_n = 0;
    for (;;)
    {
        const int sa = (next_t[0] < next_t[1]) ? ((next_t[0] < next_t[2]) ? 0 : 2) : ((next_t[1] < next_t[2]) ? 1 : 2);
        const uint64_t cell = (uint64_t) pos[0] + (uint64_t) pos[2] * g->dim[0] + (uint64_t) pos[1] * g->dim[0] * g->dim[2];
        const uint64_t len = g->cell_offset[cell + 1] - g->cell_offset[cell];
        if (lens && *n_cells < cap)
            lens[*n_cells] = (uint16_t) (len > 65535 ? 65535 : len);
        if (ids && len && *n_cells < cap)
            ids[*n_cells] = (uint32_t) cell;
        if (!ids || len)
            (*n_cells)++;
        for (uint64_t k = g->cell_offset[cell]; k < g->cell_offset[cell + 1]; k++)
        {
            const uint32_t ci = g->tri_index[k];
            const uint32_t *tr = sc->tri + (size_t) ci * 6;
            const float *v0 = sc->vtx + (size_t) tr[0] * 6, *v1 = sc->vtx + (size_t) tr[1] * 6, *v2 = sc->vtx + (size_t) tr[2] * 6;
            float ct, cu, cv;
            const int hit = rto_ray_tri(origin, dir, v0, v1, v2, &ct, &cu, &cv, NULL);
            if (cnt)
            {
                cnt->tests++;
                int found = -1;
                for (uint32_t m = 0; m < mbox_n && m < 64; m++)
                    if (mbox[(mbox_n - 1 - m) & 63] == ci) { found = (int) m; break; }
                if (found >= 0 && found < 2) cnt->rep2++;
                if (found >= 0 && found < 8) cnt->rep8++;
                if (found >= 0) cnt->rep64++;
                mbox[mbox_n & 63] = ci;
                mbox_n++;
                /* |tvec x d|^2 > thresh, all in fp32 without contraction */
                const float tv[3] = { origin[0] - v0[0], origin[1] - v0[1], origin[2] - v0[2] };
                const float e1[3] = { v1[0] - v0[0], v1[1] - v0[1], v1[2] - v0[2] };
                const float e2[3] = { v2[0] - v0[0], v2[1] - v0[1], v2[2] - v0[2] };
                const float l1 = e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2];
                const float l2 = e2[0] * e2[0] + e2[1] * e2[1] + e2[2] * e2[2];
                const float tt = tv[0] * tv[0] + tv[1] * tv[1] + tv[2] * tv[2];
                const float thresh = (l1 > l2 ? l1 : l2) * 1.01f + tt * (32.0f * 5.9604645e-8f);
                const float qx = tv[1] * dir[2] - tv[2] * dir[1];
                const float qy = tv[2] * dir[0] - tv[0] * dir[2];
                const float qz = tv[0] * dir[1] - tv[1] * dir[0];
                if (qx * qx + qy * qy + qz * qz > thresh)
                {
                    cnt->pre_reject++;
                    if (hit) cnt->pre_violation++;
                }
                else if (!hit)
                    cnt->pre_keep_fail++;
            }
            if (hit && ct < best && ct < next_t[sa])
                best = ct;
        }
        if (best != FLT_MAX)
            return 1;
        pos[sa] += step[sa];
        if (pos[sa] == out[sa])
            break;
        next_t[sa] += delta_t[sa];
    }
    return 0;
}

/* -> number of cells visited (may exceed cap; only cap entries are written); the last one is the hit's cell when *hit */
uint32_t rts_ray_walk_profile(const rto_scene *sc, const float *origin, const float *dir, uint32_t cap, uint16_t *list_lengths,
                              int *hit)
{
    uint32_t n = 0;
    *hit = walk(sc, origin, dir, list_lengths, NULL, cap, &n, NULL);
    return n;
}

/* -> number of OCCUPIED cells visited, their (unpadded) cell indices in order in cell_ids (at most cap are written; the
 * last one is the hit's cell when *hit) -- tools/warp_walk_model.py --screen-cull */
uint32_t rts_ray_walk_cells(const rto_scene *sc, const float *origin, const float *dir, uint32_t cap, uint32_t *cell_ids, int *hit)
{
    uint32_t n = 0;
    *hit = walk(sc, origin, dir, NULL, cell_ids, cap, &n, NULL);
    return n;
}

int rts_study_ray(const rto_scene *sc, const float *origin, const float *dir, rts_counters *cnt)
{
    uint32_t n = 0;
    return walk(sc, origin, dir, NULL, NULL, 0, &n, cnt);
}

/* The product's mailbox mode restated on the CPU: same walk, same 4-entry round-robin mailbox keyed by triangle index,
 * outcome (hit, t, u, v) reused when the triangle turns up again; the acceptance window is evaluated per cell. */
int rts_mailbox_walk(const rto_scene *sc, const float *origin, const float *dir, int variant, float *t, float *u, float *v,
                     uint32_t *tri_idx, uint64_t *asked, uint64_t *reused)
{
    const rto_grid *g = &sc->grid;
    float enter_t, leave_t, gi[3];
    if (rto_point_in_aabb(origin, g->aabb_min, g->aabb_max))
    {
        enter_t = 0.0f;
        gi[0] = origin[0]; gi[1] = origin[1]; gi[2] = origin[2];
    }
    else if (rto_ray_aabb(origin, dir, g->aabb_min, g->aabb_max, &enter_t, &leave_t))
        for (int a = 0; a < 3; a++)
            gi[a] = origin[a] + dir[a] * enter_t;
    else
        return 0;
    float next_t[3], delta_t[3] = { 0.0f, 0.0f, 0.0f };
    int step[3] = { 1, 1, 1 }, out[3], pos[3];
    for (int a = 0; a < 3; a++)
    {
        out[a] = (int) g->dim[a];
        pos[a] = to_voxel(g, gi, a);
        if (dir[a] == 0.0f)
            next_t[a] = FLT_MAX;
        else if (dir[a] > 0.0f)
        {
            next_t[a] = enter_t + (to_pos(g, pos[a] + 1, a) - gi[a]) / dir[a];
            delta_t[a] = g->cell_wdh / dir[a];
        }
        else
        {
            next_t[a] = enter_t + (to_pos(g, pos[a], a) - gi[a]) / dir[a];
            delta_t[a] = -g->cell_wdh / dir[a];
            step[a] = -1;
            out[a] = -1;
        }
    }
    uint32_t mb_id[4] = { 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu }, mb_next = 0;
    int mb_hit[4] = { 0, 0, 0, 0 };
    float mb_t[4] = { 0 }, mb_u[4] = { 0 }, mb_v[4] = { 0 };
    float best = FLT_MAX;
    for (;;)
    {
        const int sa = (next_t[0] < next_t[1]) ? ((next_t[0] < next_t[2]) ? 0 : 2) : ((next_t[1] < next_t[2]) ? 1 : 2);
        const uint64_t cell = (uint64_t) pos[0] + (uint64_t) pos[2] * g->dim[0] + (uint64_t) pos[1] * g->dim[0] * g->dim[2];
        for (uint64_t k = g->cell_offset[cell]; k < g->cell_offset[cell + 1]; k++)
        {
            const uint32_t ci = g->tri_index[k];
            float ct = 0.0f, cu = 0.0f, cv = 0.0f;
            int hit = 0, found = 0;
            (*asked)++;
            for (int j = 0; j < 4; j++)
                if (mb_id[j] == ci)
                {
                    found = 1;
                    hit = mb_hit[j]; ct = mb_t[j]; cu = mb_u[j]; cv = mb_v[j];
                }
            if (found)
                (*reused)++;
            else
            {
                const uint32_t *tr = sc->tri + (size_t) ci * 6;
                const float *v0 = sc->vtx + (size_t) tr[0] * 6, *v1 = sc->vtx + (size_t) tr[1] * 6, *v2 = sc->vtx + (size_t) tr[2] * 6;
                if (variant == RTO_VARIANT_BARY)
                    hit = rto_ray_tri_bary(origin, dir, v0, v1, v2, (const float *) (tr + 3), &ct, &cu, &cv, NULL);
                else
                    hit = rto_ray_tri(origin, dir, v0, v1, v2, &ct, &cu, &cv, NULL);
                const uint32_t slot = mb_next++ % 4u;
                mb_id[slot] = ci; mb_hit[slot] = hit; mb_t[slot] = ct; mb_u[slot] = cu; mb_v[slot] = cv;
            }
            if (hit && ct < best && ct < next_t[sa])
            {
                best = ct; *t = ct; *u = cu; *v = cv; *tri_idx = ci;
            }
        }
        if (best != FLT_MAX)
            return 1;
        pos[sa] += step[sa];
        if (pos[sa] == out[sa])
            break;
        next_t[sa] += delta_t[sa];
    }
    return 0;
}

/* rto_grid_intersect (grid.cpp:159-281) bounded by t_max:
 *   rule 1  a triangle is accepted only if also t < t_max;
 *   rule 2  the walk ends as a miss at the first OCCUPIED cell entered through a crossing greater than t_max (the
 *           first cell's entry is enter_t; every later cell's is the next_t[sa] of the step that entered it).
 * Returns 1 on a hit, 0 on a miss, 2 on a miss decided by rule 2. */
int rts_bounded_walk(const rto_scene *sc, const float *origin, const float *dir, int variant, float t_max, float *t,
                     float *u, float *v, uint32_t *tri_idx)
{
    const rto_grid *g = &sc->grid;
    float enter_t, leave_t, gi[3];
    if (rto_point_in_aabb(origin, g->aabb_min, g->aabb_max))
    {
        enter_t = 0.0f;
        gi[0] = origin[0]; gi[1] = origin[1]; gi[2] = origin[2];
    }
    else if (rto_ray_aabb(origin, dir, g->aabb_min, g->aabb_max, &enter_t, &leave_t))
    {
        gi[0] = origin[0] + dir[0] * enter_t;
        gi[1] = origin[1] + dir[1] * enter_t;
        gi[2] = origin[2] + dir[2] * enter_t;
    }
    else
        return 0;
    float next_t[3], delta_t[3] = { 0.0f, 0.0f, 0.0f };
    int step[3] = { 1, 1, 1 }, out[3], pos[3];
    for (int a = 0; a < 3; a++)
    {
        out[a] = (int) g->dim[a];
        pos[a] = to_voxel(g, gi, a);
        if (dir[a] == 0.0f)
            next_t[a] = FLT_MAX;
        else if (dir[a] > 0.0f)
        {
            next_t[a] = enter_t + (to_pos(g, pos[a] + 1, a) - gi[a]) / dir[a];
            delta_t[a] = g->cell_wdh / dir[a];
        }
        else
        {
            next_t[a] = enter_t + (to_pos(g, pos[a], a) - gi[a]) / dir[a];
            delta_t[a] = -g->cell_wdh / dir[a];
            step[a] = -1;
            out[a] = -1;
        }
    }
    float entry = enter_t;
    *t = FLT_MAX;
    for (;;)
    {
        const int sa = (next_t[0] < next_t[1]) ? ((next_t[0] < next_t[2]) ? 0 : 2) : ((next_t[1] < next_t[2]) ? 1 : 2);
        const uint64_t cell = (uint64_t) pos[0] + (uint64_t) pos[2] * g->dim[0] + (uint64_t) pos[1] * g->dim[0] * g->dim[2];
        if (g->cell_offset[cell] != g->cell_offset[cell + 1] && entry > t_max)
            return 2;
        for (uint64_t k = g->cell_offset[cell]; k < g->cell_offset[cell + 1]; k++)
        {
            const uint32_t ci = g->tri_index[k];
            const uint32_t *tr = sc->tri + (size_t) ci * 6;
            const float *v0 = sc->vtx + (size_t) tr[0] * 6, *v1 = sc->vtx + (size_t) tr[1] * 6, *v2 = sc->vtx + (size_t) tr[2] * 6;
            float ct, cu, cv;
            const int hit = variant == RTO_VARIANT_BARY
                                ? rto_ray_tri_bary(origin, dir, v0, v1, v2, (const float *) (tr + 3), &ct, &cu, &cv, NULL)
                                : rto_ray_tri(origin, dir, v0, v1, v2, &ct, &cu, &cv, NULL);
            if (hit && ct < *t && ct < next_t[sa] && ct < t_max)
            {
                *t = ct; *u = cu; *v = cv; *tri_idx = ci;
            }
        }
        if (*t != FLT_MAX)
            return 1;
        entry = next_t[sa];
        pos[sa] += step[sa];
        if (pos[sa] == out[sa])
            break;
        next_t[sa] += delta_t[sa];
    }
    return 0;
}

/* A batch of rts_bounded_walk: t_max per ray, or t_max_all for every ray when t_max is NULL.  Outputs as
 * cuda_trace_query_rays writes them (tri = RTO_MISS and t = u = v = 0 on a miss); stopped[i] = 1 where rule 2 decided
 * the miss (may be NULL). */
void rts_query_rays(const rto_scene *sc, uint32_t n, const float *origins, const float *dirs, const float *t_max,
                    float t_max_all, int variant, uint32_t *tri_idx, float *t, float *u, float *v, uint8_t *stopped)
{
    for (uint32_t i = 0; i < n; i++)
    {
        float ct = 0.0f, cu = 0.0f, cv = 0.0f;
        uint32_t idx = RTO_MISS;
        const int r = rts_bounded_walk(sc, origins + 3 * (size_t) i, dirs + 3 * (size_t) i, variant,
                                       t_max ? t_max[i] : t_max_all, &ct, &cu, &cv, &idx);
        tri_idx[i] = r == 1 ? idx : RTO_MISS;
        t[i] = r == 1 ? ct : 0.0f;
        u[i] = r == 1 ? cu : 0.0f;
        v[i] = r == 1 ? cv : 0.0f;
        if (stopped)
            stopped[i] = r == 2;
    }
}
