"""CPU model of K1's warp-level traversal (no GPU): where do the lanes of a warp wait?

For a sample of strips of a frame, the oracle port records for every primary ray the triangle-list lengths of the
cells it visits (tools/study/rt_study.c rts_ray_walk_profile, a study copy of the oracle's walk).  The model then replays K1's two-phase loop per warp round (32 rays,
lane = pixel-in-round * spp + sample): phase A costs the LONGEST empty-cell run among the lanes, phase B the LONGEST
list, and compares with (a) the useful work, i.e. perfect packing, and (b) re-pairing the strip's rays between phases
(the rays of one strip pooled, sorted by what they need next, and dealt to the strip's warps).

With --screen-cull it replays phase B of the same warps against the screen boxes of the pair records
(tools/screen_cull.py) instead: the fraction of pair iterations in which every lane
that owns a pair is outside its box -- the iterations K1 could skip before loading the record -- with one box per pair
and, for comparison, one per triangle.

With --warp-scan it also replays the warp scan of the cull (csrc/warp_trace.cuh test_pair_list): in a round
whose lanes with a list all stand on one cell, 32 boxes are checked at once against the footprint of the lanes' image
points (screen_cull.footprint_skips) and only the pairs left are walked; other rounds keep the serial walk.  It reports
how often the fast path applies, the 32-pair chunks, the pairs the footprint keeps against those the per-lane check
keeps, and the pair iterations before and after; and, as the alternative for phase A, the share of a lane's occupied-
cell visits whose point lies outside the cell's box (the union of its pair boxes).

python tools/warp_walk_model.py [workload] [n_strips] [--screen-cull | --warp-scan]   (test infrastructure: imports oracle/)"""
import ctypes as C
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import pyoracle  # noqa: E402

pkg = lambda s: importlib.import_module("cpp-11-ray-trace-march-framework_b200." + s)
scenes, hostapi, mr = pkg("scenes"), pkg("hostapi"), pkg("multirank")

C_DDA, C_TEST, C_ITER = 13, 61, 24  # SASS instructions: one DDA step, one triangle test, fixed cost of one A+B iteration

SCAN = "--warp-scan" in sys.argv
CULL = "--screen-cull" in sys.argv or SCAN
args = [a for a in sys.argv[1:] if a not in ("--screen-cull", "--warp-scan")]
wl = args[0] if args else "killeroo4k"
n_strips = int(args[1]) if len(args) > 1 else 1500
scene, w, h, spp, res = scenes.CONFIGS[wl]
host = hostapi.host_api()
m, fov, cam = scenes.build(host, scene)
vtx, tri = m.arrays()
port = pyoracle.Port.get()
ps = port.scene(vtx, tri, res)
lib = port.lib
F, U16 = C.POINTER(C.c_float), C.POINTER(C.c_uint16)
import subprocess  # noqa: E402
STUDY = os.path.join(os.path.dirname(os.path.abspath(__file__)), "study")
subprocess.check_call(["bash", os.path.join(STUDY, "build.sh")])
study = C.CDLL(os.path.join(STUDY, "librt_study.so"))
study.rts_ray_walk_profile.restype = C.c_uint32
study.rts_ray_walk_profile.argtypes = [C.c_void_p, F, F, C.c_uint32, U16, C.POINTER(C.c_int)]
study.rts_ray_walk_cells.restype = C.c_uint32
study.rts_ray_walk_cells.argtypes = [C.c_void_p, F, F, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_int)]
smp = port.sample_table(spp)
fov_xs, aspect = port.camera_constants(fov, w, h)
cam32 = np.ascontiguousarray(cam, np.float32)
sw, sh = mr.strip_size(spp, w * h * spp)
rs = np.random.RandomState(7)
prof_buf = np.zeros(4096, np.uint16)


def ray_profile(px, py, s):
    o, d = np.zeros(3, np.float32), np.zeros(3, np.float32)
    lib.rto_generate_ray(cam32.ctypes.data_as(F), px, py, w, h, float(smp[s, 0]), float(smp[s, 1]), float(fov_xs),
                         float(aspect), o.ctypes.data_as(F), d.ctypes.data_as(F))
    hit = C.c_int(0)
    n = study.rts_ray_walk_profile(C.byref(ps.s), o.ctypes.data_as(F), d.ctypes.data_as(F), len(prof_buf),
                                 prof_buf.ctypes.data_as(U16), C.byref(hit))
    return prof_buf[:min(n, len(prof_buf))].astype(np.int64).copy()


def segments(profile):
    """-> list of (empty_steps_before, list_len) per occupied cell visited, + trailing empty steps to the exit.
    K1 steps once after every tested cell, so the step onto the next cell belongs to the following phase A."""
    segs, run = [], 0
    for k, ln in enumerate(profile):
        if ln == 0:
            run += 1
        else:
            segs.append((run + (1 if segs else 0), int(ln)))
            run = 0
    return segs, run + (1 if segs else 0)


def model_warp(rays):
    """rays: list of (segs, tail).  -> (cost of K1's loop, useful work), in thread-instruction units / 32"""
    idx = [0] * len(rays)
    alive = [True] * len(rays)
    cost = useful = 0
    while any(alive):
        a_steps, b_len = [], []
        for r, (segs, tail) in enumerate(rays):
            if not alive[r]:
                continue
            if idx[r] < len(segs):
                a_steps.append(segs[idx[r]][0]); b_len.append(segs[idx[r]][1]); idx[r] += 1
                if idx[r] == len(segs) and tail == 0:
                    alive[r] = False
            else:
                a_steps.append(tail); b_len.append(0); alive[r] = False
        # a ray whose last occupied cell holds its hit ends there (profile ends with that cell: tail == 0)
        cost += C_ITER + max(a_steps) * C_DDA + max(b_len) * C_TEST
        useful += (sum(a_steps) * C_DDA + sum(b_len) * C_TEST) / 32.0
    return cost, useful


def model_pooled(rays, n_warps):
    """All rays of the strip advance in lock step; before each phase the pool is sorted by what the rays need next and
    dealt to n_warps warps of 32: each phase costs the sum over warps of their longest lane."""
    idx = [0] * len(rays)
    alive = [True] * len(rays)
    cost = 0
    while any(alive):
        a_steps, b_len = [], []
        for r, (segs, tail) in enumerate(rays):
            if not alive[r]:
                continue
            if idx[r] < len(segs):
                a_steps.append(segs[idx[r]][0]); b_len.append(segs[idx[r]][1]); idx[r] += 1
                if idx[r] == len(segs) and tail == 0:
                    alive[r] = False
            else:
                a_steps.append(tail); b_len.append(0); alive[r] = False
        for vals, c in ((sorted(a_steps, reverse=True), C_DDA), (sorted(b_len, reverse=True), C_TEST)):
            for k in range(0, len(vals), 32):
                cost += vals[k] * c
        cost += C_ITER * ((len(a_steps) + 31) // 32) + 40  # + a shared-memory exchange per phase pair
    return cost


def cull_model():
    """Phase B of K1's warp rounds with the screen cull: counts pair iterations, those every owning lane skips (pair
    box; per-triangle boxes), and the lane-level pair tests."""
    import screen_cull as sc
    pstart, a, b = sc.pair_records(ps)
    inv, k, ok = sc.camera_terms(cam32, fov_xs, aspect)
    org = cam32.reshape(-1)[12:15]
    ta, tb = sc.triangle_boxes(*a, org, inv, k, ok), sc.triangle_boxes(*b, org, inv, k, ok)
    pb = sc.pair_boxes(ta, tb).astype(np.float64)
    ta32, tb32 = sc.pair_boxes(ta, ta).astype(np.float64), sc.pair_boxes(tb, tb).astype(np.float64)
    print("pairs %d, never culled (whole plane) %.2f %%" % (len(pb), 100.0 * np.mean(np.isinf(pb[:, 0]) & (pb[:, 0] < 0))))
    ids = np.zeros(4096, np.uint32)
    cnt = dict(iters=0, skip_pair=0, skip_tri=0, lane_tests=0, lane_out=0)
    # --warp-scan: rounds, one-cell rounds, their chunks, pair iterations, and the pairs kept by footprint / per lane
    scan = dict(rounds=0, one_cell=0, chunks=0, iters_one=0, kept_fp=0, kept_lane=0, iters_after=0, checks_after=0,
                visits=0, visits_out=0)
    if SCAN:
        ncell = len(pstart) - 1
        cell_of = np.repeat(np.arange(ncell), np.diff(pstart))
        cb = np.empty((ncell, 4))
        cb[:, 0::2], cb[:, 1::2] = np.inf, -np.inf
        for q, fn in enumerate((np.minimum, np.maximum, np.minimum, np.maximum)):
            fn.at(cb[:, q], cell_of, pb[:, q])
    out = lambda box, j, x, y: (x < box[j, 0]) | (x > box[j, 1]) | (y < box[j, 2]) | (y > box[j, 3])
    n_x, n_y = w // sw, h // sh
    for _ in range(n_strips):
        bx, by = rs.randint(n_x) * sw, rs.randint(n_y) * sh
        lanes = []
        for slot in range(sw * sh):
            ox = (slot & 1) | ((slot >> 1) & 2) | ((slot >> 2) & 4)
            oy = ((slot >> 1) & 1) | ((slot >> 2) & 2)
            for s in range(spp):
                o, d = np.zeros(3, np.float32), np.zeros(3, np.float32)
                lib.rto_generate_ray(cam32.ctypes.data_as(F), bx + ox, by + oy, w, h, float(smp[s, 0]), float(smp[s, 1]),
                                     float(fov_xs), float(aspect), o.ctypes.data_as(F), d.ctypes.data_as(F))
                hit = C.c_int(0)
                n = study.rts_ray_walk_cells(C.byref(ps.s), o.ctypes.data_as(F), d.ctypes.data_as(F), len(ids),
                                             ids.ctypes.data_as(C.POINTER(C.c_uint32)), C.byref(hit))
                x, y = sc.image_point(bx + ox, by + oy, w, h, smp[s, 0], smp[s, 1], fov_xs, aspect)
                lanes.append((ids[:min(n, len(ids))].astype(np.int64).copy(), float(x), float(y)))
                if SCAN:
                    cells = lanes[-1][0]
                    scan["visits"] += len(cells)
                    scan["visits_out"] += int(((x < cb[cells, 0]) | (x > cb[cells, 1]) | (y < cb[cells, 2]) |
                                               (y > cb[cells, 3])).sum())
        for wbase in range(0, len(lanes), 32):
            warp = lanes[wbase:wbase + 32]
            xs = np.array([l[1] for l in warp])
            ys = np.array([l[2] for l in warp])
            for r in range(max(len(l[0]) for l in warp)):
                has = np.array([r < len(l[0]) for l in warp])
                cell = np.array([l[0][r] if r < len(l[0]) else 0 for l in warp])
                beg = pstart[cell]
                ln = np.where(has, pstart[cell + 1] - beg, 0)
                if SCAN and ln.max() > 0:
                    scan["rounds"] += 1
                    on = ln > 0
                    if len(set(beg[on])) == 1:
                        b0, n0 = int(beg[on][0]), int(ln.max())
                        sk = sc.footprint_skips(pb[b0:b0 + n0].astype(np.float32), xs[on], ys[on])
                        lane_in = ~out(pb, np.arange(b0, b0 + n0)[:, None], xs[on][None, :], ys[on][None, :])
                        assert not (sk & lane_in.any(1)).any()  # the footprint skips only pairs every lane skips
                        scan["one_cell"] += 1
                        scan["chunks"] += (n0 + 31) // 32
                        scan["iters_one"] += n0
                        scan["kept_fp"] += int((~sk).sum())
                        scan["kept_lane"] += int(lane_in.any(1).sum())
                        scan["iters_after"] += int((~sk).sum())
                        scan["checks_after"] += (n0 + 31) // 32
                    else:
                        scan["iters_after"] += int(ln.max())
                        scan["checks_after"] += int(ln.max())
                for i in range(int(ln.max())):
                    mine = i < ln
                    j = beg + np.minimum(i, np.maximum(ln - 1, 0))
                    op = out(pb, j, xs, ys)
                    ot = out(ta32, j, xs, ys) & out(tb32, j, xs, ys)
                    cnt["iters"] += 1
                    cnt["skip_pair"] += bool(np.all(~mine | op))
                    cnt["skip_tri"] += bool(np.all(~mine | ot))
                    cnt["lane_tests"] += int(mine.sum())
                    cnt["lane_out"] += int((mine & op).sum())
    fp, ft = cnt["skip_pair"] / cnt["iters"], cnt["skip_tri"] / cnt["iters"]
    print("%s: %d strips, %d warp pair-iterations" % (wl, n_strips, cnt["iters"]))
    print("skipped by the pair box %.1f %%, by per-triangle boxes %.1f %%; lane pair tests outside the pair box %.1f %%"
          % (100 * fp, 100 * ft, 100 * cnt["lane_out"] / cnt["lane_tests"]))
    # a skipped iteration saves ~37 issue slots, a kept one costs ~8 more (estimated from the r02 SASS)
    for name, f in (("pair box", fp), ("triangle boxes", ft)):
        print("  %s: net instructions saved per pair iteration %.1f (37 f - 8 (1 - f))" % (name, 37 * f - 8 * (1 - f)))
    if SCAN:
        c = scan
        print("warp scan: phase-B rounds %d, on one cell %d (%.1f %%); in those: %d pairs in %d chunks of 32, kept by the "
              "footprint %d (%.1f %%), by the per-lane check %d (%.1f %%)"
              % (c["rounds"], c["one_cell"], 100 * c["one_cell"] / c["rounds"], c["iters_one"], c["chunks"], c["kept_fp"],
                 100 * c["kept_fp"] / c["iters_one"], c["kept_lane"], 100 * c["kept_lane"] / c["iters_one"]))
        print("  warp pair iterations %d -> %d (%.1f %% fewer); box checks (serial: one per iteration) %d -> %d"
              % (cnt["iters"], c["iters_after"], 100 * (1 - c["iters_after"] / cnt["iters"]), cnt["iters"],
                 c["checks_after"]))
        print("  %d skipped iterations of %d remain (the serial walk of multi-cell rounds, and pairs the footprint keeps)"
              % (c["iters_after"] - (cnt["iters"] - cnt["skip_pair"]), c["iters_after"]))
        print("cell boxes (a phase-A alternative): lane occupied-cell visits outside the cell's box %d of %d (%.1f %%)"
              % (c["visits_out"], c["visits"], 100 * c["visits_out"] / c["visits"]))


if CULL:
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    cull_model()
    sys.exit(0)

tot = dict(k1=0.0, useful=0.0, pooled=0.0)
n_x, n_y = w // sw, h // sh
for _ in range(n_strips):
    bx, by = rs.randint(n_x) * sw, rs.randint(n_y) * sh
    rays = []
    for slot in range(sw * sh):  # Morton slot order of the strip's pixels, lanes sample-fastest (trace_kernels.cu)
        ox = (slot & 1) | ((slot >> 1) & 2) | ((slot >> 2) & 4)
        oy = ((slot >> 1) & 1) | ((slot >> 2) & 2)
        for s in range(spp):
            rays.append(segments(ray_profile(bx + ox, by + oy, s)))
    warps = [rays[k:k + 32] for k in range(0, len(rays), 32)]
    for wr in warps:
        c, u = model_warp(wr)
        tot["k1"] += c
        tot["useful"] += u
    tot["pooled"] += model_pooled(rays, len(warps))
print("%s: %d strips of %dx%d px x %d spp (%d rays)" % (wl, n_strips, sw, sh, spp, n_strips * sw * sh * spp))
print("modelled warp-instructions per ray: K1 loop %.0f   useful (perfect packing) %.0f   strip-pooled re-pairing %.0f"
      % (tot["k1"] * 32 / (n_strips * sw * sh * spp) / 32 * 32, tot["useful"] * 32 / (n_strips * sw * sh * spp),
         tot["pooled"] * 32 / (n_strips * sw * sh * spp)))
print("lane utilisation of the K1 loop %.1f %%; re-pairing within a strip would cut the loop by %.1f %%"
      % (100 * tot["useful"] / tot["k1"], 100 * (1 - tot["pooled"] / tot["k1"])))
