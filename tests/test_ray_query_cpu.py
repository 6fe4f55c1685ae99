"""CPU checks of the ray-query semantics (include/cuda_trace.h, cuda_trace_query_rays): the bounded walk's restatement
(tools/study/rt_study.c, rts_query_rays) on top of the oracle port, the ctypes mirror of the batch struct, and the
refusals that need no device.  tests/test_gpu_ray_query.py compares the device with the same restatement."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, pkg

F = C.POINTER(C.c_float)
U32 = C.POINTER(C.c_uint32)
U8 = C.POINTER(C.c_uint8)
MISS = 0xFFFFFFFF
SCENES = [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, "tiger_soup_small"]


def load_study():
    d = os.path.join(ROOT, "tools", "study")
    subprocess.check_call(["bash", os.path.join(d, "build.sh")])
    lib = C.CDLL(os.path.join(d, "librt_study.so"))
    lib.rts_query_rays.restype = None
    lib.rts_query_rays.argtypes = [C.c_void_p, C.c_uint32, F, F, F, C.c_float, C.c_int, U32, F, F, F, U8]
    return lib


def port_query(study, ps, o, d, t_max, variant):
    """Bounded closest hit on the port: t_max a float (every ray) or an (n,) array.
    -> (tri, t, u, v, stopped by rule 2)"""
    o = np.ascontiguousarray(o, np.float32)
    d = np.ascontiguousarray(d, np.float32)
    n = len(o)
    per_ray = isinstance(t_max, np.ndarray)
    tm = np.ascontiguousarray(t_max, np.float32) if per_ray else None
    tri = np.empty(n, np.uint32)
    t, u, v = (np.empty(n, np.float32) for _ in range(3))
    stopped = np.empty(n, np.uint8)
    study.rts_query_rays(C.byref(ps.s), n, o.ctypes.data_as(F), d.ctypes.data_as(F),
                         tm.ctypes.data_as(F) if per_ray else None, float("inf") if per_ray else float(t_max),
                         variant, tri.ctypes.data_as(U32), t.ctypes.data_as(F), u.ctypes.data_as(F),
                         v.ctypes.data_as(F), stopped.ctypes.data_as(U8))
    return tri, t, u, v, stopped.astype(bool)


def arbitrary_rays(g, n=20000, seed=7):
    """The ray set of test_gpu_parity.py::test_arbitrary_rays, scaled to the grid's box: axis-aligned and planar
    directions, origins inside the box, on its faces and behind it, unnormalised directions."""
    rs = np.random.RandomState(seed)
    lo, hi = np.asarray(g["aabb_min"], np.float32), np.asarray(g["aabb_max"], np.float32)
    c, h = (lo + hi) / 2, (hi - lo) / 2
    o = (c + rs.uniform(-1.5, 1.5, (n, 3)) * 2 * h).astype(np.float32)
    d = rs.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True).astype(np.float32)
    d[:3000, 0] = 0.0
    d[1000:4000, 1] = 0.0
    d[4000:4600] = np.eye(3, dtype=np.float32)[rs.randint(0, 3, 600)] * rs.choice([-1, 1], (600, 1))
    d[4600:4700, 2] = -0.0
    o[5000:9000] = (c + rs.uniform(-0.9, 0.9, (4000, 3)) * h).astype(np.float32)
    o[9000:9300, 0] = lo[0]
    o[9300:9600, 1] = hi[1]
    d[9600:10000] *= rs.uniform(0.1, 10, (400, 1)).astype(np.float32)
    keep = np.abs(d).sum(axis=1) > 0
    return o[keep], d[keep]


def box_rays(g, n=30000, seed=11):
    """The ray set of test_gpu_parity.py::test_mailboxing_mode: origins mostly outside the box, aimed at points in it."""
    rs = np.random.RandomState(seed)
    lo, hi = np.asarray(g["aabb_min"], np.float32), np.asarray(g["aabb_max"], np.float32)
    o = (rs.uniform(-1.0, 1.0, (n, 3)) * 2.0 * (hi - lo) + (lo + hi) / 2).astype(np.float32)
    target = rs.uniform(lo, hi, (n, 3)).astype(np.float32)
    d = target - o
    d /= np.linalg.norm(d, axis=1, keepdims=True).astype(np.float32)
    return o, d


def t_max_around_hits(t_hit, hit, seed=3):
    """Per-ray bounds drawn around each ray's hit parameter (misses get a bound of the same spread).  The first 30 %
    sit exactly at the hit or one ulp either side of it, where the rule-2 corner lives; the rest are uniform in
    [0.5, 1.5] times the hit parameter."""
    rs = np.random.RandomState(seed)
    scale = np.where(hit, t_hit, np.median(t_hit[hit]) if hit.any() else 1.0).astype(np.float32)
    tm = (scale * rs.uniform(0.5, 1.5, len(t_hit))).astype(np.float32)
    # a share exactly at the hit and one ulp either side
    k = len(tm) // 10
    tm[:k] = t_hit[:k]
    tm[k:2 * k] = np.nextafter(t_hit[k:2 * k], np.float32(np.inf))
    tm[2 * k:3 * k] = np.nextafter(t_hit[2 * k:3 * k], np.float32(0))
    return np.where(hit | (np.arange(len(tm)) >= 3 * k), tm, scale).astype(np.float32)


def same_bits(a, b):
    return all(np.array_equal(np.asarray(x).view(np.uint32), np.asarray(y).view(np.uint32)) for x, y in zip(a, b))


@pytest.fixture(scope="module")
def study(port):
    return load_study()


@pytest.mark.parametrize("name", SCENES)
def test_unbounded_walk_is_grid_intersect(study, port, scene_data, name):
    """t_max = +inf: the bounded walk is rto_grid_intersect (pinned to the reference's Grid::Intersect) bit for bit"""
    sd = scene_data(name)
    res = 48 if name == "tiger_soup_small" else 64
    ps = port.scene(sd.vtx, sd.tri, res, tight_ranges=True)
    g = ps.grid()
    for o, d in (arbitrary_rays(g), box_rays(g)):
        for variant in (0, 1):
            want = ps.intersect_rays(o, d, variant)
            got = port_query(study, ps, o, d, float("inf"), variant)
            assert same_bits(got[:4], want), (name, variant)
            assert not got[4].any()


@pytest.mark.parametrize("name", SCENES)
def test_bounded_walk_against_clipped_unbounded_hit(study, port, scene_data, name):
    """Against "the unbounded hit, kept if t < t_max" the bounded walk differs only in the documented corner: a miss
    decided by rule 2 where the unbounded walk found its triangle at t < t_max in a cell entered after t_max."""
    sd = scene_data(name)
    res = 48 if name == "tiger_soup_small" else 64
    ps = port.scene(sd.vtx, sd.tri, res, tight_ranges=True)
    g = ps.grid()
    total = differ = adjacent = 0
    for o, d in (arbitrary_rays(g), box_rays(g)):
        for variant in (0, 1):
            tri, t, u, v = ps.intersect_rays(o, d, variant)
            hit = tri != MISS
            tm = t_max_around_hits(t, hit)
            keep = hit & (t < tm)
            want = (np.where(keep, tri, MISS), np.where(keep, t, 0), np.where(keep, u, 0), np.where(keep, v, 0))
            btri, bt, bu, bv, stopped = port_query(study, ps, o, d, tm, variant)
            diff = ~((btri == want[0]) & (bt.view(np.uint32) == want[1].astype(np.float32).view(np.uint32)) &
                     (bu.view(np.uint32) == want[2].astype(np.float32).view(np.uint32)) &
                     (bv.view(np.uint32) == want[3].astype(np.float32).view(np.uint32)))
            # every difference: the bounded walk stopped by rule 2, the unbounded hit lies below t_max
            assert np.all(stopped[diff] & keep[diff] & (btri[diff] == MISS)), (name, variant)
            near = np.arange(len(o)) < 3 * (len(o) // 10)  # bounds at the hit or one ulp from it
            total += int((~near).sum())
            differ += int(diff[~near].sum())
            adjacent += int(diff[near].sum())
            # per-ray bounds and one bound for the batch agree
            one = port_query(study, ps, o[:2000], d[:2000], float(np.median(tm)), variant)
            per = port_query(study, ps, o[:2000], d[:2000], np.full(2000, np.median(tm), np.float32), variant)
            assert same_bits(one[:4], per[:4])
    print("%s: %d of %d bounded queries with t_max drawn around the hit differ from the clipped unbounded hit, and %d "
          "with t_max within one ulp of it (all in the rule-2 corner)" % (name, differ, total, adjacent))
    assert differ <= total * 1e-4


def test_nonpositive_and_nan_bounds_miss(study, port, scene_data):
    sd = scene_data("cornell")
    ps = port.scene(sd.vtx, sd.tri, 64)
    o, d = arbitrary_rays(ps.grid())
    for tm in (0.0, -0.0, -1.0, float("nan")):
        tri = port_query(study, ps, o, d, tm, 0)[0]
        assert np.all(tri == MISS), tm


def test_ray_batch_struct_matches_header(tmp_path):
    """capi.RayBatch has the size and field offsets of cuda_trace_ray_batch as a C compiler lays it out"""
    capi = pkg("capi")
    src = tmp_path / "layout.c"
    fields = [f for f, _ in capi.RayBatch._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "cuda_trace.h"\nint main(void){printf("%zu'
                   + "".join(" %zu" for _ in fields) + '\\n", sizeof(cuda_trace_ray_batch)'
                   + "".join(", offsetof(cuda_trace_ray_batch, %s)" % f for f in fields) + ");return 0;}\n")
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", "-I" + os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got[0] == C.sizeof(capi.RayBatch)
    assert got[1:] == [getattr(capi.RayBatch, f).offset for f in fields]
    assert capi.QUERY_CLOSEST == 0 and capi.QUERY_OCCLUSION == 1


def test_query_refuses_null_context_and_batch_without_a_device():
    capi = pkg("capi")
    lib = capi.load_library()
    b = capi.RayBatch()
    assert lib.cuda_trace_query_rays(None, None, None) == 1
    assert lib.cuda_trace_query_rays(None, C.byref(b), None) == 1
