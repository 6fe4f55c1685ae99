"""Ray queries on GPU-resident rays (cuda_trace_query_rays, CudaTrace.query_rays): bit-exact against the oracle port's
walk (unbounded: rto_grid_intersect; bounded: tools/study rts_query_rays) and the old ray-batch entry point, in every
occupancy-map mode, for closest hit and occlusion; asynchrony, refusals and scene lifetime."""
import ctypes as C

import numpy as np
import pytest

from conftest import pkg
from test_ray_query_cpu import MISS, arbitrary_rays, box_rays, load_study, port_query, same_bits, t_max_around_hits

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def study(port):
    return load_study()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def host(out):
    if isinstance(out, tuple):
        tri, t, u, v = (x.cpu().numpy() for x in out)
        return tri.view(np.uint32), t, u, v
    return out.cpu().numpy()


def scene_rays(name, g):
    return arbitrary_rays(g) if name == "cornell" else box_rays(g)


CASES = [("cornell", 64), ("killeroo", 64), ("room", 64), ("tiger_soup_small", 150), ("tiger_soup_small", 48)]


@pytest.mark.parametrize("name,res", CASES)
def test_unbounded_closest_hit(cuda_trace, port, scene_data, name, res):
    sd = scene_data(name)
    cuda_trace.upload_scene(sd.vtx, sd.tri, res)
    ps = port.scene(sd.vtx, sd.tri, res, tight_ranges=True)
    o, d = scene_rays(name, ps.grid())
    for variant in (0, 1):
        got = host(cuda_trace.query_rays(dev(o), dev(d), variant=variant))
        torch.cuda.synchronize()
        assert same_bits(got, ps.intersect_rays(o, d, variant)), (name, res, variant)
        assert same_bits(got, cuda_trace.intersect_rays(o, d, variant)), (name, res, variant)
        assert (got[0] != MISS).sum() > len(o) // 20


@pytest.mark.parametrize("mode", ["0", "1", "2", "3"])
@pytest.mark.parametrize("name,res", [("killeroo", 64), ("tiger_soup_small", 150)])
def test_occupancy_map_modes(port, study, scene_data, monkeypatch, mode, name, res):
    """Every home of the occupancy map gives the same bits, bounded or not (switches are read once per context)"""
    monkeypatch.setenv("RTM_OCC_MODE", mode)
    sd = scene_data(name)
    ct = pkg("capi").CudaTrace(1)
    ct.upload_scene(sd.vtx, sd.tri, res)
    ps = port.scene(sd.vtx, sd.tri, res, tight_ranges=True)
    o, d = box_rays(ps.grid())
    for variant in (0, 1):
        want = ps.intersect_rays(o, d, variant)
        assert same_bits(host(ct.query_rays(dev(o), dev(d), variant=variant)), want), (mode, variant)
        tm = t_max_around_hits(want[1], want[0] != MISS)
        got = host(ct.query_rays(dev(o), dev(d), t_max=dev(tm), variant=variant))
        assert same_bits(got, port_query(study, ps, o, d, tm, variant)[:4]), (mode, variant)
        occ = host(ct.query_rays(dev(o), dev(d), t_max=dev(tm), occlusion=True, variant=variant))
        assert np.array_equal(occ, got[0] != MISS)
    ct.close()


@pytest.mark.parametrize("name,res", CASES)
def test_bounded_closest_hit_and_occlusion(cuda_trace, port, study, scene_data, name, res):
    sd = scene_data(name)
    cuda_trace.upload_scene(sd.vtx, sd.tri, res)
    ps = port.scene(sd.vtx, sd.tri, res, tight_ranges=True)
    o, d = scene_rays(name, ps.grid())
    do, dd = dev(o), dev(d)
    for variant in (0, 1):
        tri, t, _, _ = ps.intersect_rays(o, d, variant)
        tm = t_max_around_hits(t, tri != MISS)
        got = host(cuda_trace.query_rays(do, dd, t_max=dev(tm), variant=variant))
        want = port_query(study, ps, o, d, tm, variant)
        assert same_bits(got, want[:4]), (name, variant)
        occ = host(cuda_trace.query_rays(do, dd, t_max=dev(tm), occlusion=True, variant=variant))
        assert occ.dtype == np.bool_ and np.array_equal(occ, got[0] != MISS)
        # one bound for the whole batch
        for s in (float("inf"), 0.0, -1.0, float("nan"), float(np.median(t[tri != MISS]))):
            got = host(cuda_trace.query_rays(do, dd, t_max=s, variant=variant))
            assert same_bits(got, port_query(study, ps, o, d, s, variant)[:4]), (name, variant, s)
            occ = host(cuda_trace.query_rays(do, dd, t_max=s, occlusion=True, variant=variant))
            assert np.array_equal(occ, got[0] != MISS), (name, variant, s)
            if not s > 0:
                assert np.all(got[0] == MISS)
            if s == float("inf"):
                assert np.array_equal(occ, tri != MISS)


def test_shadow_rays_from_a_frame(cuda_trace, port, study, scene_data):
    """Killeroo 1080p, 1 spp: rays from a point light to every hit point of the frame, t_max just short of the point"""
    sd = scene_data("killeroo")
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    w, h = 1920, 1080
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    cuda_trace.trace_tiles(cuda_trace.make_frame(w, h, 1, sd.cam16, fov_xs, aspect, keep_hits=True), want_image=False)
    tri, t, u, v = (x.reshape(-1) for x in cuda_trace.download_hits(w, h, 1))
    hit = tri != MISS
    vtx, tris = np.asarray(sd.vtx, np.float32).reshape(-1, 6), np.asarray(sd.tri, np.uint32).reshape(-1, 6)
    corners = vtx[tris[tri[hit], :3], :3]  # [k, 3 vertices, xyz]
    p = (corners[:, 0] + u[hit, None] * (corners[:, 1] - corners[:, 0]) +
         v[hit, None] * (corners[:, 2] - corners[:, 0])).astype(np.float32)
    g = port.scene(sd.vtx, sd.tri, 64).grid()
    lo, hi = np.asarray(g["aabb_min"], np.float32), np.asarray(g["aabb_max"], np.float32)
    light = ((lo + hi) / 2 + np.array([0.3, 1.2, 0.4], np.float32) * (hi - lo)).astype(np.float32)
    o = np.broadcast_to(light, p.shape).astype(np.float32)
    dist = np.linalg.norm(p - o, axis=1).astype(np.float32)
    d = ((p - o) / dist[:, None]).astype(np.float32)
    tm = (dist * np.float32(0.999)).astype(np.float32)
    ps = port.scene(sd.vtx, sd.tri, 64)
    do, dd, dtm = dev(o), dev(d), dev(tm)
    for variant in (0, 1):
        occ = host(cuda_trace.query_rays(do, dd, t_max=dtm, occlusion=True, variant=variant))
        got = host(cuda_trace.query_rays(do, dd, t_max=dtm, variant=variant))
        assert same_bits(got, port_query(study, ps, o, d, tm, variant)[:4])
        assert np.array_equal(occ, got[0] != MISS)
        frac = occ.mean()
        print("variant %d: %.1f %% of %d shadow rays occluded" % (variant, 100 * frac, len(o)))
        assert 0.0 < frac < 1.0


@pytest.mark.parametrize("n", [0, 1, 31, 33, (1 << 20) + 7])
def test_batch_sizes(cuda_trace, port, study, scene_data, n):
    sd = scene_data("room")
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    ps = port.scene(sd.vtx, sd.tri, 64)
    o, d = box_rays(ps.grid(), max(n, 1), seed=n)
    o, d = o[:n], d[:n]
    tm = np.random.RandomState(n).uniform(0.5, 4.0, n).astype(np.float32)
    got = host(cuda_trace.query_rays(dev(o), dev(d), variant=0))
    assert all(len(x) == n for x in got)
    assert same_bits(got, ps.intersect_rays(o, d, 0))
    got = host(cuda_trace.query_rays(dev(o), dev(d), t_max=dev(tm), variant=1))
    assert same_bits(got, port_query(study, ps, o, d, tm, 1)[:4])
    occ = host(cuda_trace.query_rays(dev(o), dev(d), t_max=dev(tm), occlusion=True, variant=1))
    assert np.array_equal(occ, got[0] != MISS)


def test_query_on_a_busy_side_stream_does_not_wait(cuda_trace, port, scene_data):
    sd = scene_data("killeroo")
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    ps = port.scene(sd.vtx, sd.tri, 64)
    o, d = box_rays(ps.grid(), 200000)
    do, dd = dev(o), dev(d)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(500_000_000)  # ~0.25 s of spinning ahead of the query
    out = cuda_trace.query_rays(do, dd, stream=side)
    assert not side.query(), "the query call waited for its stream"
    side.synchronize()
    assert same_bits(host(out), ps.intersect_rays(o, d, 0))


def test_refusals_enqueue_nothing(cuda_trace, port, scene_data):
    capi = pkg("capi")
    sd = scene_data("cornell")
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    o, d = arbitrary_rays(port.scene(sd.vtx, sd.tri, 64).grid())
    do, dd = dev(o), dev(d)
    n = len(o)
    tri = torch.full((n,), 7, dtype=torch.int32, device="cuda")
    occ = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    host_tri = np.zeros(n, np.uint32)
    lib = cuda_trace.lib

    def batch(kind=0, variant=0, tri_ptr=tri.data_ptr(), occ_ptr=None, origins=do.data_ptr()):
        b = capi.RayBatch()
        b.n, b.kind, b.variant, b.t_max_all = n, kind, variant, float("inf")
        b.origins, b.dirs, b.tri_idx, b.occluded = origins, dd.data_ptr(), tri_ptr, occ_ptr
        return b

    torch.cuda.synchronize()
    launches = cuda_trace.kernel_launches()
    cases = [batch(tri_ptr=host_tri.ctypes.data),              # CPU output pointer
             batch(origins=o.ctypes.data),                     # CPU input pointer
             batch(variant=0x100),                             # MAILBOX
             batch(variant=2),                                 # no such variant
             batch(kind=2),                                    # no such kind
             batch(tri_ptr=None),                              # closest hit without tri_idx
             batch(kind=1, tri_ptr=None, occ_ptr=None)]        # occlusion without occluded
    for b in cases:
        assert lib.cuda_trace_query_rays(cuda_trace.h, C.byref(b), None) == 1
        assert lib.cuda_trace_last_error(cuda_trace.h)
    fresh = capi.CudaTrace(1)
    assert lib.cuda_trace_query_rays(fresh.h, C.byref(batch()), None) == 4  # no scene
    fresh.close()
    torch.cuda.synchronize()
    assert cuda_trace.kernel_launches() == launches
    assert bool((tri == 7).all()) and bool((occ == 7).all())
    # the Python binding refuses before the C call
    with pytest.raises(ValueError):
        cuda_trace.query_rays(torch.from_numpy(o), dd)
    with pytest.raises(TypeError):
        cuda_trace.query_rays(do.double(), dd)
    with pytest.raises(ValueError):
        cuda_trace.query_rays(do, dd, t_max=dev(np.ones(n + 1)))
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            cuda_trace.query_rays(do.to("cuda:1"), dd)
    # and a valid query still works
    b = batch()
    assert lib.cuda_trace_query_rays(cuda_trace.h, C.byref(b), None) == 0
    assert lib.cuda_trace_query_rays(cuda_trace.h, C.byref(batch(kind=1, tri_ptr=None, occ_ptr=occ.data_ptr())), None) == 0
    cuda_trace.sync()
    want = cuda_trace.intersect_rays(o, d, 0)[0]
    assert np.array_equal(tri.cpu().numpy().view(np.uint32), want)
    assert np.array_equal(occ.cpu().numpy(), (want != MISS).astype(np.uint8))


def test_scene_replacement_waits_for_pending_queries(port, scene_data):
    """Replacing the scene right after enqueueing a large query on a busy side stream leaves that query reading the
    first scene's arrays until it is done"""
    a, b = scene_data("killeroo"), scene_data("cornell")
    ct = pkg("capi").CudaTrace(1)
    ct.upload_scene(a.vtx, a.tri, 64)
    ps = port.scene(a.vtx, a.tri, 64)
    o, d = box_rays(ps.grid(), 1 << 20)
    want = ps.intersect_rays(o, d, 0)
    do, dd = dev(o), dev(d)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(500_000_000)
    out = ct.query_rays(do, dd, stream=side)
    ct.upload_scene(b.vtx, b.tri, 64)
    side.synchronize()
    assert same_bits(host(out), want)
    ct.close()
