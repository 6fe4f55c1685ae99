"""Scenes uploaded from GPU-resident meshes (cuda_trace_upload_scene_device, CudaTrace.upload_scene_device): the grid,
the distance map, frames and ray queries are the host upload's bit for bit; the call orders itself after the
producer's stream, lets the caller reuse its tensors at once, leaks nothing across rebuilds, refuses bad input
without touching the previous scene, waits for pending queries, and replicates to a second device."""
import ctypes as C

import numpy as np
import pytest

from conftest import pkg
from test_ray_query_cpu import MISS, box_rays, same_bits, t_max_around_hits

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

PRESETS = ["torusknot", "cornell", "room", "table_chair", "head", "room_cat", "water_knot", "griebel_teapot",
           "killeroo", "dwarf_hand_blob"]
GRID_KEYS = ("dim", "aabb_min", "aabb_max", "cell_wdh", "inv_cell_wdh", "cell_offset", "tri_index")
F32P, U32P = C.POINTER(C.c_float), C.POINTER(C.c_uint32)


@pytest.fixture(scope="module")
def two_gpus():
    if pkg("capi").load_library().cuda_trace_device_count() < 2:
        pytest.skip("needs 2 GPUs")


@pytest.fixture(scope="module")
def contexts():
    """(host-path context, device-path context)"""
    capi = pkg("capi")
    a, b = capi.CudaTrace(1), capi.CudaTrace(1)
    yield a, b
    a.close()
    b.close()


def on_gpu(vtx, tri):
    """The Mesh arrays as CUDA tensors: float32 (V, 6) and int32 (T, 6)"""
    return (torch.from_numpy(np.ascontiguousarray(vtx, np.float32)).cuda(),
            torch.from_numpy(np.ascontiguousarray(tri, np.uint32).view(np.int32)).cuda())


def on_host(v, t):
    return v.cpu().numpy(), t.cpu().numpy().view(np.uint32)


def same_grid(a, b):
    """Two grids (download_grid dicts) hold the same bytes"""
    for k in GRID_KEYS:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes(), k


def same_scene(ca, cb):
    """Two contexts hold the same grid and the same distance map"""
    same_grid(ca.download_grid(), cb.download_grid())
    da, db = ca.download_distance_map(), cb.download_distance_map()
    assert (da is None) == (db is None)
    assert da is None or da.tobytes() == db.tobytes()


def frame(ct, port, sd, w, h, spp, **kw):
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    return ct.make_frame(w, h, spp, sd.cam16, fov_xs, aspect, **kw)


def render(ct, port, sd, w, h, spp, variant=0):
    """-> (image, per-sample hit records)"""
    img = ct.trace_tiles(frame(ct, port, sd, w, h, spp, variant=variant, keep_hits=True))
    return img, ct.download_hits(w, h, spp)


def queries(ct, o, d, tm):
    """Closest hit and occlusion, unbounded and bounded by the per-ray tm, on host copies"""
    out = []
    for t_max in (None, tm):
        for occlusion in (False, True):
            r = ct.query_rays(o, d, t_max=t_max, occlusion=occlusion)
            out.append(r.cpu().numpy() if occlusion else tuple(x.cpu().numpy() for x in r))
    return out


def same_queries(a, b):
    for x, y in zip(a, b):
        if isinstance(x, tuple):
            assert same_bits(x, y)
        else:
            assert np.array_equal(x, y)


def query_set(ct, n=30000):
    """Rays through the box of ct's scene and per-ray bounds around their hits"""
    o, d = box_rays(ct.download_grid(), n)
    do, dd = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    tri, t, _, _ = ct.query_rays(do, dd)
    tm = t_max_around_hits(t.cpu().numpy(), tri.cpu().numpy() != -1)
    return do, dd, torch.from_numpy(tm).cuda()


@pytest.mark.parametrize("name,res", [(n, 64) for n in PRESETS] + [("tiger_soup_small", 64), ("tiger_soup_small", 150)])
def test_grid_is_the_host_paths(contexts, port, scene_data, name, res):
    host_ct, dev_ct = contexts
    sd = scene_data(name)
    host_ct.upload_scene(sd.vtx, sd.tri, res)
    dev_ct.upload_scene_device(*on_gpu(sd.vtx, sd.tri), grid_res=res)
    same_scene(host_ct, dev_ct)
    if res == 150:
        assert dev_ct.download_distance_map() is not None
    if name in ("cornell", "killeroo", "tiger_soup_small"):
        same_grid(dev_ct.download_grid(), port.scene(sd.vtx, sd.tri, res, tight_ranges=True).grid())


def test_uint32_triangles_and_explicit_current_stream(contexts, scene_data):
    host_ct, dev_ct = contexts
    sd = scene_data("cornell")
    host_ct.upload_scene(sd.vtx, sd.tri, 64)
    v, t = on_gpu(sd.vtx, sd.tri)
    dev_ct.upload_scene_device(v, t.view(torch.uint32), 64, stream=torch.cuda.current_stream())
    same_scene(host_ct, dev_ct)


@pytest.mark.parametrize("variant", [0, 1])
def test_frames_are_the_host_paths(contexts, port, scene_data, variant):
    host_ct, dev_ct = contexts
    sd = scene_data("killeroo")
    host_ct.upload_scene(sd.vtx, sd.tri, 64)
    dev_ct.upload_scene_device(*on_gpu(sd.vtx, sd.tri), grid_res=64)
    (ia, ha), (ib, hb) = (render(ct, port, sd, 320, 180, 4, variant) for ct in (host_ct, dev_ct))
    assert np.array_equal(ia, ib)
    assert same_bits(ha, hb)
    assert (ha[0] != MISS).mean() > 0.1


def test_pooled_frame_is_the_host_paths(contexts, port, scene_data):
    """tiger_soup_small at res 150 has a distance map, so its frames take the pooled-ray traversal"""
    host_ct, dev_ct = contexts
    sd = scene_data("tiger_soup_small")
    host_ct.upload_scene(sd.vtx, sd.tri, 150)
    dev_ct.upload_scene_device(*on_gpu(sd.vtx, sd.tri), grid_res=150)
    f = frame(host_ct, port, sd, 320, 180, 4)
    img = host_ct.trace_tiles(f)
    assert np.array_equal(img, dev_ct.trace_tiles(f))


def test_queries_are_the_host_paths(contexts, scene_data):
    host_ct, dev_ct = contexts
    sd = scene_data("killeroo")
    host_ct.upload_scene(sd.vtx, sd.tri, 64)
    dev_ct.upload_scene_device(*on_gpu(sd.vtx, sd.tri), grid_res=64)
    o, d, tm = query_set(host_ct)
    a, b = queries(host_ct, o, d, tm), queries(dev_ct, o, d, tm)
    same_queries(a, b)
    assert 0 < (a[0][0] != -1).sum() and 0 < a[3].sum() < len(tm)


def test_upload_waits_for_the_producer_stream(contexts, scene_data):
    """The final vertex values are written on a side stream behind ~0.25 s of spinning, and the call gets no host
    synchronisation: the grid must still be the one of the final values"""
    host_ct, dev_ct = contexts
    sd = scene_data("killeroo")
    v0, t = on_gpu(sd.vtx, sd.tri)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        v = v0.clone()
        torch.cuda._sleep(500_000_000)
        v[:, :3] *= 1.75
        v[:, 1] += 0.5
    dev_ct.upload_scene_device(v, t, 64, stream=side)
    assert side.query(), "the call returned before the producer's work was done"
    host_ct.upload_scene(*on_host(v, t), 64)
    same_scene(host_ct, dev_ct)


def test_caller_buffers_may_be_reused_at_once(contexts, port, scene_data):
    host_ct, dev_ct = contexts
    sd = scene_data("killeroo")
    host_ct.upload_scene(sd.vtx, sd.tri, 64)
    v, t = on_gpu(sd.vtx, sd.tri)
    dev_ct.upload_scene_device(v, t, 64)
    v.fill_(float("nan"))
    t.zero_()
    del v, t
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    junk = torch.full((1 << 22,), -1, dtype=torch.int32, device="cuda")  # takes the freed memory, if anything would
    (ia, ha), (ib, hb) = (render(ct, port, sd, 256, 144, 4) for ct in (host_ct, dev_ct))
    assert np.array_equal(ia, ib) and same_bits(ha, hb)
    o, d, tm = query_set(host_ct)
    same_queries(queries(host_ct, o, d, tm), queries(dev_ct, o, d, tm))
    del junk


def test_dynamic_scene(contexts, scene_data):
    """20 steps of deform on the GPU -> device upload -> query; compared with the host upload of the same arrays at
    steps 0, 7 and 19, and no device memory is lost per rebuild"""
    host_ct, dev_ct = contexts
    sd = scene_data("killeroo")
    base, t = on_gpu(sd.vtx, sd.tri)
    host_ct.upload_scene(sd.vtx, sd.tri, 64)
    o, d, tm = query_set(host_ct, 20000)
    free = []
    for step in range(20):
        v = base.clone()
        p = v[:, :3]
        p += 0.05 * torch.sin(3.0 * p[:, [1, 2, 0]] + 0.4 * step)
        dev_ct.upload_scene_device(v, t, 64)
        got = queries(dev_ct, o, d, tm)
        if step in (0, 7, 19):
            host_ct.upload_scene(*on_host(v, t), 64)
            same_scene(host_ct, dev_ct)
            same_queries(got, queries(host_ct, o, d, tm))
        torch.cuda.synchronize()
        free.append(torch.cuda.mem_get_info()[0])
    # from step 2 on every allocation of a step has a same-sized predecessor
    assert min(free[2:]) >= free[2] - (16 << 20), [f >> 20 for f in free]


def test_refusals_leave_the_previous_scene(contexts, port, scene_data):
    capi = pkg("capi")
    host_ct, dev_ct = contexts
    lib = dev_ct.lib
    sd = scene_data("killeroo")
    v, t = on_gpu(sd.vtx, sd.tri)
    dev_ct.upload_scene_device(v, t, 64)
    o, d, tm = query_set(dev_ct, 20000)
    want_q = queries(dev_ct, o, d, tm)
    want_img, want_hits = render(dev_ct, port, sd, 256, 144, 4)
    nv, nt = v.shape[0], t.shape[0]
    vp, tp = C.cast(v.data_ptr(), F32P), C.cast(t.data_ptr(), U32P)
    hv, ht = np.ascontiguousarray(sd.vtx, np.float32), np.ascontiguousarray(sd.tri, np.uint32)

    def records_to_allocation_end(ptr):
        for seg in torch.cuda.memory_snapshot():
            if seg["address"] <= ptr < seg["address"] + seg["total_size"]:
                return (seg["address"] + seg["total_size"] - ptr) // 24
        raise AssertionError("no caching-allocator segment holds the tensor")

    n_refused = [0]

    def refused(*args, says):
        n_refused[0] += 1
        assert lib.cuda_trace_upload_scene_device(dev_ct.h, *args, None) == 1, says
        msg = lib.cuda_trace_last_error(dev_ct.h).decode()
        assert says in msg, msg
        same_queries(queries(dev_ct, o, d, tm), want_q)

    torch.cuda.synchronize()
    launches = dev_ct.kernel_launches()
    refused(hv.ctypes.data_as(F32P), len(hv), ht.ctypes.data_as(U32P), len(ht), 64, says="not device memory")
    refused(vp, nv, ht.ctypes.data_as(U32P), len(ht), 64, says="triangles is not device memory")
    refused(None, nv, tp, nt, 64, says="empty mesh")
    refused(vp, nv, None, nt, 64, says="empty mesh")
    refused(vp, 0, tp, nt, 64, says="empty mesh")
    refused(vp, nv, tp, 0, 64, says="empty mesh")
    refused(vp, nv, tp, nt, 0, says="grid_res")
    refused(C.cast(v.data_ptr() + 2, F32P), nv, tp, nt, 64, says="vertices is not 4-byte aligned")
    refused(vp, nv, C.cast(t.data_ptr() + 1, U32P), nt, 64, says="triangles is not 4-byte aligned")
    refused(vp, records_to_allocation_end(v.data_ptr()) + 1, tp, nt, 64, says="vertices records")
    refused(vp, nv, tp, records_to_allocation_end(t.data_ptr()) + 1, 64, says="triangles records")
    refused(vp, 0xFFFFFFFF, tp, nt, 64, says="run past the end of their allocation")
    # only the four queries after each refusal were launched: the refused uploads enqueued nothing
    assert dev_ct.kernel_launches() == launches + 4 * n_refused[0]

    bad = t.clone()
    bad[nt // 2, 1] = nv           # index == num_vertices, in the middle
    bad[nt - 3, 0] = nv + 7        # a later one: the message names the lowest
    refused(vp, nv, C.cast(bad.data_ptr(), U32P), nt, 64, says="triangle %d " % (nt // 2))
    with pytest.raises(capi.CudaTraceError) as e:
        dev_ct.upload_scene_device(v, bad, 64)
    assert e.value.code == 1 and "triangle %d " % (nt // 2) in str(e.value)
    # the binding refuses before the C call
    with pytest.raises(ValueError):
        dev_ct.upload_scene_device(v.cpu(), t, 64)
    with pytest.raises(TypeError):
        dev_ct.upload_scene_device(v.double(), t, 64)
    with pytest.raises(TypeError):
        dev_ct.upload_scene_device(v, t.long(), 64)
    with pytest.raises(ValueError):
        dev_ct.upload_scene_device(v[:, :3], t, 64)
    with pytest.raises(ValueError):
        dev_ct.upload_scene_device(v, t[:0], 64)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            dev_ct.upload_scene_device(v.to("cuda:1"), t, 64)
    img, hits = render(dev_ct, port, sd, 256, 144, 4)
    assert np.array_equal(img, want_img) and same_bits(hits, want_hits)
    same_queries(queries(dev_ct, o, d, tm), want_q)


def test_scene_replacement_waits_for_pending_queries(port, scene_data):
    """Replacing the scene through the device path right after enqueueing a large query on a busy side stream leaves
    that query reading the first scene's arrays until it is done"""
    a, b = scene_data("killeroo"), scene_data("cornell")
    ct = pkg("capi").CudaTrace(1)
    ct.upload_scene_device(*on_gpu(a.vtx, a.tri), grid_res=64)
    ps = port.scene(a.vtx, a.tri, 64)
    o, d = box_rays(ps.grid(), 1 << 20)
    want = ps.intersect_rays(o, d, 0)
    do, dd = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    vb, tb = on_gpu(b.vtx, b.tri)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        torch.cuda._sleep(500_000_000)
    out = ct.query_rays(do, dd, stream=side)
    ct.upload_scene_device(vb, tb, 64)
    side.synchronize()
    tri, t, u, v = (x.cpu().numpy() for x in out)
    assert same_bits((tri.view(np.uint32), t, u, v), want)
    ct.close()


def test_two_devices(two_gpus, port, scene_data):
    """Device 1 gets its arrays from device 0's copy: its strips of the frame must be the single-GPU frame's"""
    capi = pkg("capi")
    sd = scene_data("killeroo")
    w, h, spp = 320, 180, 16
    one = capi.CudaTrace(1)
    one.upload_scene(sd.vtx, sd.tri, 64)
    want = render(one, port, sd, w, h, spp)
    one.close()
    two = capi.CudaTrace(2)
    two.upload_scene_device(*on_gpu(sd.vtx, sd.tri), grid_res=64)
    got = render(two, port, sd, w, h, spp)
    two.close()
    assert np.array_equal(got[0], want[0]) and same_bits(got[1], want[1])
