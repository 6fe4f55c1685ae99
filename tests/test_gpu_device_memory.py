"""The tracer library gives back the device memory it takes: a context that uploads scenes three ways, renders, answers
ray and sampling queries and is destroyed leaves free device memory where it found it, calling an entry point again
does not take more, and refused uploads take nothing.  The library allocates outside torch's caching allocator, so
its memory shows in torch.cuda.mem_get_info().  Sizes stay small: killeroo at 64^3, frames of at most 1080p."""
import numpy as np
import pytest

from conftest import pkg
from test_ray_query_cpu import box_rays

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

SLACK = 2 << 20  # bytes


def free_bytes():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return torch.cuda.mem_get_info()[0]


@pytest.fixture(scope="module")
def steps(port, scene_data):
    """(name, call(ct)) for every entry point that allocates, in the order of one cycle"""
    capi = pkg("capi")
    sd = scene_data("killeroo")
    ct = capi.CudaTrace(1)
    ct.upload_scene(sd.vtx, sd.tri, 64)
    grid = ct.download_grid()
    ct.close()
    v = torch.from_numpy(np.ascontiguousarray(sd.vtx, np.float32)).cuda()
    t = torch.from_numpy(np.ascontiguousarray(sd.tri, np.uint32).view(np.int32)).cuda()
    o, d = box_rays(grid, 20000)
    do, dd = torch.from_numpy(o).cuda(), torch.from_numpy(d).cuda()
    x = np.random.RandomState(5).uniform(0.0, 1.0, 10000)

    def frame(w, h, spp, keep_hits):
        fov_xs, aspect = port.camera_constants(sd.fov, w, h)
        return capi.CudaTrace.make_frame(w, h, spp, sd.cam16, fov_xs, aspect, keep_hits=keep_hits)

    small, large = frame(320, 180, 4, True), frame(1920, 1080, 8, False)  # large: origin-relative records, screen boxes

    def render(ct):
        ct.trace_tiles(small)
        ct.download_hits(320, 180, 4)
        ct.trace_tiles(large)

    return [
        ("upload_scene", lambda ct: ct.upload_scene(sd.vtx, sd.tri, 64)),
        ("upload_scene_with_grid", lambda ct: ct.upload_scene_with_grid(sd.vtx, sd.tri, grid)),
        ("upload_scene_device", lambda ct: ct.upload_scene_device(v, t, 64)),
        ("frames", render),
        ("intersect_rays", lambda ct: ct.intersect_rays(o, d)),
        ("intersect_rays mailbox", lambda ct: ct.intersect_rays(o, d, mailbox=True)),
        ("intersect_rays_brute_force", lambda ct: ct.intersect_rays_brute_force(o[:2000], d[:2000])),
        ("query_rays", lambda ct: ct.query_rays(do, dd)),
        ("ray_march", lambda ct: ct.ray_march(o[:2000], d[:2000])),
        ("sample_table", lambda ct: ct.sample_table(16)),
        ("qmc_sequence", lambda ct: ct.qmc_sequence("halton", 0, 4096, 0, 8, scramble="faure")),
        ("qmc_cranley_patterson", lambda ct: ct.qmc_cranley_patterson(x, 0.3)),
        ("download_grid", lambda ct: ct.download_grid()),
    ]


def cycle(steps, repeats=1):
    """Create a context, run every step `repeats` times, destroy it.  -> {step: free bytes after each call}"""
    ct = pkg("capi").CudaTrace(1)
    after = {}
    for name, call in steps:
        after[name] = []
        for _ in range(repeats):
            call(ct)
            after[name].append(free_bytes())
    ct.close()
    return after


def test_a_second_cycle_gives_back_what_it_takes(steps):
    cycle(steps)  # warm-up: modules, the driver's own set-up
    start = free_bytes()
    cycle(steps)
    end = free_bytes()
    assert end >= start - SLACK, "%.1f MB lost" % ((start - end) / 2 ** 20)


def test_calls_again_take_no_more(steps):
    cycle(steps)
    after = cycle(steps, repeats=6)
    lost = {name: (f[0] - min(f[1:])) / 2 ** 20 for name, f in after.items() if min(f[1:]) < f[0] - SLACK}
    assert not lost, "MB lost over five more calls: %s" % lost


def test_refused_device_uploads_take_nothing(scene_data):
    capi = pkg("capi")
    sd = scene_data("killeroo")
    v = torch.from_numpy(np.ascontiguousarray(sd.vtx, np.float32)).cuda()
    t = torch.from_numpy(np.ascontiguousarray(sd.tri, np.uint32).view(np.int32)).cuda()
    bad = t.clone()
    bad[len(bad) // 2, 1] = len(v)  # vertex index == num_vertices
    ct = capi.CudaTrace(1)
    ct.upload_scene_device(v, t, 64)
    start = free_bytes()
    for _ in range(5):
        with pytest.raises(capi.CudaTraceError, match="vertex index out of bounds"):
            ct.upload_scene_device(v, bad, 64)
    end = free_bytes()
    ct.close()
    assert end >= start - SLACK, "%.1f MB lost" % ((start - end) / 2 ** 20)
