"""The C++ host mirror (Renderer : Framebuffer, Scene, Grid -- host/*.h) driven on one GPU and compared with the
unmodified reference's classes of the same names (oracle/_ref), or with the committed digests of their answers
(tests/golden) when it is absent.

Everything here goes Mesh -> Scene -> Renderer -> Resize/StartRendering -> WaitRendering -> tiles, i.e. the route a
viewer using the reference's API takes (INTEGRATION.md route A)."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import pkg

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))


def _host_renderer(name, grid_res=64):
    hostapi, scenes = pkg("hostapi"), pkg("scenes")
    m, fov, cam = scenes.build(hostapi.host_api(), name)
    return hostapi.HostRenderer(m, fov, cam, grid_res), fov, cam


def _ref_renderer(ref, name, grid_res=64):
    m, fov, cam = pkg("scenes").build(ref.api, name)
    return ref.renderer(m, fov, cam, grid_res)


@pytest.mark.parametrize("name,w,h,spp", [("cornell", 200, 120, 4), ("killeroo", 333, 217, 2), ("head", 128, 128, 16)])
def test_renderer_frame_matches_reference(ref_answers, name, w, h, spp):
    hr, _, _ = _host_renderer(name)
    sec, img = hr.render(w, h, spp)
    assert sec > 0 and hr.last_kernel_ms() > 0
    ref_answers.check("renderer/%s/%dx%dx%d" % (name, w, h, spp), img, lambda r: _ref_renderer(r, name).render(w, h, spp)[1])
    # a second frame at another size and sample count through the same Renderer (Resize path)
    w2, h2 = w // 2 + 1, h // 2 + 3
    _, img2 = hr.render(w2, h2, 1)
    ref_answers.check("renderer/%s/%dx%dx1" % (name, w2, h2), img2, lambda r: _ref_renderer(r, name).render(w2, h2, 1)[1])


def test_renderer_digest_without_reference():
    """Same route, checked against tests/golden/ref_digests.json -- runs on boxes without oracle/_ref."""
    with open(os.path.join(HERE, "golden", "ref_digests.json")) as f:
        digests = json.load(f)
    key = sorted(k for k, d in digests.items() if d["scene"] == "cornell")[0]
    d = digests[key]
    hr, _, _ = _host_renderer(d["scene"], d["grid_res"])
    _, img = hr.render(d["width"], d["height"], d["spp"])
    assert hashlib.md5(np.ascontiguousarray(img).tobytes()).hexdigest() == d["image_md5"]
    gi = hr.grid_info()
    assert [int(x) for x in gi["dim"]] == d["dim"] and gi["num_refs"] == d["refs"]
    assert int(np.float32(gi["cell_wdh"]).view(np.uint32)) == d["cell_wdh_bits"]


def test_save_bmp_byte_identical(ref_answers, tmp_path):
    hr, _, _ = _host_renderer("cornell")
    hr.render(96, 64, 2)
    a, b = str(tmp_path / "host.bmp"), str(tmp_path / "ref.bmp")
    hr.save_bmp(a)

    def ref_bmp(r):
        rr = _ref_renderer(r, "cornell")
        rr.render(96, 64, 2)
        rr.save_bmp(b)
        return np.fromfile(b, np.uint8)

    ref_answers.check("save_bmp/cornell/96x64x2", np.fromfile(a, np.uint8), ref_bmp)


def test_grid_intersect_and_ray_march_single_ray(ref_answers, port):
    """Grid::Intersect (grid.cpp:208-334) and Renderer::RayMarch (renderer.cpp:24-41) as one-ray queries.
    Per queried ray: hit triangle (MISS if none), t / u / v bits (0 on a miss), march hit flag, march t bits."""
    hr, _, _ = _host_renderer("cornell")
    o3, d3 = ref_answers.rays(port, "cornell", 16, 12, 1, 0, 12)
    o, d = o3.reshape(-1, 3), d3.reshape(-1, 3)
    sel = range(0, len(o), 7)
    got = np.zeros((len(sel), 6), np.uint32)
    for row, i in enumerate(sel):
        ok, tuv, tri = hr.intersect(o[i], d[i])
        got[row, 0] = tri if ok else 0xFFFFFFFF
        if ok:
            got[row, 1:4] = np.asarray(tuv, np.float32).view(np.uint32)
        got_hit, got_t = hr.ray_march(o[i], d[i])
        got[row, 4], got[row, 5] = int(bool(got_hit)), np.float32(got_t).view(np.uint32)

    def want(r):
        rr = _ref_renderer(r, "cornell")
        idx, t, u, v = rr.intersect_rays(o, d)
        mh, mt = rr.ray_march(o, d)
        w = np.zeros_like(got)
        for row, i in enumerate(sel):
            w[row, 0] = idx[i]
            if idx[i] != 0xFFFFFFFF:
                w[row, 1:4] = np.array([t[i], u[i], v[i]], np.float32).view(np.uint32)
            w[row, 4], w[row, 5] = int(bool(mh[i])), mt[i:i + 1].view(np.uint32)[0]
        return w

    ref_answers.check("intersect_and_march/cornell/16x12x1/every7", got, want)
    assert int((got[:, 0] != 0xFFFFFFFF).sum()) > 5


def test_renderer_alternates_match_port(port):
    """Renderer::SetOrthographicWidth / SetShadingMode through the C++ mirror == the port's restatement of
    camera.h:25-36 and renderer.cpp:116,118 (itself pinned to the reference on the CPU)."""
    hostapi, scenes = pkg("hostapi"), pkg("scenes")
    m, fov, cam = scenes.build(hostapi.host_api(), "cornell")
    vtx, tri = m.arrays()
    ps = port.scene(vtx, tri, 64)
    hr = hostapi.HostRenderer(m, fov, cam)
    w, h, spp = 150, 90, 4
    for ortho, mode in ((1.6, 0), (0.0, 1), (0.0, 2), (1.2, 2), (0.0, 0)):
        hr.set_alternates(ortho, mode)
        _, img = hr.render(w, h, spp)
        want = ps.render(cam, fov, w, h, spp, ortho_width=ortho if ortho else None, shade_mode=mode)["bgra"]
        assert np.array_equal(img, want), (ortho, mode)


def test_grid_info_matches_reference(ref_answers):
    """Grid dimensions, reference count, cell size bits, bounding box bits: [dim x3, refs, cell_wdh, min x3, max x3]."""
    def record(dim, refs, cell_wdh, mn, mx):
        f32 = lambda a: np.asarray(a, np.float32).reshape(-1).view(np.uint32).astype(np.uint64)
        return np.concatenate([np.asarray(dim, np.uint64), [np.uint64(refs)], f32(cell_wdh), f32(mn), f32(mx)])

    for name, res in (("killeroo", 64), ("room", 32)):
        hr, _, _ = _host_renderer(name, res)
        gi = hr.grid_info()
        got = record(gi["dim"], gi["num_refs"], gi["cell_wdh"], gi["aabb_min"], gi["aabb_max"])

        def want(r):
            g = _ref_renderer(r, name, res).grid()
            return record(g["dim"], len(g["tri_index"]), g["cell_wdh"], g["aabb_min"], g["aabb_max"])

        ref_answers.check("grid_info/%s/g%d" % (name, res), got, want)


def test_tiles_into_gives_every_tile_its_own_buffer(scene_data, port):
    """cuda_trace_tiles_into: each tile row-major in its own buffer (Framebuffer::Tile::m_bgra, framebuffer.h:64),
    reported complete in groups, every tile exactly once, top of the frame first."""
    capi = pkg("capi")
    sd = scene_data("killeroo")
    w, h, spp = 1283, 731, 4   # ragged: the last tile column / row absorb the remainder
    ct = capi.CudaTrace(1)
    ct.upload_scene(sd.vtx, sd.tri, 64)
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    f = ct.make_frame(w, h, spp, sd.cam16, fov_xs, aspect)
    want = ct.trace_tiles(f)
    rects = capi.full_frame_tiles(w, h)
    for _ in range(2):
        tiles, groups = ct.trace_tiles_into(f, rects)
        for (x0, y0, x1, y1), t in zip(rects, tiles):
            assert np.array_equal(t, want[y0:y1, x0:x1])
        flat = [i for g in groups for i in g]
        assert sorted(flat) == list(range(len(rects))) and len(groups) > 1
        last_row = [rects[g[0]][3] for g in groups]
        assert last_row == sorted(last_row)
    # a partial, unordered tile list
    some = [rects[40], rects[3], (5, 7, 5, 20), rects[100]]
    tiles, groups = ct.trace_tiles_into(f, some)
    for (x0, y0, x1, y1), t in zip(some, tiles):
        if x1 > x0 and y1 > y0:
            assert np.array_equal(t, want[y0:y1, x0:x1])
    assert sorted(i for g in groups for i in g) == [0, 1, 2, 3]
    ct.close()


def test_screenshot_of_a_frame_in_progress(tmp_path):
    """Tiles are handed back one by one while the frame is traced (the reference's worker leaves its tile lock
    when the tile is done, framebuffer.cpp:72-77): a SaveToBMP during the frame shows the finished tiles with their
    final pixels and the others black (framebuffer.cpp:203), and the count of lockable tiles grows."""
    hr, _, _ = _host_renderer("killeroo")
    w, h, spp = 1920, 1080, 256          # ~45 ms of tracing on one B200
    hr.render(w, h, 1)                    # sizes the frame buffer
    path = str(tmp_path / "partial.bmp")
    hr.start(w, h, spp)
    seen, shot, began = [], None, False
    import time
    t_end = time.time() + 10.0
    while time.time() < t_end:
        n = hr.finished_tiles()
        seen.append(n)
        began = began or n < 108          # the launcher holds the tiles: the frame has begun
        if shot is None and 20 <= n < 100:
            hr.save_bmp(path)
            shot = n
        if began and n == 108:
            break
    sec = hr.wait()
    final = hr.copy_bitmap(w, h)
    assert sec > 0 and shot is not None, "the frame went by without an intermediate state: %r" % sorted(set(seen))
    assert any(0 < n < 108 for n in seen)
    data = np.fromfile(path, np.uint8)[54:].view(np.uint32).reshape(h, w)
    black = same = 0
    for (x0, y0, x1, y1) in pkg("capi").full_frame_tiles(w, h):
        t = data[y0:y1, x0:x1]
        if not t.any():
            black += 1
        else:
            assert np.array_equal(t, final[y0:y1, x0:x1])
            same += 1
    assert black > 0 and same >= shot


def test_failed_frame_is_reported_not_fatal():
    """A device error inside the launcher thread must not terminate the application (std::terminate from an
    exception on a std::thread): WaitRendering() reports it, the tiles are released, the next frame works."""
    hr, _, _ = _host_renderer("cornell")
    _, good = hr.render(64, 48, 2)
    with pytest.raises(RuntimeError) as e:
        hr.render(64, 48, 1 << 20)   # more samples than the kernel accepts
    assert "samples per pixel" in str(e.value)
    assert hr.finished_tiles() == 108
    _, again = hr.render(64, 48, 2)
    assert np.array_equal(again, good)


def test_stop_rendering_leaves_unfinished_tiles_black():
    hr, _, _ = _host_renderer("killeroo")
    w, h = 1920, 1080
    hr.render(w, h, 1)
    hr.start(w, h, 1024)                  # ~180 ms
    while hr.finished_tiles() == 108:
        pass
    hr.stop()                             # KillAllWorkerThreads: cancel + wait
    img = hr.copy_bitmap(w, h)
    tiles = [img[y0:y1, x0:x1] for (x0, y0, x1, y1) in pkg("capi").full_frame_tiles(w, h)]
    assert sum(1 for t in tiles if not t.any()) > 0
    _, ok = hr.render(w, h, 1)            # and the renderer is still usable
    assert ok.any()
