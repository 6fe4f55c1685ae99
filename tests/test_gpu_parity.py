"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle on the same
inputs.  Bar: per-sample hit record (tri_idx, t, u, v) bit-exact AND the 8-bit image bit-exact
(north_star tolerance: hit index exact up to 0.01 % ties, image within 1 LSB on 99.9 % of pixels --
both are met with zero exceptions on every case here)."""
import numpy as np
import pytest

from conftest import pkg

pytestmark = pytest.mark.gpu

ALL_SCENES = ["torusknot", "cornell", "room", "table_chair", "head", "room_cat", "water_knot",
              "griebel_teapot", "killeroo", "dwarf_hand_blob"]


def image_diff(a, b):
    """-> (pixels differing, max per-channel abs difference)"""
    a8 = a.view(np.uint8).reshape(a.shape + (4,)).astype(np.int16)
    b8 = b.view(np.uint8).reshape(b.shape + (4,)).astype(np.int16)
    d = np.abs(a8 - b8)
    return int((d.max(axis=-1) > 0).sum()), int(d.max())


def frame_for(ct, port, sd, w, h, spp, **kw):
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    return ct.make_frame(w, h, spp, sd.cam16, fov_xs, aspect, **kw)


@pytest.mark.parametrize("spp", [1, 2, 3, 4, 5, 16, 32, 33, 64, 256, 1000])
def test_sample_table(cuda_trace, port, spp):
    assert np.array_equal(cuda_trace.sample_table(spp).view(np.uint32), port.sample_table(spp).view(np.uint32))


@pytest.mark.parametrize("name", ALL_SCENES)
def test_grid_build_matches_oracle(cuda_trace, port, scene_data, name):
    sd = scene_data(name)
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    g = cuda_trace.download_grid()
    og = port.scene(sd.vtx, sd.tri, 64).grid()
    for k in ("dim", "aabb_min", "aabb_max", "cell_wdh", "inv_cell_wdh", "cell_offset", "tri_index"):
        assert np.array_equal(np.asarray(g[k]), np.asarray(og[k])), k


@pytest.mark.parametrize("res", [1, 7, 33, 128])
def test_grid_build_other_resolutions(cuda_trace, port, scene_data, res):
    sd = scene_data("killeroo")
    cuda_trace.upload_scene(sd.vtx, sd.tri, res)
    g = cuda_trace.download_grid()
    og = port.scene(sd.vtx, sd.tri, res).grid()
    for k in ("dim", "cell_wdh", "cell_offset", "tri_index"):
        assert np.array_equal(np.asarray(g[k]), np.asarray(og[k])), k


@pytest.mark.parametrize("name", ALL_SCENES)
@pytest.mark.parametrize("variant", [0, 1])
def test_scene_parity_small(cuda_trace, port, scene_data, name, variant):
    sd = scene_data(name)
    w, h, spp = 200, 120, 4
    ps = port.scene(sd.vtx, sd.tri, 64)
    if variant == 0:
        cuda_trace.upload_scene(sd.vtx, sd.tri, 64)          # device-built grid
    else:
        cuda_trace.upload_scene_with_grid(sd.vtx, sd.tri, ps.grid())  # injected oracle grid
    f = frame_for(cuda_trace, port, sd, w, h, spp, variant=variant, keep_hits=True)
    img = cuda_trace.trace_tiles(f)
    tri, t, u, v = cuda_trace.download_hits(w, h, spp)
    o = ps.render(sd.cam16, sd.fov, w, h, spp, variant=variant, want_hits=True, want_tuv=True)
    assert np.array_equal(tri, o["tri"])
    assert np.array_equal(t.view(np.uint32), o["t"].view(np.uint32))
    assert np.array_equal(u.view(np.uint32), o["u"].view(np.uint32))
    assert np.array_equal(v.view(np.uint32), o["v"].view(np.uint32))
    # 8-bit output: IEEE sqrtf vs glibc powf(x, .5f) never changes a byte for x in [0, 1.12]
    # (exhaustive scan, tests/test_oracle_vs_ref.py), so the image is bit-exact too
    assert image_diff(img, o["bgra"]) == (0, 0)


@pytest.mark.parametrize("name,res,size", [("tiger_soup_small", 64, (200, 112)), ("tiger_soup_small", 200, (160, 90)),
                                           ("tiger_soup_medium", 128, (160, 90))])
def test_instanced_soup_parity(cuda_trace, port, scene_data, name, res, size):
    """The synthetic tiger soup (config C5's construction at test size: 108 K / 2.3 M triangles):
    device-built grid == oracle grid (array equality) and per-sample hits + image bit-exact.  The
    occupancy map does not fit shared memory at these resolutions, so this also covers the
    global-bitmap traversal mode."""
    sd = scene_data(name)
    w, h = size
    ps = port.scene(sd.vtx, sd.tri, res, tight_ranges=True)
    cuda_trace.upload_scene(sd.vtx, sd.tri, res)
    g, og = cuda_trace.download_grid(), ps.grid()
    for k in ("dim", "aabb_min", "aabb_max", "cell_wdh", "inv_cell_wdh", "cell_offset", "tri_index"):
        assert np.array_equal(np.asarray(g[k]), np.asarray(og[k])), k
    f = frame_for(cuda_trace, port, sd, w, h, 4, keep_hits=True)
    img = cuda_trace.trace_tiles(f)
    tri, t, u, v = cuda_trace.download_hits(w, h, 4)
    o = ps.render(sd.cam16, sd.fov, w, h, 4, want_hits=True, want_tuv=True)
    assert np.array_equal(tri, o["tri"])
    assert np.array_equal(t.view(np.uint32), o["t"].view(np.uint32))
    assert np.array_equal(img, o["bgra"])
    assert (tri != 0xFFFFFFFF).mean() > 0.1


@pytest.mark.parametrize("spp", [1, 2, 3, 5, 16, 32, 33, 70])
def test_sample_counts(cuda_trace, port, scene_data, spp):
    sd = scene_data("cornell")
    w, h = 67, 45  # not multiples of the 8x4 strip
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    f = frame_for(cuda_trace, port, sd, w, h, spp, keep_hits=True)
    img = cuda_trace.trace_tiles(f)
    tri, t, u, v = cuda_trace.download_hits(w, h, spp)
    o = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, w, h, spp, want_hits=True)
    assert np.array_equal(tri, o["tri"])
    assert image_diff(img, o["bgra"]) == (0, 0)


def test_ragged_tiles_and_untouched_pixels(cuda_trace, port, scene_data):
    sd = scene_data("cornell")
    w, h, spp = 131, 77, 4
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    f = frame_for(cuda_trace, port, sd, w, h, spp)
    rects = [(0, 0, 1, 1), (5, 3, 5, 9), (7, 7, 7, 7), (10, 10, 29, 13), (100, 50, 131, 77), (40, 20, 49, 55)]
    out = np.full((h, w), 0xDEADBEEF, np.uint32)
    cuda_trace.trace_tiles(f, rects, out=out)
    o = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, w, h, spp)["bgra"]
    mask = np.zeros((h, w), bool)
    for x0, y0, x1, y1 in rects:
        mask[y0:y1, x0:x1] = True
    assert (out[~mask] == 0xDEADBEEF).all()
    assert np.array_equal(out[mask], o[mask])
    # empty tile list is legal and renders nothing
    out2 = np.full((h, w), 7, np.uint32)
    cuda_trace.trace_tiles(f, [], out=out2)
    assert (out2 == 7).all()


def test_no_gamma_flag(cuda_trace, port, scene_data):
    sd = scene_data("cornell")
    w, h, spp = 64, 64, 2
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    f = frame_for(cuda_trace, port, sd, w, h, spp, gamma=False)
    img = cuda_trace.trace_tiles(f)
    o = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, w, h, spp, gamma=False)["bgra"]
    assert np.array_equal(img, o)  # without the powf/sqrtf difference the image is bit-exact


def test_arbitrary_rays(cuda_trace, port, scene_data):
    """Grid::Intersect on rays the camera never produces: axis-aligned directions (zero
    components -> +-inf slabs), origins inside / on / behind the box, unnormalised directions."""
    sd = scene_data("cornell")
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    ps = port.scene(sd.vtx, sd.tri, 64)
    g = ps.grid()
    rs = np.random.RandomState(7)
    n = 20000
    o = rs.uniform(-1.5, 1.5, (n, 3)).astype(np.float32)
    d = rs.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True).astype(np.float32)
    # axis aligned and planar directions
    d[:3000, 0] = 0.0
    d[1000:4000, 1] = 0.0
    d[4000:4600] = np.eye(3, dtype=np.float32)[rs.randint(0, 3, 600)] * rs.choice([-1, 1], (600, 1))
    d[4600:4700, 2] = -0.0
    # origins inside the box, exactly on its faces, and unnormalised directions
    o[5000:9000] = rs.uniform(-0.45, 0.45, (4000, 3)).astype(np.float32)
    o[9000:9300, 0] = g["aabb_min"][0]
    o[9300:9600, 1] = g["aabb_max"][1]
    d[9600:10000] *= rs.uniform(0.1, 10, (400, 1)).astype(np.float32)
    keep = np.abs(d).sum(axis=1) > 0
    o, d = o[keep], d[keep]
    for variant in (0, 1):
        tri, t, u, v = cuda_trace.intersect_rays(o, d, variant)
        otri, ot, ou, ov = ps.intersect_rays(o, d, variant)
        assert np.array_equal(tri, otri)
        assert np.array_equal(t.view(np.uint32), ot.view(np.uint32))
        assert np.array_equal(u.view(np.uint32), ou.view(np.uint32))
        assert np.array_equal(v.view(np.uint32), ov.view(np.uint32))
        assert (tri != 0xFFFFFFFF).sum() > 1000


@pytest.mark.parametrize("name,res", [("killeroo", 64), ("room", 64), ("torusknot", 64), ("tiger_soup_small", 48)])
def test_mailboxing_mode(cuda_trace, port, scene_data, name, res):
    """Mailboxing -- the reference author's TODO at grid.cpp:172 -- as an optional mode of the ray-batch entry point:
    a ray reuses the outcome of a triangle it has already tested in an earlier cell.  Results must be bit-identical
    to the plain walk and to the oracle; the statistics say how many tests the mailbox answered."""
    sd = scene_data(name)
    cuda_trace.upload_scene(sd.vtx, sd.tri, res)
    ps = port.scene(sd.vtx, sd.tri, res, tight_ranges=True)
    rs = np.random.RandomState(11)
    n = 30000
    g = ps.grid()
    lo, hi = np.asarray(g["aabb_min"], np.float32), np.asarray(g["aabb_max"], np.float32)
    o = (rs.uniform(-1.0, 1.0, (n, 3)) * 2.0 * (hi - lo) + (lo + hi) / 2).astype(np.float32)  # mostly outside the box
    target = rs.uniform(lo, hi, (n, 3)).astype(np.float32)
    d = target - o
    d /= np.linalg.norm(d, axis=1, keepdims=True).astype(np.float32)
    for variant in (0, 1):
        plain = cuda_trace.intersect_rays(o, d, variant)
        boxed = cuda_trace.intersect_rays(o, d, variant, mailbox=True)
        want = ps.intersect_rays(o, d, variant)
        for a, b, c in zip(plain, boxed, want):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(b.view(np.uint32), c.view(np.uint32))
        tests, reused = cuda_trace.mailbox_stats()
        assert tests > 0 and 0 < reused < tests
        print("%s variant %d: mailbox answered %.1f %% of %d tests" % (name, variant, 100.0 * reused / tests, tests))


def cityblock_distance_map(occ):
    """Exact city-block distance transform of a boolean volume (distance 0 where set), clamped to 255: the
    separable two-sweep form per axis in numpy -- the checker of the device's distance map."""
    d = np.where(occ, 0, 10 ** 6).astype(np.int64)
    for axis in range(3):
        d = np.moveaxis(d, axis, 0)
        for i in range(1, d.shape[0]):
            np.minimum(d[i], d[i - 1] + 1, out=d[i])
        for i in range(d.shape[0] - 2, -1, -1):
            np.minimum(d[i], d[i + 1] + 1, out=d[i])
        d = np.moveaxis(d, 0, axis)
    return np.minimum(d, 255).astype(np.uint8)


@pytest.mark.parametrize("name,res", [("tiger_soup_small", 150), ("killeroo", 200), ("cornell", 130)])
def test_distance_map_matches_cityblock_transform(cuda_trace, port, scene_data, name, res):
    """The second level of the empty-space walk (large grids): the device's distance map over the padded grid equals
    the exact city-block distance to the nearest non-empty or padding cell, computed here from the ORACLE's grid."""
    sd = scene_data(name)
    cuda_trace.upload_scene(sd.vtx, sd.tri, res)
    dist = cuda_trace.download_distance_map()
    assert dist is not None
    og = port.scene(sd.vtx, sd.tri, res, tight_ranges=True).grid()
    dx, dy, dz = [int(v) for v in og["dim"]]
    off = np.asarray(og["cell_offset"]).astype(np.int64)
    occ = np.ones((dy + 2, dz + 2, dx + 2), bool)  # padding cells count as occupied
    occ[1:-1, 1:-1, 1:-1] = (off[1:] != off[:-1]).reshape(dy, dz, dx)  # cell = x + z*dx + y*dx*dz (grid.h:41-42)
    want = cityblock_distance_map(occ)
    assert dist.shape == want.shape and np.array_equal(dist, want)
    assert int(dist.max()) > 3  # there is something to skip


def test_small_grids_have_no_distance_map(cuda_trace, scene_data):
    sd = scene_data("cornell")
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    assert cuda_trace.download_distance_map() is None


@pytest.mark.parametrize("threads", ["1024", "128"])
@pytest.mark.parametrize("name,spp,res", [("killeroo", 4, 64), ("room", 16, 64), ("cornell", 1, 64), ("killeroo", 5, 96),
                                          ("tiger_soup_small", 16, 150), ("torusknot", 32, 64)])
def test_pooled_traversal(port, scene_data, monkeypatch, name, spp, res, threads):
    """K7 trace_pool (pool_trace.cu): every warp keeps a pool of 64 rays and compacts, by ballot, 32 that need the
    same kind of work (walk / test); K1 then shades from the hit records.  Same per-ray arithmetic, so hit records
    and image must be bit-identical to the oracle -- with the caller's hit buffers (KEEP_HITS) and with the device's
    own, on whole frames and on a ragged tile list whose strips are clipped."""
    monkeypatch.setenv("RTM_POOL", "1")
    monkeypatch.setenv("RTM_THREADS", threads)
    sd = scene_data(name)
    w, h = 250, 138
    ct = pkg("capi").CudaTrace(1)
    ct.upload_scene(sd.vtx, sd.tri, res)
    assert ct.download_distance_map() is not None
    o = port.scene(sd.vtx, sd.tri, res, tight_ranges=True).render(sd.cam16, sd.fov, w, h, spp, want_hits=True, want_tuv=True)
    launches = ct.kernel_launches()
    f = frame_for(ct, port, sd, w, h, spp, keep_hits=True)
    img = ct.trace_tiles(f)
    assert ct.kernel_launches() - launches == 3  # sample table + K7 + K1 <from hits>
    tri, t, u, v = ct.download_hits(w, h, spp)
    assert np.array_equal(tri, o["tri"])
    for a, b in ((t, o["t"]), (u, o["u"]), (v, o["v"])):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
    assert np.array_equal(img, o["bgra"])
    # the device's own hit records + ragged tiles (pixels outside them stay untouched)
    f2 = frame_for(ct, port, sd, w, h, spp)
    assert np.array_equal(ct.trace_tiles(f2), o["bgra"])
    rects = [(3, 5, 117, 61), (117, 5, 250, 61), (0, 70, 250, 138)]
    out = np.full((h, w), 0xDEADBEEF, np.uint32)
    got = ct.trace_tiles(f2, rects=rects, out=out)
    want = np.full((h, w), 0xDEADBEEF, np.uint32)
    for x0, y0, x1, y1 in rects:
        want[y0:y1, x0:x1] = o["bgra"][y0:y1, x0:x1]
    assert np.array_equal(got, want)
    ct.close()


@pytest.mark.parametrize("mode", ["0", "1", "2", "3"])
@pytest.mark.parametrize("name,spp", [("killeroo", 4), ("room", 16), ("cornell", 1)])
def test_occupancy_map_modes(port, scene_data, monkeypatch, mode, name, spp):
    """The homes of the padded occupancy map (bits through L1 / bits in shared memory / one byte
    per cell in shared memory with the DDA tracking the byte address / the distance map through L1 with look-ups
    only every `distance` steps) and both phase-A forms must give the same bits.  Small frames default to mode 0, so the shared-memory modes are forced here (the tuning
    switches are read when a context is created)."""
    monkeypatch.setenv("RTM_OCC_MODE", mode)
    monkeypatch.setenv("RTM_THREADS", "1024" if mode in ("1", "2") else "256")
    sd = scene_data(name)
    w, h = 256, 144
    cuda_trace = pkg("capi").CudaTrace(1)
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    f = frame_for(cuda_trace, port, sd, w, h, spp, keep_hits=True)
    img = cuda_trace.trace_tiles(f)
    tri, t, u, v = cuda_trace.download_hits(w, h, spp)
    o = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, w, h, spp, want_hits=True, want_tuv=True)
    assert np.array_equal(tri, o["tri"]) and np.array_equal(img, o["bgra"])
    assert np.array_equal(t.view(np.uint32), o["t"].view(np.uint32))
    # and the plain (non-instrumented) kernel instantiation
    f2 = frame_for(cuda_trace, port, sd, w, h, spp)
    assert np.array_equal(cuda_trace.trace_tiles(f2), o["bgra"])
    cuda_trace.close()


@pytest.mark.parametrize("mode", ["0", "2"])
@pytest.mark.parametrize("name,spp", [("killeroo", 4), ("cornell", 16), ("head", 1), ("dwarf_hand_blob", 64)])
def test_origin_relative_records(port, scene_data, monkeypatch, mode, name, spp):
    """Frames of 16 M rays and more run Moeller-Trumbore on records relative to the camera position
    (tvec, qvec and e2.qvec precomputed once per camera, csrc/pack.cu).  Forced on here for small frames so that
    the per-sample t / u / v can be compared bit for bit with the oracle, in two occupancy modes, before and after
    the camera moves (the records are rebuilt), and against the plain records (forced off)."""
    capi = pkg("capi")
    sd = scene_data(name)
    w, h = 192, 128
    ps = port.scene(sd.vtx, sd.tri, 64)
    cam2 = np.array(sd.cam16, np.float32).copy()
    cam2[12:15] += np.array([0.03, -0.02, 0.05], np.float32)  # Matrix44f translation row = camera origin
    outs = {}
    for rel in ("2", "0"):
        monkeypatch.setenv("RTM_REL_RECORDS", rel)
        monkeypatch.setenv("RTM_OCC_MODE", mode)
        monkeypatch.setenv("RTM_THREADS", "1024" if mode != "0" else "256")
        ct = capi.CudaTrace(1)
        ct.upload_scene(sd.vtx, sd.tri, 64)
        fov_xs, aspect = port.camera_constants(sd.fov, w, h)
        for k, cam in enumerate((sd.cam16, cam2, sd.cam16)):
            f = ct.make_frame(w, h, spp, cam, fov_xs, aspect, keep_hits=True)
            img = ct.trace_tiles(f)
            tri, t, u, v = ct.download_hits(w, h, spp)
            outs[(rel, k)] = (img.copy(), tri, t, u, v)
            plain = ct.trace_tiles(ct.make_frame(w, h, spp, cam, fov_xs, aspect))  # non-instrumented instantiation
            assert np.array_equal(plain, img)
        ct.close()
    for k, cam in enumerate((sd.cam16, cam2)):
        o = ps.render(cam, sd.fov, w, h, spp, want_hits=True, want_tuv=True)
        for rel in ("2", "0"):
            img, tri, t, u, v = outs[(rel, k)]
            assert np.array_equal(tri, o["tri"]) and np.array_equal(img, o["bgra"]), (rel, k)
            for got, key in ((t, "t"), (u, "u"), (v, "v")):
                assert np.array_equal(got.view(np.uint32), o[key].view(np.uint32)), (rel, k, key)
    for rel in ("2", "0"):  # back at the first camera
        for a, b in zip(outs[(rel, 2)], outs[(rel, 0)]):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


@pytest.mark.parametrize("name,ortho_width", [("cornell", 1.7), ("killeroo", 1.3), ("room", 0.9)])
def test_orthographic_camera(cuda_trace, port, scene_data, name, ortho_width):
    """GenerateRay's orthographic branch (camera.h:25-36): every ray has its own origin.  Oracle = the port, whose
    ortho rays and hits are pinned to the reference's GenerateRay(ortho = true) + Grid::Intersect on the CPU
    (tests/test_oracle_vs_ref.py)."""
    sd = scene_data(name)
    w, h, spp = 160, 96, 4
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    f = cuda_trace.make_frame(w, h, spp, sd.cam16, fov_xs, aspect, keep_hits=True, ortho_width=ortho_width)
    img = cuda_trace.trace_tiles(f)
    tri, t, u, v = cuda_trace.download_hits(w, h, spp)
    o = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, w, h, spp, want_hits=True, want_tuv=True,
                                               ortho_width=ortho_width)
    assert np.array_equal(tri, o["tri"]) and np.array_equal(img, o["bgra"])
    for got, key in ((t, "t"), (u, "u"), (v, "v")):
        assert np.array_equal(got.view(np.uint32), o[key].view(np.uint32))
    assert (tri != 0xFFFFFFFF).sum() > 1000
    plain = cuda_trace.trace_tiles(cuda_trace.make_frame(w, h, spp, sd.cam16, fov_xs, aspect, ortho_width=ortho_width))
    assert np.array_equal(plain, img)


@pytest.mark.parametrize("shade_mode", [1, 2])
@pytest.mark.parametrize("name,spp", [("cornell", 1), ("head", 4), ("killeroo", 16)])
def test_shading_alternates(cuda_trace, port, scene_data, name, spp, shade_mode):
    """Face-normal and depth shading (renderer.cpp:116,118, commented out in the reference)."""
    sd = scene_data(name)
    w, h = 144, 100
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    img = cuda_trace.trace_tiles(cuda_trace.make_frame(w, h, spp, sd.cam16, fov_xs, aspect, shade_mode=shade_mode))
    o = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, w, h, spp, shade_mode=shade_mode)
    assert np.array_equal(img, o["bgra"])
    if name != "cornell" or shade_mode == 2:  # the Cornell box is flat-shaded: its face normals ARE its vertex normals
        live = cuda_trace.trace_tiles(cuda_trace.make_frame(w, h, spp, sd.cam16, fov_xs, aspect))
        assert not np.array_equal(img, live)


def test_brute_force_self_check(cuda_trace, ref_answers, port, scene_data):
    """Renderer::IntersectBruteForce on the device: bit-exact against the reference's own brute force, and
    -- the author's cross-check -- equal to the grid result except where the grid's in-cell rule decides."""
    sd = scene_data("cornell")
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    o3, d3 = ref_answers.rays(port, "cornell", 96, 64, 2, 0, 64)
    o, d = o3.reshape(-1, 3), d3.reshape(-1, 3)
    bt = cuda_trace.intersect_rays_brute_force(o, d)

    def want(r):
        m, fov, cam = pkg("scenes").build(r.api, "cornell")
        rt = r.renderer(m, fov, cam).intersect_rays_brute_force(o, d)
        return np.stack([rt[0]] + [rt[i].view(np.uint32) for i in (1, 2, 3)])

    ref_answers.check("brute_force/cornell/96x64x2", np.stack([bt[0]] + [bt[i].view(np.uint32) for i in (1, 2, 3)]), want)
    gt = cuda_trace.intersect_rays(o, d, 0)
    assert (gt[0] != bt[0]).mean() < 0.01  # grid vs brute force: only boundary / tie cases differ
    assert (bt[0] != 0xFFFFFFFF).sum() > 1000


def test_ray_march_matches_reference(cuda_trace, ref_answers, port, scene_data):
    """Renderer::RayMarch + DistanceBruteForce + DistancePointTri on the device, bit-exact (hit flag and the
    parameter t reached) against the reference's own functions, on camera rays of the Cornell scene."""
    sd = scene_data("cornell")
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    o3, d3 = ref_answers.rays(port, "cornell", 48, 32, 1, 0, 32)
    o, d = o3.reshape(-1, 3), d3.reshape(-1, 3)
    gh, gt = cuda_trace.ray_march(o, d)

    def want(r):
        m, fov, cam = pkg("scenes").build(r.api, "cornell")
        rh, rt = r.renderer(m, fov, cam).ray_march(o, d)
        return np.stack([np.asarray(rh, np.uint32), rt.view(np.uint32)])

    ref_answers.check("ray_march/cornell/48x32x1", np.stack([np.asarray(gh, np.uint32), gt.view(np.uint32)]), want)
    assert 100 < int(gh.sum()) < len(gh)


def test_counters_match_oracle(cuda_trace, port, scene_data):
    sd = scene_data("killeroo")
    w, h, spp = 160, 90, 4
    cuda_trace.upload_scene(sd.vtx, sd.tri, 64)
    cuda_trace.set_counting(True)
    try:
        f = frame_for(cuda_trace, port, sd, w, h, spp)
        cuda_trace.trace_tiles(f)
        c = cuda_trace.get_counters()
    finally:
        cuda_trace.set_counting(False)
    oc = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, w, h, spp)["counters"]
    for k in ("rays", "cells", "tri_tests", "hits"):
        assert c[k] == oc[k], k


def test_errors(cuda_trace, scene_data):
    capi = pkg("capi")
    ct = capi.CudaTrace(1)
    try:
        f = ct.make_frame(16, 16, 1, np.eye(4, dtype=np.float32).reshape(16), 0.5, 1.0)
        with pytest.raises(capi.CudaTraceError) as e:
            ct.trace_tiles(f)
        assert e.value.code == 4  # CUDA_TRACE_ERR_NO_SCENE
        sd = scene_data("cornell")
        bad = sd.tri.copy()
        bad[0, 0] = len(sd.vtx)
        with pytest.raises(capi.CudaTraceError):
            ct.upload_scene(sd.vtx, bad, 64)
        with pytest.raises(capi.CudaTraceError):
            ct.upload_scene(sd.vtx, sd.tri, 0)
        ct.upload_scene(sd.vtx, sd.tri, 64)
        with pytest.raises(capi.CudaTraceError):
            ct.trace_tiles(f, [(0, 0, 17, 16)])  # tile outside the frame
        f0 = ct.make_frame(16, 16, 0, np.eye(4, dtype=np.float32).reshape(16), 0.5, 1.0)
        with pytest.raises(capi.CudaTraceError):
            ct.trace_tiles(f0)
    finally:
        ct.close()
    with pytest.raises(capi.CudaTraceError):
        capi.CudaTrace(devices=[99])


def test_cost_ordered_split_frames_match_image_order(ref_answers, scene_data):
    """Scheduling must never change results.  Frames 2.. of one layout run through the cost order of the previous
    frame, with its expensive strips split into pieces (csrc/schedule.cu); the camera moves between frames so a
    skipped piece cannot hide behind a stale pixel.  1080p / 16 spp: 128-ray strips, 4 pieces, order on by default;
    both the plain read-back and the overlapped per-band one (whose counters count pieces) are used."""
    capi, scenes = pkg("capi"), pkg("scenes")
    api = ref_answers.api
    sd = scene_data("killeroo")
    w, h, spp = 1920, 1080, 16
    fov_xs, aspect = api.camera_constants(sd.fov, w, h)
    cams = []
    for eye_x in (-1.6, -1.5, -1.4):
        cams.append(api.look_at((eye_x, 1.2, -1.0), (0.0, 0.0, -0.1)))
    fresh = capi.CudaTrace(1)
    fresh.upload_scene(sd.vtx, sd.tri, 64)
    want = []
    for cam in cams:  # every frame in image order: a new layout (different tiles) in between invalidates the order
        fresh.trace_tiles(fresh.make_frame(64, 64, 1, cam, fov_xs, aspect))
        want.append(fresh.trace_tiles(fresh.make_frame(w, h, spp, cam, fov_xs, aspect)).copy())

    def ref_frame(r):
        m, fov, _ = scenes.build(r.api, "killeroo")
        return r.renderer(m, fov, cams[0]).render(w, h, spp)[1]

    ref_answers.check("renderer/killeroo_eye-1.6/%dx%dx%d" % (w, h, spp), want[0], ref_frame)
    fresh.close()

    ct = capi.CudaTrace(1)
    ct.upload_scene(sd.vtx, sd.tri, 64)
    pinned = capi.PinnedImage(w, h)
    for k, cam in enumerate(cams):
        f = ct.make_frame(w, h, spp, cam, fov_xs, aspect)
        ct.trace_tiles_async(f)
        got = ct.read_framebuffer(np.zeros((h, w), np.uint32))
        assert np.array_equal(got, want[k]), "frame %d (plain read-back)" % k
        cyc = ct.strip_cycles()
        assert len(cyc) == (w // 4) * (h // 2) and int((cyc == 0).sum()) == 0  # every strip was visited and timed
    for k, cam in enumerate(cams):
        pinned.array[:] = 0
        ct.trace_tiles(ct.make_frame(w, h, spp, cam, fov_xs, aspect), out=pinned.array)
        assert np.array_equal(pinned.array, want[k]), "frame %d (overlapped read-back)" % k
    heavy = ct.strip_cycles()
    assert heavy.max() > 4 * heavy.mean()  # the premise: strip costs are very uneven
    ct.close()


def test_refused_call_leaves_the_overlapped_read_back_usable(port, scene_data):
    """A call that is refused (bad sample count, tile outside the frame, counters with an alternate) must not
    advance the band completion targets of the overlapped read-back: the next ordinary frame into a host buffer
    would then wait for counts the device never reaches.  Also after a frame whose layout differs."""
    capi = pkg("capi")
    sd = scene_data("cornell")
    w, h, spp = 640, 480, 4   # > 1 MB of pixels: several row bands
    ct = capi.CudaTrace(1)
    ct.upload_scene(sd.vtx, sd.tri, 64)
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    good = ct.make_frame(w, h, spp, sd.cam16, fov_xs, aspect)
    ref_img = ct.trace_tiles(good).copy()
    assert np.array_equal(ref_img, port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, w, h, spp)["bgra"])
    # 1. sample count beyond the limit
    with pytest.raises(capi.CudaTraceError):
        ct.trace_tiles(ct.make_frame(w, h, 1 << 20, sd.cam16, fov_xs, aspect))
    assert np.array_equal(ct.trace_tiles(good), ref_img)
    # 2. a tile outside the frame
    with pytest.raises(capi.CudaTraceError):
        ct.trace_tiles(good, rects=[(0, 0, w + 1, h)])
    assert np.array_equal(ct.trace_tiles(good), ref_img)
    # 3. work counters together with the orthographic camera
    ct.set_counting(True)
    with pytest.raises(capi.CudaTraceError):
        ct.trace_tiles(ct.make_frame(w, h, spp, sd.cam16, fov_xs, aspect, ortho_width=1.5))
    ct.set_counting(False)
    assert np.array_equal(ct.trace_tiles(good), ref_img)
    # 4. overlapping tiles whose areas add up to the frame: not a partition, so no whole-band copies; pixels no
    #    tile covers keep what the host buffer held
    out = np.full((h, w), 0xDEADBEEF, np.uint32)
    ct.trace_tiles(good, rects=[(0, 0, w, h // 2), (0, 0, w, h // 2)], out=out)
    assert np.array_equal(out[: h // 2], ref_img[: h // 2]) and (out[h // 2:] == 0xDEADBEEF).all()
    assert np.array_equal(ct.trace_tiles(good), ref_img)
    ct.close()


def test_cancel_names_its_frame(port, scene_data):
    """cuda_trace_cancel stops the frame in flight (Framebuffer::m_threads_stop, framebuffer.h:32) and nothing
    else: a request issued when no frame is running must not cancel the next one."""
    import threading
    capi = pkg("capi")
    sd = scene_data("killeroo")
    w, h, spp = 1920, 1080, 64   # long enough (tens of ms) for the request to arrive while it runs
    ct = capi.CudaTrace(1)
    ct.upload_scene(sd.vtx, sd.tri, 64)
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    f = ct.make_frame(w, h, spp, sd.cam16, fov_xs, aspect)
    small = ct.make_frame(160, 96, 4, sd.cam16, *port.camera_constants(sd.fov, 160, 96))
    want_small = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, 160, 96, 4)["bgra"]
    ct.trace_tiles(small)
    ct.cancel()  # no frame running: refers to the finished frame
    assert np.array_equal(ct.trace_tiles(small), want_small)
    ct.trace_tiles_async(f)
    t = threading.Timer(0.002, ct.cancel)
    t.start()
    with pytest.raises(capi.CudaTraceError) as e:
        ct.sync()
    t.join()
    assert e.value.code == 5  # CUDA_TRACE_ERR_CANCELLED
    assert np.array_equal(ct.trace_tiles(small), want_small)   # the next frame is not affected
    ct.close()
