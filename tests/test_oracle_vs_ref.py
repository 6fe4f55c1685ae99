"""CPU tests that PIN the oracle port (oracle/rt_oracle.c) against the unmodified reference
(oracle/_ref, or the digests of its answers in tests/golden/ref_answers.json where it is not built): every
function of the hot path, bit for bit."""
import numpy as np
import pytest

from conftest import pkg

PRESETS = list(range(10))


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def grid_record(g):
    """Every field of a grid dict, in key order, as one byte string."""
    return np.concatenate([np.ascontiguousarray(g[k]).reshape(-1).view(np.uint8) for k in sorted(g)])


def ref_scene(r, name, grid_res=64):
    m, fov, cam = pkg("scenes").build(r.api, name)
    return r.renderer(m, fov, cam, grid_res)


@pytest.mark.parametrize("spp", [1, 2, 3, 4, 7, 16, 64, 100, 256])
def test_sample_table(port, ref_answers, spp):
    ref_answers.check("sample_table/%d" % spp, bits(port.sample_table(spp)), lambda r: bits(r.sample_table(spp)))


def test_sample_table_single_sample_is_pixel_corner(port):
    # N = 1: the only sample sits at (-0.5, -0.5), the pixel's lower-left corner (SURVEY a2)
    assert port.sample_table(1).tolist() == [[-0.5, -0.5]]


def test_ray_triangle_variants_against_reference_functions(port, ref_answers):
    """Per case and variant: hit flag, then t / u / v bits (0 on a miss)."""
    rs = np.random.RandomState(11)
    cases = []
    for i in range(4000):
        v = rs.uniform(-1, 1, (3, 3)).astype(np.float32)
        o = rs.uniform(-2, 2, 3).astype(np.float32)
        target = (v[0] * 0.3 + v[1] * 0.3 + v[2] * 0.4 + rs.normal(scale=0.3, size=3)).astype(np.float32)
        d = (target - o).astype(np.float32)
        d /= np.float32(np.linalg.norm(d))
        e1, e2 = v[1] - v[0], v[2] - v[0]
        n = np.cross(e1, e2).astype(np.float32)
        n /= np.float32(max(np.linalg.norm(n), 1e-20))
        if i % 50 == 0:  # degenerate: ray in the triangle's plane / zero-area triangle
            d = (e1 / np.float32(max(np.linalg.norm(e1), 1e-20))).astype(np.float32)
        if i % 97 == 0:
            v[2] = v[1]
        cases.append((o, d, v[0].copy(), v[1].copy(), v[2].copy(), n))

    def run(impl):
        out = np.zeros((len(cases), 2, 4), np.uint32)
        for i, c in enumerate(cases):
            for variant in (0, 1):
                hit, tuv = impl.tri_test(variant, *c)
                out[i, variant, 0] = hit
                if hit:
                    out[i, variant, 1:] = bits(tuv)
        return out

    got = run(port)
    ref_answers.check("tri_test/4000", got, run)
    assert got[:, :, 0].sum(axis=0).min() > 500


@pytest.mark.parametrize("name", PRESETS)
def test_grid_build_matches_reference(port, ref_answers, scene_data, name):
    sd = scene_data(name)
    got = grid_record(port.scene(sd.vtx, sd.tri, 64).grid())
    ref_answers.check("grid/%s/g64" % name, got, lambda r: grid_record(ref_scene(r, name).grid()))


@pytest.mark.parametrize("res", [1, 5, 32, 100])
def test_grid_build_other_resolutions(port, ref_answers, scene_data, res):
    sd = scene_data("torusknot")
    got = grid_record(port.scene(sd.vtx, sd.tri, res).grid())
    ref_answers.check("grid/torusknot/g%d" % res, got, lambda r: grid_record(ref_scene(r, "torusknot", res).grid()))


def test_tight_candidate_ranges_give_identical_grids(port, scene_data):
    """The literal port enumerates the reference's (FLT_MIN-seeded, hence huge) candidate ranges;
    its optional tight mode and the GPU build cut them at the true triangle maximum.  Same lists."""
    for name, res in (("killeroo", 64), ("tiger_soup_small", 48), ("cornell", 64), ("head", 33)):
        sd = scene_data(name)
        a = port.scene(sd.vtx, sd.tri, res).grid()
        b = port.scene(sd.vtx, sd.tri, res, tight_ranges=True).grid()
        for k in a:
            assert np.array_equal(np.asarray(a[k]), np.asarray(b[k])), (name, k)


@pytest.mark.parametrize("name", PRESETS)
def test_render_matches_reference(port, ref_answers, scene_data, name):
    """Image through the reference's own Renderer/worker pool, and per-sample hit records through
    its GenerateRay + Grid::Intersect, against the port."""
    sd = scene_data(name)
    w, h, spp = 160, 96, 4
    o = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, w, h, spp, want_hits=True, want_tuv=True)
    key = "port_render/%s/%dx%dx%d/" % (name, w, h, spp)
    ref_answers.check(key + "bgra", o["bgra"], lambda r: ref_scene(r, name).render(w, h, spp)[1])
    ref_answers.check(key + "tri", o["tri"], lambda r: ref_scene(r, name).trace_hits(w, h, spp)[0])
    ref_answers.check(key + "tuv", np.stack([bits(o[k]) for k in "tuv"]),
                      lambda r: np.stack([bits(a) for a in ref_scene(r, name).trace_hits(w, h, spp)[1:]]))


def test_primary_rays_match_reference(port, ref_answers, scene_data):
    import ctypes as C
    sd = scene_data("killeroo")
    w, h, spp = 97, 53, 5
    xs = (0, 1, 50, 96)
    smp = port.sample_table(spp)
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    cam32 = np.ascontiguousarray(sd.cam16, np.float32)
    F = C.POINTER(C.c_float)
    got = np.zeros((4, len(xs), spp, 2, 3), np.uint32)
    for y in range(10, 14):
        for j, x in enumerate(xs):
            for s in range(spp):
                o, d = np.zeros(3, np.float32), np.zeros(3, np.float32)
                port.lib.rto_generate_ray(cam32.ctypes.data_as(F), x, y, w, h, float(smp[s, 0]), float(smp[s, 1]),
                                          float(fov_xs), float(aspect), o.ctypes.data_as(F), d.ctypes.data_as(F))
                got[y - 10, j, s] = bits(o), bits(d)

    def want(r):
        ro, rd = ref_scene(r, "killeroo").generate_rays(w, h, spp, 10, 14)
        return np.stack([bits(ro[:, xs]), bits(rd[:, xs])], axis=3)

    ref_answers.check("primary_rays/killeroo/%dx%dx%d/rows10-14" % (w, h, spp), got, want)


def test_orthographic_rays_and_frame_match_reference(port, ref_answers, scene_data):
    """camera.h:25-36: the orthographic branch.  RenderTile never takes it, so the reference side is GenerateRay
    called with ortho = true, then Grid::Intersect on those rays; the port's whole ortho frame must carry the same
    per-sample hits."""
    import ctypes as C
    ys, xs = (0, 5, 36), (0, 1, 30, 60)
    for name, width_ortho in (("cornell", 1.7), ("killeroo", 1.3)):
        sd = scene_data(name)
        w, h, spp = 61, 37, 3
        smp = port.sample_table(spp)
        _, aspect = port.camera_constants(sd.fov, w, h)
        cam32 = np.ascontiguousarray(sd.cam16, np.float32)
        F = C.POINTER(C.c_float)
        port.lib.rto_generate_ray_ortho.argtypes = [F, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, C.c_float,
                                                    C.c_float, C.c_float, F, F]
        got = np.zeros((len(ys), len(xs), spp, 2, 3), np.uint32)
        for i, y in enumerate(ys):
            for j, x in enumerate(xs):
                for k in range(spp):
                    o, d = np.zeros(3, np.float32), np.zeros(3, np.float32)
                    port.lib.rto_generate_ray_ortho(cam32.ctypes.data_as(F), x, y, w, h, float(smp[k, 0]), float(smp[k, 1]),
                                                    width_ortho, float(aspect), o.ctypes.data_as(F), d.ctypes.data_as(F))
                    got[i, j, k] = bits(o), bits(d)

        def ref_rays(r):
            return ref_scene(r, name).generate_rays_ortho(w, h, spp, 0, h, width_ortho)

        def want_rays(r):
            ro, rd = ref_rays(r)
            return np.stack([bits(ro[ys][:, xs]), bits(rd[ys][:, xs])], axis=3)

        def want_hits(r):
            idx, t, u, v = ref_scene(r, name).intersect_rays(*ref_rays(r))
            return np.stack([idx, bits(t), bits(u), bits(v)])

        key = "ortho/%s/%r/%dx%dx%d/" % (name, width_ortho, w, h, spp)
        ref_answers.check(key + "rays", got, want_rays)
        o = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, w, h, spp, want_hits=True, want_tuv=True,
                                                  ortho_width=width_ortho)
        hits = np.stack([o["tri"].ravel()] + [bits(o[k].ravel()) for k in "tuv"])
        ref_answers.check(key + "hits", hits, want_hits)
        assert (hits[0] != 0xFFFFFFFF).sum() > 500


def test_shading_alternates_restate_the_commented_lines(port, ref_answers, scene_data):
    """renderer.cpp:116 "Vec3f n = tri.n" and :118 "col += Vec3f(t / 3)" have no call site to run; the port's two
    extra shading modes are checked against those expressions evaluated on the reference's own hits."""
    sd = scene_data("cornell")
    w, h = 48, 40
    ps = port.scene(sd.vtx, sd.tri, 64)
    cam, fov, tri = sd.cam16, sd.fov, sd.tri
    o = ps.render(cam, fov, w, h, 1, want_hits=True, want_tuv=True)
    idx, t = o["tri"], o["t"]
    ref_answers.check("hits/cornell/%dx%dx1" % (w, h), np.stack([idx, bits(t)]),
                      lambda r: (lambda a: np.stack([a[0], bits(a[1])]))(ref_scene(r, "cornell").trace_hits(w, h, 1)))
    hit = idx[:, :, 0] != 0xFFFFFFFF
    miss_grey = (np.arange(h, dtype=np.float32) / np.float32(h))[:, None] * np.ones((1, w), np.float32)

    def pack(rgb):  # lin_alg.h:125-132 after renderer.cpp:124-131 with one sample
        c = np.sqrt(rgb.astype(np.float64)).astype(np.float32)  # powf(x, .5f): never a different byte (exhaustive scan)
        b = np.where(c > 1.0, 255, (c * np.float32(255.0)).astype(np.int64) & 0xFF).astype(np.uint32)
        return (b[..., 0] << 16) | (b[..., 1] << 8) | b[..., 2]

    face = tri[:, 3:6].copy().view(np.float32)[np.where(hit, idx[:, :, 0], 0)]
    want_face = np.where(hit[..., None], (face + np.float32(1.0)) * np.float32(0.5), miss_grey[..., None])
    got_face = ps.render(cam, fov, w, h, 1, shade_mode=1)["bgra"]
    assert np.array_equal(got_face, pack(want_face))
    depth = (t[:, :, 0] / np.float32(3))[..., None] * np.ones(3, np.float32)
    want_depth = np.where(hit[..., None], depth, miss_grey[..., None])
    got_depth = ps.render(cam, fov, w, h, 1, shade_mode=2)["bgra"]
    assert np.array_equal(got_depth, pack(want_depth))
    assert not np.array_equal(got_face, got_depth)


def test_arbitrary_rays_match_reference(port, ref_answers, scene_data):
    sd = scene_data("cornell")
    ps = port.scene(sd.vtx, sd.tri, 64)
    rs = np.random.RandomState(5)
    n = 5000
    o = rs.uniform(-1.2, 1.2, (n, 3)).astype(np.float32)
    d = rs.normal(size=(n, 3)).astype(np.float32)
    d /= np.linalg.norm(d, axis=1, keepdims=True).astype(np.float32)
    d[:800, 0] = 0.0
    d[400:1200, 2] = 0.0
    o[2000:3500] = rs.uniform(-0.4, 0.4, (1500, 3)).astype(np.float32)
    keep = np.abs(d).sum(axis=1) > 0
    o, d = o[keep], d[keep]

    def record(a):
        return np.stack([a[0]] + [bits(a[i]) for i in (1, 2, 3)])

    ref_answers.check("arbitrary_rays/cornell/5000", record(ps.intersect_rays(o, d, 0)),
                      lambda r: record(ref_scene(r, "cornell").intersect_rays(o, d)))


def test_gamma_powf_vs_sqrtf_is_at_most_one_lsb(port):
    """The CUDA kernel computes gamma 1/2 with IEEE sqrtf, the reference with glibc powf(x, .5f).
    Scan EVERY float in [0, 1] (and a band above): count inputs where the two differ and where that
    changes the 8-bit channel.  Documented in DESIGN.md; the image tolerance (<= 1 LSB) rests on it."""
    one = np.array([1.0], np.float32).view(np.uint32)[0]
    diff, byte_diff = port.powf_vs_sqrtf(0, int(one) + (1 << 20))
    total = int(one) + (1 << 20)
    assert diff <= total * 1e-3
    assert byte_diff == 0, (diff, byte_diff)  # measured: 678 509 of 1 066 401 792 floats differ, none changes a byte
