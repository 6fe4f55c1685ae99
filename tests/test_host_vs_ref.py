"""CPU tests: the host library's Mesh / Matrix44f mirror against the unmodified reference
(oracle/_ref, or the digests of its answers in tests/golden/ref_answers.json where it is not built), bit for bit."""
import os

import numpy as np
import pytest

from conftest import pkg


@pytest.fixture(scope="module")
def host():
    return pkg("hostapi").host_api()


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def test_matrix_builders(host, ref_answers):
    def run(api):
        out = []
        for deg in (0.0, 30.0, 45.0, 90.0, -17.5, 123.456, 360.0):
            out += [api.rotation_x(deg), api.rotation_y(deg), api.rotation_z(deg)]
        out += [api.identity(), api.scaling(0.25), api.translation(-0.065, -0.1, 0.05)]
        for eye, at in [((-1.00001, 1.0, 1.0), (0.0, -0.2, 0.0)), ((0, 0, -2), (0, 0, 0)), ((-0.47, 0.15, -0.3), (1.0, -0.7, 0.9)),
                        ((-1.6, 1.2, -1.0), (0.0, 0.0, -0.1)), ((0.5, 0.5, 0.0), (0, 0, 0))]:
            out.append(api.look_at(eye, at))
        return np.stack([bits(np.asarray(m).reshape(-1)) for m in out])

    ref_answers.check("matrix_builders", run(host), lambda r: run(r.api))


def test_matrix_multiply_and_invert_random(host, ref_answers):
    """Per case: the product's bits, the inverse's success flag and bits."""
    rs = np.random.RandomState(3)
    cases = []
    for i in range(300):
        a = rs.normal(size=16).astype(np.float32) * np.float32(10.0 ** rs.randint(-3, 3))
        b = rs.normal(size=16).astype(np.float32)
        cases.append((a, b))

    def run(api):
        out = np.zeros((len(cases), 33), np.uint32)
        for i, (a, b) in enumerate(cases):
            ok, inv = api.invert(a)
            out[i, :16] = bits(api.multiply(a, b))
            out[i, 16] = ok
            out[i, 17:] = bits(inv)
        return out

    ref_answers.check("matrix_multiply_invert/300", run(host), lambda r: run(r.api))
    sing = np.zeros(16, np.float32)
    assert host.invert(sing)[0] is False
    if ref_answers.ref is not None:
        assert ref_answers.ref.api.invert(sing)[0] is False


def test_camera_constants(host, ref_answers, port):
    def run(api):
        out = []
        for fov in (30.0, 45.0, 51.0, 60.0, 75.0, 90.0, 1.0, 179.0):
            for w, h in ((512, 512), (1920, 1080), (3840, 2160), (67, 45)):
                out.append(bits(np.asarray(api.camera_constants(fov, w, h), np.float32)))
        return np.stack(out)

    got = run(host)
    assert np.array_equal(got, run(port))
    ref_answers.check("camera_constants", got, lambda r: run(r.api))


def test_cornell_box_and_quads(host, ref_answers):
    hv, ht = host.mesh().cornell_box().arrays()
    assert len(ht) == 32 and len(hv) == 64
    ref_answers.check("cornell_box/vtx", hv.view(np.uint32), lambda r: r.api.mesh().cornell_box().arrays()[0].view(np.uint32))
    ref_answers.check("cornell_box/tri", ht, lambda r: r.api.mesh().cornell_box().arrays()[1])


@pytest.mark.parametrize("name", list(range(10)) + ["tiger_soup_small"])
def test_scene_presets_bitwise(host, ref_answers, name):
    """Field of view and camera bits, triangles, vertex bits, bounding box bits of every preset."""
    scenes = pkg("scenes")

    def run(api):
        m, fov, cam = scenes.build(api, name)
        v, t = m.arrays()
        a, b = m.compute_aabb()
        return [bits(np.concatenate([[fov], np.asarray(cam).reshape(-1), np.asarray(a).reshape(-1),
                                     np.asarray(b).reshape(-1)])), np.ascontiguousarray(t), v.view(np.uint32)]

    got = run(host)
    for part, g in zip(("fov_cam_aabb", "tri", "vtx"), got):
        ref_answers.check("scene/%s/%s" % (name, part), g, lambda r, part=part: dict(zip(("fov_cam_aabb", "tri", "vtx"), run(r.api)))[part])


REF_MESH_DIR = "/root/reference/meshes"


@pytest.mark.skipif(not os.path.isdir(REF_MESH_DIR), reason="reference meshes not present")
def test_ascii_reader_matches_reference_and_assets(host, ref):
    meshapi = pkg("meshapi")
    names = sorted(f[:-4] for f in os.listdir(REF_MESH_DIR) if f.endswith(".dat"))
    assert len(names) == 17
    for name in names:
        for flip in ((False, True) if name == "table_chair" else (False,)):
            path = os.path.join(REF_MESH_DIR, name + ".dat")
            hm, rm = host.mesh(), ref.api.mesh()
            assert hm.read_file(path, flip) and rm.read_file(path, flip)
            hv, ht = hm.arrays()
            rv, rt = rm.arrays()
            assert np.array_equal(ht, rt), name
            assert np.array_equal(hv.view(np.uint32), rv.view(np.uint32)), name
            av, at = meshapi.load_meshbin(name, flip)
            assert np.array_equal(at, rt) and np.array_equal(av.view(np.uint32), rv.view(np.uint32)), name


def test_float_parsing_matches_reference_on_hard_decimals(host, ref_answers, tmp_path):
    """The host reader parses plain decimals on a fast exact path and leaves the rest to strtof (host/mesh.cpp);
    the reference uses fscanf("%f").  Positions written in every notation that occurs in practice plus the hard
    cases: float rounding midpoints spelled out exactly, one digit above / below them, 17+ significant digits,
    exponents, subnormals, signed zeros, huge values.  Non-indexed position-only mesh: three floats per line."""
    rs = np.random.RandomState(11)
    vals = []
    f32 = rs.standard_normal(600).astype(np.float32) * np.float32(10.0) ** rs.randint(-6, 7, 600).astype(np.float32)
    for x in f32:
        lo, hi = float(x), float(np.nextafter(x, np.float32(np.inf)))
        mid = (lo + hi) / 2                                   # exactly representable in double
        vals += ["%.6f" % lo, "%.9g" % lo, "%.17g" % lo, "%.30f" % mid, "%.25e" % mid,
                 "%.17g" % np.nextafter(mid, np.inf), "%.17g" % np.nextafter(mid, -np.inf)]
    vals += ["0", "-0", "0.0", "-0.000", "1e-45", "1.4e-45", "7e-46", "1e-40", "-3.4028235e38", "3.4028234e+38",
             "1e22", "1e23", "123456789012345678", "1234567890123456789012", "0.1", ".5", "5.", "+2.5", "1E3", "1e+3",
             "100000000000000000000e-20", "0.000000000000000000001e21", "9007199254740993", "16777217", "33554433"]
    while len(vals) % 9:
        vals.append("1")
    lines = [" ".join(vals[i:i + 3]) for i in range(0, len(vals), 3)]
    path = tmp_path / "hard.dat"
    path.write_text("\n".join(lines) + "\n")

    def run(api):
        m = api.mesh()
        assert m.read_file(str(path))
        v, _ = m.arrays()
        return np.ascontiguousarray(v[:, :3]).view(np.uint32)

    got = run(host)
    assert len(got) == len(vals) // 3
    ref_answers.check("float_parsing/hard_decimals", got, lambda r: run(r.api))


def test_reader_errors(host, tmp_path):
    m = host.mesh()
    assert not m.read_file(str(tmp_path / "missing.dat"))
    for i, text in enumerate(["", "1 2\n", "3\n\n0 0 0\n1 0 0\n", "0 0 0\n1 0 0\n0 1 0\n0 0 1\n",
                              "3\n\n0 0 0\n1 0 0\n0 1 0\n\n3\n\n0 1 7\n", "3\n\n0 0 0\n1 0 0\n0 1 0\n\n4\n\n0 1 2 0\n"]):
        p = tmp_path / ("bad%d.dat" % i)
        p.write_text(text)
        assert not m.read_file(str(p)), text
    good = tmp_path / "good.dat"
    good.write_text("0 0 0\r\n1 0 0\r\n0 1 0\r\n")  # CRLF, position only -> face normals
    assert m.read_file(str(good))
    v, t = m.arrays()
    assert len(t) == 1 and np.allclose(v[:, 3:], [[0, 0, 1]] * 3)
