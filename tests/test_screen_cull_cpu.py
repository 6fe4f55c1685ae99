"""CPU checks of the screen boxes of tools/screen_cull.py (the go / no-go model of a screen cull for K1, DESIGN.md
section 10): no ray whose image-plane point lies outside a triangle's box is accepted by the oracle port's fp32
Moeller-Trumbore (bit-exact with the reference's IntersectRayTri), and the boxes that must never cull cover the plane."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tools"))
import screen_cull as sc  # noqa: E402

F = C.POINTER(C.c_float)
W, H, SPP = 48, 27, 2


def rotated(cam16, axis, deg):
    """the camera's 3x3 turned about `axis` (same origin)"""
    a = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    t = np.radians(deg)
    k = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    r = np.eye(3) + np.sin(t) * k + (1 - np.cos(t)) * k @ k
    c = np.asarray(cam16, np.float32).reshape(4, 4).copy()
    c[:3, :3] = (c[:3, :3].astype(np.float64) @ r).astype(np.float32)
    return c.reshape(-1)


def inside(cam16, vtx):
    """the same camera moved to the centre of the scene (vertices on every side of it)"""
    c = np.asarray(cam16, np.float32).reshape(4, 4).copy()
    p = vtx.reshape(-1, 6)[:, :3]
    c[3, :3] = ((p.min(0) + p.max(0)) / 2).astype(np.float32)
    return c.reshape(-1)


def tri_geometry(vtx, tri):
    p = vtx.reshape(-1, 6)[:, :3]
    t = tri.reshape(-1, 6)[:, :3]
    v0 = p[t[:, 0]]
    return v0, p[t[:, 1]], p[t[:, 2]], (p[t[:, 1]] - v0).astype(np.float32), (p[t[:, 2]] - v0).astype(np.float32)


@pytest.mark.parametrize("name", ["killeroo", "room", "torusknot"])
def test_no_culled_ray_is_accepted(port, scene_data, name):
    sd = scene_data(name)
    v0, v1, v2, e1, e2 = tri_geometry(sd.vtx, sd.tri)
    idx = np.arange(len(v0), dtype=np.uint32)
    smp = port.sample_table(SPP)
    fov_xs, aspect = port.camera_constants(sd.fov, W, H)
    pix = float(2 * fov_xs / W)
    checked = whole = 0
    for cam in (np.asarray(sd.cam16, np.float32).reshape(-1), rotated(sd.cam16, (1, 2, 3), 7.0), inside(sd.cam16, sd.vtx)):
        inv, k, ok = sc.camera_terms(cam, fov_xs, aspect)
        assert ok
        box = sc.pair_boxes(*(2 * (sc.triangle_boxes(v0, e1, e2, idx, cam[12:15], inv, k, ok),))).astype(np.float64)
        whole += int(np.isinf(box[:, 0]).sum())
        cam32 = np.ascontiguousarray(cam, np.float32)
        m = cam32.reshape(4, 4)[:3, :3]
        for py in range(H):
            for px in range(W):
                for s in range(SPP):
                    o, d = np.zeros(3, np.float32), np.zeros(3, np.float32)
                    port.lib.rto_generate_ray(cam32.ctypes.data_as(F), px, py, W, H, float(smp[s, 0]), float(smp[s, 1]),
                                              float(fov_xs), float(aspect), o.ctypes.data_as(F), d.ctypes.data_as(F))
                    x, y = sc.image_point(px, py, W, H, smp[s, 0], smp[s, 1], fov_xs, aspect)
                    # (x, y) are the floats generate_ray normalises: the direction follows from them bit for bit
                    z = np.float32(-1)
                    ls = np.float32(0) + x * x
                    ls = ls + y * y
                    ls = ls + z * z
                    il = np.float32(1) / np.sqrt(ls)
                    n = (x * il, y * il, z * il)
                    dd = [n[0] * m[0, j] + n[1] * m[1, j] + n[2] * m[2, j] for j in range(3)]
                    assert np.array_equal(np.array(dd, np.float32).view(np.uint32), d.view(np.uint32))
                    xf, yf = float(x), float(y)
                    out = (xf < box[:, 0]) | (xf > box[:, 1]) | (yf < box[:, 2]) | (yf > box[:, 3])
                    near = ((xf > box[:, 0] - 3 * pix) & (xf < box[:, 1] + 3 * pix) &
                            (yf > box[:, 2] - 3 * pix) & (yf < box[:, 3] + 3 * pix))
                    for t in np.nonzero(out & near)[0]:
                        hit, _ = port.tri_test(0, o, d, v0[t], v1[t], v2[t], np.zeros(3, np.float32))
                        assert not hit, (name, px, py, s, int(t))
                        checked += 1
    assert checked > 1000
    assert whole > 0  # the camera inside the scene has vertices behind it


def test_never_cull_and_dummy():
    cam = np.eye(4, dtype=np.float32)  # looks down -z from the origin
    inv, k, ok = sc.camera_terms(cam.reshape(-1), 0.5, 1.5)
    assert ok
    v0 = np.float32([[0, 0, -2], [0, 0, -2], [0, 0, -2], [np.nan, 0, -2], [-1e18, 0, 0], [0, 0, -2]])
    e1 = np.float32([[0.1, 0, 0], [0.1, 0, 3], [0.1, 0, 0], [0.1, 0, 0], [1, 0, 0], [0.1, 0, 0]])
    e2 = np.float32([[0, 0.1, 0], [0, 0.1, 0], [0, np.inf, 0], [0, 0.1, 0], [0, 1, 0], [0.1, 1e-9, 0]])
    idx = np.uint32([0, 1, 2, 3, sc.DUMMY, 5])
    b = sc.triangle_boxes(v0, e1, e2, idx, np.zeros(3, np.float32), inv, k, ok)
    assert np.all(np.isfinite(b[0])) and b[0, 0] < 0.0 < b[0, 1] * 20 and b[0, 1] - b[0, 0] < 0.06
    for t in (1, 2, 3, 5):  # crosses the camera plane / infinite / NaN / degenerate in projection
        assert tuple(b[t]) == (-np.inf, np.inf, -np.inf, np.inf), t
    assert tuple(b[4]) == (np.inf, -np.inf, np.inf, -np.inf)
    # a singular camera culls nothing
    assert not sc.camera_terms(np.zeros(16, np.float32), 0.5, 1.5)[2]
