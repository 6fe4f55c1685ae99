"""Soundness of the screen boxes of tools/screen_cull.py (K1's screen cull, DESIGN.md section 3) on inputs unlike the
presets: no ray whose float32 image-plane point lies outside a triangle's box may be accepted by the fp32
Moeller-Trumbore test -- any accepted triangle, not only the closest hit.

The test and generate_ray are restated over numpy float32 arrays (IEEE, one rounding per operation, no contraction), in
the operation order of the oracle port, and pinned bit for bit to it.  The scenes are raw triangle arrays built around a
camera -- slivers, nearly edge-on triangles, vertices at the depth threshold, triangles that cross the camera plane,
sub-pixel triangles, one triangle covering the view, coplanar duplicates -- at scale 1e-3, 1 and 1e4 and translated by
1e4; the cameras include non-orthonormal 3x3s up to the gate's condition number, singular ones, extreme fields of view
and aspects.  Rays: every sample of a frame, and rays aimed a few ulps and a fraction of the push-out outside every
projected edge and vertex and every box side.  tests/test_gpu_screen_cull_boxes.py renders the same cases on the device."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_screen_cull_cpu import inside, rotated

sys.path.insert(0, os.path.join(ROOT, "tools"))
import screen_cull as sc  # noqa: E402

F = C.POINTER(C.c_float)
f32 = np.float32
W, H, SPP = 128, 96, 2
NEAR_PX = 32           # preset frame rays: those within this many pixels of a box
PRESET_TRIS = 2000     # preset triangles per case (a random sample of those with a finite box)
CHUNK = 1 << 21        # (ray, triangle) items per vectorised test


# ---------------------------------------------------------------------------------------------- restatements

def mt32(o, d, v0, e1, e2):
    """rto_ray_tri (oracle/rt_oracle.c) on broadcastable (..., 3) float32 arrays, with e1 = v1 - v0 and e2 = v2 - v0 as
    the records hold them.  -> (accepted, t, u, v)"""
    o, d, v0, e1, e2 = (np.asarray(a, f32) for a in (o, d, v0, e1, e2))
    eps = f32(0.00000001)
    with np.errstate(all="ignore"):
        p0 = d[..., 1] * e2[..., 2] - d[..., 2] * e2[..., 1]
        p1 = d[..., 2] * e2[..., 0] - d[..., 0] * e2[..., 2]
        p2 = d[..., 0] * e2[..., 1] - d[..., 1] * e2[..., 0]
        det = e1[..., 0] * p0 + e1[..., 1] * p1 + e1[..., 2] * p2
        ok = ~((det > -eps) & (det < eps))
        inv_det = f32(1) / det
        t0, t1, t2 = o[..., 0] - v0[..., 0], o[..., 1] - v0[..., 1], o[..., 2] - v0[..., 2]
        u = (t0 * p0 + t1 * p1 + t2 * p2) * inv_det
        ok &= ~((u < 0) | (u > 1))
        q0 = t1 * e1[..., 2] - t2 * e1[..., 1]
        q1 = t2 * e1[..., 0] - t0 * e1[..., 2]
        q2 = t0 * e1[..., 1] - t1 * e1[..., 0]
        v = (d[..., 0] * q0 + d[..., 1] * q1 + d[..., 2] * q2) * inv_det
        ok &= ~((v < 0) | (u + v > 1))
        t = (e2[..., 0] * q0 + e2[..., 1] * q1 + e2[..., 2] * q2) * inv_det
    return ok & (t >= 0), t, u, v


def ray_origin(cam16):
    """rto_generate_ray's origin: the 4x4 applied to (0, 0, 0, 1)"""
    m = np.asarray(cam16, f32).reshape(-1)
    z = f32(0)
    return np.array([z * m[j] + z * m[4 + j] + z * m[8 + j] + m[12 + j] for j in range(3)], f32)


def ray_dirs(x, y, cam16):
    """rto_generate_ray's direction for float32 image-plane points (x, y): normalise (x, y, -1), then the 3x3"""
    m = np.asarray(cam16, f32).reshape(4, 4)
    x, y = np.asarray(x, f32), np.asarray(y, f32)
    z = f32(-1)
    ls = f32(0) + x * x
    ls = ls + y * y
    ls = ls + z * z
    il = f32(1) / np.sqrt(ls)
    n = (x * il, y * il, z * il)
    return np.stack([n[0] * m[0, j] + n[1] * m[1, j] + n[2] * m[2, j] for j in range(3)], -1)


def frame_points(w, h, smp, fov_xs, aspect):
    """generate_ray's (x, y) of every sample of a w x h frame: two (h, w, spp) float32 arrays"""
    px = np.arange(w, dtype=f32)[None, :, None]
    py = np.arange(h, dtype=f32)[:, None, None]
    x, y = sc.image_point(px, py, w, h, smp[None, None, :, 0], smp[None, None, :, 1], fov_xs, aspect)
    return np.broadcast_to(x, (h, w, len(smp))).copy(), np.broadcast_to(y, (h, w, len(smp))).copy()


# ---------------------------------------------------------------------------------------------- cameras and scenes

def look_at(eye, target, up=(0.0, 1.0, 0.0)):
    """cam16 looking from eye at target: rows right, up, back, origin (generate_ray's dir = (x, y, -1) x 3x3)"""
    eye, target = np.asarray(eye, np.float64), np.asarray(target, np.float64)
    f = (target - eye) / np.linalg.norm(target - eye)
    r = np.cross(f, up)
    r /= np.linalg.norm(r)
    u = np.cross(r, f)
    c = np.eye(4)
    c[0, :3], c[1, :3], c[2, :3], c[3, :3] = r, u, -f, eye
    return c.astype(f32).reshape(-1)


def with_3x3(cam16, fn):
    c = np.asarray(cam16, f32).reshape(4, 4).astype(np.float64)
    c[:3, :3] = fn(c[:3, :3])
    return c.astype(f32).reshape(-1)


def sheared(cam16, kappa):
    """the 3x3 sheared in the image plane (the ray of (x, y) goes where the original camera's (x, y + a x) went), with
    a chosen so that |M|_F |M^-1|_F = kappa for a rotation M -- the condition number the cull's gate measures"""
    s = np.eye(3)
    s[0, 1] = np.sqrt(kappa - 3.0)
    return with_3x3(cam16, lambda m: s @ m)


def singular(cam16):
    return with_3x3(cam16, lambda m: np.stack([m[0], m[1], m[0]]))


def cameras(cam16, fov, pts):
    """-> [(label, cam16, fov, width, height, culls)]: the adversarial cameras derived from one camera.  culls: False
    where every box must be infinite (the gate refuses the 3x3), else the case must cull something.  pts: the scene's
    vertices (for the camera moved inside the scene)."""
    cam16 = np.asarray(cam16, f32).reshape(-1)
    return [("preset", cam16, fov, W, H, True),
            ("rotated", rotated(cam16, (1, 2, 3), 30.0), fov, W, H, True),
            ("inside", inside(cam16, np.concatenate([pts, np.zeros_like(pts)], 1)), fov, W, H, True),
            ("m_x1e-3", with_3x3(cam16, lambda m: m * 1e-3), fov, W, H, True),
            ("m_x1e3", with_3x3(cam16, lambda m: m * 1e3), fov, W, H, True),
            ("kappa10", sheared(cam16, 10.0), fov, W, H, True),
            ("kappa1e3", sheared(cam16, 1.0e3), fov, W, H, True),
            ("kappa9e3", sheared(cam16, 0.9e4), fov, W, H, True),
            ("kappa1.1e4", sheared(cam16, 1.1e4), fov, W, H, False),
            ("singular", singular(cam16), fov, W, H, False),
            ("fov1", cam16, 1.0, W, H, True),
            ("fov90", cam16, 90.0, W, H, True),
            ("fov170", cam16, 170.0, W, H, True),
            ("aspect0.05", cam16, fov, 16, 320, True),
            ("aspect1", cam16, fov, 112, 112, True),
            ("aspect20", cam16, fov, 320, 16, True)]


CAMERA_LABELS = [c[0] for c in cameras(np.eye(4, dtype=f32), 60.0, np.zeros((1, 3), f32))]
SYN_FOV = 60.0
SYN_EYE, SYN_TARGET = (0.4, 0.3, 2.5), (0.0, 0.0, 0.0)
# scale of the synthetic scenes around their camera, and a translation of scene and camera together
SCENE_FOLLOWS = ("preset", "rotated", "fov1", "fov90", "fov170", "aspect0.05", "aspect1", "aspect20")
SYN_PLACEMENTS = {"s1e-3": (1e-3, 0.0), "s1": (1.0, 0.0), "s1e4": (1e4, 0.0), "t1e4": (1.0, 1e4)}


def synthetic_tris(fx, fy, pix, rng):
    """Triangles in the camera space of a camera with half extents fx, fy of its image plane (pix = one pixel there):
    a vertex c maps to the image point (c.x / -c.z, c.y / -c.z).  -> (n, 3, 3) float64"""
    def at(x, y, z):  # camera-space point with image point (x fx, y fy) at depth z
        return np.stack([x * fx * z, y * fy * z, -z], -1)

    tris = []
    # ordinary triangles in view
    for _ in range(24):
        cxy = rng.uniform(-0.9, 0.9, 2)
        z = rng.uniform(1.0, 6.0)
        tris.append([at(*(cxy + rng.uniform(-0.15, 0.15, 2)), z * rng.uniform(0.9, 1.1)) for _ in range(3)])
    ordinary = tris[:3]
    # slivers: aspect 1e-4 (and 1e-3, 1e-2), along random directions
    for k in range(12):
        asp = (1e-4, 1e-4, 1e-3, 1e-2)[k % 4]
        a, b = rng.uniform(-0.8, 0.8, 2), rng.uniform(-0.8, 0.8, 2)
        nrm = np.array([-(b - a)[1], (b - a)[0]])
        z = rng.uniform(1.0, 4.0, 3)
        tris.append([at(*a, z[0]), at(*b, z[1]), at(*((a + b) / 2 + asp * nrm), z[2])])
    # nearly edge-on: three image points on a line at different depths lie in a plane through the camera origin; the
    # vertices are moved off it by delta x their distance
    for k in range(12):
        delta = (1e-6, 1e-6, 1e-4, 1e-2)[k % 4]
        p0, dr = rng.uniform(-0.5, 0.5, 2), rng.normal(size=2)
        dr /= np.linalg.norm(dr)
        c = np.array([at(*(p0 + s * dr), z) for s, z in zip(rng.uniform(-0.4, 0.4, 3), rng.uniform(1.0, 5.0, 3))])
        n = np.cross(c[1], c[2])
        n /= np.linalg.norm(n)
        tris.append([p + delta * np.linalg.norm(p) * n for p in c])
    # one vertex at depth tau |c| (1 -+ 1e-6): far outside the view, the other two in it
    for k in range(8):
        eps = 1e-6 if k % 2 else -1e-6
        g = sc.TAU * (1 + eps)
        r, phi = rng.uniform(0.5, 3.0), rng.uniform(0, 2 * np.pi)
        w = r * g / np.sqrt(1 - g * g)
        far = np.array([r * np.cos(phi), r * np.sin(phi), -w])
        a = rng.uniform(-0.5, 0.5, 2)
        tris.append([far, at(*a, 2.0), at(*(a + rng.uniform(-0.3, 0.3, 2)), 2.5)])
    # crossing the camera plane: two vertices in view, one behind the camera
    for _ in range(4):
        a = rng.uniform(-0.6, 0.6, 2)
        back = at(*rng.uniform(-0.5, 0.5, 2), 1.0) * np.array([1.0, 1.0, -0.5])
        tris.append([at(*a, rng.uniform(1.0, 2.0)), at(*(a + rng.uniform(-0.4, 0.4, 2)), rng.uniform(1.0, 2.0)), back])
    # sub-pixel triangles, far away: 0.05 to 0.5 pixels across
    for _ in range(30):
        cxy, z = rng.uniform(-0.9, 0.9, 2), rng.uniform(10.0, 50.0)
        size = rng.uniform(0.05, 0.5) * pix
        tris.append([at(*(cxy + size * rng.uniform(-1, 1, 2) / np.array([fx, fy])), z * rng.uniform(0.99, 1.01))
                     for _ in range(3)])
    # one triangle covering the whole view, behind everything else
    tris.append([at(-4.0, -4.0, 60.0), at(4.0, -4.0, 60.0), at(0.0, 4.0, 60.0)])
    # coplanar duplicates: the same triangle again, and with its vertices rotated
    for t in ordinary:
        tris.append(list(t))
        tris.append([t[1], t[2], t[0]])
    return np.array(tris, np.float64)


def mesh_arrays(world):
    """(n, 3, 3) world-space triangles -> the vtx (3n, 6) / tri (n, 6) arrays of a mesh (own vertices per triangle,
    face normal as vertex normal)"""
    p = np.asarray(world, f32).reshape(-1, 3, 3)
    n = np.cross((p[:, 1] - p[:, 0]).astype(np.float64), (p[:, 2] - p[:, 0]).astype(np.float64))
    with np.errstate(all="ignore"):
        n = n / np.linalg.norm(n, axis=1, keepdims=True)
    n = np.nan_to_num(n).astype(f32)
    vtx = np.concatenate([p.reshape(-1, 3), np.repeat(n, 3, 0)], 1).astype(f32)
    tri = np.zeros((len(p), 6), np.uint32)
    tri[:, :3] = np.arange(3 * len(p), dtype=np.uint32).reshape(-1, 3)
    tri[:, 3:] = n.view(np.uint32)
    return np.ascontiguousarray(vtx), tri


def synthetic_cases(port, placement):
    """-> [(label, vtx, tri, cam16, fov, width, height, culls)]: the synthetic scene of one placement under every
    adversarial camera.  The scene is built in the camera space of the unmodified camera, and follows the camera (is
    built in its camera space, so that it fills the view) only where the view turns or changes its extent.  A scaled
    3x3 sees the same image through directions of length 1e-3 or 1e3; a sheared one sees it sheared, mostly outside
    the frame, through world-space error terms that grow with the condition number."""
    scale, shift = SYN_PLACEMENTS[placement]
    base = look_at(np.asarray(SYN_EYE) * scale + shift, np.asarray(SYN_TARGET) * scale + shift)
    rng = np.random.default_rng(7)
    out = []
    for label, cam, fov, w, h, culls in cameras(base, SYN_FOV, np.zeros((1, 3), f32)):
        if label == "inside":
            continue  # the scene is built around its camera: "crossing" and "tau" cover vertices behind it
        view = cam if label in SCENE_FOLLOWS else base
        fov_xs, aspect = port.camera_constants(fov, w, h)
        fx, fy = float(fov_xs), float(fov_xs) / float(aspect)
        tris = synthetic_tris(fx, fy, 2 * fx / w, np.random.default_rng(rng.integers(1 << 30))) * scale
        c = np.asarray(view, f32).reshape(4, 4).astype(np.float64)
        world = c[3, :3] + tris @ c[:3, :3]
        vtx, tri = mesh_arrays(world)
        out.append((label, vtx, tri, cam, fov, w, h, culls))
    return out


def preset_cases(scene_data, name):
    sd = scene_data(name)
    pts = sd.vtx.reshape(-1, 6)[:, :3]
    return [(label, sd.vtx, sd.tri, cam, fov, w, h, culls) for label, cam, fov, w, h, culls in cameras(sd.cam16, sd.fov, pts)]


# ---------------------------------------------------------------------------------------------- the property

def triangle_records(vtx, tri):
    """(v0, e1, e2) float32 of every triangle as the records hold them"""
    p = vtx.reshape(-1, 6)[:, :3]
    t = tri.reshape(-1, 6)[:, :3]
    v0 = p[t[:, 0]]
    return v0, (p[t[:, 1]] - v0).astype(f32), (p[t[:, 2]] - v0).astype(f32)


def boxes_of(v0, e1, e2, cam16, fov_xs, aspect, edges=None):
    """every triangle's own box, narrowed outwards to float32 as a pair box is: (n, 4) float32"""
    inv, k, ok = sc.camera_terms(cam16, fov_xs, aspect)
    origin = np.asarray(cam16, f32).reshape(-1)[12:15]
    tb = sc.triangle_boxes(v0, e1, e2, np.arange(len(v0), dtype=np.uint32), origin, inv, k, ok, edges)
    return sc.pair_boxes(tb, tb), ok


class Tally:
    def __init__(self):
        self.outside = 0   # (ray, triangle) items whose image point is outside the triangle's box
        self.accepted = 0  # items the test accepts

    def check(self, x, y, t, cam16, v0, e1, e2, box, what):
        """the rays of the float32 image points (x, y) against triangles t: an accepted one must lie in its box"""
        o = ray_origin(cam16)
        for s in range(0, len(x), CHUNK):
            xs, ys, ts = x[s:s + CHUNK], y[s:s + CHUNK], t[s:s + CHUNK]
            b = box[ts]
            out = (xs < b[:, 0]) | (xs > b[:, 1]) | (ys < b[:, 2]) | (ys > b[:, 3])
            hit = mt32(o, ray_dirs(xs, ys, cam16), v0[ts], e1[ts], e2[ts])[0]
            bad = np.nonzero(hit & out)[0]
            assert len(bad) == 0, (what, "accepted outside the box: tri %d at (%r, %r), box %r" % (
                ts[bad[0]], xs[bad[0]], ys[bad[0]], tuple(b[bad[0]])))
            self.outside += int(out.sum())
            self.accepted += int(hit.sum())


def frame_items(box, X, Y, fov_xs, aspect, w, h, tris, near_px):
    """(x, y, tri) of every frame sample within near_px pixels of each triangle's box (near_px None: every sample
    against every triangle)"""
    xs, ys = X.reshape(-1), Y.reshape(-1)
    if near_px is None:
        tr = np.repeat(tris, len(xs))
        return np.tile(xs, len(tris)), np.tile(ys, len(tris)), tr
    fx, fy = float(fov_xs), float(fov_xs) / float(aspect)
    spp = X.shape[2]
    parts = []
    for t in tris:
        b = box[t].astype(np.float64)
        with np.errstate(all="ignore"):
            x0 = np.floor((b[0] / fx + 1) / 2 * w) - near_px
            x1 = np.ceil((b[1] / fx + 1) / 2 * w) + near_px
            y0 = np.floor((b[2] / fy + 1) / 2 * h) - near_px
            y1 = np.ceil((b[3] / fy + 1) / 2 * h) + near_px
        x0, x1 = int(np.clip(np.nan_to_num(x0), 0, w)), int(np.clip(np.nan_to_num(x1), 0, w))
        y0, y1 = int(np.clip(np.nan_to_num(y0), 0, h)), int(np.clip(np.nan_to_num(y1), 0, h))
        if x1 <= x0 or y1 <= y0:
            continue
        idx = ((np.arange(y0, y1)[:, None] * w + np.arange(x0, x1)[None, :])[..., None] * spp +
               np.arange(spp)).reshape(-1)
        parts.append((idx, np.full(len(idx), t)))
    if not parts:
        return xs[:0], ys[:0], np.zeros(0, np.int64)
    idx = np.concatenate([p[0] for p in parts])
    return xs[idx], ys[idx], np.concatenate([p[1] for p in parts])


def ulp_step(a, k, sign):
    """a (float32) moved k ulps towards sign (+1 / -1 / 0)"""
    a = np.asarray(a, f32)
    out = a.copy()
    for _ in range(k):
        out = np.where(sign > 0, np.nextafter(out, f32(np.inf)), np.where(sign < 0, np.nextafter(out, f32(-np.inf)), out))
    return out.astype(f32)


def targeted_items(box, edges, finite):
    """(x, y, tri): image points on and just outside every projected vertex and edge of the triangles with a finite
    box -- moved outwards along the edge normal by 1/16, 1/4 and 1 of that edge's push-out, or by 1, 4 and 64 ulps in
    each coordinate -- and 1, 4 and 64 ulps inside and outside each side of the box, level with the vertex that
    defines it"""
    t = np.nonzero(finite)[0]
    if len(t) == 0:
        return np.zeros(0, f32), np.zeros(0, f32), np.zeros(0, np.int64)
    cx, cy = edges["cx"][:, t], edges["cy"][:, t]
    nx, ny, off = edges["nx"][:, t], edges["ny"][:, t], edges["off"][:, t]
    px, py, nnx, nny, noff = [], [], [], [], []
    for q in range(3):  # edge q runs from vertex q to vertex q + 1
        j = (q + 1) % 3
        for a in (0.0, 0.25, 0.5, 0.75):
            px.append(cx[q] + a * (cx[j] - cx[q]))
            py.append(cy[q] + a * (cy[j] - cy[q]))
            nnx.append(nx[q])
            nny.append(ny[q])
            noff.append(off[q])
        # the vertex q again, pushed along the other edge through it
        p = (q + 2) % 3
        px.append(cx[q])
        py.append(cy[q])
        nnx.append(nx[p])
        nny.append(ny[p])
        noff.append(off[p])
    px, py, nnx, nny, noff = (np.array(a) for a in (px, py, nnx, nny, noff))
    tt = np.broadcast_to(t, px.shape)
    xs, ys, ts = [], [], []
    for frac in (1 / 16, 1 / 4, 1.0):
        xs.append(px + frac * noff * nnx)
        ys.append(py + frac * noff * nny)
        ts.append(tt)
    on_x, on_y = px.astype(f32), py.astype(f32)
    xs.append(on_x)
    ys.append(on_y)
    ts.append(tt)
    for k in (1, 4, 64):
        xs.append(ulp_step(on_x, k, np.sign(nnx)))
        ys.append(ulp_step(on_y, k, np.sign(nny)))
        ts.append(tt)
    # the box sides: level with the projected vertex that reaches furthest
    b = box[t]
    vx, vy = cx.astype(f32), cy.astype(f32)
    for side, (coord, sign) in enumerate(((0, -1), (0, 1), (1, -1), (1, 1))):
        lvl = (vy if coord == 0 else vx)[np.argmax(sign * (cx if coord == 0 else cy), 0), np.arange(len(t))]
        for k in (1, 4, 64):
            for s in (sign, -sign):
                at = ulp_step(b[:, side], k, np.full(len(t), s))
                xs.append(at if coord == 0 else lvl)
                ys.append(lvl if coord == 0 else at)
                ts.append(t)
    x = np.concatenate([np.asarray(a, f32).reshape(-1) for a in xs])
    y = np.concatenate([np.asarray(a, f32).reshape(-1) for a in ys])
    tr = np.concatenate([np.asarray(a).reshape(-1) for a in ts])
    keep = np.isfinite(x) & np.isfinite(y)
    return x[keep], y[keep], tr[keep]


def check_case(port, case, preset):
    """-> (frame items outside their box, accepted items) of one (scene, camera)"""
    label, vtx, tri, cam, fov, w, h, culls = case
    fov_xs, aspect = port.camera_constants(fov, w, h)
    v0, e1, e2 = triangle_records(vtx, tri)
    edges = {}
    box, ok = boxes_of(v0, e1, e2, cam, fov_xs, aspect, edges)
    finite = np.isfinite(box).all(1)
    if not culls:
        assert not ok and not finite.any(), label
        return 0, 0
    assert ok and finite.any(), label  # the case culls something
    tally = Tally()
    X, Y = frame_points(w, h, port.sample_table(SPP), fov_xs, aspect)
    if preset:
        # a sample of the finite boxes, those that reach within NEAR_PX of the frame first
        m = NEAR_PX * 2 * float(fov_xs) / w
        near = finite & (box[:, 1] > X.min() - m) & (box[:, 0] < X.max() + m) & (box[:, 3] > Y.min() - m) & (box[:, 2] < Y.max() + m)
        rng = np.random.default_rng(11)
        cand = np.nonzero(near)[0] if near.sum() >= PRESET_TRIS // 4 else np.nonzero(finite)[0]
        tris = np.sort(rng.choice(cand, min(PRESET_TRIS, len(cand)), replace=False))
        x, y, t = frame_items(box, X, Y, fov_xs, aspect, w, h, tris, NEAR_PX)
    else:
        x, y, t = frame_items(box, X, Y, fov_xs, aspect, w, h, np.arange(len(v0)), None)
    tally.check(x, y, t, cam, v0, e1, e2, box, (label, "frame"))
    frame_outside = tally.outside
    x, y, t = targeted_items(box, edges, finite)
    tally.check(x, y, t, cam, v0, e1, e2, box, (label, "targeted"))
    # every finite box had rays aimed just outside each of its sides
    assert tally.outside - frame_outside >= 12 * int(finite.sum()), (label, tally.outside - frame_outside)
    return frame_outside, tally.accepted


# ---------------------------------------------------------------------------------------------- tests

def test_mt32_matches_port(port):
    """the vectorised test equals the port's rto_ray_tri bit for bit (accepted, and t, u, v of an accepted hit) on
    random triangles and on rays aimed at their edges and vertices, at several scales"""
    rng = np.random.default_rng(1)
    n = 100000
    scale = 10.0 ** rng.integers(-3, 5, n)[:, None]
    v = (rng.normal(size=(n, 3, 3)) * scale[:, :, None]).astype(f32)
    o = (rng.normal(size=(n, 3)) * scale * 3).astype(f32)
    # aim: a random point of the triangle, on an edge, or at a vertex, nudged by a few ulps-worth
    b = rng.dirichlet((1, 1, 1), n)
    kind = rng.integers(0, 3, n)
    b[kind == 1, rng.integers(0, 3, (kind == 1).sum())] = 0.0
    vert = rng.integers(0, 3, (kind == 2).sum())
    b[kind == 2] = 0.0
    b[np.nonzero(kind == 2)[0], vert] = 1.0
    b /= b.sum(1, keepdims=True)
    target = np.einsum("nk,nkj->nj", b, v.astype(np.float64))
    target += rng.normal(size=(n, 3)) * scale * 1e-7
    d = target - o
    d = (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(f32)
    # a tenth: direction nearly in the triangle's plane (det near its threshold)
    ep = rng.random(n) < 0.1
    nrm = np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0]).astype(np.float64)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    dd = d.astype(np.float64) - (d * nrm).sum(1, keepdims=True) * nrm * (1 - 1e-6)
    d[ep] = (dd[ep] / np.linalg.norm(dd[ep], axis=1, keepdims=True)).astype(f32)
    e1 = (v[:, 1] - v[:, 0]).astype(f32)
    e2 = (v[:, 2] - v[:, 0]).astype(f32)
    hit, t, u, vv = mt32(o, d, v[:, 0], e1, e2)
    assert 0.2 * n < hit.sum() < 0.8 * n
    for i in range(n):
        h, tuv = port.tri_test(0, o[i], d[i], v[i, 0], v[i, 1], v[i, 2], np.zeros(3, f32))
        assert h == bool(hit[i]), i
        if h:
            assert np.array_equal(tuv.view(np.uint32), np.array([t[i], u[i], vv[i]], f32).view(np.uint32)), i


def test_generate_ray_matches_port(port):
    """frame_points + ray_dirs + ray_origin equal rto_generate_ray bit for bit, here for a sheared, scaled camera"""
    w, h, spp = 24, 10, 4
    cam = with_3x3(sheared(look_at((3.0, -2.0, 7.0), (0.2, 0.1, -0.3)), 50.0), lambda m: m * 3.7)
    fov_xs, aspect = port.camera_constants(75.0, w, h)
    smp = port.sample_table(spp)
    X, Y = frame_points(w, h, smp, fov_xs, aspect)
    d = ray_dirs(X, Y, cam)
    o = ray_origin(cam)
    cam32 = np.ascontiguousarray(cam, f32)
    for py in range(h):
        for px in range(w):
            for s in range(spp):
                ro, rd = np.zeros(3, f32), np.zeros(3, f32)
                port.lib.rto_generate_ray(cam32.ctypes.data_as(F), px, py, w, h, float(smp[s, 0]), float(smp[s, 1]),
                                          float(fov_xs), float(aspect), ro.ctypes.data_as(F), rd.ctypes.data_as(F))
                assert np.array_equal(rd.view(np.uint32), d[py, px, s].view(np.uint32)), (px, py, s)
                assert np.array_equal(ro.view(np.uint32), o.view(np.uint32))


def test_gate_condition_numbers():
    """the sheared cameras straddle the gate as labelled"""
    cam = look_at((1.0, 2.0, 3.0), (0.0, 0.0, 0.0))
    for kappa, want in ((10.0, True), (1e3, True), (0.9e4, True), (1.1e4, False)):
        assert sc.camera_terms(sheared(cam, kappa), 0.5, 1.5)[2] == want, kappa
    assert not sc.camera_terms(singular(cam), 0.5, 1.5)[2]


@pytest.mark.parametrize("placement", list(SYN_PLACEMENTS))
def test_synthetic_scenes_sound(port, placement):
    cases = synthetic_cases(port, placement)
    assert len(cases) == len(CAMERA_LABELS) - 1
    res = {case[0]: check_case(port, case, preset=False) for case in cases}
    # the frame rays tested something (at fov 1 deg the few finite boxes cover the frame), and the test accepts rays
    # (at scale 1e-3, through directions of length 1e-3, every determinant is below its threshold)
    assert all(r[0] >= 1000 for k, r in res.items() if k not in ("kappa1.1e4", "singular", "fov1")), res
    assert sum(r[1] > 0 for r in res.values()) >= len(res) - 3, res


@pytest.mark.parametrize("name", ["killeroo", "room", "torusknot"])
def test_preset_scenes_sound(port, scene_data, name):
    res = {case[0]: check_case(port, case, preset=True) for case in preset_cases(scene_data, name)}
    # (the frame of a turned or sheared camera can show only a few boxes)
    assert sum(r[0] >= 1000 for r in res.values()) >= len(res) - 6, res
    assert sum(r[1] > 0 for r in res.values()) >= len(res) - 3, res
