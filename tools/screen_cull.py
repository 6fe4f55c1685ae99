"""Screen boxes of the pair records for one camera: the CPU restatement of csrc/pack.cu screen_boxes_kernel, the
pre-pass of K1's screen cull (DESIGN.md section 3, profiles/r04_screen_cull.txt).

Every triangle gets a box in the image plane of generate_ray -- the (x, y) it forms before normalising,
x = ndc_x * fov_xs, y = ndc_y * fov_xs / aspect -- outside which no ray of that camera can be accepted by the fp32
Moeller-Trumbore test; a pair's box is the union of its two.  Computed in float64: the projected triangle with each
edge line pushed outwards by SAFETY x a bound on the image-plane error of that edge's part of the test, narrowed
outwards to float32.  Written operation by operation, without contraction, so that a device pre-pass can restate it
bit for bit.

Used by tools/warp_walk_model.py --screen-cull / --warp-scan (how many pair iterations a warp could skip) and by
tests/test_screen_cull_cpu.py (no culled ray is accepted by the oracle port) and tests/test_cull_scan_cpu.py."""
import numpy as np

EPS = 2.0 ** -24
TAU = 2.0 ** -6          # a vertex must lie clearly in front of the camera: depth w > TAU * |camera-space vector|
C_ROUND, C_DIR = 16.0, 16.0  # rounding-error constants of the test and of generate_ray's direction (DESIGN.md)
SAFETY = 16.0  # the slack used is SAFETY x the derived bound
KAPPA_MAX = 1.0e4        # cameras whose 3x3 has a larger condition number cull nothing
DUMMY = 0xFFFFFFFF       # tri index of the unhittable b half of an odd list's last pair (pack.cu)
INF = float("inf")


def camera_terms(cam16, fov_xs, aspect):
    """-> (inverse 3x3 as 9 floats, scale K, ok): the per-frame terms, as every thread of the kernel derives them."""
    m = list(np.asarray(cam16, np.float32).reshape(4, 4)[:3, :3].reshape(-1).astype(np.float64))
    m00, m01, m02, m10, m11, m12, m20, m21, m22 = m
    c00 = m11 * m22 - m12 * m21
    c01 = m12 * m20 - m10 * m22
    c02 = m10 * m21 - m11 * m20
    det = m00 * c00 + m01 * c01 + m02 * c02
    with np.errstate(all="ignore"):
        inv = [c00 / det, (m02 * m21 - m01 * m22) / det, (m01 * m12 - m02 * m11) / det,
               c01 / det, (m00 * m22 - m02 * m20) / det, (m02 * m10 - m00 * m12) / det,
               c02 / det, (m01 * m20 - m00 * m21) / det, (m00 * m11 - m01 * m10) / det]
    fro = 0.0
    for x in m:
        fro = fro + x * x
    fro = np.sqrt(fro)
    fro_inv = 0.0
    for x in inv:
        fro_inv = fro_inv + x * x
    fro_inv = np.sqrt(fro_inv)
    fx = float(np.float32(fov_xs))
    fy = fx / float(np.float32(aspect))
    l_img = np.sqrt(1.0 + 4.0 * (fx * fx) + 4.0 * (fy * fy))
    with np.errstate(all="ignore"):
        k = EPS * fro * l_img / abs(det)
    ok = bool(np.isfinite(k) and det != 0.0 and np.isfinite(fro_inv) and fro * fro_inv <= KAPPA_MAX)
    return inv, float(k), ok


def triangle_boxes(v0, e1, e2, idx, origin, inv, k, ok, edges_out=None):
    """v0, e1, e2: (n, 3) float32 as the records hold them; idx: (n,) uint32.  -> (n, 4) float64 {xmin, xmax, ymin, ymax}:
    +-inf for "never cull", an empty box (+inf, -inf, ...) for the dummy triangle.  edges_out (a dict) receives the
    projected vertices "cx", "cy" and, per edge q = 0-1, 1-2, 2-0, its outward unit normal "nx", "ny" and push-out
    "off", each (3, n) -- what tests aim rays at."""
    v0, e1, e2 = (np.asarray(a, np.float32).astype(np.float64) for a in (v0, e1, e2))
    o = np.asarray(origin, np.float32).astype(np.float64)
    n = len(v0)
    with np.errstate(all="ignore"):
        verts = (v0, v0 + e1, v0 + e2)
        V, c, w, clen = [], [], [], []
        for p in verts:
            vx, vy, vz = p[:, 0] - o[0], p[:, 1] - o[1], p[:, 2] - o[2]
            cx = vx * inv[0] + vy * inv[3] + vz * inv[6]
            cy = vx * inv[1] + vy * inv[4] + vz * inv[7]
            cz = vx * inv[2] + vy * inv[5] + vz * inv[8]
            V.append((vx, vy, vz))
            c.append((cx / -cz, cy / -cz))
            w.append(-cz)
            clen.append(np.sqrt(cx * cx + cy * cy + cz * cz))
        R = np.maximum(np.maximum(_norm(V[0]), _norm(V[1])), _norm(V[2]))
        l1, l2 = _norm((e1[:, 0], e1[:, 1], e1[:, 2])), _norm((e2[:, 0], e2[:, 1], e2[:, 2]))
        # rounding error of the three edge functions of the test: v's numerator (edge 0-1), u's (edge 2-0), and the
        # u + v <= 1 test (edge 1-2), which carries both numerators and the determinant
        base = (C_ROUND * (R * l1), C_ROUND * (R * (l1 + l2) + l1 * l2), C_ROUND * (R * l2))
        edges = ((0, 1), (1, 2), (2, 0))
        a2s = (c[1][0] - c[0][0]) * (c[2][1] - c[0][1]) - (c[1][1] - c[0][1]) * (c[2][0] - c[0][0])
        sgn = np.where(a2s < 0, -1.0, 1.0)
        nx, ny, off = [], [], []
        perim_slack = np.zeros(n)
        for q, (i, j) in enumerate(edges):
            dx, dy = c[j][0] - c[i][0], c[j][1] - c[i][1]
            lij = np.sqrt(dx * dx + dy * dy)
            cr = _norm(_cross(V[i], V[j]))
            dij = SAFETY * (k * (base[q] + C_DIR * cr) / (w[i] * w[j] * lij))
            nx.append(sgn * dy / lij)  # outward unit normal
            ny.append(-sgn * dx / lij)
            off.append(dij)
            perim_slack = perim_slack + lij * dij
        # vertex q lies on edges q-1 and q: its offset position solves n . s = slack for both lines
        px, py = [], []
        for q in range(3):
            a, b = (q + 2) % 3, q
            det2 = nx[a] * ny[b] - ny[a] * nx[b]
            px.append(c[q][0] + (off[a] * ny[b] - off[b] * ny[a]) / det2)
            py.append(c[q][1] + (nx[a] * off[b] - nx[b] * off[a]) / det2)
        box = np.stack([np.minimum(np.minimum(px[0], px[1]), px[2]), np.maximum(np.maximum(px[0], px[1]), px[2]),
                        np.minimum(np.minimum(py[0], py[1]), py[2]), np.maximum(np.maximum(py[0], py[1]), py[2])], 1)
        good = np.full(n, ok)
        for q in range(3):
            good &= w[q] > TAU * clen[q]
        good &= perim_slack < np.abs(a2s)
        good &= np.isfinite(box).all(1)
    if edges_out is not None:
        edges_out.update(cx=np.array([p[0] for p in c]), cy=np.array([p[1] for p in c]), nx=np.array(nx),
                         ny=np.array(ny), off=np.array(off))
    box[~good] = (-INF, INF, -INF, INF)
    box[np.asarray(idx) == DUMMY] = (INF, -INF, INF, -INF)
    return box


def pair_boxes(tboxes_a, tboxes_b):
    """Union of the two halves' boxes, narrowed outward to float32: (n, 4) float32 {xmin, xmax, ymin, ymax}."""
    lo_x = np.minimum(tboxes_a[:, 0], tboxes_b[:, 0])
    hi_x = np.maximum(tboxes_a[:, 1], tboxes_b[:, 1])
    lo_y = np.minimum(tboxes_a[:, 2], tboxes_b[:, 2])
    hi_y = np.maximum(tboxes_a[:, 3], tboxes_b[:, 3])
    return np.stack([round_down(lo_x), round_up(hi_x), round_down(lo_y), round_up(hi_y)], 1)


def round_down(x):
    f = np.asarray(x, np.float64).astype(np.float32)
    return np.where(f.astype(np.float64) > x, np.nextafter(f, np.float32(-INF)), f).astype(np.float32)


def round_up(x):
    f = np.asarray(x, np.float64).astype(np.float32)
    return np.where(f.astype(np.float64) < x, np.nextafter(f, np.float32(INF)), f).astype(np.float32)


def pair_records(ps):
    """The pairing of pack.cu on the port's grid: consecutive entries of each cell's ascending list.
    -> (cell_pair_start (num_cells + 1,), a (v0, e1, e2, idx), b (v0, e1, e2, idx)); b of an odd list's last pair is
    the dummy triangle."""
    g = ps.s.grid
    nc = int(g.num_cells)
    off = np.ctypeslib.as_array(g.cell_offset, (nc + 1,)).astype(np.int64)
    ti = np.ctypeslib.as_array(g.tri_index, (int(g.num_refs),)).astype(np.int64) if g.num_refs else np.zeros(0, np.int64)
    lens = np.diff(off)
    npairs = (lens + 1) // 2
    pstart = np.zeros(nc + 1, np.int64)
    np.cumsum(npairs, out=pstart[1:])
    cell_of = np.repeat(np.arange(nc), npairs)
    j = np.arange(pstart[-1]) - pstart[cell_of]
    ka = off[cell_of] + 2 * j
    kb = ka + 1
    has_b = kb < off[cell_of + 1]
    ia = ti[ka]
    ib = np.where(has_b, ti[np.minimum(kb, len(ti) - 1)], -1)
    vtx = ps.vtx.reshape(-1, 6)[:, :3]
    tri = ps.tri.reshape(-1, 6)[:, :3]

    def geom(ids):
        v = np.zeros((len(ids), 3, 3), np.float32)
        okm = ids >= 0
        v[okm] = vtx[tri[ids[okm]]]
        v0 = v[:, 0]
        e1 = (v[:, 1] - v0).astype(np.float32)
        e2 = (v[:, 2] - v0).astype(np.float32)
        idx = np.where(okm, ids, DUMMY).astype(np.uint32)
        # the dummy triangle of pack.cu (its box is empty whatever its geometry)
        v0 = np.where(okm[:, None], v0, np.float32([-1.0e18, 0, 0]))
        e1 = np.where(okm[:, None], e1, np.float32([1, 0, 0]))
        e2 = np.where(okm[:, None], e2, np.float32([0, 1, 0]))
        return v0, e1, e2, idx
    return pstart, geom(ia), geom(ib)


def scene_pair_boxes(ps, cam16, fov_xs, aspect):
    """-> (cell_pair_start, (num_pairs, 4) float32 pair boxes) of the port scene for this camera"""
    pstart, a, b = pair_records(ps)
    inv, k, ok = camera_terms(cam16, fov_xs, aspect)
    origin = np.asarray(cam16, np.float32).reshape(-1)[12:15]
    return pstart, pair_boxes(triangle_boxes(*a, origin, inv, k, ok), triangle_boxes(*b, origin, inv, k, ok))


def footprint_skips(boxes, x, y):
    """The warp scan of K1's screen cull (csrc/warp_trace.cuh test_pair_list) for the lanes standing on one
    cell: boxes (n, 4) float32 of the cell's pairs, x / y the float32 image points of those lanes.  -> (n,) bool, True
    where a pair's box is disjoint from the footprint, the bounding box of the points -- then every lane lies outside
    it.  A NaN point makes the footprint NaN, and nothing is skipped."""
    b = np.asarray(boxes, np.float32)
    x, y = np.asarray(x, np.float32), np.asarray(y, np.float32)
    if np.isnan(x).any() or np.isnan(y).any():
        return np.zeros(len(b), bool)
    x_lo, x_hi, y_lo, y_hi = x.min(), x.max(), y.min(), y.max()
    return (x_hi < b[:, 0]) | (x_lo > b[:, 1]) | (y_hi < b[:, 2]) | (y_lo > b[:, 3])


def image_point(px, py, w, h, off_x, off_y, fov_xs, aspect):
    """generate_ray's (x, y) in float32 (camera.h:8-47 before normalisation; the IEEE quotients of the exact path)"""
    f32 = np.float32
    ndc_x = (f32(px) + f32(off_x)) / f32(w) * f32(2) - f32(1)
    ndc_y = (f32(py) + f32(off_y)) / f32(h) * f32(2) - f32(1)
    return f32(ndc_x * f32(fov_xs)), f32(ndc_y * f32(fov_xs) / f32(aspect))


def _norm(v):
    return np.sqrt(v[0] * v[0] + v[1] * v[1] + v[2] * v[2])


def _cross(a, b):
    return (a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0])
