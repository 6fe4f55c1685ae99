"""The warp scan of K1's screen cull (csrc/warp_trace.cuh test_pair_list) restated on the CPU
(tools/screen_cull.py footprint_skips): a pair whose box is disjoint from the footprint of a warp's image points -- their
bounding box -- has every lane outside it, and walking only the pairs the footprint keeps, in ascending list position,
gives every lane the (tri, t, u, v) of the serial walk that checks each pair's box against every lane.  Checked on the
presets and on the adversarial scenes and cameras of test_screen_cull_adversarial_cpu.py, whose builders it reuses, and
on lists with equally close hits inside one cell, where list order decides."""
import numpy as np
import pytest

from test_screen_cull_adversarial_cpu import (SYN_PLACEMENTS, boxes_of, frame_points, mt32, preset_cases, ray_dirs,
                                              ray_origin, sc, synthetic_cases, triangle_records)

f32 = np.float32
LIST = 96  # triangles in a replayed list: 48 pairs, two chunks of the scan


def outside(box, x, y):
    """(n, 4) boxes against (m,) points -> (n, m): the point lies outside the box (the serial per-lane check)"""
    b = np.asarray(box, f32)
    return ((x[None, :] < b[:, 0:1]) | (x[None, :] > b[:, 1:2]) | (y[None, :] < b[:, 2:3]) | (y[None, :] > b[:, 3:4]))


def warps(w, h, spp, smp, fov_xs, aspect):
    """the image points of K1's warps: 32 / spp pixels of a 2 x 2-quad (Morton) block, the sample index fastest"""
    X, Y = frame_points(w, h, smp, fov_xs, aspect)
    ppr = 32 // spp
    slot = np.arange(ppr)
    ox = (slot & 1) | ((slot >> 1) & 2) | ((slot >> 2) & 4)
    oy = ((slot >> 1) & 1) | ((slot >> 2) & 2)
    bw, bh = ox.max() + 1, oy.max() + 1
    for by in range(0, h - bh + 1, bh):
        for bx in range(0, w - bw + 1, bw):
            yield X[by + oy, bx + ox].reshape(-1), Y[by + oy, bx + ox].reshape(-1)


def replay(cam16, x, y, recs, pair_box, scan):
    """phase B of one warp on one pair list, all lanes owning every pair: -> per lane (tri, t, u, v) as uint32 bits.
    recs = (v0, e1, e2, idx) of the list's triangles, pair k = triangles 2k and 2k + 1."""
    v0, e1, e2, idx = recs
    o, d = ray_origin(cam16), ray_dirs(x, y, cam16)
    if scan:
        walk = np.nonzero(~sc.footprint_skips(pair_box, x, y))[0]
    else:
        walk = np.nonzero(~outside(pair_box, x, y).all(1))[0]
    bound = np.full(len(x), np.inf, f32)
    res = np.zeros((4, len(x)), f32)
    res[0] = np.uint32(0xFFFFFFFF).view(f32)
    for k in walk:
        for j in (2 * k, 2 * k + 1):  # a before b
            if j >= len(v0):
                continue
            ok, t, u, v = mt32(o, d, v0[j], e1[j], e2[j])
            take = ok & (t < bound)
            bound = np.where(take, t, bound)
            res[:, take] = np.stack([np.full(len(x), np.uint32(idx[j]).view(f32)), t, u, v])[:, take]
    return res.view(np.uint32), len(walk)


def lists_for(rng, n_tri, ties):
    """ascending triangle lists of LIST entries; ties: every triangle three times in a row (equal t, u and v)"""
    for _ in range(4):
        base = np.sort(rng.choice(n_tri, LIST // 3 if ties else LIST, replace=False))
        yield np.repeat(base, 3) if ties else base


def check_case(cam16, fov, w, h, spp, vtx, tri, port, rng, ties):
    smp = port.sample_table(spp)
    fov_xs, aspect = port.camera_constants(fov, w, h)
    v0, e1, e2 = triangle_records(vtx, tri)
    tbox, _ = boxes_of(v0, e1, e2, cam16, fov_xs, aspect)
    all_warps = list(warps(w, h, spp, smp, fov_xs, aspect))
    walked = [0, 0]
    for lst in lists_for(rng, len(v0), ties):
        tb = tbox[lst].astype(np.float64)
        if len(lst) % 2:
            tb = np.concatenate([tb, [[np.inf, -np.inf, np.inf, -np.inf]]])
        pair_box = sc.pair_boxes(tb[0::2], tb[1::2])
        recs = (v0[lst], e1[lst], e2[lst], lst.astype(np.uint32))
        for k in rng.choice(len(all_warps), min(len(all_warps), 48), replace=False):
            x, y = all_warps[k]
            skip = sc.footprint_skips(pair_box, x, y)
            assert outside(pair_box[skip], x, y).all()  # a skipped pair has every lane outside its box
            serial, n_serial = replay(cam16, x, y, recs, pair_box, False)
            scan, n_scan = replay(cam16, x, y, recs, pair_box, True)
            assert np.array_equal(serial, scan), (k, lst[:4])
            walked[0] += n_serial
            walked[1] += n_scan
    return walked


@pytest.mark.parametrize("placement", list(SYN_PLACEMENTS))
def test_scan_equals_serial_synthetic(port, placement):
    rng = np.random.default_rng(11)
    for label, vtx, tri, cam, fov, w, h, _ in synthetic_cases(port, placement):
        for spp in (1, 16):
            check_case(cam, fov, min(w, 64), min(h, 48), spp, vtx, tri, port, rng, False)


@pytest.mark.parametrize("name", ["killeroo", "room", "torusknot"])
@pytest.mark.parametrize("ties", [False, True])
def test_scan_equals_serial_presets(port, scene_data, name, ties):
    rng = np.random.default_rng(5)
    hits = 0
    for label, vtx, tri, cam, fov, w, h, _ in preset_cases(scene_data, name)[:4]:
        for spp in (1, 16):
            walked = check_case(cam, fov, 64, 48, spp, vtx, tri, port, rng, ties)
            assert walked[1] >= walked[0]  # the footprint is conservative: it keeps every pair some lane is inside
            hits += walked[0]
    assert hits > 0


def test_footprint_nan_keeps_everything():
    box = np.array([[0, 1, 0, 1], [5, 6, 5, 6], [np.inf, -np.inf, np.inf, -np.inf]], f32)
    x = np.array([0.5, 0.6], f32)
    y = np.array([0.5, 0.6], f32)
    assert list(sc.footprint_skips(box, x, y)) == [False, True, True]
    assert not sc.footprint_skips(box, np.array([0.5, np.nan], f32), y).any()
