"""K1's screen boxes on the device (csrc/pack.cu screen_boxes_kernel, read back with cuda_trace_download_screen_boxes)
against their float64 restatement tools/screen_cull.py, bit for bit: on the adversarial scenes and cameras of
tests/test_screen_cull_adversarial_cpu.py and on the ten presets at their own cameras, with the cull automatic and
forced on.  Also: the small-box count and the automatic gate, frames with the cull forced on against the oracle port,
the camera constants the boxes are cached under, and a scene replaced under an unchanged camera."""
import numpy as np
import pytest

from conftest import pkg
from test_screen_cull_adversarial_cpu import (SYN_PLACEMENTS, preset_cases, rotated, sc, synthetic_cases)

PRESETS = ["torusknot", "cornell", "room", "table_chair", "head", "room_cat", "water_knot", "griebel_teapot", "killeroo",
           "dwarf_hand_blob"]
SMALL_PIXELS = 32  # kScreenCullSmallPixels: a box of at most this many pixels a side counts small


def context(monkeypatch, cull, occ_mode=None):
    """a context on origin-relative records at every frame size; cull None = the automatic gate"""
    monkeypatch.setenv("RTM_REL_RECORDS", "2")
    if cull is None:
        monkeypatch.delenv("RTM_SCREEN_CULL", raising=False)
    else:
        monkeypatch.setenv("RTM_SCREEN_CULL", cull)
    if occ_mode is not None:
        monkeypatch.setenv("RTM_OCC_MODE", occ_mode)
        monkeypatch.setenv("RTM_THREADS", "1024" if occ_mode != "0" else "256")
    return pkg("capi").CudaTrace(1)


def expected_small(boxes, fov_xs, width):
    """screen_boxes_kernel's count, restated in float32: max side <= 32 pixels of the image plane"""
    small_side = np.float32(SMALL_PIXELS) * (np.float32(2) * np.float32(fov_xs) / np.float32(width))
    with np.errstate(invalid="ignore"):
        side = np.fmax(boxes[:, 1] - boxes[:, 0], boxes[:, 3] - boxes[:, 2])
    return int((side <= small_side).sum())


def check_boxes(ct, ps, cam, fov_xs, aspect, width, what):
    got, small, on = ct.download_screen_boxes()
    _, want = sc.scene_pair_boxes(ps, cam, fov_xs, aspect)
    assert got.shape == want.shape, what
    bad = np.nonzero((got.view(np.uint32) != want.view(np.uint32)).any(1))[0]
    assert len(bad) == 0, (what, "%d of %d pair boxes differ, first %d: device %r, restatement %r" % (
        len(bad), len(want), bad[0], tuple(got[bad[0]]), tuple(want[bad[0]])))
    assert small == expected_small(want, fov_xs, width), what
    assert on == (small * 5 >= len(want)), what
    return got, small


def grids_equal(ct, ps):
    g, og = ct.download_grid(), ps.grid()
    return all(np.array_equal(np.asarray(g[k]), np.asarray(og[k])) for k in ("dim", "cell_offset", "tri_index"))


def all_cases(port, scene_data, group):
    if group == "presets":
        return [(name, sd.vtx, sd.tri, sd.cam16, sd.fov, 96, 64, True) for name, sd in
                ((n, scene_data(n)) for n in PRESETS)]
    if group in SYN_PLACEMENTS:
        return synthetic_cases(port, group)
    name = group.split(":")[1]
    return preset_cases(scene_data, name)


GROUPS = list(SYN_PLACEMENTS) + ["presets", "preset:killeroo", "preset:room", "preset:torusknot"]


@pytest.mark.gpu
@pytest.mark.parametrize("cull", [None, "1"])
@pytest.mark.parametrize("group", GROUPS)
def test_device_boxes_match_restatement(port, scene_data, monkeypatch, cull, group):
    ct = context(monkeypatch, cull)
    try:
        for label, vtx, tri, cam, fov, w, h, _ in all_cases(port, scene_data, group):
            ps = port.scene(vtx, tri, 64)
            ct.upload_scene(vtx, tri, 64)
            # the device pairs the references of each cell as the restatement does on the port's grid
            assert grids_equal(ct, ps), label
            assert ct.download_screen_boxes()[0].shape == (0, 4), label  # nothing built for the new scene yet
            fov_xs, aspect = port.camera_constants(fov, w, h)
            ct.trace_tiles(ct.make_frame(w, h, 1, cam, fov_xs, aspect))
            check_boxes(ct, ps, cam, fov_xs, aspect, w, (group, label))
    finally:
        ct.close()


@pytest.mark.gpu
def test_no_boxes_without_the_cull(port, scene_data, monkeypatch):
    sd = scene_data("killeroo")
    ct = context(monkeypatch, "0")
    try:
        ct.upload_scene(sd.vtx, sd.tri, 64)
        fov_xs, aspect = port.camera_constants(sd.fov, 64, 48)
        ct.trace_tiles(ct.make_frame(64, 48, 1, sd.cam16, fov_xs, aspect))
        boxes, small, on = ct.download_screen_boxes()
        assert boxes.shape == (0, 4) and small == 0 and not on
    finally:
        ct.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "2"])
@pytest.mark.parametrize("group", GROUPS)
def test_frames_under_cull_match_oracle(port, scene_data, monkeypatch, mode, group):
    spp = 2
    ct = context(monkeypatch, "1", mode)
    try:
        for label, vtx, tri, cam, fov, w, h, _ in all_cases(port, scene_data, group):
            ps = port.scene(vtx, tri, 64)
            ct.upload_scene(vtx, tri, 64)
            fov_xs, aspect = port.camera_constants(fov, w, h)
            img = ct.trace_tiles(ct.make_frame(w, h, spp, cam, fov_xs, aspect, keep_hits=True)).copy()
            got = (img,) + tuple(ct.download_hits(w, h, spp))
            plain = ct.trace_tiles(ct.make_frame(w, h, spp, cam, fov_xs, aspect))  # the non-instrumented instantiation
            o = ps.render(cam, fov, w, h, spp, want_hits=True, want_tuv=True)
            want = (o["bgra"], o["tri"], o["t"], o["u"], o["v"])
            for k, (a, b) in enumerate(zip(got, want)):
                assert np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32)), (group, label, k)
            assert np.array_equal(plain, img), (group, label)
    finally:
        ct.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["killeroo", "room"])
def test_box_cache_keys(port, scene_data, monkeypatch, name):
    """one context, a sequence of frames that each change one input; the boxes must be rebuilt for every camera
    constant they depend on (origin, 3x3, fov_xs, aspect, width) and are reused across a change of height only.
    Every frame equals the same frame rendered without the cull (and the oracle's, where aspect = width / height)."""
    sd = scene_data(name)
    ps = port.scene(sd.vtx, sd.tri, 64)
    w0, h0, spp = 96, 64, 2
    fx0, a0 = port.camera_constants(sd.fov, w0, h0)
    moved = np.array(sd.cam16, np.float32).copy()
    moved[12:15] += np.array([0.02, -0.03, 0.01], np.float32)
    turned = rotated(moved, (1, 2, 3), 4.0)
    fov1 = sd.fov * 0.8
    fx1, _ = port.camera_constants(fov1, w0, h0)
    a1 = np.float32(a0 * np.float32(1.25))
    # (label, cam, fov or None when aspect != w / h, fov_xs, aspect, width, height)
    seq = [("first", sd.cam16, sd.fov, fx0, a0, w0, h0),
           ("origin", moved, sd.fov, fx0, a0, w0, h0),
           ("3x3", turned, sd.fov, fx0, a0, w0, h0),
           ("fov_xs", turned, fov1, fx1, a0, w0, h0),
           ("aspect", turned, None, fx1, a1, w0, h0),
           ("width", turned, None, fx1, a1, 4 * w0, h0),
           ("height", turned, None, fx1, a1, 4 * w0, h0 + 24)]
    frames = {}
    for cull in ("1", "0"):
        ct = context(monkeypatch, cull)
        try:
            ct.upload_scene(sd.vtx, sd.tri, 64)
            prev = None
            for label, cam, fov, fx, a, w, h in seq:
                img = ct.trace_tiles(ct.make_frame(w, h, spp, cam, fx, a, keep_hits=True)).copy()
                frames[(cull, label)] = (img,) + tuple(ct.download_hits(w, h, spp))
                if cull == "1":
                    boxes, small = check_boxes(ct, ps, cam, fx, a, w, label)
                    if prev is not None:
                        same = np.array_equal(boxes.view(np.uint32), prev[0].view(np.uint32))
                        # the boxes do not depend on the frame size; the width sets the pixel size of the small count
                        assert same == (label in ("width", "height")), label
                        if label in ("width", "height"):
                            assert (small != prev[1]) == (label == "width"), (label, small, prev[1])
                    prev = boxes, small
        finally:
            ct.close()
    for label, cam, fov, fx, a, w, h in seq:
        for k, (x, y) in enumerate(zip(frames[("1", label)], frames[("0", label)])):
            assert np.array_equal(np.asarray(x).view(np.uint32), np.asarray(y).view(np.uint32)), (label, k)
        if fov is not None:
            o = ps.render(cam, fov, w, h, spp, want_hits=True, want_tuv=True)
            for k, (x, y) in enumerate(zip(frames[("1", label)], (o["bgra"], o["tri"], o["t"], o["u"], o["v"]))):
                assert np.array_equal(np.asarray(x).view(np.uint32), np.asarray(y).view(np.uint32)), (label, k)


@pytest.mark.gpu
@pytest.mark.parametrize("cull", [None, "1"])
def test_boxes_rebuilt_for_a_new_scene(port, scene_data, monkeypatch, cull):
    """the same grid and camera, perturbed vertices: the pair count and structure stay, so only a rebuild on upload
    keeps the boxes (and, with the cull on, the frame) right"""
    sd = scene_data("killeroo")
    grid = port.scene(sd.vtx, sd.tri, 64).grid()
    vtx2 = sd.vtx.copy()
    rng = np.random.default_rng(3)
    vtx2[:, :3] += (rng.normal(size=(len(vtx2), 3)) * 2e-3).astype(np.float32)
    w, h, spp = 96, 64, 2
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    ct = context(monkeypatch, cull)
    try:
        before = None
        for vtx in (sd.vtx, vtx2):
            ps = port.scene(vtx, sd.tri, grid=grid)
            ct.upload_scene_with_grid(vtx, sd.tri, grid)
            img = ct.trace_tiles(ct.make_frame(w, h, spp, sd.cam16, fov_xs, aspect, keep_hits=True)).copy()
            got = (img,) + tuple(ct.download_hits(w, h, spp))
            boxes = check_boxes(ct, ps, sd.cam16, fov_xs, aspect, w, "after upload")[0]
            if before is not None:
                assert not np.array_equal(boxes.view(np.uint32), before.view(np.uint32))
            before = boxes
            o = ps.render(sd.cam16, sd.fov, w, h, spp, want_hits=True, want_tuv=True)
            for k, (x, y) in enumerate(zip(got, (o["bgra"], o["tri"], o["t"], o["u"], o["v"]))):
                assert np.array_equal(np.asarray(x).view(np.uint32), np.asarray(y).view(np.uint32)), k
    finally:
        ct.close()
