"""The warp scan of K1's screen cull (csrc/warp_trace.cuh test_pair_list): with the cull forced on, frames equal the
oracle port's bit for bit -- in occupancy modes 0 and 2, in the hit-keeping and the plain instantiation, on the
adversarial scenes and cameras, the presets and the camera sequence of the screen cull's tests.  One more case aims at
the scan and at its fallback: cells of more than 64 pairs holding three copies of every triangle, so that several
32-pair chunks run and equally close hits inside one cell must go to the first copy in list order, traced at 16 samples
(two pixels a warp: the scan) and at 1 sample (eight pixels a warp: lanes on different cells take the pair-by-pair
box check)."""
import os
import sys

import numpy as np
import pytest

import test_gpu_screen_cull as cull_frames
import test_gpu_screen_cull_boxes as cull_boxes
from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tools"))
import screen_cull as sc  # noqa: E402


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "2"])
@pytest.mark.parametrize("group", cull_boxes.GROUPS)
def test_scan_frames_match_oracle(port, scene_data, monkeypatch, mode, group):
    cull_boxes.test_frames_under_cull_match_oracle(port, scene_data, monkeypatch, mode, group)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "2"])
@pytest.mark.parametrize("name,spp", [("killeroo", 4), ("room", 4), ("torusknot", 16), ("cornell", 1)])
def test_scan_camera_views_match_oracle(port, scene_data, monkeypatch, mode, name, spp):
    cull_frames.test_screen_cull_matches_oracle(port, scene_data, monkeypatch, mode, name, spp)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["killeroo", "room"])
def test_scan_camera_sequence(port, scene_data, monkeypatch, name):
    cull_boxes.test_box_cache_keys(port, scene_data, monkeypatch, name)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "2"])
def test_scan_long_lists_and_ties(port, scene_data, monkeypatch, mode):
    """killeroo with every triangle three times (consecutive indices, identical geometry: every hit is a three-way tie
    of equal t, u and v) on a coarse grid; 1 sample (8 x 4 pixels a warp: lanes on different cells, the pair-by-pair box
    check) and 16 (2 pixels: the warp scan)"""
    sd = scene_data("killeroo")
    tri3 = np.ascontiguousarray(np.repeat(sd.tri, 3, axis=0))
    res = 16
    ps = port.scene(sd.vtx, tri3, res)
    pstart, _, _ = sc.pair_records(ps)
    assert np.diff(pstart).max() > 64  # three chunks or more in the longest list
    w, h = 96, 64
    fov_xs, aspect = port.camera_constants(sd.fov, w, h)
    for spp in (1, 16):
        o = ps.render(sd.cam16, sd.fov, w, h, spp, want_hits=True, want_tuv=True)
        want = (o["bgra"], o["tri"], o["t"], o["u"], o["v"])
        hit = np.asarray(o["tri"]) != 0xFFFFFFFF
        assert hit.any() and (np.asarray(o["tri"])[hit] % 3 == 0).all()  # ties go to the first copy
        ct = cull_boxes.context(monkeypatch, "1", mode)
        try:
            ct.upload_scene(sd.vtx, tri3, res)
            img = ct.trace_tiles(ct.make_frame(w, h, spp, sd.cam16, fov_xs, aspect, keep_hits=True)).copy()
            got = (img,) + tuple(ct.download_hits(w, h, spp))
            plain = ct.trace_tiles(ct.make_frame(w, h, spp, sd.cam16, fov_xs, aspect))
        finally:
            ct.close()
        for k, (a, b) in enumerate(zip(got, want)):
            assert np.array_equal(np.asarray(a).view(np.uint32), np.asarray(b).view(np.uint32)), (spp, k)
        assert np.array_equal(plain, img), spp

