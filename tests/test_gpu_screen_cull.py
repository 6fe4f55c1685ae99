"""K1's screen cull (csrc/pack.cu screen_boxes_kernel, warp_trace.cuh test_pair_list<CULL>): with the cull forced on, the
per-sample (tri, t, u, v) and the image equal the oracle's bit for bit, for a sequence of cameras that changes each
constant the boxes are keyed on -- moved, rotated about the same origin, another field of view and aspect at the same
origin -- so that a stale box array would show."""
import numpy as np
import pytest

from conftest import pkg
from test_screen_cull_cpu import rotated


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["0", "2"])
@pytest.mark.parametrize("name,spp", [("killeroo", 4), ("room", 4), ("torusknot", 16), ("cornell", 1)])
def test_screen_cull_matches_oracle(port, scene_data, monkeypatch, mode, name, spp):
    capi = pkg("capi")
    sd = scene_data(name)
    ps = port.scene(sd.vtx, sd.tri, 64)
    moved = np.array(sd.cam16, np.float32).copy()
    moved[12:15] += np.array([0.03, -0.02, 0.05], np.float32)
    turned = rotated(moved, (1, 2, 3), 5.0)
    views = [(sd.cam16, sd.fov, 192, 128), (moved, sd.fov, 192, 128), (turned, sd.fov, 192, 128),
             (turned, sd.fov * 0.7, 160, 144)]
    monkeypatch.setenv("RTM_REL_RECORDS", "2")
    monkeypatch.setenv("RTM_OCC_MODE", mode)
    monkeypatch.setenv("RTM_THREADS", "1024" if mode != "0" else "256")
    outs = {}
    for cull in ("1", "0"):
        monkeypatch.setenv("RTM_SCREEN_CULL", cull)
        ct = capi.CudaTrace(1)
        ct.upload_scene(sd.vtx, sd.tri, 64)
        for k, (cam, fov, w, h) in enumerate(views):
            fov_xs, aspect = port.camera_constants(fov, w, h)
            f = ct.make_frame(w, h, spp, cam, fov_xs, aspect, keep_hits=True)
            img = ct.trace_tiles(f).copy()
            outs[(cull, k)] = (img,) + tuple(ct.download_hits(w, h, spp))
            plain = ct.trace_tiles(ct.make_frame(w, h, spp, cam, fov_xs, aspect))  # non-instrumented instantiation
            assert np.array_equal(plain, img), (cull, k)
        ct.close()
    for k, (cam, fov, w, h) in enumerate(views):
        o = ps.render(cam, fov, w, h, spp, want_hits=True, want_tuv=True)
        want = (o["bgra"], o["tri"], o["t"], o["u"], o["v"])
        for cull in ("1", "0"):
            for got, ref in zip(outs[(cull, k)], want):
                assert np.array_equal(np.asarray(got).view(np.uint32), np.asarray(ref).view(np.uint32)), (cull, k)
