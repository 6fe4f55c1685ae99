"""Golden vectors generated from the unmodified reference (tests/golden/make_golden.py): the oracle port
(CPU test) and the CUDA path (GPU test) must reproduce every digest.  These are the fixtures that
still pin parity on a box where oracle/_ref is absent."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import ROOT, pkg

GOLDEN = os.path.join(ROOT, "tests", "golden")
with open(os.path.join(GOLDEN, "ref_digests.json")) as f:
    DIGESTS = json.load(f)


def md5(a):
    return hashlib.md5(np.ascontiguousarray(a).tobytes()).hexdigest()


def host_scene(name):
    hostapi, scenes = pkg("hostapi"), pkg("scenes")
    m, fov, cam = scenes.build(hostapi.host_api(), name)
    vtx, tri = m.arrays()
    return vtx, tri, fov, cam


SMALL = sorted(k for k, d in DIGESTS.items() if d["width"] * d["height"] * d["spp"] <= 2000000)


@pytest.mark.parametrize("key", SMALL)
def test_port_reproduces_reference_digests(port, key):
    d = DIGESTS[key]
    vtx, tri, fov, cam = host_scene(d["scene"])  # scene through the host mirror, not the reference
    ps = port.scene(vtx, tri, d["grid_res"], tight_ranges=True)
    g = ps.grid()
    assert [int(x) for x in g["dim"]] == d["dim"] and len(g["tri_index"]) == d["refs"]
    assert int(np.float32(g["cell_wdh"]).view(np.uint32)) == d["cell_wdh_bits"]
    assert md5(g["cell_offset"]) == d["cell_offset_md5"] and md5(g["tri_index"]) == d["tri_index_md5"]
    o = ps.render(cam, fov, d["width"], d["height"], d["spp"], want_hits=True, want_tuv=True)
    assert md5(o["bgra"]) == d["image_md5"]
    assert md5(o["tri"]) == d["tri_md5"] and int((o["tri"] != 0xFFFFFFFF).sum()) == d["hits"]
    assert md5(o["t"]) == d["t_md5"] and md5(o["u"]) == d["u_md5"] and md5(o["v"]) == d["v_md5"]


def test_port_reproduces_full_golden_arrays(port):
    z = np.load(os.path.join(GOLDEN, "cornell_48x48x2.npz"))
    vtx, tri, fov, cam = host_scene("cornell")
    o = port.scene(vtx, tri, 64).render(cam, fov, 48, 48, 2, want_hits=True, want_tuv=True)
    assert np.array_equal(o["bgra"], z["image"]) and np.array_equal(o["tri"], z["tri"])
    for k in ("t", "u", "v"):
        assert np.array_equal(o[k].view(np.uint32), z[k].view(np.uint32))


@pytest.mark.gpu
@pytest.mark.parametrize("key", sorted(DIGESTS))
def test_cuda_reproduces_reference_digests(cuda_trace, key):
    d = DIGESTS[key]
    hostapi = pkg("hostapi")
    vtx, tri, fov, cam = host_scene(d["scene"])
    cuda_trace.upload_scene(vtx, tri, d["grid_res"])
    g = cuda_trace.download_grid()
    assert [int(x) for x in g["dim"]] == d["dim"] and len(g["tri_index"]) == d["refs"]
    assert md5(g["cell_offset"]) == d["cell_offset_md5"] and md5(g["tri_index"]) == d["tri_index_md5"]
    w, h, spp = d["width"], d["height"], d["spp"]
    fov_xs, aspect = hostapi.host_api().camera_constants(fov, w, h)
    f = cuda_trace.make_frame(w, h, spp, cam, fov_xs, aspect, keep_hits=True)
    img = cuda_trace.trace_tiles(f)
    hit, t, u, v = cuda_trace.download_hits(w, h, spp)
    assert md5(hit) == d["tri_md5"] and int((hit != 0xFFFFFFFF).sum()) == d["hits"]
    assert md5(t) == d["t_md5"] and md5(u) == d["u_md5"] and md5(v) == d["v_md5"]
    assert md5(img) == d["image_md5"]


FULL_SIZE = ["cornell_512x512x1_g64", "killeroo_1920x1080x4_g64", "torusknot_1920x1080x16_g64", "room_3840x2160x16_g64",
             "killeroo_3840x2160x16_g64", "tiger_soup_medium_1920x1080x4_g160"]


@pytest.mark.gpu
@pytest.mark.parametrize("key", FULL_SIZE)
def test_default_instantiation_reproduces_full_size_reference_frames(key):
    """The BASELINE configs at FULL size through the kernel instantiation bench.py times -- no per-sample records,
    no environment overrides, the launcher's own choice of records / occupancy map / CTA size -- both ways a caller
    gets the frame: cuda_trace_tiles() into a page-locked host buffer (overlapped band read-back) and
    cuda_trace_tiles_async() + cuda_trace_read_framebuffer().  The digest is the reference's own frame."""
    d = DIGESTS[key]
    capi, hostapi = pkg("capi"), pkg("hostapi")
    for var in ("RTM_REL_RECORDS", "RTM_OCC_MODE", "RTM_THREADS", "RTM_COST_ORDER", "RTM_STRIP_PIXELS", "RTM_FAST_MATH",
                "RTM_OVERLAP_D2H"):
        assert var not in os.environ
    vtx, tri, fov, cam = host_scene(d["scene"])
    w, h, spp = d["width"], d["height"], d["spp"]
    ct = capi.CudaTrace(1)
    try:
        ct.upload_scene(vtx, tri, d["grid_res"])
        fov_xs, aspect = hostapi.host_api().camera_constants(fov, w, h)
        f = ct.make_frame(w, h, spp, cam, fov_xs, aspect)
        pinned = capi.PinnedImage(w, h)
        for _ in range(2):  # the second frame runs in the cost order recorded by the first (sharded / small frames)
            pinned.array[:] = 0
            ct.trace_tiles(f, out=pinned.array)
            assert md5(pinned.array) == d["image_md5"]
        ct.trace_tiles_async(f)
        ct.sync()
        img = np.zeros((h, w), np.uint32)
        ct.read_framebuffer(img)
        assert md5(img) == d["image_md5"]
        pinned.close()
    finally:
        ct.close()


@pytest.mark.gpu
def test_cuda_reproduces_full_golden_arrays(cuda_trace):
    z = np.load(os.path.join(GOLDEN, "cornell_48x48x2.npz"))
    hostapi = pkg("hostapi")
    vtx, tri, fov, cam = host_scene("cornell")
    cuda_trace.upload_scene(vtx, tri, 64)
    fov_xs, aspect = hostapi.host_api().camera_constants(fov, 48, 48)
    f = cuda_trace.make_frame(48, 48, 2, cam, fov_xs, aspect, keep_hits=True)
    img = cuda_trace.trace_tiles(f)
    hit, t, u, v = cuda_trace.download_hits(48, 48, 2)
    assert np.array_equal(img, z["image"]) and np.array_equal(hit, z["tri"])
    assert np.array_equal(t.view(np.uint32), z["t"].view(np.uint32))
