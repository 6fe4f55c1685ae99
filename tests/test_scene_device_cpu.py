"""CPU checks of the device-side scene upload (include/cuda_trace.h, cuda_trace_upload_scene_device): the symbol is
exported, its ctypes prototype is the header's declaration, and a NULL context is refused without a device.
tests/test_gpu_scene_device.py compares the device path with the host upload on a B200."""
import ctypes as C
import os
import re

from conftest import ROOT, pkg

NAME = "cuda_trace_upload_scene_device"


def header_params(name):
    text = open(os.path.join(ROOT, "include", "cuda_trace.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)\s*;", text)
    assert m, name + " is not declared in cuda_trace.h"
    return [" ".join(p.split()) for p in m.group(1).split(",")]


def test_symbol_exported_and_prototype_matches_header():
    capi = pkg("capi")
    lib = capi.load_library()
    assert hasattr(lib, NAME)
    # C parameter type (name stripped) -> the ctypes type the binding must use for it
    ctypes_of = {"cuda_trace_ctx *": C.c_void_p, "const float *": C.POINTER(C.c_float), "uint32_t": C.c_uint32,
                 "const uint32_t *": C.POINTER(C.c_uint32), "void *": C.c_void_p}
    c_types = [re.sub(r"\w+$", "", p).strip() for p in header_params(NAME)]  # drop the parameter name
    assert c_types == ["cuda_trace_ctx *", "const float *", "uint32_t", "const uint32_t *", "uint32_t", "uint32_t",
                       "void *"]
    res, args = capi.SYMBOLS[NAME]
    assert res is C.c_int
    assert args == [ctypes_of[t] for t in c_types]
    fn = getattr(lib, NAME)
    assert fn.restype is C.c_int and list(fn.argtypes) == args


def test_upload_scene_device_refuses_null_context_without_a_device():
    lib = pkg("capi").load_library()
    assert lib.cuda_trace_upload_scene_device(None, None, 0, None, 0, 0, None) == 1
    v = (C.c_float * 6)()
    t = (C.c_uint32 * 6)()
    assert lib.cuda_trace_upload_scene_device(None, v, 1, t, 1, 64, None) == 1
