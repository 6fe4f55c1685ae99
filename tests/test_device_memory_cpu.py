"""Device and page-locked memory of the tracer library (libcuda_trace.so) is owned by the array types of
csrc/device_array.cuh, which free it on every path, failures included.  No other source of the library allocates or
frees it by hand; the exceptions are the two C ABI functions that hand a page-locked buffer to the caller and take it
back (cuda_trace_host_alloc / cuda_trace_host_free).  tests/test_gpu_device_memory.py checks on a B200 that nothing
leaks."""
import os
import re

from conftest import pkg

RAW = re.compile(r"\b(cudaMalloc|cudaFree|cudaHostAlloc|cudaFreeHost)\s*\(")
HANDED_TO_CALLER = ("cuda_trace_host_alloc", "cuda_trace_host_free")


def csrc():
    return os.path.join(os.path.dirname(pkg("build").__file__), "csrc")


def without_comments(text):
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return re.sub(r"//[^\n]*", "", text)


def without_function(text, name):
    """text with the definition of the function `name` (signature and braced body) cut out"""
    m = re.search(r"\b" + name + r"\s*\([^)]*\)\s*\{", text)
    assert m, name + " is not defined"
    depth, i = 1, m.end()
    while depth:
        depth += {"{": 1, "}": -1}.get(text[i], 0)
        i += 1
    return text[:m.start()] + text[i:]


def library_sources():
    build = pkg("build")
    names = list(build.CU_SOURCES) + [f for f in os.listdir(csrc()) if f.endswith((".cuh", ".h", ".inc"))]
    assert "api.cu" in names and "grid_build.cu" in names and "device_array.cuh" in names
    return [n for n in names if n != "device_array.cuh"]


def test_only_the_array_types_allocate_and_free():
    found = []
    for name in library_sources():
        text = without_comments(open(os.path.join(csrc(), name)).read())
        if name == "api.cu":
            for fn in HANDED_TO_CALLER:
                text = without_function(text, fn)
        found += ["%s: %s" % (name, line.strip()) for line in text.splitlines() if RAW.search(line)]
    assert not found, "\n".join(found)

