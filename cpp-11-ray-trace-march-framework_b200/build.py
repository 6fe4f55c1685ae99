"""Build the native libraries of this package in-tree (nvcc / g++, sm_100a only).

    python cpp-11-ray-trace-march-framework_b200/build.py [--force]

libcuda_trace.so          -- CUDA kernels + the C ABI of include/cuda_trace.h (csrc/*.cu)
libcuda_trace_measure.so  -- measurement / self-check helpers of include/cuda_trace_measure.h (csrc/measure.cu);
                             loaded by bench.py, tools/ and tests/ only
librtm_host.so            -- the C++ host mirror of the reference classes (host/*.cpp)
"""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB_CUDA = os.path.join(PKG, "libcuda_trace.so")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# -fmad=false: the kernels must round like the reference's FMA-free x86-64 build (DESIGN.md)
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
              "-Xcompiler", "-fPIC,-O2,-ffp-contract=off", "-Xptxas", "-v"]
CU_SOURCES = ["api.cu", "trace_kernels.cu", "ray_query.cu", "pool_trace.cu", "pack.cu", "grid_build.cu", "schedule.cu", "qmc.cu"]
LIB_MEASURE = os.path.join(PKG, "libcuda_trace_measure.so")


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_cuda(force=False, verbose=False):
    srcs = [os.path.join(CSRC, s) for s in CU_SOURCES]
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".inc"))]
    deps.append(os.path.join(ROOT, "include", "cuda_trace.h"))
    if not force and not _newer(LIB_CUDA, deps):
        return LIB_CUDA
    objs = []
    for s in srcs:
        o = s[:-3] + ".o"
        if force or _newer(o, deps):
            cmd = [NVCC] + NVCC_FLAGS + ["-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if verbose or r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode:
                raise RuntimeError("nvcc failed: " + " ".join(cmd))
            with open(o + ".ptxas.log", "w") as f:
                f.write(r.stdout + r.stderr)
        objs.append(o)
    cmd = [NVCC, "-shared", "-o", LIB_CUDA] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.check_call(cmd)
    return LIB_CUDA


def build_measure(force=False, verbose=False):
    """libcuda_trace_measure.so: roofline ceilings, L2 flush, arithmetic self-check (csrc/measure.cu)."""
    src = os.path.join(CSRC, "measure.cu")
    deps = [src, os.path.join(CSRC, "rt_device.cuh"), os.path.join(ROOT, "include", "cuda_trace_measure.h")]
    if not force and not _newer(LIB_MEASURE, deps):
        return LIB_MEASURE
    cmd = [NVCC] + NVCC_FLAGS + ["-shared", "-o", LIB_MEASURE, src, "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError("nvcc failed: " + " ".join(cmd))
    return LIB_MEASURE


HOST = os.path.join(PKG, "host")
LIB_HOST = os.path.join(PKG, "librtm_host.so")
CXX = "g++"
# -ffp-contract=off: mesh transforms must round like the reference's (no FMA), see host/lin_alg.h
CXX_FLAGS = ["-std=c++11", "-O2", "-g", "-fPIC", "-pthread", "-Wall", "-Wextra", "-ffp-contract=off"]
HOST_SOURCES = ["mesh.cpp", "grid.cpp", "framebuffer.cpp", "renderer.cpp", "bmp_writer.cpp", "trace.cpp", "capi.cpp"]


def build_host(force=False, verbose=False):
    """librtm_host.so: the C++ mirror of the reference's Mesh/Scene/Grid/Framebuffer/Renderer API
    (host/*.cpp) + flat C wrappers; links against libcuda_trace.so next to it."""
    srcs = [os.path.join(HOST, s) for s in HOST_SOURCES]
    deps = srcs + [os.path.join(HOST, f) for f in os.listdir(HOST) if f.endswith(".h")]
    deps += [os.path.join(ROOT, "include", "cuda_trace.h"), LIB_CUDA]
    if not force and not _newer(LIB_HOST, deps):
        return LIB_HOST
    cmd = [CXX] + CXX_FLAGS + ["-shared", "-o", LIB_HOST] + srcs + [
        "-L" + PKG, "-lcuda_trace", "-Wl,-rpath,$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError("g++ failed: " + " ".join(cmd))
    return LIB_HOST


CLI = os.path.join(PKG, "rtm_render")


def build_cli(force=False, verbose=False):
    """rtm_render: headless command-line renderer on the host API (tools/rtm_render.cpp)."""
    src = os.path.join(ROOT, "tools", "rtm_render.cpp")
    if not force and not _newer(CLI, [src, LIB_HOST]):
        return CLI
    cmd = [CXX] + CXX_FLAGS + ["-o", CLI, src, "-I" + HOST, "-L" + PKG, "-lrtm_host", "-lcuda_trace",
                               "-Wl,-rpath,$ORIGIN"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode:
        sys.stderr.write(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError("g++ failed: " + " ".join(cmd))
    return CLI


def build_all(force=False, verbose=False):
    return [build_cuda(force, verbose), build_measure(force, verbose), build_host(force, verbose), build_cli(force, verbose)]


if __name__ == "__main__":
    print("\n".join(build_all("--force" in sys.argv, "-v" in sys.argv)))
