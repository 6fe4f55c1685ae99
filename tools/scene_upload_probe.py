#!/usr/bin/env python
"""What a scene upload costs from host arrays (cuda_trace_upload_scene) and from CUDA tensors already resident on the
GPU (cuda_trace_upload_scene_device), on three meshes:

  killeroo            res 64
  tiger_soup_medium   cuda_trace_suggest_grid_res(T)
  tiger_soup (C5)     res 768, distance-map mode

Both paths are timed as wall clock around the call, which returns after a device synchronisation; the host path gets
pageable numpy arrays.  The two paths alternate in one context, after one warm-up call each; median, min and max
over the repetitions.  The grids of the two paths are compared at the end (whole grid and distance map, or for C5
the grid description).

Then the dynamic-scene loop on killeroo: per step, deform the positions with torch ops, upload through the device
path and run a 20 000-ray closest-hit query; wall clock per step, synchronised at its end.

    python tools/scene_upload_probe.py [out.txt]        (default profiles/r07_scene_upload.txt)
"""
import importlib
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pkg = lambda s: importlib.import_module("cpp-11-ray-trace-march-framework_b200." + s)
capi, hostapi, scenes = pkg("capi"), pkg("hostapi"), pkg("scenes")
OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r07_scene_upload.txt")
lines = []


def log(s=""):
    print(s, flush=True)
    lines.append(s)


def wall_ms(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def stats(ms):
    return "median %9.2f ms  (min %9.2f, max %9.2f, n=%d)" % (float(np.median(ms)), min(ms), max(ms), len(ms))


def same_grid(a, b, whole):
    ga, gb = a.download_grid(), b.download_grid()
    keys = ("dim", "aabb_min", "aabb_max", "cell_wdh", "inv_cell_wdh") + (("cell_offset", "tri_index") if whole else ())
    ok = all(np.asarray(ga[k]).tobytes() == np.asarray(gb[k]).tobytes() for k in keys)
    ok = ok and len(ga["tri_index"]) == len(gb["tri_index"])
    if whole:
        da, db = a.download_distance_map(), b.download_distance_map()
        ok = ok and (da is None) == (db is None) and (da is None or da.tobytes() == db.tobytes())
    return ok


def upload_case(host, name, res, reps):
    m, _, _ = scenes.build(host, name)
    vtx, tri = m.arrays()
    res = res or capi.load_library().cuda_trace_suggest_grid_res(len(tri))
    v = torch.from_numpy(vtx).cuda()
    t = torch.from_numpy(tri.view(np.int32)).cuda()
    torch.cuda.synchronize()
    mb = (vtx.nbytes + tri.nbytes) / 2 ** 20
    ct = capi.CudaTrace(1)
    ct.upload_scene(vtx, tri, res)            # warm-up
    ct.upload_scene_device(v, t, res)
    host_ms, dev_ms = [], []
    for _ in range(reps):
        host_ms.append(wall_ms(lambda: ct.upload_scene(vtx, tri, res)))
        dev_ms.append(wall_ms(lambda: ct.upload_scene_device(v, t, res)))
    ref = capi.CudaTrace(1)
    ref.upload_scene(vtx, tri, res)
    equal = same_grid(ref, ct, whole=len(tri) < 10_000_000)
    refs = int(ct.download_grid()["tri_index"].shape[0]) if len(tri) < 10_000_000 else None
    ref.close()
    ct.close()
    log("%s, res %d: %d vertices, %d triangles (%.1f MB of records)%s; grids equal: %s" % (
        name, res, len(vtx), len(tri), mb, "" if refs is None else ", %d cell references" % refs, equal))
    log("  host path   (pageable numpy)  %s" % stats(host_ms))
    log("  device path (CUDA tensors)    %s" % stats(dev_ms))
    log("  median difference host - device: %.2f ms" % (float(np.median(host_ms)) - float(np.median(dev_ms))))
    log()


def dynamic_loop(host, steps=20):
    m, _, _ = scenes.build(host, "killeroo")
    vtx, tri = m.arrays()
    base = torch.from_numpy(vtx).cuda()
    t = torch.from_numpy(tri.view(np.int32)).cuda()
    ct = capi.CudaTrace(1)
    ct.upload_scene_device(base, t, 64)
    g = ct.download_grid()
    lo, hi = torch.tensor(g["aabb_min"], device="cuda"), torch.tensor(g["aabb_max"], device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(3)
    o = ((lo + hi) / 2 + (torch.rand(20000, 3, device="cuda", generator=gen) * 2 - 1) * 2 * (hi - lo)).contiguous()
    d = lo + torch.rand(20000, 3, device="cuda", generator=gen) * (hi - lo) - o
    d = (d / d.norm(dim=1, keepdim=True)).contiguous()
    torch.cuda.synchronize()
    ms = []
    for step in range(steps + 2):
        t0 = time.perf_counter()
        v = base.clone()
        p = v[:, :3]
        p += 0.05 * torch.sin(3.0 * p[:, [1, 2, 0]] + 0.4 * step)
        ct.upload_scene_device(v, t, 64)
        ct.query_rays(o, d)
        torch.cuda.synchronize()
        if step >= 2:  # the first two steps warm up the allocator and the query kernel
            ms.append((time.perf_counter() - t0) * 1e3)
    ct.close()
    log("killeroo dynamic scene, res 64: deform (torch) + device upload + 20 000-ray query per step")
    log("  per step %s" % stats(ms))
    log()


def main():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    log("scene upload probe: %s" % time.strftime("%Y-%m-%d %H:%M:%S"))
    log("GPU (name, power limit, max SM clock): %s" % (smi[0] if smi else "unknown"))
    log("wall clock around each call (it returns after a device synchronisation); host and device path alternate in "
        "one context after one warm-up call each")
    log()
    host = hostapi.host_api()
    upload_case(host, "killeroo", 64, 20)
    upload_case(host, "tiger_soup_medium", 0, 10)
    upload_case(host, "tiger_soup", 768, 5)
    dynamic_loop(host)
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
