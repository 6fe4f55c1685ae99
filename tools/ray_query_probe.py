#!/usr/bin/env python
"""Ray queries on GPU-resident rays (cuda_trace_query_rays) against the ray-batch entry point cuda_trace_intersect_rays
(host arrays in and out), on three workloads:

  W1  coherent    killeroo, res 64, the primary rays of a 3840 x 2160 frame at 1 spp (8.3 M rays): closest hit
  W2  shadow      killeroo, rays from a point light to every W1 hit point, t_max = 0.999 x the distance: occlusion
                  and bounded closest hit
  W3  incoherent  the C5 soup (50.1 M triangles) at 768^3 (distance-map mode), 8 M rays from outside the box through
                  random points in it: closest hit
  S   small       W1's first 1 / 32 / 1024 rays: the new query + synchronise against the old entry's wall time

New kernel: CUDA events around each launch, median of warmed repetitions.  Old entry: the duration of the kernel it
launches, from torch.profiler, and its wall time.  profiles/r03_ray_query.txt was taken while that entry still ran
the one-thread-per-ray intersect_rays_kernel; on those numbers its plain mode now runs the query kernel (the
mailboxing mode keeps the old kernel), so a rerun compares the query kernel with itself plus the host staging.
The L2 is not flushed between repetitions: W1 / W2's scene stays resident in the 126 MB L2, W3's does not fit.
Results of the two paths are compared bit for bit.

    python tools/ray_query_probe.py [out.txt]        (default profiles/r03_ray_query.txt)
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
OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r03_ray_query.txt")
REPS = 10
lines = []


def log(s=""):
    print(s, flush=True)
    lines.append(s)


def primary_rays(cam16, fov_xs, aspect, w, h):
    """camera.h:8-47 perspective rays through the pixel centres (float32 torch arithmetic: rays for timing, not the
    bit-exact GenerateRay)"""
    m = torch.tensor(np.asarray(cam16, np.float32).reshape(4, 4), device="cuda")
    py, px = torch.meshgrid(torch.arange(h, device="cuda", dtype=torch.float32),
                            torch.arange(w, device="cuda", dtype=torch.float32), indexing="ij")
    x = ((px + 0.5) / w * 2 - 1) * float(fov_xs)
    y = ((py + 0.5) / h * 2 - 1) * float(fov_xs) / float(aspect)
    v = torch.stack([x, y, -torch.ones_like(x)], -1).reshape(-1, 3)
    v = v / v.norm(dim=1, keepdim=True)
    d = (v @ m[:3, :3]).contiguous()
    o = m[3, :3].expand_as(d).contiguous()
    return o, d


def time_new(ct, o, d, **kw):
    out = ct.query_rays(o, d, **kw)
    torch.cuda.synchronize()
    ms = []
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = ct.query_rays(o, d, **kw)
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms)), out


def time_old(ct, o, d, reps=3):
    """-> (median kernel ms from torch.profiler, median wall ms of the whole call, result)"""
    on, dn = o.cpu().numpy(), d.cpu().numpy()
    res = ct.intersect_rays(on, dn)  # warm-up
    walls = []
    for _ in range(reps):
        t0 = time.perf_counter()
        res = ct.intersect_rays(on, dn)
        walls.append((time.perf_counter() - t0) * 1e3)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            ct.intersect_rays(on, dn)
    ks = [e.device_time / 1e3 if hasattr(e, "device_time") else e.cuda_time / 1e3
          for e in prof.events() if "intersect_rays_kernel" in e.name or "ray_query_kernel" in e.name]
    return float(np.median(ks)) if ks else float("nan"), float(np.median(walls)), res


def same(new, old):
    return all(np.array_equal(a.cpu().numpy().view(np.uint32), np.asarray(b).view(np.uint32)) for a, b in zip(new, old))


def grays(n, ms):
    return n / ms / 1e6


def report(name, n, new_ms, old_kernel_ms=None, old_wall_ms=None, equal=None):
    s = "%-28s n=%9d  new %9.3f ms %7.3f Grays/s" % (name, n, new_ms, grays(n, new_ms))
    if old_kernel_ms is not None:
        s += "  | old kernel %9.3f ms %7.3f Grays/s, old entry wall %9.3f ms  | new/old kernel speed-up %.2fx" % (
            old_kernel_ms, grays(n, old_kernel_ms), old_wall_ms, old_kernel_ms / new_ms)
    if equal is not None:
        s += "  bit-equal=%s" % equal
    log(s)


def main():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    log("ray query probe: %s" % time.strftime("%Y-%m-%d %H:%M:%S"))
    log("GPU (name, power limit, max SM clock): %s" % smi)
    log("L2: not flushed between repetitions (killeroo's scene arrays stay resident in the 126 MB L2; the C5 soup's "
        "do not fit)")
    log("new: CUDA events, median of %d warmed launches; old: torch.profiler kernel time and wall time of "
        "cuda_trace_intersect_rays (host arrays), median of 3" % REPS)
    log()
    host = hostapi.host_api()
    m, fov, cam = scenes.build(host, "killeroo")
    vtx, tri = m.arrays()
    ct = capi.CudaTrace(1)
    ct.upload_scene(vtx, tri, 64)
    w, h = 3840, 2160
    fov_xs, aspect = host.camera_constants(fov, w, h)
    o, d = primary_rays(cam, fov_xs, aspect, w, h)
    n = o.shape[0]

    # W1
    new_ms, new = time_new(ct, o, d)
    k_ms, wall_ms, old = time_old(ct, o, d)
    report("W1 coherent, closest", n, new_ms, k_ms, wall_ms, same(new, old))

    # W2: light -> W1 hit points
    tri_w1, t_w1 = new[0], new[1]
    hit = tri_w1 >= 0
    p = o[hit] + d[hit] * t_w1[hit, None]
    g = ct.download_grid()
    lo, hi = torch.tensor(g["aabb_min"], device="cuda"), torch.tensor(g["aabb_max"], device="cuda")
    light = (lo + hi) / 2 + torch.tensor([0.3, 1.2, 0.4], device="cuda") * (hi - lo)
    so = light.expand_as(p).contiguous()
    dist = (p - so).norm(dim=1)
    sd = ((p - so) / dist[:, None]).contiguous()
    tm = (dist * 0.999).contiguous()
    ns = so.shape[0]
    occ_ms, occ = time_new(ct, so, sd, t_max=tm, occlusion=True)
    bnd_ms, bnd = time_new(ct, so, sd, t_max=tm)
    k_ms, wall_ms, old = time_old(ct, so, sd)
    # the old kernel answers the unbounded query; the bounded one must agree with it wherever no rule-2 corner is hit
    old_tri = torch.from_numpy(old[0].view(np.int32)).cuda()
    old_t = torch.from_numpy(old[1]).cuda()
    clipped = torch.where((old_tri >= 0) & (old_t < tm), old_tri, torch.full_like(old_tri, -1))
    log("W2 shadow rays: %.1f %% occluded; occlusion == bounded hit: %s; bounded differs from the clipped unbounded hit "
        "on %d rays" % (100.0 * occ.float().mean().item(), bool(torch.equal(occ, bnd[0] >= 0)),
                        int((clipped != bnd[0]).sum().item())))
    report("W2 shadow, occlusion", ns, occ_ms, k_ms, wall_ms)
    report("W2 shadow, bounded closest", ns, bnd_ms, k_ms, wall_ms)

    # S: small batches (query + synchronise on the host against the old entry's wall time)
    for k in (1, 32, 1024):
        oo, dd = o[:k].contiguous(), d[:k].contiguous()
        on, dn = oo.cpu().numpy(), dd.cpu().numpy()
        for _ in range(3):
            ct.query_rays(oo, dd)
            ct.intersect_rays(on, dn)
        torch.cuda.synchronize()
        nw, ow = [], []
        for _ in range(50):
            t0 = time.perf_counter()
            ct.query_rays(oo, dd)
            torch.cuda.synchronize()
            nw.append((time.perf_counter() - t0) * 1e3)
            t0 = time.perf_counter()
            ct.intersect_rays(on, dn)
            ow.append((time.perf_counter() - t0) * 1e3)
        log("S  %4d rays: new query + sync %.3f ms, old entry %.3f ms (median wall of 50)" % (
            k, float(np.median(nw)), float(np.median(ow))))
    ct.close()

    # W3
    t0 = time.time()
    m, fov, cam = scenes.build(host, "tiger_soup")
    vtx, tri = m.arrays()
    ct = capi.CudaTrace(1)
    ct.upload_scene(vtx, tri, 768)
    log("W3 scene: %d triangles, built and uploaded in %.1f s, distance map: %s" % (
        len(tri), time.time() - t0, ct.download_distance_map() is not None))
    g = ct.download_grid()
    lo, hi = torch.tensor(g["aabb_min"], device="cuda"), torch.tensor(g["aabb_max"], device="cuda")
    gen = torch.Generator(device="cuda").manual_seed(5)
    n3 = 8 << 20
    o3 = (lo + hi) / 2 + (torch.rand(n3, 3, device="cuda", generator=gen) * 2 - 1) * 2 * (hi - lo)
    target = lo + torch.rand(n3, 3, device="cuda", generator=gen) * (hi - lo)
    d3 = target - o3
    d3 = (d3 / d3.norm(dim=1, keepdim=True)).contiguous()
    o3 = o3.contiguous()
    new_ms, new = time_new(ct, o3, d3)
    k_ms, wall_ms, old = time_old(ct, o3, d3, reps=1)
    report("W3 incoherent, closest", n3, new_ms, k_ms, wall_ms, same(new, old))
    ct.close()

    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    with open(OUT, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
