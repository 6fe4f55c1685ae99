#!/usr/bin/env python
"""bench.py -- Mrays/s and ms/frame of the per-tile tracing hot path on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl ours|reference] [--full]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...      (N > 1: one rank per GPU)

A step is one frame of the workload (default: killeroo + ground plane, 3840x2160, 16 spp, the
north-star target scene; --workload C1..C5 selects the BASELINE.json configs).  At N > 1 the frame
is tile-sharded: every rank holds the replicated scene + grid, renders its interleaved share of the strips and
stores its pixels straight into rank 0's device framebuffer through a CUDA-IPC mapping (NVLink peer stores); no
collective is on the data path.

Prints ONE JSON line (rank 0):
  value     primary rays of the whole frame / device time of the trace kernel (CUDA events on its stream, max over
            ranks per step, L2 flushed before every step)
  e2e       the same through the reference-facing call cuda_trace_tiles() with a HOST framebuffer (tile list H2D +
            framebuffer D2H inside the timed region)
  parity    the frame the end-to-end region left in the host buffer, hashed AFTER the timed regions and compared
            with the digest of the reference's own render of this workload (tests/golden/ref_digests.json);
            a mismatch makes the run exit non-zero
  roofline  algorithmic flops (SURVEY.md 8d) against the measured FP32 ceiling without FMA for the L2-resident
            workloads, measured DRAM traffic against the measured HBM bandwidth for the 50 M-triangle soup
  extra.configs   kernel / end-to-end / parity of the other BASELINE configs (C1-C4; C5 with --full), short runs
`--impl reference` times the reference's own threaded CPU renderer (oracle/_ref), whole frames through its own
worker pool, on the host cores instead.

`--dump-outputs DIR` writes the frame the last timed step left in the host framebuffer (see dump_outputs), so that
two builds can be compared pixel for pixel on the same workload.
"""
import argparse
import hashlib
import importlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
PKG = "cpp-11-ray-trace-march-framework_b200"

METRIC = "Mrays/s"
TILES_TEXT = "12x9 (reference layout, framebuffer.h:87-88)"


def pkg(sub):
    return importlib.import_module(PKG + "." + sub)


def workload(name):
    scenes = pkg("scenes")
    if name not in scenes.CONFIGS:
        raise SystemExit("unknown workload %r (have: %s)" % (name, ", ".join(scenes.CONFIGS)))
    scene, w, h, spp, res = scenes.CONFIGS[name]
    return dict(name=name, scene=scene, width=w, height=h, spp=spp, grid_res=res)


def config_of(wl, triangles):
    """The `config` object of the JSON line -- the SAME dict in both arms (the workload, nothing about how it is run)."""
    return {"workload": wl["name"], "scene": wl["scene"], "width": wl["width"], "height": wl["height"], "spp": wl["spp"],
            "grid_res": wl["grid_res"], "triangles": int(triangles), "rays_per_frame": wl["width"] * wl["height"] * wl["spp"],
            "tiles": TILES_TEXT}


def golden_digest(wl):
    """Digest record of the reference's own render of this workload (tests/golden/make_golden.py) or None."""
    path = os.path.join(ROOT, "tests", "golden", "ref_digests.json")
    try:
        with open(path) as f:
            d = json.load(f)
    except (OSError, ValueError):
        return None, None
    key = "%s_%dx%dx%d_g%d" % (wl["scene"], wl["width"], wl["height"], wl["spp"], wl["grid_res"])
    return key, d.get(key)


def md5(a):
    return hashlib.md5(np.ascontiguousarray(a).tobytes()).hexdigest()


DUMP_MAX_PIXELS = 1 << 21  # 32 MiB of float32 BGRA + 16 MiB of float64 indices, under 64 MB in all


def dump_outputs(out_dir, image):
    """Write a BGRA frame ([H, W] uint32) as DIR/pixel_index.npy (float64 [n], row-major pixel index y * W + x) and
    DIR/bgra.npy (float32 [n, 4], the channel bytes B, G, R, A).  Frames of more than DUMP_MAX_PIXELS pixels are
    sampled at a fixed, seeded set of pixels, so every run of the same workload writes the same pixels."""
    flat = np.ascontiguousarray(image, np.uint32).reshape(-1)
    if flat.size > DUMP_MAX_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(flat.size, DUMP_MAX_PIXELS, replace=False))
    else:
        idx = np.arange(flat.size)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "bgra.npy"), flat[idx].view(np.uint8).reshape(-1, 4).astype(np.float32))


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p.get("hbm_gbs", 6650.0)), "measured (MEASURED_PEAKS.json)", float(p.get("sm_max_mhz", 1965.0))
    return 6650.0, "fallback (B200_PROFILING.md)", 1965.0


def measured_dram_traffic(name):
    """DRAM bytes (read + write) of one trace_tiles launch from the committed `ncu --set full` capture of this
    workload, with the file it comes from (profiles/dram_traffic.json), or (None, None)."""
    try:
        with open(os.path.join(ROOT, "profiles", "dram_traffic.json")) as f:
            rec = json.load(f).get(name)
        return (float(rec["bytes_per_launch"]), rec["source"]) if rec else (None, None)
    except (OSError, ValueError, KeyError, TypeError):
        return None, None


# ---------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks + throttle reasons, sampled every 200 ms while the timed region runs."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        for line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------- reference (CPU)
def time_reference_cpu(wl, steps, warmup, budget_s):
    """The reference's own CPU renderer (oracle/_ref: unmodified sources + headless driver): WHOLE frames through
    Framebuffer::WorkerThread (framebuffer.cpp:59-92) on hardware_concurrency() threads, `warmup` untimed + `steps`
    timed (BASELINE.md 3.5: >= 1 + >= 5, best and median reported).  If the warm-up frames do not fit a share of
    budget_s their number is cut; the number of timed frames is always `steps`.  The 50 M-triangle soup is the one
    exception (BASELINE.md 3.6): its CPU side is the oracle port on a band of image rows -- the reference's own grid
    build does not finish on it (FLT_MIN-seeded candidate ranges, triangle.h:123: ~10^5 cells per triangle at
    512^3); the port builds the identical grid with tight ranges.  Falls back to the port as well if oracle/_ref could not be built."""
    from oracle import pyoracle as po
    scenes = pkg("scenes")
    w, h, spp = wl["width"], wl["height"], wl["spp"]
    use_port = not po.have_ref() or wl["scene"] == "tiger_soup"
    if not use_port:
        ref = po.Ref.get()
        threads = ref.hardware_threads()
        mesh, fov, cam = scenes.build(ref.api, wl["scene"])
        triangles = mesh.num_triangles
        t0 = time.perf_counter()
        r = ref.renderer(mesh, fov, cam, wl["grid_res"])
        build_s = time.perf_counter() - t0
        # first frame: a warm-up, and the estimate the warm-up count is cut to the budget with
        sec, img = r.render(w, h, spp, want_image=True)
        done_warm = 1
        n_warm = min(warmup, max(1, int(0.15 * budget_s / max(sec, 1e-6)))) if warmup > 0 else 0
        while done_warm < n_warm:
            r.render(w, h, spp, want_image=False)
            done_warm += 1
        times = [sec] if warmup == 0 else []     # without warm-up frames the first one counts
        if warmup == 0:
            done_warm = 0
        while len(times) < steps:
            s2, img = r.render(w, h, spp, want_image=True)
            times.append(s2)
        total = sum(times)
        rays = w * h * spp * len(times)
        return dict(value=rays / total / 1e6, unit=METRIC, cores=threads, kind="reference",
                    sample="whole frames through the reference's own worker pool (Framebuffer::WorkerThread): %d warm-up + %d "
                           "timed" % (done_warm, len(times)),
                    steps_timed=len(times), warmup_done=done_warm, ms_per_step=1e3 * total / len(times),
                    ms_per_frame_best=1e3 * min(times), ms_per_frame_median=1e3 * statistics.median(times),
                    ms_per_frame_est=1e3 * total / len(times), grid_build_s=build_s, triangles=triangles,
                    image_md5=md5(img), rows=None)
    # oracle port on a band of rows
    port = po.Port.get()
    host = pkg("hostapi").host_api()
    mesh, fov, cam = scenes.build(host, wl["scene"])
    vtx, tri = mesh.arrays()
    threads = os.cpu_count() or 1
    ps = port.scene(vtx, tri, wl["grid_res"], n_threads=threads, tight_ranges=True)
    rows = max(8, h // 64) if len(tri) > 1000000 else max(8, h // 16)
    times, rays, band = [], 0, None
    for i in range(warmup + steps):
        y0 = (i * rows) % max(h - rows, 1)
        t0 = time.perf_counter()
        o = ps.render(cam, fov, w, h, spp, y_begin=y0, y_end=y0 + rows, n_threads=threads)
        sec = time.perf_counter() - t0
        if i >= warmup:
            times.append(sec)
            rays += rows * w * spp
            band = (y0, y0 + rows, o["bgra"])
    total = sum(times)
    return dict(value=rays / total / 1e6, unit=METRIC, cores=threads, kind="port",
                sample="%d image rows per step, %d steps (oracle port: %s)" % (
                    rows, steps, "reference grid build unbounded for this scene" if po.have_ref() else "oracle/_ref not built"),
                steps_timed=len(times), warmup_done=warmup, ms_per_step=1e3 * total / len(times),
                ms_per_frame_best=1e3 * min(times) / (rows * w * spp) * (w * h * spp),
                ms_per_frame_median=1e3 * statistics.median(times) / (rows * w * spp) * (w * h * spp),
                ms_per_frame_est=1e3 * total / rays * (w * h * spp), triangles=len(tri), image_md5=None, rows=band)


def run_reference_arm(args, wl, rank):
    if rank != 0:
        return
    base = time_reference_cpu(wl, args.steps, args.warmup, budget_s=170.0)
    key, gold = golden_digest(wl)
    line = {
        "impl": "reference", "metric": METRIC, "value": base["value"], "unit": METRIC, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": base["ms_per_step"],
        "ms_per_frame_est": base["ms_per_frame_est"], "ms_per_frame_best": base["ms_per_frame_best"],
        "ms_per_frame_median": base["ms_per_frame_median"], "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic camera over the reference's own mesh assets (assets/meshes)",
        "config": config_of(wl, base["triangles"]),
        "cpu_baseline": {"value": base["value"], "unit": METRIC, "cores": base["cores"], "kind": base["kind"],
                         "sample": base["sample"]},
        "e2e": {"value": base["value"], "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "extra": {"steps_timed": base["steps_timed"], "warmup_done": base["warmup_done"],
                  "grid_build_s": base.get("grid_build_s")},
    }
    if base["image_md5"] is not None and gold:
        # the reference arm's own frame against the committed digest: the golden fixtures describe THIS build of the reference
        line["parity"] = {"golden": key, "image_md5": base["image_md5"], "image_md5_ok": base["image_md5"] == gold["image_md5"]}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------ GPU (ours)
class GpuWorkload:
    """One workload on this rank's GPU: scene through the product's own host library (Mesh / Matrix44f mirror),
    upload + grid build, frame description, tile list, pinned host framebuffer."""

    def __init__(self, wl, rank, world, local_rank, group):
        capi, hostapi, scenes, multirank = pkg("capi"), pkg("hostapi"), pkg("scenes"), pkg("multirank")
        self.wl, self.rank, self.world, self.group = wl, rank, world, group
        self.w, self.h, self.spp = wl["width"], wl["height"], wl["spp"]
        self.rays = self.w * self.h * self.spp
        host = hostapi.host_api()
        mesh, fov, cam = scenes.build(host, wl["scene"])
        vtx, tri = mesh.arrays()
        self.triangles = int(len(tri))
        self.ct = capi.CudaTrace(devices=[local_rank])
        t0 = time.perf_counter()
        self.ct.upload_scene(vtx, tri, wl["grid_res"])
        self.upload_s = time.perf_counter() - t0
        self.ct.set_shard(rank, world)
        fov_xs, aspect = host.camera_constants(fov, self.w, self.h)
        self.cam, self.fov_xs, self.aspect = cam, fov_xs, aspect
        self.frame = self.ct.make_frame(self.w, self.h, self.spp, cam, fov_xs, aspect)
        self.rects = capi.CudaTrace.make_tiles(capi.full_frame_tiles(self.w, self.h))  # converted once: the layout repeats
        # rank 0 owns the framebuffer; the others map it (CUDA IPC) and store into it over NVLink
        multirank.share_framebuffer(self.ct, group, self.w, self.h)
        self.pinned = capi.PinnedImage(self.w, self.h) if rank == 0 else None  # page-locked: the D2H copy is one DMA
        self.host_fb = self.pinned.array if rank == 0 else None
        self.signals_on = False

    def close(self):
        # rank 0's framebuffer is mapped by the other ranks (CUDA IPC): they unmap it before rank 0 frees it
        if self.rank != 0:
            self.ct.close()
        self.group.barrier()
        if self.rank == 0:
            self.ct.close()
        if self.pinned is not None:
            self.pinned.close()

    def warm(self, n):
        for _ in range(n):
            self.ct.trace_tiles_async(self.frame, self.rects)
            self.ct.sync()
        self.group.barrier()

    def time_kernel(self, steps):
        """K frames, L2 flushed before each, CUDA events around the trace kernel; max over ranks per step."""
        ct, group = self.ct, self.group
        launches0 = ct.kernel_launches()
        group.barrier()
        step_ms = np.zeros(steps, np.float64)
        for i in range(steps):
            ct.flush_l2()
            ct.trace_tiles_async(self.frame, self.rects)
            ct.sync()
            step_ms[i] = ct.last_kernel_ms()
        group.barrier()
        launches = ct.kernel_launches() - launches0
        step_ms = group.allreduce_max(step_ms)      # a frame is done when its slowest rank is
        launches = int(group.allreduce_sum([launches])[0])
        return step_ms, launches

    def time_e2e(self, steps):
        """The reference-facing call with a host framebuffer: returns when the whole frame is in the HOST buffer.
        Row bands are copied out as soon as every rank's strips of that band are finished (no barrier between
        tracing and read-back)."""
        ct, group, rank = self.ct, self.group, self.rank
        if self.world > 1 and not self.signals_on:
            # every rank also counts its finished strips per row band behind rank 0's framebuffer
            ct.set_shard_signals(True)
            self.signals_on = True
            group.barrier()
        e2e_s = 0.0
        kernel_ms = np.zeros(steps, np.float64)
        marks = np.zeros(7, np.float64)
        # one untimed call first: the completion targets of the overlapped read-back are computed once per layout
        if rank == 0:
            ct.trace_tiles(self.frame, self.rects, out=self.host_fb)
        else:
            ct.trace_tiles_async(self.frame, self.rects)
            ct.sync()
        group.barrier()
        for i in range(steps):
            ct.flush_l2()
            ct.sync()
            group.barrier()
            t0 = time.perf_counter()
            if rank == 0:
                ct.trace_tiles(self.frame, self.rects, out=self.host_fb)
            else:
                ct.trace_tiles_async(self.frame, self.rects)
                ct.sync()
            group.barrier()
            e2e_s += time.perf_counter() - t0
            kernel_ms[i] = ct.last_kernel_ms()
            if rank == 0:
                marks += np.array(ct.last_call_timing()) / steps
        e2e_s = float(group.allreduce_max([e2e_s])[0])
        mine = np.zeros(self.world, np.float64)
        mine[rank] = kernel_ms.mean()
        by_rank = group.allreduce_sum(mine)
        kernel_ms = group.allreduce_max(kernel_ms)
        return e2e_s, kernel_ms, by_rank, marks

    def count_work(self):
        """Work counters of one frame (untimed, instrumented kernel), summed over the ranks' shards."""
        ct = self.ct
        ct.set_counting(True)
        ct.trace_tiles_async(self.frame, self.rects)
        ct.sync()
        c = ct.get_counters()
        ct.set_counting(False)
        keys = ("rays", "cells", "tri_tests", "hits")
        tot = self.group.allreduce_sum([float(c[k]) for k in keys])
        return {k: int(v) for k, v in zip(keys, tot)}

    def parity(self, cpu_rows=None):
        """AFTER the timed regions: the frame the end-to-end region left in rank 0's host buffer against the
        reference's digest of this workload; at N = 1 also the per-sample hit triangle indices of one more
        (untimed) frame.  cpu_rows = (y0, y1, bgra) of the oracle port, for workloads without a reference frame."""
        key, gold = golden_digest(self.wl)
        out = {"golden": key if gold else None, "image_md5": None, "image_md5_ok": None, "hits_ok": None}
        if self.rank == 0:
            out["image_md5"] = md5(self.host_fb)
            if gold:
                out["image_md5_ok"] = out["image_md5"] == gold["image_md5"]
            if cpu_rows is not None:
                y0, y1, bgra = cpu_rows
                out["rows_checked"] = [int(y0), int(y1)]
                out["rows_ok"] = bool(np.array_equal(self.host_fb[y0:y1], bgra))
        if gold and self.world == 1:
            f = self.ct.make_frame(self.w, self.h, self.spp, self.cam, self.fov_xs, self.aspect, keep_hits=True)
            self.ct.trace_tiles_async(f, self.rects)
            self.ct.sync()
            tri, _, _, _ = self.ct.download_hits(self.w, self.h, self.spp, want_tuv=False)
            out["hits_ok"] = md5(tri) == gold["tri_md5"] and int((tri != 0xFFFFFFFF).sum()) == gold["hits"]
            del tri
        elif gold:
            out["hits_note"] = "per-sample records stay on the rank that traced them; checked at N = 1 and in tests/"
        return out


def roofline_of(name, counters, pixels, sec, world, local_rank):
    """SURVEY.md section 8(d) (DESIGN.md "Algorithmic work"): per frame
         bytes = 8*C + 40*T + 48*Hh + 4*P      flops = 80*R + 4*C + 40*T + 36*Hh + 4*(R-Hh) + 12*P
    The scenes of C1-C4 / killeroo4k are L2-resident (a few MB of DRAM traffic per launch): those kernels are bound
    by instruction issue / the FP32 pipe, so the fraction is algorithmic flops against the FP32 ceiling WITHOUT FMA
    (the kernels round like the reference's FMA-free build) measured on this box in this run.  The 50 M-triangle
    soup does not fit in L2: there `achieved` is the MEASURED DRAM traffic of a launch (ncu, profiles/dram_traffic.json) over
    the kernel time against the measured HBM bandwidth -- 3 % of it: the frame's working set is L2-sized and the kernel is
    latency / issue bound, which `limiter` says next to the number."""
    capi = pkg("capi")
    R, Cc, T, Hh, P = counters["rays"], counters["cells"], counters["tri_tests"], counters["hits"], pixels
    alg_bytes = 8 * Cc + 40 * T + 48 * Hh + 4 * P
    alg_flops = 80 * R + 4 * Cc + 40 * T + 36 * Hh + 4 * (R - Hh) + 12 * P
    hbm_peak, hbm_kind, sm_max = measured_peaks()
    traffic, traffic_src = measured_dram_traffic(name)
    fp32_nominal = 148 * 128 * sm_max * 1e6 / 1e12  # non-FMA instr-flop/s at max clock
    try:
        fp32_meas, l2_meas = capi.measure_peaks(local_rank)
        fp32_kind = "measured in this run (csrc/measure.cu: FMUL + FADD chains at full occupancy)"
    except Exception as e:  # noqa: BLE001 -- the nominal figure stands in, and says so
        fp32_meas, l2_meas, fp32_kind = fp32_nominal, None, "nominal 148 SM x 128 lanes x max clock (measurement failed: %s)" % e
    hbm = None
    if traffic is not None:
        hbm = {"achieved": traffic / sec / 1e9, "peak": hbm_peak * world, "unit": "GB/s", "frac": traffic / sec / 1e9 / (hbm_peak * world),
               "peak_kind": hbm_kind, "traffic_source": traffic_src}
    fp32 = {"achieved": alg_flops / sec / 1e12, "peak": fp32_meas * world, "unit": "TFLOP/s",
            "frac": alg_flops / sec / 1e12 / (fp32_meas * world), "peak_kind": fp32_kind, "peak_nominal": fp32_nominal * world,
            "algorithmic_flops_per_launch": alg_flops}
    if name == "C5" and hbm is not None:
        r = dict(hbm, bound="hbm", traffic=traffic, fp32_nonfma=fp32,
                 limiter="neither ceiling: the pooled-ray kernel runs at ~72 % issue and ~70 % L1 utilisation with 40 % of the "
                         "stall samples on long-scoreboard waits (distance look-ups, cold triangle records); "
                         "profiles/r02_ncu_summary_C5_pool768.txt")
    else:
        r = dict(fp32, bound="fp32_nonfma", traffic=traffic, traffic_source=traffic_src, hbm=hbm)
    r["algorithmic_bytes_per_launch"] = alg_bytes
    r["algorithmic_bytes_note"] = ("L1/L2 request bytes of the reference's algorithm (SURVEY 8d), served from L1 (hit rate 92 %) "
                                   "for the L2-resident scenes; never divided by the HBM peak")
    if l2_meas:
        r["l2_read_peak_measured_gbs"] = l2_meas
    r["counters"] = counters
    return r


def bench_side_config(name, steps, rank, world, local_rank, group):
    """Short run of another BASELINE config: kernel, end to end, parity."""
    wl = workload(name)
    g = GpuWorkload(wl, rank, world, local_rank, group)
    g.warm(3)
    step_ms, _ = g.time_kernel(steps)
    e2e_s, _, _, _ = g.time_e2e(steps)
    par = g.parity()
    rec = {"scene": wl["scene"], "width": g.w, "height": g.h, "spp": g.spp, "grid_res": wl["grid_res"], "triangles": g.triangles,
           "steps": steps, "kernel_mrays_s": g.rays * steps / (step_ms.sum() * 1e-3) / 1e6, "kernel_ms": float(step_ms.mean()),
           "e2e_mrays_s": g.rays * steps / e2e_s / 1e6, "e2e_ms": 1e3 * e2e_s / steps,
           "scene_upload_and_grid_build_s": g.upload_s, "parity": par}
    g.close()
    return rec


def time_class_route(wl, steps, n_gpus=1):
    """The drop-in route a viewer written against the reference takes (application.cpp:304-517): Mesh -> Scene ->
    Renderer, then per frame StartRendering() ... WaitRendering() with the pixels in the Framebuffer::Tile buffers
    (host/*.h, INTEGRATION.md route A).  Timed inside the C++ classes, from the StartRendering call to the last
    tile handed back; L2 flushed before every frame."""
    capi, hostapi, scenes = pkg("capi"), pkg("hostapi"), pkg("scenes")
    w, h, spp = wl["width"], wl["height"], wl["spp"]
    mesh, fov, cam = scenes.build(hostapi.host_api(), wl["scene"])
    hr = hostapi.HostRenderer(mesh, fov, cam, wl["grid_res"], n_gpus)
    for _ in range(3):
        hr.start(w, h, spp)
        hr.wait()
    total = 0.0
    for _ in range(steps):
        for dev in range(n_gpus):
            capi.flush_l2(dev)
        hr.start(w, h, spp)
        total += hr.wait()
    img = hr.copy_bitmap(w, h)
    kernel_ms = hr.last_kernel_ms()
    hr.close()
    key, gold = golden_digest(wl)
    return {"value": w * h * spp * steps / total / 1e6, "unit": METRIC, "ms_per_step": 1e3 * total / steps, "n_gpus": n_gpus,
            "kernel_ms_last": kernel_ms, "what": "Renderer::StartRendering() -> WaitRendering(), pixels in the Framebuffer::Tile buffers",
            "image_md5_ok": (md5(img) == gold["image_md5"]) if gold else None}


def run_ours(args, wl, rank, world, local_rank, dist):
    multirank = pkg("multirank")
    group = multirank.RankGroup(dist, "cuda" if dist is not None else None)
    g = GpuWorkload(wl, rank, world, local_rank, group)
    warm = max(args.warmup, 3)
    g.warm(warm)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    step_ms, launches = g.time_kernel(args.steps)                     # ---- device-timed region
    e2e_s, e2e_kernel_ms, e2e_kernel_by_rank, e2e_marks = g.time_e2e(args.steps)   # ---- end-to-end region
    t0 = time.perf_counter()
    for _ in range(20):
        group.barrier()
    barrier_ms = float(group.allreduce_max([(time.perf_counter() - t0) / 20 * 1e3])[0])
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, g.host_fb)

    # ---- untimed: work counters, CPU baseline, parity, the other configs
    counters = g.count_work()
    base = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        base = time_reference_cpu(wl, 3, 1, budget_s=30.0)
    par = g.parity(cpu_rows=base["rows"] if base else None)
    class_route = time_class_route(wl, args.steps) if (rank == 0 and world == 1 and not args.no_class_route) else None
    side = {}
    if not args.no_side_configs:
        names = [n for n in ("C1", "C2", "C3", "C4") if n != wl["name"]]
        if args.full and wl["name"] != "C5":
            names.append("C5")
        for n in names:
            side[n] = bench_side_config(n, 5, rank, world, local_rank, group)
    total_ms = float(step_ms.sum())
    roof = roofline_of(wl["name"], counters, g.w * g.h, total_ms * 1e-3 / args.steps, world, local_rank) if rank == 0 else None
    triangles, upload_s, rays = g.triangles, g.upload_s, g.rays
    w, h = g.w, g.h
    g.close()
    if rank != 0:
        return 0

    line = {
        "metric": METRIC, "value": rays * args.steps / (total_ms * 1e-3) / 1e6, "unit": METRIC, "n_gpus": world,
        "steps": args.steps, "warmup": warm, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic camera over the reference's own mesh assets (assets/meshes)",
        "config": config_of(wl, triangles),
        "clocks": clocks,
        "e2e": {"value": rays * args.steps / e2e_s / 1e6, "unit": METRIC, "ms_per_step": 1e3 * e2e_s / args.steps,
                "kernel_ms_per_step": float(e2e_kernel_ms.mean()),
                "kernel_ms_by_rank": [round(float(x), 4) for x in e2e_kernel_by_rank], "barrier_ms": barrier_ms,
                "rank0_call_ms": {"prepared": e2e_marks[4], "launching": e2e_marks[5], "launched": e2e_marks[6],
                                  "submitted": e2e_marks[0], "traced": e2e_marks[1], "copied": e2e_marks[2], "returned": e2e_marks[3]},
                "h2d_bytes_per_step": 108 * 16 + 109 * 4, "d2h_bytes_per_step": w * h * 4},
        "gpu_launches": int(launches),
        "parity": par,
        "roofline": roof,
        "step_ms": [round(float(x), 4) for x in step_ms],
        "extra": {"l2": "flushed before every timed step (256 MiB memset, untimed); the scene itself is L2-resident",
                  "strips": "~128-ray pixel-block strips, chunks of 32 strips dealt round-robin over ranks",
                  "scene_upload_and_grid_build_s": upload_s, "configs": side},
    }
    if class_route:
        line["e2e"]["class_route"] = class_route
    if base:
        line["cpu_baseline"] = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")}
        line["cpu_baseline"].update(ms_per_frame_est=base["ms_per_frame_est"], ms_per_frame_best=base["ms_per_frame_best"])
    print(json.dumps(line), flush=True)
    bad = [n for n, p in [(wl["name"], par)] + [(n, r["parity"]) for n, r in side.items()]
           if p.get("image_md5_ok") is False or p.get("hits_ok") is False or p.get("rows_ok") is False]
    if class_route and class_route["image_md5_ok"] is False:
        bad.append(wl["name"] + " (class route)")
    if bad:
        sys.stderr.write("PARITY FAILURE: %s differ from the reference digests\n" % ", ".join(bad))
        return 3
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="killeroo4k")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-configs", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--no-class-route", action="store_true", help="skip the Renderer / Framebuffer class-route timing")
    ap.add_argument("--full", action="store_true", help="also run C5 (50 M triangles) among the side configs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the frame of the last timed step to DIR as .npy files")
    args = ap.parse_args()
    args.steps = max(args.steps, 1)
    if args.dump_outputs and args.impl != "ours":
        raise SystemExit("--dump-outputs writes the GPU path's frame: use it with --impl ours")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = workload(args.workload)

    if args.impl == "reference":
        run_reference_arm(args, wl, rank)
        return 0

    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    elif args.gpus > 1:
        raise SystemExit("--gpus %d needs torchrun (one rank per GPU); see the module docstring" % args.gpus)
    rc = 1
    try:
        rc = run_ours(args, wl, rank, world, local_rank, dist)
    finally:
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
    return rc


if __name__ == "__main__":
    sys.exit(main())
