"""bench.py's contract, as far as a box without a GPU can check it: the reference arm runs the reference's own CPU
renderer and prints one JSON line with the agreed keys; the product arm refuses to run without a CUDA device (there
is no CPU fallback to time by accident)."""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT


def _run(*args):
    env = dict(os.environ, RTM_QUIET="1")
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + list(args), capture_output=True, text=True,
                          timeout=600, cwd=ROOT, env=env)


def test_reference_arm_line(pyoracle):
    r = _run("--impl", "reference", "--workload", "C1", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "Mrays/s" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["config"]["workload"] == "C1" and d["config"]["width"] == 512 and d["config"]["spp"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert cb["kind"] == ("reference" if pyoracle.have_ref() else "port")
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a box WITHOUT a GPU")
def test_product_arm_fails_loudly_without_a_gpu():
    r = _run("--workload", "C1", "--steps", "1", "--warmup", "0", "--no-cpu-baseline")
    assert r.returncode != 0
    assert "no CPU fallback" in r.stderr and not [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_dump_outputs_samples_a_large_frame_the_same_way_every_time(tmp_path):
    import bench
    rs = np.random.RandomState(5)
    img = rs.randint(0, 1 << 24, size=(2160, 3840)).astype(np.uint32)
    for sub in ("a", "b"):
        bench.dump_outputs(str(tmp_path / sub), img)
    idx = np.load(tmp_path / "a" / "pixel_index.npy")
    bgra = np.load(tmp_path / "a" / "bgra.npy")
    assert idx.dtype == np.float64 and bgra.dtype == np.float32 and bgra.shape == (bench.DUMP_MAX_PIXELS, 4)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 * 2 ** 20
    assert np.array_equal(idx, np.load(tmp_path / "b" / "pixel_index.npy"))
    assert np.array_equal(bgra, np.load(tmp_path / "b" / "bgra.npy"))
    assert np.all(np.diff(idx) > 0) and idx[0] >= 0 and idx[-1] < img.size
    want = img.reshape(-1)[idx.astype(np.int64)]
    got = bgra.astype(np.uint8).view(np.uint32).reshape(-1)
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_dump_outputs_is_the_frame_of_the_last_timed_step(tmp_path):
    """C1 (512 x 512) is below the sample size: every pixel is written, and the bytes reassemble to the digest of the
    reference's own render of that workload.  --steps sets the number of timed steps."""
    r = _run("--workload", "C1", "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-side-configs",
             "--no-class-route", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 3 and len(d["step_ms"]) == 3
    idx = np.load(tmp_path / "pixel_index.npy")
    bgra = np.load(tmp_path / "bgra.npy")
    assert np.array_equal(idx, np.arange(512 * 512))
    img = bgra.astype(np.uint8).view(np.uint32).reshape(512, 512)
    with open(os.path.join(ROOT, "tests", "golden", "ref_digests.json")) as f:
        gold = json.load(f)["cornell_512x512x1_g64"]
    assert hashlib.md5(img.tobytes()).hexdigest() == gold["image_md5"]
