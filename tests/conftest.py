import ctypes
import hashlib
import importlib
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

PKG = "cpp-11-ray-trace-march-framework_b200"


def pkg(sub=None):
    return importlib.import_module(PKG + ("." + sub if sub else ""))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200)")
    config.addinivalue_line("markers", "slow: long-running")


def _have_gpu():
    try:
        lib = pkg("capi").load_library()
        return lib.cuda_trace_device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    # GPU tests are selected with -m gpu; when they are selected there must be a GPU -- they
    # then FAIL (not skip) if the CUDA library cannot be loaded, so a silent fallback is impossible
    pass


@pytest.fixture(scope="session")
def pyoracle():
    from oracle import pyoracle as po
    po.build(ref=True, port=True)
    return po


@pytest.fixture(scope="session")
def port(pyoracle):
    return pyoracle.Port.get()


@pytest.fixture(scope="session")
def ref(pyoracle):
    if not pyoracle.have_ref():
        pytest.skip("oracle/_ref/libref_oracle.so not built (needs /root/reference)")
    return pyoracle.Ref.get()


REF_ANSWERS = os.path.join(ROOT, "tests", "golden", "ref_answers.json")
# set to a file name: the run writes tests/golden/ref_answers.json there, updated with the digest of every answer
# it checked
RECORD_REF_ANSWERS = os.environ.get("RTM_RECORD_REF_ANSWERS")
_recorded = {}


class RefAnswers:
    """Comparisons with the reference.  Where oracle/_ref is built, the reference computes its answer and the result
    must equal it bit for bit.  Elsewhere the result must match the md5 digest stored under the same key in
    tests/golden/ref_answers.json, so the comparison runs on every machine.  The digests stored first were taken
    from this project's results (CUDA build, host library, oracle port) at the commit where the same tests compared
    those results bit for bit with the live reference; the file's "note" says so.  Recording needs the reference,
    except for keys passed with reference_free=True: answers no reference call produces (a test's own stand-in
    input), which only pin this project's result."""

    def __init__(self, ref):
        self.ref = ref
        self.api = ref.api if ref is not None else pkg("hostapi").host_api()
        with open(REF_ANSWERS) as f:
            self.answers = json.load(f)["md5"]

    @staticmethod
    def digest(a):
        a = np.ascontiguousarray(a)
        return hashlib.md5(repr((a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()

    def check(self, key, got, want, reference_free=False):
        """got: this project's result; want(ref) -> the reference's answer to the same query."""
        got = np.ascontiguousarray(got)
        if self.ref is not None and not reference_free:
            w = np.ascontiguousarray(want(self.ref))
            assert w.dtype == got.dtype and w.shape == got.shape and w.tobytes() == got.tobytes(), key
        if RECORD_REF_ANSWERS:
            if self.ref is None and not reference_free:
                pytest.fail("recording %s needs the reference (oracle/_ref)" % key)
            _recorded[key] = self.digest(got)
        elif self.ref is None or reference_free:
            assert key in self.answers, "no recorded answer for " + key
            assert self.digest(got) == self.answers[key], key

    def rays(self, port, name, width, height, spp, y_begin, y_end):
        """Primary rays [rows, W, spp, 3] of a scene preset: the reference's GenerateRay, or the oracle port's
        restatement of it (pinned bit for bit by tests/test_oracle_vs_ref.py) where the reference is not built."""
        m, fov, cam = pkg("scenes").build(self.api, name)
        if self.ref is not None:
            return self.ref.renderer(m, fov, cam).generate_rays(width, height, spp, y_begin, y_end)
        F = ctypes.POINTER(ctypes.c_float)
        smp = port.sample_table(spp)
        fov_xs, aspect = port.camera_constants(fov, width, height)
        cam32 = np.ascontiguousarray(cam, np.float32)
        o = np.zeros((y_end - y_begin, width, spp, 3), np.float32)
        d = np.zeros_like(o)
        for y in range(y_begin, y_end):
            for x in range(width):
                for s in range(spp):
                    port.lib.rto_generate_ray(cam32.ctypes.data_as(F), x, y, width, height, float(smp[s, 0]),
                                              float(smp[s, 1]), float(fov_xs), float(aspect),
                                              o[y - y_begin, x, s].ctypes.data_as(F), d[y - y_begin, x, s].ctypes.data_as(F))
        return o, d


@pytest.fixture(scope="session")
def ref_answers(pyoracle):
    return RefAnswers(pyoracle.Ref.get() if pyoracle.have_ref() else None)


def pytest_sessionfinish(session, exitstatus):
    if RECORD_REF_ANSWERS and _recorded:
        with open(REF_ANSWERS) as f:
            data = json.load(f)
        data["md5"].update(_recorded)
        with open(RECORD_REF_ANSWERS, "w") as f:
            json.dump(data, f, indent=1, sort_keys=True)
            f.write("\n")


class SceneData:
    """Post-transform mesh arrays + camera of one preset, built through a MeshApi backend."""

    def __init__(self, name, vtx, tri, fov, cam16):
        self.name, self.vtx, self.tri, self.fov, self.cam16 = name, vtx, tri, float(fov), cam16


_scene_cache = {}


@pytest.fixture(scope="session")
def scene_data(pyoracle):
    """scene_data(name) -> SceneData.  Built with the reference's own Mesh/Matrix44f when
    oracle/_ref exists, else with the host library (whose parity with the reference is pinned by
    tests/test_host_vs_ref.py in the build container)."""
    scenes = pkg("scenes")

    def get(name):
        if name not in _scene_cache:
            if pyoracle.have_ref():
                api = pyoracle.Ref.get().api
            else:
                api = pkg("hostapi").host_api()
            m, fov, cam = scenes.build(api, name)
            vtx, tri = m.arrays()
            _scene_cache[name] = SceneData(name, vtx, tri, fov, cam)
        return _scene_cache[name]

    return get


@pytest.fixture(scope="session")
def cuda_trace():
    capi = pkg("capi")
    ct = capi.CudaTrace(1)
    yield ct
    ct.close()
