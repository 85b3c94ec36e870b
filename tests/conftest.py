"""Shared fixtures. `-m "not gpu"`: oracle vs golden vectors, host logic, C-ABI exports (no compute calls).
`-m gpu`: the parity tests proper, all through the C ABI of libcgrt_b200.so."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import __graft_entry__ as ge  # noqa: E402
from oracle import bindings as ob  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
# data/ of a CG-RayTracer checkout (its OBJ/MTL files are not part of this repository); the loader tests skip without it
REFERENCE_DATA = os.environ.get("CGRT_REFERENCE_DATA", "")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session", autouse=True)
def _built():
    ge.build()


@pytest.fixture(scope="session")
def capi():
    return ge.load_package().capi


@pytest.fixture(scope="session")
def oracle():
    return ob.OracleLib()


@pytest.fixture(scope="session")
def reflib():
    """The reference's own TUs compiled verbatim (oracle/_ref, built where the reference's sources are present), else None."""
    try:
        return ob.RefLib()
    except (FileNotFoundError, OSError):
        return None


@pytest.fixture(scope="session")
def gpu(capi):
    if capi.device_count() < 1:
        pytest.skip("no CUDA device")
    return 0


SCENES = ["triangle", "cube", "cornell", "monkey", "dodge", "soup70"]


class Golden:
    def __init__(self, name):
        z = np.load(os.path.join(GOLDEN, f"scene_{name}.npz"))
        self.name = name
        self.z = z
        self.flat = ob.FlatScene(z["vcount"], z["tcount"], z["vertices"], z["triangles"], z["materials"], z["spheres"])
        self.lights = z["lights"]
        self.W, self.H = [int(v) for v in z["frame"]]
        self.rays = z["rays"].view(ob.RAY_DTYPE).reshape(-1)
        self.hits = z["hits"].view(ob.HIT_DTYPE).reshape(-1)
        self.counts = z["counts"]


_golden_cache = {}


def load_golden(name):
    if name not in _golden_cache:
        _golden_cache[name] = Golden(name)
    return _golden_cache[name]


@pytest.fixture(scope="session", params=SCENES)
def golden(request):
    return load_golden(request.param)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def same_bits(a, b):
    """bit-exact equality of float arrays, treating every NaN as equal to every NaN"""
    a = np.ascontiguousarray(a, np.float32)
    b = np.ascontiguousarray(b, np.float32)
    if a.shape != b.shape:
        return False
    return bool(np.all((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))))


def hits_equal(h, g, canon=None):
    """closest-hit records equal: id (canonicalised), t, barycentrics, normal — bit for bit"""
    tri = h["tri"]
    if canon is not None:
        tri = np.where(tri >= 0, canon[np.maximum(tri, 0)], tri)
    ok = np.array_equal(tri, g["tri"])
    for f in ("t", "alpha", "beta", "gamma", "n"):
        ok = ok and same_bits(h[f], g[f])
    return ok
