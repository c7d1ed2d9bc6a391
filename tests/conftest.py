import ctypes
import glob
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def golden_ct_cases():
    names = (os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, "ct_*.npz")))
    return sorted(n for n in names if "." not in n)   # <name>.<array>.npz is a part of <name> (load_golden)


def load_golden(name):
    """The arrays of tests/golden/<name>.npz, and of <name>.<array>.npz beside it where a fixture over 1 MB is split."""
    d = {}
    for path in [os.path.join(GOLDEN, name + ".npz")] + sorted(glob.glob(os.path.join(GOLDEN, glob.escape(name) + ".*.npz"))):
        z = np.load(path)
        d.update({k: z[k] for k in z.files})
    if "params" in d:
        d["params"] = json.loads(str(d["params"]))
    return d


# forward: rel 1e-5 (+ atol 1e-6), gradients: rel 1e-4 (+ 1e-4 * mean|g|)   — BASELINE.json north_star
def fwd_ok(out, ref):
    err = np.abs(out.astype(np.float64) - ref.astype(np.float64))
    tol = 1e-5 * np.abs(ref) + 1e-6
    return float((err / tol).max()), bool((err <= tol).all())


def grad_ok(g, ref):
    err = np.abs(g.astype(np.float64) - ref.astype(np.float64))
    tol = 1e-4 * np.abs(ref) + 1e-4 * np.abs(ref).mean() + 1e-12
    return float((err / tol).max()), bool((err <= tol).all())


def s2m_ok(got, ref32, ref64):
    """
    Parity of the specular->metallic conversion with an sRGB albedo (diffuse.py:129-147).  It divides by
    (decode(albedo) - 0.04 + 2e-6), which amplifies ONE ulp of the decode by up to 2e-3 relative near 0.04, so no
    implementation whose pow differs from ATen's by an ulp anywhere can be inside rel 1e-5 on every texel.  The statement
    is SURVEY.md 8c's: inside rel 1e-5 of the reference, or not further from the reference's own fp64 evaluation than
    twice the reference is.  Returns (fraction inside plain rel 1e-5, all texels pass).
    """
    got, ref32, ref64 = (np.asarray(x, np.float64) for x in (got, ref32, ref64))
    plain = np.abs(got - ref32) <= 1e-5 * np.abs(ref32) + 1e-6
    arb = np.abs(got - ref64) <= 2 * np.abs(ref32 - ref64) + 1e-6
    return float(plain.mean()), bool((plain | arb).all())


@pytest.fixture(scope="session")
def hostsim():
    """The device math headers compiled for the host (tests/hostsim/hostsim.cpp)."""
    import __graft_entry__ as g

    path = g.build_hostsim()
    lib = ctypes.CDLL(path)
    lib.hs_div_check.restype = ctypes.c_int64
    return lib


def case_inputs(z):
    """Golden case -> (maps dict of np arrays, view, lights(L,3), intensity(L,3), params, flags)."""
    p = z["params"]
    maps = {k[3:]: np.ascontiguousarray(z[k]) for k in z if k.startswith("in_")}
    lights = np.ascontiguousarray(z["lights"].reshape(-1, 3))
    L = lights.shape[0]
    inten = np.ascontiguousarray(np.broadcast_to(z["intensity"].reshape(-1, 3), (L, 3)).astype(np.float32))
    multi = z["lights"].ndim == 2
    per_light = bool(multi and not p["accumulate"])
    return maps, np.ascontiguousarray(z["view"]), lights, inten, p, multi, per_light
