"""
tests/golden/make_host_golden.py — records the regression snapshots that two host-path tests compare against:

    transforms_pipeline_24x40.npz   test_transforms.py::test_same_results_as_the_reference_on_a_seeded_pipeline
    io_folder_24x40.npz             test_io.py::test_same_maps_as_the_reference

Both tests used to import the unmodified reference package, which is not part of this repository, and were skipped
wherever it was missing. The fixtures hold what pypbr_b200's host (CPU) path returns on the same seeded cases. That path
calls the torch / torchvision / PIL operations the reference calls, and was checked against the reference's transforms
and loader on exactly these cases when it was written (bit-equal; the rotated normals within 3e-7). From here on the
stored results are what the tests compare against: re-record them only for a deliberate change of behaviour.

    python tests/golden/make_host_golden.py
"""

import json
import os
import random
import sys
import tempfile
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]

import pypbr_b200.transforms as OT  # noqa: E402
import test_io  # noqa: E402
import test_transforms  # noqa: E402
from pypbr_b200.io import load_material_from_folder  # noqa: E402
from pypbr_b200.materials import BasecolorMetallicMaterial  # noqa: E402


def make_transforms_fixture():
    maps = test_transforms._maps(H=24, W=40, seed=5)
    m = BasecolorMetallicMaterial(device=torch.device("cpu"))
    for k, v in maps.items():
        m._maps[k] = v.clone()
    random.seed(test_transforms.SEEDED_PIPELINE_SEED)
    out = test_transforms.seeded_pipeline(OT)(m)
    arrs = {f"in_{k}": v.numpy() for k, v in maps.items()}
    arrs.update({f"out_{k}": out._maps[k].numpy() for k in maps})
    meta = {"maps": list(maps), "size": list(out.size), "normal_convention": out.normal_convention.name}
    arrs["meta"] = np.array(json.dumps(meta))
    np.savez_compressed(os.path.join(HERE, "transforms_pipeline_24x40.npz"), **arrs)
    print(f"transforms_pipeline_24x40: size {out.size}")


def make_io_fixture():
    arrs, meta = {}, {}
    with tempfile.TemporaryDirectory() as folder, warnings.catch_warnings():
        warnings.simplefilter("ignore")
        test_io._write_folder(folder, seed=test_io.REFERENCE_FOLDER_SEED)
        for tag, pref in test_io.REFERENCE_WORKFLOWS.items():
            m = load_material_from_folder(folder, preferred_workflow=pref)
            meta[tag] = {"class": type(m).__name__, "maps": {k: t is not None for k, t in m._maps.items()},
                         "albedo_is_srgb": m.albedo_is_srgb}
            arrs.update({f"{tag}_{k}": t.numpy() for k, t in m._maps.items() if t is not None})
    arrs["meta"] = np.array(json.dumps(meta))
    np.savez_compressed(os.path.join(HERE, "io_folder_24x40.npz"), **arrs)
    print(f"io_folder_24x40: {meta}")


if __name__ == "__main__":
    make_transforms_fixture()
    make_io_fixture()
