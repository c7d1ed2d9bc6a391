"""
pypbr_b200.io: folder loading / saving with the reference's naming conventions and workflow selection (pypbr/io.py:22-230).
Host maps against a regression snapshot in tests/golden (recorded from this package's loader where it had been checked
equal to the reference's); CUDA loading (8-bit bytes uploaded, converted by pbr_ingest_image) bit-equal to host loading.
"""
import json
import os
import warnings

import numpy as np
import pytest
import torch
from conftest import load_golden
from PIL import Image

from pypbr_b200.io import load_material_from_folder, save_material_to_folder, select_material_class
from pypbr_b200.materials import BasecolorMetallicMaterial, DiffuseSpecularMaterial

DEV = torch.device("cuda:0") if torch.cuda.is_available() else None


def _write_folder(path, H=24, W=40, seed=0, with_specular=True, with_metallic=True, albedo_stem="basecolor"):
    rng = np.random.default_rng(seed)
    rgb = lambda: Image.fromarray(rng.integers(0, 256, (H, W, 3), dtype=np.uint8), "RGB")
    grey = lambda: Image.fromarray(rng.integers(0, 256, (H, W), dtype=np.uint8), "L")
    rgb().save(os.path.join(path, f"{albedo_stem}.png"))
    rgb().save(os.path.join(path, "diffuse.png"))
    rgb().save(os.path.join(path, "normalmap.png"))          # second accepted stem of "normal"
    grey().save(os.path.join(path, "roughness.bmp"))
    Image.fromarray(rng.integers(0, 65536, (H, W), dtype=np.uint16)).save(os.path.join(path, "displacement.png"))   # 16-bit height
    if with_metallic:
        grey().save(os.path.join(path, "metalness.png"))
    if with_specular:
        rgb().save(os.path.join(path, "specular.png"))
    return path


def _quiet(fn, *a, **k):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return fn(*a, **k)


def test_workflow_selection_and_warnings(tmp_path):
    folder = _write_folder(str(tmp_path))
    with pytest.warns(UserWarning, match="Defaulting to metallic workflow"):
        m = load_material_from_folder(folder)
    assert isinstance(m, BasecolorMetallicMaterial) and "specular" not in m._maps and m.metallic.shape == (1, 24, 40)
    with pytest.warns(UserWarning, match="Using specular workflow as preferred"):
        s = load_material_from_folder(folder, preferred_workflow="specular")
    assert isinstance(s, DiffuseSpecularMaterial) and "metallic" not in s._maps and s.specular.shape == (3, 24, 40)
    assert not torch.equal(s.albedo, m.albedo)       # diffuse.png vs basecolor.png
    assert m.height.shape == (1, 24, 40) and float(m.height.max()) <= 1.0 and m.height.dtype == torch.float32
    n = m.normal
    assert torch.allclose(n.norm(dim=0), torch.ones(24, 40), atol=1e-5)       # [0,1]-encoded RGB -> unit vectors
    lin = load_material_from_folder(folder, preferred_workflow="metallic", is_srgb=False)
    assert lin.albedo_is_srgb is False and lin.specular_is_srgb is False
    # select_material_class on its own: removes the map of the workflow that lost
    maps = {"metallic": 1, "specular": 2, "basecolor": 3}
    assert _quiet(select_material_class, maps, "specular") is DiffuseSpecularMaterial and "metallic" not in maps
    assert select_material_class({"diffuse": 1}) is DiffuseSpecularMaterial
    with pytest.warns(UserWarning, match="no albedo map found"):
        assert select_material_class({}) is BasecolorMetallicMaterial


def test_missing_albedo_custom_names_and_values(tmp_path):
    folder = _write_folder(str(tmp_path), with_specular=False, albedo_stem="colour")
    with pytest.warns(UserWarning, match="Basecolor map not found"):
        m = load_material_from_folder(folder)
    assert m._maps.get("albedo") is None and isinstance(m, BasecolorMetallicMaterial)
    named = load_material_from_folder(folder, map_names={"basecolor": ["colour"], "roughness": ["roughness"], "metallic": ["metalness"]})
    assert set(k for k, v in named._maps.items() if v is not None) == {"albedo", "roughness", "metallic"}
    raw = np.asarray(Image.open(os.path.join(folder, "colour.png")).convert("RGB"))
    assert torch.equal(named.albedo, torch.from_numpy(raw).permute(2, 0, 1).float().div(255))      # TF.to_tensor
    r = np.asarray(Image.open(os.path.join(folder, "roughness.bmp")).convert("L"))
    assert torch.equal(named.roughness, torch.from_numpy(r).unsqueeze(0).float().div(255))


def test_save_and_reload_round_trip(tmp_path):
    (tmp_path / "in").mkdir()
    src = _quiet(load_material_from_folder, _write_folder(str(tmp_path / "in")), preferred_workflow="metallic")
    out = str(tmp_path / "out")
    save_material_to_folder(src, out, map_names={"albedo": "basecolor"}, format="png")
    assert sorted(os.listdir(out)) == ["basecolor.png", "height.png", "metallic.png", "normal.png", "roughness.png"]
    back = _quiet(load_material_from_folder, out)
    assert torch.equal(back.albedo, src.albedo) and torch.equal(back.roughness, src.roughness) and torch.equal(back.metallic, src.metallic)
    assert torch.allclose(back.normal, src.normal, atol=3.0 / 255)       # [-1,1] re-quantised to 8 bits (step 2/255) and renormalised
    src.save_to_folder(str(tmp_path / "out2"))                           # the method form (base.py:869-878)
    assert "albedo.png" in os.listdir(str(tmp_path / "out2"))


REFERENCE_FOLDER_SEED = 3
REFERENCE_WORKFLOWS = {"metallic": "metallic", "specular": "specular", "auto": None}   # fixture tag -> preferred_workflow


def test_same_maps_as_the_reference(tmp_path):
    """Against a regression snapshot of the maps loaded from _write_folder(seed=REFERENCE_FOLDER_SEED),
    tests/golden/io_folder_24x40.npz: recorded from this package's loader at a commit where it had been checked equal to
    the reference's loader (tests/golden/make_host_golden.py).  Not an independent comparison with the reference: a
    snapshot re-recorded from this package carries no reference parity of its own."""
    z = load_golden("io_folder_24x40")
    meta = json.loads(str(z["meta"]))
    folder = _write_folder(str(tmp_path), seed=REFERENCE_FOLDER_SEED)
    for tag, pref in REFERENCE_WORKFLOWS.items():
        ours = _quiet(load_material_from_folder, folder, preferred_workflow=pref)
        theirs = meta[tag]
        assert type(ours).__name__ == theirs["class"]
        assert set(ours._maps) == set(theirs["maps"])
        for k, present in theirs["maps"].items():
            t = torch.from_numpy(z[f"{tag}_{k}"]) if present else None
            assert (t is None) == (ours._maps[k] is None) and (t is None or torch.equal(ours._maps[k], t)), (pref, k)
        assert ours.albedo_is_srgb == theirs["albedo_is_srgb"]


@pytest.mark.gpu
def test_loading_onto_the_device_equals_host_loading(tmp_path):
    """device=cuda uploads the decoder's bytes and converts on the device (pbr_ingest_image): same bits as the host path."""
    folder = _write_folder(str(tmp_path), H=37, W=52, seed=5)
    for pref in ("metallic", "specular"):
        host = _quiet(load_material_from_folder, folder, preferred_workflow=pref)
        dev = _quiet(load_material_from_folder, folder, preferred_workflow=pref, device=DEV)
        assert type(dev) is type(host) and set(dev._maps) == set(host._maps)
        for k, t in host._maps.items():
            assert dev._maps[k].is_cuda and dev._maps[k].dtype == torch.float32
            assert torch.equal(dev._maps[k].cpu(), t), (pref, k)
    out = str(tmp_path / "saved")
    dev.save_to_folder(out)
    assert "specular.png" in os.listdir(out)
