"""
The camera at a finite position (view_type="point") on the CPU: the device math headers compiled for the host with the
camera view type (tests/hostsim/camsim.cpp: the cam_* kernels' per-texel-pair arithmetic, V = f2) against the camera
oracle (tests/camera_oracle.py) - the forward at rel 1e-5, every map gradient at rel 1e-4, and the intensity, light and
camera gradients against the fp64 oracle at 1e-4 |g| + 1e-4 mean|g|.  Also the API's refusals, which need no GPU.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch

import camera_oracle as CO
from conftest import ROOT, fwd_ok, grad_ok

CSRC = os.path.join(ROOT, "pypbr_b200", "csrc")
SRC = os.path.join(ROOT, "tests", "hostsim", "camsim.cpp")
WFS = {"metallic": 0, "specular": 1, "metallic3": 2}
SHARED = ("intensity", "lights", "camera")


@pytest.fixture(scope="module")
def camsim(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("camsim") / "libcamsim.so")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-std=c++17", "-shared", "-fPIC", "-I", CSRC, SRC, "-o", out], check=True)
    lib = ctypes.CDLL(out)
    f, i, p = ctypes.c_float, ctypes.c_int, ctypes.c_void_p
    head = [i] * 6 + [f] + [i] * 4 + [p] * 3
    lib.cs_forward.argtypes = head + [p] * 5
    lib.cs_backward.argtypes = head + [p] * 5 + [p] * 4 + [p] * 3
    return lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _case(seed, wf, B, H, W, L, light, normal=True):
    g = torch.Generator().manual_seed(seed)
    maps = {"albedo": torch.rand(B, 3, H, W, generator=g), "roughness": torch.rand(B, 1, H, W, generator=g) * 0.8 + 0.2}
    if normal:
        n = torch.randn(B, 3, H, W, generator=g) * torch.tensor([0.3, 0.3, 0.0]).view(1, 3, 1, 1)
        maps["normal"] = torch.nn.functional.normalize(n + torch.tensor([0.0, 0.0, 1.0]).view(1, 3, 1, 1), dim=1)
    if wf == "specular":
        maps["specular"] = torch.rand(B, 3, H, W, generator=g)
    else:
        maps["metallic"] = torch.rand(B, 3 if wf == "metallic3" else 1, H, W, generator=g)
    ang = torch.arange(L, dtype=torch.float32) * (6.2831853 / L) + 0.3
    lights = torch.stack([0.4 * torch.cos(ang), 0.4 * torch.sin(ang), torch.ones(L)], dim=1)
    if light == "directional":
        lights = torch.nn.functional.normalize(lights + torch.tensor([0.0, 0.0, 1.0]), dim=-1)
    inten = (torch.tensor([1.0, 0.8, 0.6]).expand(L, 3) / L).contiguous()
    return maps, lights, inten, g


def _np(t):
    return np.ascontiguousarray(t.detach().numpy().astype(np.float32))


CASES = []
for _wf in WFS:
    for _light in ("point", "directional"):
        CASES += [
            dict(wf=_wf, light=_light, L=1, per_light=False),
            dict(wf=_wf, light=_light, L=3, per_light=False),
            dict(wf=_wf, light=_light, L=3, per_light=True),
        ]
CASES += [
    dict(wf="metallic", light="point", L=2, per_light=False, normal=False),
    dict(wf="specular", light="directional", L=1, per_light=False, albedo_srgb=False, specular_srgb=False),
    dict(wf="metallic3", light="point", L=2, per_light=True, return_srgb=False),
    dict(wf="metallic", light="point", L=1, per_light=False, camera=(0.6, -0.3, 0.05)),        # grazing, off centre
    dict(wf="specular", light="directional", L=2, per_light=False, camera=(-0.45, 0.2, 0.05)),
    dict(wf="metallic3", light="point", L=3, per_light=False, camera=(0.3, 0.35, 0.05), light_size=2.0),
]


def _id(c):
    return "-".join(str(x) for x in (c["wf"], c["light"], f"L{c['L']}", "per" if c["per_light"] else "acc",
                                     "" if c.get("normal", True) else "nonormal", "" if c.get("albedo_srgb", True) else "linalb",
                                     "" if c.get("return_srgb", True) else "linout", "grazing" if "camera" in c else "") if x != "")


@pytest.mark.parametrize("c", CASES, ids=[_id(c) for c in CASES])
def test_camera_matches_oracle_on_host(camsim, c):
    B, H, W, L = 2, 5, 9, c["L"]   # odd W: the last texel pair is ragged
    maps, lights, inten, g = _case(100 + CASES.index(c), c["wf"], B, H, W, L, c["light"], c.get("normal", True))
    camera = torch.tensor(c.get("camera", (0.1, -0.15, 1.2)))
    size = c.get("light_size")
    flags = dict(albedo_is_srgb=c.get("albedo_srgb", True), specular_is_srgb=c.get("specular_srgb", True),
                 return_srgb=c.get("return_srgb", True))
    acc = not c["per_light"]
    mkey = "specular" if c["wf"] == "specular" else "metallic"

    leaves = {k: v.clone().requires_grad_(True) for k, v in maps.items()}
    ref = CO.render(leaves, camera, lights, inten, size, c["light"], accumulate=acc, **flags)
    go = torch.rand(ref.shape, generator=g)
    ref.backward(go)
    sh = {k: t.double().clone().requires_grad_(True) for k, t in zip(SHARED, (inten, lights, camera))}
    ref64 = CO.render({k: t.double() for k, t in maps.items()}, sh["camera"], sh["lights"], sh["intensity"], size, c["light"],
                      accumulate=acc, **flags)
    ref64.backward(go.double())

    a = {k: _np(v) for k, v in maps.items()}
    head = (B, H, W, L, WFS[c["wf"]], int(c["light"] == "point"), float(size or 0.0), int(flags["albedo_is_srgb"]),
            int(flags["specular_is_srgb"]), int(flags["return_srgb"]), int(c["per_light"]))
    par = [_np(camera), _np(lights), _np(inten)]
    args = head + tuple(_ptr(x) for x in par) + tuple(_ptr(a.get(k)) for k in ("albedo", "normal", "roughness", mkey))
    out = np.zeros(ref.shape, np.float32)
    assert camsim.cs_forward(*args, _ptr(out)) == 0
    ratio, ok = fwd_ok(out, ref.detach().numpy())
    assert ok, f"forward {ratio}"

    grads = {k: np.zeros(v.shape, np.float32) for k, v in a.items()}
    d_int, d_lights, d_cam = np.zeros(3 * L), np.zeros(3 * L), np.zeros(3)
    gout = _np(go)
    assert camsim.cs_backward(*args, _ptr(gout), *(_ptr(grads.get(k)) for k in ("albedo", "normal", "roughness", mkey)),
                              _ptr(d_int), _ptr(d_lights), _ptr(d_cam)) == 0
    for k in maps:
        ratio, ok = grad_ok(grads[k], leaves[k].grad.numpy())
        assert ok, f"d_{k} {ratio}"
    for k, got in zip(SHARED, (d_int, d_lights, d_cam)):
        want = sh[k].grad.numpy().reshape(-1)
        tol = 1e-4 * np.abs(want) + 1e-4 * np.abs(want).mean()
        assert np.all(np.abs(got - want) <= tol), (k, float((np.abs(got - want) / tol).max()), got, want)


def test_far_camera_approaches_the_view_direction():
    """The camera oracle's substitution in the limit: a camera far along v shades like the reference's view direction v."""
    from oracle import pbr_oracle as O

    maps, lights, inten, _ = _case(5, "metallic", 1, 4, 6, 1, "point")
    m = {k: v[0].double() for k, v in maps.items()}
    v = torch.tensor([0.1, -0.2, 1.0], dtype=torch.float64)
    far = CO.render(m, v * 1e7, lights[0].double(), inten[0].double(), 1.0, "point")
    ortho = O.render(m, v, lights[0].double(), inten[0].double(), 1.0, "point")
    assert torch.allclose(far, ortho, rtol=0, atol=1e-6)


def test_view_type_is_validated():
    from pypbr_b200.fit import RenderingLoss
    from pypbr_b200.models import CookTorranceBRDF

    with pytest.raises(ValueError, match="view_type"):
        CookTorranceBRDF(view_type="perspective")
    with pytest.raises(ValueError, match="view_type"):
        RenderingLoss(view_type="orthographic")
    assert CookTorranceBRDF(view_type="Point").view_type == "point"
    assert CookTorranceBRDF().view_type == "directional"


def test_one_launch_fit_step_refuses_a_camera():
    from pypbr_b200.fit import fit_step, fused_fit_step

    z = torch.zeros(3, 4, 4)
    with pytest.raises(ValueError, match=r"fit_step\(fused=False\)"):
        fused_fit_step(None, None, z, torch.tensor([0.0, 0.0, 2.0]), torch.tensor([0.1, 0.1, 1.0]), torch.ones(3),
                       view_type="point")
    with pytest.raises(ValueError, match=r"fit_step\(fused=False\)"):
        fit_step(None, None, z, torch.tensor([0.0, 0.0, 2.0]), torch.tensor([0.1, 0.1, 1.0]), torch.ones(3), fused=True,
                 view_type="point")
