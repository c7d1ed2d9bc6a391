"""
Every compiled camera kernel (view_type="point": pbr::cam_{forward,backward}_kernel<WF, light>) against the camera
oracle (tests/camera_oracle.py), in the style of test_gpu_kernel_coverage.py.

Each row of CASES is one call through the public API - autograd through CookTorranceBRDF(view_type="point"),
fused_loss_step(view_type="point") or fit_step(fused=False, view_type="point") - with the exact set of cam_* kernels it
must launch.  The row compares the results with the oracle (images and map gradients with fwd_ok / grad_ok, at a grazing
camera with the fp64 arbiter of _map_grad_ok; intensity,
light and camera gradients against the fp64 oracle at 1e-4 |g| + 1e-4 mean|g|; the fit step against torch.optim.Adam
plus projection applied to the oracle's gradients) and checks under torch.profiler that exactly those kernels, and no
ct_* kernel, ran.  test_every_camera_kernel_has_a_row is the ledger: the cam_* instantiations defined in libpbrcuda.so
must be exactly the union of the rows' kernels.

Kernel names: cam_forward_kernel<WF, light>, cam_backward_kernel<WF, light> (the entry points of the generic kernels' bodies
with the camera view, kCam); WF 0 metallic (1-channel map), 1 specular, 2 metallic with a 3-channel map; light 0
directional, 1 several point lights (per texel), 2 one point light (hoisted).  test_the_two_ledgers_partition_the_library:
every Cook-Torrance kernel of the library is in exactly one ledger, this file's or test_gpu_kernel_coverage.py's.
"""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

import camera_oracle as CO
from conftest import ROOT, fwd_ok

DEV = torch.device("cuda:0") if torch.cuda.is_available() else None
LIB = os.path.join(ROOT, "pypbr_b200", "lib", "libpbrcuda.so")
DIR, PT, HOIST = 0, 1, 2
WFS = {"metallic": 0, "specular": 1, "metallic3": 2}
MAPS = ("albedo", "normal", "roughness", "metspec")
SHARED = ("intensity", "lights", "view")
CAMERA = (0.12, -0.2, 1.5)
GRAZING = (0.7, -0.35, 0.05)


def fk(wf, light):
    return f"cam_forward_kernel<{wf}, {light}>"


def bk(wf, light):
    return f"cam_backward_kernel<{wf}, {light}>"


_NAME = re.compile(r"(cam_(?:forward|backward)_kernel)\s*<([^<>]*)>")
_CT = re.compile(r"ct_(?:forward|backward)_(?:kernel|stream)\s*<")


def norm_kernel(name):
    m = _NAME.search(name)
    return f"{m.group(1)}<{', '.join(a.strip() for a in m.group(2).split(','))}>" if m else None


def _row(entry, wf, kernels, *, light="point", L=1, B=2, H=4, W=40, per_light=False, albedo_srgb=True, return_srgb=True,
         normal=True, grads=MAPS + SHARED, layout="contig", on_device=False, camera=CAMERA):
    """entry: "autograd" (CookTorranceBRDF forward + backward), "loss" (fused_loss_step; "lights" / "view" in grads request
    want_geometry_grad) or "fit" (fit_step(fused=False): loss kernel, all-reduce, FusedAdam).  layout: "contig",
    "misaligned" (first texel 4-byte aligned, element accesses) or "bcast" (one (1, C, H, W) metallic map for the batch).
    on_device: the camera, lights and intensities are CUDA tensors (PbrCtDesc.params_on_device)."""
    r = dict(entry=entry, wf=wf, kernels=tuple(kernels), light=light, L=L, B=B, H=H, W=W, per_light=per_light,
             albedo_srgb=albedo_srgb, return_srgb=return_srgb, normal=normal, grads=tuple(grads), layout=layout,
             on_device=on_device, camera=camera)
    r["id"] = "-".join(str(x) for x in (entry, wf, light, f"L{L}", f"B{B}", f"{H}x{W}", "per" if per_light else "acc", layout,
                                         "+".join(g[:3] for g in grads), "" if normal else "nonormal",
                                         "" if albedo_srgb else "linalb", "" if return_srgb else "linout",
                                         "dev" if on_device else "", "grazing" if camera == GRAZING else "") if x != "")
    return r


def _cases():
    rows = []
    for wf, c in WFS.items():
        rows += [
            _row("autograd", wf, [fk(c, DIR), bk(c, DIR)], light="directional", L=2),
            _row("autograd", wf, [fk(c, HOIST), bk(c, HOIST)], B=17, H=3, W=20),       # B = 17: two 16-material walks
            _row("autograd", wf, [fk(c, PT), bk(c, PT)], L=3, per_light=True),
            _row("loss", wf, [bk(c, PT)], L=3),                                          # accumulate mode: two passes
            _row("loss", wf, [bk(c, HOIST)], per_light=True, grads=MAPS + ("intensity",)),
            _row("fit", wf, [bk(c, PT)], L=2, per_light=True, grads=MAPS),
        ]
    rows += [
        _row("autograd", "metallic", [fk(0, HOIST), bk(0, HOIST)], B=1),
        _row("autograd", "metallic", [fk(0, PT), bk(0, PT)], L=16, B=1),
        _row("autograd", "specular", [fk(1, PT), bk(1, PT)], L=64, B=1, H=3, W=20),
        _row("autograd", "metallic3", [fk(2, PT), bk(2, PT)], L=3, B=3, layout="bcast"),
        _row("autograd", "specular", [fk(1, HOIST), bk(1, HOIST)], W=41),                  # odd W
        _row("autograd", "metallic", [fk(0, PT), bk(0, PT)], L=2, layout="misaligned"),
        _row("autograd", "metallic", [fk(0, DIR), bk(0, DIR)], light="directional", W=41, layout="misaligned",
             normal=False, albedo_srgb=False, return_srgb=False),
        _row("autograd", "metallic3", [fk(2, PT), bk(2, PT)], L=2, on_device=True),
        _row("autograd", "specular", [fk(1, DIR), bk(1, DIR)], light="directional", on_device=True),
        _row("autograd", "metallic", [fk(0, HOIST), bk(0, HOIST)], camera=GRAZING),
        _row("autograd", "specular", [fk(1, DIR), bk(1, DIR)], light="directional", L=2, camera=GRAZING),
        _row("loss", "metallic", [bk(0, PT)], L=64, B=1, H=3, W=20),
        _row("loss", "metallic3", [bk(2, DIR)], light="directional", L=2, per_light=True, on_device=True),
        _row("loss", "specular", [bk(1, PT)], L=3, camera=GRAZING, grads=("lights", "view")),   # no map gradient at all
        _row("fit", "metallic", [bk(0, HOIST)], B=17, H=3, W=20, grads=MAPS),
        _row("fit", "metallic", [bk(0, DIR)], light="directional", L=2, per_light=True, W=41, grads=MAPS),
    ]
    return rows


CASES = _cases()


# ---------------------------------------------------------------------------------------------- the ledger (CPU)
def test_every_camera_kernel_has_a_row():
    assert os.path.exists(LIB), f"{LIB} is not built"
    out = subprocess.run(["nm", "-C", "--defined-only", LIB], check=True, capture_output=True, text=True).stdout
    compiled = {norm_kernel(m.group(0)) for m in re.finditer(r"pbr::cam_(?:forward|backward)_kernel<[^<>]*>", out)}
    named = {k for r in CASES for k in r["kernels"]}
    assert compiled, "no camera kernel in the library"
    assert not compiled - named, f"instantiations without a parity row: {sorted(compiled - named)}"
    assert not named - compiled, f"rows name kernels the library does not contain: {sorted(named - compiled)}"
    ids = [r["id"] for r in CASES]
    assert len(ids) == len(set(ids))


def test_the_two_ledgers_partition_the_library():
    from test_gpu_kernel_coverage import CASES as ORTHO_CASES, norm_kernel as norm_ct

    out = subprocess.run(["nm", "-C", "--defined-only", LIB], check=True, capture_output=True, text=True).stdout
    compiled = {norm_kernel(m.group(0)) or norm_ct(m.group(0))
                for m in re.finditer(r"pbr::(?:ct|cam)_(?:forward|backward)_(?:kernel|stream)<[^<>]*>", out)}
    cam = {k for r in CASES for k in r["kernels"]}
    ortho = {k for r in ORTHO_CASES for k in r["kernels"]}
    assert not cam & ortho, sorted(cam & ortho)
    assert cam | ortho == compiled, sorted(compiled ^ (cam | ortho))


def test_kernel_names_normalise():
    assert norm_kernel("void pbr::cam_backward_kernel<2, 1>(pbr::CtKParams)") == "cam_backward_kernel<2, 1>"
    assert norm_kernel("pbr::cam_forward_kernel<0,2>") == "cam_forward_kernel<0, 2>"
    assert norm_kernel("void pbr::ct_backward_kernel<0, 3, false, true, 1>(pbr::CtKParams)") is None


# ---------------------------------------------------------------------------------------------- parity rows (GPU)
def _random_case(seed, B, H, W, L, workflow, normal=True):
    g = torch.Generator().manual_seed(seed)
    shp = lambda c: (B, c, H, W)
    maps = {"albedo": torch.rand(shp(3), generator=g), "roughness": torch.rand(shp(1), generator=g) * 0.8 + 0.2}
    if normal:
        n = torch.randn(shp(3), generator=g) * torch.tensor([0.3, 0.3, 0.0]).view(1, 3, 1, 1)
        maps["normal"] = torch.nn.functional.normalize(n + torch.tensor([0.0, 0.0, 1.0]).view(1, 3, 1, 1), dim=1)
    if workflow == "specular":
        maps["specular"] = torch.rand(shp(3), generator=g)
    else:
        maps["metallic"] = torch.rand(shp(3 if workflow == "metallic3" else 1), generator=g)
    ang = torch.arange(L, dtype=torch.float32) * (6.2831853 / L) + 0.2
    lights = torch.stack([0.4 * torch.cos(ang), 0.4 * torch.sin(ang), torch.ones(L)], dim=1) if L > 1 else torch.tensor([0.1, 0.1, 1.0])
    inten = torch.tensor([1.0, 0.8, 0.6]).expand(L, 3) / L if L > 1 else torch.tensor([1.0, 0.8, 0.6])
    return maps, lights, inten.contiguous(), g


def _launched(fn):
    """fn() under torch.profiler -> (its result, the cam_* kernels it launched, whether any ct_* kernel ran)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    return res, {k for k in map(norm_kernel, names) if k}, any(_CT.search(n) for n in names)


def _device_material(r, maps):
    from pypbr_b200.materials import BasecolorMetallicMaterial, DiffuseSpecularMaterial

    cls = DiffuseSpecularMaterial if r["wf"] == "specular" else BasecolorMetallicMaterial
    m = cls(albedo_is_srgb=r["albedo_srgb"], device=DEV)
    if cls is DiffuseSpecularMaterial:
        m.specular_is_srgb = True
    want = {("metspec" if k in ("metallic", "specular") else k) for k in maps} & set(r["grads"]) if r["entry"] == "autograd" else set()
    leaves = {}
    for k, v in maps.items():
        t = v.to(DEV)
        if r["layout"] == "bcast" and k == "metallic":
            t = t[:1].contiguous()
        elif r["layout"] == "misaligned":
            wide = torch.zeros(*t.shape[:-1], r["W"] + 8, device=DEV)
            wide[..., 1:1 + r["W"]] = t
            t = wide[..., 1:1 + r["W"]]
        t = t.detach().requires_grad_(("metspec" if k in ("metallic", "specular") else k) in want)
        leaves[k] = t
        m._maps[k] = t
    if "normal" not in maps:
        m._maps["normal"] = None
    return m, leaves


def _map_grad_ok(got, ref32, ref64):
    """Map gradients: conftest.grad_ok, or - per texel, for the grazing rows only - not further from the fp64 oracle than
    twice the fp32 oracle is.  At a grazing camera N.V is near 0, where the specular term's 1/(4 N.V N.L + 1e-7) and
    G1(N.V) amplify one ulp of N.V in the normal's gradient beyond rel 1e-4 (the rule conftest.s2m_ok states for the
    same kind of amplification in the specular -> metallic conversion)."""
    err = np.abs(got.astype(np.float64) - ref32.astype(np.float64))
    tol = 1e-4 * np.abs(ref32) + 1e-4 * np.abs(ref32).mean() + 1e-12
    ok = err <= tol
    if ref64 is not None:
        ok |= np.abs(got - ref64) <= 2 * np.abs(ref32.astype(np.float64) - ref64) + tol
    return float((err / tol).max()), bool(ok.all())


def _check_shared(got, want, key):
    got, want = np.asarray(got, np.float64).reshape(-1), np.asarray(want, np.float64).reshape(-1)
    tol = 1e-4 * np.abs(want) + 1e-4 * np.abs(want).mean()
    assert np.all(np.abs(got - want) <= tol), (key, float((np.abs(got - want) / tol).max()), got, want)


@pytest.mark.gpu
@pytest.mark.parametrize("r", CASES, ids=[r["id"] for r in CASES])
def test_camera_kernel_against_oracle(r):
    from oracle import pbr_oracle as O
    from pypbr_b200.fit import FusedAdam, fit_step, fused_loss_step
    from pypbr_b200.models import CookTorranceBRDF

    seed = 9000 + CASES.index(r)
    B, H, W, L, wf = r["B"], r["H"], r["W"], r["L"], r["wf"]
    maps, lights, inten, g = _random_case(seed, B, H, W, L, wf, normal=r["normal"])
    light_type = r["light"]
    if light_type == "directional":
        lights = torch.nn.functional.normalize(lights + torch.tensor([0.0, 0.0, 1.0]), dim=-1)
    if r["layout"] == "bcast":
        maps["metallic"] = maps["metallic"][:1].expand_as(maps["metallic"]).clone()
    camera = torch.tensor(r["camera"])
    size = 1.0 if light_type == "point" else None   # the plane keeps its default side with a directional light
    flags = dict(albedo_is_srgb=r["albedo_srgb"], specular_is_srgb=True, return_srgb=r["return_srgb"])
    acc = not r["per_light"]
    mkey = "specular" if wf == "specular" else "metallic"
    name = lambda k: "metspec" if k == mkey else k
    entry, grads = r["entry"], set(r["grads"])
    want_maps = {k for k in maps if name(k) in grads} if entry == "autograd" else (set(maps) if (entry == "fit" or grads & set(MAPS)) else set())
    want_shared = grads & set(SHARED) if entry != "fit" else set()
    if entry == "loss" and want_shared & {"lights", "view"}:
        want_shared |= {"lights", "view"}

    leaves_ref = {k: v.clone().requires_grad_(k in want_maps) for k, v in maps.items()}
    ref = CO.render(leaves_ref, camera, lights, inten, size, light_type, accumulate=acc, **flags)
    go = torch.rand(ref.shape, generator=g)   # grad_out, or the target of the loss
    if entry == "autograd":
        if want_maps:
            ref.backward(go)
    else:
        loss_ref = ((ref - go) ** 2).mean()
        if want_maps:
            loss_ref.backward()
    shared64, maps64 = {}, {}
    grazing = r["camera"] == GRAZING
    if want_shared or grazing:
        sh = {k: t.double().clone().requires_grad_(k in want_shared) for k, t in zip(SHARED, (inten, lights, camera))}
        m64 = {k: t.double().requires_grad_(grazing and k in want_maps) for k, t in maps.items()}
        ref64 = CO.render(m64, sh["view"], sh["lights"], sh["intensity"], size, light_type, accumulate=acc, **flags)
        (ref64.backward(go.double()) if entry == "autograd" else ((ref64 - go.double()) ** 2).mean().backward())
        shared64 = {k: sh[k].grad.numpy() for k in want_shared}
        maps64 = {k: m64[k].grad.numpy() for k in want_maps} if grazing else {}

    mat, leaves = _device_material(r, maps)
    multi = "per_light" if r["per_light"] else "accumulate"
    where = DEV if r["on_device"] else torch.device("cpu")
    if entry == "autograd":
        sh_dev = {k: t.clone().to(where).requires_grad_(k in want_shared) for k, t in zip(SHARED, (inten, lights, camera))}

        def call():
            out = CookTorranceBRDF(light_type, multi_light=multi, view_type="point")(
                mat, sh_dev["view"], sh_dev["lights"], sh_dev["intensity"], size, r["return_srgb"])
            out.backward(go.to(DEV))
            return out

        out, launched, ct_ran = _launched(call)
        assert out.shape == ref.shape
        ratio, ok = fwd_ok(out.detach().cpu().numpy(), ref.detach().numpy())
        assert ok, f"forward {ratio}"
        for k in maps:
            if k not in want_maps:
                assert leaves[k].grad is None, k
                continue
            exp = leaves_ref[k].grad
            if r["layout"] == "bcast" and k == "metallic":
                exp = exp.sum(0, keepdim=True)
            ratio, ok = _map_grad_ok(leaves[k].grad.cpu().numpy(), exp.numpy(), maps64.get(k))
            assert ok, f"d_{k} {ratio}"
        for k in want_shared:
            _check_shared(sh_dev[k].grad.cpu().numpy(), shared64[k], k)
    elif entry == "loss":
        args = [t.to(where) for t in (camera, lights, inten)]

        def call():
            return fused_loss_step(mat, go.to(DEV), *args, light_type, size, r["return_srgb"], multi,
                                   want_intensity_grad="intensity" in want_shared,
                                   want_geometry_grad=bool(want_shared & {"lights", "view"}), want_map_grads=bool(want_maps),
                                   view_type="point")

        (buf, dgrads), launched, ct_ran = _launched(call)
        buf = buf.cpu().numpy().astype(np.float64)
        assert buf.size == 1 + 3 * L + (3 * L + 3 if "lights" in want_shared else 0)
        lr = float(loss_ref.detach())
        assert abs(buf[0] / go.numel() - lr) <= 2e-6 * lr, (buf[0] / go.numel(), lr)
        for k in maps:
            if k in want_maps:
                ratio, ok = _map_grad_ok(dgrads[k].cpu().numpy(), leaves_ref[k].grad.numpy(), maps64.get(k))
                assert ok, f"d_{k} {ratio}"
            else:
                assert dgrads.get(k) is None, k
        if "intensity" in want_shared:
            _check_shared(buf[1:1 + 3 * L], shared64["intensity"], "intensity")
        if "lights" in want_shared:
            _check_shared(buf[1 + 3 * L:1 + 6 * L], shared64["lights"], "lights")
            _check_shared(buf[1 + 6 * L:], shared64["view"], "view")
    else:
        opt = FusedAdam({k: mat._maps[k] for k in maps}, lr=0.01)

        def call():
            return fit_step(mat, opt, go.to(DEV), camera, lights, inten, light_type, size, multi, fused=False,
                            view_type="point")

        buf, launched, ct_ran = _launched(call)
        lr = float(loss_ref.detach())
        assert abs(float(buf[0]) / go.numel() - lr) <= 2e-6 * lr
        want = O.adam_fit_steps(maps, [{k: leaves_ref[k].grad for k in maps}], lr=0.01)
        for k in maps:
            a, b = mat._maps[k].cpu(), want[k]
            # an Adam step is lr * g / (|g| + eps) whatever the gradient's size: it is defined to the test's precision only where
            # |g| is above noise level and well above eps = 1e-8 (the B = 17 row's gradients are ~1e-5: 1/numel is small)
            big = leaves_ref[k].grad.abs() > torch.clamp(1e-3 * leaves_ref[k].grad.abs().mean(), min=1e-5)
            if k == "normal":   # the projection F.normalize couples the channels: every channel's step must be defined
                big = big.all(dim=-3, keepdim=True).expand_as(big)
            assert bool(((a - b).abs()[big] <= 2e-5 * b.abs()[big] + 2e-6).all()), (k, float((a - b).abs()[big].max()))
    assert launched == set(r["kernels"]), f"launched {sorted(launched)}, row names {sorted(r['kernels'])}"
    assert not ct_ran, "an orthographic ct_* kernel ran for a camera call"


@pytest.mark.gpu
def test_fit_with_a_camera_cuts_the_loss():
    """40 steps of fit_step(fused=False, view_type="point") on 4 x 256^2 from flat maps: the loss falls at least 4x."""
    from pypbr_b200.fit import FusedAdam, fit_step
    from pypbr_b200.materials import BasecolorMetallicMaterial
    from pypbr_b200.models import CookTorranceBRDF

    B, H, W = 4, 256, 256
    maps, _, _, _ = _random_case(31, B, H, W, 1, "metallic")
    camera = torch.tensor([0.1, -0.1, 1.2])
    lights = torch.tensor([[0.3, 0.2, 1.0], [-0.3, -0.1, 0.8]])
    inten = torch.tensor([[1.0, 1.0, 1.0], [0.8, 0.8, 0.8]])
    gt = BasecolorMetallicMaterial(albedo_is_srgb=True, device=DEV)
    gt._maps.update({k: v.to(DEV) for k, v in maps.items()})
    with torch.no_grad():
        target = CookTorranceBRDF("point", multi_light="per_light", view_type="point")(gt, camera, lights, inten, 1.0)
    mat = BasecolorMetallicMaterial(albedo_is_srgb=True, device=DEV)
    flat = torch.tensor([0.0, 0.0, 1.0], device=DEV).view(1, 3, 1, 1).expand(B, 3, H, W)
    mat._maps.update(albedo=torch.full((B, 3, H, W), 0.5, device=DEV), roughness=torch.full((B, 1, H, W), 0.5, device=DEV),
                     metallic=torch.full((B, 1, H, W), 0.5, device=DEV), normal=flat.contiguous())
    opt = FusedAdam({k: mat._maps[k] for k in maps}, lr=0.05)
    losses = [float(fit_step(mat, opt, target, camera, lights, inten, "point", 1.0, fused=False, view_type="point")[0])
              for _ in range(40)]
    assert losses[-1] * 4 <= losses[0], losses
