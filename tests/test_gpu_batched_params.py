"""
Per-material view, lights and intensities on the GPU (the pbr_ct_*_pb entry points).  A batched call with per-material
parameters is B independent calls, so each row checks

  * bitwise equality with a loop of B single-material calls (FORCE_GENERIC, so both pick the same generic instantiation,
    which torch.profiler confirms): outputs and map gradients with torch.equal; the sums over texels (shared-parameter
    gradients, per-material parameter gradients, the loss) with grad_ok, since their atomics add in another order;
  * parity with the oracle (oracle/pbr_oracle.py, tests/camera_oracle.py for the camera) looped over b, fwd_ok / grad_ok,
    including gradients of per-material (B, L, 3) / (B, 3) leaves and of a shared leaf mixed with them;
  * the kernel set: no streamed kernel, no cached light mode, and every kernel is in the existing ledgers.
"""
import numpy as np
import pytest
import torch

import camera_oracle as CO
from conftest import fwd_ok, grad_ok
from test_gpu_camera import CASES as CAM_CASES, norm_kernel as norm_cam
from test_gpu_kernel_coverage import CASES as CT_CASES, norm_kernel

DEV = torch.device("cuda:0") if torch.cuda.is_available() else None
LEDGER = {k for r in CT_CASES + CAM_CASES for k in r["kernels"]}   # every kernel the two kernel ledgers test
PARAMS = ("intensity", "lights", "view")


def _case(seed, B, H, W, L, wf, light_type, camera, normal=True):
    g = torch.Generator().manual_seed(seed)
    shp = lambda c: (B, c, H, W)
    maps = {"albedo": torch.rand(shp(3), generator=g), "roughness": torch.rand(shp(1), generator=g) * 0.8 + 0.2}
    if normal:
        n = torch.randn(shp(3), generator=g) * torch.tensor([0.3, 0.3, 0.0]).view(1, 3, 1, 1)
        maps["normal"] = torch.nn.functional.normalize(n + torch.tensor([0.0, 0.0, 1.0]).view(1, 3, 1, 1), dim=1)
    if wf == "specular":
        maps["specular"] = torch.rand(shp(3), generator=g)
    else:
        maps["metallic"] = torch.rand(shp(3 if wf == "metallic3" else 1), generator=g)
    lights = torch.rand(B, L, 3, generator=g) * torch.tensor([0.8, 0.8, 0.5]) - torch.tensor([0.4, 0.4, -0.8])
    if light_type == "directional":
        lights = torch.nn.functional.normalize(lights * torch.tensor([0.5, 0.5, 1.0]), dim=-1)
    inten = (torch.rand(B, L, 3, generator=g) * 0.5 + 0.5) / L
    if camera:
        view = torch.rand(B, 3, generator=g) * torch.tensor([0.4, 0.4, 0.5]) - torch.tensor([0.2, 0.2, -1.2])
    else:
        view = torch.nn.functional.normalize(torch.rand(B, 3, generator=g) * torch.tensor([0.3, 0.3, 0.0])
                                             + torch.tensor([0.0, 0.0, 1.0]), dim=-1)
    return maps, lights, inten, view, g


def _material(maps, wf, misaligned=False, grad=True):
    from pypbr_b200.materials import BasecolorMetallicMaterial, DiffuseSpecularMaterial

    cls = DiffuseSpecularMaterial if wf == "specular" else BasecolorMetallicMaterial
    m = cls(albedo_is_srgb=True, device=DEV)
    leaves = {}
    for k, v in maps.items():
        t = v.to(DEV)
        if misaligned:   # first texel 4-byte aligned: the element-access flavour
            wide = torch.zeros(*t.shape[:-1], t.shape[-1] + 8, device=DEV)
            wide[..., 1:1 + t.shape[-1]] = t
            t = wide[..., 1:1 + t.shape[-1]]
        leaves[k] = t.detach().requires_grad_(grad)
        m._maps[k] = leaves[k]
    if "normal" not in maps:
        m._maps["normal"] = None
    return m, leaves


def _launched(fn):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    return res, {k for k in (norm_kernel(n) or norm_cam(n) for n in names) if k}


def _check_kernels(launched):
    """Per-material calls: generic kernels only, light modes directional / per-texel point / hoisted, all in the ledgers."""
    assert launched, "no Cook-Torrance kernel ran"
    for k in launched:
        assert "stream" not in k, k
        light = int(k.split("<")[1].rstrip(">").split(",")[1])
        assert light in (0, 1, 2), f"{k}: a cached light mode"
    assert launched <= LEDGER, sorted(launched - LEDGER)


def _close(got, want, what):
    ratio, ok = grad_ok(np.asarray(got, np.float64), np.asarray(want, np.float64))
    assert ok, f"{what}: {ratio}"


# (wf, light type, camera, multi_light, normal map, L, B, H, W, misaligned)
ROWS = [
    ("metallic", "point", False, "accumulate", True, 1, 3, 4, 40, False),
    ("metallic", "point", True, "per_light", True, 1, 17, 3, 20, False),
    ("metallic", "point", False, "accumulate", True, 3, 17, 3, 20, False),
    ("metallic", "directional", False, "per_light", True, 3, 3, 4, 40, False),
    ("metallic", "directional", True, "accumulate", False, 3, 3, 4, 41, False),
    ("specular", "point", False, "per_light", False, 20, 3, 3, 20, False),
    ("specular", "point", True, "accumulate", True, 3, 3, 4, 41, False),
    ("specular", "directional", False, "accumulate", True, 1, 17, 3, 20, False),
    ("metallic3", "point", False, "per_light", True, 3, 3, 4, 40, True),
    ("metallic3", "point", True, "accumulate", True, 20, 3, 3, 20, False),
    ("metallic3", "directional", False, "accumulate", True, 20, 1, 4, 40, False),
    ("metallic", "point", False, "accumulate", True, 3, 3, 4, 41, True),
    ("specular", "point", False, "accumulate", True, 1, 3, 4, 40, True),
]
IDS = ["-".join(str(x) for x in (wf, lt, "cam" if cam else "dir", ml[:3], "n" if nrm else "nonormal", f"L{L}", f"B{B}",
                                 f"{H}x{W}", "misaligned" if mis else ""))
       for wf, lt, cam, ml, nrm, L, B, H, W, mis in ROWS]


@pytest.mark.gpu
@pytest.mark.parametrize("row", ROWS, ids=IDS)
def test_batched_call_is_the_loop_of_single_calls(row):
    """autograd through CookTorranceBRDF: per-material lights, intensities and view, every leaf requiring a gradient."""
    from pypbr_b200.models import CookTorranceBRDF
    from pypbr_b200.models import cooktorrance as ct

    wf, light_type, camera, multi, normal, L, B, H, W, mis = row
    maps, lights, inten, view, g = _case(1000 + ROWS.index(row), B, H, W, L, wf, light_type, camera, normal)
    brdf = CookTorranceBRDF(light_type, multi_light=multi, view_type="point" if camera else "directional")
    size = 1.0 if light_type == "point" else None
    mat, leaves = _material(maps, wf, mis)
    sh = {k: t.to(DEV).requires_grad_(True) for k, t in zip(PARAMS, (inten, lights, view))}
    ct.FORCE_GENERIC = True
    try:
        def batched():
            out = brdf(mat, sh["view"], sh["lights"], sh["intensity"], size)
            out.backward(go)
            return out

        with torch.no_grad():
            go = torch.rand(brdf(mat, sh["view"], sh["lights"], sh["intensity"], size).shape, generator=g).to(DEV)
        out, kb = _launched(batched)
        one, one_leaves = _material({k: v[:1] for k, v in maps.items()}, wf, mis)
        outs, grads, kl = [], {k: [] for k in list(maps) + list(PARAMS)}, set()
        for b in range(B):
            for k, v in maps.items():
                with torch.no_grad():
                    one_leaves[k].copy_(v[b:b + 1])
                one_leaves[k].grad = None
            p1 = {k: t[b].to(DEV).requires_grad_(True) for k, t in zip(PARAMS, (inten, lights, view))}

            def single():
                o = brdf(one, p1["view"], p1["lights"], p1["intensity"], size)
                o.backward(go[b:b + 1])
                return o

            o, k1 = _launched(single)
            kl |= k1
            outs.append(o.detach())
            for k in maps:
                grads[k].append(one_leaves[k].grad.clone())
            for k in PARAMS:
                grads[k].append(p1[k].grad)
    finally:
        ct.FORCE_GENERIC = False
    assert kb == kl, (sorted(kb), sorted(kl))
    _check_kernels(kb)
    assert torch.equal(out.detach(), torch.cat(outs)), "output"
    for k in maps:
        assert torch.equal(leaves[k].grad, torch.cat(grads[k])), f"d_{k}"
    for k in PARAMS:
        assert sh[k].grad.shape == sh[k].shape
        _close(sh[k].grad.cpu(), torch.stack(grads[k]).cpu(), f"d_{k}")


def _oracle(maps, view, lights, inten, size, light_type, camera, accumulate, want, go):
    """The oracle looped over b; returns the render and the gradients of every leaf in `want` (fp32, the oracle's own)."""
    from oracle import pbr_oracle as O

    R = CO.render if camera else O.render
    leaves = {k: v.clone().requires_grad_(k in want) for k, v in maps.items()}
    sh = {k: t.clone().requires_grad_(k in want) for k, t in zip(PARAMS, (inten, lights, view))}
    outs = []
    for b in range(maps["albedo"].shape[0]):
        mb = {k: v[b] for k, v in leaves.items()}
        # material b's parameters: row b of a per-material one, row 0 of a (1, ...) shared one
        pick = lambda t, nd: (t[b] if t.shape[0] > 1 else t[0]) if t.dim() == nd else t
        lb = pick(sh["lights"], 3)
        ib = pick(sh["intensity"], 3)
        ib = ib.view(-1, 3).expand(lb.view(-1, 3).shape[0], 3) if ib.numel() == 3 else ib
        outs.append(R(mb, pick(sh["view"], 2), lb, ib, size, light_type, accumulate=accumulate))
    ref = torch.stack(outs)
    ref.backward(go)
    return ref, {k: t.grad for k, t in {**leaves, **sh}.items() if k in want}


# (wf, light type, camera, multi_light, which parameters are per material, L, B, W)
ORACLE_ROWS = [
    ("metallic", "point", True, "per_light", ("lights", "view", "intensity"), 3, 3, 40),
    ("metallic", "point", False, "accumulate", ("lights",), 1, 17, 20),                  # shared view and intensity
    ("specular", "directional", False, "per_light", ("view", "intensity"), 3, 3, 41),    # shared lights
    ("metallic3", "point", True, "accumulate", ("lights", "intensity1"), 20, 3, 20),     # (B, 1, 3) intensity, shared camera
    ("metallic3", "directional", True, "accumulate", ("view",), 1, 3, 40),
]


@pytest.mark.gpu
@pytest.mark.parametrize("row", ORACLE_ROWS, ids=["-".join(str(x) for x in (r[0], r[1], "cam" if r[2] else "dir", r[3][:3],
                                                                            "+".join(r[4]), f"L{r[5]}", f"B{r[6]}", f"W{r[7]}"))
                                                  for r in ORACLE_ROWS])
def test_batched_call_against_the_oracle(row):
    from pypbr_b200.models import CookTorranceBRDF

    wf, light_type, camera, multi, pm, L, B, W = row
    H = 4
    maps, lights, inten, view, g = _case(2000 + ORACLE_ROWS.index(row), B, H, W, L, wf, light_type, camera)
    if "lights" not in pm:
        lights = lights[0]
    if "view" not in pm:
        view = view[0]
    if "intensity1" in pm:
        inten = inten[:, :1].contiguous()
    elif "intensity" not in pm:
        inten = inten[:1]                  # (1, L, 3): shared
    size = 1.0 if light_type == "point" else None
    want = set(maps) | set(PARAMS)
    acc = multi == "accumulate"
    with torch.no_grad():
        shape = CO.render({k: v[0] for k, v in maps.items()}, view.reshape(-1, 3)[0], lights.reshape(-1, L, 3)[0],
                          torch.ones(L, 3), size, light_type, accumulate=acc).shape
    go = torch.rand(B, *shape, generator=g)
    ref, rg = _oracle(maps, view, lights, inten, size, light_type, camera, acc, want, go)
    mat, leaves = _material(maps, wf)
    sh = {k: t.to(DEV).requires_grad_(True) for k, t in zip(PARAMS, (inten, lights, view))}
    brdf = CookTorranceBRDF(light_type, multi_light=multi, view_type="point" if camera else "directional")
    out, launched = _launched(lambda: brdf(mat, sh["view"], sh["lights"], sh["intensity"], size))
    _check_kernels(launched)
    ratio, ok = fwd_ok(out.detach().cpu().numpy(), ref.detach().numpy())
    assert ok, f"forward {ratio}"
    _, launched = _launched(lambda: out.backward(go.to(DEV)))
    _check_kernels(launched)
    for k in maps:
        _close(leaves[k].grad.cpu(), rg[k], f"d_{k}")
    for k in PARAMS:
        assert sh[k].grad.shape == sh[k].shape, k
        _close(sh[k].grad.cpu(), rg[k], f"d_{k}")


@pytest.mark.gpu
@pytest.mark.parametrize("camera", [False, True])
def test_fused_loss_step_with_per_material_parameters(camera):
    """buf keeps its layout with the per-material sections zero; their gradients come back in grads, in the parameters'
    shapes; a shared intensity's stays in buf.  Loss and map gradients against the oracle."""
    from pypbr_b200.fit import fused_loss_step

    B, H, W, L, wf = 5, 4, 40, 3, "metallic"
    maps, lights, inten, view, g = _case(3000 + camera, B, H, W, L, wf, "point", camera)
    inten = inten[:1]   # shared
    target = torch.rand(B, L, 3, H, W, generator=g)
    want = set(maps) | set(PARAMS)
    from oracle import pbr_oracle as O
    R = CO.render if camera else O.render
    lv = {k: v.clone().requires_grad_(True) for k, v in maps.items()}
    sh = {k: t.clone().requires_grad_(True) for k, t in zip(PARAMS, (inten, lights, view))}
    ref = torch.stack([R({k: v[b] for k, v in lv.items()}, sh["view"][b], sh["lights"][b], sh["intensity"][0], 1.0, "point",
                         accumulate=False) for b in range(B)])
    loss = ((ref - target) ** 2).mean()
    loss.backward()
    mat, _ = _material(maps, wf, grad=False)
    out = {}
    for _ in range(2):   # the second call reuses the buffers in `out`
        (buf, grads), launched = _launched(lambda: fused_loss_step(
            mat, target.to(DEV), view.to(DEV), lights.to(DEV), inten, "point", 1.0, multi_light="per_light", out=out,
            want_intensity_grad=True, want_geometry_grad=True, view_type="point" if camera else "directional"))
        _check_kernels(launched)
        buf = buf.cpu().double()
        assert buf.numel() == 1 + 6 * L + 3
        assert abs(float(buf[0]) / target.numel() - float(loss)) <= 2e-6 * float(loss)
        assert torch.count_nonzero(buf[1 + 3 * L:]) == 0, "per-material sections of buf must stay zero"
        _close(buf[1:1 + 3 * L].view(1, L, 3), sh["intensity"].grad, "d_intensity (shared)")
        for k in ("lights", "view"):
            assert grads[k].shape == sh[k].shape and grads[k] is out[k]
            _close(grads[k].cpu(), sh[k].grad, f"d_{k}")
        assert "intensity" not in grads
        for k in maps:
            _close(grads[k].cpu(), lv[k].grad, f"d_{k}")


@pytest.mark.gpu
def test_fused_loss_step_broadcast_intensity_gradient_has_the_parameters_shape():
    from pypbr_b200.fit import fused_loss_step
    from oracle import pbr_oracle as O

    B, H, W, L = 3, 4, 40, 2
    maps, lights, inten, view, g = _case(3100, B, H, W, L, "specular", "point", False)
    inten = inten[:, :1].contiguous()   # (B, 1, 3)
    target = torch.rand(B, L, 3, H, W, generator=g)
    iv = inten.clone().requires_grad_(True)
    ref = torch.stack([O.render({k: v[b] for k, v in maps.items()}, view[0], lights[b], iv[b].expand(L, 3), 1.0, "point",
                                accumulate=False) for b in range(B)])
    ((ref - target) ** 2).mean().backward()
    mat, _ = _material(maps, "specular", grad=False)
    out = {}
    for _ in range(2):   # the second call reduces into the buffer the first one left in `out`
        buf, grads = fused_loss_step(mat, target.to(DEV), view[0], lights.to(DEV), inten.to(DEV), "point", 1.0,
                                     multi_light="per_light", want_intensity_grad=True, out=out)
        assert grads["intensity"].shape == (B, 1, 3) and grads["intensity"] is out["intensity_sum"]
        assert torch.count_nonzero(buf[1:]) == 0
        _close(grads["intensity"].cpu(), iv.grad, "d_intensity")


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 8])
def test_one_launch_fit_step_with_per_material_lights(L):
    """fused_fit_step with per-material lights and intensities == fused_loss_step + FusedAdam.step (the tolerance of
    test_one_launch_fit_step_equals_loss_kernel_plus_adam_kernel); its per-material intensity gradient goes to
    scratch["d_intensity"]."""
    from pypbr_b200.fit import FusedAdam, fused_fit_step, fused_loss_step
    from pypbr_b200.models import cooktorrance as ct

    B, H, W = 3, 27, 44
    maps, lights, inten, view, g = _case(4000 + L, B, H, W, L, "metallic", "point", False)
    target = torch.rand(B, L, 3, H, W, generator=g).to(DEV)
    args = (view[0], lights.to(DEV), inten.to(DEV), "point", 1.0)

    def make():
        m, lv = _material({k: v * 0.7 + 0.1 if k != "normal" else v for k, v in maps.items()}, "metallic", grad=False)
        return m, lv, FusedAdam(lv, lr=0.03)

    (ma, la, oa), (mb, lb, ob) = make(), make()
    scratch = {}
    ct.FORCE_GENERIC = True
    try:
        for step in (1, 2):
            # one step from identical state each time (as test_one_launch_fit_step_equals_loss_kernel_plus_adam_kernel);
            # the step counts advance on their own: the second step's bias correction reads them
            for k in la:
                lb[k].copy_(la[k]); ob.state[k][0].copy_(oa.state[k][0]); ob.state[k][1].copy_(oa.state[k][1])
            red_a, grads = fused_loss_step(ma, target, *args, multi_light="per_light", loss_scale=1.0 / target.numel(),
                                           want_intensity_grad=True)
            oa.step({k: grads[k] for k in oa.params})
            red_b, launched = _launched(lambda: fused_fit_step(mb, ob, target, *args, multi_light="per_light",
                                                               want_intensity_grad=True, scratch=scratch))
            assert type(ob.step_count) is int and ob.step_count == oa.step_count == step
            _check_kernels(launched)
            assert abs(float(red_a[0]) - float(red_b[0])) <= 1e-6 * abs(float(red_a[0]))
            assert torch.count_nonzero(red_b[1:]) == 0
            _close(scratch["d_intensity"].cpu(), grads["intensity"].cpu(), "d_intensity")
            for k in la:
                for a, b, what in ((la[k], lb[k], "param"), (oa.state[k][0], ob.state[k][0], "exp_avg"),
                                   (oa.state[k][1], ob.state[k][1], "exp_avg_sq")):
                    err = (a - b).abs()
                    tol = 1e-5 * a.abs() + 2e-5 * a.abs().mean() + (2e-7 if what == "param" else 0.0)
                    ok = err <= tol
                    if what == "param":
                        m1 = oa.state[k][0].abs()
                        ok = ok | (m1 <= 1e-4 * m1.mean())
                    assert bool(ok.all()), (step, k, what, float((err / tol)[~ok].max()))
    finally:
        ct.FORCE_GENERIC = False


@pytest.mark.gpu
def test_rendering_loss_and_fit_step_take_per_material_parameters():
    """RenderingLoss maps the per-material gradients onto its leaves; fit_step(fused=False) runs and lowers the loss."""
    from pypbr_b200.fit import FusedAdam, RenderingLoss, fit_step
    from oracle import pbr_oracle as O

    B, H, W, L = 3, 4, 40, 2
    maps, lights, inten, view, g = _case(5000, B, H, W, L, "metallic", "point", False)
    lt = lights.to(DEV).requires_grad_(True)
    it = inten[:, :1].contiguous().to(DEV).requires_grad_(True)
    target = torch.rand(B, L, 3, H, W, generator=g)
    crit = RenderingLoss("point", view_dir=view[0], light_dir=lt, light_intensity=it, light_size=1.0)
    mat, leaves = _material(maps, "metallic")
    loss = crit(mat, target.to(DEV))
    loss.backward()
    lr_, ir = lights.clone().requires_grad_(True), inten[:, :1].clone().requires_grad_(True)
    lv = {k: v.clone().requires_grad_(True) for k, v in maps.items()}
    ref = torch.stack([O.render({k: v[b] for k, v in lv.items()}, view[0], lr_[b], ir[b].expand(L, 3), 1.0, "point",
                                accumulate=False) for b in range(B)])
    rl = ((ref - target) ** 2).mean()
    rl.backward()
    assert abs(float(loss) - float(rl)) <= 2e-6 * float(rl)
    _close(lt.grad.cpu(), lr_.grad, "d_lights")
    _close(it.grad.cpu(), ir.grad, "d_intensity")
    for k in maps:
        _close(leaves[k].grad.cpu(), lv[k].grad, f"d_{k}")
    for fused in (False, True):
        m, lv2 = _material({k: v * 0.5 + 0.25 if k != "normal" else v for k, v in maps.items()}, "metallic", grad=False)
        opt = FusedAdam(lv2, lr=0.05)
        losses = [float(fit_step(m, opt, target.to(DEV), view[0], lights.to(DEV), inten.to(DEV), "point", 1.0,
                                 fused=fused)[0]) for _ in range(10)]
        assert losses[-1] < losses[0], losses
