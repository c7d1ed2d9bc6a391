"""
Every compiled Cook-Torrance kernel at the edges of its inputs: the rows of the two kernel ledgers
(test_gpu_kernel_coverage.CASES, test_gpu_camera.CASES), each run on the edge atlas of tests/test_edges_host.py instead
of the benign random material.

For every row the atlas is tiled to the row's (B, H, W), and the row's L lights are taken in turn from the edge lightings
(test_edges_host.point_lightings / dir_lightings; camera rows also cycle through test_edges_host.cameras), as many runs
as it takes for every edge lighting to reach the row.  Each run goes through the row's own entry (autograd, fused loss,
one-launch fit step, conversion, camera) and asserts under torch.profiler that exactly the row's kernels launched, so the
edges reach the streamed kFast and general kernels, the 64-bit-access and element-access flavours, every geometry-cache
mode, the plain-case flavour, the loss kernel and the fit step on both sides of each shared-memory reduction boundary.

The comparison rules are test_edges_host.py's (its docstring): the image with fwd_ok or the fp64 arbiter, map gradients
with grad_ok per atlas category or the fp64 arbiter, finiteness wherever the fp32 oracle is finite, the shared-parameter
gradients against the fp64 oracle.  The fit step compares the updated maps with an Adam step on the oracle's gradients
where that step is defined to the test's precision: the fp32 and fp64 gradients agree to 1e-3 and are above 1e-3 of
their category's mean (an Adam step has the size lr whatever the gradient, so its sign must be defined).
test_every_compiled_kernel_is_reached: the rows are every row of both ledgers, so they cover every name in
compiled_kernels() and every camera kernel.
"""
import numpy as np
import pytest
import torch

import camera_oracle as CO
import test_gpu_camera as CAM
import test_gpu_kernel_coverage as KC
from test_edges_host import (SHARED, VIEW_UP, _labels_like, cameras, check_finite, check_forward, check_map_grad,
                             check_shared, dir_lightings, edge_atlas, in_plane, oracle, point_lightings)
from test_gpu_kernel_coverage import CASES, _device_material

DEV = KC.DEV
ROWS = [("ct", r) for r in CASES] + [("cam", r) for r in CAM.CASES]


def _runs(kind, r, H, W):
    """The (view / camera, lights, intensities) of each run of a row: every edge lighting reaches the row."""
    edges = point_lightings(H, W) if r["light"] == "point" else dir_lightings()
    L, n = r["L"], len(edges)
    starts = list(range(0, n, L)) if L < n else [0]
    cams = [c for _, c in cameras(H, W)]
    if kind == "cam":
        starts = [starts[k % len(starts)] for k in range(max(len(starts), len(cams)))]
    runs = []
    for k, s in enumerate(starts):
        pick = [edges[(s + i) % n] for i in range(L)]
        view = cams[k % len(cams)] if kind == "cam" else VIEW_UP
        runs.append((torch.tensor(view), torch.tensor([p for _, p, _ in pick]), torch.tensor([i for _, _, i in pick])))
    return runs


def _atlas(r):
    B = r["B"] or 1
    wf_maps = "specular" if r["entry"] == "convert" else r["wf"]
    maps, cat = edge_atlas(B, r["H"], r["W"], wf_maps)
    if not r["normal"]:
        del maps["normal"]
    if r["layout"] == "bcast":   # one metallic map for the batch: the same values for every material
        maps["metallic"] = maps["metallic"][:1].expand_as(maps["metallic"]).clone()
    return maps, cat


def _launched(kind, fn):
    """fn() under torch.profiler -> (its result, the Cook-Torrance kernels of the row's ledger that it launched); a camera
    call must launch no orthographic kernel."""
    if kind == "cam":
        res, launched, ct_ran = CAM._launched(fn)
        assert not ct_ran, "an orthographic ct_* kernel ran for a camera call"
        return res, launched
    return KC._launched(fn)


def _unbatch(lights, inten, L):
    return (lights, inten) if L > 1 else (lights[0], inten[0])


def test_every_compiled_kernel_is_reached():
    """Every row of both ledgers is a row here, so the edges reach every kernel that test_every_compiled_kernel_has_a_row
    and test_every_camera_kernel_has_a_row tie to the library; in particular every name in compiled_kernels()."""
    assert [r["id"] for _, r in ROWS] == [r["id"] for r in CASES] + [r["id"] for r in CAM.CASES]
    assert KC.compiled_kernels() <= {k for _, r in ROWS for k in r["kernels"]}


def _check_fit(mat, maps, g32, g64, cat, projection):
    from oracle import pbr_oracle as O

    want = O.adam_fit_steps(maps, [{k: torch.from_numpy(g32[k]) for k in maps}], lr=0.01, projection=projection)
    for k in maps:
        a, b = mat._maps[k].detach().cpu().numpy(), want[k].numpy()
        check_finite(f"fit {k}", a, b)
        r32, r64 = np.abs(g32[k]), g64[k]
        lab = _labels_like(r32, cat)
        big = np.zeros(r32.shape, bool)
        for c in np.unique(lab):
            sel = lab == c
            big[sel] = r32[sel] > 1e-3 * r32[sel].mean()
        big &= np.abs(g32[k] - r64) <= 1e-3 * np.abs(r64)
        if k == "normal":   # F.normalize couples the channels: every channel's step must be defined
            big = np.broadcast_to(big.all(axis=-3, keepdims=True), big.shape)
        err = np.abs(a - b)
        ok = err[big] <= 2e-5 * np.abs(b[big]) + 2e-6
        assert ok.all(), (k, float(err[big].max()))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,r", ROWS, ids=[f"{kind}-{r['id']}" for kind, r in ROWS])
def test_kernel_at_the_edges(kind, r):
    for run, (view, lights, inten) in enumerate(_runs(kind, r, r["H"], r["W"])):
        try:
            _run_row(kind, r, run, view, lights, inten)
        except AssertionError as e:
            raise AssertionError(f"run {run}: view {view.tolist()}, lights {lights.tolist()}: {e}") from None


def _run_row(kind, r, run, view, lights, inten):
    from oracle import pbr_oracle as O
    from pypbr_b200.fit import FusedAdam, fit_step, fused_fit_step, fused_loss_step
    from pypbr_b200.materials import DiffuseSpecularMaterial
    from pypbr_b200.models import CookTorranceBRDF

    H, W, L, wf, entry = r["H"], r["W"], r["L"], r["wf"], r["entry"]
    light_type = r["light"]
    size = 1.0 if light_type == "point" else None
    flags = dict(albedo_is_srgb=r["albedo_srgb"], specular_is_srgb=True, return_srgb=r["return_srgb"])
    acc = not r["per_light"]
    multi = "per_light" if r["per_light"] else "accumulate"
    render = CO.render if kind == "cam" else O.render
    maps, cat = _atlas(r)
    lights, inten = _unbatch(lights, inten, L)
    gen = torch.Generator().manual_seed(run)
    if entry == "convert":
        ref = {k: v[0].clone().requires_grad_(True) for k, v in maps.items()}
        b, m = O.specular_to_metallic(ref["albedo"], ref["specular"], True)
        conv = dict(albedo=b, metallic=m, normal=ref["normal"], roughness=ref["roughness"])
        out_ref = O.render(conv, view, lights, inten, size, light_type, albedo_is_srgb=False)
        go = torch.rand(out_ref.shape, generator=gen) + 0.5
        out_ref.backward(go)
        r64 = {k: v[0].double().requires_grad_(True) for k, v in maps.items()}
        b64, m64 = O.specular_to_metallic(r64["albedo"], r64["specular"], True)
        out64 = O.render(dict(albedo=b64, metallic=m64, normal=r64["normal"], roughness=r64["roughness"]), view.double(),
                         lights.double(), inten.double(), size, light_type, albedo_is_srgb=False)
        out64.backward(go.double())
        lv = {k: v[0].to(DEV).requires_grad_(True) for k, v in maps.items()}
        mat = DiffuseSpecularMaterial(albedo_is_srgb=True, device=DEV)
        mat._maps.update(lv)

        def call():
            res = CookTorranceBRDF(light_type)(mat.to_basecolor_metallic_material(), view, lights, inten, size)
            res.backward(go.to(DEV))
            return res

        out, launched = _launched(kind, call)
        check_forward(out.detach().cpu().numpy()[None], out_ref.detach().numpy()[None], out64.detach().numpy()[None], cat)
        for k in maps:
            check_map_grad(k, lv[k].grad.cpu().numpy()[None], ref[k].grad.numpy()[None], r64[k].grad.numpy()[None], cat,
                           in_plane(light_type, lights))
        assert launched == set(r["kernels"]), f"launched {sorted(launched)}, row names {sorted(r['kernels'])}"
        return

    mkey = "specular" if wf == "specular" else "metallic"
    name = lambda k: "metspec" if k == mkey else k
    grads = set(r["grads"])
    want_maps = {k for k in maps if name(k) in grads} if entry == "autograd" else (
        set(maps) if (entry == "fit" or grads & set(KC.MAPS)) else set())
    want_shared = grads & set(SHARED) if not (kind == "cam" and entry == "fit") else set()
    if entry == "loss" and want_shared & {"lights", "view"}:
        want_shared |= {"lights", "view"}
    img = render(maps, view, lights, inten, size, light_type, accumulate=acc, **flags)
    go = torch.rand(img.shape, generator=gen) + (0.5 if entry == "autograd" else 0.0)   # grad_out, or the loss target
    if entry == "autograd":
        ref = oracle(render, maps, view, lights, inten, size, light_type, acc, flags, go)
    else:   # the gradients of the mean squared error: its d loss / d image as the output gradient
        loss_ref = float(((img - go) ** 2).mean())
        ref = oracle(render, maps, view, lights, inten, size, light_type, acc, flags, 2.0 * (img - go) / go.numel())
    mat, leaves = (CAM._device_material if kind == "cam" else _device_material)(r, maps)
    bcast = r["layout"] == "bcast"

    def expect(k, g):
        return g.sum(0, keepdims=True) if bcast and k == "metallic" else g

    where = DEV if r.get("on_device") else torch.device("cpu")
    vt = dict(view_type="point") if kind == "cam" else {}
    if entry == "autograd":
        sh_dev = {k: t.clone().to(where).requires_grad_(k in want_shared) for k, t in zip(SHARED, (inten, lights, view))}

        def call():
            out = CookTorranceBRDF(light_type, multi_light=multi, **vt)(mat, sh_dev["view"], sh_dev["lights"],
                                                                       sh_dev["intensity"], size, r["return_srgb"])
            out.backward(go.to(DEV))
            return out

        res, launched = _launched(kind, call)
        check_forward(res.detach().cpu().numpy(), ref["out"], ref["out64"], cat)
        for k in maps:
            if k in want_maps:
                check_map_grad(k, leaves[k].grad.cpu().numpy(), expect(k, ref["g32"][k]), expect(k, ref["g64"][k]), cat,
                               in_plane(light_type, lights))
        for k in want_shared:
            check_shared(k, sh_dev[k].grad.cpu().numpy(), ref["shared64"][k], ref["shared32"][k])
    elif entry == "loss":
        args = [t.to(where) for t in (view, lights, inten)]

        def call():
            return fused_loss_step(mat, go.to(DEV), *args, light_type, size, r["return_srgb"], multi,
                                   want_intensity_grad="intensity" in want_shared,
                                   want_geometry_grad=bool(want_shared & {"lights", "view"}),
                                   want_map_grads=bool(want_maps), **vt)

        (buf, dgrads), launched = _launched(kind, call)
        buf = buf.cpu().numpy().astype(np.float64)
        assert np.isfinite(buf).all(), buf
        assert abs(buf[0] / go.numel() - loss_ref) <= 2e-6 * loss_ref + 1e-12, (buf[0] / go.numel(), loss_ref)
        for k in want_maps:
            check_map_grad(k, dgrads[k].cpu().numpy(), ref["g32"][k], ref["g64"][k], cat, in_plane(light_type, lights))
        if "intensity" in want_shared:
            check_shared("intensity", buf[1:1 + 3 * L], ref["shared64"]["intensity"], ref["shared32"]["intensity"])
        if "lights" in want_shared:
            check_shared("lights", buf[1 + 3 * L:1 + 6 * L], ref["shared64"]["lights"], ref["shared32"]["lights"])
            check_shared("view", buf[1 + 6 * L:], ref["shared64"]["view"], ref["shared32"]["view"])
    else:
        project = None if r.get("project", True) else {k: None for k in maps}
        opt = FusedAdam({k: mat._maps[k] for k in maps}, lr=0.01, project=project)
        if kind == "cam":
            def call():
                return fit_step(mat, opt, go.to(DEV), view, lights, inten, light_type, size, multi, fused=False,
                                view_type="point")
        else:
            def call():
                return fused_fit_step(mat, opt, go.to(DEV), view, lights, inten, light_type, size, r["return_srgb"], multi,
                                      want_intensity_grad="intensity" in want_shared)

        buf, launched = _launched(kind, call)
        buf = buf.cpu().numpy().astype(np.float64).reshape(-1)
        assert np.isfinite(buf).all(), buf
        assert abs(buf[0] / go.numel() - loss_ref) <= 2e-6 * loss_ref + 1e-12, (buf[0] / go.numel(), loss_ref)
        _check_fit(mat, maps, ref["g32"], ref["g64"], cat, project)
        if "intensity" in want_shared:
            check_shared("intensity", buf[1:1 + 3 * L], ref["shared64"]["intensity"], ref["shared32"]["intensity"])
    assert launched == set(r["kernels"]), f"run {run}: launched {sorted(launched)}, row names {sorted(r['kernels'])}"
