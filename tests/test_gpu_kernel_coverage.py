"""
Every compiled Cook-Torrance kernel against the oracle.

The host dispatch (pbr_kernels.cu: light_mode, launch_fwd / launch_bwd, stream_shape, ct_dispatch) picks one of the
library's ct_{forward,backward}_{kernel,stream} instantiations from the workflow, the light type and count, the batch,
the alignment and the gradients requested.  Each row of CASES is one call through the public API with the exact set of
instantiations it must launch; the row compares the call's results with the oracle and checks, under torch.profiler,
that those kernels (and no other Cook-Torrance kernel) ran.  test_every_compiled_kernel_has_a_row is the ledger: the
instantiations defined in libpbrcuda.so must be exactly the union of the kernels named in CASES, so a new instantiation
without a parity row, or a row naming a kernel that no longer exists, fails the CPU suite.

Kernel names are written as ncu prints them, booleans as 0 / 1:
  ct_forward_kernel<WF, light, kVec, kFM>           ct_backward_kernel<WF, light, kGeom, kVec, kFM>
  ct_forward_stream<WF, light, kFast>               ct_backward_stream<WF, light, mode, kFast>   (mode: 1 loss | 2 d_intensity)
WF: 0 metallic (1-channel map), 1 specular, 2 metallic with a 3-channel map.  Light modes: pbr_shade.cuh, LightMode.
"""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, fwd_ok, grad_ok

DEV = torch.device("cuda:0") if torch.cuda.is_available() else None
LIB = os.path.join(ROOT, "pypbr_b200", "lib", "libpbrcuda.so")

DIR, PT, HOIST, C6, C8, C8BIG = range(6)   # LightMode: directional, per-texel point, hoisted, 6-field / 8-field / 8-field big cache
WFS = {"metallic": 0, "specular": 1, "metallic3": 2}
MAPS = ("albedo", "normal", "roughness", "metspec")
SHARED = ("intensity", "lights", "view")


def fk(wf, light, vec, fm=0):
    return f"ct_forward_kernel<{wf}, {light}, {int(vec)}, {fm}>"


def bk(wf, light, geom, vec, fm=0):
    return f"ct_backward_kernel<{wf}, {light}, {int(geom)}, {int(vec)}, {fm}>"


def fs(wf, light, fast):
    return f"ct_forward_stream<{wf}, {light}, {int(fast)}>"


def bs(wf, light, mode, fast):
    return f"ct_backward_stream<{wf}, {light}, {mode}, {int(fast)}>"


_NAME = re.compile(r"(ct_(?:forward|backward)_(?:kernel|stream))\s*<([^<>]*)>")


def norm_kernel(name):
    """'void pbr::ct_backward_kernel<0, 3, false, true, 1>(pbr::CtKParams)' or 'ct_backward_kernel<0, 3, 0, 1, 1>' ->
    'ct_backward_kernel<0, 3, 0, 1, 1>'; None for anything that is not a Cook-Torrance kernel."""
    m = _NAME.search(name)
    if not m:
        return None
    args = [a.strip().replace("true", "1").replace("false", "0") for a in m.group(2).split(",")]
    return f"{m.group(1)}<{', '.join(args)}>"


def _row(entry, wf, kernels, *, light="point", L=1, B=2, H=4, W=40, per_light=False, albedo_srgb=True, return_srgb=True,
         normal=True, grads=MAPS, layout="contig", project=True):
    """entry: "autograd" (CookTorranceBRDF forward + backward), "loss" (fused_loss_step), "fit" (fused_fit_step) or
    "convert" (DiffuseSpecularMaterial -> to_basecolor_metallic_material() -> render -> backward).
    grads: the map leaves (MAPS) and shared parameters (SHARED) whose gradients the call requests.  For "loss", any map
    requests every map gradient and "lights" / "view" request both (want_geometry_grad); "fit" updates every map.
    layout: "contig", "strided" (rows of a wider tensor, 16-byte aligned: still the 64-bit-access flavours), "misaligned"
    (first texel 4-byte aligned: the element-access flavours) or "bcast" (one (1, 3, H, W) metallic map for the batch)."""
    assert entry in ("autograd", "loss", "fit", "convert") and wf in WFS and set(grads) <= set(MAPS + SHARED)
    r = dict(entry=entry, wf=wf, kernels=tuple(kernels), light=light, L=L, B=B, H=H, W=W, per_light=per_light,
             albedo_srgb=albedo_srgb, return_srgb=return_srgb, normal=normal, grads=tuple(grads), layout=layout,
             project=project)
    r["id"] = "-".join(str(x) for x in (entry, wf, light, f"L{L}", f"B{B}", f"{H}x{W}", "per" if per_light else "acc", layout,
                                         "+".join(g[:3] for g in grads), "" if normal else "nonormal",
                                         "" if albedo_srgb else "linalb", "" if return_srgb else "linout",
                                         "" if project else "noproj") if x != "")
    return r


def _cases():
    rows = []
    for wf, c in WFS.items():
        # -- streamed kernels: one light, W % 4 == 0, at least 32 four-texel groups per row.  kFast: W % 512 == 0 (one
        #    128 x 1 block per tile row), a normal map, sRGB in and out, every map gradient; anything else: the general
        #    flavour.  Backward mode = loss bit | intensity-gradient bit: "autograd" gives 0 / 2, "loss" 1 / 3.
        for light, lc in (("point", HOIST), ("directional", DIR)):
            for mode in range(4):
                entry = "loss" if mode & 1 else "autograd"
                grads = MAPS + (("intensity",) if mode & 2 else ())
                for fast in (True, False):
                    kw = dict(light=light, B=2, H=3, W=512, grads=grads)
                    if not fast:   # a different reason for the general flavour in each mode
                        kw.update([dict(W=256), dict(normal=False), dict(albedo_srgb=False), dict(return_srgb=False)][mode])
                    ks = [bs(c, lc, mode, fast)] + ([fs(c, lc, fast)] if entry == "autograd" else [])
                    rows.append(_row(entry, wf, ks, **kw))
        # -- generic kernels, map gradients (autograd)
        rows += [
            _row("autograd", wf, [fk(c, DIR, 1), bk(c, DIR, 0, 1)], light="directional", L=2),
            _row("autograd", wf, [fk(c, DIR, 0), bk(c, DIR, 0, 0)], light="directional", W=41),          # odd W: element access
            _row("autograd", wf, [fk(c, PT, 1), bk(c, PT, 0, 1)], L=3, B=1, per_light=True),             # one material: per-texel geometry
            _row("autograd", wf, [fk(c, PT, 1, 1), bk(c, PT, 0, 1, 1)], L=3, B=1),                       # ... plain-case flavour
            _row("autograd", wf, [fk(c, PT, 0), bk(c, PT, 0, 0)], L=3, layout="misaligned"),
            _row("autograd", wf, [fk(c, HOIST, 1), bk(c, HOIST, 0, 1)], W=40),                          # < 32 groups: not streamed
            _row("autograd", wf, [fk(c, C8, 1), bk(c, C8, 0, 1)], L=2, per_light=True, layout="strided"),  # all-field cache, L <= 4
            _row("autograd", wf, [fk(c, C8, 1, 1), bk(c, C8, 0, 1, 1)], L=4, B=3),
            _row("autograd", wf, [fk(c, C6, 1), bk(c, C8BIG, 0, 1)], L=5, per_light=True),              # 4 < L <= 8: big backward cache
            _row("autograd", wf, [fk(c, C6, 1, 1), bk(c, C8BIG, 0, 1, 1)], L=8, layout="strided"),
            _row("autograd", wf, [fk(c, C6, 1), bk(c, C6, 0, 1)], L=9, per_light=True),                 # 6-field cache, L <= 16
            _row("autograd", wf, [fk(c, C6, 1, 1), bk(c, C6, 0, 1, 1)], L=16),
            # geometry gradients (kGeom): 6-field cache, per-texel, directional, and the element-access flavours
            _row("autograd", wf, [fk(c, C8, 1, 1), bk(c, C6, 1, 1)], L=3, grads=MAPS + ("lights", "view")),
            _row("autograd", wf, [fk(c, PT, 1), bk(c, PT, 1, 1)], L=2, B=1, per_light=True,
                 grads=("albedo", "roughness", "lights", "view")),
            _row("autograd", wf, [fk(c, DIR, 1), bk(c, DIR, 1, 1)], light="directional", L=2, grads=MAPS + SHARED),
            _row("autograd", wf, [fk(c, PT, 0), bk(c, PT, 1, 0)], L=2, W=41, grads=MAPS + ("lights", "view")),
            _row("autograd", wf, [fk(c, DIR, 0), bk(c, DIR, 1, 0)], light="directional", W=41, grads=("lights", "view")),
        ]
        # -- accumulate mode, loss kernel and one-launch fit step: with L > 1 no forward output exists, so the backward
        #    runs two passes with is_loss set (and the Adam epilogue for the fit step, which never takes the big cache)
        for L, lc_loss, lc_fit in ((1, HOIST, HOIST), (2, C8, C8), (6, C8BIG, C6), (12, C6, C6), (20, PT, PT)):
            want_int = ("intensity",) if L in (6, 20) else ()
            rows.append(_row("loss", wf, [bk(c, lc_loss, 0, 1)], L=L, grads=MAPS + want_int))
            rows.append(_row("fit", wf, [bk(c, lc_fit, 0, 1)], L=L, grads=MAPS + (("intensity",) if L == 12 else ())))
    rows += [
        # -- the one-launch fit step off its benchmarked shape
        _row("fit", "metallic", [bk(0, C8, 0, 1)], L=3, B=17, per_light=True),        # two 16-material walks of a CTA
        _row("fit", "specular", [bk(1, C8, 0, 1)], L=3, B=17, per_light=True),
        _row("fit", "metallic", [bk(0, PT, 0, 0)], L=2, W=41, per_light=True),        # odd W: element access
        _row("fit", "metallic3", [bk(2, PT, 0, 0)], L=2, W=41, per_light=True),
        _row("fit", "metallic", [bk(0, DIR, 0, 1)], light="directional", L=2, per_light=True),
        _row("fit", "specular", [bk(1, DIR, 0, 0)], light="directional", W=41),
        _row("fit", "metallic", [bk(0, PT, 0, 1)], L=3, B=1, per_light=True),
        _row("fit", "metallic3", [bk(2, PT, 0, 1)], L=3, B=1, per_light=True),
        _row("fit", "metallic3", [bk(2, C8, 0, 1)], L=3, per_light=True),
        _row("fit", "metallic3", [bk(2, C8, 0, 1)], L=3, per_light=True, project=False),
        _row("fit", "metallic3", [bk(2, C6, 0, 1)], L=7, per_light=True, normal=False, project=False),
        # -- 3-channel metallic: one map for the whole batch (its gradient is the sum over the batch), some gradients only
        _row("autograd", "metallic3", [fk(2, C8, 1, 1), bk(2, C8, 0, 1, 1)], L=3, B=3, layout="bcast"),
        _row("autograd", "metallic3", [fs(2, HOIST, 1), bs(2, HOIST, 0, 0)], B=2, H=3, W=512, grads=("albedo", "metspec")),
        _row("autograd", "metallic3", [fk(2, C8, 1, 1), bk(2, C8, 0, 1)], L=3, grads=("normal", "metspec")),
        _row("loss", "metallic3", [bs(2, HOIST, 3, 0)], B=3, H=3, W=256, grads=("intensity",)),   # no map gradient at all
        # -- the user's path to a 3-channel metallic map: the converted material is linear (albedo_is_srgb=False), so the
        #    general streamed flavour
        _row("convert", "metallic3", [fs(2, HOIST, 0), bs(2, HOIST, 0, 0)], B=None, H=3, W=512),
    ]
    # -- both sides of each reduction boundary of the shared-parameter gradients.  launch_bwd gives every thread its own
    #    shared-memory slots (part_on) when the slots take <= 48 KB and slots + geometry cache + Adam staging fit in
    #    kMaxDynSmem = 100 KB + 30 KB = 133 120 B; otherwise each light goes through a warp shuffle and shared atomics
    #    (CtaGeomSink::add, int_sink).  128 threads a CTA; slots: 6 floats a light with d_lights / d_view (3 072 B),
    #    3 without (1 536 B); 6-field geometry cache: 6 x 8 B x 128 = 6 144 B a light; Adam staging 30 720 B.
    #  d_lights / d_view on the 6-field cache (B >= 2): 6 144 L + 3 072 L <= 133 120  <=>  L <= 14; L = 15, 16 shuffle
    for L in (14, 15, 16):
        rows.append(_row("autograd", "metallic3", [fk(2, C6, 1, 1), bk(2, C6, 1, 1)], L=L, grads=MAPS + SHARED))
    #  d_lights / d_view on per-texel geometry (B = 1): 3 072 L <= 49 152  <=>  L <= 16; L = 17 .. 64 shuffle
    for L in (16, 17, 64):
        rows.append(_row("autograd", "metallic", [fk(0, PT, 1, 1), bk(0, PT, 1, 1)], L=L, B=1, grads=MAPS + SHARED))
    rows.append(_row("loss", "specular", [bk(1, PT, 1, 1)], L=17, B=1, per_light=True, grads=MAPS + SHARED))
    #  d_intensity alone, per-texel geometry: 1 536 L <= 49 152  <=>  L <= 32; L = 33 .. 64 shuffle
    for L in (32, 33, 64):
        rows.append(_row("autograd", "specular", [fk(1, PT, 1, 1), bk(1, PT, 0, 1)], L=L, B=1, grads=MAPS + ("intensity",)))
    #  fit step with want_intensity_grad on the 6-field cache: 30 720 + 6 144 L + 1 536 L <= 133 120  <=>  L <= 13; 14 .. 16 shuffle
    for L in (13, 14, 16):
        rows.append(_row("fit", "metallic3", [bk(2, C6, 0, 1)], L=L, per_light=True, grads=MAPS + ("intensity",)))
    return rows


CASES = _cases()


# ---------------------------------------------------------------------------------------------- the ledger (CPU)
def compiled_kernels():
    """The Cook-Torrance kernel instantiations defined in the built library."""
    assert os.path.exists(LIB), f"{LIB} is not built"
    out = subprocess.run(["nm", "-C", "--defined-only", LIB], check=True, capture_output=True, text=True).stdout
    return {norm_kernel(m.group(0)) for m in re.finditer(r"pbr::ct_(?:forward|backward)_(?:kernel|stream)<[^<>]*>", out)}


def test_every_compiled_kernel_has_a_row():
    compiled = compiled_kernels()
    named = {k for r in CASES for k in r["kernels"]}
    assert not compiled - named, f"instantiations without a parity row: {sorted(compiled - named)}"
    assert not named - compiled, f"rows name kernels the library does not contain: {sorted(named - compiled)}"
    ids = [r["id"] for r in CASES]
    assert len(ids) == len(set(ids))
    print(f"{len(compiled)} of {len(compiled)} Cook-Torrance instantiations covered by {len(CASES)} rows")


def test_kernel_names_normalise_from_every_spelling():
    want = "ct_backward_kernel<0, 3, 0, 1, 1>"
    assert norm_kernel("void pbr::ct_backward_kernel<0, 3, false, true, 1>(pbr::CtKParams)") == want
    assert norm_kernel("ct_backward_kernel<0, 3, 0, 1, 1>") == want
    assert norm_kernel("pbr::ct_backward_kernel<0,3,false,true,1>") == want
    assert norm_kernel("void pbr::convert_kernel<true>(pbr::ConvKParams)") is None


# ---------------------------------------------------------------------------------------------- parity rows (GPU)
def _random_case(seed, B, H, W, L, workflow="metallic", rough_lo=0.2, normal=True):
    g = torch.Generator().manual_seed(seed)
    shp = lambda c: (B, c, H, W)
    maps = {"albedo": torch.rand(shp(3), generator=g), "roughness": torch.rand(shp(1), generator=g) * (1 - rough_lo) + rough_lo}
    if normal:
        n = torch.randn(shp(3), generator=g)
        maps["normal"] = torch.nn.functional.normalize(n * torch.tensor([0.3, 0.3, 0.0]).view(1, 3, 1, 1)
                                                       + torch.tensor([0.0, 0.0, 1.0]).view(1, 3, 1, 1), dim=1)
    if workflow == "specular":
        maps["specular"] = torch.rand(shp(3), generator=g)
    else:
        maps["metallic"] = torch.rand(shp(3 if workflow == "metallic3" else 1), generator=g)
    ang = torch.arange(L, dtype=torch.float32) * (6.2831853 / max(L, 1))
    lights = torch.stack([0.4 * torch.cos(ang), 0.4 * torch.sin(ang), torch.ones(L)], dim=1) if L > 1 else torch.tensor([0.1, 0.1, 1.0])
    # a different intensity per colour channel: a channel mix-up of d_intensity does not cancel
    inten = torch.tensor([1.0, 0.8, 0.6]).expand(L, 3) / L if L > 1 else torch.tensor([1.0, 0.8, 0.6])
    return maps, lights, inten.contiguous(), g


def _shared_tol(want):
    want = np.asarray(want, np.float64)
    return 1e-4 * np.abs(want) + 1e-4 * np.abs(want).mean()


def _launched(fn):
    """fn() under torch.profiler (CUDA activities) -> (its result, the Cook-Torrance kernels it launched)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, {k for k in (norm_kernel(e.name) for e in prof.events()) if k}


def _metspec_key(wf):
    return "specular" if wf == "specular" else "metallic"


def _device_material(r, maps):
    """The material of a row, its map leaves laid out as the row says."""
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
        elif r["layout"] in ("strided", "misaligned"):
            off = 4 if r["layout"] == "strided" else 1
            wide = torch.zeros(*t.shape[:-1], r["W"] + 8, device=DEV)
            wide[..., off:off + r["W"]] = t
            t = wide[..., off:off + r["W"]]
        t = t.detach().requires_grad_(("metspec" if k in ("metallic", "specular") else k) in want)
        leaves[k] = t
        m._maps[k] = t
    if "normal" not in maps:
        m._maps["normal"] = None
    return m, leaves


def _check_shared(got, want, key):
    got, want = np.asarray(got, np.float64).reshape(-1), np.asarray(want, np.float64).reshape(-1)
    assert np.all(np.abs(got - want) <= _shared_tol(want)), (key, float((np.abs(got - want) / _shared_tol(want)).max()), got, want)


def _run_convert(r, seed):
    """DiffuseSpecularMaterial -> to_basecolor_metallic_material() -> CookTorranceBRDF -> backward to the specular-workflow
    leaves, against O.specular_to_metallic + O.render under autograd.  The specular map lies strictly between 0.04 and the
    linear diffuse (0.2 .. 1), so the conversion divides by at least ~0.16 and its metallic stays inside (0, 0.9): no
    texel sits where one ulp of the sRGB decode is amplified (conftest.s2m_ok is the rule there, test_gpu_autograd)."""
    from oracle import pbr_oracle as O
    from pypbr_b200.materials import DiffuseSpecularMaterial
    from pypbr_b200.models import CookTorranceBRDF

    g = torch.Generator().manual_seed(seed)
    H, W = r["H"], r["W"]
    albedo = 0.5 + 0.5 * torch.rand(3, H, W, generator=g)
    d = O.srgb_to_linear(albedo)
    specular = 0.04 + (0.05 + 0.8 * torch.rand(3, H, W, generator=g)) * (d - 0.04)
    maps, lights, inten, _ = _random_case(seed, 1, H, W, 1)
    maps = dict(albedo=albedo, specular=specular, roughness=maps["roughness"][0], normal=maps["normal"][0])
    view = torch.tensor([0.04, -0.07, 1.0])
    ref = {k: v.clone().requires_grad_(True) for k, v in maps.items()}
    b, m = O.specular_to_metallic(ref["albedo"], ref["specular"], True)
    out_ref = O.render(dict(albedo=b, metallic=m, normal=ref["normal"], roughness=ref["roughness"]), view, lights, inten, 1.0,
                       "point", albedo_is_srgb=False)
    go = torch.rand(out_ref.shape, generator=g)
    out_ref.backward(go)

    lv = {k: v.to(DEV).requires_grad_(True) for k, v in maps.items()}
    mat = DiffuseSpecularMaterial(albedo_is_srgb=True, device=DEV)
    mat._maps.update(lv)

    def call():
        conv = mat.to_basecolor_metallic_material()
        assert conv.metallic.shape == (3, H, W)
        out = CookTorranceBRDF("point")(conv, view, lights, inten, 1.0)
        out.backward(go.to(DEV))
        return out

    out, launched = _launched(call)
    ratio, ok = fwd_ok(out.detach().cpu().numpy(), out_ref.detach().numpy())
    assert ok, f"forward {ratio}"
    for k in maps:
        ratio, ok = grad_ok(lv[k].grad.cpu().numpy(), ref[k].grad.numpy())
        assert ok, f"d_{k} {ratio}"
    return launched


@pytest.mark.gpu
@pytest.mark.parametrize("r", CASES, ids=[r["id"] for r in CASES])
def test_kernel_against_oracle(r):
    from oracle import pbr_oracle as O
    from pypbr_b200.fit import FusedAdam, fused_fit_step, fused_loss_step
    from pypbr_b200.models import CookTorranceBRDF

    seed = 7000 + CASES.index(r)
    if r["entry"] == "convert":
        launched = _run_convert(r, seed)
        assert launched == set(r["kernels"]), f"launched {sorted(launched)}, row names {sorted(r['kernels'])}"
        return
    B, H, W, L, wf = r["B"], r["H"], r["W"], r["L"], r["wf"]
    maps, lights, inten, g = _random_case(seed, B, H, W, L, wf, normal=r["normal"])
    light_type = r["light"]
    if light_type == "directional":
        lights = torch.nn.functional.normalize(lights + torch.tensor([0.0, 0.0, 1.0]), dim=-1)
    if r["layout"] == "bcast":   # one metallic map shared by the batch: the same values for every material
        maps["metallic"] = maps["metallic"][:1].expand_as(maps["metallic"]).clone()
    view = torch.tensor([0.04, -0.07, 1.0])
    size = 1.0 if light_type == "point" else None
    flags = dict(albedo_is_srgb=r["albedo_srgb"], specular_is_srgb=True, return_srgb=r["return_srgb"])
    acc = not r["per_light"]
    mkey = _metspec_key(wf)
    name = lambda k: "metspec" if k == mkey else k
    entry, grads = r["entry"], set(r["grads"])
    want_maps = {k for k in maps if name(k) in grads} if entry == "autograd" else (set(maps) if (entry == "fit" or grads & set(MAPS)) else set())
    want_shared = grads & set(SHARED)
    if entry == "loss" and want_shared & {"lights", "view"}:
        want_shared |= {"lights", "view"}

    # the oracle: fp32 for the image, the loss and the map gradients; fp64 for the shared parameters (sums over the image)
    leaves_ref = {k: v.clone().requires_grad_(k in want_maps) for k, v in maps.items()}
    ref = O.render(leaves_ref, view, lights, inten, size, light_type, accumulate=acc, **flags)
    go = torch.rand(ref.shape, generator=g)   # grad_out, or the target of the loss
    if entry == "autograd":
        if want_maps:
            ref.backward(go)
    else:
        loss_ref = ((ref - go) ** 2).mean()
        if want_maps:
            loss_ref.backward()
    shared64 = {}
    if want_shared:
        sh = {k: t.double().clone().requires_grad_(k in want_shared) for k, t in zip(SHARED, (inten, lights, view))}
        ref64 = O.render({k: t.double() for k, t in maps.items()}, sh["view"], sh["lights"], sh["intensity"], size, light_type,
                         accumulate=acc, **flags)
        (ref64.backward(go.double()) if entry == "autograd" else ((ref64 - go.double()) ** 2).mean().backward())
        shared64 = {k: sh[k].grad.numpy() for k in want_shared}

    mat, leaves = _device_material(r, maps)
    multi = "per_light" if r["per_light"] else "accumulate"
    if entry == "autograd":
        sh_dev = {k: t.clone().requires_grad_(k in want_shared) for k, t in zip(SHARED, (inten, lights, view))}

        def call():
            out = CookTorranceBRDF(light_type, multi_light=multi)(mat, sh_dev["view"], sh_dev["lights"], sh_dev["intensity"], size,
                                                                   r["return_srgb"])
            out.backward(go.to(DEV))
            return out

        out, launched = _launched(call)
        assert out.shape == ref.shape
        ratio, ok = fwd_ok(out.detach().cpu().numpy(), ref.detach().numpy())
        assert ok, f"forward {ratio}"
        for k in maps:
            if k not in want_maps:
                assert leaves[k].grad is None, k
                continue
            exp = leaves_ref[k].grad
            if r["layout"] == "bcast" and k == "metallic":
                exp = exp.sum(0, keepdim=True)   # the shared map collects every material's gradient
            ratio, ok = grad_ok(leaves[k].grad.cpu().numpy(), exp.numpy())
            assert ok, f"d_{k} {ratio}"
        for k in want_shared:
            _check_shared(sh_dev[k].grad.numpy(), shared64[k], k)
    elif entry == "loss":
        def call():
            return fused_loss_step(mat, go.to(DEV), view, lights, inten, light_type, size, r["return_srgb"], multi,
                                   want_intensity_grad="intensity" in want_shared,
                                   want_geometry_grad=bool(want_shared & {"lights", "view"}), want_map_grads=bool(want_maps))

        (buf, dgrads), launched = _launched(call)
        buf = buf.cpu().numpy().astype(np.float64)
        lr = float(loss_ref.detach())
        assert abs(buf[0] / go.numel() - lr) <= 2e-6 * lr, (buf[0] / go.numel(), lr)
        for k in maps:
            if k in want_maps:
                ratio, ok = grad_ok(dgrads[k].cpu().numpy(), leaves_ref[k].grad.numpy())
                assert ok, f"d_{k} {ratio}"
            else:
                assert dgrads.get(k) is None, k
        if "intensity" in want_shared:
            _check_shared(buf[1:1 + 3 * L], shared64["intensity"], "intensity")
        if "lights" in want_shared:
            _check_shared(buf[1 + 3 * L:1 + 6 * L], shared64["lights"], "lights")
            _check_shared(buf[1 + 6 * L:], shared64["view"], "view")
    else:
        opt = FusedAdam({k: mat._maps[k] for k in maps}, lr=0.01, project=None if r["project"] else {k: None for k in maps})

        def call():
            return fused_fit_step(mat, opt, go.to(DEV), view, lights, inten, light_type, size, r["return_srgb"], multi,
                                  want_intensity_grad="intensity" in want_shared)

        buf, launched = _launched(call)
        buf = buf.cpu().numpy().astype(np.float64)
        lr = float(loss_ref.detach())
        assert abs(buf[0] / go.numel() - lr) <= 2e-6 * lr, (buf[0] / go.numel(), lr)
        want = O.adam_fit_steps(maps, [{k: leaves_ref[k].grad for k in maps}], lr=0.01,
                                projection=None if r["project"] else {k: None for k in maps})
        for k in maps:
            a, b = mat._maps[k].cpu(), want[k]
            # an Adam step is lr-sized whatever the gradient: where |g| is at noise level its sign is not defined to 1e-4
            big = leaves_ref[k].grad.abs() > 1e-3 * leaves_ref[k].grad.abs().mean()
            assert bool(((a - b).abs()[big] <= 2e-5 * b.abs()[big] + 2e-6).all()), (k, float((a - b).abs()[big].max()))
        if "intensity" in want_shared:
            _check_shared(buf[1:1 + 3 * L], shared64["intensity"], "intensity")
    assert launched == set(r["kernels"]), f"launched {sorted(launched)}, row names {sorted(r['kernels'])}"
