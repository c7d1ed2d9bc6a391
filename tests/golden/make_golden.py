"""
tests/golden/make_golden.py — generates the golden fixtures in this directory.

Run ONLY in the build container, where the reference lives at /root/reference:
    python tests/golden/make_golden.py
It imports the UNMODIFIED reference (copied to a temp dir only to add the git-ignored
`_version.py` stub that `pypbr/__init__.py:22` needs), executes it in fp32 (the parity target) and
fp64 (the arbiter; maps injected through `_maps`, which bypasses the FloatTensor gate of
`materials/base.py:96-101`), asserts that oracle/pbr_oracle.py is BIT-IDENTICAL to the reference
on every case (outputs and autograd gradients), and writes one .npz per case.

Nothing at test / bench / smoke time reads /root/reference; they replay these files.
"""

import json
import os
import shutil
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

REF_SRC = "/root/reference"


def import_reference():
    tmp = tempfile.mkdtemp(prefix="pypbr_ref_")
    shutil.copytree(os.path.join(REF_SRC, "pypbr"), os.path.join(tmp, "pypbr"))
    with open(os.path.join(tmp, "pypbr", "_version.py"), "w") as f:
        f.write('version = "0.1.0"\n')
    sys.path.insert(0, tmp)
    import pypbr  # noqa: F401

    return tmp


import_reference()
from pypbr.blending.functional import blend_materials as ref_blend_materials  # noqa: E402
from pypbr.io import load_material_from_folder  # noqa: E402
from pypbr.materials import BasecolorMetallicMaterial, DiffuseSpecularMaterial  # noqa: E402
from pypbr.models import CookTorranceBRDF  # noqa: E402
from pypbr.utils import linear_to_srgb as ref_l2s  # noqa: E402

from oracle import pbr_oracle as O  # noqa: E402


def bits_equal(a, b):
    if a is None and b is None:
        return True
    a = a.detach().contiguous()
    b = b.detach().contiguous()
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    return bool(torch.all((a == b) | (torch.isnan(a) & torch.isnan(b))))


# ------------------------------------------------------------------------------------------
# input synthesis (SURVEY.md §8d)
# ------------------------------------------------------------------------------------------


def synth_maps(gen, H, W, workflow, normal="unit", rough_lo=0.2, B=None):
    shp = (lambda c: (c, H, W)) if B is None else (lambda c: (B, c, H, W))
    cdim = 0 if B is None else 1
    maps = {"albedo": torch.rand(shp(3), generator=gen)}
    if normal == "unit":
        n = torch.randn(shp(3), generator=gen)
        scale = torch.tensor([0.3, 0.3, 0.0]).view((3, 1, 1) if B is None else (1, 3, 1, 1))
        up = torch.tensor([0.0, 0.0, 1.0]).view((3, 1, 1) if B is None else (1, 3, 1, 1))
        maps["normal"] = torch.nn.functional.normalize(n * scale + up, dim=cdim)
    elif normal == "raw":  # tests/test_models.py:17,34: un-normalised, any sign
        maps["normal"] = torch.rand(shp(3), generator=gen) * 2 - 1
    maps["roughness"] = torch.rand(shp(1), generator=gen) * (1 - rough_lo) + rough_lo
    if workflow == "metallic":
        maps["metallic"] = torch.rand(shp(1), generator=gen)
    else:
        maps["specular"] = torch.rand(shp(3), generator=gen)
    return maps


def ref_material(maps, dtype, flags, requires_grad=False):
    cls = BasecolorMetallicMaterial if "metallic" in maps else DiffuseSpecularMaterial
    m = cls()
    m.albedo_is_srgb = flags.get("albedo_is_srgb", True)
    if cls is DiffuseSpecularMaterial:
        m.specular_is_srgb = flags.get("specular_is_srgb", True)
    leaves = {}
    for k, t in maps.items():
        leaf = t.to(dtype).clone().requires_grad_(requires_grad)
        leaves[k] = leaf
        m._maps[k] = leaf
    if "normal" not in maps:
        # `material.normal` raises AttributeError unless the key exists (base.py:105-120); the
        # default +Z branch of cooktorrance.py:143-151 is only reachable with an explicit None entry.
        m._maps["normal"] = None
    return m, leaves


def ref_render(maps, view, lights, intens, p, dtype, grad_out=None):
    """Loop of reference calls combined per the module docstring of oracle/pbr_oracle.py."""
    batched = maps["albedo"].dim() == 4
    multi = lights.dim() == 2
    B = maps["albedo"].shape[0] if batched else 1
    lts = lights if multi else lights.view(1, 3)
    ins = intens if intens.dim() == 2 else intens.view(1, 3).expand(lts.shape[0], 3)
    brdf = CookTorranceBRDF(light_type=p["light_type"])
    leaves_all, outs = [], []
    for b in range(B):
        mb = {k: (t[b] if batched else t) for k, t in maps.items()}
        mat, leaves = ref_material(mb, dtype, p, requires_grad=grad_out is not None)
        leaves_all.append(leaves)
        single = (not multi) and True
        if single:
            outs.append(brdf(mat, view.to(dtype), lts[0].to(dtype), ins[0].to(dtype), p["light_size"], p["return_srgb"]))
            continue
        per = [brdf(mat, view.to(dtype), lts[l].to(dtype), ins[l].to(dtype), p["light_size"], False) for l in range(lts.shape[0])]
        enc = ref_l2s if p["return_srgb"] else (lambda c: c)
        if p["accumulate"]:
            tot = per[0]
            for q in per[1:]:
                tot = tot + q
            outs.append(enc(torch.clamp(tot, 0.0, 1.0)))
        else:
            outs.append(torch.stack([enc(q) for q in per], dim=0))
    out = torch.stack(outs, dim=0) if batched else outs[0]
    grads = None
    if grad_out is not None:
        out.backward(grad_out.to(dtype))
        grads = {}
        for k in maps:
            gs = [lv[k].grad for lv in leaves_all]
            grads[k] = torch.stack(gs, dim=0) if batched else gs[0]
    return out.detach(), grads


def oracle_render(maps, view, lights, intens, p, dtype, grad_out=None):
    leaves = {k: t.to(dtype).clone().requires_grad_(grad_out is not None) for k, t in maps.items()}
    out = O.render(
        leaves, view.to(dtype), lights.to(dtype), intens.to(dtype), p["light_size"], p["light_type"],
        p.get("albedo_is_srgb", True), p.get("specular_is_srgb", True), p["return_srgb"], p["accumulate"],
    )
    grads = None
    if grad_out is not None:
        out.backward(grad_out.to(dtype))
        grads = {k: leaves[k].grad for k in maps}
    return out.detach(), grads


def ring_lights(L):
    if L == 1:
        return torch.tensor([0.1, 0.1, 1.0])
    ang = torch.arange(L, dtype=torch.float64) * (2 * np.pi / L)
    return torch.stack([0.4 * torch.cos(ang), 0.4 * torch.sin(ang), torch.ones(L, dtype=torch.float64)], dim=1).float()


CT_CASES = [
    # name, H, W, B, L, params
    dict(name="ct_metal_point_37x53", H=37, W=53, B=None, L=1, workflow="metallic", normal="unit", rough_lo=0.2,
         light_type="point", light_size=1.0, return_srgb=True, albedo_is_srgb=True, accumulate=True),
    dict(name="ct_metal_point_stress_40x64", H=40, W=64, B=None, L=1, workflow="metallic", normal="unit", rough_lo=0.0,
         light_type="point", light_size=1.0, return_srgb=True, albedo_is_srgb=True, accumulate=True),
    dict(name="ct_metal_dir_reftest_64x64", H=64, W=64, B=None, L=1, workflow="metallic", normal="raw", rough_lo=0.0,
         light_type="directional", light_size=None, return_srgb=True, albedo_is_srgb=True, accumulate=True,
         light=[0.0, 0.0, 1.0]),  # tests/test_models.py:12-27
    dict(name="ct_spec_point_reftest_64x64", H=64, W=64, B=None, L=1, workflow="specular", normal="raw", rough_lo=0.0,
         light_type="point", light_size=5.0, return_srgb=True, albedo_is_srgb=True, accumulate=True,
         light=[0.0, 10.0, 10.0]),  # tests/test_models.py:30-43
    dict(name="ct_spec_dir_linear_33x47", H=33, W=47, B=None, L=1, workflow="specular", normal="unit", rough_lo=0.2,
         light_type="directional", light_size=None, return_srgb=False, albedo_is_srgb=False, specular_is_srgb=False,
         accumulate=True, light=[0.3, -0.2, 0.9], intensity=[2.0, 1.5, 1.0], view=[0.1, 0.2, 1.0]),
    dict(name="ct_metal_nonormal_32x40", H=32, W=40, B=None, L=1, workflow="metallic", normal=None, rough_lo=0.2,
         light_type="point", light_size=None, return_srgb=True, albedo_is_srgb=True, accumulate=True,
         view=[0.2, -0.1, 1.0], intensity=[3.0, 2.5, 2.0]),
    dict(name="ct_metal_point_B3_L4_acc_24x36", H=24, W=36, B=3, L=4, workflow="metallic", normal="unit", rough_lo=0.2,
         light_type="point", light_size=1.0, return_srgb=True, albedo_is_srgb=True, accumulate=True),
    dict(name="ct_metal_point_B2_L3_per_24x36", H=24, W=36, B=2, L=3, workflow="metallic", normal="unit", rough_lo=0.2,
         light_type="point", light_size=1.0, return_srgb=True, albedo_is_srgb=True, accumulate=False),
    dict(name="ct_spec_point_B2_L2_acc_20x28", H=20, W=28, B=2, L=2, workflow="specular", normal="unit", rough_lo=0.2,
         light_type="point", light_size=2.0, return_srgb=True, albedo_is_srgb=True, specular_is_srgb=True, accumulate=True),
    dict(name="ct_metal_dir_B2_L3_acc_16x20", H=16, W=20, B=2, L=3, workflow="metallic", normal="unit", rough_lo=0.2,
         light_type="directional", light_size=None, return_srgb=True, albedo_is_srgb=True, accumulate=True),
]


def make_ct_case(idx, c):
    gen = torch.Generator().manual_seed(1000 + idx)
    maps = synth_maps(gen, c["H"], c["W"], c["workflow"], c["normal"], c["rough_lo"], c["B"])
    L = c["L"]
    lights = torch.tensor(c["light"]) if "light" in c else ring_lights(L)
    if L > 1:
        intens = torch.ones(L, 3) * (1.5 / L if c["accumulate"] else 1.0)
        intens = intens * torch.tensor([1.0, 0.9, 0.8])
    else:
        intens = torch.tensor(c.get("intensity", [1.0, 1.0, 1.0]))
    view = torch.tensor(c.get("view", [0.0, 0.0, 1.0]))
    p = {k: c.get(k) for k in ("light_type", "light_size", "return_srgb", "albedo_is_srgb", "specular_is_srgb", "accumulate")}
    p = {k: (True if (v is None and k.endswith("is_srgb")) else v) for k, v in p.items()}

    out32, _ = ref_render(maps, view, lights, intens, p, torch.float32)
    grad_out = torch.rand(out32.shape, generator=gen)
    out32, g32 = ref_render(maps, view, lights, intens, p, torch.float32, grad_out)
    out64, g64 = ref_render(maps, view, lights, intens, p, torch.float64, grad_out)
    o32, og32 = oracle_render(maps, view, lights, intens, p, torch.float32, grad_out)
    o64, og64 = oracle_render(maps, view, lights, intens, p, torch.float64, grad_out)
    assert bits_equal(o32, out32), f"{c['name']}: oracle fp32 forward differs from reference"
    assert bits_equal(o64, out64), f"{c['name']}: oracle fp64 forward differs from reference"
    for k in maps:
        assert bits_equal(og32[k], g32[k]), f"{c['name']}: oracle fp32 grad {k} differs"
        assert bits_equal(og64[k], g64[k]), f"{c['name']}: oracle fp64 grad {k} differs"

    arrs = {f"in_{k}": v.numpy() for k, v in maps.items()}
    arrs.update(view=view.numpy(), lights=lights.numpy(), intensity=intens.numpy(), grad_out=grad_out.numpy(),
                out32=out32.numpy(), out64=out64.numpy().astype(np.float64))
    for k in maps:
        arrs[f"g32_{k}"] = g32[k].numpy()
        arrs[f"g64_{k}"] = g64[k].numpy()
    arrs["params"] = np.array(json.dumps(p))
    np.savez_compressed(os.path.join(HERE, c["name"] + ".npz"), **arrs)
    e = (out32.double() - out64).abs() / out64.abs().clamp_min(1e-6)
    print(f"{c['name']}: ok  out mean {out32.mean():.6f}  ref32-vs-ref64 max rel {e.max():.2e}")


# ------------------------------------------------------------------------------------------
# workflow conversions, blends
# ------------------------------------------------------------------------------------------


def make_conversion_cases():
    gen = torch.Generator().manual_seed(77)
    H, W = 31, 45
    maps = synth_maps(gen, H, W, "metallic")
    arrs = {}
    for srgb in (True, False):
        m = BasecolorMetallicMaterial(albedo=maps["albedo"], normal=maps["normal"], roughness=maps["roughness"],
                                      metallic=maps["metallic"], albedo_is_srgb=srgb)
        d = m.to_diffuse_specular_material()
        od, os_ = O.metallic_to_specular(maps["albedo"], maps["metallic"], srgb)
        assert bits_equal(od, d.albedo) and bits_equal(os_, d.specular)
        assert d.normal is m.normal and d.roughness is m.roughness and d.specular_is_srgb is True and d.albedo_is_srgb is False
        arrs[f"m2s_diffuse_srgb{int(srgb)}"] = d.albedo.numpy()
        arrs[f"m2s_specular_srgb{int(srgb)}"] = d.specular.numpy()
    # edge values through the metallic→specular path
    smaps = synth_maps(gen, H, W, "specular")
    # push some texels to the branches of diffuse.py:134-145 (den < eps, m >= 0.95)
    smaps["albedo"][:, :4] = 0.04
    smaps["specular"][:, 4:8] = 0.99
    smaps["albedo"][:, 8:10] = 0.0
    for srgb in (True, False):
        m = DiffuseSpecularMaterial(albedo=smaps["albedo"], normal=smaps["normal"], roughness=smaps["roughness"],
                                    specular=smaps["specular"], albedo_is_srgb=srgb)
        bm = m.to_basecolor_metallic_material()
        ob, om = O.specular_to_metallic(smaps["albedo"], smaps["specular"], srgb)
        assert bits_equal(ob, bm.albedo) and bits_equal(om, bm.metallic)
        assert bm.metallic.shape[0] == 3
        arrs[f"s2m_basecolor_srgb{int(srgb)}"] = bm.albedo.numpy()
        arrs[f"s2m_metallic_srgb{int(srgb)}"] = bm.metallic.numpy()
        # fp64 arbiter: the division by (diffuse - 0.04) amplifies an ulp of the sRGB decode without bound near 0.04, so
        # parity there is stated against the reference's own distance from its fp64 evaluation (SURVEY.md 8c)
        m64 = DiffuseSpecularMaterial()
        m64.albedo_is_srgb = srgb
        for k in ("albedo", "normal", "roughness", "specular"):
            m64._maps[k] = smaps[k].double()
        bm64 = m64.to_basecolor_metallic_material()
        ob64, om64 = O.specular_to_metallic(smaps["albedo"].double(), smaps["specular"].double(), srgb)
        assert bits_equal(ob64, bm64.albedo) and bits_equal(om64, bm64.metallic)
        arrs[f"s2m_basecolor64_srgb{int(srgb)}"] = bm64.albedo.numpy()
        arrs[f"s2m_metallic64_srgb{int(srgb)}"] = bm64.metallic.numpy()
    arrs.update({f"in_m_{k}": v.numpy() for k, v in maps.items()})
    arrs.update({f"in_s_{k}": v.numpy() for k, v in smaps.items()})
    np.savez_compressed(os.path.join(HERE, "convert_31x45.npz"), **arrs)
    print("convert_31x45: ok")


def make_blend_cases():
    gen = torch.Generator().manual_seed(99)
    H, W = 29, 43
    m1 = synth_maps(gen, H, W, "metallic")
    m2 = synth_maps(gen, H, W, "metallic", normal="raw")
    m1["height"] = torch.rand(1, H, W, generator=gen)
    m2["height"] = torch.rand(1, H, W, generator=gen)
    m2["opacity"] = torch.rand(1, H, W, generator=gen)  # one-sided map: passed through by reference
    mask = torch.rand(1, H, W, generator=gen)
    mats = [BasecolorMetallicMaterial(albedo=m["albedo"], normal=m["normal"], roughness=m["roughness"],
                                      metallic=m["metallic"], **{k: m[k] for k in ("height", "opacity") if k in m})
            for m in (m1, m2)]
    arrs = {f"in1_{k}": v.numpy() for k, v in m1.items()}
    arrs.update({f"in2_{k}": v.numpy() for k, v in m2.items()})
    arrs["mask"] = mask.numpy()
    runs = {
        "mask": dict(method="mask", mask=mask),
        "mask2d": dict(method="mask", mask=mask[0]),
        "height": dict(method="height", blend_width=0.1),
        "height_w03": dict(method="height", blend_width=0.3),
        "prop_metallic": dict(method="properties", property_name="metallic", blend_width=0.1),
        "prop_roughness": dict(method="properties", property_name="roughness", blend_width=0.05),
        "grad_h": dict(method="gradient", direction="horizontal"),
        "grad_v": dict(method="gradient", direction="vertical"),
    }
    for tag, kw in runs.items():
        blended, used_mask = ref_blend_materials(mats[0], mats[1], **kw)
        # oracle: mask builders + map arithmetic + the setattr normal re-ingestion quirk
        if kw["method"] == "mask":
            om = kw["mask"]
        elif kw["method"] == "height":
            om = O.sigmoid_mask(m1["height"], m2["height"], kw["blend_width"])
        elif kw["method"] == "properties":
            om = O.property_mask(m1[kw["property_name"]], m2[kw["property_name"]], kw["blend_width"])
        else:
            om = O.gradient_mask(H, W, kw["direction"])
        ob = O.blend_maps(m1, m2, om)
        ob["normal"] = O.process_normal_map(ob["normal"])
        om3 = om.unsqueeze(0) if om.dim() == 2 else om
        assert bits_equal(om3, used_mask), tag
        for k, v in blended._maps.items():
            assert bits_equal(ob[k], v), (tag, k)
            arrs[f"{tag}_{k}"] = v.numpy()
        arrs[f"{tag}_mask"] = used_mask.numpy()
    np.savez_compressed(os.path.join(HERE, "blend_29x43.npz"), **arrs)
    print("blend_29x43: ok")


def make_config1_fixture():
    """BASELINE.json configs[0]: tiles fixture, metallic workflow, 256x256, example lighting."""
    mat = load_material_from_folder(os.path.join(REF_SRC, "tests", "data", "tiles"), preferred_workflow="metallic")
    mat.resize((256, 256))
    brdf = CookTorranceBRDF(light_type="point")
    view = torch.tensor([0.0, 0.0, 1.0])
    light = torch.tensor([0.1, 0.1, 1.0])
    inten = torch.tensor([1.0, 1.0, 1.0])
    out = brdf(mat, view, light, inten, 1.0)
    names = [k for k in ("albedo", "normal", "roughness", "metallic") if mat._maps.get(k) is not None]
    maps = {k: mat._maps[k] for k in names}
    p = dict(light_type="point", light_size=1.0, return_srgb=True, albedo_is_srgb=mat.albedo_is_srgb, accumulate=True)
    o32, _ = oracle_render(maps, view, light, inten, p, torch.float32)
    assert bits_equal(o32, out)
    arrs = {f"in_{k}": v.numpy() for k, v in maps.items()}
    arrs.update(view=view.numpy(), lights=light.numpy(), intensity=inten.numpy(), out32=out.numpy(),
                params=np.array(json.dumps(p)))
    # three files, none over 1 MB: the normal map and the output each in config1_tiles_256.<array>.npz
    split = ("in_normal", "out32")
    np.savez_compressed(os.path.join(HERE, "config1_tiles_256.npz"), **{k: v for k, v in arrs.items() if k not in split})
    for k in split:
        np.savez_compressed(os.path.join(HERE, f"config1_tiles_256.{k}.npz"), **{k: arrs[k]})
    print(f"config1_tiles_256: ok  mean {out.mean():.7f} min {out.min():.5f} max {out.max():.5f}")


def make_geomgrad_cases():
    """Gradients of the shared geometry parameters (view_dir, light position / direction) and of the intensity, from
    the reference's own autograd (cooktorrance.py:95,125-140), fp32 and fp64; the oracle must agree bit for bit."""
    arrs = {}
    cases = [dict(tag="point_metal", workflow="metallic", light_type="point", light_size=1.0, H=24, W=36,
                  view=[0.15, -0.1, 0.9], light=[0.3, 0.2, 0.8], intensity=[1.2, 1.0, 0.8]),
             dict(tag="dir_spec", workflow="specular", light_type="directional", light_size=None, H=20, W=28,
                  view=[-0.2, 0.1, 1.0], light=[0.3, -0.2, 0.9], intensity=[2.0, 1.5, 1.0])]
    for ci, c in enumerate(cases):
        gen = torch.Generator().manual_seed(4000 + ci)
        maps = synth_maps(gen, c["H"], c["W"], c["workflow"])
        grad_out = torch.rand(3, c["H"], c["W"], generator=gen)
        p = dict(light_type=c["light_type"], light_size=c["light_size"], return_srgb=True, albedo_is_srgb=True,
                 specular_is_srgb=True, accumulate=True)
        for dtype, tag in ((torch.float32, "32"), (torch.float64, "64")):
            shared = [torch.tensor(c[k], dtype=dtype, requires_grad=True) for k in ("view", "light", "intensity")]
            mat, _ = ref_material(maps, dtype, p)
            out = CookTorranceBRDF(light_type=c["light_type"])(mat, shared[0], shared[1], shared[2], c["light_size"], True)
            out.backward(grad_out.to(dtype))
            oshared = [torch.tensor(c[k], dtype=dtype, requires_grad=True) for k in ("view", "light", "intensity")]
            oout = O.render({k: t.to(dtype) for k, t in maps.items()}, oshared[0], oshared[1], oshared[2], c["light_size"],
                            c["light_type"], True, True, True, True)
            oout.backward(grad_out.to(dtype))
            assert bits_equal(oout, out), f"geomgrad {c['tag']}: oracle forward differs ({tag})"
            for a, b, nm in zip(shared, oshared, ("view", "light", "intensity")):
                assert bits_equal(a.grad, b.grad), f"geomgrad {c['tag']}: oracle d_{nm} differs ({tag})"
                arrs[f"{c['tag']}_g{tag}_{nm}"] = a.grad.numpy()
        for k, v in maps.items():
            arrs[f"{c['tag']}_in_{k}"] = v.numpy()
        arrs[f"{c['tag']}_grad_out"] = grad_out.numpy()
        arrs[f"{c['tag']}_params"] = np.array(json.dumps({**p, **{k: c[k] for k in ("view", "light", "intensity", "workflow")}}))
        print(f"geomgrad {c['tag']}: ok  d_view64 {arrs[c['tag'] + '_g64_view']}  d_light64 {arrs[c['tag'] + '_g64_light']}")
    np.savez_compressed(os.path.join(HERE, "geomgrad_shared_params.npz"), **arrs)


def make_autograd_cases():
    """
    Autograd THROUGH the conversions, blends, normal ingestion and index transforms, from the reference's own torch graph
    (metallic.py:103-109, diffuse.py:129-147, blending/functional.py:104-145,187-194, materials/base.py:215-242,521-537,
    605-655), fp32 and fp64; the oracle's restatement must agree bit for bit.  Written to autograd_convert_blend.npz.
    """
    gen = torch.Generator().manual_seed(2025)
    H, W = 23, 38
    arrs = {}

    def leafs(d, dtype):
        return {k: v.to(dtype).clone().requires_grad_(True) for k, v in d.items()}

    def put(cls, leaves, **flags):
        m = cls()
        for k, v in flags.items():
            setattr(m, k, v)
        for k, v in leaves.items():
            m._maps[k] = v   # (bypasses the FloatTensor gate: fp64 and requires_grad leaves, as for the shading cases)
        for k in ("normal", "roughness"):
            m._maps.setdefault(k, None)   # the conversions read both attributes (metallic.py:115-116)
        return m

    # ---- conversions
    mm = synth_maps(gen, H, W, "metallic")
    sm = synth_maps(gen, H, W, "specular")
    sm["albedo"][:, :3] = 0.04
    sm["specular"][:, 3:6] = 0.99
    sm["albedo"][:, 6:8] = 0.0
    g0, g1 = torch.randn(3, H, W, generator=gen), torch.randn(3, H, W, generator=gen)
    arrs.update({f"m2s_in_{k}": mm[k].numpy() for k in ("albedo", "metallic")})
    arrs.update({f"s2m_in_{k}": sm[k].numpy() for k in ("albedo", "specular")})
    arrs.update(conv_g0=g0.numpy(), conv_g1=g1.numpy())
    for srgb in (True, False):
        for dtype, tag in ((torch.float32, "32"), (torch.float64, "64")):
            lv = leafs({k: mm[k] for k in ("albedo", "metallic")}, dtype)
            d = put(BasecolorMetallicMaterial, lv, albedo_is_srgb=srgb).to_diffuse_specular_material()
            ((d.albedo * g0.to(dtype)).sum() + (d.specular * g1.to(dtype)).sum()).backward()
            ol = leafs({k: mm[k] for k in ("albedo", "metallic")}, dtype)
            od, os_ = O.metallic_to_specular(ol["albedo"], ol["metallic"], srgb)
            ((od * g0.to(dtype)).sum() + (os_ * g1.to(dtype)).sum()).backward()
            for k in lv:
                assert bits_equal(lv[k].grad, ol[k].grad), ("m2s", k, srgb, tag)
                arrs[f"m2s_srgb{int(srgb)}_g{tag}_{k}"] = lv[k].grad.numpy()
            lv = leafs({k: sm[k] for k in ("albedo", "specular")}, dtype)
            b = put(DiffuseSpecularMaterial, lv, albedo_is_srgb=srgb).to_basecolor_metallic_material()
            ((b.albedo * g0.to(dtype)).sum() + (b.metallic * g1.to(dtype)).sum()).backward()
            ol = leafs({k: sm[k] for k in ("albedo", "specular")}, dtype)
            ob, om = O.specular_to_metallic(ol["albedo"], ol["specular"], srgb)
            ((ob * g0.to(dtype)).sum() + (om * g1.to(dtype)).sum()).backward()
            for k in lv:
                assert bits_equal(lv[k].grad, ol[k].grad), ("s2m", k, srgb, tag)
                arrs[f"s2m_srgb{int(srgb)}_g{tag}_{k}"] = lv[k].grad.numpy()

    # ---- blends (mask given / height sigmoid), every map a leaf
    m1 = synth_maps(gen, H, W, "metallic")
    m2 = synth_maps(gen, H, W, "metallic", normal="raw")
    m1["height"] = torch.rand(1, H, W, generator=gen)
    m2["height"] = torch.rand(1, H, W, generator=gen)
    mask = torch.rand(1, H, W, generator=gen)
    names = ("albedo", "normal", "roughness", "metallic", "height")
    gout = {k: torch.randn(m1[k].shape, generator=gen) for k in names}
    gmask = torch.randn(1, H, W, generator=gen)
    arrs.update({f"blend_in1_{k}": m1[k].numpy() for k in names})
    arrs.update({f"blend_in2_{k}": m2[k].numpy() for k in names})
    arrs["blend_mask"] = mask.numpy()
    arrs.update({f"blend_gout_{k}": v.numpy() for k, v in gout.items()})
    arrs["blend_gmask"] = gmask.numpy()
    for mode in ("mask", "height"):
        for dtype, tag in ((torch.float32, "32"), (torch.float64, "64")):
            l1, l2 = leafs(m1, dtype), leafs(m2, dtype)
            mk = mask.to(dtype).clone().requires_grad_(True)
            a, b = put(BasecolorMetallicMaterial, l1), put(BasecolorMetallicMaterial, l2)
            kw = dict(method="mask", mask=mk) if mode == "mask" else dict(method="height", blend_width=0.15)
            blended, used = ref_blend_materials(a, b, **kw)
            # (fp64 maps fail the FloatTensor gate of base.py:96-101 and land as plain attributes: getattr finds both)
            assert float(getattr(blended, "normal").detach().min()) < 0   # the setattr re-ingestion keeps the blended normal as it is
            loss = sum((getattr(blended, k) * gout[k].to(dtype)).sum() for k in names)
            if mode == "height":
                loss = loss + (used * gmask.to(dtype)).sum()
            loss.backward()
            o1, o2 = leafs(m1, dtype), leafs(m2, dtype)
            omk = mask.to(dtype).clone().requires_grad_(True)
            om = omk if mode == "mask" else O.sigmoid_mask(o1["height"], o2["height"], 0.15)
            ob = O.blend_maps(o1, o2, om)
            oloss = sum((ob[k] * gout[k].to(dtype)).sum() for k in names)
            if mode == "height":
                oloss = oloss + (om * gmask.to(dtype)).sum()
            oloss.backward()
            for k in names:
                if mode == "height" and k == "height":   # sums over the maps again (through the sigmoid): order, see below
                    assert torch.allclose(l1[k].grad, o1[k].grad, rtol=1e-5, atol=1e-6) and torch.allclose(l2[k].grad, o2[k].grad, rtol=1e-5, atol=1e-6)
                else:
                    assert bits_equal(l1[k].grad, o1[k].grad) and bits_equal(l2[k].grad, o2[k].grad), (mode, k, tag)
                arrs[f"blend_{mode}_g{tag}_in1_{k}"] = l1[k].grad.numpy()
                arrs[f"blend_{mode}_g{tag}_in2_{k}"] = l2[k].grad.numpy()
            if mode == "mask":
                # the mask gradient is a sum over the maps, accumulated by autograd in graph order: the reference walks a
                # Python set of names (functional.py:92), the oracle a sorted list - same terms, another order
                assert torch.allclose(mk.grad, omk.grad, rtol=1e-5, atol=1e-6)
                arrs[f"blend_mask_g{tag}_mask"] = mk.grad.numpy()

    # ---- normal ingestion: 3-channel RGB-encoded and 2-channel maps (base.py:215-217, :235-242)
    rgb = torch.rand(3, H, W, generator=gen)
    two = torch.rand(2, H, W, generator=gen)
    gn = torch.randn(3, H, W, generator=gen)
    arrs.update(ingest_in3=rgb.numpy(), ingest_in2=two.numpy(), ingest_gout=gn.numpy())
    from pypbr.materials import MaterialBase as RefBase

    for dtype, tag in ((torch.float32, "32"), (torch.float64, "64")):
        for key, src in (("3", rgb), ("2", two)):
            leaf = src.to(dtype).clone().requires_grad_(True)
            out = RefBase()._process_normal_map(leaf)
            (out * gn.to(dtype)).sum().backward()
            ol = src.to(dtype).clone().requires_grad_(True)
            (O.process_normal_map(ol) * gn.to(dtype)).sum().backward()
            assert bits_equal(leaf.grad, ol.grad), ("ingest", key, tag)
            arrs[f"ingest{key}_g{tag}"] = leaf.grad.numpy()

    # ---- index transforms: flip / roll / tile of a material whose maps are leaves
    tm = {"albedo": torch.rand(3, 10, 14, generator=gen), "normal": torch.randn(3, 10, 14, generator=gen)}
    arrs.update({f"index_in_{k}": v.numpy() for k, v in tm.items()})
    ops = {"flip_h": lambda m: m.flip_horizontal(), "flip_v": lambda m: m.flip_vertical(), "roll": lambda m: m.roll((3, -5)),
           "tile": lambda m: m.tile(3)}
    for op, fn in ops.items():
        lv = leafs(tm, torch.float32)
        m = fn(put(BasecolorMetallicMaterial, lv))
        gs = {k: torch.randn(m._maps[k].shape, generator=gen) for k in tm}
        sum((m._maps[k] * gs[k]).sum() for k in tm).backward()
        for k in tm:
            arrs[f"index_{op}_gout_{k}"] = gs[k].numpy()
            arrs[f"index_{op}_g32_{k}"] = lv[k].grad.numpy()
    np.savez_compressed(os.path.join(HERE, "autograd_convert_blend.npz"), **arrs)
    print("autograd_convert_blend: ok")



def make_height_from_normal_fixture():
    """compute_height_from_normal / compute_normal_from_height of the reference itself (utils/functions.py:123-323)."""
    from pypbr.utils import NormalConvention as RefConv
    from pypbr.utils import compute_height_from_normal as ref_h_from_n
    from pypbr.utils import compute_normal_from_height as ref_n_from_h

    gen = torch.Generator().manual_seed(606)
    H, W = 48, 72
    yy, xx = torch.meshgrid(torch.linspace(0, 3.0, H), torch.linspace(0, 5.0, W), indexing="ij")
    height = 0.5 + 0.25 * torch.sin(2.1 * xx) * torch.cos(1.3 * yy) + 0.05 * torch.rand(H, W, generator=gen)
    height = height.unsqueeze(0)
    arrs = {"height": height.numpy()}
    for conv, tag in ((RefConv.OPENGL, "gl"), (RefConv.DIRECTX, "dx")):
        n = ref_n_from_h(height, 4.0, conv)
        arrs[f"normal_{tag}"] = n.numpy()
        arrs[f"height_back_{tag}"] = ref_h_from_n(n.clone(), 1.0, conv).numpy()
    np.savez_compressed(os.path.join(HERE, "height_normal_48x72.npz"), **arrs)
    print("height_normal_48x72: ok")


def make_normal_ops_autograd_fixture():
    """The reference's own autograd through rotate_normals (utils/functions.py:69-108; in place, hence run on a non-leaf),
    MaterialBase.adjust_normal_strength (materials/base.py:689-706; in place as well) and compute_height_from_normal
    (utils/functions.py:180-323), fp32 (the target) and fp64 (the arbiter)."""
    from pypbr.utils import NormalConvention as RefConv
    from pypbr.utils import compute_height_from_normal as ref_h_from_n
    from pypbr.utils import rotate_normals as ref_rotate

    gen = torch.Generator().manual_seed(707)
    H, W = 20, 28
    up = torch.tensor([0.0, 0.0, 1.0]).view(3, 1, 1)
    n0 = torch.nn.functional.normalize(torch.randn(3, H, W, generator=gen) * 0.45 + up, dim=0)
    w3 = torch.rand(3, H, W, generator=gen)
    w1 = torch.rand(1, H, W, generator=gen)
    arrs = {"normal": n0.numpy(), "w3": w3.numpy(), "w1": w1.numpy(), "angle": np.float32(37.0), "strength": np.float32(2.5),
            "scale": np.float32(1.5)}
    for dtype, tag in ((torch.float32, "32"), (torch.float64, "64")):
        x = n0.detach().to(dtype).clone().requires_grad_(True)
        y = ref_rotate(x * 1.0, 37.0)
        (y * w3.to(dtype)).sum().backward()
        arrs[f"rot_out{tag}"], arrs[f"rot_g{tag}"] = y.detach().numpy(), x.grad.numpy()

        x = n0.detach().to(dtype).clone().requires_grad_(True)
        m = BasecolorMetallicMaterial()
        m._maps["normal"] = x * 1.0
        m.adjust_normal_strength(2.5)
        y = m._maps["normal"]
        (y * w3.to(dtype)).sum().backward()
        arrs[f"str_out{tag}"], arrs[f"str_g{tag}"] = y.detach().numpy(), x.grad.numpy()

        for conv, ctag in ((RefConv.OPENGL, "gl"), (RefConv.DIRECTX, "dx")):
            x = n0.detach().to(dtype).clone().requires_grad_(True)
            h = ref_h_from_n(x, 1.5, conv)
            (h * w1.to(dtype)).sum().backward()
            arrs[f"hfn_out_{ctag}{tag}"], arrs[f"hfn_g_{ctag}{tag}"] = h.detach().numpy(), x.grad.numpy()
    np.savez_compressed(os.path.join(HERE, "autograd_normal_ops.npz"), **arrs)
    print("autograd_normal_ops: ok")


if __name__ == "__main__":
    torch.set_num_threads(8)
    if len(sys.argv) > 1 and sys.argv[1] == "normalops":   # only this fixture (the others are unchanged)
        make_normal_ops_autograd_fixture()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "height":
        make_height_from_normal_fixture()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "convert":
        make_conversion_cases()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "autograd":   # only this fixture (the others are unchanged)
        make_autograd_cases()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "geomgrad":   # only this fixture (the others are unchanged)
        make_geomgrad_cases()
        sys.exit(0)
    for i, c in enumerate(CT_CASES):
        make_ct_case(i, c)
    make_conversion_cases()
    make_blend_cases()
    make_config1_fixture()
    make_geomgrad_cases()
    make_autograd_cases()
    make_height_from_normal_fixture()
    make_normal_ops_autograd_fixture()
