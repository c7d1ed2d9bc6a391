"""
tools/bench_batched_params.py — what per-material view, lights and intensities cost (CookTorranceBRDF with (B, 3) / (B, L, 3)
parameters, the pbr_ct_*_pb entry points: the generic kernels with one material per CTA), against the two ways to get the
same images without them, in the same process, legs alternating step by step, timed with CUDA events.

  train  64 x 256^2, metallic, forward + backward through autograd, L = 1 and L = 4, a camera (view_type="point") and point
         lights of their own per material.  Legs: one call with per-material lights and cameras; a Python loop of 64
         single-material calls (one per material, each with its own lights and camera); one call with one shared set (the
         bound).  Maps, grad_out and gradients: ~340 MB, over the 126 MB of L2.
  c2     bench.py's C2 shape (64 x 1024^2, one point light, the orthographic view), forward + backward: per-material lights
         against one shared light, which the streamed TMA-fed kernels shade.
  c5     bench.py's C5 shape, the one-launch fit step (fit_step(fused=True)): 512 x 512^2, 8 point lights, per-light targets,
         per-material lights against shared ones (which the generic kernels shade with a geometry cache over a 16-material
         walk).

    python tools/bench_batched_params.py [--steps 20] [--warmup 3] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402


def power_limit() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def random_maps(B, H, W, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    n = torch.randn(B, 3, H, W, generator=g, device=dev) * torch.tensor([0.3, 0.3, 0.0], device=dev).view(1, 3, 1, 1)
    return dict(albedo=torch.rand(B, 3, H, W, generator=g, device=dev),
                normal=torch.nn.functional.normalize(n + torch.tensor([0.0, 0.0, 1.0], device=dev).view(1, 3, 1, 1), dim=1),
                roughness=torch.rand(B, 1, H, W, generator=g, device=dev) * 0.8 + 0.2,
                metallic=torch.rand(B, 1, H, W, generator=g, device=dev)), g


def random_lights(B, L, dev, g):
    """(B, L, 3) point lights around the plane's centre and (B, 3) cameras above it, one set per material."""
    lights = torch.rand(B, L, 3, generator=g, device=dev) * torch.tensor([0.8, 0.8, 0.5], device=dev) - torch.tensor([0.4, 0.4, -0.8], device=dev)
    cams = torch.rand(B, 3, generator=g, device=dev) * torch.tensor([0.4, 0.4, 0.5], device=dev) - torch.tensor([0.2, 0.2, -1.2], device=dev)
    return lights, cams


def timed(legs, steps, warmup, work):
    for _ in range(max(warmup, 3)):
        for leg in legs.values():
            leg()
    torch.cuda.synchronize()
    evs = {name: [] for name in legs}
    for _ in range(steps):
        for name, leg in legs.items():   # alternating: every leg sees the same clocks and neighbours
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            leg()
            e1.record()
            evs[name].append((e0, e1))
    torch.cuda.synchronize()
    res = {}
    for name, ev in evs.items():
        t = sorted(a.elapsed_time(b) for a, b in ev)
        med = t[len(t) // 2]
        res[name] = dict(median_ms=round(med, 4), min_ms=round(t[0], 4), max_ms=round(t[-1], 4),
                         gtexel_lights_per_s=round(work / (med * 1e-3) / 1e9, 2))
    return res


def run_train(L, steps, warmup, dev):
    from pypbr_b200.materials import BasecolorMetallicMaterial
    from pypbr_b200.models import CookTorranceBRDF

    B, H, W = 64, 256, 256
    maps, g = random_maps(B, H, W, dev, 5 + L)
    lights, cams = random_lights(B, L, dev, g)
    inten = torch.ones(L, 3, device=dev) / L
    grad_out = torch.rand(B, 3, H, W, generator=g, device=dev)
    leaves = {k: v.requires_grad_(True) for k, v in maps.items()}
    mat = BasecolorMetallicMaterial(albedo_is_srgb=True, device=dev)
    mat._maps.update(leaves)
    brdf = CookTorranceBRDF("point", view_type="point")
    one = BasecolorMetallicMaterial(albedo_is_srgb=True, device=dev)

    def clear():
        for t in leaves.values():
            t.grad = None

    def per_material():
        clear()
        brdf(mat, cams, lights, inten, 1.0).backward(grad_out)

    def loop():   # what a user writes without per-material parameters: one call per material
        clear()
        for b in range(B):
            one._maps.update({k: v[b:b + 1] for k, v in leaves.items()})
            brdf(one, cams[b], lights[b], inten, 1.0).backward(grad_out[b:b + 1])

    def shared():
        clear()
        brdf(mat, cams[0], lights[0], inten, 1.0).backward(grad_out)

    res = timed(dict(per_material=per_material, loop=loop, shared=shared), steps, warmup, B * H * W * L)
    res["shape"] = dict(B=B, H=H, W=W, L=L)
    res["loop_over_per_material"] = round(res["loop"]["median_ms"] / res["per_material"]["median_ms"], 2)
    res["per_material_over_shared"] = round(res["per_material"]["median_ms"] / res["shared"]["median_ms"], 3)
    return res


def run_c2(steps, warmup, dev):
    from pypbr_b200.materials import BasecolorMetallicMaterial
    from pypbr_b200.models import CookTorranceBRDF

    B, H, W = 64, 1024, 1024
    maps, g = random_maps(B, H, W, dev, 7)
    lights, _ = random_lights(B, 1, dev, g)
    view, inten = torch.tensor([0.0, 0.0, 1.0], device=dev), torch.ones(3, device=dev)
    grad_out = torch.rand(B, 3, H, W, generator=g, device=dev)
    leaves = {k: v.requires_grad_(True) for k, v in maps.items()}
    mat = BasecolorMetallicMaterial(albedo_is_srgb=True, device=dev)
    mat._maps.update(leaves)
    brdf = CookTorranceBRDF("point")

    def leg(light):
        def step():
            for t in leaves.values():
                t.grad = None
            brdf(mat, view, light, inten, 1.0).backward(grad_out)
        return step

    res = timed(dict(per_material=leg(lights), shared=leg(lights[0, 0])), steps, warmup, B * H * W)
    res["shape"] = dict(B=B, H=H, W=W, L=1)
    res["per_material_over_shared"] = round(res["per_material"]["median_ms"] / res["shared"]["median_ms"], 3)
    return res


def run_c5(steps, warmup, dev):
    from pypbr_b200.fit import FusedAdam, fit_step
    from pypbr_b200.materials import BasecolorMetallicMaterial

    B, H, W, L = 512, 512, 512, 8
    maps, g = random_maps(B, H, W, dev, 9)
    lights, _ = random_lights(B, L, dev, g)
    view, inten = torch.tensor([0.0, 0.0, 1.0], device=dev), torch.ones(L, 3, device=dev)
    target = torch.rand(B, L, 3, H, W, generator=g, device=dev)
    legs = {}
    for name, light in (("per_material", lights), ("shared", lights[0])):
        mat = BasecolorMetallicMaterial(albedo_is_srgb=True, device=dev)
        mat._maps.update({k: v.clone() for k, v in maps.items()})
        opt = FusedAdam(dict(mat._maps), lr=0.01)
        scratch = {}
        legs[name] = (lambda mat=mat, opt=opt, light=light, scratch=scratch:
                      fit_step(mat, opt, target, view, light, inten, "point", 1.0, fused=True, scratch=scratch))
    del maps
    res = timed(legs, steps, warmup, B * H * W * L)
    res["shape"] = dict(B=B, H=H, W=W, L=L, multi_light="per_light")
    res["per_material_over_shared"] = round(res["per_material"]["median_ms"] / res["shared"]["median_ms"], 3)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_batched_params.py needs a CUDA device")
    dev = torch.device("cuda:0")
    line = dict(device=torch.cuda.get_device_name(0), power_limit=power_limit(),
                rate="Gtexel-lights/s of the whole step (median)")
    for L in (1, 4):
        line[f"train_L{L}"] = run_train(L, args.steps, args.warmup, dev)
        torch.cuda.empty_cache()
    line["c2"] = run_c2(args.steps, args.warmup, dev)
    torch.cuda.empty_cache()
    with torch.no_grad():
        line["c5_fit_step"] = run_c5(args.steps, args.warmup, dev)
    print(json.dumps(line))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
