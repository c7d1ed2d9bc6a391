"""
tools/bench_camera.py — what a camera at a finite position costs: one forward + backward step through autograd
(CookTorranceBRDF(view_type="point"), the cam_* kernels) against the same step with the orthographic view (the ct_*
kernels), in the same process, the two alternating step by step, timed with CUDA events.

Shapes: the C2 shape of bench.py (64 x 1024^2, one point light) and its C3 shape (16 x 2048^2, 16 point lights,
accumulated), metallic workflow, every map gradient requested.  The maps, grad_out and gradients of either shape take
about 4 GB, far more than the 126 MB of L2.

    python tools/bench_camera.py [--steps 20] [--warmup 3] [--out result.json]
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

SHAPES = {"c2": dict(B=64, H=1024, W=1024, L=1), "c3": dict(B=16, H=2048, W=2048, L=16)}


def power_limit() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def run_shape(name, B, H, W, L, steps, warmup, dev):
    from pypbr_b200.materials import BasecolorMetallicMaterial
    from pypbr_b200.models import CookTorranceBRDF

    g = torch.Generator(device=dev).manual_seed(5)
    n = torch.randn(B, 3, H, W, generator=g, device=dev) * torch.tensor([0.3, 0.3, 0.0], device=dev).view(1, 3, 1, 1)
    maps = dict(albedo=torch.rand(B, 3, H, W, generator=g, device=dev),
                normal=torch.nn.functional.normalize(n + torch.tensor([0.0, 0.0, 1.0], device=dev).view(1, 3, 1, 1), dim=1),
                roughness=torch.rand(B, 1, H, W, generator=g, device=dev) * 0.8 + 0.2,
                metallic=torch.rand(B, 1, H, W, generator=g, device=dev))
    mat = BasecolorMetallicMaterial(albedo_is_srgb=True, device=dev)
    mat._maps.update({k: v.requires_grad_(True) for k, v in maps.items()})
    ang = torch.arange(L, dtype=torch.float32) * (6.2831853 / L)
    lights = torch.stack([0.4 * torch.cos(ang), 0.4 * torch.sin(ang), torch.ones(L)], dim=1) if L > 1 else torch.tensor([0.1, 0.1, 1.0])
    inten = torch.ones(L, 3) / L if L > 1 else torch.ones(3)
    grad_out = torch.rand(B, 3, H, W, generator=g, device=dev)
    legs = {"ortho": (CookTorranceBRDF("point"), torch.tensor([0.0, 0.0, 1.0])),
            "camera": (CookTorranceBRDF("point", view_type="point"), torch.tensor([0.1, -0.1, 1.5]))}

    def step(leg):
        brdf, view = legs[leg]
        for t in maps.values():
            t.grad = None
        brdf(mat, view, lights, inten, 1.0).backward(grad_out)

    for _ in range(max(warmup, 3)):
        for leg in legs:
            step(leg)
    torch.cuda.synchronize()
    ms = {leg: [] for leg in legs}
    for _ in range(steps):
        for leg in legs:   # alternating: both legs see the same clocks and neighbours
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step(leg)
            e1.record()
            ms[leg].append((e0, e1))
    torch.cuda.synchronize()
    res = dict(shape=dict(B=B, H=H, W=W, L=L), steps=steps)
    for leg, evs in ms.items():
        t = sorted(a.elapsed_time(b) for a, b in evs)
        med = t[len(t) // 2]
        res[leg] = dict(median_ms=round(med, 4), min_ms=round(t[0], 4), max_ms=round(t[-1], 4),
                        gtexel_lights_per_s=round(B * H * W * L / (med * 1e-3) / 1e9, 2))
    res["camera_over_ortho"] = round(res["camera"]["median_ms"] / res["ortho"]["median_ms"], 3)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--shapes", default="c2,c3")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_camera.py needs a CUDA device")
    dev = torch.device("cuda:0")
    line = dict(device=torch.cuda.get_device_name(0), power_limit=power_limit(),
                step="CookTorranceBRDF forward + backward through autograd, metallic, every map gradient")
    for name in args.shapes.split(","):
        line[name] = run_shape(name, **SHAPES[name], steps=args.steps, warmup=args.warmup, dev=dev)
        torch.cuda.empty_cache()
    print(json.dumps(line))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
