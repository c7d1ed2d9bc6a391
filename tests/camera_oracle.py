"""
tests/camera_oracle.py — TEST INFRASTRUCTURE: the checker of the camera at a finite position (view_type="point").

The reference shades with one view direction, so it has no camera to pin this path against.  The oracle is therefore
oracle.pbr_oracle's restatement of the reference's op sequence (pypbr/models/cooktorrance.py:92-177) with ONE
substitution: the constant view map becomes the per-texel view vector of a camera at position `camera`,

    pos  = the fp32 plane grid the point-light branch builds, (x_j, -y_i, 0), side s = light_size or 1.0 (for both
           light types);
    vmap = F.normalize(camera.view(3, 1, 1) - pos, dim=0)

and every later use of the view (N.V twice, h = normalize(v + l), clamp(h.v) in the Fresnel term) reads vmap.  The same
code in fp64 is the arbiter of the shared-parameter gradients, as for the orthographic path.
"""

from __future__ import annotations

import math
import os
import sys
from typing import Dict, Optional

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import pbr_oracle as O  # noqa: E402

Tensor = torch.Tensor


def plane_grid(H: int, W: int, light_size, device) -> Tensor:
    """The reference's point-light grid (cooktorrance.py:128-133): (3, H, W) fp32 positions (x_j, -y_i, 0)."""
    s = light_size or 1.0
    x = torch.linspace(-s / 2, s / 2, W, device=device)
    y = torch.linspace(-s / 2, s / 2, H, device=device)
    yv, xv = torch.meshgrid(y, x, indexing="ij")
    return torch.stack([xv, -yv, torch.zeros_like(xv)], dim=0)


def shade_linear(maps: Dict[str, Tensor], camera: Tensor, light: Tensor, intensity: Tensor, light_size: Optional[float] = None,
                 light_type: str = "point", albedo_is_srgb: bool = True, specular_is_srgb: bool = True) -> Tensor:
    """oracle.pbr_oracle.shade_linear with the camera's per-texel view vector in place of the constant view map."""
    dt = maps["albedo"].dtype
    inten = intensity.view(3, 1, 1)
    rough = maps["roughness"]
    nmap = maps.get("normal")
    albedo = maps["albedo"]
    base = O.srgb_to_linear(albedo) if albedo_is_srgb else albedo
    metallic = maps.get("metallic")
    if metallic is not None:
        f0 = torch.lerp(torch.full_like(base, 0.04), base, metallic)
    elif maps.get("specular") is not None:
        spec_map = maps["specular"]
        f0 = O.srgb_to_linear(spec_map) if specular_is_srgb else spec_map
    else:
        raise ValueError("Material must have either 'metallic' or 'specular' property.")

    _, H, W = base.shape
    pos = plane_grid(H, W, light_size, base.device)
    vmap = F.normalize(camera.view(3, 1, 1) - pos, dim=0)   # the substitution
    att = 1.0
    if light_type == "directional":
        ldir = F.normalize(light, dim=0)
        lmap = ldir.view(3, 1, 1).expand(3, H, W)
    elif light_type == "point":
        lmap = light.view(3, 1, 1) - pos
        dist = torch.norm(lmap, dim=0, keepdim=True)
        lmap = lmap / (dist + 1e-7)
        att = 1.0 / (dist**2 + 1e-7)
    else:
        raise ValueError("Invalid light_type")

    if nmap is None:
        nmap = torch.tensor([0.0, 0.0, 1.0], dtype=dt, device=base.device).view(3, 1, 1).expand(3, H, W)
    n = F.normalize(nmap, dim=0)
    h = F.normalize(vmap + lmap, dim=0)
    cos_t = torch.clamp((h * vmap).sum(dim=0, keepdim=True), 0.0, 1.0)
    fs = f0 + (1.0 - f0) * torch.pow(1.0 - cos_t.expand_as(f0), 5.0)
    ndf = O._ggx_ndf(n, h, rough)
    g_ndv = torch.clamp((n * vmap).sum(dim=0, keepdim=True), 0.0, 1.0)
    g_ndl = torch.clamp((n * lmap).sum(dim=0, keepdim=True), 0.0, 1.0)
    g = O._g1(g_ndv, rough) * O._g1(g_ndl, rough)
    ndv = torch.clamp((n * vmap).sum(dim=0, keepdim=True), 0.0, 1.0)
    ndl = torch.clamp((n * lmap).sum(dim=0, keepdim=True), 0.0, 1.0)
    spec = (fs * ndf * g) / (4.0 * ndv * ndl + 1e-7)
    kd = (1.0 - fs) * (1.0 - metallic) if metallic is not None else 1.0 - fs
    diff = kd * base / math.pi
    rad = inten * (ndl * att)
    return torch.clamp((diff + spec) * rad, 0.0, 1.0)


def render(maps: Dict[str, Tensor], camera: Tensor, lights: Tensor, intensities: Tensor, light_size: Optional[float] = None,
           light_type: str = "point", albedo_is_srgb: bool = True, specular_is_srgb: bool = True, return_srgb: bool = True,
           accumulate: bool = True) -> Tensor:
    """oracle.pbr_oracle.render (batches, several lights, per-light or accumulated) with a camera at `camera`."""
    batched = maps["albedo"].dim() == 4
    multi = lights.dim() == 2
    B = maps["albedo"].shape[0] if batched else 1
    lts = lights if multi else lights.view(1, 3)
    ins = intensities if intensities.dim() == 2 else intensities.view(1, 3).expand(lts.shape[0], 3)
    enc = O.linear_to_srgb if return_srgb else (lambda c: c)
    outs = []
    for b in range(B):
        mb = {k: (t[b] if batched else t) for k, t in maps.items() if t is not None}
        per = [shade_linear(mb, camera, lts[l], ins[l], light_size, light_type, albedo_is_srgb, specular_is_srgb)
               for l in range(lts.shape[0])]
        if accumulate or not multi:
            if len(per) == 1:
                outs.append(enc(per[0]))
            else:
                tot = per[0]
                for p in per[1:]:
                    tot = tot + p
                outs.append(enc(torch.clamp(tot, 0.0, 1.0)))
        else:
            outs.append(torch.stack([enc(p) for p in per], dim=0))
    return torch.stack(outs, dim=0) if batched else outs[0]
