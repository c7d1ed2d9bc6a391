"""
pypbr_b200.models.cooktorrance — CookTorranceBRDF behind the reference's API.

Mirrors pypbr/models/cooktorrance.py: same class names, constructor and call signature, same return
shape, same exceptions.  `forward` validates on the host, then issues ONE kernel launch
(pbr_ct_forward); autograd's backward is ONE launch (pbr_ct_backward) that recomputes the forward in
registers and writes d(albedo, normal, roughness, metallic | specular) - no intermediate tensor is
ever materialised.

Extensions over the reference (which is single-material, single-light, cooktorrance.py:120):
  * maps may be batched (B, C, H, W) -> (B, 3, H, W);
  * `light_dir_or_position` / `light_intensity` may be (L, 3):
      multi_light="accumulate" -> encode(clamp(sum_l clamp(shade_l, 0, 1), 0, 1)), shape (..., 3, H, W)
      multi_light="per_light"  -> one image per light, shape (..., L, 3, H, W)
    both reduce to the reference for L = 1;
  * view_type="point": `view_dir` is the position of a camera at a finite distance, and every texel is shaded with its own
    view vector F.normalize(camera - P) (texel (i, j) at P = (x_j, -y_i, 0) on the plane of side `light_size or 1.0`);
  * per-material parameters for batched maps: `view_dir` (B, 3), `light_dir_or_position` (B, L, 3), `light_intensity`
    (B, L, 3) or (B, 1, 3), each on its own; a leading dimension of 1 is shared by the batch.  Material b is shaded exactly
    as a call with material[b], view_dir[b], lights[b], intensity[b] would shade it (pbr_ct_*_pb).
"""

from __future__ import annotations

from abc import ABC
from typing import Optional

import torch
import torch.nn as nn
from torch import Tensor

from .. import _cabi
from ..materials import MaterialBase


# A/B switch for tests and tuning: True routes every call to the generic kernels (PbrCtDesc.force_generic).
FORCE_GENERIC = False
NO_SAVED_OUT = False   # tests: make the accumulate-mode backward recompute the summed image (two passes) as the C ABI does without fwd_out


class BRDFModel(nn.Module, ABC):
    """Abstract base class for BRDF models."""


def _as_f32_rows(t: Tensor, name: str) -> Tensor:
    if not isinstance(t, Tensor):
        t = torch.as_tensor(t, dtype=torch.float32)
    if t.dim() == 1:
        t = t.view(1, -1)
    if t.dim() not in (2, 3) or t.shape[-1] != 3:
        raise ValueError(f"{name} must have shape (3,), (L, 3) or (B, L, 3), got {tuple(t.shape)}")
    return t


def _per_material(t: Tensor, B: int, batched: bool, name: str) -> bool:
    """Whether a parameter with a leading batch dimension holds one set per material (B) or one for the batch (1)."""
    if t.shape[0] == 1:
        return False
    if not batched:
        raise ValueError(f"{name} of shape {tuple(t.shape)} holds per-material parameters, which need batched (B, 3, H, W) maps")
    if t.shape[0] != B:
        raise ValueError(f"{name} has {t.shape[0]} parameter sets for a batch of {B} materials; expected {B} or 1")
    return True


def _parse_params(view_dir, light, intensity, B: int, batched: bool):
    """The view, lights and intensities of a call on B materials -> (view, lights (L, 3) | (B, L, 3), intensities of the
    lights' shape, whether the lights count as several, which of (intensity, lights, view) are per material).  Each is
    shared by the batch or, with a leading dimension of B, one set per material; a leading dimension of 1 is shared."""
    view = torch.as_tensor(view_dir, dtype=torch.float32) if not isinstance(view_dir, Tensor) else view_dir
    lights = _as_f32_rows(light, "light_dir_or_position")
    multi = lights.dim() == 3 or (isinstance(light, Tensor) and light.dim() == 2)
    pm_lights = lights.dim() == 3 and _per_material(lights, B, batched, "light_dir_or_position")
    if lights.dim() == 3 and not pm_lights:
        lights = lights[0]
    inten = _as_f32_rows(intensity, "light_intensity")   # (a 2-D intensity is (L, 3), whatever B is)
    pm_inten = inten.dim() == 3 and _per_material(inten, B, batched, "light_intensity")
    if inten.dim() == 3 and not pm_inten:
        inten = inten[0]
    L = lights.shape[-2]
    if inten.shape[-2] != L:
        if inten.shape[-2] != 1:
            raise ValueError(f"light_intensity has {inten.shape[-2]} rows for {L} lights")
        inten = inten.expand(*inten.shape[:-2], L, 3)
    if L > _cabi.PBR_MAX_LIGHTS:
        raise ValueError(f"at most {_cabi.PBR_MAX_LIGHTS} lights per call, got {L}")
    pm_view = view.numel() != 3 and view.dim() == 2 and view.shape[1] == 3 and _per_material(view, B, batched, "view_dir")
    if view.numel() != 3 and not pm_view:
        raise ValueError(f"view_dir must have shape (3,) or (B, 3), got {tuple(view.shape)}")
    return view, lights, inten, multi, (pm_inten, pm_lights, pm_view)


class _ShadeCfg:
    """Everything about one shading call that is not a texture map."""

    __slots__ = ("workflow", "metallic_channels", "light_type", "albedo_is_srgb", "specular_is_srgb", "return_srgb",
                 "per_light", "light_size", "L", "view", "lights", "intensity", "on_device", "batched", "multi", "camera",
                 "pb", "param_shapes")


def ct_call(kind: str, cfg: _ShadeCfg, desc, *args, device) -> None:
    """pbr_ct_<kind>: with per-material parameters its _pb form, with a camera its _camera form."""
    lib = _cabi.load()
    if cfg.pb is not None:
        fn = f"pbr_ct_{kind}_pb"
        rc = getattr(lib, fn)(_cabi.byref(desc), _cabi.byref(cfg.pb), *args, _cabi.stream_ptr(device))
    else:
        fn = f"pbr_ct_{kind}_camera" if cfg.camera else f"pbr_ct_{kind}"
        rc = getattr(lib, fn)(_cabi.byref(desc), *args, _cabi.stream_ptr(device))
    _cabi.check(rc, fn)


def _fill_desc(cfg: _ShadeCfg, albedo, normal, roughness, metspec, keep: list) -> "_cabi.PbrCtDesc":
    d = _cabi.PbrCtDesc()
    d.B = albedo.shape[0] if albedo.dim() == 4 else 1
    d.H, d.W = albedo.shape[-2], albedo.shape[-1]
    d.L = cfg.L
    d.workflow = cfg.workflow
    d.metallic_channels = cfg.metallic_channels
    d.light_type = cfg.light_type
    d.albedo_is_srgb = int(cfg.albedo_is_srgb)
    d.specular_is_srgb = int(cfg.specular_is_srgb)
    d.return_srgb = int(cfg.return_srgb)
    d.per_light = int(cfg.per_light)
    d.light_size = float(cfg.light_size)
    d.albedo = _cabi.plane(albedo)
    d.normal = _cabi.plane(normal)
    d.roughness = _cabi.plane(roughness)
    d.metspec = _cabi.plane(metspec)
    d.params_on_device = int(cfg.on_device)
    d.force_generic = int(FORCE_GENERIC)
    if cfg.on_device:
        d.view, d.lights, d.intensity = cfg.view.data_ptr(), cfg.lights.data_ptr(), cfg.intensity.data_ptr()
    else:
        hv = _cabi.host_floats(cfg.view)
        hl = _cabi.host_floats(cfg.lights)
        hi = _cabi.host_floats(cfg.intensity)
        keep.extend((hv, hl, hi))
        d.view = _cabi.ctypes.cast(hv, _cabi.c_void_p)
        d.lights = _cabi.ctypes.cast(hl, _cabi.c_void_p)
        d.intensity = _cabi.ctypes.cast(hi, _cabi.c_void_p)
    return d


def _out_plane(t: Tensor, per_light: bool, batched: bool):
    """Plane + per-light stride for an output-shaped tensor ((B,)(L,)3,H,W), contiguous."""
    HW3 = 3 * t.shape[-2] * t.shape[-1]
    L = t.shape[-4] if per_light else 1
    sb = HW3 * L if batched else 0
    return _cabi.PbrPlane(t.data_ptr(), sb, t.shape[-2] * t.shape[-1], t.shape[-1]), (HW3 if per_light else 0)


def _out_shape(cfg: _ShadeCfg, albedo: Tensor):
    shape = []
    if cfg.batched:
        shape.append(albedo.shape[0])
    if cfg.per_light:
        shape.append(cfg.L)
    return (*shape, 3, albedo.shape[-2], albedo.shape[-1])


def check_view_type(view_type: str) -> str:
    view_type = view_type.lower()
    if view_type not in ("directional", "point"):
        raise ValueError(f"Unsupported view_type: {view_type}. Must be 'directional' or 'point'.")
    return view_type


class _CookTorranceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, cfg: _ShadeCfg, albedo, normal, roughness, metspec, intensity_leaf, lights_leaf=None, view_leaf=None):
        keep: list = []
        d = _fill_desc(cfg, albedo, normal, roughness, metspec, keep)
        out = torch.empty(_out_shape(cfg, albedo), dtype=torch.float32, device=albedo.device)
        d.out, d.out_sl = _out_plane(out, cfg.per_light, cfg.batched)
        with _cabi.device_guard(albedo.device):
            ct_call("forward", cfg, d, device=albedo.device)
        ctx.cfg = cfg
        ctx.has_normal = normal is not None
        # the shared parameters may live on another device than the maps (the reference moves them with .to(device))
        ctx.leaf_meta = [(t.device, tuple(t.shape)) if t is not None else None for t in (intensity_leaf, lights_leaf, view_leaf)]
        # accumulate mode with several lights: the output (which the caller holds anyway) lets the backward skip its
        # first pass, the recomputation of the summed image (PbrCtGrads.fwd_out; the camera kernels do not use it)
        ctx.keep_out = cfg.L > 1 and not cfg.per_light and not cfg.camera
        ctx.save_for_backward(albedo, normal if normal is not None else albedo.new_empty(0), roughness, metspec,
                              out if ctx.keep_out else albedo.new_empty(0))
        return out

    @staticmethod
    def backward(ctx, grad_out):
        cfg = ctx.cfg
        albedo, normal, roughness, metspec, fwd_out = ctx.saved_tensors
        if not ctx.has_normal:
            normal = None
        keep: list = []
        d = _fill_desc(cfg, albedo, normal, roughness, metspec, keep)
        grad_out = grad_out.contiguous()
        g = _cabi.PbrCtGrads()
        g.grad_out, g.grad_out_sl = _out_plane(grad_out, cfg.per_light, cfg.batched)
        if ctx.keep_out and not NO_SAVED_OUT:
            g.fwd_out = _out_plane(fwd_out, False, cfg.batched)[0]
        need = ctx.needs_input_grad  # (cfg, albedo, normal, roughness, metspec, intensity, lights, view)
        dev = albedo.device
        d_albedo = torch.empty(albedo.shape, dtype=torch.float32, device=dev) if need[1] else None
        d_normal = torch.empty(normal.shape, dtype=torch.float32, device=dev) if (need[2] and normal is not None) else None
        d_rough = torch.empty(roughness.shape, dtype=torch.float32, device=dev) if need[3] else None
        d_met = torch.empty(metspec.shape, dtype=torch.float32, device=dev) if need[4] else None
        # the shared parameters' gradients are sums over the batch; a per-material parameter's, one set per material
        # (the gradient buffers take the parameters' strides)
        d_int, d_lights, d_view = (torch.zeros(shape, dtype=torch.float32, device=dev) if want else None
                                   for shape, want in zip(cfg.param_shapes, need[5:8]))
        g.d_albedo = _cabi.plane(d_albedo)
        g.d_normal = _cabi.plane(d_normal)
        g.d_roughness = _cabi.plane(d_rough)
        g.d_metspec = _cabi.plane(d_met)
        g.d_intensity = d_int.data_ptr() if d_int is not None else None
        # gradients of the light positions / directions and of the view direction (plain autograd in the reference)
        g.d_lights = d_lights.data_ptr() if d_lights is not None else None
        g.d_view = d_view.data_ptr() if d_view is not None else None
        with _cabi.device_guard(dev):
            ct_call("backward", cfg, d, _cabi.byref(g), device=dev)
        shared = []
        for t, meta in zip((d_int, d_lights, d_view), ctx.leaf_meta):
            shared.append(t.reshape(meta[1]).to(meta[0]) if (t is not None and meta is not None) else None)
        return (None, d_albedo, d_normal, d_rough, d_met, *shared)


def _prepare(material: MaterialBase, device, view_dir, light, intensity, light_type: str, light_size, return_srgb: bool,
             multi_light: str, view_type: str = "directional"):
    """Host-side validation in the reference's order (cooktorrance.py:92-118); returns (cfg, maps, shared-parameter
    leaves (intensity, lights, view - None where no gradient is wanted), device).  view_type="point": view_dir is the
    camera position."""
    # attribute / workflow errors first, exactly where the reference raises them (cooktorrance.py:99-118)
    roughness = material.roughness  # AttributeError if the map was never set
    normal = material.normal  # AttributeError unless the key exists (None selects the +Z default)
    cfg = _ShadeCfg()
    cfg.camera = check_view_type(view_type) == "point"
    cfg.specular_is_srgb = True
    cfg.metallic_channels = 1
    if hasattr(material, "metallic") and material.metallic is not None:
        albedo = material._maps.get("albedo", None)
        metspec = material.metallic
        cfg.workflow = _cabi.WORKFLOW_METALLIC
    elif hasattr(material, "specular") and material.specular is not None:
        albedo = material._maps.get("albedo", None)
        metspec = material.specular
        cfg.workflow = _cabi.WORKFLOW_SPECULAR
        cfg.specular_is_srgb = bool(getattr(material, "specular_is_srgb", True))
    else:
        raise ValueError("Material must have either 'metallic' or 'specular' property.")
    if albedo is None:
        # the reference fails on `material.linear_albedo.to(device)` with linear_albedo == None
        raise AttributeError("'NoneType' object has no attribute 'to'")

    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError(
            f"pypbr_b200: CookTorranceBRDF runs on CUDA only (material.device is {device}); there is no CPU fallback. "
            "Use material.to('cuda') or CookTorranceBRDF(override_device='cuda')."
        )
    # the reference moves every map with .to(device) on every call (cooktorrance.py:99-112); a map that is already there is
    # handed on untouched (Tensor.to would return it as well, several microseconds later)
    want = device.index if device.index is not None else torch.cuda.current_device()

    def mv(t):
        return t if (t is None or (t.is_cuda and t.device.index == want)) else t.to(device)

    roughness, normal, metspec, albedo = mv(roughness), mv(normal), mv(metspec), mv(albedo)
    cfg.albedo_is_srgb = bool(material.albedo_is_srgb)

    for name, t in (("albedo", albedo), ("roughness", roughness), ("normal", normal), ("metallic/specular", metspec)):
        if t is not None:
            _cabi.require_cuda(t, name)
    if albedo.dim() not in (3, 4) or albedo.shape[-3] != 3:
        raise ValueError(f"albedo must have shape (3, H, W) or (B, 3, H, W), got {tuple(albedo.shape)}")
    cfg.batched = albedo.dim() == 4
    H, W = albedo.shape[-2:]

    def fit(t, channels, name):
        if t.dim() == albedo.dim() - 1:
            t = t.unsqueeze(-3)
        if t.dim() != albedo.dim() or t.shape[-2:] != (H, W) or t.shape[-3] not in channels:
            raise ValueError(f"{name} of shape {tuple(t.shape)} does not match albedo {tuple(albedo.shape)}")
        if cfg.batched and t.shape[0] != albedo.shape[0]:
            if t.shape[0] != 1:
                raise ValueError(f"{name} batch {t.shape[0]} does not match albedo batch {albedo.shape[0]}")
            t = t.expand(albedo.shape[0], *t.shape[1:])
        return _cabi.rowmajor(t)

    albedo = _cabi.rowmajor(albedo)
    roughness = fit(roughness, (1,), "roughness")
    if normal is not None:
        normal = fit(normal, (3,), "normal")
    if cfg.workflow == _cabi.WORKFLOW_METALLIC:
        metspec = fit(metspec, (1, 3), "metallic")
        cfg.metallic_channels = metspec.shape[-3]
    else:
        metspec = fit(metspec, (3,), "specular")

    cfg.light_type = _cabi.LIGHT_POINT if light_type == "point" else _cabi.LIGHT_DIRECTIONAL
    # the plane's size places the texels: a point light's position, or a camera's, is relative to it
    cfg.light_size = float(light_size or 1.0) if (light_type == "point" or cfg.camera) else 0.0
    cfg.return_srgb = bool(return_srgb)

    B = albedo.shape[0] if cfg.batched else 1
    view, lights, inten, cfg.multi, (pm_inten, pm_lights, pm_view) = _parse_params(view_dir, light, intensity, B, cfg.batched)
    cfg.L = lights.shape[-2]
    cfg.per_light = cfg.multi and multi_light == "per_light"
    # shapes of the kernels' gradient buffers (intensity, lights, view): one set per material, or the sum over the batch
    cfg.param_shapes = ((B, cfg.L, 3) if pm_inten else (cfg.L, 3), (B, cfg.L, 3) if pm_lights else (cfg.L, 3),
                        (B, 3) if pm_view else (3,))

    # views of the caller's tensors: their (L, 3) / (3,) gradients reach the caller through autograd's view tracking
    shared_leaves = (inten if inten.requires_grad else None,
                     lights if lights.requires_grad else None,
                     view if view.requires_grad else None)
    # compare with the device the maps actually live on: torch.device("cuda") (no index) never equals "cuda:0", and the
    # device-resident fast path (no .tolist() sync, graph-capturable) would be dead for material.to("cuda")
    device = albedo.device
    cfg.pb = None
    if pm_view or pm_lights or pm_inten:
        # per-material parameters are read from device memory (the launch carries one set only): all three go there
        cfg.pb = _cabi.PbrCtParamBatch(int(cfg.camera), 0, 3 if pm_view else 0, 3 * cfg.L if pm_lights else 0,
                                       3 * cfg.L if pm_inten else 0)
    all_dev = cfg.pb is not None or all(t.is_cuda and t.device == device for t in (view, lights, inten))
    cfg.on_device = all_dev
    if all_dev:
        def f32c(t):
            t = t.detach().to(device=device, dtype=torch.float32)
            return t if t.is_contiguous() else t.contiguous()

        cfg.view = f32c(view).reshape(cfg.param_shapes[2])
        cfg.lights = f32c(lights)
        cfg.intensity = f32c(inten)
    else:  # small host arrays are copied into the kernel launch parameters: no H2D copy, no sync for CPU inputs
        cfg.view = view.detach().reshape(3).to(torch.float32).cpu().tolist()
        cfg.lights = lights.detach().to(torch.float32).cpu().reshape(-1).tolist()
        cfg.intensity = inten.detach().to(torch.float32).cpu().reshape(-1).tolist()
    return cfg, (albedo, normal, roughness, metspec), shared_leaves, device


class CookTorranceBRDF(BRDFModel):
    """
    Cook-Torrance BRDF (GGX D, Smith-Schlick G, Schlick F) for directional and point lights.

    view_type: "directional" (the reference: `view_dir` is one view direction for the whole image) or "point"
    (`view_dir` is the position of a camera at a finite distance, in the frame of a point light's position; each
    texel is shaded with its own view vector).

    Per-material parameters (batched maps only): view_dir (B, 3), light_dir_or_position (B, L, 3), light_intensity
    (B, L, 3) or (B, 1, 3), each on its own; material b is shaded as a call on material[b] with view_dir[b], lights[b],
    intensity[b] would shade it.  Such a call reads all three parameters from the maps' device, so any of them given on
    the CPU is copied there (a synchronous copy from pageable memory) on every call: keep them on the maps' device in a
    loop.

    Example:
        brdf = CookTorranceBRDF(light_type="point")
        color = brdf(material, view_dir, light_pos, light_intensity, light_size)   # (3, H, W)
        color = CookTorranceBRDF(light_type="point", view_type="point")(material, camera_pos, light_pos, light_intensity)
    """

    def __init__(self, light_type: str = "point", override_device: torch.device = None, multi_light: str = "accumulate",
                 view_type: str = "directional"):
        super().__init__()
        self.light_type = light_type.lower()
        if self.light_type not in ["directional", "point"]:
            raise ValueError(f"Unsupported light_type: {self.light_type}. Must be 'directional' or 'point'.")
        if multi_light not in ("accumulate", "per_light"):
            raise ValueError(f"Unsupported multi_light: {multi_light}. Must be 'accumulate' or 'per_light'.")
        self.override_device = override_device
        self.multi_light = multi_light
        self.view_type = check_view_type(view_type)

    def forward(
        self,
        material: MaterialBase,
        view_dir: Tensor,
        light_dir_or_position: Tensor,
        light_intensity: Tensor,
        light_size: Optional[float] = None,
        return_srgb: bool = True,
    ) -> Tensor:
        """
        Evaluate the BRDF.  Arguments as in the reference (cooktorrance.py:68-91).

        Returns:
            Tensor (3, H, W); (B, 3, H, W) for batched maps; (..., L, 3, H, W) in per_light mode.
        """
        device = self.override_device or material.device
        cfg, (albedo, normal, roughness, metspec), shared_leaves, _ = _prepare(
            material, device, view_dir, light_dir_or_position, light_intensity, self.light_type, light_size,
            return_srgb, self.multi_light, self.view_type,
        )
        # the shared-parameter leaves are views of the caller's tensors, so e.g. the (L, 3) intensity gradient reaches
        # the caller's (3,) or (L, 3) tensor through autograd's view tracking.
        return _CookTorranceFn.apply(cfg, albedo, normal, roughness, metspec, *shared_leaves)
