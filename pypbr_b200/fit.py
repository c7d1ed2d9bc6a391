"""
pypbr_b200.fit — the rendering-loss step of an SVBRDF inverse-rendering fit, fused and sharded.

The reference only documents this loop (docs/source/tutorials/06_advanced.rst:73-107):
``RenderingLoss.forward = MSELoss()(brdf(pred, ...), brdf(gt, ...))`` over a DataLoader of materials.
Here one kernel launch (pbr_ct_loss_fwd_bwd) renders the predicted material, compares it with the
target image, reduces the squared error (warp shuffle -> shared -> one atomic per CTA) and writes
d loss / d(albedo, normal, roughness, metallic | specular) - the rendered image never reaches HBM.

Multi-GPU: materials are independent, so the batch is sharded across ranks with no data-path
collective; the only exchange is ONE all-reduce per step over a (1 + 3L)-float buffer holding the
loss sum and the gradients of the shared parameters - light intensities and, on request, light positions /
directions and the view direction (`allreduce_loss_and_shared`).
"""

from __future__ import annotations

import ctypes
from typing import Dict, Optional, Tuple

import torch
import torch.nn as nn

from . import _cabi
from .materials import MaterialBase
from .models.cooktorrance import _fill_desc, _out_plane, _prepare, check_view_type


def shard_range(total: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous slice [lo, hi) of `total` materials owned by `rank` (remainder spread over the first ranks)."""
    base, rem = divmod(total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def fused_loss_step(
    material: MaterialBase,
    target: torch.Tensor,
    view_dir: torch.Tensor,
    lights: torch.Tensor,
    intensity: torch.Tensor,
    light_type: str = "point",
    light_size: Optional[float] = None,
    return_srgb: bool = True,
    multi_light: str = "per_light",
    loss_scale: Optional[float] = None,
    want_intensity_grad: bool = False,
    out: Optional[Dict[str, torch.Tensor]] = None,
    want_geometry_grad: bool = False,
    want_map_grads: bool = True,
    device=None,
    view_type: str = "directional",
):
    """
    One fused forward + MSE + backward pass over a (batched) material.

    target: the reference render, same shape as CookTorranceBRDF would return for these arguments.
    loss_scale: factor applied to the gradients (default 1/target.numel(), i.e. nn.MSELoss()).
    out: optional dict of preallocated gradient / scratch buffers to reuse between steps
         (keys d_albedo, d_normal, d_roughness, d_metspec, buf).
    want_geometry_grad: also the gradients of the light positions / directions and of the view direction (shared
         parameters of a fit with unknown lighting); buf then has 1 + 6L + 3 floats.
    want_map_grads: False -> loss (and shared-parameter gradients) only: no gradient buffer is allocated or written.
    device: where to shade (default material.device; maps living elsewhere are moved, like CookTorranceBRDF's override_device).
    view_type: as CookTorranceBRDF's; "point" reads view_dir as the camera position, and the last 3 floats of buf (with
         want_geometry_grad) are then the gradient w.r.t. that position.
    Returns (buf, grads): buf is a device tensor [loss_sum, d_intensity(L*3)..., (d_lights(L*3)..., d_view(3))]
    (loss_sum is the UNscaled sum of squared errors; multiply by loss_scale for the mean), grads a dict of tensors.
    """
    lib = _cabi.load()
    cfg, (albedo, normal, roughness, metspec), _leaf, device = _prepare(
        material, device if device is not None else material.device, view_dir, lights, intensity, light_type, light_size,
        return_srgb, multi_light, view_type
    )
    _cabi.require_cuda(target, "target")
    target = target.contiguous()
    expect = ((albedo.shape[0],) if cfg.batched else ()) + ((cfg.L,) if cfg.per_light else ()) + (3, *albedo.shape[-2:])
    if tuple(target.shape) != expect:
        raise ValueError(f"target has shape {tuple(target.shape)}, expected {expect}")
    if loss_scale is None:
        loss_scale = 1.0 / target.numel()
    out = out if out is not None else {}

    def buf(key, like):
        t = out.get(key)
        if t is None or t.shape != like.shape or t.device != like.device:
            t = torch.empty(like.shape, dtype=torch.float32, device=device)
            out[key] = t
        return t

    keep: list = []
    d = _fill_desc(cfg, albedo, normal, roughness, metspec, keep)
    g = _cabi.PbrCtGrads()
    d_albedo = buf("d_albedo", albedo) if want_map_grads else None
    d_normal = buf("d_normal", normal) if (normal is not None and want_map_grads) else None
    d_rough = buf("d_roughness", roughness) if want_map_grads else None
    d_met = buf("d_metspec", metspec) if want_map_grads else None
    g.d_albedo, g.d_normal = _cabi.plane(d_albedo), _cabi.plane(d_normal)
    g.d_roughness, g.d_metspec = _cabi.plane(d_rough), _cabi.plane(d_met)
    red = out.get("buf")
    n_red = 1 + 3 * cfg.L + ((3 * cfg.L + 3) if want_geometry_grad else 0)
    if red is None or red.numel() != n_red:
        red = torch.empty(n_red, dtype=torch.float32, device=device)
        out["buf"] = red
    red.zero_()
    g.d_intensity = red[1:].data_ptr() if want_intensity_grad else None
    if want_geometry_grad:
        g.d_lights = red[1 + 3 * cfg.L:].data_ptr()
        g.d_view = red[1 + 6 * cfg.L:].data_ptr()
    ls = _cabi.PbrCtLoss()
    ls.target, ls.target_sl = _out_plane(target, cfg.per_light, cfg.batched)
    ls.loss_scale = float(loss_scale)
    ls.loss_sum = red.data_ptr()
    fn = "pbr_ct_loss_fwd_bwd_camera" if cfg.camera else "pbr_ct_loss_fwd_bwd"
    with torch.cuda.device(device):
        _cabi.check(getattr(lib, fn)(_cabi.byref(d), _cabi.byref(ls), _cabi.byref(g), _cabi.stream_ptr(device)), fn)
    grads = {"albedo": d_albedo, "normal": d_normal, "roughness": d_rough,
             ("metallic" if cfg.workflow == _cabi.WORKFLOW_METALLIC else "specular"): d_met}
    return red, grads


def allreduce_loss_and_shared(buf: torch.Tensor, group=None) -> torch.Tensor:
    """
    The ONLY collective of the sharded fit: SUM all-reduce of [loss_sum, d_intensity...] (1 + 3L floats)
    over NCCL / NVLink.  Per-material map gradients are never communicated.  No-op without an
    initialised process group (single GPU).  Issued on the current stream: whatever is launched next waits for it.
    """
    import torch.distributed as dist

    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    return buf


class PendingLoss:
    """
    Handle of a loss all-reduce that was issued OFF the compute stream (`allreduce_loss_async`).  The update of a
    `fit_step(..., fused=True)` does not depend on the reduced loss (its gradient scale 1/global_numel is known up
    front), so the next step's kernel must not wait for the slowest rank's previous step: the collective runs on a side
    stream behind an event and only whoever reads the loss waits for it.

    wait()  : the CURRENT stream waits for the all-reduce; returns the reduced device buffer.
    item()  : host-synchronises on the all-reduce only (not on the compute stream) and returns buf[0] * scale.
    """

    def __init__(self, buf: torch.Tensor, work=None, done: Optional["torch.cuda.Event"] = None, scale: float = 1.0):
        self.buf, self._work, self._done, self.scale = buf, work, done, scale

    def wait(self) -> torch.Tensor:
        if self._done is not None:
            torch.cuda.current_stream(self.buf.device).wait_event(self._done)
        elif self._work is not None:   # CPU group (gloo): the work object blocks the host
            self._work.wait()
            self._work = None
        return self.buf

    def item(self) -> float:
        if self._done is not None:
            self._done.synchronize()
        elif self._work is not None:
            self._work.wait()
            self._work = None
        elif self.buf.is_cuda:
            torch.cuda.current_stream(self.buf.device).synchronize()
        return float(self.buf[0]) * self.scale


_side_streams: Dict[int, "torch.cuda.Stream"] = {}


def _side_stream(device: torch.device) -> "torch.cuda.Stream":
    idx = device.index if device.index is not None else torch.cuda.current_device()
    st = _side_streams.get(idx)
    if st is None:
        st = torch.cuda.Stream(device=device)
        _side_streams[idx] = st
    return st


def allreduce_loss_async(buf: torch.Tensor, group=None, scale: float = 1.0, timing: Optional[list] = None) -> PendingLoss:
    """
    `allreduce_loss_and_shared` off the compute stream: a side stream waits (event) for what the compute stream has
    enqueued so far - the kernel that fills `buf` - and carries the collective; the compute stream goes on at once.
    The caller must not touch `buf` on the compute stream before `PendingLoss.wait()` (fit_step alternates two buffers).
    timing: optional list that receives a (start, end) CUDA-event pair bracketing the collective on the side stream.
    """
    import torch.distributed as dist

    multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
    if not buf.is_cuda:   # CPU tensors (gloo tests): plain asynchronous work object
        return PendingLoss(buf, dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group, async_op=True) if multi else None, None, scale)
    side = _side_stream(buf.device)
    side.wait_stream(torch.cuda.current_stream(buf.device))
    done = torch.cuda.Event(enable_timing=timing is not None)
    with torch.cuda.stream(side):
        if timing is not None:
            t0 = torch.cuda.Event(enable_timing=True)
            t0.record(side)
        if multi:
            dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group, async_op=True).wait()   # side stream waits, not the host
        done.record(side)
        if timing is not None:
            timing.append((t0, done))
    return PendingLoss(buf, None, done, scale)


# projection that keeps a fitted map valid after every optimiser step
DEFAULT_PROJECTION = {
    "albedo": ("clamp", 0.0, 1.0), "roughness": ("clamp", 0.0, 1.0), "metallic": ("clamp", 0.0, 1.0),
    "specular": ("clamp", 0.0, 1.0), "height": ("clamp", 0.0, 1.0), "normal": ("normalize", 0.0, 0.0),
}


class FusedAdam:
    """
    Adam on every parameter map of a (batched) material in ONE kernel launch per step (pbr_adam_step), fused with
    the projection onto the valid range: clamp to [0, 1] for albedo / roughness / metallic / specular, renormalise
    for the normal map.  The update rule is torch.optim.Adam's (no weight decay, no amsgrad); the reference has no
    optimiser code (docs/source/tutorials/06_advanced.rst:136-137 leaves it to the reader).

    params: dict name -> CUDA float32 tensor (C,H,W) or (B,C,H,W), updated in place.
    project: dict name -> ("clamp", lo, hi) | ("normalize",) | None; defaults to DEFAULT_PROJECTION by map name.
    """

    def __init__(self, params: Dict[str, torch.Tensor], lr: float = 1e-2, betas=(0.9, 0.999), eps: float = 1e-8,
                 project: Optional[Dict[str, Optional[tuple]]] = None):
        if not params:
            raise ValueError("FusedAdam needs at least one parameter map")
        if len(params) > _cabi.PBR_MAX_ADAM_MAPS:
            raise ValueError(f"at most {_cabi.PBR_MAX_ADAM_MAPS} maps per optimiser")
        self.params = {}
        shape = None
        for name, t in params.items():
            _cabi.require_cuda(t, name)
            if t.dim() not in (3, 4) or not t.is_contiguous():
                raise ValueError(f"{name}: parameter maps must be contiguous (C,H,W) or (B,C,H,W) tensors")
            key = (t.shape[0] if t.dim() == 4 else 1, t.shape[-2], t.shape[-1])
            if shape is None:
                shape = key
            elif key != shape:
                raise ValueError("all parameter maps must share batch and spatial size")
            self.params[name] = t
        self.B, self.H, self.W = shape
        self.lr, self.betas, self.eps = float(lr), (float(betas[0]), float(betas[1])), float(eps)
        self.step_count = 0
        self.state = {n: (torch.zeros_like(t), torch.zeros_like(t)) for n, t in self.params.items()}
        proj = dict(DEFAULT_PROJECTION)
        if project is not None:
            proj.update(project)
        self.project = {n: proj.get(n) for n in self.params}

    def step(self, grads: Dict[str, torch.Tensor], grad_scale: float = 1.0) -> None:
        """One Adam step with gradient `grads[name] * grad_scale` for every map (grads are not modified)."""
        lib = _cabi.load()
        t_step = self.step_count + 1   # committed only once the launch has been accepted
        b1, b2 = self.betas
        d = _cabi.PbrAdamDesc()
        d.B, d.H, d.W, d.n_maps = self.B, self.H, self.W, len(self.params)
        d.step_size = self.lr / (1.0 - b1 ** t_step)
        d.one_minus_beta1, d.beta2, d.one_minus_beta2 = 1.0 - b1, b2, 1.0 - b2
        d.bias2_sqrt = (1.0 - b2 ** t_step) ** 0.5
        d.eps, d.grad_scale = self.eps, float(grad_scale)
        device = None
        for i, (name, t) in enumerate(self.params.items()):
            g = grads[name]
            _cabi.require_cuda(g, f"grad of {name}")
            if g.shape != t.shape or not g.is_contiguous():
                raise ValueError(f"grad of {name} must be a contiguous tensor of shape {tuple(t.shape)}")
            m, v = self.state[name]
            pr = self.project[name]
            kind = _cabi.PROJECT_NONE if pr is None else (_cabi.PROJECT_CLAMP if pr[0] == "clamp" else _cabi.PROJECT_NORMALIZE)
            lo, hi = (float(pr[1]), float(pr[2])) if kind == _cabi.PROJECT_CLAMP else (0.0, 0.0)
            d.maps[i] = _cabi.PbrAdamMap(_cabi.plane(t), _cabi.plane(g), _cabi.plane(m), _cabi.plane(v), t.shape[-3], kind, lo, hi)
            device = t.device
        with torch.cuda.device(device):
            _cabi.check(lib.pbr_adam_step(_cabi.byref(d), _cabi.stream_ptr(device)), "pbr_adam_step")
        _cabi.touch(*self.params.values())
        self.step_count = t_step


def _no_camera(view_type: str) -> None:
    if check_view_type(view_type) == "point":
        raise ValueError("the one-launch fit step has no camera at a finite position (view_type='point'): "
                         "use fit_step(fused=False)")


def fused_fit_step(
    material: MaterialBase,
    optimizer: FusedAdam,
    target: torch.Tensor,
    view_dir: torch.Tensor,
    lights: torch.Tensor,
    intensity: torch.Tensor,
    light_type: str = "point",
    light_size: Optional[float] = None,
    return_srgb: bool = True,
    multi_light: str = "per_light",
    loss_scale: Optional[float] = None,
    want_intensity_grad: bool = False,
    scratch: Optional[Dict[str, torch.Tensor]] = None,
    view_type: str = "directional",
) -> torch.Tensor:
    """
    Render + MSE + backward + Adam + projection in ONE kernel launch (pbr_ct_fit_step): the map gradients stay in
    registers and the optimiser's pass over parameters and moments rides along the shading kernel.  Numerically the
    same step as `fused_loss_step` followed by `optimizer.step(grads)`.

    The optimiser must own exactly the maps the kernel shades (albedo, roughness, metallic | specular, and normal
    if the material has one) - the very tensors stored in the material, contiguous, not batch-broadcast - with the
    default projection for all of them or none at all.  Anything else: use `fit_step(..., fused=False)`.
    The one-launch kernel shades with the view direction only: view_type="point" (a camera position) raises ValueError.
    Returns the device buffer [sum of squared errors, d_intensity(L*3)...] (not all-reduced).
    """
    _no_camera(view_type)
    lib = _cabi.load()
    cfg, (albedo, normal, roughness, metspec), _leaf, device = _prepare(
        material, material.device, view_dir, lights, intensity, light_type, light_size, return_srgb, multi_light
    )
    _cabi.require_cuda(target, "target")
    target = target.contiguous()
    expect = ((albedo.shape[0],) if cfg.batched else ()) + ((cfg.L,) if cfg.per_light else ()) + (3, *albedo.shape[-2:])
    if tuple(target.shape) != expect:
        raise ValueError(f"target has shape {tuple(target.shape)}, expected {expect}")
    if loss_scale is None:
        loss_scale = 1.0 / target.numel()
    met_name = "metallic" if cfg.workflow == _cabi.WORKFLOW_METALLIC else "specular"
    shaded = {"albedo": albedo, "roughness": roughness, met_name: metspec}
    if normal is not None:
        shaded["normal"] = normal
    if set(optimizer.params) != set(shaded):
        raise ValueError(f"fused_fit_step: the optimiser holds {sorted(optimizer.params)}, the kernel updates {sorted(shaded)}")
    kinds = set()
    for name, t in shaded.items():
        p = optimizer.params[name]
        if p.data_ptr() != t.data_ptr() or tuple(p.shape[-3:]) != tuple(t.shape[-3:]) or not t.is_contiguous():
            raise ValueError(f"fused_fit_step: {name} is updated in place and must be the optimiser's own contiguous tensor")
        pr, want = optimizer.project[name], DEFAULT_PROJECTION[name]
        kinds.add(None if pr is None else (pr[0] == want[0] and (pr[0] == "normalize" or tuple(pr[1:3]) == tuple(want[1:3]))))
    if kinds not in ({None}, {True}):
        raise ValueError("fused_fit_step: projection must be the default for every map or None for every map")
    scratch = scratch if scratch is not None else {}
    red = scratch.get("buf")
    if red is None or red.numel() != 1 + 3 * cfg.L:
        red = torch.empty(1 + 3 * cfg.L, dtype=torch.float32, device=device)
        scratch["buf"] = red
    red.zero_()
    keep: list = []
    d = _fill_desc(cfg, albedo, normal, roughness, metspec, keep)
    ls = _cabi.PbrCtLoss()
    ls.target, ls.target_sl = _out_plane(target, cfg.per_light, cfg.batched)
    ls.loss_scale = float(loss_scale)
    ls.loss_sum = red.data_ptr()
    t = optimizer.step_count + 1   # committed only once the launch has been accepted
    b1, b2 = optimizer.betas
    a = _cabi.PbrCtAdam()
    for key, name in (("albedo", "albedo"), ("normal", "normal"), ("roughness", "roughness"), ("metspec", met_name)):
        if name in optimizer.state:
            m, v = optimizer.state[name]
            setattr(a, "m_" + key, _cabi.plane(m))
            setattr(a, "v_" + key, _cabi.plane(v))
    a.step_size = optimizer.lr / (1.0 - b1 ** t)
    a.one_minus_beta1, a.beta2, a.one_minus_beta2 = 1.0 - b1, b2, 1.0 - b2
    a.bias2_sqrt = (1.0 - b2 ** t) ** 0.5
    a.eps = optimizer.eps
    a.project = 1 if kinds == {True} else 0
    d_int = ctypes.c_void_p(red[1:].data_ptr()) if want_intensity_grad else None
    with torch.cuda.device(device):
        _cabi.check(
            lib.pbr_ct_fit_step(_cabi.byref(d), _cabi.byref(ls), _cabi.byref(a), d_int, _cabi.stream_ptr(device)),
            "pbr_ct_fit_step",
        )
    _cabi.touch(*optimizer.params.values())
    optimizer.step_count = t
    return red


def fit_step(material: MaterialBase, optimizer: FusedAdam, target: torch.Tensor, view_dir, lights, intensity,
             light_type: str = "point", light_size: Optional[float] = None, multi_light: str = "per_light",
             scratch: Optional[Dict[str, torch.Tensor]] = None, global_numel: Optional[int] = None,
             fused: bool = False, async_loss: bool = False, timing: Optional[list] = None, view_type: str = "directional"):
    """
    One step of the sharded inverse-rendering fit on this rank's materials: fused render + MSE + backward
    (pbr_ct_loss_fwd_bwd), ONE all-reduce of the loss buffer, fused Adam + projection (pbr_adam_step).
    `fused=True`: all of it in one launch (pbr_ct_fit_step, see fused_fit_step); the all-reduce then only serves
    the reported loss.  With `async_loss=True` it therefore leaves the compute stream (allreduce_loss_async) and the
    call returns a PendingLoss; the loss buffers alternate between two slots of `scratch`, and a slot is only reused
    after its all-reduce of two steps ago has completed.
    `global_numel`: element count of the target over ALL ranks (the MSE denominator); default: this rank's.
    `view_type`: as CookTorranceBRDF's ("point": view_dir is the camera position); "point" needs fused=False.
    Returns the all-reduced buffer [sum of squared errors, ...] (device tensor; multiply [0] by 1/global_numel), or
    the PendingLoss that will deliver it.
    """
    numel = global_numel if global_numel is not None else target.numel()
    if fused:
        _no_camera(view_type)
        if async_loss:
            scratch = scratch if scratch is not None else {}
            ring = scratch.setdefault("loss_ring", [None, None])
            pend = scratch.setdefault("loss_pending", [None, None])
            i = scratch["loss_slot"] = 1 - scratch.get("loss_slot", 1)
            if pend[i] is not None:
                pend[i].wait()   # stream-level: the all-reduce of two steps ago, long finished
            scratch["buf"] = ring[i]
        buf = fused_fit_step(material, optimizer, target, view_dir, lights, intensity, light_type, light_size,
                             multi_light=multi_light, loss_scale=1.0 / numel, scratch=scratch)
        if async_loss:
            ring[i] = buf
            pend[i] = allreduce_loss_async(buf, scale=1.0 / numel, timing=timing)
            return pend[i]
        return allreduce_loss_and_shared(buf)
    buf, grads = fused_loss_step(material, target, view_dir, lights, intensity, light_type, light_size,
                                 multi_light=multi_light, loss_scale=1.0 / numel, out=scratch, view_type=view_type)
    allreduce_loss_and_shared(buf)
    optimizer.step({k: grads[k] for k in optimizer.params})
    return buf


class RenderingLoss(nn.Module):
    """
    The tutorial's RenderingLoss (06_advanced.rst:73-107) with the predicted render, the MSE and the
    backward pass fused in one kernel.  `forward(predicted_material, ground_truth_material)` returns the
    scalar loss; calling `.backward()` on it delivers the map gradients computed by that same launch.
    """

    def __init__(self, light_type="point", view_dir=torch.tensor([0.0, 0.0, 1.0]), light_dir=torch.tensor([0.1, 0.1, 1.0]),
                 light_intensity=torch.tensor([1.0, 1.0, 1.0]), light_size: Optional[float] = None,
                 view_type: str = "directional"):
        super().__init__()
        from .models import CookTorranceBRDF

        self.light_type = light_type
        self.brdf = CookTorranceBRDF(light_type=light_type, multi_light="per_light", view_type=view_type)
        self.view_type = self.brdf.view_type
        self.view_dir = view_dir
        self.light_dir = light_dir
        self.light_intensity = light_intensity
        self.light_size = light_size

    def forward(self, predicted_material: MaterialBase, ground_truth_material) -> torch.Tensor:
        if isinstance(ground_truth_material, torch.Tensor):
            target = ground_truth_material
        else:
            with torch.no_grad():
                target = self.brdf(ground_truth_material, self.view_dir, self.light_dir, self.light_intensity, self.light_size)
        names = [k for k in ("albedo", "normal", "roughness", "metallic", "specular")
                 if predicted_material._maps.get(k) is not None]
        leaves = [predicted_material._maps[k] for k in names]
        shared = [t if isinstance(t, torch.Tensor) else torch.as_tensor(t, dtype=torch.float32)
                  for t in (self.light_intensity, self.light_dir, self.view_dir)]
        grad_on = torch.is_grad_enabled()
        want_maps = grad_on and any(t.requires_grad for t in leaves)
        want_int = grad_on and shared[0].requires_grad
        want_geo = grad_on and (shared[1].requires_grad or shared[2].requires_grad)
        kw = dict(light_type=self.light_type, light_size=self.light_size, multi_light="per_light",
                  want_map_grads=want_maps, want_intensity_grad=want_int, want_geometry_grad=want_geo,
                  device=self.brdf.override_device, view_type=self.view_type)
        L = shared[1].shape[0] if shared[1].dim() == 2 else 1

        class _Fn(torch.autograd.Function):
            @staticmethod
            def forward(ctx, *inputs):
                red, grads = fused_loss_step(predicted_material, target, shared[2], shared[1], shared[0], **kw)
                # gradients come back in the shape the kernel shaded ((1,H,W) for an (H,W) map, a broadcast map expanded to
                # the batch): reduce them onto the leaves' own shapes
                ctx.grads = [grads[k].sum_to_size(t.shape) if (want_maps and grads.get(k) is not None) else None
                             for k, t in zip(names, leaves)]
                red = red.detach()
                g_int = red[1:1 + 3 * L].view(L, 3) if want_int else None
                g_light = red[1 + 3 * L:1 + 6 * L].view(L, 3) if want_geo else None
                g_view = red[1 + 6 * L:1 + 6 * L + 3] if want_geo else None
                def onto(g, t):   # (L,3) rows onto a (3,) or (L,3) leaf; (3,) onto any 3-element view tensor
                    if g is None:
                        return None
                    g = g.reshape(t.shape) if g.numel() == t.numel() else g.sum_to_size(t.shape)
                    return g.to(t.device)

                ctx.shared = [onto(g, t) for g, t in zip((g_int, g_light, g_view), shared)]
                return red[0] / target.numel()

            @staticmethod
            def backward(ctx, g):
                maps = tuple((gr * g if gr is not None else None) for gr in ctx.grads)
                sh = tuple((gr * g.to(gr.device) if gr is not None else None) for gr in ctx.shared)
                return maps + sh

        return _Fn.apply(*leaves, *shared)
