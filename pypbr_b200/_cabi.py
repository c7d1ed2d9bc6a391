"""
pypbr_b200._cabi — ctypes binding of libpbrcuda.so (include/pbrcuda.h).

This is the only place the package touches native code.  There is NO fallback: if the shared library
is missing or a tensor is not a CUDA float32 tensor, the call raises.  PyTorch is used for device
memory, streams and autograd plumbing only; every per-texel operation of the hot path runs in the
kernels behind these entry points.
"""

from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, byref, c_char_p, c_float, c_int, c_int32, c_int64, c_uint64, c_void_p
from typing import Optional, Sequence

import torch

ABI_VERSION = 5
PBR_MAX_LIGHTS = 64
PBR_MAX_BLEND_MAPS = 12
PBR_MAX_INDEX_MAPS = 12
PBR_MAX_ADAM_MAPS = 8

WORKFLOW_METALLIC, WORKFLOW_SPECULAR = 0, 1
LIGHT_DIRECTIONAL, LIGHT_POINT = 0, 1
MASK_GIVEN, MASK_SIGMOID, MASK_GRADIENT_H, MASK_GRADIENT_V = 0, 1, 2, 3
INGEST_PLAIN, INGEST_NORMAL3, INGEST_NORMAL2 = 0, 1, 2
PROJECT_NONE, PROJECT_CLAMP, PROJECT_NORMALIZE = 0, 1, 2

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libpbrcuda.so")


class PbrPlane(Structure):
    _fields_ = [("ptr", c_void_p), ("sb", c_int64), ("sc", c_int64), ("sh", c_int64)]


class PbrCtDesc(Structure):
    _fields_ = [
        ("B", c_int32), ("H", c_int32), ("W", c_int32), ("L", c_int32),
        ("workflow", c_int32), ("light_type", c_int32),
        ("albedo_is_srgb", c_int32), ("specular_is_srgb", c_int32), ("return_srgb", c_int32),
        ("per_light", c_int32), ("params_on_device", c_int32),
        ("light_size", c_float),
        ("albedo", PbrPlane), ("normal", PbrPlane), ("roughness", PbrPlane), ("metspec", PbrPlane),
        ("metallic_channels", c_int32),
        ("view", c_void_p), ("lights", c_void_p), ("intensity", c_void_p),
        ("out", PbrPlane), ("out_sl", c_int64),
        ("force_generic", c_int32),
    ]


class PbrCtGrads(Structure):
    _fields_ = [
        ("grad_out", PbrPlane), ("grad_out_sl", c_int64),
        ("d_albedo", PbrPlane), ("d_normal", PbrPlane), ("d_roughness", PbrPlane), ("d_metspec", PbrPlane),
        ("d_intensity", c_void_p), ("d_lights", c_void_p), ("d_view", c_void_p),
        ("fwd_out", PbrPlane),
    ]


class PbrCtLoss(Structure):
    _fields_ = [("target", PbrPlane), ("target_sl", c_int64), ("loss_scale", c_float), ("loss_sum", c_void_p)]


class PbrCtParamBatch(Structure):
    _fields_ = [("camera", c_int32), ("pad", c_int32), ("view_sb", c_int64), ("lights_sb", c_int64), ("intensity_sb", c_int64)]


class PbrConvDesc(Structure):
    _fields_ = [
        ("B", c_int32), ("H", c_int32), ("W", c_int32), ("albedo_is_srgb", c_int32),
        ("albedo", PbrPlane), ("metspec", PbrPlane), ("out0", PbrPlane), ("out1", PbrPlane),
        ("metallic_channels", c_int32),
    ]


class PbrConvGrads(Structure):
    _fields_ = [("g_out0", PbrPlane), ("g_out1", PbrPlane), ("d_albedo", PbrPlane), ("d_metspec", PbrPlane)]


class PbrBlendMap(Structure):
    _fields_ = [("a", PbrPlane), ("b", PbrPlane), ("out", PbrPlane), ("channels", c_int32), ("is_normal", c_int32)]


class PbrBlendDesc(Structure):
    _fields_ = [
        ("B", c_int32), ("H", c_int32), ("W", c_int32), ("n_maps", c_int32), ("mask_mode", c_int32),
        ("blend_width", c_float), ("shift", c_float), ("apply_shift", c_int32),
        ("mask", PbrPlane), ("prop1", PbrPlane), ("prop2", PbrPlane), ("mask_out", PbrPlane),
        ("normal_min", c_void_p),
        ("maps", PbrBlendMap * PBR_MAX_BLEND_MAPS),
    ]


class PbrBlendGradMap(Structure):
    _fields_ = [("g_out", PbrPlane), ("d_a", PbrPlane), ("d_b", PbrPlane)]


class PbrBlendGrads(Structure):
    _fields_ = [
        ("mask", PbrPlane), ("g_mask_out", PbrPlane), ("d_mask", PbrPlane), ("d_prop1", PbrPlane), ("d_prop2", PbrPlane),
        ("maps", PbrBlendGradMap * PBR_MAX_BLEND_MAPS),
    ]


class PbrColorDesc(Structure):
    _fields_ = [
        ("B", c_int32), ("C", c_int32), ("H", c_int32), ("W", c_int32), ("to_linear", c_int32),
        ("in_", PbrPlane), ("out", PbrPlane),
    ]


class PbrNormalDesc(Structure):
    _fields_ = [("B", c_int32), ("H", c_int32), ("W", c_int32), ("channels", c_int32), ("in_", PbrPlane), ("out", PbrPlane),
                ("cond_min", c_void_p)]


class PbrNormalGrads(Structure):
    _fields_ = [("g_out", PbrPlane), ("d_in", PbrPlane)]


class PbrIngestDesc(Structure):
    _fields_ = [
        ("B", c_int32), ("H", c_int32), ("W", c_int32), ("bits", c_int32), ("src_channels", c_int32),
        ("channels", c_int32), ("mode", c_int32),
        ("src", c_void_p), ("src_batch_stride", c_int64), ("src_row_stride", c_int64),
        ("out", PbrPlane),
    ]


class PbrIndexMap(Structure):
    _fields_ = [("in_", PbrPlane), ("out", PbrPlane), ("channels", c_int32), ("negate_mask", c_int32)]


class PbrIndexDesc(Structure):
    _fields_ = [
        ("B", c_int32), ("H_in", c_int32), ("W_in", c_int32), ("H_out", c_int32), ("W_out", c_int32),
        ("origin_y", c_int32), ("step_y", c_int32), ("origin_x", c_int32), ("step_x", c_int32),
        ("wrap", c_int32), ("n_maps", c_int32), ("reduce_y", c_int32), ("reduce_x", c_int32),
        ("maps", PbrIndexMap * PBR_MAX_INDEX_MAPS),
    ]


class PbrAdamMap(Structure):
    _fields_ = [
        ("param", PbrPlane), ("grad", PbrPlane), ("exp_avg", PbrPlane), ("exp_avg_sq", PbrPlane),
        ("channels", c_int32), ("project", c_int32), ("lo", c_float), ("hi", c_float),
    ]


class PbrAdamDesc(Structure):
    _fields_ = [
        ("B", c_int32), ("H", c_int32), ("W", c_int32), ("n_maps", c_int32),
        ("step_size", c_float), ("one_minus_beta1", c_float), ("beta2", c_float), ("one_minus_beta2", c_float),
        ("bias2_sqrt", c_float), ("eps", c_float), ("grad_scale", c_float),
        ("maps", PbrAdamMap * PBR_MAX_ADAM_MAPS),
    ]


class PbrCtAdam(Structure):
    _fields_ = [
        ("m_albedo", PbrPlane), ("v_albedo", PbrPlane), ("m_normal", PbrPlane), ("v_normal", PbrPlane),
        ("m_roughness", PbrPlane), ("v_roughness", PbrPlane), ("m_metspec", PbrPlane), ("v_metspec", PbrPlane),
        ("step_size", c_float), ("one_minus_beta1", c_float), ("beta2", c_float), ("one_minus_beta2", c_float),
        ("bias2_sqrt", c_float), ("eps", c_float), ("project", c_int32),
    ]


class PbrNormalOpDesc(Structure):
    _fields_ = [
        ("B", c_int32), ("H", c_int32), ("W", c_int32), ("op", c_int32),
        ("cos_a", c_float), ("sin_a", c_float), ("scale", c_float), ("flip_y", c_int32),
        ("in_", PbrPlane), ("out", PbrPlane), ("aux", PbrPlane),
    ]


NORMAL_OP_ROTATE, NORMAL_OP_FROM_HEIGHT, NORMAL_OP_DIVERGENCE, NORMAL_OP_FROM_HEIGHT_BWD = 0, 1, 2, 3
NORMAL_OP_ROTATE_BWD, NORMAL_OP_DIVERGENCE_BWD = 4, 5

# order = the `which` argument of pbr_sizeof()
STRUCTS = (PbrPlane, PbrCtDesc, PbrCtGrads, PbrCtLoss, PbrConvDesc, PbrBlendMap, PbrBlendDesc, PbrColorDesc, PbrNormalDesc,
           PbrIngestDesc, PbrIndexMap, PbrIndexDesc, PbrAdamMap, PbrAdamDesc, PbrCtAdam, PbrNormalOpDesc,
           PbrConvGrads, PbrBlendGradMap, PbrBlendGrads, PbrNormalGrads, PbrCtParamBatch)

_lib = None

# every symbol include/pbrcuda.h declares (tests check that the built library exports all of them)
EXPORTS = (
    "pbr_abi_version", "pbr_strerror", "pbr_ct_forward", "pbr_ct_backward", "pbr_ct_loss_fwd_bwd", "pbr_ct_fit_step",
    "pbr_convert_m2s", "pbr_convert_s2m", "pbr_blend", "pbr_color_convert", "pbr_normal_min",
    "pbr_normal_ingest", "pbr_ingest_image", "pbr_index_transform", "pbr_adam_step", "pbr_normal_op", "pbr_launch_count", "pbr_sizeof",
    "pbr_convert_m2s_backward", "pbr_convert_s2m_backward", "pbr_blend_backward", "pbr_normal_ingest_backward",
    "pbr_ct_forward_camera", "pbr_ct_backward_camera", "pbr_ct_loss_fwd_bwd_camera",
    "pbr_ct_forward_pb", "pbr_ct_backward_pb", "pbr_ct_loss_fwd_bwd_pb", "pbr_ct_fit_step_pb",
)


def lib_path() -> str:
    return _LIB_PATH


def load():
    """Load libpbrcuda.so (once).  Raises ImportError if it was not built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise ImportError(
            f"pypbr_b200: native library not found at {_LIB_PATH}. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
            "There is no CPU or PyTorch fallback for the shading path."
        )
    lib = ctypes.CDLL(_LIB_PATH)
    lib.pbr_abi_version.restype = c_int
    lib.pbr_strerror.restype = c_char_p
    lib.pbr_strerror.argtypes = [c_int]
    lib.pbr_launch_count.restype = c_uint64
    lib.pbr_sizeof.restype = c_uint64
    lib.pbr_sizeof.argtypes = [c_int]
    lib.pbr_ct_forward.argtypes = [POINTER(PbrCtDesc), c_void_p]
    lib.pbr_ct_backward.argtypes = [POINTER(PbrCtDesc), POINTER(PbrCtGrads), c_void_p]
    lib.pbr_ct_loss_fwd_bwd.argtypes = [POINTER(PbrCtDesc), POINTER(PbrCtLoss), POINTER(PbrCtGrads), c_void_p]
    lib.pbr_ct_fit_step.argtypes = [POINTER(PbrCtDesc), POINTER(PbrCtLoss), POINTER(PbrCtAdam), c_void_p, c_void_p]
    lib.pbr_ct_forward_camera.argtypes = [POINTER(PbrCtDesc), c_void_p]
    lib.pbr_ct_backward_camera.argtypes = [POINTER(PbrCtDesc), POINTER(PbrCtGrads), c_void_p]
    lib.pbr_ct_loss_fwd_bwd_camera.argtypes = [POINTER(PbrCtDesc), POINTER(PbrCtLoss), POINTER(PbrCtGrads), c_void_p]
    lib.pbr_ct_forward_pb.argtypes = [POINTER(PbrCtDesc), POINTER(PbrCtParamBatch), c_void_p]
    lib.pbr_ct_backward_pb.argtypes = [POINTER(PbrCtDesc), POINTER(PbrCtParamBatch), POINTER(PbrCtGrads), c_void_p]
    lib.pbr_ct_loss_fwd_bwd_pb.argtypes = [POINTER(PbrCtDesc), POINTER(PbrCtParamBatch), POINTER(PbrCtLoss), POINTER(PbrCtGrads),
                                           c_void_p]
    lib.pbr_ct_fit_step_pb.argtypes = [POINTER(PbrCtDesc), POINTER(PbrCtParamBatch), POINTER(PbrCtLoss), POINTER(PbrCtAdam),
                                       c_void_p, c_void_p]
    lib.pbr_convert_m2s.argtypes = [POINTER(PbrConvDesc), c_void_p]
    lib.pbr_convert_s2m.argtypes = [POINTER(PbrConvDesc), c_void_p]
    lib.pbr_blend.argtypes = [POINTER(PbrBlendDesc), c_void_p]
    lib.pbr_convert_m2s_backward.argtypes = [POINTER(PbrConvDesc), POINTER(PbrConvGrads), c_void_p]
    lib.pbr_convert_s2m_backward.argtypes = [POINTER(PbrConvDesc), POINTER(PbrConvGrads), c_void_p]
    lib.pbr_blend_backward.argtypes = [POINTER(PbrBlendDesc), POINTER(PbrBlendGrads), c_void_p]
    lib.pbr_normal_ingest_backward.argtypes = [POINTER(PbrNormalDesc), POINTER(PbrNormalGrads), c_void_p]
    lib.pbr_color_convert.argtypes = [POINTER(PbrColorDesc), c_void_p]
    lib.pbr_normal_min.argtypes = [POINTER(PbrNormalDesc), c_void_p, c_void_p]
    lib.pbr_normal_ingest.argtypes = [POINTER(PbrNormalDesc), c_void_p]
    lib.pbr_ingest_image.argtypes = [POINTER(PbrIngestDesc), c_void_p]
    lib.pbr_index_transform.argtypes = [POINTER(PbrIndexDesc), c_void_p]
    lib.pbr_adam_step.argtypes = [POINTER(PbrAdamDesc), c_void_p]
    lib.pbr_normal_op.argtypes = [POINTER(PbrNormalOpDesc), c_void_p]
    for name in EXPORTS:
        fn = getattr(lib, name)
        if name not in ("pbr_strerror", "pbr_launch_count", "pbr_sizeof"):
            fn.restype = c_int
    if lib.pbr_abi_version() != ABI_VERSION:
        raise ImportError(f"pypbr_b200: ABI version mismatch in {_LIB_PATH}")
    for which, st in enumerate(STRUCTS):
        if lib.pbr_sizeof(which) != ctypes.sizeof(st):
            raise ImportError(f"pypbr_b200: layout of {st.__name__} differs between _cabi.py and {_LIB_PATH}")
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().pbr_strerror(rc).decode()
        raise RuntimeError(f"pypbr_b200: {what} failed: {msg} (code {rc})")


def launch_count() -> int:
    return int(load().pbr_launch_count())


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t)}")
    if not t.is_cuda:
        raise RuntimeError(
            f"pypbr_b200: {name} lives on {t.device}; the shading path runs on CUDA only (no CPU fallback). "
            "Move the material with material.to('cuda') or construct CookTorranceBRDF(override_device='cuda')."
        )
    if t.dtype != torch.float32:
        raise TypeError(f"pypbr_b200: {name} must be float32, got {t.dtype}")


def rowmajor(t: torch.Tensor) -> torch.Tensor:
    """The kernels need unit stride along W; everything else is expressed through strides."""
    return t if (t.stride(-1) == 1 or t.shape[-1] == 1) else t.contiguous()


def plane(t: Optional[torch.Tensor]) -> PbrPlane:
    """(C,H,W) or (B,C,H,W) tensor -> PbrPlane (strides in elements).  None -> NULL plane."""
    if t is None:
        return PbrPlane(None, 0, 0, 0)
    st = t.stride()
    n = len(st)
    assert st[-1] == 1 or t.shape[-1] == 1, "call rowmajor() first"
    if n == 3:
        return PbrPlane(t.data_ptr(), 0, st[0], st[1])
    if n == 4:
        return PbrPlane(t.data_ptr(), st[0], st[1], st[2])
    raise ValueError(f"maps must be (C,H,W) or (B,C,H,W), got shape {tuple(t.shape)}")


class device_guard:
    """`with torch.cuda.device(dev)` only when `dev` is not already current (the context manager costs ~5 us per entry,
    a tenth of a small-image call)."""

    __slots__ = ("ctx",)

    def __init__(self, dev: torch.device):
        idx = dev.index
        self.ctx = None if (idx is None or idx == torch.cuda.current_device()) else torch.cuda.device(dev)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *a):
        if self.ctx is not None:
            self.ctx.__exit__(*a)


def touch(*tensors) -> None:
    """A kernel has written these tensors IN PLACE through their raw pointers: bump torch's version counter, so that
    autograd notices a modified saved tensor and the memoised normal-map probe (materials/base.py) is invalidated."""
    for t in tensors:
        if t is not None:
            torch.autograd.graph.increment_version(t)


def stream_ptr(device: torch.device) -> c_void_p:
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def host_floats(values: Sequence[float]):
    arr = (c_float * len(values))(*values)
    return arr
