"""Per-material view, lights and intensities without a GPU: the shapes the host layer accepts and refuses, and the argument
errors of the pbr_ct_*_pb entry points, which come back before any launch."""
import ctypes

import pytest
import torch

from pypbr_b200 import _cabi
from pypbr_b200.models.cooktorrance import _parse_params

PM = ("intensity", "lights", "view")


def parse(view, lights, inten, B=4, batched=True):
    v, l, i, multi, pm = _parse_params(view, lights, inten, B, batched)
    return v, l, i, multi, {k for k, on in zip(PM, pm) if on}


V3, L1 = torch.tensor([0.0, 0.1, 1.0]), torch.tensor([0.2, 0.1, 1.0])


def test_shared_shapes_keep_their_meaning():
    v, l, i, multi, pm = parse(V3, L1, torch.ones(3))
    assert (tuple(l.shape), tuple(i.shape), multi, pm) == ((1, 3), (1, 3), False, set())
    # a 2-D (B, 3) intensity is still (L, 3): here L = 4 lights
    v, l, i, multi, pm = parse(V3, torch.rand(4, 3), torch.rand(4, 3))
    assert (tuple(l.shape), tuple(i.shape), multi, pm) == ((4, 3), (4, 3), True, set())
    _, l, i, _, _ = parse(V3, torch.rand(4, 3), torch.rand(1, 3))
    assert tuple(i.shape) == (4, 3)
    # any 3-element view is one view, a (1, 3) one included
    for view in (V3, V3.view(1, 3), V3.view(3, 1), [0.0, 0.0, 1.0]):
        assert parse(view, L1, torch.ones(3))[4] == set()


def test_per_material_shapes():
    B, L = 4, 3
    v, l, i, multi, pm = parse(torch.rand(B, 3), torch.rand(B, L, 3), torch.rand(B, L, 3), B=B)
    assert (tuple(v.shape), tuple(l.shape), tuple(i.shape), multi, pm) == ((B, 3), (B, L, 3), (B, L, 3), True, set(PM))
    # (B, 1, 3) intensities are broadcast over the lights
    _, _, i, _, pm = parse(V3, torch.rand(B, L, 3), torch.rand(B, 1, 3), B=B)
    assert tuple(i.shape) == (B, L, 3) and pm == {"intensity", "lights"}
    # (1, L, 3) is shared, and counts as several lights even for L = 1
    _, l, i, multi, pm = parse(torch.rand(B, 3), torch.rand(1, 1, 3), torch.rand(1, 1, 3), B=B)
    assert (tuple(l.shape), tuple(i.shape), multi, pm) == ((1, 3), (1, 3), True, {"view"})
    # each parameter on its own: per-material intensities with shared lights
    _, l, i, _, pm = parse(V3, torch.rand(L, 3), torch.rand(B, L, 3), B=B)
    assert (tuple(l.shape), tuple(i.shape), pm) == ((L, 3), (B, L, 3), {"intensity"})
    # unbatched maps take a leading dimension of 1
    _, _, _, multi, pm = parse(V3, torch.rand(1, 2, 3), torch.rand(1, 2, 3), B=1, batched=False)
    assert multi and pm == set()


@pytest.mark.parametrize("args, match", [
    ((torch.rand(3, 3), L1, torch.ones(3)), "view_dir has 3 parameter sets for a batch of 4"),
    ((V3, torch.rand(2, 1, 3), torch.ones(3)), "light_dir_or_position has 2 parameter sets"),
    ((V3, L1, torch.rand(5, 1, 3)), "light_intensity has 5 parameter sets"),
    ((V3, torch.rand(4, 2, 3), torch.rand(4, 3, 3)), "light_intensity has 3 rows for 2 lights"),
    ((V3, torch.rand(4, 2, 3), torch.rand(3, 3)), "light_intensity has 3 rows for 2 lights"),
    ((V3, torch.rand(4, 65, 3), torch.ones(3)), "at most 64 lights"),
    ((V3, torch.rand(1, 65, 3), torch.ones(3)), "at most 64 lights"),
    ((torch.rand(4, 4), L1, torch.ones(3)), r"view_dir must have shape \(3,\) or \(B, 3\)"),
    ((torch.rand(4, 3, 1), L1, torch.ones(3)), r"view_dir must have shape"),
    ((V3, torch.rand(4, 2, 2), torch.ones(3)), r"must have shape \(3,\), \(L, 3\) or \(B, L, 3\)"),
    ((V3, torch.rand(1, 4, 2, 3), torch.ones(3)), r"must have shape"),
])
def test_bad_shapes_raise(args, match):
    with pytest.raises(ValueError, match=match):
        _parse_params(*args, 4, True)


@pytest.mark.parametrize("args", [
    (torch.rand(2, 3), L1, torch.ones(3)),
    (V3, torch.rand(2, 1, 3), torch.ones(3)),
    (V3, L1, torch.rand(2, 1, 3)),
])
def test_per_material_parameters_need_batched_maps(args):
    with pytest.raises(ValueError, match="need batched"):
        _parse_params(*args, 1, False)


def test_param_batch_struct_layout():
    assert ctypes.sizeof(_cabi.PbrCtParamBatch) == 2 * 4 + 3 * 8
    assert _cabi.STRUCTS.index(_cabi.PbrCtParamBatch) == 20
    assert _cabi.load().pbr_sizeof(20) == ctypes.sizeof(_cabi.PbrCtParamBatch)


_HOST = (ctypes.c_float * (3 * 65))()


def _desc(L=2, B=3, on_device=1):
    fake = 0x1000   # never dereferenced: argument checks only
    d = _cabi.PbrCtDesc()
    d.B, d.H, d.W, d.L = B, 4, 4, L
    for pl in ("albedo", "roughness", "metspec", "out"):
        setattr(d, pl, _cabi.PbrPlane(fake, 48, 16, 4))
    # host parameters are copied into the launch by the argument checks: they must be readable
    d.view = d.lights = d.intensity = ctypes.cast(_HOST, ctypes.c_void_p) if not on_device else fake
    d.params_on_device = on_device
    return d


def _calls(lib, d, pb):
    """Every _pb entry point on descriptors that pass their own checks (a NULL stream: nothing may be launched)."""
    fake = 0x1000
    g = _cabi.PbrCtGrads()
    g.grad_out = _cabi.PbrPlane(fake, 48, 16, 4)
    ls = _cabi.PbrCtLoss()
    ls.target, ls.loss_sum = _cabi.PbrPlane(fake, 48, 16, 4), fake
    a = _cabi.PbrCtAdam()
    for f in ("m_albedo", "v_albedo", "m_roughness", "v_roughness", "m_metspec", "v_metspec"):
        setattr(a, f, _cabi.PbrPlane(fake, 48, 16, 4))
    pbp = ctypes.byref(pb) if pb is not None else None
    return {
        "forward": lib.pbr_ct_forward_pb(ctypes.byref(d), pbp, None),
        "backward": lib.pbr_ct_backward_pb(ctypes.byref(d), pbp, ctypes.byref(g), None),
        "loss": lib.pbr_ct_loss_fwd_bwd_pb(ctypes.byref(d), pbp, ctypes.byref(ls), ctypes.byref(g), None),
        "fit": lib.pbr_ct_fit_step_pb(ctypes.byref(d), pbp, ctypes.byref(ls), ctypes.byref(a), None, None),
    }


def test_param_batch_argument_errors_come_back_before_any_launch():
    lib = _cabi.load()
    launches = _cabi.launch_count()
    pb = _cabi.PbrCtParamBatch(0, 0, 3, 6, 6)
    assert lib.pbr_ct_forward_pb(None, ctypes.byref(pb), None) == -1          # NULL descriptor
    assert lib.pbr_ct_backward_pb(None, ctypes.byref(pb), None, None) == -1
    assert lib.pbr_ct_loss_fwd_bwd_pb(None, ctypes.byref(pb), None, None, None) == -1
    assert lib.pbr_ct_fit_step_pb(None, ctypes.byref(pb), None, None, None, None) == -1
    assert set(_calls(lib, _desc(), None).values()) == {-1}                    # NULL parameter batch
    assert set(_calls(lib, _desc(on_device=0), pb).values()) == {-3}           # per-material strides need device parameters
    for bad in (_cabi.PbrCtParamBatch(0, 0, 2, 0, 0), _cabi.PbrCtParamBatch(0, 0, 0, 5, 0),
                _cabi.PbrCtParamBatch(0, 0, 0, 0, 3), _cabi.PbrCtParamBatch(0, 0, -3, 0, 0)):
        assert set(_calls(lib, _desc(L=2), bad).values()) == {-2}              # a stride below 3 (view) or 3L
    assert set(_calls(lib, _desc(), _cabi.PbrCtParamBatch(2, 0, 0, 0, 0)).values()) == {-3}   # camera is 0 or 1
    # the one-launch fit step has no camera; the other three take it
    rc = _calls(lib, _desc(L=65), _cabi.PbrCtParamBatch(1, 0, 0, 0, 0))
    assert set(rc.values()) == {-4}                                            # the descriptor's own checks come first
    d = _desc()
    d.view = None
    assert set(_calls(lib, d, _cabi.PbrCtParamBatch(1, 0, 3, 0, 0)).values()) == {-1}
    assert lib.pbr_ct_fit_step_pb(ctypes.byref(_desc()), ctypes.byref(_cabi.PbrCtParamBatch(1, 0, 0, 0, 0)),
                                  None, None, None, None) == -3
    assert _cabi.launch_count() == launches
