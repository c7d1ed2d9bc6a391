"""
The Cook-Torrance math at the edges of its inputs, on the CPU: the device math headers compiled for the host (hostsim)
against the oracle, on an "edge atlas" - a deterministic material whose texels sit on the non-smooth points of the
reference's op chain - under "edge lightings" that put the light and the view on those points too.

The rest of the suite draws its inputs from one benign distribution (roughness in [0.2, 1], unit normals near +z, maps in
[0, 1], lights above the plane), where N.L, N.V, N.H and h.v almost never reach a clamp.  The kernels' gates (the
inclusive clamp gates rebuilt by `gated()`, the saturating adds and multiplies, the normalize eps branches, the seeded
reciprocals of the point-light geometry) are written for exactly the points this file visits.  Such inputs also occur in
real use: a crop past the border pads with zero maps, FusedAdam(project=None) lets maps leave [0, 1], and a low light
sits on or just above the plane.

The atlas (`edge_atlas`): CATEGORIES lists the texels, each a labelled set of map values exactly at a singular point or one
fp32 ulp either side of it.  The material repeats the list in row-major order (rows padded to an even length); the list's
length is odd, so every category falls on both lanes of a texel pair, and tiled to a kernel's (B, H, W) it reaches full 4-texel and 512-texel tiles.
Lightings (`point_lightings`, `dir_lightings`, `cameras`): the light and the view on +z (N.L = N.V = N.H = h.v = 1 on the
(0, 0, 1) normal), a directional light opposite the view (h has zero length), point lights at z = 0, 1e-7, 1e-6 and
1e-4 above a texel centre (exact plane coordinates taken from the grid, so d is exactly z there), a point light below the
plane, a zero-intensity and a saturating light in accumulate mode, and for the camera at a finite position, a camera on
the plane at a texel centre and one directly above a texel.

Comparison rules (`check_forward`, `check_map_grad`, `check_shared`, `check_finite`), shared with tests/test_gpu_edges.py:
  * forward: conftest.fwd_ok against the fp32 oracle, or per texel the fp64 arbiter |y - y64| <= max(2 |y32 - y64|, tol);
  * map gradients: conftest.grad_ok applied per atlas category (the 1e-4 mean|g| term is the category's own mean: one
    1e12 eps-branch gradient would otherwise widen the tolerance of every other texel), but no tighter than grad_ok over
    the texels off the eps branch (EPS_CATS).  A category can be all cancellation, where no fp32 evaluation order is
    within rel 1e-4 of another: at the grazing normal N.V ~ 1e-3, d/d N.V is a difference of two terms ~1/N.V.  Then
    the fp64 arbiter per texel, |g - g64| <= 2 |g32 - g64| + tol: where the fp32 and fp64 oracles fall on different
    sides of a gate it accepts either side, and those texels are listed in the failure message.  One more cancellation
    gets 10x the tolerance, and only where it occurs: at roughness -1 (K0_CATS, k = 0) d/d roughness is the a2 path
    alone, weighted (1 - 2 N.H^2), and a light in the plane (`in_plane`) makes N.H^2 ~ 1/2 on the +z normal - the
    gradient is ~1e-7 of O(1) terms, and the fp32 oracle is 30 % off its fp64 run there;
  * shared-parameter gradients (sums over the image): 1e-4 |g| + 1e-4 mean|g| of the fp64 oracle, as in the kernel
    ledger, or per element the same fp64 arbiter.  The arbiter is what a camera ON the plane needs: on the camera's own
    row the view is exactly (-+1, 0, 0), and a point light 1e-6 above that row, across the camera, makes l the view's
    near-opposite; h = normalize(v + l) then normalizes a sum whose horizontal part, ~1e-7 / d, is one fp32 ulp of the
    parts it cancels, so its direction is set by rounding.  The fp32 oracle's d_intensity / d_lights are up to 200x the
    tolerance off its fp64 run there (4 x 40; the 9 x 9 atlas puts no texel on that row between them), and the kernels
    agree with the fp32 oracle to 1e-2 of the tolerance - the light = -view edge, approached continuously;
  * finiteness: wherever the fp32 oracle is finite, the image, every map gradient, the loss and d_intensity / d_lights /
    d_view are finite.
Known difference, not tested: NaN / Inf INPUTS.  The kernels clamp with saturating instructions, which map NaN to 0,
where torch propagates it.
"""
import ctypes

import numpy as np
import pytest
import torch

from conftest import fwd_ok

F32 = np.float32
WFS = {"metallic": 0, "specular": 1, "metallic3": 2}
SHARED = ("intensity", "lights", "view")


def _up(x):
    return float(np.nextafter(F32(x), F32(np.inf)))


def _dn(x):
    return float(np.nextafter(F32(x), F32(-np.inf)))


# ---------------------------------------------------------------------------------------------- the edge atlas
# A benign texel, and per category the values that differ from it.  "n": raw normal (the kernels normalize it, as the
# reference does), "r": roughness, "m": metallic (metallic workflows) / "s": specular (specular workflow), "a": albedo.
BASE = dict(a=(0.6, 0.45, 0.3), n=(0.1, -0.05, 0.99), r=0.5, m=0.4, s=(0.3, 0.25, 0.2))
_K = 0.04045   # the sRGB decode knee
CATEGORIES = [
    ("base", {}),
    # normals: the upper gate (N.L = N.V = N.H = h.v = 1 under the +z light and view) and one ulp either side
    ("n_up", dict(n=(0.0, 0.0, 1.0))),
    ("n_up+ulp", dict(n=(0.0, 0.0, _up(1.0)))),
    ("n_up-ulp", dict(n=(0.0, 0.0, _dn(1.0)))),
    ("n_up_r0", dict(n=(0.0, 0.0, 1.0), r=0.0)),          # N.H = 1 and a2 = 0: the GGX denominator is 1e-7 alone
    ("n_up_r-1", dict(n=(0.0, 0.0, 1.0), r=-1.0)),
    # the lower gate (N.L = 0 under +z) and one step of z either side
    ("n_side", dict(n=(1.0, 0.0, 0.0))),
    ("n_side+", dict(n=(1.0, 0.0, 6e-8))),
    ("n_side-", dict(n=(1.0, 0.0, -6e-8))),
    ("n_down", dict(n=(0.0, 0.0, -1.0))),                 # below the horizon
    ("n_raw2", dict(n=(0.0, 0.0, 2.0))),                  # raw, not unit
    ("n_raw34", dict(n=(0.3, 0.0, 0.4))),
    ("n_zero", dict(n=(0.0, 0.0, 0.0))),                  # F.normalize's eps branch: gradients ~ 1e12
    ("n_tiny", dict(n=(0.0, 0.0, 1e-13))),
    ("n_tiny_xz", dict(n=(6e-14, 0.0, 8e-14))),
    ("n_graze", dict(n=(1.0, 0.0, 1e-3))),
    # roughness: the reference does not clamp it; at -1, k = (r + 1)^2 / 8 = 0
    ("r0", dict(r=0.0)),
    ("r1", dict(r=1.0)),
    ("r1.5", dict(r=1.5)),
    ("r-0.3", dict(r=-0.3)),
    ("r-1", dict(r=-1.0)),
    # metallic / specular, in and out of [0, 1]
    ("m0", dict(m=0.0, s=(0.0, 0.0, 0.0))),
    ("m1", dict(m=1.0, s=(1.0, 1.0, 1.0))),
    ("m-0.2", dict(m=-0.2, s=(1.2, 1.2, 1.2))),
    ("m1.3", dict(m=1.3, s=(1.0, 0.0, 1.2))),
    # albedo: the decode's input clamp gates (0 and 1 inclusive) and the knee with its neighbours
    ("a0", dict(a=(0.0, 0.0, 0.0))),
    ("a_knee", dict(a=(_K, _K, _K))),
    ("a_knee+", dict(a=(_up(_K), _up(_K), _up(_K)))),
    ("a_knee-", dict(a=(_dn(_K), _dn(_K), _dn(_K)))),
    ("a1", dict(a=(1.0, 1.0, 1.0))),
    ("a1-ulp", dict(a=(_dn(1.0), _dn(1.0), _dn(1.0)))),
    ("a_out", dict(a=(1.2, -0.1, 1.2))),
    ("a_out2", dict(a=(-0.1, 1.2, _up(0.0)))),
    # a crop past the border: every map zero
    ("zero_pad", dict(a=(0.0, 0.0, 0.0), n=(0.0, 0.0, 0.0), r=0.0, m=0.0, s=(0.0, 0.0, 0.0))),
    ("mix_out", dict(a=(1.2, 1.0, 0.0), n=(0.3, 0.0, 0.4), r=1.5, m=1.3, s=(1.2, 1.0, 0.0))),
]
# roughness -1: k = 0, so d/d roughness is the a2 path alone, 2 r (1 - 2 N.H^2) D' - a cancellation near N.H^2 = 1/2 (the +z
# normal under a light in the plane) that the kernels' MUFU reciprocals resolve to ~3x grad_ok's tolerance on the B200
K0_CATS = [i for i, (name, _) in enumerate(CATEGORIES) if name in ("r-1", "n_up_r-1")]


def in_plane(light_type, lights):
    """Whether a light lies in the plane or within 1e-4 above it, seen from most texels edge-on: h then makes N.H^2 ~ 1/2
    with the +z normal, the cancellation of K0_CATS (check_map_grad's light_in_plane)."""
    p = np.asarray(lights, np.float64).reshape(-1, 3)
    if light_type == "point":
        return bool(((p[:, 2] >= 0) & (p[:, 2] <= 1e-4)).any())
    return bool((np.abs(p[:, 2]) <= 1e-3 * np.linalg.norm(p, axis=1)).any())
EPS_CATS = [i for i, (name, _) in enumerate(CATEGORIES) if name in ("n_zero", "n_tiny", "n_tiny_xz", "zero_pad")]
assert len(CATEGORIES) % 2 == 1   # row-major repetition then puts every category on both lanes of a texel pair
NCAT = len(CATEGORIES)
CAT_NAMES = [c[0] for c in CATEGORIES]


def edge_atlas(B, H, W, wf):
    """The atlas tiled to (B, H, W): maps as (B, C, H, W) fp32 tensors, and the (B, H, W) category index of every texel.
    Material b starts b categories further on, so the batch walk of the kernels meets every category at every position."""
    vals = {k: [] for k in ("a", "n", "r", "m", "s")}
    for _, over in CATEGORIES:
        t = dict(BASE, **over)
        for k in vals:
            vals[k].append(np.atleast_1d(np.asarray(t[k], np.float64)))
    table = {k: np.stack(v).astype(F32) for k, v in vals.items()}           # (NCAT, C)
    we = W + W % 2                                                          # a row starts on lane 0 even for odd W
    pos = (np.arange(H)[:, None] * we + np.arange(W)[None, :]).reshape(-1)
    idx = (pos[None, :] + np.arange(B)[:, None]) % NCAT                     # (B, H*W)
    pick = lambda k: torch.from_numpy(np.ascontiguousarray(table[k][idx].transpose(0, 2, 1).reshape(B, -1, H, W)))
    maps = {"albedo": pick("a"), "normal": pick("n"), "roughness": pick("r")}
    if wf == "specular":
        maps["specular"] = pick("s")
    else:
        m = pick("m")
        maps["metallic"] = m.expand(B, 3, H, W).contiguous() if wf == "metallic3" else m
        if wf == "metallic3":   # channel 1 of the 3-channel map takes the next category's value: channels differ
            maps["metallic"][:, 1] = torch.from_numpy(table["m"][(idx + 1) % NCAT][..., 0].reshape(B, H, W))
    return maps, idx.reshape(B, H, W)


def grid(H, W, size=1.0):
    """The plane coordinates of the texel centres exactly as the reference forms them (fp32 linspace)."""
    return torch.linspace(-size / 2, size / 2, W).numpy(), torch.linspace(-size / 2, size / 2, H).numpy()


def above(H, W, i, j, z, size=1.0):
    """A point light or camera exactly above texel (i, j): the reference's light vector there is (0, 0, z)."""
    xs, ys = grid(H, W, size)
    return [float(xs[j % W]), float(-ys[i % H]), z]


def point_lightings(H, W):
    """(name, position, intensity) of the point-light edges, each above its own texel (or below the plane)."""
    return [
        ("benign", [0.2, -0.1, 1.0], [1.0, 0.8, 0.6]),
        ("z0", above(H, W, H // 2, W // 2, 0.0), [1.0, 0.8, 0.6]),
        ("z1e-7", above(H, W, H // 2 + 1, W // 3, 1e-7), [1.0, 0.8, 0.6]),
        ("z1e-6", above(H, W, H // 3, W // 2 + 1, 1e-6), [0.7, 0.8, 0.9]),
        ("z1e-4", above(H, W, 0, W - 1, 1e-4), [1.0, 0.8, 0.6]),
        ("below", [0.1, 0.05, -0.5], [1.0, 1.0, 1.0]),
        ("dark", [-0.2, 0.1, 0.7], [0.0, 0.0, 0.0]),
        ("strong", [0.05, -0.05, 0.6], [8.0, 6.0, 40.0]),   # saturates the accumulated sum
    ]


VIEW_UP = [0.0, 0.0, 1.0]


def dir_lightings():
    """(name, direction, intensity) of the directional edges; the view is VIEW_UP."""
    return [
        ("benign", [0.3, 0.2, 0.93], [1.0, 0.8, 0.6]),
        ("up", [0.0, 0.0, 1.0], [1.0, 0.8, 0.6]),          # = view: the upper gates
        ("down", [0.0, 0.0, -1.0], [1.0, 0.8, 0.6]),       # = -view: h = normalize(0)
        ("graze", [1.0, 0.0, 0.0], [1.0, 0.8, 0.6]),       # N.L = 0 on the +z normals
        ("dark", [-0.3, 0.1, 0.9], [0.0, 0.0, 0.0]),
        ("strong", [0.1, -0.2, 0.97], [8.0, 6.0, 40.0]),
    ]


def cameras(H, W):
    """(name, camera position) for view_type="point"."""
    return [
        ("cam_above", above(H, W, H // 2, W // 2, 0.7)),   # the view is exactly +z at one texel
        ("cam_plane", above(H, W, 1, 2, 0.0)),             # on the plane, at a texel centre: a zero-length view there,
                                                           # horizontal views everywhere else
        ("cam_low", [0.3, -0.2, 1e-6]),
    ]


# ---------------------------------------------------------------------------------------------- comparison rules
def _labels_like(arr, cat):
    """Broadcast the (B, H, W) category map to an output / gradient of shape (B, [L,] C, H, W) or (1, C, H, W)."""
    cat = np.asarray(cat)
    if arr.shape[0] != cat.shape[0]:
        cat = cat[:arr.shape[0]]
    shape = (cat.shape[0],) + (1,) * (arr.ndim - 3) + cat.shape[1:]
    return np.broadcast_to(cat.reshape(shape), arr.shape)


def _where(bad, cat, limit=8):
    pos = np.argwhere(bad)[:limit]
    lab = _labels_like(bad, cat)
    return [(tuple(int(v) for v in p), CAT_NAMES[int(lab[tuple(p)])]) for p in pos]


def check_finite(what, got, ref32):
    got, ref32 = np.asarray(got), np.asarray(ref32)
    bad = np.isfinite(ref32) & ~np.isfinite(got)
    assert not bad.any(), f"{what}: non-finite where the oracle is finite at {np.argwhere(bad)[:8].tolist()}"


def check_forward(got, ref32, ref64, cat):
    """conftest.fwd_ok, or per texel the fp64 arbiter."""
    got, ref32, ref64 = (np.asarray(x, np.float64) for x in (got, ref32, ref64))
    check_finite("forward", got, ref32)
    err = np.abs(got - ref32)
    tol = 1e-5 * np.abs(ref32) + 1e-6
    ok = (err <= tol) | (np.abs(got - ref64) <= np.maximum(2 * np.abs(ref32 - ref64), tol))
    assert ok.all(), f"forward: max err/tol {float((err / tol).max()):.3g} at {_where(~ok, cat)}"
    return fwd_ok(got, ref32)[0]


def check_map_grad(name, got, ref32, ref64, cat, light_in_plane=False):
    """conftest.grad_ok per atlas category, or per texel the fp64 arbiter (which accepts either side of a gate where
    the fp32 and fp64 oracles disagree on it)."""
    got, r32, r64 = (np.asarray(x, np.float64) for x in (got, ref32, ref64))
    check_finite(f"d_{name}", got, r32)
    lab = _labels_like(r32, cat)
    err = np.abs(got - r32)
    tol = np.empty_like(r32)
    regular = ~np.isin(lab, EPS_CATS)
    floor = np.abs(r32[regular]).mean() if regular.any() else 0.0
    for c in np.unique(lab):
        sel = lab == c
        tol[sel] = 1e-4 * np.abs(r32[sel]) + 1e-4 * max(np.abs(r32[sel]).mean(), floor) + 1e-12
        if light_in_plane and name == "roughness" and c in K0_CATS:
            tol[sel] *= 10
    plain = err <= tol
    arb = np.abs(got - r64) <= 2 * np.abs(r32 - r64) + tol
    ok = plain | arb
    gate = ~plain & arb & (np.abs(r32 - r64) > tol)   # the two oracles disagree beyond the tolerance: a gate split
    assert ok.all(), (f"d_{name}: max err/tol {float((err / tol)[~ok].max()):.3g} at {_where(~ok, cat)}; "
                      f"accepted on the fp64 side of a gate: {_where(gate, cat)}")


def check_shared(name, got, want64, want32):
    """A sum over the image: 1e-4 |g| + 1e-4 mean|g| of the fp64 oracle, or per element the fp64 arbiter.  The arbiter
    matters where a gate splits the fp32 and fp64 oracles inside the sum (a camera on the plane puts N.V of every +z
    normal exactly on its lower gate, and texels fall on either side of it)."""
    got, w64, w32 = (np.asarray(x, np.float64).reshape(-1) for x in (got, want64, want32))
    assert np.isfinite(got).all(), (name, got)
    tol = 1e-4 * np.abs(w64) + 1e-4 * np.abs(w64).mean()
    ok = (np.abs(got - w64) <= tol) | (np.abs(got - w64) <= 2 * np.abs(w32 - w64) + tol)
    assert ok.all(), (name, float((np.abs(got - w64) / tol)[~ok].max()), got, w32, w64)


# ---------------------------------------------------------------------------------------------- the oracle
def oracle(render, maps, view, lights, inten, size, light_type, acc, flags, go):
    """fp32 image and map gradients, the fp64 image, map gradients and shared-parameter gradients of render(...) with the
    output gradient go (same shape as the image)."""
    leaves = {k: v.clone().requires_grad_(True) for k, v in maps.items()}
    sh32 = {k: t.clone().requires_grad_(True) for k, t in zip(SHARED, (inten, lights, view))}
    out = render(leaves, sh32["view"], sh32["lights"], sh32["intensity"], size, light_type, accumulate=acc, **flags)
    out.backward(go)
    m64 = {k: v.double().requires_grad_(True) for k, v in maps.items()}
    sh = {k: t.double().clone().requires_grad_(True) for k, t in zip(SHARED, (inten, lights, view))}
    out64 = render(m64, sh["view"], sh["lights"], sh["intensity"], size, light_type, accumulate=acc, **flags)
    out64.backward(go.double())
    return dict(out=out.detach().numpy(), out64=out64.detach().numpy(),
                g32={k: v.grad.numpy() for k, v in leaves.items()}, g64={k: v.grad.numpy() for k, v in m64.items()},
                shared32={k: sh32[k].grad.numpy() for k in SHARED}, shared64={k: sh[k].grad.numpy() for k in SHARED})


# ---------------------------------------------------------------------------------------------- hostsim runs
FP = ctypes.POINTER(ctypes.c_float)
DP = ctypes.POINTER(ctypes.c_double)
B_, H_, W_ = 2, 9, 9   # 81 texels a material: every category at least twice, on both lanes


def _fp(a):
    return None if a is None else a.ctypes.data_as(FP)


def _np(t):
    return np.ascontiguousarray(t.detach().numpy().astype(F32))


def _runs():
    """(id, light_type, lights, intensities, per_light, flags) for the orthographic view VIEW_UP."""
    pl, dl = point_lightings(H_, W_), dir_lightings()
    srgb = dict(albedo_is_srgb=True, specular_is_srgb=True, return_srgb=True)
    runs = [(f"point-{n}", "point", [p], [i], False, srgb) for n, p, i in pl]
    runs += [(f"dir-{n}", "directional", [p], [i], False, srgb) for n, p, i in dl]
    for per in (False, True):
        tag = "per" if per else "acc"
        runs.append((f"point-all-{tag}", "point", [p for _, p, _ in pl], [i for _, _, i in pl], per, srgb))
        runs.append((f"dir-all-{tag}", "directional", [p for _, p, _ in dl], [i for _, _, i in dl], per, srgb))
    lin = dict(albedo_is_srgb=False, specular_is_srgb=False, return_srgb=False)
    runs.append(("point-all-acc-linear", "point", [p for _, p, _ in pl], [i for _, _, i in pl], False, lin))
    runs.append(("point-z1e-7-linear", "point", [pl[2][1]], [pl[2][2]], False, lin))
    return runs


RUNS = _runs()
_CACHE = {}


def _case(wf, run):
    key = (wf, run[0])
    if key not in _CACHE:
        from oracle import pbr_oracle as O

        _, light_type, lights, inten, per, flags = run
        maps, cat = edge_atlas(B_, H_, W_, wf)
        view, lt, it = torch.tensor(VIEW_UP), torch.tensor(lights), torch.tensor(inten)
        size = 1.0 if light_type == "point" else None
        shape = (B_, len(lights), 3, H_, W_) if per else (B_, 3, H_, W_)
        go = torch.rand(shape, generator=torch.Generator().manual_seed(len(_CACHE) + 1)) + 0.5
        ref = oracle(O.render, maps, view, lt, it, size, light_type, not per, flags, go)
        _CACHE[key] = (maps, cat, view, lt, it, go, ref)
    return _CACHE[key]


def _args(wf, run, maps, view, lights, inten):
    _, light_type, _, _, per, flags = run
    a = {k: _np(v) for k, v in maps.items()}
    ms = a["specular" if wf == "specular" else "metallic"]
    keep = (a, ms, _np(view), _np(lights), _np(inten))
    args = (B_, H_, W_, lights.shape[0], WFS[wf], int(light_type == "point"), int(flags["albedo_is_srgb"]),
            int(flags["specular_is_srgb"]), int(flags["return_srgb"]), int(per), ctypes.c_float(1.0 if light_type == "point" else 0.0),
            _fp(a["albedo"]), _fp(a["normal"]), _fp(a["roughness"]), _fp(ms), _fp(keep[2]), _fp(keep[3]), _fp(keep[4]))
    return args, keep


def test_atlas_puts_every_category_on_both_lanes():
    for B, H, W in ((B_, H_, W_), (2, 3, 512), (2, 4, 40), (1, 4, 41)):
        _, cat = edge_atlas(B, H, W, "metallic")
        col = np.broadcast_to(np.arange(W) % 2, cat.shape)
        for lane in (0, 1):
            assert set(np.unique(cat[col == lane])) == set(range(NCAT)), (B, H, W, lane)


def test_edge_lights_sit_exactly_above_their_texels():
    """The reference's light vector at the texel under a light is (0, 0, z) exactly: torch.linspace's grid is used."""
    xs, ys = grid(H_, W_)
    for name, p, _ in point_lightings(H_, W_):
        if name.startswith("z"):
            j = int(np.flatnonzero(xs == F32(p[0]))[0]); i = int(np.flatnonzero(-ys == F32(p[1]))[0])
            assert F32(p[0]) - xs[j] == 0 and F32(p[1]) + ys[i] == 0, name


@pytest.mark.parametrize("generic", [0, 1, 2, 3, 5, 7, 15])   # the bits of test_hostsim.py
@pytest.mark.parametrize("run", RUNS, ids=[r[0] for r in RUNS])
@pytest.mark.parametrize("wf", list(WFS))
def test_forward_edges(hostsim, wf, run, generic):
    maps, cat, view, lights, inten, go, ref = _case(wf, run)
    args, keep = _args(wf, run, maps, view, lights, inten)
    out = np.zeros(ref["out"].shape, F32)
    assert hostsim.hs_ct_forward(*args, _fp(out), generic) == 0
    check_forward(out, ref["out"], ref["out64"], cat)


@pytest.mark.parametrize("generic", [0, 1, 2, 3, 5, 7, 15, 17, 23])
@pytest.mark.parametrize("run", RUNS, ids=[r[0] for r in RUNS])
@pytest.mark.parametrize("wf", list(WFS))
def test_backward_edges(hostsim, wf, run, generic):
    maps, cat, view, lights, inten, go, ref = _case(wf, run)
    args, (a, ms, *_) = _args(wf, run, maps, view, lights, inten)
    L = lights.shape[0]
    da, dn, dr, dm = np.zeros_like(a["albedo"]), np.zeros_like(a["normal"]), np.zeros_like(a["roughness"]), np.zeros_like(ms)
    di = np.zeros((L, 3), np.float64)
    loss = ctypes.c_double(0)
    gon = _np(go)
    assert hostsim.hs_ct_backward(*args, _fp(gon), None, ctypes.c_float(0), ctypes.byref(loss), _fp(da), _fp(dn), _fp(dr),
                                  _fp(dm), di.ctypes.data_as(DP), generic) == 0
    mkey = "specular" if wf == "specular" else "metallic"
    for k, g in (("albedo", da), ("normal", dn), ("roughness", dr), (mkey, dm)):
        check_map_grad(k, g, ref["g32"][k], ref["g64"][k], cat, in_plane(run[1], lights))
    check_shared("intensity", di, ref["shared64"]["intensity"], ref["shared32"]["intensity"])


@pytest.mark.parametrize("packed", [0, 2])
@pytest.mark.parametrize("run", RUNS, ids=[r[0] for r in RUNS])
def test_light_and_view_gradients_at_the_edges(hostsim, run, packed):
    wf = "metallic"
    maps, cat, view, lights, inten, go, ref = _case(wf, run)
    args, (a, ms, *_) = _args(wf, run, maps, view, lights, inten)
    L = lights.shape[0]
    da, dn, dr, dm = np.zeros_like(a["albedo"]), np.zeros_like(a["normal"]), np.zeros_like(a["roughness"]), np.zeros_like(ms)
    di, dl, dv = np.zeros((L, 3), np.float64), np.zeros((L, 3), np.float64), np.zeros(3, np.float64)
    loss = ctypes.c_double(0)
    gon = _np(go)
    assert hostsim.hs_ct_backward_geom(*args, _fp(gon), None, ctypes.c_float(0), ctypes.byref(loss), _fp(da), _fp(dn), _fp(dr),
                                       _fp(dm), di.ctypes.data_as(DP), dl.ctypes.data_as(DP), dv.ctypes.data_as(DP), packed) == 0
    for k, g in (("albedo", da), ("normal", dn), ("roughness", dr), ("metallic", dm)):
        check_map_grad(k, g, ref["g32"][k], ref["g64"][k], cat, in_plane(run[1], lights))
    for k, got in zip(SHARED, (di, dl, dv)):
        check_shared(k, got, ref["shared64"][k], ref["shared32"][k])


def test_loss_sum_and_gradients_at_the_edges(hostsim):
    """The fused-loss path (target instead of grad_out) on the lighting that broke the point-light geometry."""
    from oracle import pbr_oracle as O

    run = next(r for r in RUNS if r[0] == "point-all-acc")
    maps, cat, view, lights, inten, _, _ = _case("metallic", run)
    target = torch.rand(B_, 3, H_, W_, generator=torch.Generator().manual_seed(3))
    leaves = {k: v.clone().requires_grad_(True) for k, v in maps.items()}
    out = O.render(leaves, view, lights, inten, 1.0, "point", accumulate=True)
    loss = ((out - target) ** 2).mean()
    loss.backward()
    m64 = {k: v.double().requires_grad_(True) for k, v in maps.items()}
    loss64 = ((O.render(m64, view.double(), lights.double(), inten.double(), 1.0, "point") - target.double()) ** 2).mean()
    loss64.backward()
    args, (a, ms, *_) = _args("metallic", run, maps, view, lights, inten)
    tgt = _np(target)
    da, dn, dr, dm = np.zeros_like(a["albedo"]), np.zeros_like(a["normal"]), np.zeros_like(a["roughness"]), np.zeros_like(ms)
    lsum = ctypes.c_double(0)
    scale = 1.0 / target.numel()
    for generic in (0, 3, 7, 23):
        lsum.value = 0.0
        assert hostsim.hs_ct_backward(*args, None, _fp(tgt), ctypes.c_float(scale), ctypes.byref(lsum), _fp(da), _fp(dn),
                                      _fp(dr), _fp(dm), None, generic) == 0
        assert np.isfinite(lsum.value) and abs(lsum.value * scale - float(loss.detach())) <= 1e-5 * float(loss.detach()), (lsum.value * scale, float(loss.detach()))
        for k, g in (("albedo", da), ("normal", dn), ("roughness", dr), ("metallic", dm)):
            check_map_grad(k, g, leaves[k].grad.numpy(), m64[k].grad.numpy(), cat, in_plane("point", lights))


# ---------------------------------------------------------------------------------------------- camera
@pytest.fixture(scope="module")
def camera_sim(hostsim):
    f, i, p = ctypes.c_float, ctypes.c_int, ctypes.c_void_p
    head = [i] * 6 + [f] + [i] * 4 + [p] * 3
    hostsim.hs_ct_forward_camera.argtypes = head + [p] * 5
    hostsim.hs_ct_backward_camera.argtypes = head + [p] * 5 + [p] * 4 + [p] * 3
    return hostsim


def _cam_runs():
    """(id, H, W, camera, light type, lights, intensities, per_light).  Two shapes: the atlas's 9 x 9, and the 4 x 40 of the
    camera ledger's rows, where a camera on the plane makes the shared-parameter sums a cancellation (check_shared)."""
    runs = []
    for H, W in ((H_, W_), (4, 40)):
        pl, dl, cams = point_lightings(H, W), dir_lightings(), cameras(H, W)
        tag = f"{H}x{W}"
        for cname, cpos in cams:
            runs.append((f"{tag}-{cname}-point-benign", H, W, cpos, "point", [pl[0][1]], [pl[0][2]], False))
            runs.append((f"{tag}-{cname}-point-all-acc", H, W, cpos, "point", [p for _, p, _ in pl], [i for _, _, i in pl], False))
            runs.append((f"{tag}-{cname}-point-all-per", H, W, cpos, "point", [p for _, p, _ in pl], [i for _, _, i in pl], True))
            runs.append((f"{tag}-{cname}-dir-all-acc", H, W, cpos, "directional", [p for _, p, _ in dl], [i for _, _, i in dl], False))
        runs.append((f"{tag}-cam_above-point-z0", H, W, cams[0][1], "point", [pl[1][1]], [pl[1][2]], False))
        runs.append((f"{tag}-cam_above-point-z1e-7", H, W, cams[0][1], "point", [pl[2][1]], [pl[2][2]], False))
    return runs


CAM_RUNS = _cam_runs()


@pytest.mark.parametrize("run", CAM_RUNS, ids=[r[0] for r in CAM_RUNS])
@pytest.mark.parametrize("wf", list(WFS))
def test_camera_edges(camera_sim, wf, run):
    import camera_oracle as CO

    _, H, W, cam, light_type, lights, inten, per = run
    maps, cat = edge_atlas(B_, H, W, wf)
    camera, lt, it = torch.tensor(cam), torch.tensor(lights), torch.tensor(inten)
    size = 1.0 if light_type == "point" else None
    flags = dict(albedo_is_srgb=True, specular_is_srgb=True, return_srgb=True)
    shape = (B_, len(lights), 3, H, W) if per else (B_, 3, H, W)
    go = torch.rand(shape, generator=torch.Generator().manual_seed(CAM_RUNS.index(run))) + 0.5
    ref = oracle(CO.render, maps, camera, lt, it, size, light_type, not per, flags, go)
    mkey = "specular" if wf == "specular" else "metallic"
    a = {k: _np(v) for k, v in maps.items()}
    ptr = lambda x: None if x is None else x.ctypes.data_as(ctypes.c_void_p)
    par = [_np(camera), _np(lt), _np(it)]
    head = (B_, H, W, len(lights), WFS[wf], int(light_type == "point"), float(size or 0.0), 1, 1, 1, int(per))
    args = head + tuple(ptr(x) for x in par) + tuple(ptr(a[k]) for k in ("albedo", "normal", "roughness", mkey))
    out = np.zeros(ref["out"].shape, F32)
    assert camera_sim.hs_ct_forward_camera(*args, ptr(out)) == 0
    check_forward(out, ref["out"], ref["out64"], cat)
    grads = {k: np.zeros(v.shape, F32) for k, v in a.items()}
    d_int, d_lights, d_cam = np.zeros(3 * len(lights)), np.zeros(3 * len(lights)), np.zeros(3)
    gout = _np(go)
    assert camera_sim.hs_ct_backward_camera(*args, ptr(gout), *(ptr(grads[k]) for k in ("albedo", "normal", "roughness", mkey)),
                                            ptr(d_int), ptr(d_lights), ptr(d_cam)) == 0
    for k in maps:
        check_map_grad(k, grads[k], ref["g32"][k], ref["g64"][k], cat, in_plane(light_type, lights))
    for k, got in zip(SHARED, (d_int, d_lights, d_cam)):
        check_shared(k, got, ref["shared64"][k], ref["shared32"][k])
