#!/usr/bin/env python
"""
bench.py — CookTorrance forward+backward throughput (BASELINE.json metric), one JSON line on stdout.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c1|c3|c4|c5|aux]
                  [--dump-outputs DIR]

Every GPU timing of our arm (the config's value, the configs block, the e2e legs, the c4 / aux kernel rows, the c1 CUDA
graph replay) runs max(W, 3) warm-up steps and then exactly K timed steps.  The cpu_baseline and gpu_eager_baseline
samples do not follow K: they are best-of-a-few samples bounded in time, so that the line stays affordable.

Main line (default --config c2, N=1): BASELINE.json configs[1] — batch 64 materials 1024x1024, CookTorrance
forward+backward, 1 point light, fp32, metallic workflow, sRGB albedo in / sRGB colour out.  A step = one forward pass
(pbr_ct_forward) + one backward pass (pbr_ct_backward) over the whole batch through the public API
(CookTorranceBRDF.__call__ + torch.autograd.grad).  N>1 (torchrun): every rank owns its own 64-material shard (weak
scaling, no data-path collective - materials are independent); value = texel-lights of all ranks / max-over-ranks
device time.

  value     : Gtexel-lights/s, maps resident in HBM, timed with CUDA events on the launch stream
  roofline  : the backward kernel (dominant): algorithmic bytes (76 B/texel, DESIGN.md §5) / its own CUDA-event
              duration, against the measured HBM peak of MEASURED_PEAKS.json; `traffic` = the ncu DRAM bytes of that
              kernel from profiles/traffic.json, dropped when that capture was taken from other kernel sources
  e2e       : the same two kernels (brdf() + autograd backward) fed from PINNED HOST memory with 8-bit textures (the
              form the reference's material constructors accept): per step the H2D of every texture (chunked,
              double-buffered against compute), pbr_ingest_image, forward, backward, and the D2H of the step's result
              (the light-intensity gradient the backward reduces, 12 bytes).  e2e.legs holds the float32-maps-in /
              map-gradients-out leg (32 B/texel each way) and the fit-style leg (fused loss kernel, loss read back).
  configs   : the other BASELINE.json configs measured in the same run, same rules (barrier, CUDA events, max over
              ranks): c1 (single 256x256 material, launch-latency bound: microseconds per call), c3 (16 x 2048^2,
              16 lights, forward+backward), c5 (one step of the sharded inverse-rendering fit: 512 materials 512x512
              per GPU, 8 lights, ONE launch per step + the NCCL all-reduce of the loss, timed per step)
  cpu_baseline / --impl reference : the oracle port of the reference's PyTorch eager CPU path (oracle/pbr_oracle.py,
              bit-identical to the reference, tests/golden/make_golden.py) timed on the host cores on a bounded sample
  gpu_eager_baseline : the same port run with CUDA tensors (what `.to("cuda")` gives a reference user on this B200):
              one material, forward+backward through autograd, CUDA events, kernel-launch count
"""

from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

CONFIGS = {
    # name: (B per GPU, H, W, L, per_light)
    "c2": dict(B=64, H=1024, W=1024, L=1, per_light=False,
               workload="batch 64 materials 1024x1024, CookTorrance forward+backward, 1 point light, fp32"),
    "c3": dict(B=16, H=2048, W=2048, L=16, per_light=False,
               workload="batch 16 materials 2048x2048, 16 point lights, forward+backward shading"),
    "c5": dict(B=512, H=512, W=512, L=8, per_light=True,
               workload="SVBRDF inverse-rendering fit step, 512 materials 512x512 per GPU, 8 lights: fused render+MSE+backward, "
                        "loss all-reduce, fused Adam+projection"),
}
C1 = dict(H=256, W=256,
          workload="single 256x256 BasecolorMetallicMaterial, CookTorranceBRDF point light, one view/light (examples/example_brdf.py, CPU)")
C4 = dict(H=4096, W=4096,
          workload="4096x4096 metallic->diffuse-specular conversion + mask/height blend_materials pipeline")
FWD_BYTES, BWD_BYTES = 44, 76  # algorithmic bytes per texel, metallic workflow, accumulate mode (SURVEY.md §8d)
METRIC = "Gtexel-lights/sec CookTorrance fwd+bwd"
UNIT = "Gtexel-lights/s"


def csrc_sha16():
    """Hash of the kernel sources the library is built from (the .cu / .cuh files and the C-ABI header)."""
    h = hashlib.sha256()
    csrc = os.path.join(ROOT, "pypbr_b200", "csrc")
    for path in sorted(os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cu", ".cuh"))) + [os.path.join(ROOT, "include", "pbrcuda.h")]:
        with open(path, "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def measured_traffic(key):
    """Per-launch DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) of a kernel from the committed `ncu --set full`
    capture of this same command (profiles/traffic.json, written by tools/ncu_traffic.py).  The file carries the hash of
    the kernel sources it was captured from: a stale capture (sources changed since) is not reported."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tr = json.load(f)
        if tr.get("_csrc_sha16") != csrc_sha16():
            return None
        return tr.get(key)
    except Exception:
        return None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    BAD = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "hw_power_brake": 0x80}
    NOTE = {"sw_power_cap": 0x4}

    def __init__(self, index: int):
        self.samples, self.reasons, self.stop_flag = [], set(), False
        self.max_mhz = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop_flag and self.nv is not None:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for k, bit in {**self.BAD, **self.NOTE}.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop_flag = True
        self.t.join(timeout=2)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ---------------------------------------------------------------------------------------------- inputs
def synth_maps(B, H, W, device, seed, pin=False, rough_lo=0.2):
    """SURVEY.md §8d: albedo U[0,1] sRGB, metallic U[0,1], roughness U[0.2,1], unit normals around +Z."""
    g = torch.Generator(device=device).manual_seed(seed)
    albedo = torch.rand(B, 3, H, W, generator=g, device=device)
    metallic = torch.rand(B, 1, H, W, generator=g, device=device)
    roughness = torch.rand(B, 1, H, W, generator=g, device=device) * (1.0 - rough_lo) + rough_lo
    n = torch.randn(B, 3, H, W, generator=g, device=device)
    n[:, 0:2] *= 0.3
    n[:, 2] = 1.0
    normal = torch.nn.functional.normalize(n, dim=1)
    del n
    maps = dict(albedo=albedo, normal=normal, roughness=roughness, metallic=metallic)
    if pin:
        maps = {k: v.pin_memory() for k, v in maps.items()}
    return maps


def lights_for(L):
    if L == 1:
        return torch.tensor([0.1, 0.1, 1.0]), torch.tensor([1.0, 1.0, 1.0])
    pts = [[0.4 * math.cos(2 * math.pi * l / L), 0.4 * math.sin(2 * math.pi * l / L), 1.0] for l in range(L)]
    return torch.tensor(pts), torch.ones(L, 3)


def config1_fixture():
    """BASELINE.json configs[0]: the reference's tests/data/tiles material at 256x256 with example_brdf.py's lighting
    (tests/golden/config1_tiles_256.npz and its normal map in config1_tiles_256.in_normal.npz, written by
    tests/golden/make_golden.py from the reference's own loader)."""
    import numpy as np

    golden = os.path.join(ROOT, "tests", "golden", "config1_tiles_256")
    z = np.load(golden + ".npz")
    normal = np.load(golden + ".in_normal.npz")["in_normal"]
    maps = {k: torch.from_numpy(normal if k == "normal" else z["in_" + k]) for k in ("albedo", "normal", "roughness", "metallic")}
    return maps, torch.from_numpy(z["view"]), torch.from_numpy(z["lights"]), torch.from_numpy(z["intensity"])


# ---------------------------------------------------------------------------------------------- baselines (oracle port)
def port_sample(maps, view, lights, inten, device, reps=8, budget_s=12.0, backward=True, accumulate=True):
    """One material through the oracle port of the reference's eager path (autograd backward) on `device`.
    Returns (best seconds, timed repetitions).  CPU: wall clock; CUDA: CUDA events."""
    from oracle import pbr_oracle as O

    maps = {k: v.to(device) for k, v in maps.items()}
    view, lights, inten = view.to(device), lights.to(device), inten.to(device)
    cuda = torch.device(device).type == "cuda"
    go = None
    best, n_timed, t_begin = None, 0, time.perf_counter()
    for it in range(reps + 1):
        leaves = {k: v.clone().requires_grad_(backward) for k, v in maps.items()}
        if cuda:
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
        t0 = time.perf_counter()
        with torch.set_grad_enabled(backward):
            out = O.render(leaves, view, lights, inten, 1.0, "point", accumulate=accumulate)
        if backward:
            if go is None:
                go = torch.rand(out.shape, device=device)
            out.backward(go)
        if cuda:
            e1.record()
            torch.cuda.synchronize()
            dt = e0.elapsed_time(e1) * 1e-3
        else:
            dt = time.perf_counter() - t0
        if it > 0:
            best = dt if best is None else min(best, dt)
            n_timed += 1
        if n_timed >= 2 and time.perf_counter() - t_begin > budget_s:
            break
    return best, n_timed


def cpu_baseline_for(name, reps=8, budget_s=12.0):
    """`cpu_baseline` object of one config: a bounded sample of the workload on all host threads."""
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    if name == "c1":
        maps, view, lights, inten = config1_fixture()
        fb, n = port_sample(maps, view, lights, inten, "cpu", reps, budget_s)
        f, _ = port_sample(maps, view, lights, inten, "cpu", reps, budget_s, backward=False)
        return {"value": C1["H"] * C1["W"] / fb / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
                "fwd_us": f * 1e6, "fwd_bwd_us": fb * 1e6,
                "sample": f"the whole config (1 material 256x256, 1 light), forward and forward+backward through autograd, best of {n}; "
                          "oracle/pbr_oracle.py, bit-identical to the reference"}
    cfg = CONFIGS[name]
    H, W, L = cfg["H"], cfg["W"], cfg["L"]
    maps = {k: v[0] for k, v in synth_maps(1, H, W, torch.device("cpu"), 7).items()}
    lights, inten = lights_for(min(L, 2))
    nl = lights.shape[0] if lights.dim() == 2 else 1
    if L > 1 and not cfg["per_light"]:
        inten = inten / L
    best, n = port_sample(maps, torch.tensor([0.0, 0.0, 1.0]), lights, inten, "cpu", reps, budget_s, accumulate=not cfg["per_light"])
    return {"value": H * W * nl / best / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"1 material {H}x{W} x {nl} light(s) of the batch, fwd+bwd through autograd, best of {n} "
                      f"after 1 warm-up ({best:.2f} s each); oracle/pbr_oracle.py, bit-identical to the reference"}


def gpu_eager_baseline(name, dev, our_value):
    """The reference's eager path on the same GPU (the port on CUDA tensors): what `material.to('cuda')` buys a reference
    user.  One material x one light, forward+backward through autograd; CUDA events; kernel launches counted by the profiler."""
    from oracle import pbr_oracle as O  # noqa: F401  (checker / baseline only)

    if name == "c1":
        maps, view, lights, inten = config1_fixture()
        H, W = C1["H"], C1["W"]
    else:
        cfg = CONFIGS[name]
        H, W = cfg["H"], cfg["W"]
        maps = {k: v[0] for k, v in synth_maps(1, H, W, dev, 7).items()}
        view, (lights, inten) = torch.tensor([0.0, 0.0, 1.0]), lights_for(1)
    best, n = port_sample(maps, view, lights, inten, dev, reps=10, budget_s=5.0)
    f_best, _ = port_sample(maps, view, lights, inten, dev, reps=10, budget_s=5.0, backward=False)
    launches = None
    try:
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            port_sample(maps, view, lights, inten, dev, reps=0, budget_s=0.0)
            torch.cuda.synchronize()
        launches = sum(1 for e in prof.events() if e.device_type.name == "CUDA" and "memcpy" not in e.name.lower() and "memset" not in e.name.lower())
    except Exception:
        pass
    v = H * W / best / 1e9
    return {"value": v, "unit": UNIT, "kind": "port on CUDA tensors (PyTorch eager, ATen kernels)", "fwd_ms": f_best * 1e3, "fwd_bwd_ms": best * 1e3,
            "kernel_launches_per_fwd_bwd": launches, "ours_over_eager": (our_value / v) if our_value else None,
            "sample": f"1 material {H}x{W} x 1 light, fwd+bwd through autograd, best of {n} (CUDA events)"}


# ---------------------------------------------------------------------------------------------- reference arm
def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the path (the oracle port, bit-identical to it) on all
    host threads, on our arm's config / metric / unit; rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    if args.config == "c4":
        return run_reference_c4(args, threads)
    name = args.config if args.config in ("c1", "c2", "c3", "c5") else "c2"
    if name == "c1":
        maps, view, lights, inten = config1_fixture()
        H, W, nl, B, per_light = C1["H"], C1["W"], 1, 1, False
        workload = C1["workload"]
        sample = "the whole config: 1 material 256x256, 1 light, fwd+bwd (autograd) per step"
    else:
        cfg = CONFIGS[name]
        H, W, L, B, per_light = cfg["H"], cfg["W"], cfg["L"], cfg["B"], cfg["per_light"]
        maps = {k: v[0] for k, v in synth_maps(1, H, W, torch.device("cpu"), 7).items()}
        lights, inten = lights_for(min(L, 2))
        nl = lights.shape[0] if lights.dim() == 2 else 1
        if L > 1 and not per_light:
            inten = inten / L
        view = torch.tensor([0.0, 0.0, 1.0])
        workload = cfg["workload"]
        sample = f"1 material {H}x{W} x {nl} light(s) per step, fwd+bwd (autograd), of the batch of {B}"
    from oracle import pbr_oracle as O

    go = torch.rand(((nl,) if (per_light and nl > 1) else ()) + (3, H, W))

    def step():
        leaves = {k: v.clone().requires_grad_(True) for k, v in maps.items()}
        out = O.render(leaves, view, lights, inten, 1.0, "point", accumulate=not per_light)
        out.backward(go)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = time.perf_counter() - t0
    value = H * W * nl * args.steps / dt / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if name == "c2" and not args.no_configs:
        # the other shading configs on the same host cores, bounded samples (independent of --steps)
        line["configs"] = {k: {"workload": (C1 if k == "c1" else CONFIGS[k])["workload"], **cpu_baseline_for(k, reps=2, budget_s=6.0)}
                           for k in ("c1", "c3", "c5")}
    print(json.dumps(line), flush=True)


def c4_cpu_pipeline(H, W):
    """BASELINE.json configs[3] on the host: the port's conversions + blends (oracle/pbr_oracle.py restates
    metallic.py:90-109 and blending/functional.py:64-196 op for op).  Returns a callable running one pipeline."""
    from oracle import pbr_oracle as O

    mats = []
    for seed in (4001, 4002):
        m = {k: v[0] for k, v in synth_maps(1, H, W, torch.device("cpu"), seed).items()}
        m["height"] = torch.rand(1, H, W, generator=torch.Generator().manual_seed(seed + 50))
        mats.append(m)
    mask = torch.rand(1, H, W, generator=torch.Generator().manual_seed(4003))

    def pipeline():
        ds = []
        for m in mats:
            d, s = O.metallic_to_specular(m["albedo"], m["metallic"], True)
            ds.append(dict(albedo=d, specular=s, normal=O.process_normal_map(m["normal"]), roughness=m["roughness"]))
        b1 = O.blend_maps(ds[0], ds[1], mask)
        b1["normal"] = O.process_normal_map(b1["normal"])
        hm = O.sigmoid_mask(mats[0]["height"], mats[1]["height"], 0.1, 0.0)
        b2 = O.blend_maps(mats[0], mats[1], hm)
        b2["normal"] = O.process_normal_map(b2["normal"])
        return b1, b2

    return pipeline


C4_SAMPLE_HW = 2048   # bounded sample: a quarter of the 4096 x 4096 texels (every op is per-texel: cost is linear in the texel count)


def c4_cpu_sample(reps=1):
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    pipe = c4_cpu_pipeline(C4_SAMPLE_HW, C4_SAMPLE_HW)
    pipe()
    best = None
    for _ in range(reps):
        t0 = time.perf_counter()
        pipe()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {"value": C4_SAMPLE_HW * C4_SAMPLE_HW / best / 1e9, "unit": "Gtexel/s", "cores": threads, "kind": "port",
            "sample": f"the same pipeline on two {C4_SAMPLE_HW}x{C4_SAMPLE_HW} materials (1/4 of the texels), best of {reps} after 1 warm-up "
                      f"({best:.2f} s each); oracle/pbr_oracle.py"}


def run_reference_c4(args, threads):
    """--impl reference --config c4: the conversion + blend pipeline of the port on the host cores, a bounded sample per step."""
    H = W = C4_SAMPLE_HW
    pipeline = c4_cpu_pipeline(H, W)
    for _ in range(max(args.warmup, 1)):
        pipeline()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        pipeline()
    dt = (time.perf_counter() - t0) / args.steps
    value = H * W / dt / 1e9
    sample = f"the same pipeline on two {H}x{W} materials (1/4 of the 4096x4096 texels) per step"
    print(json.dumps({
        "impl": "reference", "metric": "Gtexel/s conversion + blend pipeline", "value": value, "unit": "Gtexel/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": {"workload": C4["workload"], "sample": sample},
        "cpu_baseline": {"value": value, "unit": "Gtexel/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Gtexel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}), flush=True)


# ---------------------------------------------------------------------------------------------- our arm
class Ctx:
    """Process-level state of the GPU arm: rank / device / process group, and the barrier + max-over-ranks helpers."""

    def __init__(self):
        import torch.distributed as dist

        self.dist = dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the shading path has no CPU fallback)")
        self.dev = torch.device(f"cuda:{self.local}")
        torch.cuda.set_device(self.dev)
        self.numa = bind_to_gpu_numa(self.local)
        if self.world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("nccl", device_id=self.dev)
        from pypbr_b200 import _cabi

        self.cabi = _cabi
        _cabi.load()

    def barrier(self):
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        if self.world == 1:
            return x
        t = torch.tensor([x], device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def bind_to_gpu_numa(index):
    """Pin this process (and with it the first-touch placement of the pinned host buffers it allocates) to the CPUs
    NVML reports as local to its GPU.  Best effort: returns what was done for the JSON line."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        node = None
        try:
            nm = pynvml.nvmlDeviceGetMemoryAffinity(h, 4, pynvml.NVML_AFFINITY_SCOPE_NODE)
            node = [64 * w + b for w, m in enumerate(nm) for b in range(64) if (m >> b) & 1]
        except Exception:
            pass
        return {"cpus_bound": len(cpus), "cpu_range": f"{min(cpus)}-{max(cpus)}" if cpus else None, "numa_nodes": node}
    except Exception as e:  # pragma: no cover
        return {"error": str(e)[:80]}


def make_material(maps, dev, requires_grad):
    from pypbr_b200.materials import BasecolorMetallicMaterial

    mat = BasecolorMetallicMaterial(albedo_is_srgb=True, device=dev)
    leaves = []
    for k, v in maps.items():
        v.requires_grad_(requires_grad)
        mat._maps[k] = v
        leaves.append(v)
    return mat, leaves


DUMP_BYTES = 60_000_000   # --dump-outputs: what the sampled arrays may take, under a 64 MB cap for the whole directory


def dump_outputs(out_dir, arrays, B, H, W):
    """--dump-outputs: each (B, ..., H, W) array of `arrays` (or (C, H, W) with B = 1) as out_dir/<name>.npy in float32,
    shaped (texels, channels) and taken at the same texel positions: all B*H*W in order when they fit DUMP_BYTES, else a
    fixed sample (seed 0, sorted, no repeats).  Any other array is written whole, in float64."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    texels = B * H * W
    planes = {k: v.detach().reshape(B, -1, H * W) for k, v in arrays.items() if v.dim() >= 3 and tuple(v.shape[-2:]) == (H, W)}
    n = min(texels, DUMP_BYTES // (4 * sum(v.shape[1] for v in planes.values())))
    idx = torch.randint(0, texels, (n,), generator=torch.Generator().manual_seed(0)).unique() if n < texels else torch.arange(texels)
    idx = idx.to(next(iter(planes.values())).device)
    b, p = idx // (H * W), idx % (H * W)
    for k, v in arrays.items():
        a = planes[k][b, :, p].float() if k in planes else v.detach().double()
        np.save(os.path.join(out_dir, k + ".npy"), a.cpu().numpy())


def measure_shading(name, args, ctx, steps, warmup, dump_dir=None):
    """One shading config (c2 / c3 / c5) on this rank's shard: W warm-up steps, then `steps` steps between two CUDA events,
    bracketed by barrier + synchronize, max over ranks.  Returns the config's result object.
    dump_dir: write what the last timed step returned to its caller there (dump_outputs; rank 0's shard): the forward output
    and the map gradients, or for the fit (c5) the maps after the update and the step's loss buffer."""
    from pypbr_b200.fit import FusedAdam, allreduce_loss_and_shared, fit_step, fused_loss_step
    from pypbr_b200.models import CookTorranceBRDF

    cfg = CONFIGS[name]
    dev, world, rank = ctx.dev, ctx.world, ctx.rank
    B, H, W, L, per_light = cfg["B"], cfg["H"], cfg["W"], cfg["L"], cfg["per_light"]
    fused_fit = name == "c5"
    one_launch = fused_fit and args.fit.startswith("one-launch")
    async_loss = one_launch and args.fit == "one-launch"
    maps = synth_maps(B, H, W, dev, 1000 * 2 + rank)
    mat, leaves = make_material(maps, dev, not fused_fit)
    lights, inten = lights_for(L)
    if L > 1 and not per_light:
        inten = inten / L
    view = torch.tensor([0.0, 0.0, 1.0])
    brdf = CookTorranceBRDF("point", multi_light="per_light" if per_light else "accumulate")
    out_shape = (B, L, 3, H, W) if per_light else (B, 3, H, W)
    g = torch.Generator(device=dev).manual_seed(99 + rank)
    ar_events, adam_ms = [], []
    if fused_fit:
        target = torch.rand(out_shape, generator=g, device=dev)
        bufs = {}
        adam = FusedAdam({k: mat._maps[k] for k in ("albedo", "normal", "roughness", "metallic")}, lr=1e-3)
    else:
        grad_out = torch.rand(out_shape, generator=g, device=dev)

    ev = lambda: torch.cuda.Event(enable_timing=True)
    fwd_ms, bwd_ms = [], []
    last = [None]
    kept = {}   # what the last timed step returned, held only when it is to be dumped

    def step(record=False, keep=False):
        if fused_fit:
            # one full step of the sharded fit: fused render + MSE + backward, ONE all-reduce, fused Adam + projection
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            if one_launch:
                # ... all of it in ONE launch (pbr_ct_fit_step: Adam + projection in the loss kernel's epilogue); the
                # all-reduce only serves the reported loss and runs on a side stream (fit.allreduce_loss_async)
                last[0] = fit_step(mat, adam, target, view, lights, inten, "point", 1.0, scratch=bufs,
                                   global_numel=target.numel() * world, fused=True, async_loss=async_loss,
                                   timing=ar_events if (record and async_loss) else None)
                e1.record()
                if record:
                    bwd_ms.append((e0, e1))
                if keep:
                    kept["loss_buffer"] = last[0].buf if async_loss else last[0]
                return
            # --shared-grads: the fit with unknown lighting - intensity, light position and view gradients ride along
            # (PbrCtGrads.d_intensity / d_lights / d_view; 1 + 6L + 3 floats to all-reduce instead of 1 + 3L)
            buf, grads = fused_loss_step(mat, target, view, lights, inten, "point", 1.0, multi_light="per_light",
                                         loss_scale=1.0 / (target.numel() * world), out=bufs,
                                         want_intensity_grad=args.shared_grads, want_geometry_grad=args.shared_grads)
            e1.record()
            allreduce_loss_and_shared(buf)
            adam.step({k: grads[k] for k in adam.params})
            e2.record()
            if record:
                bwd_ms.append((e0, e1))
                adam_ms.append((e1, e2))
            if keep:
                kept["loss_buffer"] = buf
            return
        e0, e1, e2 = ev(), ev(), ev()
        e0.record()
        out = brdf(mat, view, lights, inten, 1.0)
        e1.record()
        grads = torch.autograd.grad(out, leaves, grad_out)
        e2.record()
        if record:
            fwd_ms.append((e0, e1))
            bwd_ms.append((e1, e2))
        if keep:
            kept.update(out=out, **{"grad_" + k: t for k, t in zip(maps, grads)})

    for _ in range(warmup):
        step()
    ctx.barrier()
    launches0 = ctx.cabi.launch_count()
    t_start, t_end = ev(), ev()
    with ClockSampler(ctx.local) as clk:
        t_start.record()
        for i in range(steps):
            step(record=True, keep=dump_dir is not None and i == steps - 1)
        if async_loss and last[0] is not None:
            last[0].wait()   # the timed region ends when the last step's loss has been reduced as well
        t_end.record()
        torch.cuda.synchronize()
    launches = ctx.cabi.launch_count() - launches0
    elapsed_ms = ctx.max_over_ranks(t_start.elapsed_time(t_end))
    ctx.barrier()
    if dump_dir is not None and rank == 0:
        if fused_fit:
            kept.update((k, mat._maps[k]) for k in maps)   # the parameters as the last step's update left them
        dump_outputs(dump_dir, kept, B, H, W)
    kept.clear()

    texel_lights_per_step = B * H * W * L * world
    value = texel_lights_per_step * steps / (elapsed_ms * 1e-3) / 1e9
    peak, peak_src = measured_peak()
    texels = B * H * W
    bwd_avg = sum(a.elapsed_time(b) for a, b in bwd_ms) / len(bwd_ms)
    fwd_avg = None
    if one_launch:
        # maps in (32) + per-light targets (12 L) + maps out (32) + both Adam moments of the 8 planes read (64) and
        # written (64); the epilogue's re-read of the parameters is served by L2 and not counted (ncu: 288 B per texel)
        kbytes = texels * (32 + 12 * L + 32 + 128)
        kname = "ct_backward_kernel<0,3,0> (fused loss + Adam epilogue, cached light geometry)"
    elif fused_fit:
        kbytes = texels * (32 + 12 * L + 32)
        kname = "ct_backward_kernel<0,5,0> (fused loss, cached light geometry)" if not args.shared_grads else \
                "ct_backward_kernel<0,3,1> (fused loss + d_intensity / d_lights / d_view, cached light geometry)"
    else:
        fwd_avg = sum(a.elapsed_time(b) for a, b in fwd_ms) / len(fwd_ms)
        # accumulate mode with several lights: + the forward output the one-pass backward reads (12 B per texel)
        kbytes = texels * ((BWD_BYTES + (12 if L > 1 else 0)) if not per_light else 64 + 12 * L)
        kname = "ct_backward_stream<0,2,0> (TMA-fed)" if L == 1 else "ct_backward_kernel<0,3,0> (cached light geometry, one pass from the saved forward output)"
    achieved = kbytes / (bwd_avg * 1e-3) / 1e9
    tr = measured_traffic(f"{name}:backward" + (":two-kernel" if fused_fit and not one_launch else ""))
    roofline = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": (tr or {}).get("bytes"), "traffic_source": (tr or {}).get("source"),
                "peak_source": peak_src, "algorithmic_bytes_per_launch": kbytes, "kernel_ms": bwd_avg}
    if tr and tr.get("fma_pipe_busy_pct") is not None and L > 1:
        # the multi-light kernels sit under the FP32 roof, not the HBM one (SURVEY.md 8d): what the committed ncu capture
        # of this command says about the instruction side
        roofline["compute_side"] = {"fma_pipe_busy_pct": tr["fma_pipe_busy_pct"], "issue_slots_busy_pct": tr.get("issue_active_pct"),
                                    "warp_instructions": tr.get("warp_instructions"), "source": tr.get("source")}
    if fused_fit and not one_launch:
        a_avg = sum(a.elapsed_time(b) for a, b in adam_ms) / len(adam_ms)
        ab = texels * 8 * 28   # 8 parameter planes: read p, g, m, v and write p, m, v
        roofline["adam"] = {"kernel": "adam_kernel (+ the loss all-reduce when n_gpus > 1)", "kernel_ms": a_avg,
                            "algorithmic_bytes_per_launch": ab, "achieved": ab / (a_avg * 1e-3) / 1e9,
                            "frac": ab / (a_avg * 1e-3) / 1e9 / peak}
    if fwd_avg is not None:
        fb = texels * (FWD_BYTES if not per_light else 32 + 12 * L)
        roofline["forward"] = {"kernel": "ct_forward_stream<0,2> (TMA-fed)" if L == 1 else "ct_forward_kernel<0,3> (cached light geometry)", "achieved": fb / (fwd_avg * 1e-3) / 1e9, "kernel_ms": fwd_avg,
                               "frac": fb / (fwd_avg * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": fb}
        roofline["fwd_plus_bwd_frac"] = (fb + kbytes) / ((fwd_avg + bwd_avg) * 1e-3) / 1e9 / peak
    res = {
        "value": value, "unit": UNIT, "ms_per_step": elapsed_ms / steps, "steps": steps, "warmup": warmup,
        "config": {"workload": cfg["workload"], "per_gpu_batch": B, "H": H, "W": W, "lights": L,
                   "mode": ("per_light fused loss + Adam, " + args.fit + (", shared-parameter gradients" if args.shared_grads else "")) if fused_fit else "accumulate", "parallelism": f"batch-shard x{world}",
                   "l2": f"inputs ({texels * 32 / 1e9:.1f} GB per GPU) exceed the 126 MB L2; no flush needed"},
        "roofline": roofline, "gpu_launches": int(launches), "clocks": clk.summary(),
    }
    if fused_fit:
        ar = None
        if ar_events:
            torch.cuda.synchronize()
            ar = sum(a.elapsed_time(b) for a, b in ar_events) / len(ar_events)
        res["allreduce"] = {
            "collective": f"NCCL all_reduce(SUM) of {1 + 3 * L} floats per step" + ("" if world > 1 else " (single rank: no-op)"),
            "where": "side stream behind an event; the compute stream never waits for it" if async_loss else "compute stream (blocking)",
            # from the fit kernel's completion to the reduced loss: includes waiting for the slowest rank's kernel and for an SM
            # slot under the NEXT step's kernel, which is already running - it is off the critical path by construction
            "completion_latency_ms": ar, "world": world}
        if last[0] is not None and async_loss:
            res["loss"] = last[0].item()
    return res


def measure_c1(ctx, steps, warmup, dump_dir=None):
    """BASELINE.json configs[0]: one 256x256 material, one point light - a launch-latency-bound call.  Microseconds per
    `brdf()` call (forward) and per forward+backward through autograd, back to back, CUDA events around the loop (host
    launch overhead included: that is what a caller sees).  `warmup` + `steps` calls of each, and as many replays of the
    CUDA graph.  dump_dir: write what the last timed forward+backward returned there (dump_outputs)."""
    from pypbr_b200.models import CookTorranceBRDF

    maps, view, lights, inten = config1_fixture()
    dev = ctx.dev
    mat, leaves = make_material({k: v.to(dev) for k, v in maps.items()}, dev, True)
    brdf = CookTorranceBRDF("point")
    go = torch.rand(3, C1["H"], C1["W"], device=dev)
    view_d, lights_d, inten_d = view.to(dev), lights.to(dev), inten.to(dev)   # device-resident parameters: no staging, no sync
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def fwd():
        with torch.no_grad():
            return brdf(mat, view_d, lights_d, inten_d, 1.0)

    def fwd_bwd():
        out = brdf(mat, view_d, lights_d, inten_d, 1.0)
        return out, torch.autograd.grad(out, leaves, go)

    res, last = {}, None
    launches0 = ctx.cabi.launch_count()
    with ClockSampler(ctx.local) as clk:
        for key, fn in (("fwd_us", fwd), ("fwd_bwd_us", fwd_bwd)):
            for _ in range(warmup):
                fn()
            ctx.barrier()
            a, b = ev(), ev()
            a.record()
            for i in range(steps):
                r = fn()
                if dump_dir is not None and fn is fwd_bwd and i == steps - 1:
                    last = r
                del r
            b.record()
            torch.cuda.synchronize()
            res[key] = ctx.max_over_ranks(a.elapsed_time(b)) / steps * 1e3
    launches = ctx.cabi.launch_count() - launches0
    if last is not None and ctx.rank == 0:
        out, grads = last
        dump_outputs(dump_dir, {"out": out, **{"grad_" + k: t for k, t in zip(maps, grads)}}, 1, C1["H"], C1["W"])
    del last
    # the kernels alone (CUDA graph replay of the same two launches: no host time between them)
    graph_us = None
    try:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            fwd_bwd()
        torch.cuda.current_stream().wait_stream(s)
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            fwd_bwd()
        for _ in range(warmup):
            gr.replay()
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        for _ in range(steps):
            gr.replay()
        b.record()
        torch.cuda.synchronize()
        graph_us = a.elapsed_time(b) / steps * 1e3
    except Exception as e:  # pragma: no cover
        graph_us = f"capture failed: {str(e)[:80]}"
    texels = C1["H"] * C1["W"]
    return {"value": texels * ctx.world / (res["fwd_bwd_us"] * 1e-6) / 1e9, "unit": UNIT, "ms_per_step": res["fwd_bwd_us"] * 1e-3,
            "steps": steps, "warmup": warmup, **res, "fwd_bwd_cuda_graph_us": graph_us,
            "config": {"workload": C1["workload"], "H": C1["H"], "W": C1["W"], "lights": 1,
                       "inputs": "tests/golden/config1_tiles_256.npz + config1_tiles_256.in_normal.npz (the reference's tests/data/tiles "
                                 "material, its own loader + resize)",
                       "l2": "2 MB of maps: L2-resident by nature of the config (a single small material); the number is launch latency, not bandwidth"},
            "roofline": {"bound": "launch latency", "note": "0.26 Mtexel per call: 120 B/texel x 65536 texels = 7.9 MB per fwd+bwd, ~1.2 us at the HBM roof"},
            "gpu_launches": int(launches), "clocks": clk.summary()}


# ---------------------------------------------------------------------------------------------- e2e legs (host buffers)
class _Pipe:
    """Software pipeline over (step, chunk) units: the H2D copy of unit i+1 runs on a copy stream while unit i is
    computed; two device staging slots, guarded by events (ready: copy done; free: compute done with the slot)."""

    def __init__(self, dev):
        self.dev = dev
        self.copy = torch.cuda.Stream(device=dev)
        self.ready = [torch.cuda.Event(), torch.cuda.Event()]
        self.free = [torch.cuda.Event(), torch.cuda.Event()]
        self.used = [False, False]

    def upload(self, slot, fn):
        with torch.cuda.stream(self.copy):
            if self.used[slot]:
                self.copy.wait_event(self.free[slot])
            fn()
            self.ready[slot].record(self.copy)

    def acquire(self, slot):
        torch.cuda.current_stream(self.dev).wait_event(self.ready[slot])

    def release(self, slot):
        self.free[slot].record(torch.cuda.current_stream(self.dev))
        self.used[slot] = True


def measure_e2e(ctx, cfg, steps, warmup):
    """End to end through the public API with HOST buffers (C2 shape).  Three legs, all chunk-pipelined (H2D of the next
    chunk overlaps the kernels of the current one), wall clock between two device synchronisations, max over ranks:
      primary      : uint8 textures (B,H,W,C) in pinned memory -> H2D -> pbr_ingest_image -> brdf() (K1) -> autograd backward
                     (K2) -> D2H of d(light intensity), the reduction the backward delivers (12 bytes)
      f32_maps_grads_to_host : float32 maps in pinned memory -> H2D -> K1 -> K2 -> D2H of every map gradient (32 B/texel)
      fit_uint8    : uint8 textures -> H2D -> ingest -> fused loss kernel (K3: render + MSE + backward) -> D2H of the loss
    Each leg: `warmup` steps, then `steps` timed steps.
    """
    from pypbr_b200.fit import fused_loss_step
    from pypbr_b200.materials import BasecolorMetallicMaterial
    from pypbr_b200.materials._ingest import NORMAL3, PLAIN, ingest_uint
    from pypbr_b200.models import CookTorranceBRDF

    dev, rank, world = ctx.dev, ctx.rank, ctx.world
    B, H, W, L = cfg["B"], cfg["H"], cfg["W"], cfg["L"]
    chunk = 8
    n_chunks = B // chunk
    texel_lights_per_step = B * H * W * L * world
    lights, inten = lights_for(L)
    view = torch.tensor([0.0, 0.0, 1.0], device=dev)
    lights_d, inten_d = lights.to(dev), inten.to(dev)
    brdf = CookTorranceBRDF("point")
    names = (("albedo", 3), ("normal", 3), ("roughness", 1), ("metallic", 1))
    g = torch.Generator(device=dev).manual_seed(123 + rank)
    grad_out = torch.rand(chunk, 3, H, W, generator=g, device=dev)      # upstream gradient: resident, like in `value`
    target = torch.rand(chunk, 3, H, W, generator=g, device=dev)

    def timed(run_step, finish, n):
        for s in range(warmup):
            run_step(s)
        finish()
        ctx.barrier()
        t0 = time.perf_counter()
        for s in range(n):
            run_step(s)
        finish()
        torch.cuda.synchronize()
        return ctx.max_over_ranks(time.perf_counter() - t0)

    legs = {}
    # ---- uint8 textures
    g8 = torch.Generator().manual_seed(77 + rank)
    host8 = {k: torch.randint(0, 256, (B, H, W, c), dtype=torch.uint8, generator=g8).pin_memory() for k, c in names}
    h2d8 = sum(v.numel() for v in host8.values())
    stage8 = [{k: torch.empty((chunk, H, W, c), dtype=torch.uint8, device=dev) for k, c in names} for _ in range(2)]
    result_host = torch.zeros(16, 3, dtype=torch.float32).pin_memory()
    loss_host = torch.zeros(16, dtype=torch.float32).pin_memory()
    pipe = _Pipe(dev)
    unit = [0]

    # the ceiling of this leg on this host at this N: the same pinned buffers copied to the device with nothing else going on,
    # every rank at once (tools/h2d_scaling.py: 55 / 111 / 115 / 187 GB/s in total at 1 / 2 / 4 / 8 ranks on the 8-GPU box)
    ceil_dst = {k: torch.empty_like(v, device=dev) for k, v in host8.items()}

    def copy_all():
        for k in host8:
            ceil_dst[k].copy_(host8[k], non_blocking=True)

    copy_all()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(4):
        copy_all()
    torch.cuda.synchronize()
    h2d_ceiling = 4 * h2d8 / ctx.max_over_ranks(time.perf_counter() - t0) / 1e9
    del ceil_dst

    def chunk_material(slot, requires_grad):
        m = BasecolorMetallicMaterial(albedo_is_srgb=True, device=dev)
        leaves = []
        for k, _c in names:
            t = ingest_uint(stage8[slot][k], dev, NORMAL3 if k == "normal" else PLAIN)
            t.requires_grad_(requires_grad)
            m._maps[k] = t
            leaves.append(t)
        return m, leaves

    def upload8(i):
        slot, c = i % 2, i % n_chunks
        pipe.upload(slot, lambda: [stage8[slot][k].copy_(host8[k][c * chunk:(c + 1) * chunk], non_blocking=True) for k, _ in names])

    def step_render_grad_u8(s):
        acc = torch.zeros(1, 3, device=dev)
        for c in range(n_chunks):
            i = unit[0]
            if i == 0:
                upload8(0)
            upload8(i + 1)                      # next unit (of this or the next step) travels while this one is shaded
            slot = i % 2
            pipe.acquire(slot)
            m, leaves = chunk_material(slot, True)
            it = inten_d.clone().requires_grad_(True)
            out = brdf(m, view, lights_d, it, 1.0)
            grads = torch.autograd.grad(out, leaves + [it], grad_out)
            pipe.release(slot)
            acc += grads[-1]
            unit[0] += 1
        result_host[s % 16].copy_(acc[0], non_blocking=True)   # D2H of the step's result

    def finish():
        torch.cuda.synchronize()
        unit[0] = 0
        pipe.used = [False, False]

    dt = timed(step_render_grad_u8, finish, steps)
    primary = {"value": texel_lights_per_step * steps / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d8, "d2h_bytes_per_step": 12,
               "steps": steps, "warmup": warmup, "ms_per_step": dt / steps * 1e3,
               "path": "pinned host uint8 (B,H,W,C) textures -> H2D in chunks of 8 materials (copy stream, double-buffered) -> pbr_ingest_image x4 -> "
                       "CookTorranceBRDF.__call__ (pbr_ct_forward) -> torch.autograd.grad (pbr_ct_backward; map gradients stay in HBM for the optimiser) -> "
                       "D2H of d(light_intensity) (12 bytes)",
               "h2d_gbs": h2d8 / (dt / steps) / 1e9, "h2d_ceiling_gbs": h2d_ceiling,
               "frac_of_h2d_ceiling": h2d8 / (dt / steps) / 1e9 / h2d_ceiling,
               "bound": "host->device copy rate of this host at this many ranks (h2d_ceiling_gbs: the same buffers copied with no kernels "
                        "running, all ranks at once, measured in this run)", "numa": ctx.numa}

    def step_fit_u8(s):
        for c in range(n_chunks):
            i = unit[0]
            if i == 0:
                upload8(0)
            upload8(i + 1)
            slot = i % 2
            pipe.acquire(slot)
            m, _ = chunk_material(slot, False)
            buf, _g = fused_loss_step(m, target, view, lights_d, inten_d, "point", 1.0, multi_light="accumulate", out=fit_bufs)
            pipe.release(slot)
            loss_acc.add_(buf[0])
            unit[0] += 1
        loss_host[s % 16].copy_(loss_acc[0], non_blocking=True)
        loss_acc.zero_()

    fit_bufs, loss_acc = {}, torch.zeros(1, device=dev)
    dt = timed(step_fit_u8, finish, steps)
    legs["fit_uint8"] = {"value": texel_lights_per_step * steps / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d8, "d2h_bytes_per_step": 4,
                         "steps": steps, "ms_per_step": dt / steps * 1e3, "h2d_gbs": h2d8 / (dt / steps) / 1e9,
                         "path": "pinned host uint8 textures -> H2D (chunked, overlapped) -> pbr_ingest_image x4 -> pypbr_b200.fit.fused_loss_step "
                                 "(pbr_ct_loss_fwd_bwd: render + MSE + backward in one launch) -> D2H of the loss (4 bytes)"}
    del host8, stage8

    # ---- float32 maps in, every map gradient out (full duplex over PCIe)
    host = synth_maps(B, H, W, torch.device("cpu"), 5 + rank, pin=True)
    h2d = sum(v.numel() * 4 for v in host.values())
    host_grads = {k: torch.empty(v.shape, dtype=torch.float32).pin_memory() for k, v in host.items()}
    stage = [{k: torch.empty((chunk, *v.shape[1:]), dtype=torch.float32, device=dev) for k, v in host.items()} for _ in range(2)]
    d2h_stream = torch.cuda.Stream(device=dev)

    def upload32(i):
        slot, c = i % 2, i % n_chunks
        pipe.upload(slot, lambda: [stage[slot][k].copy_(host[k][c * chunk:(c + 1) * chunk], non_blocking=True) for k in host])

    def step_f32(s):
        for c in range(n_chunks):
            i = unit[0]
            if i == 0:
                upload32(0)
            upload32(i + 1)
            slot = i % 2
            pipe.acquire(slot)
            m, leaves = make_material({k: stage[slot][k].detach() for k in host}, dev, True)
            out = brdf(m, view, lights_d, inten_d, 1.0)
            grads = torch.autograd.grad(out, leaves, grad_out)
            pipe.release(slot)
            done = torch.cuda.Event()
            done.record()
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(done)
                for k, gt in zip(host, grads):
                    host_grads[k][c * chunk:(c + 1) * chunk].copy_(gt, non_blocking=True)
                    gt.record_stream(d2h_stream)
            unit[0] += 1

    dt = timed(step_f32, finish, steps)
    legs["f32_maps_grads_to_host"] = {
        "value": texel_lights_per_step * steps / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": h2d,
        "steps": steps, "ms_per_step": dt / steps * 1e3, "h2d_gbs": h2d / (dt / steps) / 1e9,
        "path": "pinned host float32 maps -> H2D (chunked, overlapped) -> pbr_ct_forward -> pbr_ct_backward -> D2H of all four map gradients "
                "into pinned host memory (third stream; PCIe full duplex)"}
    primary["legs"] = legs
    return primary


def run_ours(args):
    ctx = Ctx()
    name = args.config
    steps, warmup = args.steps, max(args.warmup, 3)
    if name == "c1":
        res = measure_c1(ctx, steps, warmup, dump_dir=args.dump_outputs)
    else:
        res = measure_shading(name, args, ctx, steps, warmup, dump_dir=args.dump_outputs)
    line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": ctx.world, "steps": res["steps"], "warmup": res["warmup"],
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": res["config"], "roofline": res["roofline"]}
    for k in ("allreduce", "loss", "fwd_us", "fwd_bwd_us", "fwd_bwd_cuda_graph_us"):
        if k in res:
            line[k] = res[k]
    torch.cuda.empty_cache()
    solo = ctx.rank == 0 and ctx.world == 1
    line["cpu_baseline"] = cpu_baseline_for(name) if (solo and not args.no_cpu) else None
    line["gpu_eager_baseline"] = gpu_eager_baseline(name, ctx.dev, res["value"]) if (solo and not args.no_eager) else None
    line["e2e"] = measure_e2e(ctx, CONFIGS["c2"], steps, warmup) if (name == "c2" and not args.no_e2e) else None
    torch.cuda.empty_cache()
    line["gpu_launches"] = res["gpu_launches"]
    line["clocks"] = res["clocks"]
    if name == "c2" and not args.no_configs:
        # the other shading configs of BASELINE.json under the same clock (VERDICT r1: the multi-light kernels and the one
        # path with a collective must be in the driver-run line, at every N)
        cfgs = {}
        for k in ("c1", "c3", "c5"):
            r = measure_c1(ctx, steps, warmup) if k == "c1" else measure_shading(k, args, ctx, steps, warmup)
            if solo and not args.no_cpu:
                r["cpu_baseline"] = cpu_baseline_for(k, reps=2, budget_s=6.0)
            if solo and not args.no_eager and k == "c1":
                r["gpu_eager_baseline"] = gpu_eager_baseline(k, ctx.dev, r["value"])
            cfgs[k] = r
            torch.cuda.empty_cache()
        # the conversion + blend pipeline has no multi-GPU dimension (two materials): rank 0's GPU alone
        if ctx.rank == 0:
            c4 = run_c4(args, emit=False)
            cfgs["c4"] = {"value": c4["value"], "unit": c4["unit"], "metric": c4["metric"], "ms_per_step": c4["ms_per_step"], "steps": c4["steps"],
                          "warmup": c4["warmup"], "config": c4["config"], "roofline": c4["roofline"], "gpu_launches": c4["gpu_launches"],
                          "clocks": c4["clocks"]}
            if solo and not args.no_cpu:
                cfgs["c4"]["cpu_baseline"] = c4_cpu_sample(reps=1)
            torch.cuda.empty_cache()
        ctx.barrier()
        line["configs"] = cfgs
    if ctx.rank == 0:
        print(json.dumps(line), flush=True)
    ctx.close()


# ---------------------------------------------------------------------------------------------- config 4
def run_c4(args, emit=True, dump_dir=None):
    """
    BASELINE.json configs[3] (SURVEY.md §8d "C4"): two 4096x4096 metallic materials (albedo, normal, roughness,
    metallic, height) -> to_diffuse_specular_material() on each -> blend_materials(d1, d2, "mask", mask) ->
    blend_materials(m1, m2, "height").  Two measurements:
      pipeline : the four public-API calls back to back (host allocation and descriptor setup included; no device->host
                 read-back happens inside: the stream is never drained), CUDA-event time per pipeline
      kernels  : every kernel on its own through the C ABI on preallocated buffers (launches back to back between
                 two CUDA events), algorithmic bytes / time against the measured HBM peak
    Each: warm-up, then --steps timed repetitions.  dump_dir: write what the last timed pipeline returned there
    (dump_outputs): the maps of both blended materials and the height blend's mask.
    """
    from pypbr_b200 import _cabi
    from pypbr_b200.blending import blend_materials
    from pypbr_b200.materials import BasecolorMetallicMaterial

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the conversion / blend path has no CPU fallback)")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    lib = _cabi.load()
    H, W = C4["H"], C4["W"]
    texels = H * W
    peak, peak_src = measured_peak()
    st = _cabi.stream_ptr(dev)

    def material(seed):
        m = synth_maps(1, H, W, dev, seed)
        g = torch.Generator(device=dev).manual_seed(seed + 50)
        mat = BasecolorMetallicMaterial(albedo_is_srgb=True, device=dev)
        for k, v in m.items():
            mat._maps[k] = v[0]
        mat._maps["height"] = torch.rand(1, H, W, generator=g, device=dev)
        return mat

    m1, m2 = material(4001), material(4002)
    mask = torch.rand(1, H, W, generator=torch.Generator(device=dev).manual_seed(4003), device=dev)

    def pipeline():
        d1 = m1.to_diffuse_specular_material()
        d2 = m2.to_diffuse_specular_material()
        b1, _ = blend_materials(d1, d2, "mask", mask=mask)
        b2, mk = blend_materials(m1, m2, "height", blend_width=0.1)
        return b1, b2, mk

    ev = lambda: torch.cuda.Event(enable_timing=True)
    steps, warmup = args.steps, max(args.warmup, 3)
    for _ in range(warmup):
        pipeline()
    torch.cuda.synchronize()
    l0 = _cabi.launch_count()
    e0, e1 = ev(), ev()
    with ClockSampler(local) as clk:
        e0.record()
        for i in range(steps):
            r = pipeline()
            if dump_dir is not None and i == steps - 1:
                last = r
            del r
        e1.record()
        torch.cuda.synchronize()
    launches = _cabi.launch_count() - l0
    pipe_ms = e0.elapsed_time(e1) / steps
    if dump_dir is not None:
        b1, b2, mk = last
        out = {f"mask_blend_{k}": t for k, t in b1._maps.items() if t is not None}
        out.update({f"height_blend_{k}": t for k, t in b2._maps.items() if t is not None}, height_mask=mk)
        dump_outputs(dump_dir, out, 1, H, W)
        del last, b1, b2, mk, out

    # kernel-only legs through the C ABI
    d1 = m1.to_diffuse_specular_material()
    d2 = m2.to_diffuse_specular_material()

    def timed(fn):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps

    kernels = {}

    def add(name, ms, bytes_per_texel):
        ach = bytes_per_texel * texels / (ms * 1e-3) / 1e9
        kernels[name] = {"ms": ms, "bytes_per_texel": bytes_per_texel, "achieved": ach, "frac": ach / peak}

    o0, o1 = torch.empty(3, H, W, device=dev), torch.empty(3, H, W, device=dev)
    cd = _cabi.PbrConvDesc(1, H, W, 1, _cabi.plane(m1.albedo), _cabi.plane(m1.metallic), _cabi.plane(o0), _cabi.plane(o1))
    add("convert_m2s (K4)", timed(lambda: _cabi.check(lib.pbr_convert_m2s(_cabi.byref(cd), st), "m2s")), 16 + 24)
    cs = _cabi.PbrConvDesc(1, H, W, 0, _cabi.plane(d1.albedo), _cabi.plane(d1.specular), _cabi.plane(o0), _cabi.plane(o1))
    add("convert_s2m (K5)", timed(lambda: _cabi.check(lib.pbr_convert_s2m(_cabi.byref(cs), st), "s2m")), 24 + 24)
    res = torch.full((1,), float("inf"), device=dev)
    nd = _cabi.PbrNormalDesc(1, H, W, 3, _cabi.plane(m1.normal), _cabi.plane(None))
    add("normal_min probe (K7)", timed(lambda: _cabi.check(lib.pbr_normal_min(_cabi.byref(nd), res.data_ptr(), st), "nmin")), 12)

    def blend_desc(a, b, names, mode):
        d = _cabi.PbrBlendDesc()
        d.B, d.H, d.W, d.mask_mode = 1, H, W, mode
        d.blend_width, d.shift, d.apply_shift = 0.1, 0.0, 1
        outs, ch_total = [], 0
        for i, n in enumerate(names):
            ta, tb = a._maps[n], b._maps[n]
            out = torch.empty_like(ta)
            outs.append(out)
            d.maps[i] = _cabi.PbrBlendMap(_cabi.plane(ta), _cabi.plane(tb), _cabi.plane(out), ta.shape[0], int(n == "normal"))
            ch_total += ta.shape[0]
        d.n_maps = len(names)
        d.normal_min = res.data_ptr()
        return d, outs, ch_total

    bd, keep1, ch = blend_desc(d1, d2, ["albedo", "normal", "roughness", "specular"], _cabi.MASK_GIVEN)
    bd.mask = _cabi.plane(mask)
    add("blend, given mask, diffuse-specular pair (K6)", timed(lambda: _cabi.check(lib.pbr_blend(_cabi.byref(bd), st), "blend")),
        4 * (2 * ch + 1) + 4 * ch)
    bh, keep2, ch2 = blend_desc(m1, m2, ["albedo", "height", "metallic", "normal", "roughness"], _cabi.MASK_SIGMOID)
    mask_out = torch.empty(1, H, W, device=dev)
    bh.prop1, bh.prop2, bh.mask_out = _cabi.plane(m1.height), _cabi.plane(m2.height), _cabi.plane(mask_out)
    # the two height planes are read twice by one thread (mask builder + the height map's own lerp): second read is L1/L2
    add("blend, height sigmoid, metallic pair (K6)", timed(lambda: _cabi.check(lib.pbr_blend(_cabi.byref(bh), st), "blend")),
        4 * (2 * ch2) + 4 * ch2 + 4)

    # what the pipeline has to move: two conversions + the two blends.  The `normal.min() < 0` probes of base.py:212 cost no
    # bytes here: the converted materials re-use the probe result of the very same normal tensor (memoised by identity and
    # version counter), the blends fold the probe into the blend kernel and decide the remap on the device.
    total_bytes = texels * (2 * 40 + kernels["blend, given mask, diffuse-specular pair (K6)"]["bytes_per_texel"]
                            + kernels["blend, height sigmoid, metallic pair (K6)"]["bytes_per_texel"])
    dom = max(kernels.items(), key=lambda kv: kv[1]["ms"])
    line = {
        "metric": "Gtexel/s conversion + blend pipeline", "value": texels / (pipe_ms * 1e-3) / 1e9, "unit": "Gtexel/s",
        "n_gpus": 1, "steps": steps, "warmup": warmup, "ms_per_step": pipe_ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": C4["workload"], "H": H, "W": W,
                   "pipeline": "2 x to_diffuse_specular_material + blend_materials(mask) + blend_materials(height), public API",
                   "l2": "every kernel streams 0.6-2 GB, far above the 126 MB L2; no flush needed"},
        "roofline": {"bound": "hbm", "kernel": dom[0], "achieved": dom[1]["achieved"], "peak": peak, "unit": "GB/s",
                     "frac": dom[1]["frac"], "traffic": None, "peak_source": peak_src,
                     "pipeline_algorithmic_bytes": total_bytes,
                     "pipeline_frac": total_bytes / (pipe_ms * 1e-3) / 1e9 / peak, "kernels": kernels},
        "cpu_baseline": None, "e2e": None, "gpu_launches": int(launches), "clocks": clk.summary(),
    }
    if not emit:
        return line
    if not args.no_cpu:
        line["cpu_baseline"] = c4_cpu_sample(reps=1)
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------- aux rows (SURVEY.md 8f)
def run_aux(args):
    """Kernel-only timings of the rows either side of the shading path: image ingestion, index transforms, Adam.  Each
    kernel: warm-up, then --steps timed launches."""
    from pypbr_b200 import _cabi
    from pypbr_b200.fit import FusedAdam
    from pypbr_b200.materials import BasecolorMetallicMaterial
    from pypbr_b200.materials._ingest import NORMAL3, PLAIN, ingest_uint

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device")
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    _cabi.load()
    B, H, W = 16, 2048, 2048
    texels = B * H * W
    peak, peak_src = measured_peak()
    ev = lambda: torch.cuda.Event(enable_timing=True)
    steps, warmup = args.steps, max(args.warmup, 3)

    def timed(fn):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        a, b = ev(), ev()
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / steps

    kernels = {}

    def add(name, ms, nbytes):
        ach = nbytes / (ms * 1e-3) / 1e9
        kernels[name] = {"ms": ms, "algorithmic_bytes": nbytes, "achieved": ach, "frac": ach / peak}

    l0 = _cabi.launch_count()
    with ClockSampler(local) as clk:
        g = torch.Generator(device=dev).manual_seed(8)
        rgb8 = torch.randint(0, 256, (B, H, W, 3), dtype=torch.uint8, device=dev, generator=g)
        add("ingest uint8 RGB -> float32 planar", timed(lambda: ingest_uint(rgb8, dev, PLAIN)), texels * (3 + 12))
        add("ingest uint8 RGB -> unit normal", timed(lambda: ingest_uint(rgb8, dev, NORMAL3)), texels * (3 + 12))
        del rgb8
        maps = synth_maps(B, H, W, dev, 9)
        mat = BasecolorMetallicMaterial(albedo_is_srgb=True, device=dev)

        def reset():
            for k, v in maps.items():
                mat._maps[k] = v

        def flip():
            reset()
            mat.flip_horizontal()

        def rollit():
            reset()
            mat.roll((17, -33))

        add("flip_horizontal, 4 maps (8 channels) in one gather", timed(flip), texels * 8 * 8)
        add("roll, 4 maps (8 channels) in one gather", timed(rollit), texels * 8 * 8)
        reset()
        # the functional transform a user calls (pypbr_b200.transforms): a NEW material, the source untouched.  It starts from a
        # tensor-sharing copy, so the step moves 8 B per channel-texel; the reference's scheme (deep clone, then the method on
        # the clone) moves 16.
        from pypbr_b200.transforms import functional as TFn

        add("transforms.functional.flip_horizontal (public API, new material)", timed(lambda: TFn.flip_horizontal(mat)), texels * 8 * 8)

        def clone_then_flip():
            m2 = mat.clone()
            m2.flip_horizontal()

        add("clone() + flip_horizontal() (the reference's scheme, same kernels)", timed(clone_then_flip), texels * 8 * 8)
        opt = FusedAdam({k: v for k, v in maps.items()}, lr=1e-3)
        grads = {k: torch.rand_like(v) for k, v in maps.items()}
        add("Adam + projection, 4 maps (8 channels)", timed(lambda: opt.step(grads)), texels * 8 * 28)
        del opt, grads
        from pypbr_b200.utils import compute_normal_from_height, rotate_normals

        height = torch.rand(B, 1, H, W, device=dev, generator=g)
        add("compute_normal_from_height (1 ch in, 3 ch out)", timed(lambda: compute_normal_from_height(height, 2.0)), texels * 16)
        nrm = maps["normal"].clone()
        add("rotate_normals in place (3 ch)", timed(lambda: rotate_normals(nrm, 33.0)), texels * 24)
    launches = _cabi.launch_count() - l0
    dom = max(kernels.items(), key=lambda kv: kv[1]["ms"])
    line = {
        "metric": "GB/s of the ingestion / index-transform / optimiser kernels", "value": dom[1]["achieved"], "unit": "GB/s",
        "n_gpus": 1, "steps": steps, "warmup": warmup, "ms_per_step": dom[1]["ms"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"SURVEY 8f rows on {B} materials {H}x{W}: image ingestion, index transforms, Adam step, normal utilities",
                   "l2": "every kernel streams 1-15 GB, far above the 126 MB L2; no flush needed"},
        "roofline": {"bound": "hbm", "kernel": dom[0], "achieved": dom[1]["achieved"], "peak": peak, "unit": "GB/s",
                     "frac": dom[1]["frac"], "traffic": None, "peak_source": peak_src, "kernels": kernels},
        "cpu_baseline": None, "e2e": None, "gpu_launches": int(launches), "clocks": clk.summary(),
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=["c1"] + sorted(list(CONFIGS) + ["c4", "aux"]))
    ap.add_argument("--fit", default="one-launch", choices=["one-launch", "one-launch-sync", "two-kernel"],
                    help="c5: pbr_ct_fit_step with the loss all-reduce on a side stream (default) or on the compute stream, "
                         "or pbr_ct_loss_fwd_bwd + pbr_adam_step")
    ap.add_argument("--shared-grads", action="store_true",
                    help="c5 --fit two-kernel: also d(light intensity, light position, view direction), the fit with unknown lighting")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-eager", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="c2: skip the c1 / c3 / c5 block of the line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="c1-c5: after the timed steps, write what the last one returned as DIR/<name>.npy (a fixed "
                         "sample of texel positions, under 64 MB in all); the inputs are the same on every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "ours" or args.config == "aux"):
        ap.error("--dump-outputs covers the timed paths of --config c1-c5 (--impl ours)")
    if args.impl == "reference":
        if args.config == "aux":
            raise SystemExit("bench.py: the reference arm is defined for c1-c5")
        return run_reference_arm(args)
    if args.config == "c4":
        return run_c4(args, dump_dir=args.dump_outputs)
    if args.config == "aux":
        return run_aux(args)
    run_ours(args)


if __name__ == "__main__":
    main()
