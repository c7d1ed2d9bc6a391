"""bench.py's reference arm runs on the host cores, so its JSON line - and with it the key contract the driver reads
from both arms - can be checked without a GPU."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["gpu_launches"] == 0
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["unit"] == "Gtexel-lights/s" and d["higher_is_better"] is True and d["vs_baseline"] is None and d["value"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the other shading configs of BASELINE.json ride along as bounded samples on the same host cores
    assert set(d["configs"]) == {"c1", "c3", "c5"}
    for k, c in d["configs"].items():
        assert c["value"] > 0 and c["kind"] == "port" and c["cores"] >= 1 and c["sample"] and c["workload"], k
    assert d["configs"]["c1"]["fwd_us"] > 0 and d["configs"]["c1"]["fwd_bwd_us"] >= d["configs"]["c1"]["fwd_us"] * 0.5


def test_reference_arm_times_the_conversion_and_blend_pipeline():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "c4", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][0])
    assert d["impl"] == "reference" and d["unit"] == "Gtexel/s" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port"
    assert "2048x2048" in d["config"]["sample"]


def test_traffic_capture_is_dropped_when_the_kernel_sources_changed(tmp_path, monkeypatch):
    """roofline.traffic comes from a committed ncu capture; it is only reported while profiles/traffic.json carries the hash
    of the very kernel sources the library is built from."""
    sys.path.insert(0, ROOT)
    import bench

    prof = tmp_path / "profiles"
    prof.mkdir()
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    os.makedirs(tmp_path / "pypbr_b200" / "csrc")
    os.makedirs(tmp_path / "include")
    (tmp_path / "pypbr_b200" / "csrc" / "k.cu").write_text("__global__ void k() {}")
    (tmp_path / "include" / "pbrcuda.h").write_text("/* abi */")
    h = bench.csrc_sha16()
    (prof / "traffic.json").write_text(json.dumps({"_csrc_sha16": h, "c2:backward": {"bytes": 5.0e9}}))
    assert bench.measured_traffic("c2:backward") == {"bytes": 5.0e9}
    (tmp_path / "pypbr_b200" / "csrc" / "k.cu").write_text("__global__ void k() { }")
    assert bench.measured_traffic("c2:backward") is None


def test_dump_outputs_writes_the_same_texel_sample_of_every_array(tmp_path, monkeypatch):
    """--dump-outputs: float32 (texels, channels) arrays at one fixed set of positions, the whole arrays when they fit, the
    budget kept, other arrays whole in float64."""
    import numpy as np
    import torch

    sys.path.insert(0, ROOT)
    import bench

    B, H, W = 3, 20, 24
    out = torch.arange(B * 3 * H * W, dtype=torch.float32).reshape(B, 3, H, W)
    arrays = {"out": out, "grad_roughness": out[:, :1] * 2 + 1, "loss_buffer": torch.tensor([5.0, 1.0])}
    bench.dump_outputs(str(tmp_path / "all"), arrays, B, H, W)
    a = np.load(tmp_path / "all" / "out.npy")
    assert a.dtype == np.float32 and np.array_equal(a, out.permute(0, 2, 3, 1).reshape(-1, 3).numpy())
    assert np.load(tmp_path / "all" / "loss_buffer.npy").dtype == np.float64
    monkeypatch.setattr(bench, "DUMP_BYTES", 4 * 4 * 500)   # room for 500 texels of 4 channels
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, B, H, W)
    o, r = np.load(tmp_path / "a" / "out.npy"), np.load(tmp_path / "a" / "grad_roughness.npy")
    assert 400 < o.shape[0] <= 500 and o.shape == (r.shape[0], 3) and r.shape[1] == 1
    assert np.array_equal(r[:, 0], o[:, 0] * 2 + 1)                    # same positions in every array
    assert np.all(np.diff(o[:, 0]) > 0)                                 # sorted, no repeats
    for k in arrays:
        assert np.array_equal(np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy")), k
    bench.dump_outputs(str(tmp_path / "one"), {"mask": out[0, :1], "albedo": out[1]}, 1, H, W)   # (C, H, W) maps, B = 1
    m, a = np.load(tmp_path / "one" / "mask.npy"), np.load(tmp_path / "one" / "albedo.npy")
    assert m.shape == (m.shape[0], 1) and a.shape == (m.shape[0], 3) and 400 < m.shape[0] <= 500
    assert np.array_equal(a[:, 0] - m[:, 0], np.full(m.shape[0], 3 * H * W, np.float32))   # same positions


@pytest.mark.gpu
@pytest.mark.parametrize("config", ["c1", "c4"])
def test_steps_and_dump_outputs_of_the_gpu_arm(config, tmp_path):
    """--steps sets the timed steps of the line, and --dump-outputs writes what the last one returned."""
    import numpy as np

    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", config, "--steps", "4", "--warmup", "1",
                          "--no-cpu", "--no-eager", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])
    assert d["steps"] == 4 and d["warmup"] == 3
    arrays = {p.name[:-4]: np.load(p) for p in tmp_path.glob("*.npy")}
    assert sum(p.stat().st_size for p in tmp_path.glob("*.npy")) < 64e6
    want = {"out", "grad_albedo", "grad_normal", "grad_roughness", "grad_metallic"} if config == "c1" else {"height_mask", "mask_blend_albedo"}
    assert want <= set(arrays), sorted(arrays)
    n = arrays["out" if config == "c1" else "height_mask"].shape[0]
    assert all(a.dtype == np.float32 and a.ndim == 2 and a.shape[0] == n and np.isfinite(a).all() for a in arrays.values())
    if config == "c1":
        assert n == 256 * 256 and d["fwd_bwd_us"] > 0


def test_baseline_metric_and_configs_are_the_ones_benched():
    sys.path.insert(0, ROOT)
    import bench

    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert bench.C1["workload"] == base["configs"][0]
    assert bench.CONFIGS["c2"]["workload"] == base["configs"][1]
    assert bench.CONFIGS["c3"]["workload"] == base["configs"][2]
    assert bench.C4["workload"] == base["configs"][3]
    assert (bench.CONFIGS["c2"]["B"], bench.CONFIGS["c2"]["H"], bench.CONFIGS["c2"]["L"]) == (64, 1024, 1)
    assert (bench.CONFIGS["c3"]["B"], bench.CONFIGS["c3"]["H"], bench.CONFIGS["c3"]["L"]) == (16, 2048, 16)
    assert (bench.CONFIGS["c5"]["B"], bench.CONFIGS["c5"]["H"], bench.CONFIGS["c5"]["L"]) == (512, 512, 8)
