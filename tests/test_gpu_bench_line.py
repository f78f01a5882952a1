"""The bench contract on a tiny swarm: `python bench.py` prints exactly ONE JSON line on stdout with the keys the driver
and the judge read, for both arms."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from multidronesim_b200._lib import STAT_NAMES

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
            "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"}


def run(args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    return json.loads(lines[0])


@pytest.mark.gpu
def test_gpu_arm_line(tmp_path):
    d = run(["--envs", "2048", "--steps", "3", "--warmup", "3", "--fuse", "8", "--settle", "16", "--e2e-steps", "4", "--cpu-seconds", "1",
             "--dump-outputs", str(tmp_path)])
    obs_log, st = np.load(tmp_path / "obs_log.npy"), np.load(tmp_path / "rollout_stats.npy")
    assert obs_log.shape == (8, 2048, 8, 20) and obs_log.dtype == np.float32 and np.isfinite(obs_log).all()   # every env fits the sample
    assert st.dtype == np.float64 and st.tolist() == [d["rollout_stats"][k] for k in STAT_NAMES]
    assert REQUIRED <= set(d), REQUIRED - set(d)
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 3 and d["gpu_launches"] == 3 * 2 and d["dtype"] == "f32"   # two sub-swarm streams, one launch each per step
    assert d["rollout_stats"]["drone_steps"] == 2048 * 8 * 8 * 3
    r = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and 0 < r["frac"] < 1.5
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    for k in ("roofline_ctrl", "roofline_physics"):
        assert d[k]["bound"] == "hbm" and 0 < d[k]["frac"] < 1.5
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] == 2048 * 8 * 11 * 4 and e["d2h_bytes_per_step"] == 2048 * 8 * 20 * 4
    assert e["pcie_ceiling"]["value"] > 0 and 0 < e["frac_of_pcie_ceiling"] < 1.5 and e["fused"]["value"] > 0
    c = d["cpu_baseline"]
    assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["value"] > 0 and "sample" in c
    if c["kind"] == "reference":   # the reference's own classes were importable: the numpy port is reported beside them
        assert d["cpu_baseline_port"]["kind"] == "port" and d["cpu_baseline_port"]["value"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    assert d["strong"]["efficiency"] == 1.0 and d["strong"]["total_envs"] == 2048
    assert "frac_counters" in r and "peak_nominal" in r
    cf = d["configs"]
    assert set(cf) == {"C2_4096", "C3_o2_16384", "C4_65536_f64", "C5_f64"}
    for k, v in cf.items():
        assert v["value"] > 0 and 0 < v["roofline"]["frac"] < 1.5 and "clocks" in v, k


def test_dump_outputs_samples_and_crops(monkeypatch, tmp_path):
    """bench.dump_outputs on host tensors: a seeded sample of environments drawn across two sub-swarm logs, and the last
    control steps only when one environment's log exceeds the byte budget"""
    import torch
    import bench
    F, sizes = 6, (9, 14)
    rings = [torch.randn(F, e, 8, 20, generator=torch.Generator().manual_seed(p)) for p, e in enumerate(sizes)]
    whole = torch.cat(rings, dim=1).numpy()
    stats = torch.arange(8, dtype=torch.float64)
    slot = 8 * 20 * 4
    for n_envs, budget, T in ((5, 1 << 20, F), (23, 1 << 20, F), (4, 4 * slot, 4)):
        monkeypatch.setattr(bench, "DUMP_ENVS", n_envs)
        monkeypatch.setattr(bench, "DUMP_BYTES", budget)
        bench.dump_outputs(str(tmp_path), rings, stats)
        n = min(n_envs, budget // (T * slot))
        envs = np.sort(np.random.default_rng(0).choice(sum(sizes), n, replace=False))
        got = np.load(tmp_path / "obs_log.npy")
        assert got.shape == (T, n, 8, 20) and np.array_equal(got, whole[F - T:, envs]), (n_envs, budget)
        assert np.array_equal(np.load(tmp_path / "rollout_stats.npy"), stats.numpy())
        assert n == 1 or ((envs < sizes[0]).any() and (envs >= sizes[0]).any())   # the sample spans both sub-swarms


def test_reference_arm_line():
    d = run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-steps-per-step", "2", "--settle", "2"])
    assert d["impl"] == "reference" and d["value"] > 0 and d["gpu_launches"] == 0
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    from oracle import ref_pipeline
    want = "reference" if ref_pipeline.reference_root() is not None else "port"
    assert d["cpu_baseline"]["kind"] == want and d["cpu_baseline"]["value"] == d["value"]
