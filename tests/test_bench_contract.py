"""bench.py prints ONE JSON line with the contract's keys: a small configuration on the GPU (`-m gpu`) and the CPU
reference arm on a tiny sample (CPU suite)."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
COMMON = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
          "vs_baseline", "dtype", "data", "config", "e2e"}


def run_bench(*args, timeout=600):
  r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                     text=True, timeout=timeout, cwd=ROOT)
  assert r.returncode == 0, r.stderr[-2000:]
  lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
  assert len(lines) == 1, f"expected exactly one JSON line, got {len(lines)}"
  return json.loads(lines[0])


@pytest.mark.gpu
def test_bench_line_has_the_contract_keys(cuda_device, tmp_path):
  d = run_bench("--steps", "2", "--warmup", "3", "--views-per-rank", "2", "--num-gaussians", "200000",
                "--image-size", "640", "480", "--cpu-budget", "1", "--dump-outputs", str(tmp_path))
  assert d["steps"] == 2
  assert COMMON <= set(d) and {"roofline", "cpu_baseline", "clocks", "gpu_launches", "stage_ms_per_frame"} <= set(d)
  assert d["value"] > 0 and d["e2e"]["value"] > 0 and d["gpu_launches"] > 0
  assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] == 4
  r = d["roofline"]
  assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(r) and r["bound"] == "hbm"
  assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] == "port"
  assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
  assert "workload" in d["config"] and "model" not in d["config"]
  # the timed step is the CUDA-graph replay of the read-back free path, checked against the eager default path
  assert d["config"]["cuda_graph"] is True, d["config"].get("cuda_graph_error")
  assert d["config"]["graph_vs_eager_grad_rel_l2"] < 1e-5
  assert d["config"]["overlap_total_max"] <= d["config"]["overlap_capacity"]
  # the last timed step's loss and gradients, every row (200000 gaussians fit in 64 MB)
  files = {f.stem: f for f in tmp_path.glob("*.npy")}
  assert set(files) == {"loss", "grad_position", "grad_log_scaling", "grad_rotation", "grad_alpha_logit", "grad_feature"}
  assert sum(f.stat().st_size for f in files.values()) <= 64_000_000
  out = {k: np.load(f) for k, f in files.items()}
  assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in out.values())
  assert out["loss"].shape == (1,) and out["loss"][0] > 0
  assert out["grad_position"].shape == (200000, 3) and out["grad_feature"].shape[0] == 200000
  assert np.abs(out["grad_position"]).sum() > 0 and np.abs(out["grad_feature"]).sum() > 0


def test_dump_sample_is_fixed_and_bounded():
  """Gradients larger than the budget are cut down to the same seeded rows of every parameter, run after run."""
  sys.path.insert(0, str(ROOT))
  import torch
  from bench import sample_outputs
  n = 10000
  grads = {"position": torch.arange(3 * n, dtype=torch.float32).view(n, 3), "feature": torch.rand(n, 16, 3)}
  budget = (1 << 16) + 1000 * 4 * (3 + 48)
  a = sample_outputs(torch.tensor(2.5), grads, budget=budget)
  b = sample_outputs(torch.tensor(2.5), grads, budget=budget)
  assert set(a) == {"loss", "grad_position", "grad_feature"} and a["loss"].tolist() == [2.5]
  assert a["grad_position"].shape == (1000, 3) and a["grad_feature"].shape == (1000, 16, 3)
  assert sum(x.nbytes for x in a.values()) <= budget
  rows = a["grad_position"][:, 0].astype(np.int64) // 3
  assert np.all(np.diff(rows) > 0)
  assert np.array_equal(a["grad_feature"], grads["feature"].numpy()[rows])
  assert all(np.array_equal(a[k], b[k]) for k in a)
  full = sample_outputs(torch.tensor(2.5), grads)
  assert np.array_equal(full["grad_feature"], grads["feature"].numpy())


def test_reference_arm_line(monkeypatch):
  d = run_bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--num-gaussians", "80000",
                "--image-size", "320", "240")
  assert d["impl"] == "reference" and COMMON <= set(d) and d["steps"] == 1
  assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
  assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
