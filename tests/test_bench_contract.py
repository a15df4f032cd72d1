"""bench.py's host-side contract, checked without a GPU: the algorithmic-byte formulas (SURVEY 8d), the config table
(BASELINE.json configs), the committed ncu traffic number, and the failure mode of the GPU arm on a box without a GPU."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_algorithmic_bytes_match_survey_8d():
  E, V = 400000, 8000
  assert bench.algorithmic_bytes_per_step(dict(node_only=False, E=E, V=V)) == 24576 * E          # 2 L E H 4
  mis = bench.algorithmic_bytes_per_step(dict(node_only=True, E=E, V=V))
  assert mis == (2 * 12 - 2) * E * 256 * 4 + 2 * 12 * V * 256 * 4
  # per TSP-500 graph (E = 25 000, 50 steps): 30.72 GB -> the 213.8 graphs/s ceiling DESIGN.md quotes at 6567.7 GB/s
  per_graph = 24576 * 25000 * 50
  assert abs(per_graph / 1e9 - 30.72) < 1e-9
  assert abs(6567.7e9 / per_graph - 213.8) < 0.05


def test_config_table_covers_baseline_configs():
  base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
  assert sorted(bench.CONFIGS) == ["B1", "C1", "C2", "C3", "C4", "C5"]
  assert len(base["configs"]) == 5
  c2 = bench.CONFIGS["C2"]
  assert (c2["nodes"], c2["knn"], c2["batch"], c2["diffusion"]) == (500, 50, 16, "categorical")
  assert bench.METRIC.startswith("TSP-500 graphs/sec") and bench.UNIT == "graphs/s"
  wl = bench.workload_config(8)
  assert wl["global_batch"] == 16 * 8 and "model" not in wl


def test_committed_ncu_traffic_is_close_to_the_algorithmic_bytes():
  t = bench.ncu_traffic()
  assert t is not None
  algo = 24576 * 400000
  assert 1.0 <= t / algo < 1.25          # DRAM bytes of a whole step: no wasted re-reads


def test_small_workloads_build_on_cpu():
  for name in ("C1", "B1"):
    wl = bench.build_workload(bench.CONFIGS[name], rank=0)
    assert wl["edge_index"].shape == (2, wl["E"]) and wl["xt0"].shape[0] == wl["n_state"]
    assert np.all(np.diff(wl["edge_index"][0]) >= 0) or name == "C1"      # sparse TSP lists arrive row-sorted


def test_dump_outputs_float32_and_seeded_sample_within_budget(tmp_path, monkeypatch):
  hm = np.arange(1000, dtype=np.float64) / 1000
  bench.dump_outputs(str(tmp_path / "full"), {"heatmap": hm})
  got = np.load(tmp_path / "full" / "heatmap.npy")
  assert got.dtype == np.float32 and np.array_equal(got, hm.astype(np.float32))
  monkeypatch.setattr(bench, "DUMP_BYTES", 1000)             # 4000 bytes of output: a quarter survives
  for run in ("a", "b"):
    bench.dump_outputs(str(tmp_path / run), {"heatmap": hm})
  a, b = np.load(tmp_path / "a" / "heatmap.npy"), np.load(tmp_path / "b" / "heatmap.npy")
  assert a.size == 250 and np.array_equal(a, b) and np.all(np.diff(a) > 0)


def test_steps_below_one_is_rejected():
  r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], stdout=subprocess.PIPE,
                     stderr=subprocess.STDOUT, text=True, timeout=600)
  assert r.returncode == 2 and "--steps" in r.stdout


def test_gpu_arm_fails_loudly_without_a_gpu():
  import torch
  if torch.cuda.is_available():
    return
  r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--no-cpu-baseline"],
                     stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
  assert r.returncode != 0          # no CPU fallback: the product path needs the CUDA library and a device
  assert "graphs/s" not in r.stdout.splitlines()[-1] if r.stdout.strip() else True
