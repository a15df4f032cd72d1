"""Parity on the BENCHMARKED shapes (VERDICT round 1, "parity gaps"): the CUDA path through the C-ABI against the CPU
oracle at BASELINE.json's own sizes, the fused device loop (`dfb_denoise`) step for step against golden trajectories,
and the aggregation modes on the TSP (edge-valued) encoder.  Run with -m gpu on a B200.

Tolerance: 1e-4 relative (north_star) on network outputs, softmax probabilities and final heat maps."""
import numpy as np
import pytest
import torch

from conftest import golden, rel_linf
from difusco_b200 import _cabi, synthetic as syn
from oracle import difusco_oracle as orc
import gpu_util as G

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _prob_rel(out, ref):
  p = torch.softmax(torch.as_tensor(out), -1).numpy()
  pr = torch.softmax(torch.as_tensor(ref), -1).numpy()
  return float(np.abs(p / pr - 1).max())


# ------------------------------------------------------------------------------------------------
# configs[1], the headline workload: TSP-500 k=50, batch 16 in one block-diagonal call (E = 400 000)
# ------------------------------------------------------------------------------------------------
def test_config2_tsp500_batch16_forward_vs_oracle(weights2):
  pts, ei = syn.tsp_sparse_batch(500, 50, 16, seed=1234)
  xt = (syn.initial_noise(ei.shape[1], 0) > 0).astype(np.float32)
  torch.set_num_threads(max(1, min(32, torch.get_num_threads())))
  # the oracle evaluates V(h[col]) gather-then-GEMM exactly as gnn_encoder.py:99 does
  ref = orc.encoder_forward_sparse_tsp(orc.Weights(weights2), pts, xt, np.array([969.0]), ei).numpy()
  enc = G.encoder(weights2, 2, impl="tc")
  out = enc(G.cu(pts), torch.tensor([969.0]), G.cu(xt), G.cu(ei)).cpu().numpy()
  assert rel_linf(out, ref) < TOL and _prob_rel(out, ref) < TOL, (rel_linf(out, ref), _prob_rel(out, ref))


def test_config2_tsp500_teacher_forced_50_steps(weights2):
  """50-step categorical trajectory of one TSP-500 instance (the reference's own test_step shape, batch 1) through
  dfb_denoise_step: every step is fed the oracle's xt_in; network output, pre-sampling probability and the final heat
  map within 1e-4; sampled states may differ only where |p - u| is inside fp32 noise."""
  steps = 50
  pts, ei = syn.tsp_sparse_batch(500, 50, 1, seed=4321)
  n = ei.shape[1]
  xt0 = (syn.initial_noise(n, 3) > 0).astype(np.float32)
  us = [syn.uniforms(n, 500, i) for i in range(steps)]
  rec = []
  orc.denoise(orc.Weights(weights2), "tsp", "categorical", ei, xt0, points=pts, steps=steps, uniforms=us, record=rec)
  m = G.tsp_model(weights2, "tc", sparse_factor=50, inference_diffusion_steps=steps)
  dev = torch.device("cuda")
  m._prepare(G.cu(pts), G.cu(ei), dev)
  ctx = m.model.engine()
  st = torch.cuda.current_stream().cuda_stream
  worst_net = worst_p = 0.0
  for i, r in enumerate(rec):
    consts, last = m.posterior_consts(r["t1"], r["t2"])
    x = G.cu(r["xt_in"].numpy().astype(np.float32))
    u = G.cu(us[i])
    xo, p, net = torch.empty(n, device=dev), torch.empty(n, device=dev), torch.empty((n, 2), device=dev)
    ctx.denoise_step(_cabi.CATEGORICAL, x.data_ptr(), float(r["t1"]), consts, last, u.data_ptr(), 0, i, xo.data_ptr(),
                     p.data_ptr(), net.data_ptr(), st)
    torch.cuda.synchronize()
    ref_net = r["net_out"].numpy()
    worst_net = max(worst_net, rel_linf(net.cpu().numpy(), ref_net))
    assert worst_net < TOL, (i, worst_net)
    ref_p = r["p"].numpy()
    if i < steps - 1:
      worst_p = max(worst_p, float(np.abs(p.cpu().numpy().clip(0, 1) - ref_p.clip(0, 1)).max()))
      assert worst_p < TOL, (i, worst_p)
      flips = xo.cpu().numpy() != r["xt_out"].numpy()
      near = np.abs(ref_p - us[i]) < 10 * TOL
      assert not np.any(flips & ~near), (i, int(flips.sum()))
    else:
      hm, ref = xo.cpu().numpy(), r["xt_out"].numpy()
      assert np.abs(hm - ref).max() < TOL * max(ref.max(), 1e-3)
      big = ref > 1e-3
      assert np.abs(hm[big] / ref[big] - 1).max() < TOL


# ------------------------------------------------------------------------------------------------
# the fused device loop (what bench.py times) against reference trajectories, same injected uniforms
# ------------------------------------------------------------------------------------------------
def _fused_vs_golden(model, task, g, useed, diffusion):
  V, K, P, steps = [int(x) for x in g["meta"]]
  dev = torch.device("cuda")
  xt0 = g["xt0"].astype(np.float32).reshape(-1)
  n = xt0.size
  if task == "tsp":
    model._prepare(G.cu(np.tile(g["points"], (P, 1))), G.cu(g["edge_index"]), dev)
  else:
    model.model.set_graph(G.cu(g["edge_index"]), n, 1)
  ctx = model.model.engine()
  sched = orc.inference_schedule(model.args.inference_schedule, 1000, steps)
  t1s, cs, ls = [], [], []
  for t1, t2 in sched:
    c, last = model.posterior_consts(t1, t2)
    t1s.append(int(t1)); cs.append(c); ls.append(last)
  u = np.stack([syn.uniforms(n, useed, i) for i in range(steps)]).astype(np.float32)
  x = G.cu(xt0)
  mode = _cabi.CATEGORICAL if diffusion == "categorical" else _cabi.GAUSSIAN
  ctx.denoise(mode, x.data_ptr(), t1s, cs, ls, G.cu(u).data_ptr() if diffusion == "categorical" else None, 0,
              torch.cuda.current_stream().cuda_stream)
  torch.cuda.synchronize()
  got = x.cpu().numpy()
  ref = g["xt_out"][-1].reshape(-1)
  if diffusion == "categorical":
    big = ref > 1e-3
    ok = np.abs(got - ref).max() < TOL * max(ref.max(), 1e-3) and np.abs(got[big] / ref[big] - 1).max() < TOL
    if not ok:
      # a sample can only differ from the reference's where |p - u| is inside the 1e-4 contract on p; such a flip
      # legitimately changes everything downstream, so a mismatch is excused ONLY when the golden trajectory has such a tie
      near = [np.abs(g["p"][i].reshape(-1) - u[i]) < TOL for i in range(steps - 1)]
      if any(nm.any() for nm in near):
        pytest.skip("golden trajectory has a tie |p - u| < 1e-4 and the free-running loop took the other branch")
    assert ok
  else:
    assert rel_linf(got, ref) < TOL


def test_fused_loop_tsp_categorical_vs_golden_trajectory(weights2):
  g = golden("traj_tsp_cat")
  m = G.tsp_model(weights2, "tc", sparse_factor=6, parallel_sampling=2, inference_diffusion_steps=10)
  _fused_vs_golden(m, "tsp", g, 100, "categorical")


def test_fused_loop_mis_categorical_vs_golden_trajectory(weights2):
  g = golden("traj_mis_cat")
  m = G.mis_model(weights2, "tc", parallel_sampling=2, inference_diffusion_steps=8)
  _fused_vs_golden(m, "mis", g, 102, "categorical")


def test_fused_loop_tsp_gaussian_vs_golden_trajectory(weights1):
  g = golden("traj_tsp_gauss")
  m = G.tsp_model(weights1, "tc", diffusion_type="gaussian", sparse_factor=8, inference_diffusion_steps=6)
  _fused_vs_golden(m, "tsp", g, 101, "gaussian")


def test_fused_loop_tsp500_vs_oracle_free_running(weights2):
  """Free-running 10-step loop on one TSP-500 instance with injected uniforms, both sides: identical samples unless a
  near-tie occurs (then the step where the trajectories may part is reported and the test is skipped)."""
  steps = 10
  pts, ei = syn.tsp_sparse_batch(500, 50, 1, seed=99)
  n = ei.shape[1]
  xt0 = (syn.initial_noise(n, 5) > 0).astype(np.float32)
  us = [syn.uniforms(n, 900, i) for i in range(steps)]
  rec = []
  ref = orc.denoise(orc.Weights(weights2), "tsp", "categorical", ei, xt0, points=pts, steps=steps, uniforms=us,
                    record=rec).numpy()
  m = G.tsp_model(weights2, "tc", sparse_factor=50, inference_diffusion_steps=steps)
  m._prepare(G.cu(pts), G.cu(ei), torch.device("cuda"))
  sched = orc.inference_schedule("cosine", 1000, steps)
  t1s, cs, ls = [], [], []
  for t1, t2 in sched:
    c, last = m.posterior_consts(t1, t2)
    t1s.append(int(t1)); cs.append(c); ls.append(last)
  x = G.cu(xt0)
  m.model.engine().denoise(_cabi.CATEGORICAL, x.data_ptr(), t1s, cs, ls, G.cu(np.stack(us)).data_ptr(), 0,
                           torch.cuda.current_stream().cuda_stream)
  got = x.cpu().numpy()
  ok = np.abs(got - ref).max() < TOL * max(ref.max(), 1e-3)
  if not ok:
    for i, r in enumerate(rec[:-1]):
      if (np.abs(r["p"].numpy() - us[i]) < TOL).any():
        pytest.skip(f"tie |p - u| < 1e-4 at step {i}: the trajectories may legitimately part there")
  assert ok


# ------------------------------------------------------------------------------------------------
# configs[0]: TSP-50 dense, 1 instance, 50 steps (the reference's CPU-runnable case), teacher-forced vs the oracle
# ------------------------------------------------------------------------------------------------
def test_config1_tsp50_dense_50_steps_vs_oracle(weights2):
  V, steps = 50, 50
  pts = syn.tsp_points(V, 1234, 0).astype(np.float32)
  w = orc.Weights(weights2)
  sched = orc.inference_schedule("cosine", 1000, steps)
  _, Q_bar = orc.categorical_tables(1000, "linear")
  m = G.tsp_model(weights2, "tc", sparse_factor=-1, inference_diffusion_steps=steps)
  dev = torch.device("cuda")
  xt = (syn.initial_noise(V * V, 21) > 0).astype(np.float32).reshape(1, V, V)
  for i, (t1, t2) in enumerate(sched):
    ref_out = orc.encoder_forward_dense(w, pts[None], xt, np.array([float(t1)], np.float32))   # (1, 2, V, V)
    p0 = ref_out.permute(0, 2, 3, 1).softmax(-1)
    u = syn.uniforms(V * V, 333, i).reshape(1, V, V)
    p_ref, nxt = orc.categorical_posterior(Q_bar, t1, t2, p0, torch.from_numpy(xt), u)
    got_net = m.model(G.cu(pts[None]), torch.tensor([float(t1)]), G.cu(xt), None).cpu().numpy()
    assert rel_linf(got_net, ref_out.numpy()) < TOL, (i, rel_linf(got_net, ref_out.numpy()))
    if t2 == 0:   # the deterministic last step through the reference-signature method: the heat map
      hm = m.categorical_denoise_step(G.cu(pts[None]), G.cu(xt), np.array([t1]), dev, None, target_t=np.array([t2]))
      ref = nxt.numpy()
      assert hm.shape == (1, V, V)
      assert np.abs(hm.cpu().numpy() - ref).max() < TOL * max(ref.max(), 1e-3)
    xt = nxt.numpy().astype(np.float32)


# ------------------------------------------------------------------------------------------------
# configs[3]: MIS ER-[700,800], several graphs in one call (unsorted edge lists, node head, shared GroupNorm)
# ------------------------------------------------------------------------------------------------
def test_config4_mis_batch4_vs_oracle(weights2):
  ei, sizes = syn.mis_batch(700, 800, 0.15, 4, seed=41)
  V = sum(sizes)
  xt = (syn.initial_noise(V, 7) > 0).astype(np.float32)
  ref = orc.encoder_forward_mis(orc.Weights(weights2), xt, np.array([905.0]), ei).numpy()
  enc = G.encoder(weights2, 2, node_only=True, impl="tc")
  out = enc(G.cu(xt), torch.tensor([905.0]), edge_index=G.cu(ei)).cpu().numpy()
  assert rel_linf(out, ref) < TOL and _prob_rel(out, ref) < TOL, (rel_linf(out, ref), _prob_rel(out, ref))


# ------------------------------------------------------------------------------------------------
# --aggregation mean / max on the TSP (edge-valued) encoder
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("impl", ["fp32", "tc"])
@pytest.mark.parametrize("agg", ["mean", "max"])
def test_forward_tsp_aggregation_modes_vs_oracle(weights2, impl, agg):
  pts, ei = syn.tsp_sparse_batch(150, 20, 2, seed=5)
  xt = (syn.initial_noise(ei.shape[1], 15) > 0).astype(np.float32)
  ref = orc.encoder_forward_sparse_tsp(orc.Weights(weights2), pts, xt, np.array([412.0]), ei, aggregation=agg).numpy()
  enc = G.encoder(weights2, 2, impl=impl, aggregation=agg)
  out = enc(G.cu(pts), torch.tensor([412.0]), G.cu(xt), G.cu(ei)).cpu().numpy()
  assert rel_linf(out, ref) < G.TOL[impl], rel_linf(out, ref)


# ------------------------------------------------------------------------------------------------
# the single-CTA tcgen05 kernel (round 1) stays a validated fallback for every layer
# ------------------------------------------------------------------------------------------------
def test_forward_tsp_single_cta_kernel_vs_pair_kernel(weights2):
  pts, ei = syn.tsp_sparse_batch(300, 30, 3, seed=8)
  xt = (syn.initial_noise(ei.shape[1], 16) > 0).astype(np.float32)
  a = G.encoder(weights2, 2, impl="tc")(G.cu(pts), torch.tensor([555.0]), G.cu(xt), G.cu(ei)).cpu().numpy()
  b = G.encoder(weights2, 2, impl="tc1")(G.cu(pts), torch.tensor([555.0]), G.cu(xt), G.cu(ei)).cpu().numpy()
  assert rel_linf(a, b) < 2e-5


# ------------------------------------------------------------------------------------------------
# the captured CUDA graph of the loop == plain launches, across seeds / schedules / re-captures
# ------------------------------------------------------------------------------------------------
def test_fused_loop_graph_capture_matches_plain_launches(weights2):
  m = G.tsp_model(weights2, "tc", sparse_factor=10, inference_diffusion_steps=8)
  pts, ei = syn.tsp_sparse_batch(80, 10, 2, seed=12)
  xt0 = (syn.initial_noise(ei.shape[1], 4) > 0).astype(np.float32)
  ctx = m.model.engine()
  ctx.set_graph_capture(True)
  a1 = m.denoise_heatmap(G.cu(pts), G.cu(ei), G.cu(xt0), seed=5).cpu().numpy()    # captures
  b1 = m.denoise_heatmap(G.cu(pts), G.cu(ei), G.cu(xt0), seed=6).cpu().numpy()    # replays with another seed
  a2 = m.denoise_heatmap(G.cu(pts), G.cu(ei), G.cu(xt0), seed=5).cpu().numpy()    # replays
  ctx.set_graph_capture(False)
  a3 = m.denoise_heatmap(G.cu(pts), G.cu(ei), G.cu(xt0), seed=5).cpu().numpy()    # plain launches
  b3 = m.denoise_heatmap(G.cu(pts), G.cu(ei), G.cu(xt0), seed=6).cpu().numpy()
  ctx.set_graph_capture(True)
  assert np.array_equal(a1, a2) and np.array_equal(a1, a3) and np.array_equal(b1, b3) and not np.array_equal(a1, b1)
  # another graph shape -> re-capture; back to the first shape -> re-capture again, same answer
  pts2, ei2 = syn.tsp_sparse_batch(60, 10, 3, seed=13)
  x2 = (syn.initial_noise(ei2.shape[1], 5) > 0).astype(np.float32)
  c1 = m.denoise_heatmap(G.cu(pts2), G.cu(ei2), G.cu(x2), seed=9).cpu().numpy()
  a4 = m.denoise_heatmap(G.cu(pts), G.cu(ei), G.cu(xt0), seed=5).cpu().numpy()
  assert np.array_equal(a1, a4) and np.isfinite(c1).all()


def test_bench_dump_outputs_identical_across_runs(tmp_path):
  """bench.py --dump-outputs: the heat map of the last timed step; a second run with the same arguments writes the
  same bits, so two builds can be compared output for output."""
  import json
  import os
  import subprocess
  import sys
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  dumps = []
  for run in range(2):
    d = tmp_path / str(run)
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--config", "B1", "--steps", "2", "--warmup", "1",
                        "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    dumps.append(np.load(d / "heatmap.npy"))
  a, b = dumps
  assert a.dtype == np.float32 and a.shape == (500 * 50,) and np.array_equal(a, b)
  assert np.isfinite(a).all() and a.min() >= 0 and a.max() <= 1 + 1e-5    # the last step returns probabilities


# ------------------------------------------------------------------------------------------------
# N-GPU sharding on real GPUs (NCCL): per-instance heat maps bitwise equal to the single-GPU answer
# ------------------------------------------------------------------------------------------------
def test_multi_gpu_sharding_bitwise_equal_to_single_gpu():
  import os
  import socket
  import subprocess
  import sys
  n = torch.cuda.device_count()
  if n < 2:
    pytest.skip("needs >= 2 GPUs (run under `gpurun --gpus 2`; log committed as profiles/r02_multi_gpu_check.txt)")
  s = socket.socket()
  s.bind(("127.0.0.1", 0))
  port = s.getsockname()[1]
  s.close()
  root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
  r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={min(n, 2)}",
                      "--master-addr", "127.0.0.1", "--master-port", str(port),
                      os.path.join(root, "scripts", "multi_gpu_check.py")], capture_output=True, text=True, timeout=900)
  assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
  assert '"bitwise_equal_to_single_gpu": true' in r.stdout
