"""Benchmark of the denoise hot path (BASELINE.json metric: TSP-500 graphs/sec, 50-step categorical).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

A "step" = one pass of the hot path over one batch: the full 50-step categorical denoise of
16 TSP-500 (k=50) instances batched block-diagonally in one call (BASELINE config[1]), per GPU.
Weak scaling: every rank owns its own batch; no collective inside the loop; for N > 1 the final
heatmaps are all-gathered over NCCL inside the timed region (north_star).
Prints ONE JSON line on rank 0.  --dump-outputs DIR writes the heat map(s) of the last timed step as DIR/heatmap.npy
(float32; inputs and sampling seeds are fixed, so runs with the same arguments are comparable output for output).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_NODES, KNN, BATCH, DENOISE_STEPS, T = 500, 50, 16, 50, 1000
H, L = 256, 12
METRIC = "TSP-500 graphs/sec, 50-step categorical denoise"
UNIT = "graphs/s"


def model_args():
  from types import SimpleNamespace as NS
  return NS(diffusion_type="categorical", diffusion_schedule="linear", diffusion_steps=T, sparse_factor=KNN,
            n_layers=L, hidden_dim=H, aggregation="sum", parallel_sampling=1, sequential_sampling=1,
            inference_schedule="cosine", inference_diffusion_steps=DENOISE_STEPS, inference_trick="ddim")


def workload_config(n_gpus):
  return {"workload": f"TSP-{N_NODES} sparse k={KNN}, categorical diffusion, {DENOISE_STEPS} denoise steps, "
                      f"batch {BATCH} instances per GPU in one block-diagonal call (BASELINE configs[1])",
          "nodes_per_graph": N_NODES, "knn": KNN, "batch_per_gpu": BATCH, "denoise_steps": DENOISE_STEPS,
          "global_batch": BATCH * n_gpus, "parallelism": f"dp{n_gpus} (independent batches, no in-loop collective)",
          "weights": "seeded random init of the reference architecture (12 layers, hidden 256), per_layer_out de-zeroed",
          "l2_policy": "working set (edge stream 410 MB/GPU) exceeds the 126 MB L2; no explicit flush needed"}


# ------------------------------------------------------------------------------------------------
class ClockSampler(object):
  """nvidia-smi clocks + throttle reasons sampled during the timed region."""
  Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
       "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
       "clocks_event_reasons.sw_power_cap")

  def __init__(self, gpu_index):
    self.idx, self.rows, self.proc = gpu_index, [], None

  def start(self):
    try:
      self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                    "-i", str(self.idx), "-lms", "200"], stdout=subprocess.PIPE,
                                   stderr=subprocess.DEVNULL, text=True)
      self.th = threading.Thread(target=self._read, daemon=True)
      self.th.start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append([x.strip() for x in line.split(",")])

  def stop(self):
    if not self.proc:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    self.proc.terminate()
    try:
      self.proc.wait(timeout=2)
    except Exception:
      self.proc.kill()
    sm, mx, reasons = [], [], set()
    for r in self.rows:
      try:
        sm.append(float(r[1])); mx.append(float(r[2]))
      except Exception:
        continue
      for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
        if v.lower().startswith("active"):
          reasons.add(name)
    return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
            "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
  p = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(p):
    d = json.load(open(p))
    return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, sustained copy)"
  return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic():
  """dram__bytes_read.sum + dram__bytes_write.sum of ALL launches of one denoise step of the headline workload, from the
  committed ncu pass (profiles/r02_step_traffic.json; same scope as roofline.achieved: the whole step)."""
  p = os.path.join(ROOT, "profiles", "r02_step_traffic.json")
  if os.path.exists(p):
    try:
      return json.load(open(p)).get("dram_bytes_per_step")
    except Exception:
      return None
  return None


# ------------------------------------------------------------------------------------------------
_CPU_SETUP = {}


def _cpu_setup():
  """Build the CPU-oracle workload once and pick the thread count that runs one forward fastest
  (all visible cores is often NOT fastest for E = 25 000 rows: oversubscription / cgroup quotas)."""
  if _CPU_SETUP:
    return _CPU_SETUP
  import torch
  from difusco_b200 import synthetic as syn
  from oracle import difusco_oracle as orc
  w = orc.Weights(syn.make_encoder_weights(0, out_channels=2))
  pts, ei = syn.tsp_sparse_batch(N_NODES, KNN, 1, seed=1234)
  xt0 = (syn.initial_noise(ei.shape[1], 0) > 0).astype(np.float32)
  ei_t = torch.from_numpy(ei)
  try:
    avail = len(os.sched_getaffinity(0))
  except Exception:
    avail = os.cpu_count() or 1
  best = None
  with torch.no_grad():
    for th in sorted({t for t in (4, 8, 16, 32, 64, avail) if t <= avail}):
      torch.set_num_threads(th)
      orc.encoder_forward_sparse_tsp(w, pts, torch.from_numpy(xt0), torch.tensor([1000.0]), ei_t, gather_then_gemm=False)
      t0 = time.perf_counter()
      orc.encoder_forward_sparse_tsp(w, pts, torch.from_numpy(xt0), torch.tensor([1000.0]), ei_t, gather_then_gemm=False)
      dt = time.perf_counter() - t0
      if best is None or dt < best[1]:
        best = (th, dt)
      if dt > 3 * best[1]:
        break
  torch.set_num_threads(best[0])
  _CPU_SETUP.update(w=w, pts=pts, ei_t=ei_t, xt0=xt0, threads=best[0], fwd_s=best[1], avail=avail)
  return _CPU_SETUP


def cpu_oracle_graphs_per_s(budget_s=20.0):
  """The oracle port (oracle/difusco_oracle.py, torch CPU fp32) on ONE TSP-500 k=50 instance for as many of
  the 50 denoise steps as fit in ~budget_s (2..50), extrapolated to 50 steps.
  Returns (graphs/s, seconds spent, threads, steps run)."""
  import torch
  from oracle import difusco_oracle as orc
  c = _cpu_setup()
  n = int(max(2, min(DENOISE_STEPS, budget_s / max(c["fwd_s"], 1e-3))))
  sched = orc.inference_schedule("cosine", T, DENOISE_STEPS)
  _, Qbar = orc.categorical_tables(T, "linear")
  xt = torch.from_numpy(c["xt0"])
  torch.set_num_threads(c["threads"])
  with torch.no_grad():
    t0 = time.perf_counter()
    for (t1, t2) in sched[:n]:
      out = orc.encoder_forward_sparse_tsp(c["w"], c["pts"], xt, torch.tensor([float(t1)]), c["ei_t"],
                                           gather_then_gemm=False)
      _, xt = orc.categorical_posterior(Qbar, t1, t2, out.softmax(-1), xt)
    dt = time.perf_counter() - t0
  per_graph = dt * DENOISE_STEPS / n
  return 1.0 / per_graph, dt, c["threads"], n


def reference_graphs_per_s(budget_s=20.0):
  """The UNMODIFIED reference (oracle/_ref/difusco, copied by oracle/make_ref.py) on the host cores: its own TSPModel.
  categorical_denoise_step (pl_tsp_model.py:122-138 -> GNNEncoder.forward + categorical_posterior) on ONE block-diagonal
  batch of BATCH TSP-500 k=50 instances - the same call shape as the GPU arm - for as many of the 50 denoise steps as
  fit in ~budget_s (at least 1), extrapolated to 50.  Returns (graphs/s, seconds, threads, steps run) or None."""
  sys.path.insert(0, os.path.join(ROOT, "oracle"))
  import make_ref
  if not make_ref.available():
    return None
  import torch
  sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
  import ref_shims
  ref_shims.install(os.path.join(ROOT, "oracle", "_ref", "difusco"))
  from pl_tsp_model import TSPModel as RefTSPModel   # the reference's own class, stock code path
  from utils.diffusion_schedulers import InferenceSchedule as RefSchedule
  from difusco_b200 import synthetic as syn
  a = model_args()
  for k, v in dict(task="tsp", storage_path="", training_split="", validation_split="", test_split="", batch_size=1,
                   num_workers=0, learning_rate=2e-4, weight_decay=0.0, lr_scheduler="constant", num_epochs=1,
                   use_activation_checkpoint=False, save_numpy_heatmap=False, two_opt_iterations=0, fp16=False).items():
    setattr(a, k, v)
  model = RefTSPModel.__new__(RefTSPModel)
  from pl_meta_model import COMetaModel
  COMetaModel.__init__(model, param_args=a, node_feature_only=False)   # TSPModel.__init__ additionally opens dataset files
  w = syn.make_encoder_weights(0, out_channels=2)
  model.model.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
  model.eval()
  pts, ei = syn.tsp_sparse_batch(N_NODES, KNN, BATCH, seed=1234)
  xt = torch.from_numpy((syn.initial_noise(ei.shape[1], 0) > 0).astype(np.int64))
  points, edge_index = torch.from_numpy(pts), torch.from_numpy(ei)
  try:
    avail = len(os.sched_getaffinity(0))
  except Exception:
    avail = os.cpu_count() or 1
  # "all the host threads it can use": torch's intra-op pool does not scale to every core for E = 400 000 rows x 256
  # (128 threads were 5x SLOWER than 32 on the round-2 box), so the arm uses the thread count that runs ONE forward of a
  # single TSP-500 instance fastest - the most favourable setting for the reference
  p1, e1 = syn.tsp_sparse_batch(N_NODES, KNN, 1, seed=1)
  x1 = torch.zeros(e1.shape[1], dtype=torch.int64)
  best = None
  with torch.no_grad():
    for th in sorted({t for t in (8, 16, 32, 64, avail) if t <= avail}):
      torch.set_num_threads(th)
      t0 = time.perf_counter()
      model.categorical_denoise_step(torch.from_numpy(p1), x1, np.array([500]).astype(int), torch.device("cpu"),
                                     torch.from_numpy(e1), target_t=np.array([400]).astype(int))
      dt = time.perf_counter() - t0
      if best is None or dt < best[1]:
        best = (th, dt)
  avail = best[0]
  torch.set_num_threads(avail)
  dev = torch.device("cpu")
  sched = RefSchedule(inference_schedule="cosine", T=T, inference_T=DENOISE_STEPS)
  with torch.no_grad():   # untimed warm-up on a tiny instance: thread pool, allocator, lazy imports
    wp, we = syn.tsp_sparse_batch(50, 10, 1, seed=1)
    model.categorical_denoise_step(torch.from_numpy(wp), torch.zeros(we.shape[1], dtype=torch.int64),
                                   np.array([500]).astype(int), dev, torch.from_numpy(we), target_t=np.array([400]).astype(int))
  n, t0 = 0, time.perf_counter()
  with torch.no_grad():
    while n < DENOISE_STEPS:
      t1, t2 = sched(n)
      xt = model.categorical_denoise_step(points, xt, np.array([t1]).astype(int), dev, edge_index,
                                          target_t=np.array([t2]).astype(int))
      n += 1
      if time.perf_counter() - t0 > budget_s:
        break
  dt = time.perf_counter() - t0
  per_batch = dt * DENOISE_STEPS / n
  return BATCH / per_batch, dt, avail, n


def run_reference(args, rank, world):
  """--impl reference: the reference's own CPU implementation of the path on the box's host cores - the unmodified
  reference files (oracle/_ref, kind "reference") through dependency shims; the oracle port only if they are missing."""
  if rank != 0:
    return
  vals, secs, steps_run, threads, kind = [], 0.0, 0, 1, "reference"
  for _ in range(max(args.steps, 1)):
    r = reference_graphs_per_s(budget_s=20.0)
    if r is None:
      kind = "port"
      r = cpu_oracle_graphs_per_s(budget_s=15.0)
    v, dt, threads, steps_run = r
    vals.append(v); secs += dt
  value = float(np.mean(vals))
  if kind == "reference":
    sample = (f"unmodified reference (oracle/_ref: TSPModel.categorical_denoise_step = GNNEncoder.forward + "
              f"categorical_posterior, torch CPU fp32, stock gather-then-GEMM) on one block-diagonal batch of {BATCH} "
              f"TSP-500 k=50 instances, {steps_run} of {DENOISE_STEPS} denoise steps per timed step (~20 s), extrapolated "
              f"x{DENOISE_STEPS / steps_run:.1f}; torch.set_num_threads({threads}) = the fastest of 8/16/32/64/all visible cores on one forward")
  else:
    sample = (f"oracle port: 1 TSP-500 k=50 instance, {steps_run} of {DENOISE_STEPS} denoise steps per timed step, "
              f"extrapolated x{DENOISE_STEPS / steps_run:.1f}; thread count auto-picked ({threads})")
  line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": 1000.0 / value * BATCH, "higher_is_better": True,
          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
          "config": workload_config(args.gpus),
          "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                           "ref_kind": "_ref" if kind == "reference" else "port", "sample": sample,
                           "extrapolated": steps_run < DENOISE_STEPS, "measured_seconds": secs},
          "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
          "gpu_launches": 0}
  print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# BASELINE.json configs.  configs[1] (C2) is the headline workload the default run times; --config C1|C3|C4|C5 time the
# other ones through the same code path and print the same JSON schema (profiles/r02_other_configs.jsonl).
CONFIGS = {
    "C1": dict(task="tsp", nodes=50, knn=-1, batch=1, diffusion="categorical",
               label="TSP-50 dense graph, categorical diffusion, 1 instance, 50 denoise steps (BASELINE configs[0])"),
    "C2": dict(task="tsp", nodes=N_NODES, knn=KNN, batch=BATCH, diffusion="categorical", label=None),
    "C3": dict(task="tsp", nodes=1000, knn=100, batch=8, diffusion="gaussian",
               label="TSP-1000 sparse k=100, Gaussian diffusion, 50 denoise steps, batch 8 (BASELINE configs[2])"),
    "C4": dict(task="mis", nodes=(700, 800), knn=0, batch=32, diffusion="categorical",
               label="MIS ER-[700,800] p=0.15, categorical, 50 denoise steps, batch 32 (BASELINE configs[3])"),
    "C5": dict(task="tsp", nodes=10000, knn=50, batch=4, diffusion="categorical",
               label="TSP-10000 sparse k=50, categorical, 50 denoise steps, 4x parallel sampling per GPU (BASELINE configs[4])"),
    "B1": dict(task="tsp", nodes=N_NODES, knn=KNN, batch=1, diffusion="categorical",
               label="TSP-500 sparse k=50, categorical, 50 denoise steps, batch 1 (the reference test loader's shape)"),
}


def build_workload(cfg, rank):
  """-> dict(points, edge_index, xt0, V, E, n_state, graphs, node_only, gn_segments, args)."""
  from types import SimpleNamespace as NS
  from difusco_b200 import synthetic as syn
  a = model_args()
  a.diffusion_type = cfg["diffusion"]
  seed = 1234 + 1000 * rank
  if cfg["task"] == "mis":
    ei, sizes = syn.mis_batch(cfg["nodes"][0], cfg["nodes"][1], 0.15, cfg["batch"], seed=seed)
    V, E = int(sum(sizes)), ei.shape[1]
    xt0 = (syn.initial_noise(V, rank) > 0).astype(np.float32)
    a.sparse_factor = -1
    return dict(points=None, edge_index=ei, xt0=xt0, V=V, E=E, n_state=V, graphs=cfg["batch"], node_only=True,
                gn_segments=1, args=a)
  if cfg["knn"] <= 0:      # dense: the complete graph incl. self pairs, per-sample GroupNorm
    n, B = cfg["nodes"], cfg["batch"]
    pts = np.concatenate([syn.tsp_points(n, seed, i) for i in range(B)]).astype(np.float32)
    ei = np.concatenate([syn.complete_edge_index(n) + i * n for i in range(B)], axis=1)
    xt0 = (syn.initial_noise(ei.shape[1], rank) > 0).astype(np.float32)
    a.sparse_factor = -1
    return dict(points=pts, edge_index=ei, xt0=xt0, V=B * n, E=ei.shape[1], n_state=ei.shape[1], graphs=B,
                node_only=False, gn_segments=B, args=a)
  pts, ei = syn.tsp_sparse_batch(cfg["nodes"], cfg["knn"], cfg["batch"], seed=seed)
  a.sparse_factor = cfg["knn"]
  noise = syn.initial_noise(ei.shape[1], rank)
  xt0 = (noise > 0).astype(np.float32) if cfg["diffusion"] == "categorical" else noise.astype(np.float32)
  return dict(points=pts, edge_index=ei, xt0=xt0, V=pts.shape[0], E=ei.shape[1], n_state=ei.shape[1],
              graphs=cfg["batch"], node_only=False, gn_segments=1, args=a)


DUMP_BYTES = 60 * 10**6   # --dump-outputs budget: under 64 MB with the .npy headers


def dump_outputs(out_dir, arrays):
  """Writes each array as <out_dir>/<name>.npy in float32.  When together they exceed DUMP_BYTES, each one is cut to a
  fixed, seeded sample of its flattened elements: the same elements for the same arguments, so runs stay comparable."""
  os.makedirs(out_dir, exist_ok=True)
  total = sum(np.size(a) * 4 for a in arrays.values())
  for name, a in arrays.items():
    a = np.asarray(a, dtype=np.float32)
    if total > DUMP_BYTES:
      keep = a.size * DUMP_BYTES // total
      a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
    np.save(os.path.join(out_dir, name + ".npy"), a)


def algorithmic_bytes_per_step(wl):
  """SURVEY 8(d): sparse / dense TSP 2 L E H 4 = 24 576 E per denoise step (L-1 inter-layer reads + the head's read,
  L writes; layer 0 reads xt instead of a materialised e0); MIS (2L-2) E H 4 (no e0 read, the last layer's e is never
  consumed) + 2 L V H 4 (the node stream)."""
  if wl["node_only"]:
    return (2 * L - 2) * wl["E"] * H * 4 + 2 * L * wl["V"] * H * 4
  return 2 * L * wl["E"] * H * 4


def run_ours(args, rank, world, local_rank):
  import torch
  import torch.distributed as dist
  from difusco_b200 import _cabi
  from difusco_b200.pl_mis_model import MISModel
  from difusco_b200.pl_tsp_model import TSPModel
  from difusco_b200 import synthetic as syn
  from difusco_b200.utils.diffusion_schedulers import InferenceSchedule

  torch.cuda.set_device(local_rank)
  dev = torch.device("cuda", local_rank)
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
  cfg = CONFIGS[args.config]
  wl = build_workload(cfg, rank)
  categorical = cfg["diffusion"] == "categorical"
  model = (MISModel if wl["node_only"] else TSPModel)(wl["args"])
  w = syn.make_encoder_weights(0, out_channels=2 if categorical else 1)
  model.model.load_state_dict({k: torch.from_numpy(v) for k, v in w.items()})
  model.cuda(local_rank).eval()
  ctx = model.model.engine()
  impl = os.environ.get("DFB_EDGE_IMPL", "tc")
  if impl != "tc":
    ctx.set_edge_impl({"fp32": _cabi.EDGE_IMPL_FP32, "tc1": _cabi.EDGE_IMPL_TC1}[impl])
  stream = torch.cuda.current_stream().cuda_stream
  V, E, n_state, graphs = wl["V"], wl["E"], wl["n_state"], wl["graphs"]
  d_ei = torch.from_numpy(wl["edge_index"]).to(dev)
  d_xt0 = torch.from_numpy(wl["xt0"]).to(dev)
  d_pts = torch.from_numpy(wl["points"]).to(dev) if wl["points"] is not None else None
  mode = _cabi.CATEGORICAL if categorical else _cabi.GAUSSIAN

  sched = InferenceSchedule("cosine", T, DENOISE_STEPS)
  t1s, cs, ls = [], [], []
  for i in range(DENOISE_STEPS):
    t1, t2 = sched(i)
    c, last = model.posterior_consts(int(t1), int(t2))
    t1s.append(int(t1)); cs.append(c); ls.append(last)

  model.model.set_graph(d_ei, V, wl["gn_segments"])
  if d_pts is not None:
    model.model.set_points(d_pts)
  gathered = [torch.empty(n_state, device=dev) for _ in range(world)] if world > 1 else None
  x = torch.empty(n_state, device=dev)

  def one_step(seed):
    x.copy_(d_xt0)
    ctx.denoise(mode, x.data_ptr(), t1s, cs, ls, None, seed, stream)
    if world > 1:
      dist.all_gather(gathered, x)

  def fence():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  for i in range(args.warmup):
    one_step(i)
  fence()
  sampler = ClockSampler(local_rank)
  if rank == 0:
    sampler.start()
  launches0 = ctx.launch_count()
  ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ev0.record()
  for i in range(args.steps):
    one_step(100 + i)
  ev1.record()
  fence()
  ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev)
  launches = ctx.launch_count() - launches0
  clocks = sampler.stop() if rank == 0 else None
  if world > 1:
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
  total_ms = float(ms.item())
  hm = x.cpu().numpy()
  assert np.isfinite(hm).all()
  if categorical:
    assert hm.min() >= 0.0 and hm.max() <= 1.0 + 1e-5
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, {"heatmap": np.stack([g.cpu().numpy() for g in gathered]) if world > 1 else hm})

  # ---- the dominant kernel on its own: ONE more batch with per-launch CUDA events on the launching stream (plain
  #      launches: events cannot be recorded inside the captured graph the timed region replays); not part of `value`
  ctx.set_graph_capture(False)
  ctx.profile_begin()
  one_step(999)
  torch.cuda.synchronize()
  edge_ms, edge_n = ctx.profile_end()
  pev0, pev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  pev0.record()
  one_step(998)
  pev1.record()
  torch.cuda.synchronize()
  plain_ms = pev0.elapsed_time(pev1)
  ctx.set_graph_capture(True)

  # ---- e2e: same metric through the host-buffer C-ABI call (H2D of inputs + D2H of the heatmap per step)
  p_ei = torch.from_numpy(wl["edge_index"]).pin_memory()
  p_xt0 = torch.from_numpy(wl["xt0"]).pin_memory()
  p_pts = torch.from_numpy(wl["points"]).pin_memory() if wl["points"] is not None else None
  p_hm = torch.empty(n_state, dtype=torch.float32).pin_memory()

  def e2e_step(seed):
    ctx.denoise_host(mode, p_pts.data_ptr() if p_pts is not None else None, p_ei.data_ptr(), V, E, wl["gn_segments"],
                     p_xt0.data_ptr(), t1s, cs, ls, seed, p_hm.data_ptr(), stream)
  e2e_step(0)
  fence()
  t0 = time.perf_counter()
  for i in range(args.steps):
    e2e_step(200 + i)
  fence()
  e2e_s = torch.tensor([time.perf_counter() - t0], device=dev)
  if world > 1:
    dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
  e2e_value = graphs * world * args.steps / float(e2e_s.item())
  h2d = wl["edge_index"].nbytes + wl["xt0"].nbytes + (wl["points"].nbytes if wl["points"] is not None else 0)
  d2h = p_hm.numel() * 4

  if rank == 0:
    value = graphs * world * args.steps / (total_ms / 1e3)
    peak, peak_src = measured_peaks()
    # whole-step accounting (SURVEY 8d): every launch of a denoise step is inside the number, nothing is booked elsewhere
    step_bytes = algorithmic_bytes_per_step(wl)
    achieved = step_bytes * DENOISE_STEPS * args.steps / (total_ms / 1e3) / 1e9
    n_layer_launches = max(int(edge_n), 1)
    per_launch_bytes = ((2 * L - 1) * E * H * 4 / L) if not wl["node_only"] else (2 * L - 2) * E * H * 4 / L
    k_ms = edge_ms / n_layer_launches
    k_achieved = per_launch_bytes / (k_ms / 1e3) / 1e9 if k_ms > 0 else 0.0
    wlc = workload_config(world)
    if cfg["label"]:
      wlc["workload"] = cfg["label"] + ", per GPU"
      wlc.update(nodes_per_graph=cfg["nodes"], knn=cfg["knn"], batch_per_gpu=cfg["batch"], global_batch=cfg["batch"] * world)
      wlc["l2_policy"] = (f"edge stream {E * H * 4 / 1e6:.0f} MB per GPU" +
                          (" exceeds the 126 MB L2" if E * H * 4 > 126e6 else " fits the 126 MB L2 (no flush: the loop streams it 24x per step)"))
    line = {"metric": METRIC if args.config == "C2" else f"{args.config} graphs/sec, 50-step denoise ({cfg['label']})",
            "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32 (3-term bf16 split on tcgen05, fp32 accumulate)",
            "data": "synthetic", "config": wlc,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ncu_traffic(), "peak_source": peak_src,
                         "scope": "whole denoise step: every launch of the timed loop (CUDA-graph replay), timed with CUDA "
                                  "events around the loop; algorithmic bytes = SURVEY 8(d) per step",
                         "algorithmic_bytes_per_step": step_bytes, "denoise_steps_timed": DENOISE_STEPS * args.steps,
                         "kernel": {"name": "k_edge_layer_pair (CTA-pair fused edge layer, all 12 layers; layer 0 in table-lookup "
                                            "mode without the input read; the MIS last layer: k_edge_layer_tc16w)"
                                    if impl == "tc" else impl,
                                    "algorithmic_bytes_per_launch": per_launch_bytes, "launches_timed": int(edge_n),
                                    "ms_per_launch": k_ms, "achieved": k_achieved, "frac": k_achieved / peak,
                                    "share_of_step": edge_ms / plain_ms if plain_ms > 0 else None,
                                    "how": "per-launch CUDA events on the launching stream over one extra batch with plain "
                                           "launches (events cannot be recorded inside the replayed graph)"}},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches), "launches_per_denoise_step": launches / (DENOISE_STEPS * args.steps),
            "graph_replay_vs_plain_launches_ms": [total_ms / args.steps, plain_ms], "clocks": clocks}
    if world == 1 and not args.no_cpu_baseline and args.config == "C2":
      r = reference_graphs_per_s(budget_s=20.0)
      if r is not None:
        v, dt, threads, n_run = r
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "reference", "ref_kind": "_ref",
                                "sample": f"unmodified reference (oracle/_ref, TSPModel.categorical_denoise_step, torch CPU fp32) "
                                          f"on one block-diagonal batch of {BATCH} TSP-500 k=50 instances, {n_run} of "
                                          f"{DENOISE_STEPS} denoise steps ({dt:.1f} s), extrapolated x{DENOISE_STEPS / n_run:.1f}; "
                                          f"{threads} host threads"}
      else:
        v, dt, threads, n_run = cpu_oracle_graphs_per_s(budget_s=20.0)
        line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"oracle port (torch CPU fp32) on 1 TSP-500 k=50 instance, {n_run} of "
                                          f"{DENOISE_STEPS} denoise steps ({dt:.1f} s), extrapolated x{DENOISE_STEPS / n_run:.1f}; "
                                          f"thread count auto-picked ({threads} of {_CPU_SETUP.get('avail')} visible cores "
                                          f"was fastest)"}
    print(json.dumps(line))
  if world > 1:
    dist.destroy_process_group()


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=3)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--config", default="C2", choices=sorted(CONFIGS), help="BASELINE.json config (default C2 = configs[1], the headline)")
  ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
  ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                  help="write the heat map(s) of the last timed step as DIR/heatmap.npy")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and args.impl != "ours":
    ap.error("--dump-outputs needs --impl ours")
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  local_rank = int(os.environ.get("LOCAL_RANK", "0"))
  if args.impl == "reference":
    run_reference(args, rank, world)
    return
  if world != args.gpus and world == 1 and args.gpus > 1:
    raise SystemExit("launch with torchrun for --gpus > 1 (one process per GPU)")
  run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
  main()
