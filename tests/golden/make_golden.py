"""Generate tests/golden/*.npz by running the UNMODIFIED reference (/root/reference/difusco).

Run in the build container only (the reference tree does not exist on the GPU box):
    python tests/golden/make_golden.py
The reference is imported through tests/golden/ref_shims.py (stand-ins for its missing
third-party dependencies, nothing of the reference itself).  Inputs and weights come from
difusco_b200/synthetic.py, so the fixtures only need to carry the reference's OUTPUTS (plus the
small inputs, for self-containment); tests rebuild the weights from the seed.

Sampling: the reference draws torch.bernoulli(p).  To make the trajectory a pure function of the
inputs, torch.bernoulli is replaced *in this script* by (u < p) with u from synthetic.uniforms -
the same semantic torch's CPU kernel has - and p is recorded on the way through.  The reference's
test_step itself is not callable here past the heatmap (it needs the Cython merge extension,
which is decode and out of the path), so the loop at pl_tsp_model.py:185-222 /
pl_mis_model.py:156-192 is driven from here through the reference's OWN methods
(duplicate_edge_index, categorical_denoise_step, gaussian_denoise_step, InferenceSchedule).
"""
import argparse
import os
import sys
import tempfile

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import ref_shims  # noqa: E402

ref_shims.install()

from models.gnn_encoder import GNNEncoder  # noqa: E402  (reference)
from utils.diffusion_schedulers import (CategoricalDiffusion, GaussianDiffusion,  # noqa: E402
                                        InferenceSchedule)
import pl_tsp_model  # noqa: E402
import pl_mis_model  # noqa: E402

from difusco_b200 import synthetic as syn  # noqa: E402

torch.set_grad_enabled(False)


def sd_torch(w):
  return {k: torch.from_numpy(v.copy()) for k, v in w.items()}


def save(name, **arrs):
  path = os.path.join(HERE, name + ".npz")
  np.savez_compressed(path, **arrs)
  print(f"wrote {path}  ({os.path.getsize(path) / 1024:.1f} KiB)")


# ------------------------------------------------------------------------------------------
def gen_schedules():
  out = {}
  for sch in ("linear", "cosine"):
    c = CategoricalDiffusion(1000, sch)
    g = GaussianDiffusion(1000, sch)
    out[f"cat_{sch}_Qs"] = c.Qs
    out[f"cat_{sch}_Qbar"] = c.Q_bar
    out[f"gau_{sch}_beta"] = g.beta
    out[f"gau_{sch}_alpha"] = g.alpha
    out[f"gau_{sch}_alphabar"] = g.alphabar
  for kind in ("linear", "cosine"):
    for steps in (50, 10, 1000):
      s = InferenceSchedule(kind, 1000, steps)
      out[f"infer_{kind}_{steps}"] = np.array([[int(a), int(b)] for a, b in map(s, range(steps))])
  save("schedules", **out)


# ------------------------------------------------------------------------------------------
def ref_encoder(weights, out_channels, node_feature_only, sparse=True, aggregation="sum"):
  m = GNNEncoder(n_layers=12, hidden_dim=256, out_channels=out_channels, aggregation=aggregation,
                 sparse=sparse, use_activation_checkpoint=False,
                 node_feature_only=node_feature_only)
  missing = m.load_state_dict(sd_torch(weights), strict=True)
  assert not missing.missing_keys and not missing.unexpected_keys
  assert list(m.state_dict().keys()) == list(weights.keys()), "key order differs from reference"
  return m.eval()


def gen_forward():
  # --- sparse TSP, categorical (out=2), block-diagonal batch of 2 (couples through the head GN, D4)
  w2 = syn.make_encoder_weights(seed=0, out_channels=2)
  pts, ei = syn.tsp_sparse_batch(30, 6, 2, seed=1234)
  xt = (syn.initial_noise(ei.shape[1], 0) > 0).astype(np.float32)
  m = ref_encoder(w2, 2, False)
  taps = []
  hooks = [m.per_layer_out[l].register_forward_hook(lambda mod, i, o, l=l: taps.append(o.clone()))
           for l in (0, 11)]
  logits = m(torch.from_numpy(pts), torch.tensor([517.0]), torch.from_numpy(xt),
             torch.from_numpy(ei)).numpy()
  for h in hooks:
    h.remove()
  save("fwd_tsp_cat", points=pts, edge_index=ei, xt=xt, t=np.array([517.0], np.float32),
       logits=logits, out_layer0_rows=taps[0].numpy()[::7], out_layer11_rows=taps[1].numpy()[::7])

  # --- sparse TSP, Gaussian (out=1), continuous xt
  w1 = syn.make_encoder_weights(seed=1, out_channels=1)
  pts, ei = syn.tsp_sparse_batch(24, 8, 1, seed=77)
  xtg = syn.initial_noise(ei.shape[1], 3)
  m = ref_encoder(w1, 1, False)
  pred = m(torch.from_numpy(pts), torch.tensor([930.0]), torch.from_numpy(xtg),
           torch.from_numpy(ei)).numpy()
  save("fwd_tsp_gauss", points=pts, edge_index=ei, xt=xtg, t=np.array([930.0], np.float32), pred=pred)

  # --- MIS node-only, unsorted edges, 2 graphs
  ei, sizes = syn.mis_batch(30, 40, 0.15, 2, seed=5)
  V = sum(sizes)
  xtn = (syn.initial_noise(V, 9) > 0).astype(np.float32)
  m = ref_encoder(w2, 2, True)
  logits = m(torch.from_numpy(xtn), torch.tensor([256.0]), edge_index=torch.from_numpy(ei)).numpy()
  save("fwd_mis_cat", edge_index=ei, sizes=np.array(sizes), xt=xtn, t=np.array([256.0], np.float32),
       logits=logits)
  # mean / max aggregation are reachable flags (--aggregation); pin them on the same graph
  for agg in ("mean", "max"):
    m = ref_encoder(w2, 2, True, aggregation=agg)
    lg = m(torch.from_numpy(xtn), torch.tensor([256.0]), edge_index=torch.from_numpy(ei)).numpy()
    save(f"fwd_mis_cat_{agg}", logits=lg)

  # --- dense TSP (config C1 family), B=2 with different timesteps per sample
  B, V = 2, 12
  ptsd = np.stack([syn.tsp_points(V, 4321, b) for b in range(B)])
  xtd = (syn.initial_noise(B * V * V, 11) > 0).astype(np.float32).reshape(B, V, V)
  m = ref_encoder(w2, 2, False, sparse=False)
  td = np.array([801.0, 33.0], np.float32)
  out = m(torch.from_numpy(ptsd), torch.from_numpy(td), torch.from_numpy(xtd), None).numpy()
  save("fwd_dense_cat", points=ptsd, xt=xtd, t=td, out=out)


def gen_ref_copy():
  """What tests/test_reference_copy.py compares against: the sha256 of every reference file oracle/make_ref.py copies,
  and the reference GNNEncoder's forward on the instance that test feeds the oracle port."""
  sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(HERE)), "oracle"))
  import hashlib
  import make_ref
  path = os.path.join(HERE, "ref_sources.sha256")
  with open(path, "w") as f:
    for rel in make_ref.FILES:
      with open(os.path.join(ref_shims.REFERENCE_ROOT, rel), "rb") as src:
        f.write(f"{hashlib.sha256(src.read()).hexdigest()}  {rel}\n")
  print(f"wrote {path}")
  w2 = syn.make_encoder_weights(0, out_channels=2)
  pts, ei = syn.tsp_sparse_batch(30, 7, 2, seed=5)
  xt = (syn.initial_noise(ei.shape[1], 3) > 0).astype(np.float32)
  m = ref_encoder(w2, 2, False)
  logits = m(torch.from_numpy(pts), torch.tensor([321.0]), torch.from_numpy(xt), torch.from_numpy(ei)).numpy()
  save("fwd_tsp_cat_k7", points=pts, edge_index=ei, xt=xt, t=np.array([321.0], np.float32), logits=logits)


# ------------------------------------------------------------------------------------------
class Args(object):
  def __init__(self, **kw):
    self.diffusion_schedule = "linear"
    self.diffusion_steps = 1000
    self.inference_schedule = "cosine"
    self.inference_trick = "ddim"
    self.sequential_sampling = 1
    self.parallel_sampling = 1
    self.n_layers = 12
    self.hidden_dim = 256
    self.aggregation = "sum"
    self.use_activation_checkpoint = False
    self.two_opt_iterations = 0
    self.save_numpy_heatmap = False
    self.training_split_label_dir = None
    self.__dict__.update(kw)


def make_tsp_model(tmp, **kw):
  f = os.path.join(tmp, "tsp.txt")
  with open(f, "w") as fh:
    fh.write("0.1 0.2 0.3 0.4 0.5 0.6 output 1 2 3 1\n")
  a = Args(storage_path=tmp, training_split="tsp.txt", validation_split="tsp.txt",
           test_split="tsp.txt", **kw)
  return pl_tsp_model.TSPModel(param_args=a).eval()


def make_mis_model(tmp, **kw):
  a = Args(storage_path=tmp, training_split="none*", validation_split="none*", test_split="none*",
           sparse_factor=-1, **kw)
  return pl_mis_model.MISModel(param_args=a).eval()


class BernoulliTap(object):
  """Replace torch.bernoulli by (u < p) with injected uniforms and record p."""

  def __init__(self, seed):
    self.seed, self.step, self.ps = seed, 0, []

  def __enter__(self):
    self.orig = torch.bernoulli

    def fake(p, *a, **k):
      u = torch.from_numpy(syn.uniforms(p.numel(), self.seed, self.step)).reshape(p.shape)
      self.ps.append(p.clone().reshape(-1).numpy())
      self.step += 1
      return (u < p).to(p.dtype)
    torch.bernoulli = fake
    return self

  def __exit__(self, *a):
    torch.bernoulli = self.orig


def run_loop(model, task, diffusion_type, steps, points, edge_index, xt, useed):
  """The loop of pl_tsp_model.py:202-217 / pl_mis_model.py:171-186, through the reference methods."""
  device = torch.device("cpu")
  sched = InferenceSchedule(inference_schedule=model.args.inference_schedule, T=model.diffusion.T,
                            inference_T=steps)
  net_out, xts = [], []
  hook = model.model.register_forward_hook(lambda m, i, o: net_out.append(o.clone().numpy()))
  with BernoulliTap(useed) as tap:
    for i in range(steps):
      t1, t2 = sched(i)
      t1 = np.array([t1]).astype(int)
      t2 = np.array([t2]).astype(int)
      fn = model.gaussian_denoise_step if diffusion_type == "gaussian" else model.categorical_denoise_step
      if task == "tsp":
        xt = fn(points, xt, t1, device, edge_index, target_t=t2)
      else:
        xt = fn(xt, t1, device, edge_index, target_t=t2)
      xts.append(xt.clone().float().numpy())
  hook.remove()
  return np.stack(net_out), np.stack(xts), (np.stack(tap.ps) if tap.ps else np.zeros((0,), np.float32))


def gen_trajectories():
  tmp = tempfile.mkdtemp()
  # --- TSP sparse categorical, parallel_sampling = 2 (duplicate_edge_index), 10 steps
  w2 = syn.make_encoder_weights(seed=0, out_channels=2)
  N, K, P, steps = 30, 6, 2, 10
  model = make_tsp_model(tmp, diffusion_type="categorical", sparse_factor=K, parallel_sampling=P,
                         inference_diffusion_steps=steps)
  model.model.load_state_dict(sd_torch(w2), strict=True)
  pts = syn.tsp_points(N, 1234, 0)
  ei1 = syn.knn_edge_index(pts, K)
  points = torch.from_numpy(pts).repeat(P, 1)                                   # pl_tsp_model.py:182
  edge_index = model.duplicate_edge_index(torch.from_numpy(ei1), N, torch.device("cpu"))   # :183
  xt0 = (torch.from_numpy(syn.initial_noise(P * N * K, 21)) > 0).long()          # :186-200
  net, xts, ps = run_loop(model, "tsp", "categorical", steps, points, edge_index, xt0, useed=100)
  save("traj_tsp_cat", points=pts, edge_index_single=ei1, edge_index=edge_index.numpy(),
       xt0=xt0.numpy().astype(np.uint8), net_out=net, xt_out=xts, p=ps,
       meta=np.array([N, K, P, steps]))

  # --- TSP sparse Gaussian (inference works for sparse graphs, SURVEY D7), 6 steps
  w1 = syn.make_encoder_weights(seed=1, out_channels=1)
  N, K, steps = 24, 8, 6
  model = make_tsp_model(tmp, diffusion_type="gaussian", sparse_factor=K, parallel_sampling=1,
                         inference_diffusion_steps=steps)
  model.model.load_state_dict(sd_torch(w1), strict=True)
  pts = syn.tsp_points(N, 77, 0)
  ei1 = syn.knn_edge_index(pts, K)
  xt0 = torch.from_numpy(syn.initial_noise(N * K, 22))
  net, xts, _ = run_loop(model, "tsp", "gaussian", steps, torch.from_numpy(pts), torch.from_numpy(ei1),
                         xt0, useed=101)
  save("traj_tsp_gauss", points=pts, edge_index=ei1, xt0=xt0.numpy(), net_out=net, xt_out=xts,
       meta=np.array([N, K, 1, steps]))

  # --- MIS categorical, parallel_sampling = 2, 8 steps
  steps, P = 8, 2
  model = make_mis_model(tmp, diffusion_type="categorical", parallel_sampling=P,
                         inference_diffusion_steps=steps)
  model.model.load_state_dict(sd_torch(w2), strict=True)
  ei1 = syn.er_graph_edge_index(36, 0.15, seed=5, instance=0)
  V = 36
  edge_index = model.duplicate_edge_index(torch.from_numpy(ei1), V, torch.device("cpu"))
  xt0 = (torch.from_numpy(syn.initial_noise(P * V, 23)) > 0).long()
  net, xts, ps = run_loop(model, "mis", "categorical", steps, None, edge_index, xt0, useed=102)
  save("traj_mis_cat", edge_index_single=ei1, edge_index=edge_index.numpy(),
       xt0=xt0.numpy().astype(np.uint8), net_out=net, xt_out=xts, p=ps, meta=np.array([V, 0, P, steps]))

  # --- MIS Gaussian, 5 steps, linear inference schedule
  steps = 5
  model = make_mis_model(tmp, diffusion_type="gaussian", parallel_sampling=1,
                         inference_diffusion_steps=steps, inference_schedule="linear")
  model.model.load_state_dict(sd_torch(w1), strict=True)
  xt0 = torch.from_numpy(syn.initial_noise(V, 24))
  net, xts, _ = run_loop(model, "mis", "gaussian", steps, None, torch.from_numpy(ei1), xt0, useed=103)
  save("traj_mis_gauss", edge_index=ei1, xt0=xt0.numpy(), net_out=net, xt_out=xts,
       meta=np.array([V, 0, 1, steps]))

  # --- TSP dense categorical (config C1 family: TSP-50 dense is the same code at V=50), V=10, 6 steps
  steps, V = 6, 10
  model = make_tsp_model(tmp, diffusion_type="categorical", sparse_factor=-1, parallel_sampling=1,
                         inference_diffusion_steps=steps)
  model.model.load_state_dict(sd_torch(w2), strict=True)
  pts = syn.tsp_points(V, 999, 0)
  xt0 = (torch.from_numpy(syn.initial_noise(V * V, 25)).reshape(1, V, V) > 0).long()
  net, xts, ps = run_loop(model, "tsp", "categorical", steps, torch.from_numpy(pts)[None], None, xt0,
                          useed=104)
  save("traj_dense_cat", points=pts, xt0=xt0.numpy().astype(np.uint8), net_out=net, xt_out=xts, p=ps,
       meta=np.array([V, 0, 1, steps]))


def gen_mis_decode():
  """utils/mis_utils.py:mis_decode_np of the reference on seeded ER graphs (one case with many exact score ties)."""
  import scipy.sparse
  from utils.mis_utils import mis_decode_np as ref_decode
  out = {}
  for case, (n, p, seed, ties) in enumerate([(60, 0.1, 1, False), (120, 0.15, 2, False), (80, 0.1, 3, True)]):
    ei = syn.er_graph_edge_index(n, p, seed, 0)
    adj = scipy.sparse.coo_matrix((np.ones_like(ei[0]), (ei[0], ei[1])))
    pred = np.random.default_rng(seed).random(n)
    if ties:
      pred = np.round(pred * 4) / 4
    out[f"ei{case}"], out[f"pred{case}"], out[f"sol{case}"] = ei, pred, ref_decode(pred, adj)
  save("mis_decode", **out)



def _reference_tsp_utils():
  """The reference's utils/tsp_utils.py with its real Cython merge: the .pyx is compiled from where it lies in
  /root/reference into a scratch directory under /tmp (nothing is copied into this repository)."""
  import importlib, subprocess, tempfile, shutil
  build = os.path.join(tempfile.gettempdir(), "dfb_ref_cython_merge")
  os.makedirs(build, exist_ok=True)
  if not any(f.startswith("cython_merge.") and f.endswith(".so") for f in os.listdir(build)):
    shutil.copy(os.path.join(ref_shims.REFERENCE_ROOT, "utils", "cython_merge", "cython_merge.pyx"), build)
    with open(os.path.join(build, "setup.py"), "w") as f:
      f.write("from setuptools import setup, Extension\nfrom Cython.Build import cythonize\nimport numpy\n"
              "setup(ext_modules=cythonize([Extension('cython_merge', ['cython_merge.pyx'], "
              "include_dirs=[numpy.get_include()])], language_level=3))\n")
    subprocess.run([sys.executable, "setup.py", "build_ext", "--inplace"], cwd=build, check=True,
                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
  sys.path.insert(0, build)
  real = importlib.import_module("cython_merge")
  import utils.tsp_utils as tu
  tu.merge_cython = real.merge_cython
  return tu


def tsp_decode_cases():
  """(name, N, K (0 = dense), P, heat kind) of the decode fixtures; shared with the tests."""
  return [("s50", 50, 8, 1, "good"), ("s200", 200, 10, 2, "noisy"), ("s120r", 120, 5, 1, "random"),
          ("s300g", 300, 12, 1, "gauss"), ("s30full", 30, 30, 2, "noisy"), ("s40fullg", 40, 40, 1, "gauss"), ("d20", 20, 0, 2, "noisy"), ("d45", 45, 0, 1, "good")]


def tsp_decode_inputs(name, n, k, par, kind):
  """Synthetic heatmaps with the layout test_step hands to merge_tours (pl_tsp_model.py:218-231): sparse ->
  (P*E,) float32 over the kNN edge list; dense -> (P, N, N) float32."""
  rng = np.random.default_rng(sum(map(ord, name)))
  pts = syn.tsp_points(n, seed=7 + n, instance=0).astype(np.float32)
  if k:
    ei = syn.knn_edge_index(pts, k)
    d = np.linalg.norm(pts[ei[0]] - pts[ei[1]], axis=-1)
    shape = (par * ei.shape[1],)
    d = np.tile(d, par)
  else:
    ei = None
    d = np.linalg.norm(pts[:, None] - pts[None], axis=-1)
    shape = (par, n, n)
    d = np.broadcast_to(d, shape)
  u = rng.random(shape)
  if kind == "good":
    heat = np.exp(-8.0 * d * np.sqrt(n)) * (0.7 + 0.3 * u) + 1e-6
  elif kind == "noisy":
    heat = np.exp(-3.0 * d * np.sqrt(n)) * u + 1e-6
  elif kind == "random":
    heat = u + 1e-6
  else:                      # gaussian-diffusion style output: xt * 0.5 + 0.5 may leave [0, 1]
    heat = (np.exp(-6.0 * d * np.sqrt(n)) * 2 - 1 + 0.4 * rng.standard_normal(shape)) * 0.5 + 0.5
  return pts, ei, heat.astype(np.float32)


def gen_tsp_decode():
  """utils/tsp_utils.py of the reference: merge_tours (with the real Cython merge), batched_two_opt_torch on
  the CPU device, TSPEvaluator."""
  tu = _reference_tsp_utils()
  out = {}
  for name, n, k, par, kind in tsp_decode_cases():
    pts, ei, heat = tsp_decode_inputs(name, n, k, par, kind)
    import warnings
    with warnings.catch_warnings():
      warnings.simplefilter("ignore")
      tours, merge_it = tu.merge_tours(heat, pts, ei, sparse_graph=bool(k), parallel_sampling=par)
    tours = np.array(tours).astype("int64")
    out[f"{name}/points"], out[f"{name}/heat"] = pts, heat
    if k:
      out[f"{name}/edge_index"] = ei
    out[f"{name}/tours"], out[f"{name}/merge_iterations"] = tours, np.float64(merge_it)
    for cap in (3, 1000):
      solved, ns = tu.batched_two_opt_torch(pts.astype("float64"), tours, max_iterations=cap, device="cpu")
      out[f"{name}/two_opt_{cap}"], out[f"{name}/two_opt_{cap}_iters"] = solved, np.int64(ns)
    ev = tu.TSPEvaluator(pts)
    out[f"{name}/cost_merged"] = np.array([ev.evaluate(t) for t in tours])
    out[f"{name}/cost_solved"] = np.array([ev.evaluate(t) for t in out[f"{name}/two_opt_1000"]])
    print(name, "merge_it", merge_it, "2opt", int(out[f"{name}/two_opt_1000_iters"]),
          out[f"{name}/cost_merged"], out[f"{name}/cost_solved"])
  save("tsp_decode", **out)


def gen_mcts_txt():
  """tsp_mcts/convert_numpy_to_txt.py of the reference, run unmodified on small dense heat maps.  The script needs
  `fire` (absent: stubbed, main() is called directly) and np.bool (removed in numpy >= 1.24: aliased here only)."""
  import importlib.util, types
  sys.modules.setdefault("fire", types.ModuleType("fire"))
  if not hasattr(np, "bool"):
    np.bool = np.bool_
  spec = importlib.util.spec_from_file_location(
      "ref_convert", os.path.join(os.path.dirname(ref_shims.REFERENCE_ROOT), "tsp_mcts", "convert_numpy_to_txt.py"))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  out = {}
  import contextlib, io
  for case, (n, prob, seed) in enumerate([(40, 0.2, 0), (64, 0.05, 1)]):
    rng = np.random.default_rng(seed)
    pts = syn.tsp_points(n, seed=20 + seed, instance=0).astype(np.float32)
    d = np.linalg.norm(pts[:, None] - pts[None], axis=-1)
    heat = (np.exp(-5.0 * d * np.sqrt(n)) * rng.random((n, n)) + 1e-6).astype(np.float32)
    with tempfile.TemporaryDirectory() as tmp:
      os.makedirs(os.path.join(tmp, "numpy_heatmap"))
      np.save(os.path.join(tmp, "numpy_heatmap", "test-heatmap-0.npy"), heat)
      np.save(os.path.join(tmp, "numpy_heatmap", "test-points-0.npy"), pts)
      with contextlib.redirect_stdout(io.StringIO()):
        mod.main(tmp, os.path.join(tmp, "out"), num_nodes=n, num_files=1, expected_valid_prob=prob)
      with open(os.path.join(tmp, "out", "heatmap", f"tsp{n}", f"heatmaptsp{n}_0.txt"), "rb") as fh:
        text = fh.read()
    out[f"heat{case}"], out[f"points{case}"], out[f"prob{case}"] = heat, pts, np.float64(prob)
    out[f"txt{case}"] = np.frombuffer(text, dtype=np.uint8)
    print("case", case, "n", n, len(text), "bytes")
  save("mcts_txt", **out)


if __name__ == "__main__":
  ap = argparse.ArgumentParser()
  ap.add_argument("--only", default="")
  a = ap.parse_args()
  if a.only in ("", "schedules"):
    gen_schedules()
  if a.only in ("", "forward"):
    gen_forward()
  if a.only in ("", "ref_copy"):
    gen_ref_copy()
  if a.only in ("", "traj"):
    gen_trajectories()
  if a.only in ("", "mis_decode"):
    gen_mis_decode()
  if a.only in ("", "tsp_decode"):
    gen_tsp_decode()
  if a.only in ("", "mcts_txt"):
    gen_mcts_txt()
