"""How much of the tolerance each implementation uses on the irregular graph classes of tests/graph_shapes.py: worst
forward error against the float64 oracle per (class, implementation), over the three encoders and three aggregations."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from conftest import rel_linf
from difusco_b200 import synthetic as syn
from oracle import difusco_oracle as orc
import gpu_util as G
import graph_shapes as GS
import test_gpu_graph_shapes as TG

W = {"tsp_categorical": syn.make_encoder_weights(seed=0, out_channels=2),
     "tsp_gaussian": syn.make_encoder_weights(seed=1, out_channels=1),
     "mis": syn.make_encoder_weights(seed=0, out_channels=2)}
W64 = {k: orc.Weights(v, dtype=torch.float64) for k, v in W.items()}
ENC = {}

print(f"{torch.cuda.get_device_name(0)}; rel-Linf vs the float64 oracle (logits), max |p/p_ref - 1| of the softmax "
      "probabilities (categorical encoders); worst over tasks x aggregations x graphs of the class", flush=True)
for cls, graphs in TG.CLASSES.items():
  segs = max(int(GS.segments(g.edge_index[0])[0].max()) for g in graphs)
  worst = {impl: [0.0, 0.0, ""] for impl in ("fp32", "tc1", "tc")}
  for task in TG.TASKS:
    for agg in TG.AGGS:
      for g in graphs:
        xt = TG._inputs(g, task)
        if task == "mis":
          ref = orc.encoder_forward_mis(W64[task], xt, np.array([TG.T]), g.edge_index, aggregation=agg).numpy()
        else:
          ref = orc.encoder_forward_sparse_tsp(W64[task], g.points, xt, np.array([TG.T]), g.edge_index,
                                               aggregation=agg).numpy()
        for impl in worst:
          key = (task, impl, agg)
          if key not in ENC:
            ENC[key] = G.encoder(W[task], W[task]["out.2.weight"].shape[0], node_only=task == "mis", impl=impl,
                                 aggregation=agg)
          out = TG._run(ENC[key], task, g, G.cu(g.edge_index), xt)
          e = rel_linf(out, ref)
          p = TG._prob_rel(out, ref) if task != "tsp_gaussian" else 0.0
          w = worst[impl]
          if e > w[0]:
            w[0], w[2] = e, f"{task}/{agg}/{g.name}"
          w[1] = max(w[1], p)
  Es = sorted(g.E for g in graphs)
  print(f"class {cls:8s} max_seg {segs:2d}  E {Es[0]}..{Es[-1]} ({len(graphs)} graphs)", flush=True)
  for impl, (e, p, where) in worst.items():
    print(f"   impl={impl:4s}: logits {e:.2e} (tol {G.TOL[impl]:.0e}, at {where})  probs {p:.2e} (tol 1e-04)", flush=True)
