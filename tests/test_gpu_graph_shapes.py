"""The edge kernels on irregular graphs, against the float64 oracle.

k-NN and ER workloads give every 32-edge group at most two node segments.  These graphs reach the other paths of the
tensor-core edge layer (see tests/graph_shapes.py): the pair kernel's general per-segment reduce, the single-CTA
fallback for groups with more than 8 segments, degree-0 nodes between rows, hubs spanning dozens of tiles, and edge
lists of 1 to 641 edges.  Each class runs the three encoders (TSP with categorical xt through the layer-0 table, TSP
with Gaussian xt through the scalar features, MIS) under every implementation and aggregation, fed once row sorted and
once shuffled.  The class checks run on the CPU; the rest needs a GPU."""
import numpy as np
import pytest
import torch

from conftest import rel_linf
import graph_shapes as GS

CLASSES = GS.graph_classes()
TASKS = ["tsp_categorical", "tsp_gaussian", "mis"]
AGGS = ["sum", "mean", "max"]
T = 437.0
PROB_TOL = 1e-4
# Sorted vs shuffled input: the stable sort by row keeps the caller's order inside a row, so the aggregation sums run in
# another order and differ by an fp32 ulp.  The fp32 kernel passes that on at the ulp level.  The split-bf16 products of
# the tensor-core kernels are not continuous in their inputs: an ulp can move the bf16 split of a value and change a
# product by up to its ~2^-17 error, so the two runs differ at the level of the kernel's own error (B200: up to 1.9e-5,
# also for a single node whose edges are only reordered, where no permutation is involved).  Any indexing error
# (caller order lost, a stale graph reused) is O(1).
SHUFFLE_TOL = {"fp32": 1e-5, "tc": 5e-5, "tc1": 5e-5}


# ------------------------------------------------------------------------------------------------
# CPU: every case lands in the class it claims
# ------------------------------------------------------------------------------------------------
def test_fast_class():
  (g,) = CLASSES["fast"]
  segs, span = GS.segments(g.edge_index[0])
  assert GS.path_of(segs.max()) == "fast" and segs.max() == 2
  assert g.degrees[g.degrees > 0].min() >= 32 and g.E <= 30000
  first, last = g.rowptr[:-1], g.rowptr[1:] - 1
  hub = (g.degrees > 0) & (last // GS.TILE - first // GS.TILE >= 2) & (first // (2 * GS.TILE) != last // (2 * GS.TILE))
  assert hub.any()                                          # a hub over more than 2 tiles, crossing a tile pair
  assert (last // GS.TILE - first // GS.TILE).max() >= 24   # and one over dozens of tiles
  assert g.E % GS.TILE != 0                                 # a partial last tile
  assert (span > segs).any()                                # degree-0 nodes inside a group


def test_general_class():
  (g,) = CLASSES["general"]
  segs, span = GS.segments(g.edge_index[0])
  assert GS.path_of(segs.max()) == "general" and segs.max() == GS.MAXSEG
  assert set(np.unique(g.degrees[g.degrees > 0])) <= set(range(5, 32)) and g.E <= 30000
  assert (g.degrees == 0).sum() > 50 and g.degrees[0] == 0
  assert (span > segs).any() and (span[segs == GS.MAXSEG] > GS.MAXSEG).any()   # gaps inside the 8-segment group


def test_fallback_class():
  (g,) = CLASSES["fallback"]
  segs, _ = GS.segments(g.edge_index[0])
  assert GS.path_of(segs.max()) == "fallback"
  assert (segs == GS.MAXSEG + 1).any()
  assert g.degrees.min() >= 1 and g.degrees.max() <= 4 and g.E <= 30000
  assert (g.edge_index[0] == g.edge_index[1]).any()       # SATLIB-like self-loops


def test_tiny_class():
  gs = CLASSES["tiny"]
  assert sorted({g.E for g in gs}) == sorted(GS.TINY_SIZES)
  tiles = {-(-g.E // GS.TILE) for g in gs}
  assert {1, 3} <= tiles and any(t % 2 for t in tiles if t > 1)     # odd tile counts: a cluster with one idle CTA
  assert any(g.V == 1 and g.E == 1 and g.edge_index[0, 0] == g.edge_index[1, 0] for g in gs)
  paths = {GS.path_of(GS.segments(g.edge_index[0])[0].max()) for g in gs if g.E >= 33}
  assert paths == {"fast", "general"}


# ------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------
def _inputs(g, task):
  rng = np.random.default_rng(g.E * 7 + len(task))
  n = g.V if task == "mis" else g.E
  z = rng.standard_normal(n).astype(np.float32)
  return z if task == "tsp_gaussian" else (z > 0).astype(np.float32)


@pytest.fixture(scope="module")
def oracle_out(weights1, weights2):
  """float64 oracle output per (class, graph, task, aggregation), shared by the three implementations."""
  from oracle import difusco_oracle as orc
  w = {1: orc.Weights(weights1, dtype=torch.float64), 2: orc.Weights(weights2, dtype=torch.float64)}
  cache = {}

  def get(cls, i, task, agg):
    key = (cls, i, task, agg)
    if key not in cache:
      g = CLASSES[cls][i]
      xt = _inputs(g, task)
      if task == "mis":
        out = orc.encoder_forward_mis(w[2], xt, np.array([T]), g.edge_index, aggregation=agg)
      else:
        out = orc.encoder_forward_sparse_tsp(w[1 if task == "tsp_gaussian" else 2], g.points, xt, np.array([T]),
                                             g.edge_index, aggregation=agg)
      cache[key] = out.numpy()
    return cache[key]
  return get


@pytest.fixture(scope="module")
def encoders(weights1, weights2):
  """One encoder per (task, impl, aggregation); each counts the graphs its context prepares."""
  import gpu_util as G
  cache = {}

  def get(task, impl, agg):
    key = (task, impl, agg)
    if key not in cache:
      if task == "mis":
        enc = G.encoder(weights2, 2, node_only=True, impl=impl, aggregation=agg)
      elif task == "tsp_gaussian":
        enc = G.encoder(weights1, 1, impl=impl, aggregation=agg)
      else:
        enc = G.encoder(weights2, 2, impl=impl, aggregation=agg)
      ctx = enc.engine()
      prepared = []
      real = ctx.prepare_graph

      def counting(ptr, *a, **k):
        prepared.append(ptr)
        return real(ptr, *a, **k)
      ctx.prepare_graph = counting
      enc.prepared = prepared
      cache[key] = enc
    return cache[key]
  return get


def _run(enc, task, g, ei, xt):
  """ei (2, E) int64 CUDA tensor, xt in the order of ei's edges (TSP) or nodes (MIS) -> output rows."""
  import gpu_util as G
  from difusco_b200 import _cabi
  if task == "mis":
    return enc(G.cu(xt), torch.tensor([T]), edge_index=ei).cpu().numpy()
  if task == "tsp_gaussian":
    return enc(G.cu(g.points), torch.tensor([T]), G.cu(xt), ei).cpu().numpy()
  # categorical xt through the denoise step: layer 0 reads the two-row table, the head returns the logits as net_out
  ctx = enc.set_graph(ei, g.V, 1)
  enc.set_points(G.cu(g.points))
  x = G.cu(xt)
  xo, net = torch.empty(g.E, device="cuda"), torch.empty((g.E, 2), device="cuda")
  ctx.denoise_step(_cabi.CATEGORICAL, x.data_ptr(), T, [0.5, 0.5, 0.5, 0.5], 1, None, 0, 0, xo.data_ptr(), None,
                   net.data_ptr(), torch.cuda.current_stream().cuda_stream)
  return net.cpu().numpy()


def _prob_rel(out, ref):
  p = torch.softmax(torch.as_tensor(out, dtype=torch.float64), -1).numpy()
  pr = torch.softmax(torch.as_tensor(ref), -1).numpy()
  return float(np.abs(p / pr - 1).max())


@pytest.mark.gpu
@pytest.mark.parametrize("impl", ["tc", "tc1", "fp32"])
@pytest.mark.parametrize("agg", AGGS)
@pytest.mark.parametrize("task", TASKS)
@pytest.mark.parametrize("cls", list(CLASSES))
def test_graph_class_vs_oracle(encoders, oracle_out, cls, task, agg, impl):
  import gpu_util as G
  enc = encoders(task, impl, agg)
  for i, g in enumerate(CLASSES[cls]):
    ref = oracle_out(cls, i, task, agg)
    xt = _inputs(g, task)
    ei = G.cu(g.edge_index)
    out = _run(enc, task, g, ei, xt)
    assert out.shape == ref.shape and np.isfinite(out).all(), g
    err = rel_linf(out, ref)
    assert err < G.TOL[impl], (g, err)
    if task != "tsp_gaussian":
      assert _prob_rel(out, ref) < PROB_TOL, (g, _prob_rel(out, ref))
    # the same graph shuffled: a fresh graph is prepared, and the output permuted back matches the sorted run
    q = np.random.default_rng(g.E).permutation(g.E)
    eis = G.cu(g.edge_index[:, q])
    n_prepared = len(enc.prepared)
    out_s = _run(enc, task, g, eis, xt if task == "mis" else xt[q])
    assert enc.prepared[n_prepared:] == [eis.data_ptr()], g
    back = out_s if task == "mis" else out_s[np.argsort(q)]
    assert rel_linf(back, out) < SHUFFLE_TOL[impl], (g, rel_linf(back, out))
    assert rel_linf(back, ref) < G.TOL[impl], (g, rel_linf(back, ref))
