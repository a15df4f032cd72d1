"""The in-kernel sampler against a numpy reference.

`dfb_denoise` (what bench.py, TSPModel.denoise_heatmap and MISModel.denoise_labels run) passes no uniforms, so every
Bernoulli draw is philox_uniform(seed, step, element) and every DDPM noise value is philox_normal(seed, step, element)
(csrc/common.cuh).  These tests pin both bit for bit (the uniform) or to a few fp32 ulp (the normal):
  * CPU: tests/philox_ref.py against the Random123 known-answer vectors and a scalar Python port;
  * GPU: one step with uniforms = NULL against the reference on a shuffled TSP edge list and an MIS batch;
  * GPU: the fused loop (captured graph and plain launches) equals the same steps run one by one with step_index = i;
  * GPU: the DDPM noise of a Gaussian model with inference_trick=None."""
import math

import numpy as np
import pytest
import torch

import philox_ref as PR
from conftest import rel_linf

SEED = 0x0123456789ABCDEF          # both 32-bit halves non-zero and different: a swapped key split changes every draw
STEP_INDICES = [0, 1, 70001, 2 ** 31 - 1]   # includes one >= 2^16 and the largest step_index the C-ABI takes
M32 = 0xFFFFFFFF


# ------------------------------------------------------------------------------------------------
# CPU: the reference itself
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ctr,key,expect", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((M32, M32, M32, M32), (M32, M32), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox4x32_10_known_answers(ctr, key, expect):
  """Random123's known-answer vectors for philox4x32_10."""
  got = PR.philox4x32_10(ctr, key)
  assert tuple(int(x) for x in got) == expect
  # the vectorised form gives the same words in every lane
  many = PR.philox4x32_10([np.full(5, c, dtype=np.uint64) for c in ctr], key)
  for w, e in zip(many, expect):
    assert (w == e).all()


def _philox_scalar(ctr, key):
  c0, c1, c2, c3 = ctr
  k0, k1 = key
  for _ in range(10):
    p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
    c0, c1, c2, c3 = ((p1 >> 32) ^ c1 ^ k0) & M32, p1 & M32, ((p0 >> 32) ^ c3 ^ k1) & M32, p0 & M32
    k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
  return c0, c1, c2, c3


def _scalar_draws(seed, step, elem):
  key = (seed & M32, seed >> 32)
  x = _philox_scalar((elem & M32, elem >> 32, step & M32, 0), key)[0]
  u = (x >> 8) / 2.0 ** 24
  x, y = _philox_scalar((elem & M32, elem >> 32, step & M32, 1), key)[:2]
  u1 = float(np.float32((x >> 8) + 0.5)) / 2.0 ** 24     # one fp32 rounding of the exact sum, as (float)(x >> 8) + 0.5f
  u2 = (y >> 8) / 2.0 ** 24
  return u, math.sqrt(-2.0 * math.log(u1)) * math.cos(2.0 * math.pi * u2)


@pytest.mark.parametrize("seed", [0, SEED, 2 ** 64 - 1])
@pytest.mark.parametrize("step", [0, 1, 65537, 2 ** 32 - 1])
def test_uniform_and_normal_match_scalar_port(seed, step):
  elems = [0, 1, 255, 2 ** 32 - 1, 2 ** 32, 2 ** 40 + 12345, 2 ** 63 + 5]
  u = PR.uniform(seed, step, np.array(elems, dtype=np.uint64))
  z = PR.normal(seed, step, np.array(elems, dtype=np.uint64))
  assert u.dtype == np.float32
  for i, e in enumerate(elems):
    su, sz = _scalar_draws(seed, step, e)
    assert float(u[i]) == su, (e, float(u[i]), su)
    assert abs(z[i] - sz) <= 1e-14 * max(1.0, abs(sz)), (e, z[i], sz)


def test_uniform_layout_properties():
  e = np.arange(1 << 16, dtype=np.uint64)
  u = PR.uniform(SEED, 3, e)
  k = u.astype(np.float64) * 2.0 ** 24
  assert (k == np.floor(k)).all() and u.min() >= 0.0 and u.max() < 1.0     # 24-bit lattice in [0, 1)
  assert abs(u.mean() - 0.5) < 5 * math.sqrt(1 / 12 / e.size)
  # every input word matters: element high word, step, seed halves
  assert not np.array_equal(u, PR.uniform(SEED, 3, e + np.uint64(1 << 32)))
  assert not np.array_equal(u, PR.uniform(SEED, 4, e))
  assert not np.array_equal(u, PR.uniform(SEED ^ 1, 3, e))
  assert not np.array_equal(u, PR.uniform(SEED ^ (1 << 32), 3, e))
  # the normal uses counter word 3 = 1: its first word is not the uniform's
  u1, _ = PR.normal_uniforms(SEED, 3, e)
  assert np.mean(np.abs(u1 - u) < 2.0 ** -23) < 0.01


# ------------------------------------------------------------------------------------------------
# GPU helpers
# ------------------------------------------------------------------------------------------------
def _stream():
  return torch.cuda.current_stream().cuda_stream


def _tsp_graph(seed=17, n=120, k=12, batch=2):
  """A k-NN TSP batch and the same edge list shuffled (the caller's order is not row sorted, so the kernels carry a
  permutation)."""
  from difusco_b200 import synthetic as syn
  pts, ei = syn.tsp_sparse_batch(n, k, batch, seed=seed)
  q = np.random.default_rng(seed).permutation(ei.shape[1])
  eis = np.ascontiguousarray(ei[:, q])
  assert (np.diff(eis[0]) < 0).any()
  return pts, ei, eis, q


def _categorical_step(ctx, xt, t1, consts, step_index, seed=SEED):
  import gpu_util as G
  from difusco_b200 import _cabi
  n = xt.size
  x = G.cu(xt.astype(np.float32))
  xo, p, net = (torch.empty(n, device="cuda"), torch.empty(n, device="cuda"), torch.empty((n, 2), device="cuda"))
  ctx.denoise_step(_cabi.CATEGORICAL, x.data_ptr(), float(t1), consts, 0, None, seed, step_index, xo.data_ptr(),
                   p.data_ptr(), net.data_ptr(), _stream())
  torch.cuda.synchronize()
  return xo.cpu().numpy(), p.cpu().numpy(), net.cpu().numpy()


def _check_bernoulli(xo, p, seed, step):
  """xt_out[o] == (u(seed, step, o) < clip(p_out[o], 0, 1)), exactly; and the check has teeth: a wrong key split or a
  wrong step would change at least 1 % of the decisions on this input."""
  n = xo.size
  o = np.arange(n, dtype=np.uint64)
  pc = np.minimum(np.maximum(p, np.float32(0)), np.float32(1))
  expect = (PR.uniform(seed, step, o) < pc).astype(np.float32)
  bad = np.flatnonzero(xo != expect)
  assert bad.size == 0, (step, bad.size, bad[:8])
  swapped = ((seed & M32) << 32) | (seed >> 32)
  for wrong in (PR.uniform(swapped, step, o), PR.uniform(seed, (step + 1) & M32, o), PR.uniform(seed, step, o[::-1])):
    assert np.mean((wrong < pc) != expect) > 0.01


# ------------------------------------------------------------------------------------------------
# GPU: one categorical step, uniforms = NULL
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_categorical_step_philox_bitwise_tsp_shuffled(weights2):
  import gpu_util as G
  from difusco_b200 import synthetic as syn
  pts, ei, eis, q = _tsp_graph()
  n = ei.shape[1]
  dev = torch.device("cuda")
  m = G.tsp_model(weights2, "tc", sparse_factor=12)
  m._prepare(G.cu(pts), G.cu(eis), dev)
  ctx = m.model.engine()
  ref = G.tsp_model(weights2, "tc", sparse_factor=12)      # the same graph in row order: no permutation
  ref._prepare(G.cu(pts), G.cu(ei), dev)
  for j, step in enumerate(STEP_INDICES):
    xt = (syn.initial_noise(n, 40 + j) > 0).astype(np.float32)     # caller order
    t1 = 900 - 120 * j
    consts, last = m.posterior_consts(t1, t1 - 20)
    assert last == 0
    xo, p, net = _categorical_step(ctx, xt, t1, consts, step)
    _check_bernoulli(xo, p, SEED, step)
    assert 0.05 < xo.mean() < 0.95
    # outputs are in the caller's order: element o of the shuffled list is sorted edge q[o]
    _, ps, ns = _categorical_step(ref.model.engine(), xt[np.argsort(q)], t1, consts, step)
    # (5e-5: the tensor-core kernel's own error level, see SHUFFLE_TOL in test_gpu_graph_shapes.py; a lost caller order
    # is O(1) on the logits)
    assert rel_linf(net, ns[q]) < 5e-5, rel_linf(net, ns[q])
    assert np.abs(p - ps[q]).max() < 5e-5


@pytest.mark.gpu
def test_categorical_step_philox_bitwise_mis_batch(weights2):
  import gpu_util as G
  from difusco_b200 import synthetic as syn
  ei, sizes = syn.mis_batch(60, 90, 0.15, 3, seed=5)
  V = int(sum(sizes))
  m = G.mis_model(weights2, "tc")
  m.model.set_graph(G.cu(ei), V, 1)
  ctx = m.model.engine()
  for j, step in enumerate(STEP_INDICES):
    xt = (syn.initial_noise(V, 60 + j) > 0).astype(np.float32)
    t1 = 800 - 100 * j
    consts, _ = m.posterior_consts(t1, t1 - 50)
    xo, p, _ = _categorical_step(ctx, xt, t1, consts, step)
    _check_bernoulli(xo, p, SEED, step)


# ------------------------------------------------------------------------------------------------
# GPU: the fused loop equals the same steps run one by one
# ------------------------------------------------------------------------------------------------
def _schedule(m, steps):
  from oracle import difusco_oracle as orc
  t1s, cs, ls = [], [], []
  for t1, t2 in orc.inference_schedule(m.args.inference_schedule, 1000, steps):
    c, last = m.posterior_consts(t1, t2)
    t1s.append(int(t1)); cs.append(c); ls.append(last)
  return t1s, cs, ls


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["tsp_categorical", "mis_categorical", "tsp_ddpm"])
def test_fused_loop_equals_step_loop(weights1, weights2, case):
  import gpu_util as G
  from difusco_b200 import _cabi, synthetic as syn
  dev = torch.device("cuda")
  S = 6
  if case == "mis_categorical":
    ei, sizes = syn.mis_batch(60, 90, 0.15, 3, seed=6)
    n = int(sum(sizes))
    m = G.mis_model(weights2, "tc", inference_diffusion_steps=S)
    m.model.set_graph(G.cu(ei), n, 1)
  else:
    pts, _, eis, _ = _tsp_graph(seed=23, n=90, k=10)
    n = eis.shape[1]
    if case == "tsp_ddpm":
      m = G.tsp_model(weights1, "tc", diffusion_type="gaussian", inference_trick=None, sparse_factor=10,
                      inference_diffusion_steps=S)
    else:
      m = G.tsp_model(weights2, "tc", sparse_factor=10, inference_diffusion_steps=S)
    m._prepare(G.cu(pts), G.cu(eis), dev)
  ctx = m.model.engine()
  gauss = case == "tsp_ddpm"
  mode = _cabi.GAUSSIAN if gauss else _cabi.CATEGORICAL
  xt0 = syn.initial_noise(n, 31).astype(np.float32)
  if not gauss:
    xt0 = (xt0 > 0).astype(np.float32)
  t1s, cs, ls = _schedule(m, S)
  if gauss:
    assert all(c[3] != 0 for c in cs)     # DDPM: noise at every step

  state = G.cu(xt0)
  for i in range(S):
    out = torch.empty(n, device=dev)
    ctx.denoise_step(mode, state.data_ptr(), float(t1s[i]), cs[i], ls[i], None, SEED, i, out.data_ptr(), None, None,
                     _stream())
    state = out
  stepped = state.cpu().numpy()

  results = []
  for capture in (True, True, False):     # capture, replay, plain launches
    ctx.set_graph_capture(capture)
    x = G.cu(xt0)
    ctx.denoise(mode, x.data_ptr(), t1s, cs, ls, None, SEED, _stream())
    results.append(x.cpu().numpy())
  ctx.set_graph_capture(True)
  for r in results:
    assert np.array_equal(r, stepped), int((r != stepped).sum())
  assert np.isfinite(stepped).all() and not np.array_equal(stepped, xt0)


# ------------------------------------------------------------------------------------------------
# GPU: DDPM noise (philox_normal) of one Gaussian step
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gaussian_ddpm_step_noise_matches_reference(weights1):
  import gpu_util as G
  from difusco_b200 import _cabi, synthetic as syn
  from oracle import difusco_oracle as orc
  dev = torch.device("cuda")
  pts, _, eis, _ = _tsp_graph(seed=29, n=200, k=16, batch=2)
  n = eis.shape[1]
  m = G.tsp_model(weights1, "tc", diffusion_type="gaussian", inference_trick=None, sparse_factor=16,
                  inference_diffusion_steps=50)
  m._prepare(G.cu(pts), G.cu(eis), dev)
  ctx = m.model.engine()
  o = np.arange(n, dtype=np.uint64)
  sched = orc.inference_schedule("cosine", 1000, 50)
  for j, step in enumerate(STEP_INDICES):
    t1, t2 = sched[[0, 17, 35, 45][j]]
    c, _ = m.posterior_consts(t1, t2)
    assert c[3] != 0
    xt = syn.initial_noise(n, 70 + j).astype(np.float32)
    x = G.cu(xt)
    xo, net = torch.empty(n, device=dev), torch.empty((n, 1), device=dev)
    ctx.denoise_step(_cabi.GAUSSIAN, x.data_ptr(), float(t1), c, 0, None, SEED, step, xo.data_ptr(), None,
                     net.data_ptr(), _stream())
    torch.cuda.synchronize()
    xo, l0 = xo.cpu().numpy(), net.cpu().numpy()[:, 0]
    # y with the kernel's fp32 operation order (head_posterior): y = c0 (x - c1 l0); y = y + c2 l0
    y = c[0] * (xt - c[1] * l0)
    y = y + c[2] * l0
    assert y.dtype == np.float32
    z = PR.normal(SEED, step, o)
    ref = y.astype(np.float64) + float(c[3]) * z
    # tolerance: the device z differs from the float64 z by the error of logf (1 ulp), sqrtf (0.5 ulp), cospif (1 ulp)
    # and the product (0.5 ulp): <= 3 ulp of |z| <= 3 * 2^-23 |z|, taken as 2^-20 |z|; fmaf rounds xt_out once
    # (0.5 ulp), taken as 2 ulp = 2^-22 |xt_out|.
    tol = abs(float(c[3])) * 2.0 ** -20 * np.abs(z) + 2.0 ** -22 * np.abs(ref) + 1e-30
    err = np.abs(xo - ref)
    assert (err <= tol).all(), (step, float((err / tol).max()))
    # the tolerance is far below what a layout error would cause: counter word 3 = 0 instead of 1, or u1 / u2 swapped
    u1, u2 = PR.normal_uniforms(SEED, step, o)
    wrong_word = y + float(c[3]) * PR.box_muller(*PR.normal_uniforms(SEED, step, o, counter_word3=0))
    swapped = y + float(c[3]) * PR.box_muller(u2.astype(np.float64) + 2.0 ** -25, u1.astype(np.float64) - 2.0 ** -25)
    for alt in (wrong_word, swapped):
      assert np.median(np.abs(alt - ref)) > 100 * tol.max()
    # sanity of the reference itself: N(0, 1) over the elements, and the device's implied noise agrees
    for zz in (z, (xo.astype(np.float64) - y) / float(c[3])):
      assert abs(zz.mean()) < 5 / math.sqrt(n) and abs(zz.var() - 1) < 5 * math.sqrt(2 / n), (zz.mean(), zz.var())
