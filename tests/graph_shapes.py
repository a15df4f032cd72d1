"""Seeded irregular edge lists, one family per code path of the edge layer.

dfb_prepare_graph counts max_seg, the most node segments (runs of equal row) inside one 32-edge group of the row-sorted
edge list, and the tensor-core edge layer picks its kernel by it:
  fast      max_seg <= 2        the pair kernel's prefix-sum reduce
  general   3 <= max_seg <= 8   the pair kernel's per-segment reduce (edge_layer_v2.cuh, MAXSEG = 8)
  fallback  max_seg > 8         the single-CTA kernel for every layer
Every generator returns row-sorted lists and the tests count max_seg themselves (`segments`), so a change to a generator
cannot move a case to another path unnoticed.  All graphs are valid inputs of the C-ABI: degree-0 nodes, self-loops and
hubs included."""
import numpy as np

GROUP = 32     # edges per aggregation group (csrc/common.cuh)
TILE = 128     # edge rows per tensor-core tile; the pair kernel's cluster of two CTAs takes two tiles
MAXSEG = 8     # node segments per group the pair kernel handles

TINY_SIZES = [1, 31, 32, 33, 127, 128, 129, 255, 256, 257, 3 * 128, 5 * 128 + 1]


class Graph(object):
  def __init__(self, name, degrees, col, rng):
    self.name = name
    self.degrees = np.asarray(degrees, dtype=np.int64)
    self.V = int(self.degrees.size)
    self.rowptr = np.concatenate([[0], np.cumsum(self.degrees)])
    self.E = int(self.rowptr[-1])
    row = np.repeat(np.arange(self.V, dtype=np.int64), self.degrees)
    self.edge_index = np.stack([row, np.asarray(col, dtype=np.int64)])
    self.points = rng.random((self.V, 2))

  def __repr__(self):
    return f"{self.name}(V={self.V}, E={self.E})"


def segments(row):
  """Per 32-edge group of a row-sorted list: (node segments, nodes spanned first..last incl. degree-0 ones)."""
  row = np.asarray(row)
  n_groups = (row.size + GROUP - 1) // GROUP
  segs = np.empty(n_groups, dtype=np.int64)
  span = np.empty(n_groups, dtype=np.int64)
  for g in range(n_groups):
    r = row[g * GROUP:(g + 1) * GROUP]
    segs[g] = 1 + int(np.count_nonzero(r[1:] != r[:-1]))
    span[g] = int(r[-1] - r[0] + 1)
  return segs, span


def path_of(max_seg):
  return "fast" if max_seg <= 2 else ("general" if max_seg <= MAXSEG else "fallback")


def _pad_to_group_start(degrees, lo, hi, rng):
  """Append degrees in [lo, hi] until the edge count is 1 mod 32: the last node then has exactly one edge at the start
  of the next group."""
  while sum(degrees) % GROUP != 1:
    r = (1 - sum(degrees)) % GROUP
    degrees.append(r if lo <= r <= hi else int(rng.integers(lo, hi + 1)))


def _with_gaps(degrees, rng, p):
  """Insert degree-0 nodes after each node with probability p (they own no edges: the segments do not change)."""
  out = [0]
  for d in degrees:
    out.append(d)
    if d and rng.random() < p:
      out.extend([0] * int(rng.integers(1, 3)))
  return out


def fast_graph(seed=0):
  """Degrees in [32, 600] with two hubs (1500 and 3100 edges, 12 and 25 tiles, crossing tile-pair boundaries),
  degree-0 nodes between them, and a last partial tile."""
  rng = np.random.default_rng(seed)
  degrees = [int(d) for d in rng.integers(32, 601, size=34)]
  degrees[5], degrees[20] = 1500, 3100
  degrees = _with_gaps(degrees, rng, 0.15)
  if sum(degrees) % TILE == 0:
    degrees[-1] += 1
  V = len(degrees)
  return Graph("fast", degrees, rng.integers(0, V, sum(degrees)), rng)


def general_graph(seed=0):
  """Degrees in [5, 31] with degree-0 nodes interleaved; one group is planted to hold exactly 8 segments: the last edge
  of a node, six nodes of degree 5 (degree-0 nodes between them), the first edge of the next node."""
  rng = np.random.default_rng(seed)
  head = [int(d) for d in rng.integers(5, 32, size=300)]
  _pad_to_group_start(head, 5, 31, rng)
  planted = []
  for _ in range(6):
    planted += [5, 0]
  tail = [int(d) for d in rng.integers(5, 32, size=300)]
  degrees = _with_gaps(head, rng, 0.2) + planted + _with_gaps(tail, rng, 0.2)
  V = len(degrees)
  return Graph("general", degrees, rng.integers(0, V, sum(degrees)), rng)


def fallback_graph(seed=0):
  """Degrees 1 to 4: paths, stars of up to 4 leaves, and SATLIB-like nodes (a self-loop plus 1 to 3 neighbours); one
  group is planted to hold exactly 9 segments (1 + 7 x 4 + 3 edges)."""
  rng = np.random.default_rng(seed)
  degrees, cols = [], []

  def path(n):
    b = len(degrees)
    for i in range(n):
      nb = [b + j for j in (i - 1, i + 1) if 0 <= j < n]
      degrees.append(len(nb)); cols.extend(nb)

  def star(k):
    c = len(degrees)
    degrees.append(k); cols.extend(range(c + 1, c + 1 + k))
    for _ in range(k):
      degrees.append(1); cols.append(c)

  def satlib(d):            # neighbours are drawn once V is known
    i = len(degrees)
    degrees.append(d); cols.append(i); cols.extend([-1] * (d - 1))

  for _ in range(100):
    path(int(rng.integers(2, 30)))
    star(int(rng.integers(1, 5)))
    for _ in range(int(rng.integers(1, 20))):
      satlib(int(rng.integers(2, 5)))
  while sum(degrees) % GROUP != 1:
    satlib(min(4, (1 - sum(degrees)) % GROUP))
  for _ in range(8):        # seven whole nodes of degree 4 and the first three edges of the eighth
    satlib(4)
  for _ in range(300):
    satlib(int(rng.integers(2, 5)))
  V = len(degrees)
  cols = np.asarray(cols)
  free = cols < 0
  cols[free] = rng.integers(0, V, int(free.sum()))
  return Graph("fallback", degrees, cols, rng)


def tiny_graphs(seed=0):
  """Edge lists of 1 to 641 edges (odd and even tile counts, partial and whole last tiles) in two layouts: degree 40
  (pair kernel, fast reduce) and degree 7 (pair kernel, general reduce); E = 1 is one node with one self-loop."""
  rng = np.random.default_rng(seed)
  out = [Graph("tiny-E1-V1-selfloop", [1], [0], rng)]
  for deg in (40, 7):
    for E in TINY_SIZES[1:]:
      degrees = [deg] * (E // deg) + ([E % deg] if E % deg else [])
      V = len(degrees)
      out.append(Graph(f"tiny-E{E}-d{deg}", degrees, rng.integers(0, V, E), rng))
  return out


def graph_classes():
  """{class name: [Graph, ...]}"""
  return {"fast": [fast_graph(1)], "general": [general_graph(2)], "fallback": [fallback_graph(3)],
          "tiny": tiny_graphs(4)}
