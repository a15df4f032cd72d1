"""oracle/_ref (the UNMODIFIED reference files that travel with a built tree for `bench.py --impl reference`): the recipe
oracle/make_ref.py copies byte for byte and writes a matching manifest, a copy that is present is the reference as
pinned by tests/golden/ref_sources.sha256, and the reference GNNEncoder's own forward (tests/golden/fwd_tsp_cat_k7.npz)
matches the oracle port.  Both fixtures are written by tests/golden/make_golden.py from the unmodified reference."""
import hashlib
import os
import sys

from conftest import GOLDEN, ROOT, golden, rel_linf
from difusco_b200 import synthetic as syn
from oracle import difusco_oracle as orc

sys.path.insert(0, os.path.join(ROOT, "oracle"))
import make_ref  # noqa: E402


def _sha(path):
  return hashlib.sha256(open(path, "rb").read()).hexdigest()


def _manifest(path):
  out = {}
  for line in open(path):
    h, rel = line.split()
    out[rel] = h
  return out


def test_ref_copy_is_byte_identical_and_manifest_matches(tmp_path):
  # the recipe on a stand-in tree with the reference's layout
  src, dst = tmp_path / "src", tmp_path / "dst"
  for i, rel in enumerate(make_ref.FILES):
    (src / rel).parent.mkdir(parents=True, exist_ok=True)
    (src / rel).write_bytes(f"# stand-in {i} for {rel}\n".encode())
  assert make_ref.make(verbose=False, src=str(src), dst=str(dst)) == str(dst)
  manifest = _manifest(dst / "MANIFEST.sha256")
  assert sorted(manifest) == sorted(make_ref.FILES)
  for rel in make_ref.FILES:
    assert (dst / rel).read_bytes() == (src / rel).read_bytes(), rel
    assert _sha(dst / rel) == manifest[rel], rel
  # the pinned hashes of the reference cover the recipe's files; a copy that is present is unmodified
  ref = _manifest(os.path.join(GOLDEN, "ref_sources.sha256"))
  assert sorted(ref) == sorted(make_ref.FILES)
  if make_ref.available():
    assert _manifest(os.path.join(make_ref.DST, "MANIFEST.sha256")) == ref
    for rel in make_ref.FILES:
      assert _sha(os.path.join(make_ref.DST, rel)) == ref[rel], rel
  # no reference source may enter the history: the directory is git-ignored
  assert "oracle/_ref/" in open(os.path.join(ROOT, ".gitignore")).read()


def test_ref_copy_forward_matches_oracle_port():
  g = golden("fwd_tsp_cat_k7")
  w = syn.make_encoder_weights(0, out_channels=2)
  out = orc.encoder_forward_sparse_tsp(orc.Weights(w), g["points"], g["xt"], g["t"], g["edge_index"])
  err = rel_linf(out.numpy(), g["logits"])
  assert err < 1e-5, err
