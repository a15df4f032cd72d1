"""Recipe for oracle/_ref/: the UNMODIFIED reference sources of the denoise path, copied where they can travel.

Test / baseline infrastructure only (never imported by the product).  /root/reference does not exist on the GPU box,
so the `bench.py --impl reference` arm cannot read it there; this script copies the reference's own Python files
(difusco/{pl_meta_model,pl_tsp_model,pl_mis_model}.py, models/, utils/*.py, co_datasets/*.py - the six files SURVEY 8a
cites plus the modules they import) byte for byte into oracle/_ref/difusco/.  The directory is git-ignored (no reference
source enters the history) but NOT gpurun-ignored, so it ships to the box with the snapshot like a built .so.
Run by __graft_entry__.build() whenever /root/reference is present:

    python oracle/make_ref.py            # copy + verify (sha256 of every file against the source)
"""
import hashlib
import os
import shutil
import sys

SRC = "/root/reference/difusco"
DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "difusco")
FILES = [
    "pl_meta_model.py", "pl_tsp_model.py", "pl_mis_model.py",
    "models/__init__.py", "models/gnn_encoder.py", "models/nn.py",
    "utils/__init__.py", "utils/diffusion_schedulers.py", "utils/lr_schedulers.py", "utils/tsp_utils.py",
    "utils/mis_utils.py",
    "co_datasets/__init__.py", "co_datasets/tsp_graph_dataset.py", "co_datasets/mis_dataset.py",
]


def _sha(path):
  return hashlib.sha256(open(path, "rb").read()).hexdigest()


def make(verbose=True, src=SRC, dst=DST):
  """Returns the destination directory, or None when the reference tree is not mounted (the GPU box)."""
  if not os.path.isdir(src):
    return dst if os.path.isdir(dst) else None
  for rel in FILES:
    s, d = os.path.join(src, rel), os.path.join(dst, rel)
    os.makedirs(os.path.dirname(d), exist_ok=True)
    if not os.path.exists(d) or _sha(s) != _sha(d):
      shutil.copyfile(s, d)
    assert _sha(s) == _sha(d), rel
  with open(os.path.join(dst, "MANIFEST.sha256"), "w") as f:
    for rel in FILES:
      f.write(f"{_sha(os.path.join(dst, rel))}  {rel}\n")
  if verbose:
    print(f"oracle/_ref: {len(FILES)} reference files copied unmodified to {dst}")
  return dst


def available():
  return os.path.isdir(DST) and all(os.path.exists(os.path.join(DST, rel)) for rel in FILES)


if __name__ == "__main__":
  sys.exit(0 if make() else 1)
