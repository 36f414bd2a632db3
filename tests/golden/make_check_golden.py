#!/usr/bin/env python3
# coding: utf-8
"""Generate `tests/golden/reference_checks.json`: which (rule, n, f, extra arguments) the UNMODIFIED
reference's own `aggregators.gars[name].check(...)` accepts on the grid of the test, Multi-Krum's
`upper_bound(25, 5, 10)`, and how often each statement group tools/drive_attack.py rewrites occurs in
the reference's attack.py, by SHA-256 (tests/test_reference_integration.py and the stand-in under
tests/standin/ use them).  Needs the reference checkout:

    BYZ_REFERENCE=<ByzantineMomentum checkout> python tests/golden/make_check_golden.py
"""

import hashlib
import importlib.util
import json
import pathlib
import sys

HERE = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent))

from oracle import reference  # noqa: E402
from test_reference_integration import check_grid  # noqa: E402

def main():
  import torch
  root, aggregators = reference.load()
  if aggregators is None:
    raise SystemExit("set BYZ_REFERENCE to the root of a ByzantineMomentum checkout")
  accepted = []
  for name, n, f, extra in check_grid():
    try:
      if aggregators.gars[name].check(gradients=[torch.zeros(4) for _ in range(n)], f=f, **extra) is None:
        accepted.append([name, n, f, extra])
    except TypeError:
      pass
  spec = importlib.util.spec_from_file_location("drive_attack", HERE.parent.parent / "tools" / "drive_attack.py")
  drive = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(drive)
  source = (root / "attack.py").read_text()
  lo, hi = source.index(drive.STUDY_BEGIN), source.index(drive.STUDY_END)
  sha = lambda text: hashlib.sha256(text.encode()).hexdigest()
  attack_py = {sha(text): source.count(text) for text in (drive.CLIP_AND_CLONE, drive.MOMENTUM, drive.STUDY_BEGIN, drive.STUDY_END)}
  attack_py["study_block"] = sha(source[lo:hi])
  lines = ",\n  ".join(json.dumps(entry) for entry in accepted)
  (HERE / "reference_checks.json").write_text(
    f'{{"krum_upper_bound_25_5_10": {aggregators.gars["krum"].upper_bound(25, 5, 10)!r},\n "attack_py": {json.dumps(attack_py)},\n'
    f' "accepted": [\n  {lines}]}}\n')

if __name__ == "__main__":
  main()
