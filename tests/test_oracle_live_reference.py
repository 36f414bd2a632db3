# coding: utf-8
"""Beyond the committed goldens: reference outputs for other seeds and shapes (`tests/golden/live/`,
written by `tests/golden/make_golden.py --live` from the unmodified reference), checked against the
oracle with the same comparisons as the goldens."""

import pathlib

import conftest
from test_oracle_golden import test_oracle_matches_reference as check_call

LIVE_DIR = pathlib.Path(__file__).resolve().parent / "golden" / "live"

def test_oracle_matches_fresh_reference_outputs():
  paths = sorted(LIVE_DIR.glob("golden_live_*.npz"))
  assert len(paths) == 21, [p.name for p in paths]
  checked = 0
  for path in paths:
    golden = conftest.Golden(path)
    for call in golden.calls:
      check_call(golden, call)
      checked += 1
  assert checked > 450, checked
