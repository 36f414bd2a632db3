# coding: utf-8
"""Shared test plumbing: markers, path setup, golden-fixture loading."""

import json
import pathlib
import sys

import numpy as np
import pytest

ROOT = pathlib.Path(__file__).resolve().parent.parent
if str(ROOT) not in sys.path:
  sys.path.insert(0, str(ROOT))

GOLDEN_DIR = ROOT / "tests" / "golden"

def reference_root():
  """ Root of the unmodified reference checkout named by $BYZ_REFERENCE, or None. """
  from oracle import reference
  return reference.find_root()

needs_reference = pytest.mark.skipif(reference_root() is None, reason="needs a reference checkout: set BYZ_REFERENCE")

def pytest_configure(config):
  config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")

class Golden:
  """One golden fixture: input rows + the reference's recorded outputs."""
  def __init__(self, path):
    self.path = path
    self.data = np.load(path, allow_pickle=False)
    self.manifest = json.loads(str(self.data["manifest"]))
    self.rows = self.data["rows"]
    self.name = self.manifest["name"]
    self.n = self.manifest["n"]
    self.nb = self.manifest["nb_byz"]
    self.nh = self.n - self.nb
    self.calls = self.manifest["calls"]
  def get(self, tag, what):
    key = f"{tag}/{what}"
    return self.data[key] if key in self.data.files else None

def golden_paths():
  return sorted(GOLDEN_DIR.glob("golden_*.npz"))

def load_goldens():
  return [Golden(p) for p in golden_paths()]

def golden_calls():
  """ Flat list of (golden, call) for parametrisation. """
  out = []
  for g in load_goldens():
    for call in g.calls:
      out.append(pytest.param(g, call, id=f"{g.name}:{call['tag']}"))
  return out

def canon_alias(indices, nh):
  """ Byzantine rows are one aliased object in the reference: all indices >= nh are equivalent. """
  return [min(int(i), nh) for i in indices]
