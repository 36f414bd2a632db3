# coding: utf-8
"""TEST INFRASTRUCTURE — locating and importing the UNMODIFIED reference (LPD-EPFL/ByzantineMomentum).

Only `tests/`, `__graft_entry__.smoke()` and `bench.py`'s CPU legs (`--impl reference`,
`cpu_baseline`) may import this module; nothing under `byzantinemomentum_b200/` does.

The reference is found through `$BYZ_REFERENCE`, the root of a ByzantineMomentum checkout; it is
never part of this repository.  A root counts when it holds `aggregators/__init__.py` and `attack.py`.

Importing the reference's `tools` package rewires `sys.stdout`, `sys.stderr` and `sys.excepthook`
(tools/__init__.py:215-216,246); `load()` restores them, so a test or the bench keeps its own
streams.  The reference's `aggregators/__init__.py:95-110` imports every sibling module, each of
which registers its rules; nothing of it is modified or copied here.
"""

import importlib
import os
import pathlib
import sys

ROOT = pathlib.Path(__file__).resolve().parent.parent

def candidates():
  env = os.environ.get("BYZ_REFERENCE")
  return [pathlib.Path(env)] if env else []

def find_root():
  """ Root of the first usable reference checkout, or None. """
  for path in candidates():
    if (path / "aggregators" / "__init__.py").exists() and (path / "attack.py").exists():
      return path.resolve()
  return None

_loaded = None

def load():
  """ (root, aggregators module) of the unmodified reference, imported once per process, or
  (None, None) when no reference is present.  The reference root is put FIRST on sys.path so that
  `tools` / `aggregators` / `experiments` / `attacks` resolve to its packages. """
  global _loaded
  if _loaded is not None:
    return _loaded
  root = find_root()
  if root is None:
    _loaded = (None, None)
    return _loaded
  saved = (sys.stdout, sys.stderr, sys.excepthook)
  sys.path.insert(0, str(root))
  try:
    aggregators = importlib.import_module("aggregators")
  finally:
    sys.stdout, sys.stderr, sys.excepthook = saved
  if pathlib.Path(aggregators.__file__).resolve().parent.parent != root:
    raise RuntimeError(f"'aggregators' resolved to {aggregators.__file__}, not to the reference at {root}")
  _loaded = (root, aggregators)
  return _loaded

def describe():
  """ One line for reports: where the reference came from. """
  root = find_root()
  if root is None:
    return "reference not present"
  try:
    rel = root.relative_to(ROOT)
    return f"unmodified reference at <repo>/{rel}"
  except ValueError:
    return f"unmodified reference at {root}"
