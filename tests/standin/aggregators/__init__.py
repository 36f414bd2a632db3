# coding: utf-8
"""Stand-in for the `aggregators` package of the original ByzantineMomentum project, written for the
tests of this repository (it is not the original).  It keeps the original's registry interface:
`gars`, `make_gar` (the rule with its `check`, `checked`, `unchecked`, `upper_bound` and `influence`
members; `checked` raises `tools.UserException` when `check` returns a message), `register` (which
refuses a name in use), and the probe that registers `native-<rule>` when the top-level `native`
package provides it, called positionally.  Its stock rules answer `check()` and Multi-Krum's
`upper_bound(25, 5, 10)` as the original did (tests/golden/reference_checks.json) and aggregate with
this repository's NumPy oracle."""

import json
import math
import pathlib

import torch

import tools
from oracle import byzoracle

RECORDED = json.loads((pathlib.Path(__file__).resolve().parents[2] / "golden" / "reference_checks.json").read_text())
ACCEPTED = {json.dumps(entry) for entry in RECORDED["accepted"]}

def make_gar(unchecked, check, upper_bound=None, influence=None):
  def checked(**kwargs):
    message = check(**kwargs)
    if message is not None:
      raise tools.UserException(f"Aggregation rule cannot be used with the given parameters: {message}")
    return unchecked(**kwargs)
  func = checked if __debug__ else unchecked
  func.check, func.checked, func.unchecked, func.upper_bound, func.influence = check, checked, unchecked, upper_bound, influence
  return func

def register(name, unchecked, check, upper_bound=None, influence=None):
  if name in gars:
    tools.warning(f"Unable to register {name!r} GAR: name already in use")
    return
  gars[name] = make_gar(unchecked, check, upper_bound=upper_bound, influence=influence)

gars = dict()

def _stock(name):
  def unchecked(gradients, f=None, **kwargs):
    rows = [g.detach().cpu().numpy() for g in gradients]
    out = getattr(byzoracle, name)(rows, f=f, **kwargs)
    return torch.from_numpy(out.astype("float32")).to(gradients[0].device)
  def check(gradients, f=None, **kwargs):
    if json.dumps([name, len(gradients), f, kwargs]) in ACCEPTED:
      return None
    return f"{name} does not accept n={len(gradients)}, f={f!r}, {kwargs}"
  def upper_bound(n, f, d):
    return RECORDED["krum_upper_bound_25_5_10"] if (name, n, f, d) == ("krum", 25, 5, 10) else math.nan
  return unchecked, check, upper_bound

for _name in ("average", "median", "trmean", "phocas", "meamed", "krum", "bulyan", "brute", "aksel", "cge"):
  register(_name, *_stock(_name))

try:
  import native
except ImportError:
  native = None

_NATIVE = {"median": lambda mod: lambda gradients, **kwargs: mod.aggregate(gradients),
           "krum": lambda mod: lambda gradients, f, m=None, **kwargs: mod.aggregate(gradients, f, m),
           "bulyan": lambda mod: lambda gradients, f, m=None, **kwargs: mod.aggregate(gradients, f, m),
           "brute": lambda mod: lambda gradients, f, **kwargs: mod.aggregate(gradients, f)}
if native is not None:
  for _name, _wrap in _NATIVE.items():
    if _name in dir(native):
      register("native-" + _name, _wrap(getattr(native, _name)), gars[_name].check, gars[_name].upper_bound)

for _name, _rule in gars.items():
  globals()[_name] = _rule
