#!/usr/bin/env python3
# coding: utf-8
"""Generate the golden fixtures `tests/golden/golden_*.npz` by running the UNMODIFIED
reference (`/root/reference`, or $BYZ_REFERENCE) on seeded inputs.

Run in the build container only (the reference does not exist on the GPU box):

    python tests/golden/make_golden.py

Each fixture holds, per case: the [n, d] fp32 input rows (Byzantine rows last; in the
reference call they are ONE tensor object repeated, as `attacks/identical.py:86` produces),
and, for every rule/parameter combination the reference's own `check()` accepts, the
reference's output vector plus — for the selection rules — the indices it selected
(recovered by object identity from `_compute_scores` / `_compute_selection` /
`_compute_distances` / `_compute_normed`) and its `influence()` value.
The manifest (JSON string inside the npz) records torch/numpy versions and thread count.
"""

import json
import os
import pathlib
import sys

import numpy as np
import torch

REF = os.environ.get("BYZ_REFERENCE", "/root/reference")
sys.path.insert(0, REF)
_stdout, _stderr, _hook = sys.stdout, sys.stderr, sys.excepthook
import aggregators  # noqa: E402  (wraps stdout/stderr at import: tools/__init__.py:215-216,246)
sys.stdout, sys.stderr, sys.excepthook = _stdout, _stderr, _hook

HERE = pathlib.Path(__file__).resolve().parent

# ---------------------------------------------------------------------------- #
# Input distributions (SURVEY.md §8(d))

def make_rows(kind, n, nb, d, seed):
  """ Returns (honest rows [n-nb, d], one Byzantine row [d] or None). """
  gen = torch.Generator().manual_seed(seed)
  nh = n - nb
  if kind == "iid":
    honest = torch.randn(nh, d, generator=gen)
    byz = torch.randn(d, generator=gen) if nb else None
  elif kind in ("empire", "nan", "little"):
    mu = torch.randn(d, generator=gen)
    sigma = torch.linspace(0.5, 1.5, nh)
    honest = mu[None, :] + sigma[:, None] * torch.randn(nh, d, generator=gen)
    if kind == "empire":
      byz = honest.mean(dim=0).mul(-1.1)
    elif kind == "little":
      byz = honest.mean(dim=0) - 1.5 * honest.var(dim=0).sqrt()
    else:
      byz = torch.full((d,), float("nan"))
  elif kind == "quant":
    # Heavily tied values: exercises equal keys, equal distances, -0.0
    honest = torch.randint(-3, 4, (nh, d), generator=gen).to(torch.float32)
    honest[honest == 0] = honest[honest == 0] * -1.  # some -0.0
    byz = torch.randint(-3, 4, (d,), generator=gen).to(torch.float32) if nb else None
  elif kind == "inf":
    honest = torch.randn(nh, d, generator=gen)
    mask = torch.rand(nh, d, generator=gen) < 0.02
    honest[mask] = float("inf")
    mask = torch.rand(nh, d, generator=gen) < 0.02
    honest[mask] = float("-inf")
    byz = torch.randn(d, generator=gen) if nb else None
  else:
    raise KeyError(kind)
  return honest.contiguous(), (None if byz is None else byz.contiguous())

KAT_HONEST = [[1.0, 2.0, -1.0, 0.5], [1.5, 1.0, -2.0, 0.0], [0.5, 3.0, -1.5, 1.0],
              [2.0, 2.5, -0.5, -0.5], [1.2, 1.8, -1.1, 0.4]]

# (name, kind, n, nb_byz, d, seed, f list)
CASES = [
  ("kat_finite", "kat", 7, 2, 4, 0, [1, 2, 3]),
  ("kat_nan", "katnan", 7, 2, 4, 0, [1, 2, 3]),
  ("iid_n5_d33", "iid", 5, 1, 33, 101, [1, 2]),
  ("iid_n7_d257", "iid", 7, 2, 257, 102, [1, 2, 3]),
  ("empire_n11_d1000", "empire", 11, 3, 1000, 103, [2, 3, 5]),
  ("little_n12_d515", "little", 12, 2, 515, 104, [2, 4]),
  ("iid_n11_d79", "iid", 11, 0, 79, 105, [1, 2, 5]),
  ("empire_n25_d4099", "empire", 25, 5, 4099, 106, [2, 5, 10, 11, 12]),
  ("nan_n25_d1031", "nan", 25, 5, 1031, 107, [5, 10]),
  ("iid_n25_d2048", "iid", 25, 0, 2048, 108, [5, 10]),
  ("iid_n26_d300", "iid", 26, 5, 300, 109, [5, 12]),
  ("empire_n51_d1031", "empire", 51, 12, 1031, 110, [12, 24]),
  ("iid_n51_d160", "iid", 51, 0, 160, 111, [12, 25]),
  ("quant_n9_d400", "quant", 9, 2, 400, 112, [1, 2, 4]),
  ("quant_n25_d512", "quant", 25, 5, 512, 113, [5, 10]),
  ("inf_n11_d600", "inf", 11, 2, 600, 114, [2, 3]),
  ("nan_n11_d64", "nan", 11, 3, 64, 115, [3, 5]),
  ("iid_n1_d50", "iid", 1, 0, 50, 116, [1]),
  ("iid_n2_d50", "iid", 2, 0, 50, 117, [1]),
  ("iid_n3_d1", "iid", 3, 1, 1, 118, [1]),
  ("iid_n64_d130", "iid", 64, 10, 130, 119, [10, 15, 31]),
  ("empire_n33_d777", "empire", 33, 7, 777, 120, [7, 16]),
  ("iid_n19_d100", "iid", 19, 0, 100, 121, [1, 4, 9]),
]

def module(name):
  return sys.modules["aggregators." + name]

def ident_index(rows, tensor):
  for i, row in enumerate(rows):
    if row is tensor:
      return i
  raise RuntimeError("selected tensor not found by identity")

def run_case(name, kind, n, nb, d, seed, fs):
  if kind in ("kat", "katnan"):
    honest = torch.tensor(KAT_HONEST, dtype=torch.float32)
    byz = torch.tensor([9.0, -9.0, 9.0, -9.0]) if kind == "kat" else torch.full((4,), float("nan"))
  else:
    honest, byz = make_rows(kind, n, nb, d, seed)
  honests = [honest[i] for i in range(honest.shape[0])]
  attacks = [byz] * nb if nb else []
  rows = honests + attacks
  assert len(rows) == n
  out = {"rows": torch.stack(rows).numpy().copy()}
  calls = []
  def record(gar, params, tag):
    rule = aggregators.gars[gar]
    kw = dict(gradients=rows, **params)
    if rule.check(**kw) is not None:
      return
    entry = dict(gar=gar, params=params, tag=tag)
    # Selection first (cheap ones only), so a failing rule is skipped as a whole
    try:
      if gar == "krum":
        n_ = len(rows)
        m = params.get("m") or (n_ - params["f"] - 2)
        scores = module("krum")._compute_scores(rows, params["f"], m)
        out[tag + "/order"] = np.array([ident_index(rows, g) for _, g in scores], dtype=np.int64)
        out[tag + "/scores"] = np.array([s for s, _ in scores], dtype=np.float64)
      elif gar == "brute":
        out[tag + "/selection"] = np.array(module("brute")._compute_selection(rows, params["f"]), dtype=np.int64)
      elif gar == "aksel":
        dlist, c = module("aksel")._compute_distances(rows, params["f"], params.get("mode", "mid"))
        out[tag + "/order"] = np.array([i for i, _ in dlist], dtype=np.int64)
        out[tag + "/dists"] = np.array([x for _, x in dlist], dtype=np.float64)
        entry["c"] = c
      elif gar == "cge":
        normed = module("cge")._compute_normed(rows)
        out[tag + "/order"] = np.array([ident_index(rows, g) for _, g in normed], dtype=np.int64)
        out[tag + "/norms"] = np.array([s for s, _ in normed], dtype=np.float64)
      res = rule.unchecked(**kw)
    except Exception as err:  # the reference itself fails on this input (e.g. brute with NaN rows)
      entry["raises"] = type(err).__name__
      calls.append(entry)
      return
    out[tag + "/out"] = res.numpy().copy()
    if rule.influence is not None and nb > 0:
      ikw = {k: v for k, v in params.items()}
      try:
        entry["influence"] = float(rule.influence(honests, attacks, **ikw))
      except Exception as err:
        entry["influence_raises"] = type(err).__name__
    calls.append(entry)
  record("average", {}, "average")
  record("median", {}, "median")
  for f in fs:
    for gar in ("trmean", "phocas", "meamed", "cge"):
      record(gar, dict(f=f), f"{gar}_f{f}")
    for mode in ("mid", "n-f"):
      record("aksel", dict(f=f, mode=mode), f"aksel_f{f}_{mode}")
    m_max = n - f - 2
    for m in sorted({None, 1, max(1, m_max // 2)}, key=lambda x: -1 if x is None else x):
      params = dict(f=f) if m is None else dict(f=f, m=m)
      suffix = "" if m is None else f"_m{m}"
      record("krum", params, f"krum_f{f}{suffix}")
      record("bulyan", params, f"bulyan_f{f}{suffix}")
    # brute is exponential in Python: keep C(n, n-f) * pairs small
    import math
    if math.comb(n, n - f) <= 1000:
      record("brute", dict(f=f), f"brute_f{f}")
  manifest = dict(name=name, kind=kind, n=n, nb_byz=nb, d=int(out["rows"].shape[1]), seed=seed, calls=calls,
                  torch=torch.__version__, numpy=np.__version__, threads=torch.get_num_threads())
  out["manifest"] = np.array(json.dumps(manifest))
  return out

# Other seeds and shapes than CASES, kept apart under live/ (tests/test_oracle_live_reference.py):
# (name, kind, n, nb_byz, d, seed, fs), three seeds each
LIVE_CASES = [
  ("live_iid_n13", "iid", 13, 3, 211, 9001, [1, 2, 3, 5]),
  ("live_empire_n17", "empire", 17, 4, 333, 9002, [2, 3, 4, 7]),
  ("live_little_n10", "little", 10, 2, 97, 9003, [1, 2, 3]),
  ("live_nan_n9", "nan", 9, 2, 65, 9004, [1, 2, 3]),
  ("live_inf_n15", "inf", 15, 3, 130, 9005, [1, 3, 5]),
  ("live_quant_n21", "quant", 21, 4, 96, 9006, [2, 4, 9]),
  ("live_iid_n40", "iid", 40, 9, 75, 9007, [3, 9, 18]),
]
LIVE_CASES = [(f"{name}_s{k}", kind, n, nb, d + 7 * k, seed + 100 * k, fs) for (name, kind, n, nb, d, seed, fs) in LIVE_CASES for k in range(3)]

def main():
  """ `make_golden.py` writes CASES, `make_golden.py --live` writes LIVE_CASES under live/. """
  torch.set_num_threads(1)  # thread-count independent results where ATen's order depends on it
  live = sys.argv[1:] == ["--live"]
  total = 0
  for case in (LIVE_CASES if live else CASES):
    data = run_case(*case)
    path = (HERE / "live" if live else HERE) / f"golden_{case[0]}.npz"
    np.savez_compressed(path, **data)
    total += path.stat().st_size
    man = json.loads(str(data["manifest"]))
    print(f"{path.name}: {len(man['calls'])} calls, {path.stat().st_size / 1024:.0f} KiB")
  print(f"total {total / 1024:.0f} KiB")

if __name__ == "__main__":
  main()
