#!/usr/bin/env python3
# coding: utf-8
"""Generate `tests/golden/fullsize/c*.npz`: what the UNMODIFIED reference's
`aggregators.gars[g].unchecked(gradients=<cpu rows>, f=f)` and `influence()` return on the rows of
`tests/test_cuda_vs_reference_fullsize.py` (BASELINE.json's full sizes), reduced to what that test
compares: SHA-256 digests of the bit-exact outputs, the trimmed-mean tail columns, every output at a
seeded sample of columns, and the influence values.  Needs the reference checkout:

    BYZ_REFERENCE=<ByzantineMomentum checkout> python tests/golden/make_fullsize_golden.py
"""

import pathlib
import sys

import numpy as np

HERE = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent.parent))
sys.path.insert(0, str(HERE.parent))

import test_cuda_vs_reference_fullsize as t  # noqa: E402
from oracle import reference  # noqa: E402

def main():
  import torch
  root, ref = reference.load()
  if ref is None:
    raise SystemExit("set BYZ_REFERENCE to the root of a ByzantineMomentum checkout")
  out_dir = HERE / "fullsize"
  out_dir.mkdir(exist_ok=True)
  files = {}
  def case(name, n, nb, d, seed, dist):
    x, nh = t.host_stack(n, nb, d, seed, dist)
    data = files.setdefault(name.split("/")[0], {})
    cols = t.sample_columns(d)
    data[f"columns_{d}"] = cols.astype(np.int32)
    data[name + "/rows"] = np.array(t.digest(x))
    return x, nh, t.as_rows(x, nh), cols, data
  def record(data, key, value, cols, trmean=False):
    value = value.numpy()
    data[key + "/sample"] = value[cols]
    if trmean:
      body = value.shape[0] - value.shape[0] % 32
      data[key + "/body"] = np.array(t.digest(value[:body]))
      data[key + "/tail"] = value[body:]
    else:
      data[key + "/digest"] = np.array(t.digest(value))
  gars = ref.gars
  for dist in ("iid", "empire"):
    x, nh, cpu, cols, data = case(f"c1/{dist}", 11, 0 if dist == "iid" else 5, 79_510, 11, dist)
    record(data, f"c1/{dist}/median", gars["median"].unchecked(gradients=cpu, f=5), cols)
  for dist, nb in (("iid", 0), ("empire", 10)):
    x, nh, cpu, cols, data = case(f"c2/{dist}", 25, nb, 1_310_922, 12, dist)
    for name in ("trmean", "median", "phocas", "meamed", "average"):
      record(data, f"c2/{dist}/{name}", gars[name].unchecked(gradients=cpu, f=10), cols, trmean=name == "trmean")
  for dist, nbyz in (("empire", 5), ("iid", 0)):
    x, nh, cpu, cols, data = case(f"c3/{dist}", 25, nbyz, 1_310_922, t.C3_SEED, dist)
    for name, kwargs, tag in t.C3_RULES + (("bulyan", {}, "bulyan"),):
      key = f"c3/{dist}/{tag}"
      record(data, key, gars[name].unchecked(gradients=cpu, f=5, **kwargs), cols)
      if nbyz and name != "bulyan":
        data[key + "/influence"] = np.float64(gars[name].influence(cpu[:nh], cpu[nh:], f=5, **kwargs))
  for dist, nb in (("empire", 3), ("iid", 0)):
    x, nh, cpu, cols, data = case(f"c5/{dist}", 11, nb, 1_310_922, 15, dist)
    record(data, f"c5/{dist}/brute", gars["brute"].unchecked(gradients=cpu, f=3), cols)
    if nb:
      data[f"c5/{dist}/brute/influence"] = np.float64(gars["brute"].influence(cpu[:nh], cpu[nh:], f=3))
  x, nh, cpu, cols, data = case("c4/empire", 51, 12, 36_546_980 // 8, 14, "empire")
  record(data, "c4/empire/trmean", gars["trmean"].unchecked(gradients=cpu, f=12), cols, trmean=True)
  record(data, "c4/empire/median", gars["median"].unchecked(gradients=cpu, f=12), cols)
  for name, data in files.items():
    path = out_dir / f"{name}.npz"
    np.savez_compressed(path, torch=np.array(torch.__version__), threads=np.int64(torch.get_num_threads()), **data)
    print(f"{path.name}: {len(data)} arrays, {path.stat().st_size / 1024:.0f} KiB")

if __name__ == "__main__":
  main()
