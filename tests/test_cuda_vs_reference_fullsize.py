# coding: utf-8
"""GPU parity pinned to the REFERENCE ITSELF at BASELINE.json's full sizes (VERDICT r1 weak #2).

The goldens stop at d = 4,099 and `tests/test_cuda_fullsize.py` checks against the C oracle (a
restatement).  Here the CUDA rules are compared with what the unmodified reference's
`aggregators.gars[g].unchecked(gradients=<cpu rows>, f=f)` returned on the SAME seeded rows,
recorded by `tests/golden/make_fullsize_golden.py` in `tests/golden/fullsize/`:
  * bit-exact values are stored as a SHA-256 digest of the whole output (value equality:
    -0.0 and +0.0, and every NaN, are hashed alike) plus a seeded sample of columns, so a
    mismatch names a column where it can;
  * trimmed mean: digest of the bit-exact body, and the `d mod 32` ATen tail columns in full;
  * closest-m means (phocas, meamed, bulyan stage 2): the values at 8,192 seeded columns;
  * selections: the reference does not return them, so they are compared through what they
    determine — `influence()` (exact) and the ordered-subset mean itself, which is bit-exact
    when and only when the same rows were picked in the same order (krum, brute, aksel, cge).
Sizes: C1 (median n=11 d=79,510), C2 (trmean n=25 f=10 d=1,310,922), C3 (Multi-Krum + Bulyan
n=25 f=5 d=1,310,922, empire), C5 (brute n=11 f=3 d=1,310,922), plus one C4 shard (n=51 f=12,
d=4,568,372 = 36,546,980 / 8).
"""

import hashlib

import numpy as np
import pytest

import conftest
import parity

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLDEN = conftest.GOLDEN_DIR / "fullsize"
SAMPLE = 8_192

def host_stack(n, nb, d, seed, dist="empire"):
  """ [n, d] fp32 rows and the number of honest ones.  Distribution B of SURVEY §8(d) (shared
  mean + per-worker noise scale, nb Byzantine rows = -1.1 * mean(honest)) or A (i.i.d. N(0, 1),
  no Byzantine rows), drawn with NumPy's PCG64 so that every machine builds the same bits. """
  rng = np.random.default_rng(seed)
  nh = n - nb
  if dist == "iid":
    return rng.standard_normal((n, d), dtype=np.float32), nh
  x = np.empty((n, d), dtype=np.float32)
  mu = rng.standard_normal(d, dtype=np.float32)
  for i in range(nh):
    x[i] = mu + np.float32(0.5 + i / max(nh - 1, 1)) * rng.standard_normal(d, dtype=np.float32)
  if nb:
    x[nh:] = (x[:nh].astype(np.float64).mean(axis=0) * -1.1).astype(np.float32)
  return x, nh

def as_rows(x, nh, device=None):
  """ One tensor per row; the Byzantine rows are ONE tensor object repeated, as the reference's
  attacks produce them. """
  rows = [torch.from_numpy(x[i]) for i in range(nh)]
  if device is not None:
    rows = [r.to(device) for r in rows]
  if nh < x.shape[0]:
    byz = torch.from_numpy(x[nh])
    rows += [byz if device is None else byz.to(device)] * (x.shape[0] - nh)
  return rows

def sample_columns(d):
  """ The columns whose values are stored (the recorded file keeps them too). """
  return np.sort(np.random.default_rng(d).choice(d, size=min(SAMPLE, d), replace=False))

def digest(values):
  """ SHA-256 of fp32 values up to value equality (-0.0 -> +0.0, every NaN -> one NaN). """
  a = np.array(values, dtype=np.float32)
  a[a == 0] = 0
  a[np.isnan(a)] = np.nan
  return hashlib.sha256(a.tobytes()).hexdigest()

class Recorded:
  """ The reference's outputs of one test, as stored by make_fullsize_golden.py. """
  def __init__(self, name):
    self.z = np.load(GOLDEN / f"{name}.npz", allow_pickle=False)
  def __getitem__(self, key):
    return self.z[key]
  def text(self, key):
    return str(self.z[key])
  def rows(self, case, x):
    assert digest(x) == self.text(case + "/rows"), f"{case}: the seeded rows differ from the recorded ones"
    return self.z[f"columns_{x.shape[1]}"]
  def exact(self, key, got, cols, what):
    parity.assert_bit_exact(got[cols], self[key + "/sample"], what + " [sampled columns]")
    assert digest(got) == self.text(key + "/digest"), f"{what}: differs from the reference outside the sampled columns"
  def trmean(self, key, got, x, cols, what):
    d = got.shape[0]
    body = d - d % 32
    inside = cols[cols < body]
    parity.assert_bit_exact(got[inside], self[key + "/sample"][:inside.size], what + " [body, sampled columns]")
    assert digest(got[:body]) == self.text(key + "/body"), f"{what} [body]: differs from the reference outside the sampled columns"
    if body < d:
      parity.assert_close_scaled(got[body:], self[key + "/tail"], parity.column_scale(x[:, body:]), what + " [ATen tail columns]")

def _np(t):
  return t.detach().cpu().numpy()

def test_c1_median():
  import byzantinemomentum_b200 as bz
  ref = Recorded("c1")
  for dist in ("iid", "empire"):
    x, nh = host_stack(11, 0 if dist == "iid" else 5, 79_510, 11, dist)
    cols = ref.rows(f"c1/{dist}", x)
    ref.exact(f"c1/{dist}/median", _np(bz.gars["median"](gradients=as_rows(x, nh, DEV), f=5)), cols, f"C1 median {dist}")

def test_c2_trmean_phocas_meamed():
  import byzantinemomentum_b200 as bz
  ref = Recorded("c2")
  n, f, d = 25, 10, 1_310_922
  for dist, nb in (("iid", 0), ("empire", 10)):
    x, nh = host_stack(n, nb, d, 12, dist)
    cols = ref.rows(f"c2/{dist}", x)
    dev = as_rows(x, nh, DEV)
    key = f"c2/{dist}/"
    ref.trmean(key + "trmean", _np(bz.gars["trmean"](gradients=dev, f=f)), x, cols, f"C2 trmean {dist}")
    ref.exact(key + "median", _np(bz.gars["median"](gradients=dev, f=f)), cols, f"C2 median {dist}")
    xs = x[:, cols]
    for name, center in (("phocas", "trmean"), ("meamed", "median")):
      amb = parity.closest_ambiguous(xs, n - f, ref[key + center + "/sample"])
      parity.assert_close_scaled(_np(bz.gars[name](gradients=dev, f=f))[cols], ref[key + name + "/sample"], parity.column_scale(xs),
                                 f"C2 {name} {dist} [sampled columns]", exempt=amb)
    ref.exact(key + "average", _np(bz.gars["average"](gradients=dev, f=f)), cols, f"C2 average {dist}")

# cge sums the selected rows in the order of their norms: on i.i.d. rows the norms lie within
# ~1e-6 of each other, so the seed is one where they are apart by more than fp32 rounding
# (2.5e-6 at the closest), or the reference's own order would depend on its reduction order
C3_SEED = 413
C3_RULES = (("krum", {}, "krum"), ("krum", dict(m=1), "krum_m1"), ("aksel", {}, "aksel"), ("aksel", dict(mode="n-f"), "aksel_n-f"), ("cge", {}, "cge"))

def test_c3_krum_bulyan_and_the_other_distance_rules():
  import byzantinemomentum_b200 as bz
  ref = Recorded("c3")
  n, nb, f, d = 25, 5, 5, 1_310_922
  for dist, nbyz in (("empire", nb), ("iid", 0)):
    x, nh = host_stack(n, nbyz, d, C3_SEED, dist)
    cols = ref.rows(f"c3/{dist}", x)
    dev = as_rows(x, nh, DEV)
    xs = x[:, cols]
    scale = parity.column_scale(xs)
    for name, kwargs, tag in C3_RULES:
      key = f"c3/{dist}/{tag}"
      got = _np(bz.gars[name](gradients=dev, f=f, **kwargs))
      if name == "aksel":
        # aksel.py:41: distances are an fp32 ATen sum whose order depends on the thread count; the
        # selection is compared through influence below and the mean to 1e-6 (it is bit-exact
        # when the selection agrees — asserted too, on these seeds it does)
        parity.assert_close_scaled(got[cols], ref[key + "/sample"], scale, f"C3 {name} {kwargs} {dist} [sampled columns]")
      ref.exact(key, got, cols, f"C3 {name} {kwargs} {dist}")
      if nbyz:
        assert bz.gars[name].influence(dev[:nh], dev[nh:], f=f, **kwargs) == float(ref[key + "/influence"]), (name, kwargs)
    want = ref[f"c3/{dist}/bulyan/sample"]
    got = _np(bz.gars["bulyan"](gradients=dev, f=f))[cols]
    # stage 2 is a closest-beta mean in topk's unspecified order: 1e-6 of the summed magnitude
    # (a different stage-1 selection would move whole coordinates by O(1)).  Coordinates with an
    # exact key tie across the closest-beta boundary (a handful in 1.3M) have two valid answers:
    # they are identified by redoing stages 1-2 with the oracle on exactly those columns.
    off = np.abs(got.astype(np.float64) - want) > 2e-6 * np.maximum(np.abs(want), scale)
    exempt = np.zeros(cols.size, dtype=bool)
    if off.any():
      idx = np.flatnonzero(off)
      assert idx.size <= 50, f"C3 bulyan {dist}: {idx.size} sampled coordinates differ"
      from oracle import byzoracle as orc, corc
      D = corc.pairwise_distances(list(x))
      border, _ = orc.bulyan_order(D, f, n - f - 2)
      stage1 = orc.bulyan_stage1(orc.as_matrix([h[cols[idx]] for h in x]), border, f, n - f - 2)
      _, amb = orc.closest_mean(stage1, stage1.shape[0] - 2 * f, orc.median(stage1), return_info=True)
      exempt[idx] = amb
    parity.assert_close_scaled(got, want, scale, f"C3 bulyan {dist} [sampled columns]", rtol=2e-6, exempt=exempt)

def test_c5_brute():
  import byzantinemomentum_b200 as bz
  ref = Recorded("c5")
  n, f, d = 11, 3, 1_310_922
  for dist, nb in (("empire", 3), ("iid", 0)):
    x, nh = host_stack(n, nb, d, 15, dist)
    cols = ref.rows(f"c5/{dist}", x)
    dev = as_rows(x, nh, DEV)
    ref.exact(f"c5/{dist}/brute", _np(bz.gars["brute"](gradients=dev, f=f)), cols, f"C5 brute {dist}")
    if nb:
      assert bz.gars["brute"].influence(dev[:nh], dev[nh:], f=f) == float(ref[f"c5/{dist}/brute/influence"])

def test_c4_shard_median_trmean_n51():
  import byzantinemomentum_b200 as bz
  ref = Recorded("c4")
  n, f, d = 51, 12, 36_546_980 // 8
  x, nh = host_stack(n, 12, d, 14, "empire")
  cols = ref.rows("c4/empire", x)
  dev = as_rows(x, nh, DEV)
  ref.trmean("c4/empire/trmean", _np(bz.gars["trmean"](gradients=dev, f=f)), x, cols, "C4 shard trmean")
  ref.exact("c4/empire/median", _np(bz.gars["median"](gradients=dev, f=f)), cols, "C4 shard median")
