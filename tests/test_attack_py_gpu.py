# coding: utf-8
"""The drop-in INSIDE the unmodified reference, on the GPU (VERDICT r1 weak #1, SURVEY §8 a16/b).

`tools/drive_attack.py` executes the reference's own `attack.py` (from the checkout named by
$BYZ_REFERENCE: skipped without one; nothing of it is edited) with `runpy`, synthetic batches in
place of the dataset download, and the CUDA rules registered through the reference's own
`aggregators.register` (`b200-<name>`) and through the `native.<rule>.aggregate` hook it probes
(`native-<name>`).  Everything of attack.py:799-827 then runs against the CUDA rules on cuda:0:
the attack's line search (`attacks/identical.py:68-77`: GAR called once per evaluated factor, the
result modified IN PLACE by `aggregated.sub_(grad_avg)`), `defense.checked(...)`, `influence`
right after it, the `--device-gar` hops (attack.py:811-815,824-827), the study metrics
(`tools.compute_avg_dev_max` swapped for the one-pass kernel).

Parity: the same command with the STOCK rule (the reference's own PyTorch code, same device, same
seed, stock study metrics) must log the same accept ratios and the same study columns up to float
noise.  All runs share one process (`--batch`): one interpreter start, one CUDA context.
"""

import json
import math
import pathlib
import subprocess
import sys

import pytest

import conftest

ROOT = pathlib.Path(__file__).resolve().parent.parent
pytestmark = [pytest.mark.gpu, conftest.needs_reference]

STEPS = 3
EVALS = 4

def _args(out, gar, n, f, attack_args, device="cuda:0", device_gar="same", model="simples-full", dataset="mnist", momentum_at="update"):
  return ["--gar", gar, "--nb-workers", str(n), "--nb-decl-byz", str(f), "--nb-real-byz", str(f), "--attack", "empire",
          "--attack-args", *attack_args, "--model", model, "--dataset", dataset, "--nb-steps", str(STEPS), "--device", device,
          "--device-gar", device_gar, "--batch-size", "8", "--evaluation-delta", "0", "--nb-for-study", str(n - f),
          "--nb-for-study-past", "2", "--seed", "7", "--momentum-at", momentum_at, "--result-directory", str(out)]

# tag -> (our rule, the stock rule it replaces, n, f, extra keyword arguments of _args)
LINE_SEARCH = {
  "b200-krum": ("krum", 11, 3), "native-krum": ("krum", 11, 3), "native-bulyan": ("bulyan", 11, 2), "b200-bulyan": ("bulyan", 15, 3),
  "b200-trmean": ("trmean", 11, 4), "native-median": ("median", 11, 4), "b200-phocas": ("phocas", 11, 4), "b200-meamed": ("meamed", 11, 4),
  "native-brute": ("brute", 9, 2), "b200-aksel": ("aksel", 11, 3), "b200-cge": ("cge", 11, 3), "b200-average": ("average", 11, 3),
}
OTHER = {
  # `--device cpu --device-gar cuda:0` (attack.py:811-815,824-827)
  "hop": ("b200-krum", "krum", 11, 3, dict(attack_args=["factor:1.1"], device="cpu", device_gar="cuda:0")),
  # `--device cpu`: the rule stages the host rows itself and returns a host tensor
  "cpu": ("b200-trmean", "trmean", 11, 4, dict(attack_args=["factor:1.1"], device="cpu")),
  # worker-side momentum (attack.py:799-804: the GAR receives the momentum buffers, updated in
  # place every step) on CIFAR-10 `empire-cnn` (d = 1,310,922), n = 25, f = 5: BASELINE configs[2]
  "c3-krum": ("b200-krum", "krum", 25, 5, dict(attack_args=["factor:1.1"], model="empire-cnn", dataset="cifar10", momentum_at="worker")),
  "c3-bulyan": ("b200-bulyan", "bulyan", 25, 5, dict(attack_args=["factor:1.1"], model="empire-cnn", dataset="cifar10", momentum_at="worker")),
}
# gradient production fused into GradientStack.push (tools/drive_attack.py --fuse-gradients: attack.py's
# clip / clone / momentum statements swapped IN MEMORY): tag -> (rule, n, f, momentum placement, clip)
FUSED = {
  "fuse-update": ("b200-krum", 11, 3, "update", "2"),
  "fuse-worker": ("b200-krum", 11, 3, "worker", "2"),
  "fuse-server": ("b200-trmean", 11, 3, "server", "0.5"),
  "fuse-noclip": ("b200-median", 11, 3, "worker", None),
}
# the study block (attack.py:846-866) as ONE engine.study_step call (tools/drive_attack.py --fuse-study):
# tag -> (rule, n, f, real Byzantine workers, momentum placement)
STUDY = {
  "study-krum": ("b200-krum", 11, 3, 3, "update"),
  "study-bulyan-worker": ("b200-bulyan", 11, 2, 2, "worker"),
  "study-trmean-server": ("b200-trmean", 11, 4, 4, "server"),
  "study-no-attack": ("b200-median", 11, 4, 0, "update"),        # no attack gradients: NaN columns (attack.py:855-859)
}
INFLUENCE = ("krum", "brute", "aksel", "cge", "average")

@pytest.fixture(scope="module")
def runs(tmp_path_factory):
  tmp = tmp_path_factory.mktemp("attack")
  jobs = []
  for ours, (stock, n, f) in LINE_SEARCH.items():
    jobs.append(dict(tag=ours, install_tools=True, args=_args(tmp / ours, ours, n, f, [f"factor:-{EVALS}"])))
    jobs.append(dict(tag=ours + "/stock", install_tools=False, args=_args(tmp / (ours + "-stock"), stock, n, f, [f"factor:-{EVALS}"])))
  for tag, (ours, stock, n, f, kw) in OTHER.items():
    jobs.append(dict(tag=tag, install_tools=True, args=_args(tmp / tag, ours, n, f, **kw)))
    jobs.append(dict(tag=tag + "/stock", install_tools=False, args=_args(tmp / (tag + "-stock"), stock, n, f, **kw)))
  for tag, (gar, n, f, where, clip) in FUSED.items():
    extra = [] if clip is None else ["--gradient-clip", clip]
    jobs.append(dict(tag=tag, install_tools=True, fuse_gradients=True, args=_args(tmp / tag, gar, n, f, ["factor:1.1"], momentum_at=where)[:-2] + extra + ["--result-directory", str(tmp / tag)]))
    jobs.append(dict(tag=tag + "/stock", install_tools=True, fuse_gradients=False, args=_args(tmp / (tag + "-stock"), gar, n, f, ["factor:1.1"], momentum_at=where)[:-2] + extra + ["--result-directory", str(tmp / (tag + "-stock"))]))
  for tag, (gar, n, f, real, where) in STUDY.items():
    for suffix, fused in (("", True), ("/stock", False)):
      out = tmp / (tag + ("" if fused else "-stock"))
      argv = _args(out, gar, n, f, ["factor:1.1"], momentum_at=where)
      argv[argv.index("--nb-real-byz") + 1] = str(real)
      argv[argv.index("--nb-for-study") + 1] = str(n - real)
      jobs.append(dict(tag=tag + suffix, install_tools=False, fuse_study=fused, args=argv))
  batch = tmp / "batch.json"
  batch.write_text(json.dumps(jobs))
  cmd = [sys.executable, str(ROOT / "tools" / "drive_attack.py"), "--count-calls", "--install-tools", "--batch", str(batch)]
  proc = subprocess.run(cmd, cwd=tmp, capture_output=True, text=True, timeout=1500)
  assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
  result = {}
  for job in jobs:
    result[job["tag"]] = dict(ok=False, calls={}, rows=None, dir=pathlib.Path(job["args"][-1]), pushes=0, studies=0)
  for line in proc.stdout.splitlines():
    if line.startswith("run-ok "):
      result[line.split()[1]]["ok"] = True
    elif line.startswith("run-failed "):
      result[line.split()[1]]["error"] = line
    elif line.startswith("fused-pushes "):
      result[line.split()[1]]["pushes"] = int(line.split()[2])
    elif line.startswith("fused-studies "):
      result[line.split()[1]]["studies"] = int(line.split()[2])
    elif line.startswith("gar-calls "):
      _, tag, name, calls, infl = line.split()
      result[tag]["calls"][name] = (int(calls), int(infl))
  for tag, entry in result.items():
    study = entry["dir"] / "study"
    if study.exists():
      entry["rows"] = [l.split("\t") for l in study.read_text().strip().splitlines()[1:]]
  result["__stdout__"] = proc.stdout
  return result

def _close(a, b, rel=2e-4):
  a, b = float(a), float(b)
  if math.isnan(a) or math.isnan(b):
    return math.isnan(a) and math.isnan(b)
  return abs(a - b) <= rel * max(abs(a), abs(b)) + 2e-6

def _same_study(mine, theirs, exact_ratio, rel=2e-4, ratio_nan=False):
  assert len(mine) == STEPS and len(theirs) == STEPS
  for step, (a_row, b_row) in enumerate(zip(mine, theirs)):
    assert a_row[0] == b_row[0]
    if exact_ratio:      # a count of selected attack rows over a count: exact
      assert float(a_row[-1]) == float(b_row[-1]), (step, a_row[-1], b_row[-1])
    elif ratio_nan:
      assert math.isnan(float(a_row[-1]))
    else:
      assert math.isnan(float(a_row[-1])) and math.isnan(float(b_row[-1]))
    for col, (a, b) in enumerate(zip(a_row[2:-1], b_row[2:-1])):
      assert _close(a, b, rel), (step, col + 2, a, b)

@pytest.mark.parametrize("ours", sorted(LINE_SEARCH))
def test_attack_py_with_line_search_matches_the_stock_rule(runs, ours):
  """ empire with factor:-4 = a 4-evaluation line search per step -> 5 GAR calls per step, the
  fifth followed by influence() (attack.py:821-822). """
  stock = LINE_SEARCH[ours][0]
  mine, theirs = runs[ours], runs[ours + "/stock"]
  assert mine["ok"], mine.get("error", runs["__stdout__"][-3000:])
  assert theirs["ok"], theirs.get("error")
  # the reference registers its native-<name> rules WITHOUT influence (krum.py:159-166): nan there
  has_influence = stock in INFLUENCE and not ours.startswith("native-")
  assert mine["calls"][ours] == (STEPS * (EVALS + 1), STEPS if has_influence else 0), mine["calls"]
  assert theirs["calls"][stock][0] == STEPS * (EVALS + 1)
  _same_study(mine["rows"], theirs["rows"], has_influence, ratio_nan=not has_influence)

@pytest.mark.parametrize("tag", sorted(OTHER))
def test_attack_py_device_hops_momentum_and_cifar_shape(runs, tag):
  ours, stock = OTHER[tag][0], OTHER[tag][1]
  mine, theirs = runs[tag], runs[tag + "/stock"]
  assert mine["ok"], mine.get("error", runs["__stdout__"][-3000:])
  assert theirs["ok"], theirs.get("error")
  assert mine["calls"][ours][0] == STEPS
  _same_study(mine["rows"], theirs["rows"], stock in INFLUENCE, rel=5e-4)

@pytest.mark.parametrize("tag", sorted(FUSED))
def test_attack_py_with_fused_gradient_production(runs, tag):
  """ SURVEY §8(f) row 2: attack.py:775-780 / 790-795 (clip + clone) and :799-808 (momentum placement)
  executed as `GradientStack.push` — one kernel per worker writing rows of one [n, d] buffer — inside
  the otherwise unmodified attack.py; the run must log what the unfused run logs. """
  gar, n, f, where, clip = FUSED[tag]
  mine, theirs = runs[tag], runs[tag + "/stock"]
  assert mine["ok"], mine.get("error", runs["__stdout__"][-3000:])
  assert theirs["ok"], theirs.get("error")
  assert mine["pushes"] == STEPS * (n - f) and theirs["pushes"] == 0        # nb_for_study = nb_honests = n - f gradients per step
  _same_study(mine["rows"], theirs["rows"], gar[5:] in INFLUENCE, rel=5e-4)

@pytest.mark.parametrize("tag", sorted(STUDY))
def test_attack_py_with_fused_study_step(runs, tag):
  """ SURVEY §8(f) row 3: attack.py:846-866 (three compute_avg_dev_max, the defense norm, six cosines, the
  past cosine, the curvature: 9 + nb_for_study_past host syncs plus those of the stock compute_avg_dev_max)
  executed as ONE `engine.study_step` call with one host read, inside the otherwise unmodified attack.py
  against the run with the STOCK study code: the same study file up to float rounding. """
  gar, n, f, real, where = STUDY[tag]
  mine, theirs = runs[tag], runs[tag + "/stock"]
  assert mine["ok"], mine.get("error", runs["__stdout__"][-3000:])
  assert theirs["ok"], theirs.get("error")
  assert mine["studies"] == STEPS and theirs["studies"] == 0
  _same_study(mine["rows"], theirs["rows"], real > 0 and gar[5:] in INFLUENCE, rel=5e-4)
  if real == 0:        # the attack columns are NaN in both runs (checked equal above): make sure they are there
    assert any(math.isnan(float(x)) for x in mine["rows"][0][2:-1])
