# coding: utf-8
"""Drop-in registration inside the UNMODIFIED reference.  The tests run against the checkout named by
$BYZ_REFERENCE and, without one, against `tests/standin/`: a stand-in written for these tests with
the reference's registry, `tools`, `experiments` and attack.py interfaces, whose stock rules answer
`check()` and `upper_bound()` as the reference did.  What the reference's `check()`, `upper_bound()`
and attack.py hold is recorded in `tests/golden/reference_checks.json`
(tests/golden/make_check_golden.py).  They run in a subprocess because importing the reference
replaces sys.stdout / sys.stderr / sys.excepthook (tools/__init__.py:215-216,246)."""

import json
import os
import pathlib
import subprocess
import sys

import pytest

import conftest

ROOT = pathlib.Path(__file__).resolve().parent.parent
STANDIN = ROOT / "tests" / "standin"
REF = conftest.reference_root() or STANDIN

def check_grid():
  """ (rule, n, f, extra keyword arguments) on which the rules' `check()` verdicts are compared. """
  return [(name, n, f, extra) for n in (1, 3, 7, 11, 25) for f in (0, 1, 2, 3, 5, 12, "x")
          for name in ("trmean", "phocas", "meamed", "krum", "bulyan", "brute", "aksel", "cge", "median", "average")
          for extra in ({}, {"m": 1}, {"m": 99}, {"mode": "n-f"}, {"mode": "zzz"})]

def test_checks_and_upper_bound_match_the_reference():
  """ The CUDA rules accept exactly the (n, f, extra) the reference's own check() accepts, and
  Multi-Krum's upper bound is the reference's (study.py:361-366 reads it). """
  import torch
  import byzantinemomentum_b200 as bz
  recorded = json.loads((conftest.GOLDEN_DIR / "reference_checks.json").read_text())
  want = {json.dumps(entry) for entry in recorded["accepted"]}
  assert len(want) > 100, len(want)
  differs = []
  for name, n, f, extra in check_grid():
    try:
      got = bz.gars[name].check(gradients=[torch.zeros(4) for _ in range(n)], f=f, **extra) is None
    except TypeError:
      got = False
    if got != (json.dumps([name, n, f, extra]) in want):
      differs.append((name, n, f, extra, got))
  assert not differs, differs[:10]
  assert bz.gars["krum"].upper_bound(25, 5, 10) == recorded["krum_upper_bound_25_5_10"]

SCRIPT = r"""
import sys
sys.path.insert(0, {root!r}); sys.path.insert(0, {ref!r})
out = sys.stdout
import aggregators
import byzantinemomentum_b200 as bz
import torch
res = []
# Route 1: the reference found our top-level `native` package and registered native-<gar>
res.append(sorted(k for k in aggregators.gars if k.startswith("native-")) == ["native-brute", "native-bulyan", "native-krum", "native-median"])
# Route 2: register through the reference's own register()
names = bz.plugin.install(aggregators)
res.append(all(name in aggregators.gars for name in names) and len(names) == 10)
rows = [torch.zeros(8) for _ in range(7)]
# the reference's wrapper validates with OUR check functions and raises ITS UserException
import tools
try:
  aggregators.gars["b200-krum"].checked(gradients=rows, f=3)
  res.append(False)
except tools.UserException:
  res.append(True)
# members the rest of the reference relies on (study.py:361-366, attack.py:822)
rule = aggregators.gars["b200-krum"]
res.append(rule.upper_bound(25, 5, 10) == aggregators.gars["krum"].upper_bound(25, 5, 10))
res.append(callable(rule.influence) and aggregators.gars["b200-median"].influence is None)
# same verdicts as the reference's own check() on a grid of (n, f, m)
same = True
for n in (1, 3, 7, 11, 25):
  g = [torch.zeros(4) for _ in range(n)]
  for f in (0, 1, 2, 3, 5, 12, "x"):
    for name in ("trmean", "phocas", "meamed", "krum", "bulyan", "brute", "aksel", "cge", "median", "average"):
      for extra in ({{}}, {{"m": 1}}, {{"m": 99}}, {{"mode": "n-f"}}, {{"mode": "zzz"}}):
        try:
          a = aggregators.gars[name].check(gradients=g, f=f, **extra)
        except TypeError:
          a = "TypeError"
        try:
          b = aggregators.gars["b200-" + name].check(gradients=g, f=f, **extra)
        except TypeError:
          b = "TypeError"
        if (a is None) != (b is None):
          same = False
          out.write(f"check differs: {{name}} n={{n}} f={{f}} {{extra}}: {{a!r}} vs {{b!r}}\n")
res.append(same)
# override: --gar krum now resolves to the CUDA rule
bz.plugin.install(aggregators, override=True, names=["krum"])
res.append(aggregators.gars["krum"].unchecked.__module__.startswith("byzantinemomentum_b200"))
# study metrics: the swap keeps the reference's function for CPU samples, same results
stock = tools.compute_avg_dev_max
before = stock([torch.arange(6.), torch.ones(6)])
previous = bz.plugin.install_tools(tools)
after = tools.compute_avg_dev_max([torch.arange(6.), torch.ones(6)])
res.append(previous is stock and tools.compute_avg_dev_max is not stock and torch.equal(before[0], after[0]) and before[1:] == after[1:]
           and tools.compute_avg_dev_max([])[0] is None)
out.write("RESULT " + " ".join(str(int(x)) for x in res) + "\n")
out.flush()
"""

def test_rules_register_inside_the_unmodified_reference(tmp_path):
  script = tmp_path / "drive.py"
  script.write_text(SCRIPT.format(root=str(ROOT), ref=str(REF)))
  proc = subprocess.run([sys.executable, str(script)], cwd=tmp_path, capture_output=True, text=True, timeout=300)
  lines = [l for l in proc.stdout.splitlines() if l.startswith("RESULT")]
  assert lines, proc.stdout[-2000:] + proc.stderr[-2000:]
  assert lines[-1] == "RESULT 1 1 1 1 1 1 1 1", proc.stdout[-3000:]

ATTACK_ARGS = ["--nb-workers", "7", "--nb-decl-byz", "1", "--nb-real-byz", "1", "--attack", "empire", "--attack-args", "factor:1.1",
               "--model", "simples-full", "--nb-steps", "2", "--device", "cpu", "--batch-size", "8", "--evaluation-delta", "0",
               "--nb-for-study", "7", "--nb-for-study-past", "2"]

def _drive(tmp_path, gar):
  cmd = [sys.executable, str(ROOT / "tools" / "drive_attack.py"), "--reference", str(REF), "--shape", "mnist", "--install-tools",
         "--", "--gar", gar] + ATTACK_ARGS
  return subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=600)

def test_unmodified_attack_py_runs_offline_with_the_rules_registered(tmp_path):
  """ SURVEY.md §8(b): the runpy recipe.  The stock rule drives two full steps (synthetic data,
  study metrics through the swapped `compute_avg_dev_max`), with every b200-<name> registered. """
  proc = _drive(tmp_path, "krum")
  assert proc.returncode == 0, proc.stdout[-3000:] + proc.stderr[-3000:]
  assert "registered: b200-average" in proc.stdout and "b200-cge" in proc.stdout
  assert "Training..." in proc.stdout

def test_cuda_rule_inside_attack_py_fails_loudly_without_a_gpu(tmp_path):
  """ No CPU fallback: selecting a CUDA rule on a box without a GPU stops attack.py with the
  library's error instead of silently computing on the host. """
  import torch
  if torch.cuda.is_available():
    pytest.skip("this box has a GPU")
  proc = _drive(tmp_path, "b200-krum")
  assert proc.returncode != 0
  assert "no CUDA device available" in proc.stdout + proc.stderr

def test_in_memory_rewrites_of_attack_py_match_their_anchors_and_compile(monkeypatch):
  """ tools/drive_attack.py --fuse-gradients / --fuse-study: every anchor is found exactly as often as
  expected in the reference's attack.py, the study block has the known digest, the rewritten source
  compiles and calls the helper; a source that differs is refused. """
  import hashlib
  import importlib.util
  spec = importlib.util.spec_from_file_location("drive_attack", ROOT / "tools" / "drive_attack.py")
  drive = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(drive)
  sha = lambda text: hashlib.sha256(text.encode()).hexdigest()
  recorded = json.loads((conftest.GOLDEN_DIR / "reference_checks.json").read_text())["attack_py"]
  expected = {drive.CLIP_AND_CLONE: 2, drive.MOMENTUM: 1, drive.STUDY_BEGIN: 1, drive.STUDY_END: 1}
  assert {sha(text): count for text, count in expected.items()} == {k: v for k, v in recorded.items() if k != "study_block"}
  assert drive.STUDY_SHA256 == recorded["study_block"]
  source = (REF / "attack.py").read_text()
  if REF == STANDIN:          # the stand-in's study block is its own text, not the reference's
    monkeypatch.setattr(drive, "STUDY_SHA256", sha(source[source.index(drive.STUDY_BEGIN):source.index(drive.STUDY_END)]))
  both = drive.rewrite(source, True, True)
  compile(both, "attack.py", "exec")
  assert both.count("__bz_rows.push(") == 2 and both.count("__bz_rows.study(") == 1
  assert "cosin_splhon = torch.dot" not in both and "cosin_splhon = torch.dot" in drive.rewrite(source, True, False)
  assert "grad_pasts.appendleft(PastGrad(sampled_grad_avg, sampled_norm_avg))" in both          # the statement after the block stays
  with pytest.raises(SystemExit):
    drive.rewrite(source.replace("cosin_hondef = ", "cosin_hondef  = "), False, True)
  with pytest.raises(SystemExit):
    drive.rewrite(source.replace("grad.clone().detach_()", "grad.clone()"), True, False)
