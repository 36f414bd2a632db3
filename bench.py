#!/usr/bin/env python3
# coding: utf-8
"""bench.py — throughput of the aggregation hot path on synthetic [n, d] gradients.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--gar trmean --nb-workers 25 --nb-byz 10 --dim 1310922] [--no-sweep]
                    [--dump-outputs DIR]

A "step" is ONE aggregation call over one stack of n worker gradients (fp32, length d per
GPU).  Default workload = BASELINE.json configs[1]: trimmed mean, n=25, f=10, d=1,310,922
(CIFAR-10 `empire-cnn`), the configuration the headline metric is quoted on.
N > 1 (launched by torchrun, one rank per GPU, NCCL): the d axis is sharded, every rank
aggregates its own [n, d] shard; coordinate-wise rules need no collective, distance-based
rules all-gather their n x n partial-distance blocks (byzantinemomentum_b200.sharded).
Per-GPU work is fixed as N grows -> "scaling": "weak"; `value` = N*d / step time.

One JSON line is printed by rank 0 (see the driver contract in the task statement):
  value       params/s with inputs resident in HBM, device-timed (CUDA events, max over ranks)
  roofline    dominant kernel: algorithmic bytes / average per-launch duration vs the measured
              HBM peak of MEASURED_PEAKS.json
  e2e         the same metric through the reference-facing call `gars[gar](gradients=<host
              tensors>, f=f)`: pinned host rows -> H2D -> kernel -> D2H of the result, per step
  cpu_baseline  the UNMODIFIED reference's `aggregators.gars[gar].unchecked` on CPU tensors, on the host
                cores (the checkout named by $BYZ_REFERENCE; without one, its port oracle/refcost.py)
  sweep       (N=1) kernel time / GB/s / roofline fraction of the other rules and sizes
`--impl reference` times the reference's CPU aggregation alone, on the same workload.
`--steps K` is the number of timed steps of every timed loop: the headline region, the plugin and e2e
calls and the sharded block (the sweep keeps the median of 7-15 samples per point).
`--dump-outputs DIR` writes what the last timed step returned as DIR/aggregate.npy (fp32; with N > 1
each rank writes DIR/aggregate_rank<r>.npy).  The inputs are seeded, so two builds run with the same
arguments can be compared output for output.  Above 60 MB in all, a fixed seeded sample of the
elements is written instead, with their positions in DIR/<name>_index.npy (fp64).
"""

import argparse
import json
import math
import os
import pathlib
import sys
import threading
import time

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True     # the tree may be read-only: leave nothing in it

DUMP_BYTES = 60_000_000         # --dump-outputs: under 64 MB with the .npy headers

L2_BYTES = 126 * 1024 * 1024
FALLBACK_HBM_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md, used only without MEASURED_PEAKS.json

# kernels of libbyzagg launched per aggregation call (single device)
LAUNCHES = dict(average=1, median=1, trmean=1, phocas=1, meamed=1, krum=2, bulyan=2, brute=2, aksel=3, cge=2)

def algorithmic_bytes(gar, n, f, d, m=None):
  """ SURVEY.md §8(d): bytes one call must move, per GAR (no credit for aliases or L2 hits). """
  if gar in ("average", "median", "trmean", "phocas", "meamed"):
    units = n + 1
  elif gar in ("krum", "bulyan"):
    units = n + (m if m is not None else n - f - 2) + 1
  elif gar in ("brute", "cge"):
    units = n + (n - f) + 1
  elif gar == "aksel":
    units = n + (n + 1) // 2 + 1
  else:
    raise KeyError(gar)
  return units * d * 4

def default_f(gar, n, f):
  if gar in ("bulyan",):
    return min(f, (n - 3) // 4)
  if gar in ("krum",):
    return min(f, (n - 3) // 2)
  return f

# ---------------------------------------------------------------------------- #
# Clock sampling (NVML), during the timed regions

class ClockSampler:
  REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
             0x80: "hw_power_brake", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}
  def __init__(self, index):
    self.samples, self.reasons, self.max_mhz = [], set(), None
    self._stop = threading.Event()
    self._thread = None
    try:
      import pynvml
      pynvml.nvmlInit()
      self.nv = pynvml
      self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
      self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
    except Exception:
      self.nv = None
  def _loop(self):
    nv = self.nv
    while not self._stop.is_set():
      try:
        self.samples.append(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
        mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
          else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        for bit, name in self.REASONS.items():
          if mask & bit:
            self.reasons.add(name)
      except Exception:
        pass
      self._stop.wait(0.005)
  def __enter__(self):
    if self.nv is not None:
      self._thread = threading.Thread(target=self._loop, daemon=True)
      self._thread.start()
    return self
  def __exit__(self, *exc):
    self._stop.set()
    if self._thread is not None:
      self._thread.join()
  def summary(self):
    if not self.samples:
      return dict(sm_mhz=None, sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons), samples=0)
    s = sorted(self.samples)
    return dict(sm_mhz=s[len(s) // 2], sm_max_mhz=self.max_mhz, reasons=sorted(self.reasons), samples=len(s))

# ---------------------------------------------------------------------------- #

def make_rows(torch, n, d, device, seed, sets):
  """ `sets` independent stacks of n rows ~ N(0, 1) (distribution A of SURVEY.md §8(d)). """
  gen = torch.Generator(device=device).manual_seed(seed)
  return [[torch.randn(d, device=device, generator=gen) for _ in range(n)] for _ in range(sets)]

EXCHANGE = "auto"

def call_device(bz, sharded, gar, rows, f, world):
  """ One aggregation of device-resident rows (the step of the timed region). """
  if world > 1:
    if EXCHANGE == "p2p":
      return sharded.aggregate_p2p(gar, rows, f=f)
    return sharded.aggregate(gar, rows, f=f)
  return bz.gars[gar].unchecked(gradients=rows, f=f)

def time_steps(torch, fn, steps, pairs=True):
  """ K steps on the current stream between two CUDA events; with `pairs`, also one event pair
  around every step (per-launch durations).  Returns (total_ms, per_step_ms list or None, what
  the last step returned). """
  if not pairs:
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for k in range(steps):
      out = fn(k)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), None, out
  ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
  for k in range(steps):
    ev[k][0].record()
    out = fn(k)
    ev[k][1].record()
  torch.cuda.synchronize()
  total = ev[0][0].elapsed_time(ev[-1][1])
  return total, [a.elapsed_time(b) for a, b in ev], out

def dump_outputs(directory, outputs):
  """ Each array of `outputs` (name -> NumPy array) as <directory>/<name>.npy, DUMP_BYTES in all at most:
  an array over its share is replaced by a sample of its elements at fixed seeded positions, which go
  to <name>_index.npy. """
  import numpy as np
  os.makedirs(directory, exist_ok=True)
  share = DUMP_BYTES // max(len(outputs), 1)
  for name, value in outputs.items():
    value = np.ascontiguousarray(value).reshape(-1)
    if value.nbytes > share:
      index = np.sort(np.random.default_rng(0).choice(value.size, share // (value.itemsize + 8), replace=False))
      np.save(os.path.join(directory, name + "_index.npy"), index.astype(np.float64))
      value = value[index]
    np.save(os.path.join(directory, name + ".npy"), value)

def peak_hbm():
  path = ROOT / "MEASURED_PEAKS.json"
  try:
    return float(json.loads(path.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
  except Exception:
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"

def recorded_traffic(gar, n, f, d):
  """ dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture. """
  try:
    table = json.loads((ROOT / "profiles" / "traffic.json").read_text())
    return table.get(f"{gar}:n{n}:f{f}:d{d}")
  except Exception:
    return None

def cpu_info():
  model = "unknown"
  try:
    for line in pathlib.Path("/proc/cpuinfo").read_text().splitlines():
      if line.startswith("model name"):
        model = line.split(":", 1)[1].strip()
        break
  except OSError:
    pass
  try:
    allowed = len(os.sched_getaffinity(0))
  except AttributeError:
    allowed = os.cpu_count() or 1
  return dict(cpu_model=model, cpus_online=os.cpu_count() or 1, cpus_allowed=allowed)

def reference_callable(gar):
  """ (fn(rows, f), kind, path): the UNMODIFIED reference's `aggregators.gars[gar].unchecked`
  (BASELINE.md §4.2; the checkout named by $BYZ_REFERENCE) — nothing of this repository is on
  that path — or, only when no reference checkout is given, the port of its
  ATen operator sequence (oracle/refcost.py). """
  from oracle import reference
  root, aggregators = reference.load()
  if aggregators is not None and gar in aggregators.gars:
    rule = aggregators.gars[gar].unchecked
    return (lambda rows, f: rule(gradients=rows, f=f)), "reference", f"{reference.describe()}: aggregators.gars[{gar!r}].unchecked(gradients=<cpu rows>, f=f)"
  from oracle import refcost
  return (lambda rows, f: refcost.run(gar, rows, f=f)), "port", "oracle/refcost.py: the reference's ATen operator sequence on CPU tensors (no reference checkout found)"

def cpu_reference(torch, gar, n, f, d, seed, budget_s, repeats):
  """ The reference's CPU aggregation on the host cores, bounded: shrinks d so that `repeats`
  calls fit `budget_s`. """
  run, kind, path = reference_callable(gar)
  gen = torch.Generator().manual_seed(seed)
  probe_d = min(d, 65536)
  rows = [torch.randn(probe_d, generator=gen) for _ in range(n)]
  # "all the host threads it can use": os.cpu_count() may exceed what the container is allowed to
  # run, which makes ATen's parallel loops thrash; probe a few thread counts, keep the fastest
  info = cpu_info()
  allowed = info["cpus_allowed"]
  candidates = sorted({torch.get_num_threads(), allowed, os.cpu_count() or 1, 8, 16, 32} & set(range(1, allowed + 1)) | {min(allowed, 8)})
  best_threads, per_elem = None, None
  for threads in candidates:
    torch.set_num_threads(threads)
    run(rows, f)
    t0 = time.perf_counter()
    run(rows, f)
    cost = (time.perf_counter() - t0) / probe_d
    if per_elem is None or cost < per_elem:
      best_threads, per_elem = threads, cost
  torch.set_num_threads(best_threads)
  sample_d = int(min(d, max(4096, budget_s / max(repeats, 1) / max(per_elem, 1e-12))))
  rows = [torch.randn(sample_d, generator=gen) for _ in range(n)]
  run(rows, f)  # warm
  times = []
  for _ in range(repeats):
    t0 = time.perf_counter()
    run(rows, f)
    times.append(time.perf_counter() - t0)
  return dict(times=times, sample_d=sample_d, threads=torch.get_num_threads(), kind=kind, path=path, torch=torch.__version__, **info)

def make_config(gar, n, f, d, world):
  """ The workload description, identical in both arms (the driver compares the dicts). """
  return dict(workload=f"{gar} GAR, n={n} f={f}, d={d} per GPU (BASELINE.json configs[1]: CIFAR-10 empire-cnn shape)",
              gar=gar, n=n, f=f, d=d, parallelism=f"d-sharded x{world}" if world > 1 else "single GPU",
              l2="GPU arm: inputs rotate over independent [n, d] stacks totalling more than 3x the 126 MB L2; CPU arm: not applicable")

# ---------------------------------------------------------------------------- #

def run_reference(args):
  import torch
  rank = int(os.environ.get("RANK", "0"))
  world = int(os.environ.get("WORLD_SIZE", "1"))
  if rank != 0:
    return
  f = default_f(args.gar, args.n, args.f)
  res = cpu_reference(torch, args.gar, args.n, f, args.d, 4321, budget_s=120.0, repeats=args.steps + args.warmup)
  times = res["times"][args.warmup:] or res["times"]
  ms = 1e3 * sum(times) / len(times)
  value = res["sample_d"] / (ms * 1e-3)
  sample = f"{args.gar} n={args.n} f={f} on d={res['sample_d']} of {args.d} columns per step, {len(times)} timed steps"
  line = dict(impl="reference", metric="aggregated-params/sec", value=value, unit="params/s", n_gpus=args.gpus, steps=len(times),
              warmup=args.warmup, ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
              config=make_config(args.gar, args.n, f, args.d, world),
              cpu_baseline=dict(value=value, unit="params/s", cores=res["threads"], kind=res["kind"], sample=sample, path=res["path"],
                                cpu_model=res["cpu_model"], cpus_allowed=res["cpus_allowed"], torch=res["torch"]),
              e2e=dict(value=value, unit="params/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
  print(json.dumps(line), flush=True)

def timed_max_over_ranks(torch, dist, device, fn, steps, warmup=5):
  """ µs per step of `fn(k)`: `steps` calls between two CUDA events on the current stream after a
  barrier + synchronize, the MAX over the ranks (every rank issues the same collectives). """
  for k in range(warmup):
    fn(k)
  if dist is not None:
    dist.barrier()
  torch.cuda.synchronize()
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record()
  for k in range(steps):
    fn(k)
  b.record()
  torch.cuda.synchronize()
  ms = a.elapsed_time(b)
  if dist is not None:
    t = torch.tensor([ms], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
  return ms / steps * 1e3

def sharded_block(torch, dist, bz, sharded, device, world, rank, peak, steps):
  """ The multi-GPU path BASELINE.json's north_star names (SURVEY §8(e)), timed on the device:
    collective  Multi-Krum + Bulyan at C3 (n = 25, f = 5, d = 1,310,922 PER GPU: weak scaling)
                through the prepared sharded call: with the NCCL all-gather of the R n x n blocks
                ("nccl"), with the blocks read in place over NVLink peer memory by the selection
                kernel after a device barrier ("p2p"), and with the exchange INSIDE the distance
                pass ("fused": bz_krum_peers, two launches per step); beside the same rule on one GPU
                without any exchange (engine.Plan) in the same process;
    c4_strong   median + trimmed mean at C4 (n = 51, f = 12, d = 36,546,980 TOTAL, split over the
                N ranks: strong scaling; no collective on this path). """
  out = dict(world=world)
  # ---- collective path, weak scaling --------------------------------------------------------------
  n, f, d = 25, 5, 1_310_922
  sets = 4                                           # 4 x 131 MB > 3 x L2
  gen = torch.Generator(device=device).manual_seed(77 + rank)
  stacks = [[torch.randn(d, device=device, generator=gen) for _ in range(n)] for _ in range(sets)]
  rows = []
  for gar in ("krum", "bulyan"):
    rec = dict(gar=gar, n=n, f=f, d_per_gpu=d, steps=steps)
    local = [bz.Plan(gar, st, f=f) for st in stacks]
    rec["single_gpu_us"] = timed_max_over_ranks(torch, dist, device, lambda k: local[k % sets](), steps)
    for exchange in (("nccl", "p2p", "fused") if world > 1 else ("nccl",)):
      try:
        plans = [sharded.ShardedPlan(gar, st, f=f, exchange=exchange) for st in stacks]
        rec[exchange + "_us"] = timed_max_over_ranks(torch, dist, device, lambda k: plans[k % sets](), steps)
        rec[exchange + "_vs_single"] = rec[exchange + "_us"] / rec["single_gpu_us"]
        del plans
      except Exception as err:
        rec[exchange + "_error"] = f"{type(err).__name__}: {err}"[:200]
    alg = (n + (n - f - 2) + 1) * d * 4
    best = min(rec.get("nccl_us", math.inf), rec.get("p2p_us", math.inf), rec.get("fused_us", math.inf))
    if math.isfinite(best):
      rec["aggregate_gbs"] = world * alg / (best * 1e-6) / 1e9
      rec["hbm_frac_per_gpu"] = alg / (best * 1e-6) / 1e9 / peak
    rows.append(rec)
    del local
  # ---- closing the loop (SURVEY §8(f) row 4): SGD step on the shard + one all-gather of the parameters ----
  try:
    params = torch.zeros(world * d, device=device)
    shard = torch.randn(d, device=device, generator=gen)
    upd_us = timed_max_over_ranks(torch, dist, device, lambda k: sharded.apply_update(params, shard, 0.01, weight_decay=1e-4), steps)
    out["model_update"] = dict(what="sharded.apply_update: p -= lr (g + w p) on this rank's d columns, then ONE all-gather of the parameters (experiments/model.py:368-380 for a d-sharded trainer)",
                               d_total=world * d, us_per_step=upd_us, allgather_bytes_per_rank=d * 4)
    del params, shard
  except Exception as err:
    out["model_update"] = dict(error=f"{type(err).__name__}: {err}"[:200])
  out["collective"] = dict(what="weak scaling: n=25 f=5 d=1,310,922 per GPU; one exchange of R blocks of n*n fp64 per step; us per step, max over ranks",
                           exchange_bytes_per_rank=n * n * 8, rules=rows)
  del stacks
  torch.cuda.empty_cache()
  # ---- C4, strong scaling ------------------------------------------------------------------------
  n, f, total = 51, 12, 36_546_980
  per = (total + world - 1) // world
  d = min(per, total - rank * per)
  sets = max(1, min(3, math.ceil(3 * L2_BYTES / (n * d * 4))))
  gen = torch.Generator(device=device).manual_seed(177 + rank)
  stacks = [[torch.randn(d, device=device, generator=gen) for _ in range(n)] for _ in range(sets)]
  rows = []
  for gar in ("median", "trmean"):
    plans = [sharded.ShardedPlan(gar, st, f=f) for st in stacks]
    us = timed_max_over_ranks(torch, dist, device, lambda k: plans[k % sets](), steps, warmup=3)
    alg = (n + 1) * total * 4
    rows.append(dict(gar=gar, n=n, f=f, d_total=total, d_this_rank=d, us_per_step=us, params_per_s=total / (us * 1e-6),
                     aggregate_gbs=alg / (us * 1e-6) / 1e9, hbm_frac_per_gpu=alg / world / (us * 1e-6) / 1e9 / peak))
    del plans
  out["c4_strong"] = dict(what="strong scaling: n=51 f=12 d=36,546,980 split over the ranks (BASELINE.json configs[3]); us per step, max over ranks; speed-up = the N=1 line of the same run series / this",
                          rules=rows)
  del stacks
  torch.cuda.empty_cache()
  return out

def h2d_probe(torch, device, n, d):
  """ Measured host->device rate on this box for the step's input size, outside the library: ONE contiguous
  pinned copy of n*d*4 bytes, and n separate pinned rows of d*4 bytes on one stream (on some boxes the
  single large copy is the slower of the two).  The faster one is the PCIe floor of the e2e leg. """
  try:
    nbytes = n * d * 4
    host = torch.empty(n * d, dtype=torch.float32).pin_memory()
    rows = [torch.empty(d, dtype=torch.float32).pin_memory() for _ in range(n)]
    dst = torch.empty(n * d, dtype=torch.float32, device=device)
    def rate(fn):
      for _ in range(2):
        fn()
      torch.cuda.synchronize()
      a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a.record()
      for _ in range(5):
        fn()
      b.record()
      torch.cuda.synchronize()
      return a.elapsed_time(b) / 5
    ms_one = rate(lambda: dst.copy_(host, non_blocking=True))
    ms_rows = rate(lambda: [dst[i * d:(i + 1) * d].copy_(r, non_blocking=True) for i, r in enumerate(rows)])
    best = min(ms_one, ms_rows)
    return dict(contiguous_gbs=nbytes / (ms_one * 1e-3) / 1e9, rows_gbs=nbytes / (ms_rows * 1e-3) / 1e9, ms=best, bytes=nbytes)
  except Exception as err:
    return dict(error=str(err)[:120])

def run_b200(args):
  import torch
  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  if not torch.cuda.is_available():
    raise SystemExit("bench.py needs a CUDA device (the CUDA path has no CPU fallback); use --impl reference for the CPU arm")
  torch.cuda.set_device(local)
  device = torch.device("cuda", local)
  dist = None
  if world > 1:
    import torch.distributed as dist
    import datetime
    dist.init_process_group("nccl", device_id=device, timeout=datetime.timedelta(seconds=120))
  import byzantinemomentum_b200 as bz
  from byzantinemomentum_b200 import sharded
  bz._lib.lib()
  gar, n, d = args.gar, args.n, args.d
  f = default_f(gar, n, args.f)
  set_bytes = n * d * 4
  sets = max(1, min(8, math.ceil(3 * L2_BYTES / set_bytes)))
  inputs = make_rows(torch, n, d, device, 1234 + rank, sets)
  def barrier():
    if dist is not None:
      dist.barrier()
    torch.cuda.synchronize()
  # The timed step is the prepared call (byzantinemomentum_b200.Plan: the public API for steady
  # state loops): the arguments are resolved once per input stack, each step is one C-ABI call.
  # Distance-based rules under N > 1 need the all-gather and go through sharded.aggregate.
  if world == 1 or gar in sharded.COORDINATE_WISE:
    plans = [bz.Plan(gar, rows, f=f) for rows in inputs]
    step = lambda k: plans[k % sets]()
    api = f"byzantinemomentum_b200.Plan({gar!r}, rows, f={f})()"
  else:
    splans = [sharded.ShardedPlan(gar, rows, f=f, exchange=EXCHANGE) for rows in inputs]
    step = lambda k: splans[k % sets]()
    api = f"byzantinemomentum_b200.sharded.ShardedPlan({gar!r}, rows, f={f}, exchange={splans[0].exchange!r})()"
  for k in range(max(args.warmup, 3)):
    step(k)
  barrier()
  with ClockSampler(local) as clocks:
    total_ms, _, last = time_steps(torch, step, args.steps, pairs=False)     # THE timed region: K steps, two events
    if args.dump_outputs:
      dumped = last.detach().cpu().numpy()
    barrier()
    _, per_step, _ = time_steps(torch, step, args.steps, pairs=True)      # second pass: per-launch durations
    barrier()
    # keep the sampler alive a little when the region is very short
    # (a FIXED number of extra steps: every rank must issue the same collectives)
    # NVML queries take tens of milliseconds each: keep the same load running for ~0.4 s more
    if total_ms < 400:
      extra = int(min(20000, max(10, 400.0 / max(total_ms / args.steps, 1e-3))))
      if dist is not None:
        count = torch.tensor([extra], device=device, dtype=torch.int64)
        dist.broadcast(count, src=0)
        extra = int(count.item())
      for k in range(extra):
        step(k)
      torch.cuda.synchronize()
  if dist is not None:
    t = torch.tensor([total_ms], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
  ms_per_step = total_ms / args.steps
  value = world * d / (ms_per_step * 1e-3)
  # Average duration of one launch of the dominant kernel over the timed region: the launch-to-
  # launch period (total / K, conservative: it includes the inter-launch gap); the mean of the
  # per-step event pairs is kept beside it (each pair adds ~3-5 us of event overhead).
  event_pair_ms = sum(per_step) / len(per_step)
  kernel_ms = min(event_pair_ms, ms_per_step) if LAUNCHES[gar] == 1 and (world == 1 or gar in sharded.COORDINATE_WISE) else event_pair_ms
  peak, peak_src = peak_hbm()
  alg = algorithmic_bytes(gar, n, f, d)
  achieved = alg / (kernel_ms * 1e-3) / 1e9
  roofline = dict(bound="hbm", achieved=achieved, peak=peak, unit="GB/s", frac=achieved / peak, traffic=recorded_traffic(gar, n, f, d),
                  kernel=("k1_sorted" if gar in ("trmean", "phocas", "meamed") else "k1_median" if gar == "median" else "k3_average" if gar == "average" else "k2_pairdist"),
                  algorithmic_bytes=alg, read_only_frac=(n * d * 4) / (kernel_ms * 1e-3) / 1e9 / peak, kernel_ms=kernel_ms,
                  event_pair_ms=event_pair_ms, peak_source=peak_src)

  # ---- the reference-facing plugin call on the same device-resident stacks (host-side cost shows) ----
  plugin_step = lambda k: bz.gars[gar].unchecked(gradients=inputs[k % sets], f=f)
  if world == 1:
    for k in range(3):
      plugin_step(k)
    barrier()
    plugin_total, _, _ = time_steps(torch, plugin_step, args.steps)
    plugin_ms = plugin_total / args.steps
  else:
    plugin_ms = None

  # ---- end to end through the reference-facing call with HOST buffers ---------------------------
  e2e_steps = args.steps
  host_sets = 2
  # pinned host buffers, allocated while bound to the GPU-local CPUs (first touch puts the pages on
  # the GPU's NUMA node: a copy from the other socket runs at a fraction of the PCIe rate)
  with bz.hostmem.gpu_local_cpus(device.index) as numa_local:
    host = [[torch.randn(d, generator=torch.Generator().manual_seed(99 + 7 * s + r)).pin_memory() for r in range(n)] for s in range(host_sets)]
  def e2e_step(k):
    out = bz.gars[gar].unchecked(gradients=host[k % host_sets], f=f)
    assert out.device.type == "cpu"
    return out
  for k in range(12):             # the engine measures its host->device candidates during the first calls (engine._HostPath)
    e2e_step(k)
  barrier()
  e2e_total, e2e_each, _ = time_steps(torch, e2e_step, e2e_steps)
  if dist is not None:
    t = torch.tensor([e2e_total], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_total = float(t.item())
  e2e_ms = e2e_total / e2e_steps
  probe = h2d_probe(torch, device, n, d)
  e2e = dict(value=world * d / (e2e_ms * 1e-3), unit="params/s", h2d_bytes_per_step=n * d * 4, d2h_bytes_per_step=d * 4,
             h2d_probe=probe, pcie_floor_ms=probe.get("ms"), host_path=bz.engine.host_path_report(device.index), h2d_rate_achieved_gbs=n * d * 4 / (e2e_ms * 1e-3) / 1e9,
             note="pcie_floor_ms = the faster of one contiguous pinned copy and n pinned row copies of the step's bytes on THIS box, outside the library (PCIe Gen5 x16 nominal: 2.1-2.4 ms); the step adds the kernel (~23 us), the 5 MB result copy and its synchronisation; host_path 'pipeline' = bz_coordinate_host (column chunks: batched H2D of chunk c+1, kernel of chunk c and D2H of chunk c-1 overlap)",
             ms_per_step=e2e_ms, ms_per_step_min=min(e2e_each), ms_per_step_median=sorted(e2e_each)[len(e2e_each) // 2], ms_per_step_max=max(e2e_each), steps=e2e_steps, host_buffers="pinned" + (", allocated under the NVML ideal-affinity binding" if numa_local else "") + "; host->device path chosen by measurement (see host_path)", call=f"byzantinemomentum_b200.gars[{gar!r}].unchecked(gradients=<{n} pinned host tensors>, f={f})")
  del host

  line = dict(metric="aggregated-params/sec", value=value, unit="params/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
              ms_per_step=ms_per_step, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32", data="synthetic",
              config=make_config(gar, n, f, d, world),
              details=dict(api=api, plugin_call_ms_per_step=plugin_ms,
                           l2="inputs rotate over %d independent [n, d] stacks (%.0f MB > L2)" % (sets, sets * set_bytes / 1e6)),
              roofline=roofline, e2e=e2e, gpu_launches=args.steps * LAUNCHES[gar], clocks=clocks.summary())
  if rank == 0 and world == 1:
    # ---- CPU baseline: the reference's operator sequence on the host cores (bounded sample) --------
    res = cpu_reference(torch, gar, n, f, d, 4321, budget_s=20.0, repeats=3)
    best = min(res["times"])
    line["cpu_baseline"] = dict(value=res["sample_d"] / best, unit="params/s", cores=res["threads"], kind=res["kind"],
                                sample=f"best of 3 calls ({gar}, n={n}, f={f}) on d={res['sample_d']} of {d} columns", ms_per_call=best * 1e3,
                                path=res["path"], cpu_model=res["cpu_model"], cpus_allowed=res["cpus_allowed"], torch=res["torch"])
    # the same operator sequence on CUDA tensors ("PyTorch on B200" incumbent, BASELINE.md §4.5)
    try:
      from oracle import refcost
      for _ in range(2):
        refcost.run(gar, inputs[0], f=f)
      torch.cuda.synchronize()
      t0 = time.perf_counter()
      for k in range(5):
        refcost.run(gar, inputs[k % sets], f=f)
      torch.cuda.synchronize()
      line["torch_cuda_baseline"] = dict(ms_per_call=(time.perf_counter() - t0) / 5 * 1e3, what="oracle/refcost.py on CUDA tensors (library kernels)")
    except Exception as err:
      line["torch_cuda_baseline"] = dict(error=str(err)[:200])
    if not args.no_sweep:
      line["sweep"] = sweep(torch, bz, device, peak)
  if not args.no_sharded:
    try:
      line["sharded"] = sharded_block(torch, dist, bz, sharded, device, world, rank, peak, args.steps)
    except Exception as err:
      line["sharded"] = dict(error=f"{type(err).__name__}: {err}"[:300])
  if args.dump_outputs:
    dump_outputs(args.dump_outputs, {"aggregate" if world == 1 else f"aggregate_rank{rank}": dumped})
  if rank == 0:
    print(json.dumps(line), flush=True)
  if dist is not None:
    dist.destroy_process_group()

def sweep(torch, bz, device, peak):
  """ Kernel-level numbers for the other rules / sizes (single GPU; not part of `value`). """
  rows_out = []
  flush = torch.empty(2 * L2_BYTES, dtype=torch.uint8, device=device)
  full = ["average", "median", "trmean", "phocas", "meamed", "krum", "bulyan", "aksel", "cge"]
  short = ["median", "trmean", "krum", "bulyan"]
  # every rule at BASELINE.json's shapes, plus the d sweep at n = 25 (metric: "per GAR at n=25, d sweep")
  c3 = ["krum", "bulyan", "aksel", "cge"]
  plan = [(25, 5, 1_310_922, c3), (25, 5, 36_489_290, ["krum", "bulyan"]), (25, 10, 79_510, full), (25, 10, 1_310_922, full), (25, 10, 36_489_290, full), (11, 5, 79_510, full + ["brute"]),
          (11, 3, 1_310_922, full + ["brute"]), (51, 12, 4_568_373, full),
          (25, 10, 1 << 16, short), (25, 10, 431_080, short), (25, 10, 2_384_036, short), (25, 10, 1 << 23, short), (25, 10, 1 << 25, short)]
  for n, f, d, gars in plan:
    gen = torch.Generator(device=device).manual_seed(5)
    rows = [torch.randn(d, device=device, generator=gen) for _ in range(n)]
    for gar in gars:
      ff = default_f(gar, n, f)
      if gar == "bulyan" and n < 4 * ff + 3:
        continue
      fn = lambda: bz.gars[gar].unchecked(gradients=rows, f=ff)
      try:
        for _ in range(3):
          fn()
        torch.cuda.synchronize()
        times = []
        for _ in range(7 if d > 4e6 else 15):
          if n * d * 4 < 4 * L2_BYTES:
            flush.zero_()
          a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
          a.record(); fn(); b.record()
          torch.cuda.synchronize()
          times.append(a.elapsed_time(b))
        times.sort()
        ms = times[len(times) // 2]
        alg = algorithmic_bytes(gar, n, ff, d)
        rows_out.append(dict(gar=gar, n=n, f=ff, d=d, ms=ms, params_per_s=d / (ms * 1e-3), gbs=alg / (ms * 1e-3) / 1e9,
                             frac=alg / (ms * 1e-3) / 1e9 / peak, read_only_frac=n * d * 4 / (ms * 1e-3) / 1e9 / peak))
      except Exception as err:
        rows_out.append(dict(gar=gar, n=n, f=ff, d=d, error=str(err)[:200]))
    if (n, d) in ((25, 1_310_922), (25, 36_489_290)):
      rows_out.append(study_metrics_row(torch, bz, rows, n, d, flush, peak))
    del rows
    torch.cuda.empty_cache()
  return rows_out

def study_metrics_row(torch, bz, rows, n, d, flush, peak):
  """ `tools.compute_avg_dev_max` (attack.py:846-848): bz_avg_dev_max on the device (CUDA events)
  and through its public call with the host read (wall clock), beside the reference's operator
  sequence on the same CUDA tensors (oracle/refcost.py, library kernels, wall clock). """
  import time
  from oracle import refcost
  try:
    times = []
    for k in range(10):
      if n * d * 4 < 4 * L2_BYTES:
        flush.zero_()
      a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      a.record(); bz.engine.avg_dev_max_async(rows); b.record()
      torch.cuda.synchronize()
      times.append(a.elapsed_time(b))
    ms = sorted(times[3:])[len(times[3:]) // 2]
    def wall(fn):
      fn(); torch.cuda.synchronize()
      t0 = time.perf_counter()
      for _ in range(5):
        fn()
      torch.cuda.synchronize()
      return (time.perf_counter() - t0) / 5 * 1e3
    alg = (n + 1) * d * 4              # one pass: every row read once, the average written once
    return dict(gar="avg_dev_max", n=n, f=0, d=d, ms=ms, params_per_s=d / (ms * 1e-3), gbs=alg / (ms * 1e-3) / 1e9,
                frac=alg / (ms * 1e-3) / 1e9 / peak, read_only_frac=n * d * 4 / (ms * 1e-3) / 1e9 / peak,
                call_ms=wall(lambda: bz.compute_avg_dev_max(rows)), torch_cuda_ms=wall(lambda: refcost.study_metrics(rows)))
  except Exception as err:
    return dict(gar="avg_dev_max", n=n, f=0, d=d, error=str(err)[:200])

def main():
  ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=200)
  ap.add_argument("--warmup", type=int, default=10)
  ap.add_argument("--impl", choices=("b200", "reference"), default="b200")
  ap.add_argument("--gar", default="trmean")
  ap.add_argument("--nb-workers", dest="n", type=int, default=25)
  ap.add_argument("--nb-byz", dest="f", type=int, default=10)
  ap.add_argument("--dim", dest="d", type=int, default=1_310_922)
  ap.add_argument("--no-sweep", action="store_true")
  ap.add_argument("--no-sharded", action="store_true", help="skip the `sharded` block (collective path at C3 per GPU + C4 strong scaling; at N = 1 it is the reference line of the series)")
  ap.add_argument("--exchange", choices=("auto", "nccl", "p2p"), default="auto",
                  help="N > 1, distance-based rules: all-gather (NCCL) or blocks read in place over NVLink peer memory")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="write what the last timed step returned to DIR/<name>.npy (b200 implementation)")
  args = ap.parse_args()
  if args.steps < 1:
    ap.error("--steps must be at least 1")
  if args.dump_outputs and args.impl != "b200":
    ap.error("--dump-outputs writes the outputs of the b200 implementation")
  global EXCHANGE
  EXCHANGE = args.exchange
  if args.impl == "reference":
    run_reference(args)
  else:
    run_b200(args)

if __name__ == "__main__":
  main()
