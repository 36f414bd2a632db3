# coding: utf-8
"""Stand-in for the `tools` package of the original ByzantineMomentum project, written for the tests
of this repository (it is not the original): the members the rule registry, attack.py and
`byzantinemomentum_b200.plugin.install_tools` use."""

import contextlib
import math
import sys

class UserException(Exception):
  """ Error the original reports to the user (its registry raises it from `checked`). """

def warning(message):
  print(f"warning: {message}", file=sys.stderr)

@contextlib.contextmanager
def Context(name, level):
  yield

def compute_avg_dev_max(samples):
  """ Average of the samples (None without samples), its norm, the norm deviation of the samples
  around it (NaN below two samples) and its largest absolute coordinate. """
  if len(samples) == 0:
    return None, math.nan, math.nan, math.nan
  avg = samples[0].clone().detach_()
  for grad in samples[1:]:
    avg.add_(grad)
  avg.div_(len(samples))
  dev = math.nan
  if len(samples) >= 2:
    dev = math.sqrt(sum(grad.sub(avg).dot(grad.sub(avg)).item() for grad in samples) / (len(samples) - 1))
  return avg, avg.norm().item(), dev, avg.abs().max().item()
