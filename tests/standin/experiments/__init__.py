# coding: utf-8
"""Stand-in for the `experiments` package of the original ByzantineMomentum project, written for the
tests of this repository: a dataset is an endless iterator of (inputs, labels) batches, and
`make_datasets` has no data of its own (tools/drive_attack.py replaces it with synthetic batches)."""

class Dataset:
  def __init__(self, data, name=None):
    self.data, self.name = data, name
  def sample(self):
    return next(self.data)

def make_datasets(dataset, train_batch, test_batch, **kwargs):
  raise RuntimeError(f"no data for {dataset!r}: replace experiments.make_datasets")
