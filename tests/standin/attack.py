# coding: utf-8
"""Stand-in for the original ByzantineMomentum project's attack.py, written for the tests of this
repository (it is not the original): its command line, the calls it makes into `aggregators`,
`experiments` and `tools`, and the statement groups tools/drive_attack.py rewrites, training a
linear least-squares model on the batches `experiments.make_datasets` yields."""

import argparse
import collections
import sys

import torch

import aggregators
import experiments
import tools

parser = argparse.ArgumentParser()
for flag, kind, default in (("--seed", int, -1), ("--device", str, "auto"), ("--device-gar", str, "same"), ("--nb-steps", int, 300),
                            ("--nb-workers", int, 11), ("--nb-for-study", int, 1), ("--nb-for-study-past", int, 1),
                            ("--nb-decl-byz", int, 4), ("--nb-real-byz", int, 0), ("--gar", str, "average"), ("--attack", str, "nan"),
                            ("--model", str, "simples-full"), ("--dataset", str, "mnist"), ("--batch-size", int, 25),
                            ("--learning-rate", float, 0.5), ("--momentum", float, 0.9), ("--dampening", float, 0.),
                            ("--momentum-at", str, "update"), ("--gradient-clip", float, None), ("--result-directory", str, None),
                            ("--evaluation-delta", int, 100)):
  parser.add_argument(flag, type=kind, default=default)
parser.add_argument("--attack-args", nargs="*", default=[])
args = parser.parse_args(sys.argv[1:])
args.nb_honests = args.nb_workers - args.nb_real_byz
args.device = "cpu" if args.device == "auto" else args.device
factor = float(dict(arg.split(":", 1) for arg in args.attack_args).get("factor", 1.))
defense = aggregators.gars[args.gar]
device = torch.device(args.device)
if args.seed >= 0:
  torch.manual_seed(args.seed)

train, _ = experiments.make_datasets(args.dataset, args.batch_size, args.batch_size)
x, y = train.sample()
theta = torch.zeros(x[0].numel() * 10, device=device)
def gradient(theta, x, y):
  """ Least squares of the one-hot labels: (X^T (X W - Y)) / b, flattened. """
  x = x.reshape(x.shape[0], -1).to(device)
  target = torch.nn.functional.one_hot(y.to(device), 10).to(x.dtype)
  return (x.t() @ (x @ theta.view(x.shape[1], 10) - target)).div_(x.shape[0]).reshape(-1)

grad_momentum_workers = [torch.zeros_like(theta) for _ in range(args.nb_honests)]
grad_momentum_server = torch.zeros_like(theta)
PastGrad = collections.namedtuple("PastGrad", ("grad", "norm"))
grad_pasts = collections.deque(maxlen=args.nb_for_study_past)

with tools.Context("training", "info"):
  print("Training...", flush=True)
  for step in range(args.nb_steps):
    grad_sampleds = list()
    for worker in range(args.nb_honests):
      for x, y in [train.sample()]:
        with torch.no_grad():
          grad = gradient(theta, x, y)
          # Gradient clip and append
          if args.gradient_clip is not None:
            grad_norm = grad.norm().item()
            if grad_norm > args.gradient_clip:
              grad.mul_(args.gradient_clip / grad_norm)
          grad_sampleds.append(grad.clone().detach_())
    for worker in range(max(args.nb_for_study - args.nb_honests, 0)):
      for x, y in [train.sample()]:
        with torch.no_grad():
          grad = gradient(theta, x, y)
          # Gradient clip and append
          if args.gradient_clip is not None:
            grad_norm = grad.norm().item()
            if grad_norm > args.gradient_clip:
              grad.mul_(args.gradient_clip / grad_norm)
          grad_sampleds.append(grad.clone().detach_())
    if args.momentum_at == "worker":
      grad_honests = list()
      for gmtm, grad in zip(grad_momentum_workers, grad_sampleds[:args.nb_honests]):
        gmtm.mul_(args.momentum).add_(grad, alpha=(1. - args.dampening))
        grad_honests.append(gmtm)
    elif args.momentum_at == "server":
      grad_honests = list()
      for grad in grad_sampleds[:args.nb_honests]:
        grad_honests.append(grad.mul(1. - args.dampening).add_(grad_momentum_server, alpha=args.momentum))
    else:
      grad_honests = grad_sampleds[:args.nb_honests]
    grad_attacks = [torch.stack(grad_honests).mean(dim=0).mul_(-factor)] * args.nb_real_byz
    grad_defense = defense(gradients=grad_honests + grad_attacks, f=args.nb_decl_byz)
    if args.momentum_at == "update":
      grad_momentum_server.mul_(args.momentum).add_(grad_defense, alpha=1. - args.dampening)
      grad_defense = grad_momentum_server
    theta.sub_(grad_defense, alpha=args.learning_rate)
    with torch.no_grad():
      # Compute the sampled and honest gradients norm average, norm deviation and max absolute coordinate
      sampled_grad_avg, sampled_norm_avg, sampled_norm_dev, sampled_norm_max = tools.compute_avg_dev_max(grad_sampleds)
      honest_grad_avg, honest_norm_avg, honest_norm_dev, honest_norm_max = tools.compute_avg_dev_max(grad_honests)
      attack_grad_avg, attack_norm_avg, attack_norm_dev, attack_norm_max = tools.compute_avg_dev_max(grad_attacks)
      defense_norm = grad_defense.norm().item()
      cosin_splhon = torch.dot(sampled_grad_avg, honest_grad_avg).item() / (sampled_norm_avg * honest_norm_avg)
      cosin_hondef = torch.dot(honest_grad_avg, grad_defense).item() / (honest_norm_avg * defense_norm)
      # Store the new past gradient (automatic rolling)
      grad_pasts.appendleft(PastGrad(sampled_grad_avg, sampled_norm_avg))
      print(f"step {step}: defense norm {defense_norm:.6g}, cosine honest/defense {cosin_hondef:.6g}", flush=True)
