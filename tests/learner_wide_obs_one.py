"""Diagnostics (not a test): the fused learner on wide observations.

  python tests/learner_wide_obs_one.py measure
      CUDA-graph steps at B = 512, K = 5, A = 18, AdamW for input_dim 128, 147, 512, 1024: the bf16 FusedLearner, the
      f32 FusedLearner and learners.Learner (torch modules) in one process, with the card's name and power limit.
  python tests/learner_wide_obs_one.py dump OUT.npz
      Losses, priority errors and weights after a few seeded captured steps at input_dim 8 and 128 in both precisions,
      and steps/s: run once per library (MZB200_LIB=..., tests/ab_build.sh) and compare the files with `compare`.
  python tests/learner_wide_obs_one.py compare A.npz B.npz
"""
import os
import subprocess
import sys
import time
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

B, K, A = 512, 5, 18


def _cfg():
  return types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=False, no_target_transform=False,
                               num_unroll_steps=K, optimizer="AdamW", lr_init=0.0008, momentum=0.9, weight_decay=1e-4,
                               clip_grad=0, lr_scheduler=None, norm_obs=False)


def _batch(D, seed, dev):
  g = torch.Generator(device=dev).manual_seed(seed)
  r = lambda *shape: torch.rand(*shape, device=dev, generator=g)
  pol = r(B, K + 1, A)
  return ((r(B, D), torch.randint(0, A, (B, K), device=dev, generator=g),
           ((r(B, K + 1) < 0.1).float(), 4 * torch.randn(B, K + 1, device=dev, generator=g), pol / pol.sum(-1, keepdim=True))),
          None, r(B).double())


def _learner(kind, D, dev, cfg, weights):
  from model_based_rl_b200 import fused_learner, learners
  if kind == "torch":
    net = learners.FCNetworkTrain(D, A, dev, cfg)
    net.load_weights(weights)
    return learners.Learner(cfg, net, use_graph=True), net
  net = fused_learner.FusedFCNetwork(D, A, dev, cfg)
  net.load_weights(weights)
  return fused_learner.FusedLearner(cfg, net, use_graph=True, precision=kind), net


def _time(lr, batch, n):
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  for _ in range(10):
    lr.update_weights(batch)
  torch.cuda.synchronize()
  a.record()
  for _ in range(n):
    lr.update_weights(batch)
  b.record()
  torch.cuda.synchronize()
  return a.elapsed_time(b) * 1e3 / n


def _card():
  q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
  return q[torch.cuda.current_device()] if q else torch.cuda.get_device_name()


def measure():
  from model_based_rl_b200 import learners
  dev = torch.device("cuda:0")
  cfg = _cfg()
  print("card: %s" % _card())
  print("B = %d, K = %d, A = %d, AdamW, CUDA graphs; us per step (device events over 200 steps, after 10 warm-up)" % (B, K, A))
  print("%6s %10s %10s %10s %12s" % ("D", "bf16", "f32", "torch", "torch / bf16"))
  for D in (128, 147, 512, 1024):
    torch.manual_seed(D)
    w = learners.FCNetworkTrain(D, A, "cpu", cfg).state_dict()
    batch = _batch(D, 7, dev)
    t = {kind: _time(_learner(kind, D, dev, cfg, w)[0], batch, 200) for kind in ("bf16", "f32", "torch")}
    print("%6d %10.1f %10.1f %10.1f %11.1fx" % (D, t["bf16"], t["f32"], t["torch"], t["torch"] / t["bf16"]), flush=True)


def dump(out):
  from model_based_rl_b200 import learners
  dev = torch.device("cuda:0")
  cfg = _cfg()
  res = {}
  for D in (8, 128):
    torch.manual_seed(D)
    w = learners.FCNetworkTrain(D, A, "cpu", cfg).state_dict()
    for kind in ("bf16", "f32"):
      lr, net = _learner(kind, D, dev, cfg, w)
      for step in range(3):
        lr.update_weights(_batch(D, 100 + step, dev))
        res["%s_%d_losses_%d" % (kind, D, step)] = lr.last_losses.cpu().numpy()
        res["%s_%d_errors_%d" % (kind, D, step)] = lr.last_errors.cpu().numpy()
      res["%s_%d_weights" % (kind, D)] = net.flat.cpu().numpy()
      us = _time(lr, _batch(D, 7, dev), 300)
      res["%s_%d_us" % (kind, D)] = np.array(us)
      print("%s D=%d: %.1f us/step, %.0f steps/s" % (kind, D, us, 1e6 / us), flush=True)
  np.savez(out, **res)


def compare(a, b):
  x, y = np.load(a), np.load(b)
  same = True
  for k in sorted(x.files):
    if k.endswith("_us"):
      print("%-22s %8.1f us  %8.1f us" % (k, float(x[k]), float(y[k])))
    elif not np.array_equal(x[k], y[k]):
      same = False
      print("DIFFERENT: %s (max |diff| %g)" % (k, float(np.abs(x[k] - y[k]).max())))
  print("bit-identical" if same else "NOT bit-identical")
  return same


if __name__ == "__main__":
  if sys.argv[1] == "measure":
    measure()
  elif sys.argv[1] == "dump":
    dump(sys.argv[2])
  else:
    sys.exit(0 if compare(sys.argv[2], sys.argv[3]) else 1)
