"""Measurement (not a test): device time per learner step of FusedLearner(precision='tf32x3') against the bf16 and f32
steps and learners.Learner (torch modules), all in CUDA graphs, in one process, at B = 512, K = 5, 128 features,
AdamW, 31 + 31-bin supports: A = 4, A = 18, and A = 4 with a --no_support MSE network.  Each learner is warmed up,
then the four alternate over ROUNDS rounds of N steps; the card's name, power limit and maximum SM clock are read in the
same run.

  python tests/learner_tf32x3_one.py [--rounds 3] [--steps 50] [--json out.json] [--profile dir]

--profile: afterwards, one torch.profiler trace of 20 tf32x3 steps per case, per-kernel device times printed."""
import argparse
import json
import os
import subprocess
import sys
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from model_based_rl_b200 import fused_learner, learners

B, K, E = 512, 5, 128
KINDS = ("tf32x3", "bf16", "f32", "torch")


def card():
  q = "name,power.limit,clocks.max.sm"
  try:
    line = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"], capture_output=True,
                          text=True, check=True).stdout.strip().splitlines()[0]
    return dict(zip(q.split(","), [s.strip() for s in line.split(",")]))
  except (OSError, subprocess.CalledProcessError, IndexError):
    return {"name": torch.cuda.get_device_name(0)}


def make_case(A, no_support):
  cfg = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=no_support,
                              no_target_transform=False, num_unroll_steps=K, optimizer="AdamW", lr_init=0.0008, momentum=0.9,
                              weight_decay=1e-4, clip_grad=0, lr_scheduler=None, norm_obs=False)
  if no_support:
    cfg.scalar_loss = "MSE"
  dev = torch.device("cuda:0")
  g = torch.Generator(device=dev).manual_seed(7 + A)
  r = lambda *shape: torch.rand(*shape, device=dev, generator=g)
  pol = r(B, K + 1, A)
  batch = ((r(B, E), torch.randint(0, A, (B, K), device=dev, generator=g),
            ((r(B, K + 1) < 0.1).float(), 4 * torch.randn(B, K + 1, device=dev, generator=g), pol / pol.sum(-1, keepdim=True))),
           None, r(B).double())
  torch.manual_seed(A)
  w = learners.FCNetworkTrain(E, A, "cpu", cfg).get_weights()
  out = {}
  for kind in KINDS:
    if kind == "torch":
      net = learners.FCNetworkTrain(E, A, dev, cfg)
      net.load_weights(w)
      out[kind] = learners.Learner(cfg, net, use_graph=True)
    else:
      net = fused_learner.FusedFCNetwork(E, A, dev, cfg)
      net.load_weights(w)
      out[kind] = fused_learner.FusedLearner(cfg, net, use_graph=True, precision=kind)
  return out, batch


def time_steps(learner, batch, n):
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  a.record()
  for _ in range(n):
    learner.update_weights(batch)
  b.record()
  torch.cuda.synchronize()
  return a.elapsed_time(b) * 1e3 / n


def profile(learner, batch, path):
  from torch.profiler import ProfilerActivity, profile as prof
  with prof(activities=[ProfilerActivity.CUDA]) as p:
    for _ in range(20):
      learner.update_weights(batch)
    torch.cuda.synchronize()
  p.export_chrome_trace(path)
  rows = {}
  for e in p.events():
    if e.device_type == torch.autograd.DeviceType.CUDA:
      r = rows.setdefault(e.name, [0, 0.0])
      r[0] += 1
      r[1] += e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
  for name, (cnt, us) in sorted(rows.items(), key=lambda kv: -kv[1][1]):
    print("    %9.1f us/step  %4d calls  %s" % (us / 20, cnt, name[:110]))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--rounds", type=int, default=3)
  ap.add_argument("--steps", type=int, default=50)
  ap.add_argument("--json", default=None)
  ap.add_argument("--profile", default=None)
  args = ap.parse_args()
  info = card()
  print("card: %s" % json.dumps(info))
  cases = {"A4": (4, False), "A18": (18, False), "A4_no_support_mse": (4, True)}
  result = {"card": info, "B": B, "K": K, "features": E, "rounds": args.rounds, "steps": args.steps, "cases": {}}
  built = {}
  for name, (A, ns) in cases.items():
    learners_, batch = make_case(A, ns)
    for kind in KINDS:  # warm-up: graph capture, module loading, a few steps
      for _ in range(5):
        learners_[kind].update_weights(batch)
    torch.cuda.synchronize()
    built[name] = (learners_, batch)
  for name, (learners_, batch) in built.items():
    times = {k: [] for k in KINDS}
    for _ in range(args.rounds):
      for kind in KINDS:
        times[kind].append(time_steps(learners_[kind], batch, args.steps))
    result["cases"][name] = times
    print("%s (A = %d%s):" % (name, cases[name][0], ", --no_support MSE" if cases[name][1] else ""))
    for kind in KINDS:
      t = sorted(times[kind])
      print("  %-7s median %8.1f us/step  (rounds: %s)" % (kind, t[len(t) // 2], ", ".join("%.1f" % x for x in times[kind])))
    tf, to = sorted(times["tf32x3"])[args.rounds // 2], sorted(times["torch"])[args.rounds // 2]
    print("  tf32x3 / torch-module step: %.3f" % (tf / to))
  if args.json:
    with open(args.json, "w") as f:
      json.dump(result, f, indent=1)
  if args.profile:
    os.makedirs(args.profile, exist_ok=True)
    for name, (learners_, batch) in built.items():
      print("profile %s, tf32x3 step:" % name)
      profile(learners_["tf32x3"], batch, os.path.join(args.profile, "tf32x3_%s.json" % name))


if __name__ == "__main__":
  main()
