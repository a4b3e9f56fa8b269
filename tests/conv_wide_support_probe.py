"""Times the wide support head (mz_conv_support_head_tc) and what a 601-bin support costs a C5-shaped move.
Not a test; prints one JSON line (and writes it to --out when given).

  python tests/conv_wide_support_probe.py [--games 4096] [--sims 50] [--repeats 5] [--out FILE]

1. Head kernel alone, per call, CUDA events over `--calls` back-to-back launches on the [games][1536] fc buffer:
   mz_conv_support_head_tc at 64, 601 and 1024 bins against mz_conv_head at 31 bins.
2. ConvSearch move (ConvSearch.search: initial inference + search in one CUDA graph), 96 x 96 x 32 frames,
   A = 18, at 31-bin value and reward supports and at 601-bin ([-300, 300]) ones: the two engines alternate,
   `--repeats` timed moves each, and the spread between repeats is reported.
The card's name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def card():
  try:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True, timeout=30).stdout.strip().splitlines()[0]
    name, limit = [s.strip() for s in q.split(",")]
  except Exception:  # noqa: BLE001 -- the name alone still identifies the card
    name, limit = torch.cuda.get_device_name(0), "unknown"
  return {"gpu": name, "power_limit": limit}


def time_heads(G, calls):
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  dev = "cuda"
  P, st = _lib.ptr, _lib.current_stream()
  torch.manual_seed(0)
  fc = torch.relu(torch.randn((G, 1536), device=dev))
  out = torch.zeros(G, device=dev)
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  res = {}
  for bins in (31, 64, 601, 1024):
    w = torch.randn((bins, 512), device=dev) * 0.05
    bias = torch.randn(bins, device=dev) * 0.1
    if bins <= 32:
      launch = lambda: _lib.check(lib.mz_conv_head(G, fc[:, 512:].data_ptr(), 1536, P(w), P(bias), bins, 1, -15, 0,
                                                   P(out), 1, st), "mz_conv_head")
      name = "mz_conv_head"
    else:
      wb = w.to(torch.bfloat16).contiguous()
      launch = lambda: _lib.check(lib.mz_conv_support_head_tc(G, fc[:, 512:].data_ptr(), 1536, P(wb), P(bias), bins,
                                                              -(bins // 2), 0, P(out), 1, st),
                                  "mz_conv_support_head_tc")
      name = "mz_conv_support_head_tc"
    for _ in range(10):
      launch()
    torch.cuda.synchronize()
    a.record()
    for _ in range(calls):
      launch()
    b.record()
    torch.cuda.synchronize()
    res["%s_%d_bins_us" % (name, bins)] = round(a.elapsed_time(b) * 1e3 / calls, 2)
  return res


def time_moves(G, S, repeats):
  from model_based_rl_b200.muzero import ConvSearch, MuZeroNetwork, random_state_dict
  A, C_in = 18, 32
  rng = np.random.default_rng(77)
  noise, u = rng.dirichlet([0.25] * A, size=G), rng.random(G)
  obs = torch.from_numpy(rng.random((G, C_in, 96, 96), dtype=np.float32)).cuda()
  engines = {}
  for label, sup in (("31_bins", (-15, 15)), ("601_bins", (-300, 300))):
    cfg = types.SimpleNamespace(num_simulations=S, action_space=A, two_players=False, discount=0.997,
                                pb_c_base=19652, pb_c_init=1.25, init_value_score=0.0, known_bounds=[None, None],
                                root_exploration_fraction=0.25, value_support=list(sup), reward_support=list(sup),
                                no_support=False, no_target_transform=False)
    net = MuZeroNetwork(C_in, A, "cuda", cfg)
    bins = sup[1] - sup[0] + 1
    net.load_weights(random_state_dict(C_in, A, value_bins=bins, reward_bins=bins))
    cs = ConvSearch(cfg, net, G)
    for _ in range(2):
      cs.search(obs, noise, u)
    engines[label] = cs
  torch.cuda.synchronize()
  a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  ms = {k: [] for k in engines}
  for _ in range(repeats):
    for label, cs in engines.items():
      a.record()
      cs.search(obs)
      b.record()
      torch.cuda.synchronize()
      ms[label].append(a.elapsed_time(b))
  res = {}
  for label, t in ms.items():
    res["move_ms_" + label] = round(float(np.median(t)), 3)
    res["move_ms_%s_min_max" % label] = [round(min(t), 3), round(max(t), 3)]
  res["move_601_over_31"] = round(res["move_ms_601_bins"] / res["move_ms_31_bins"], 4)
  return res


def main():
  p = argparse.ArgumentParser()
  p.add_argument("--games", type=int, default=4096)
  p.add_argument("--sims", type=int, default=50)
  p.add_argument("--repeats", type=int, default=5)
  p.add_argument("--calls", type=int, default=200)
  p.add_argument("--out", default=None)
  args = p.parse_args()
  torch.cuda.set_device(0)
  res = card()
  res.update(time_heads(args.games, args.calls))
  res.update(time_moves(args.games, args.sims, args.repeats))
  line = json.dumps(res)
  print(line)
  if args.out:
    with open(args.out, "w") as f:
      f.write(line + "\n")


if __name__ == "__main__":
  main()
