"""Diagnostics (not a test): one move of G = 4096 games x S = 50 simulations with the float32-accurate tensor-core
FCNetwork (precision='tf32x3', per-launch path) at 64 actions and, for comparison, at 32: expansions/s of the whole
move (CUDA graph, CUDA events over timed moves) and the tree-step kernel's time per simulation (events around each
launch of an un-graphed move), with the step kernel on a shared-memory image of each tree and on the global blocks
(mz_debug_set_tree_staging).  Prints one JSON line per (A, staging) and the card it ran on.

  python tests/wide_probe.py [--games 4096] [--sims 50] [--moves 30]"""
import argparse
import json
import os
import subprocess
import sys
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from model_based_rl_b200 import _lib  # noqa: E402
from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict  # noqa: E402


def card():
  try:
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
  except (OSError, subprocess.SubprocessError, IndexError):
    return "unknown"


def probe(G, S, A, D, moves, staging, streams):
  lib = _lib.load()
  lib.mz_debug_set_tree_staging(staging)
  cfg = types.SimpleNamespace(num_simulations=S, action_space=A, two_players=False, discount=0.997, pb_c_base=19652,
                              pb_c_init=1.25, init_value_score=0.0, known_bounds=[None, None],
                              root_exploration_fraction=0.25, value_support=[-15, 15], reward_support=[-15, 15],
                              no_support=False, no_target_transform=False)
  net = FCNetwork(D, A, "cuda", cfg, precision="tf32x3")
  net.load_weights(random_state_dict(D, A))
  rng = np.random.default_rng(0)
  obs = rng.random((G, D)).astype(np.float32)
  noise = rng.dirichlet([0.25] * A, size=G)
  # whole move: graph replays on device-resident inputs
  fs = FCSearch(cfg, net, G, use_graph=True, num_streams=streams)
  assert fs.fused is None
  fs.search_host(obs, noise, rng.random(G), np.ones(G))
  for _ in range(3):
    fs.run()
  torch.cuda.synchronize()
  t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  t0.record()
  for _ in range(moves):
    fs.run()
  t1.record()
  torch.cuda.synchronize()
  move_ms = t0.elapsed_time(t1) / moves
  # tree-step kernel alone: events around every launch of one un-graphed single-slice move
  fs1 = FCSearch(cfg, net, G, use_graph=False, num_streams=1)
  fs1.search_host(obs, noise, rng.random(G), np.ones(G))
  plan = fs1.lanes[0]._plan(fs1.use_noise, fs1.noise_frac, torch.cuda.current_stream().cuda_stream)
  steps = []
  for rep in range(3):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(plan) + 1)]
    ev[0].record()
    for i, (fn, args) in enumerate(plan):
      _lib.check(fn(*args), fn.__name__)
      ev[i + 1].record()
    torch.cuda.synchronize()
    dur = [ev[i].elapsed_time(ev[i + 1]) * 1e3 for i in range(len(plan))]
    if rep:
      steps.append(np.mean([dur[4 + 2 * s] for s in range(S - 1)]))  # backup of s + descent of s + 1
  lib.mz_debug_set_tree_staging(0)
  return {"actions": A, "games": G, "sims": S, "obs_dim": D, "precision": "tf32x3", "streams": streams,
          "tree_image": "global" if staging else "shared", "move_ms": round(move_ms, 4),
          "expansions_per_s": round(G * S / (move_ms * 1e-3)), "tree_step_us_per_sim": round(float(np.mean(steps)), 2)}


def main():
  p = argparse.ArgumentParser()
  p.add_argument("--games", type=int, default=4096)
  p.add_argument("--sims", type=int, default=50)
  p.add_argument("--obs-dim", type=int, default=128)
  p.add_argument("--moves", type=int, default=30)
  p.add_argument("--streams", type=int, default=4)
  a = p.parse_args()
  print(json.dumps({"card": card()}))
  for A in (64, 32):
    for staging in (0, 1):
      print(json.dumps(probe(a.games, a.sims, A, a.obs_dim, a.moves, staging, a.streams)), flush=True)


if __name__ == "__main__":
  main()
