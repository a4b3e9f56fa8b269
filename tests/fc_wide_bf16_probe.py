"""Diagnostics (not a test): the bf16 FCNetwork against tf32x3 at 33..64 actions on the per-launch search path.

1. recurrent_inference per call at 4096 rows (CUDA events over --calls back-to-back launches; the 800 KB of hidden
   input stay in L2, as in a search) for each --actions value, bf16 and tf32x3;
2. one move of G = 4096 games x S = 50 simulations (CUDA graph, --streams slices) at A = 64 and 50, bf16 and tf32x3
   alternated over --rounds rounds, and where a single-slice un-graphed move spends its time: the network launch and
   the tree step per simulation (events around every launch).
Prints one JSON line per measurement and the card it ran on (name, power limit, max SM clock).

  python tests/fc_wide_bf16_probe.py [--games 4096] [--sims 50] [--moves 20] [--rounds 3]"""
import argparse
import json
import os
import sys
import types

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from model_based_rl_b200 import _lib  # noqa: E402
from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict  # noqa: E402
from wide_probe import card  # noqa: E402

PRECISIONS = ("bf16", "tf32x3")


def _cfg(S, A):
  return types.SimpleNamespace(num_simulations=S, action_space=A, two_players=False, discount=0.997, pb_c_base=19652,
                               pb_c_init=1.25, init_value_score=0.0, known_bounds=[None, None],
                               root_exploration_fraction=0.25, value_support=[-15, 15], reward_support=[-15, 15],
                               no_support=False, no_target_transform=False)


def _net(D, A, precision):
  net = FCNetwork(D, A, "cuda", _cfg(1, A), precision=precision)
  net.load_weights(random_state_dict(D, A))
  return net


def per_call(A, D, rows, calls):
  out = {}
  rng = np.random.default_rng(A)
  h = torch.from_numpy(np.maximum(rng.normal(0.3, 1.0, size=(rows, 50)), 0).astype(np.float32)).cuda()
  a = torch.from_numpy(rng.integers(0, A, size=rows).astype(np.int32)).cuda()
  for prec in PRECISIONS:
    net = _net(D, A, prec)
    v, r, l, ho = net._buffers(rows)
    call = lambda: net.recurrent_into(h, 50, None, a, ho, 50, 0, v, r, l)
    for _ in range(20):
      call()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(calls):
      call()
    t1.record()
    torch.cuda.synchronize()
    out[prec] = round(t0.elapsed_time(t1) * 1e3 / calls, 2)
  return {"what": "recurrent_inference_us_per_call", "actions": A, "rows": rows, **out}


def moves(G, S, A, D, n_moves, rounds, streams):
  rng = np.random.default_rng(0)
  obs = rng.random((G, D)).astype(np.float32)
  noise = rng.dirichlet([0.25] * A, size=G)
  cfg = _cfg(S, A)
  searches, res = {}, {}
  for prec in PRECISIONS:
    net = _net(D, A, prec)
    fs = FCSearch(cfg, net, G, use_graph=True, num_streams=streams)
    assert fs.fused is None
    fs.search_host(obs, noise, rng.random(G), np.ones(G))
    for _ in range(3):
      fs.run()
    # where one un-graphed single-slice move spends its time
    fs1 = FCSearch(cfg, net, G, use_graph=False, num_streams=1)
    fs1.search_host(obs, noise, rng.random(G), np.ones(G))
    plan = fs1.lanes[0]._plan(fs1.use_noise, fs1.noise_frac, torch.cuda.current_stream().cuda_stream)
    nets, steps = [], []
    for rep in range(3):
      ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(plan) + 1)]
      ev[0].record()
      for i, (fn, args) in enumerate(plan):
        _lib.check(fn(*args), fn.__name__)
        ev[i + 1].record()
      torch.cuda.synchronize()
      dur = [ev[i].elapsed_time(ev[i + 1]) * 1e3 for i in range(len(plan))]
      if rep:
        nets.append(np.mean([dur[3 + 2 * s] for s in range(S)]))
        steps.append(np.mean([dur[4 + 2 * s] for s in range(S - 1)]))
    searches[prec] = fs
    res[prec] = dict(ms=[], network_us_per_sim=round(float(np.mean(nets)), 2),
                     tree_step_us_per_sim=round(float(np.mean(steps)), 2))
  torch.cuda.synchronize()
  for _ in range(rounds):
    for prec in PRECISIONS:
      fs = searches[prec]
      t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      t0.record()
      for _ in range(n_moves):
        fs.run()
      t1.record()
      torch.cuda.synchronize()
      res[prec]["ms"].append(round(t0.elapsed_time(t1) / n_moves, 4))
  for prec in PRECISIONS:
    ms = float(np.median(res[prec]["ms"]))
    res[prec]["expansions_per_s"] = round(G * S / (ms * 1e-3))
  return {"what": "move", "actions": A, "games": G, "sims": S, "streams": streams, **res}


def main():
  p = argparse.ArgumentParser()
  p.add_argument("--games", type=int, default=4096)
  p.add_argument("--sims", type=int, default=50)
  p.add_argument("--obs-dim", type=int, default=128)
  p.add_argument("--moves", type=int, default=20)
  p.add_argument("--rounds", type=int, default=3)
  p.add_argument("--streams", type=int, default=4)
  p.add_argument("--calls", type=int, default=200)
  p.add_argument("--actions", default="18,32,45,50,64")
  p.add_argument("--move-actions", default="64,50")
  a = p.parse_args()
  print(json.dumps({"card": card()}), flush=True)
  for A in [int(x) for x in a.actions.split(",")]:
    print(json.dumps(per_call(A, a.obs_dim, a.games, a.calls)), flush=True)
  for A in [int(x) for x in a.move_actions.split(",")]:
    print(json.dumps(moves(a.games, a.sims, A, a.obs_dim, a.moves, a.rounds, a.streams)), flush=True)


if __name__ == "__main__":
  main()
