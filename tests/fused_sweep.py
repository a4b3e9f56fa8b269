"""Timing sweep (not a pytest): per-launch path vs the fused kernel, with and without programmatic dependent
launches, on the BASELINE shapes."""
import sys, types
import numpy as np
import torch
sys.path.insert(0, ".")
from model_based_rl_b200 import _lib
from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict

lib = _lib.load()
SHAPES = {"C4": (4096, 18, 50, 128, False, [None, None]), "C1": (4096, 9, 30, 9, True, [-1, 1]),
          "C2": (1024, 4, 30, 8, False, [None, None]), "C3": (4096, 4, 50, 128, False, [None, None]),
          "C4x4": (16384, 18, 50, 128, False, [None, None]), "C4/4": (1024, 18, 50, 128, False, [None, None])}


def run(name, variant, moves=20):
  G, A, S, D, two, kb = SHAPES[name]
  cfg = types.SimpleNamespace(
      num_simulations=S, action_space=A, two_players=two, discount=1.0 if two else 0.997, pb_c_base=19652,
      pb_c_init=1.25, init_value_score=0.0, known_bounds=kb, root_exploration_fraction=0.25,
      value_support=[-15, 15], reward_support=[-15, 15], no_support=False, no_target_transform=False)
  net = FCNetwork(D, A, "cuda", cfg)
  net.load_weights(random_state_dict(D, A))
  rng = np.random.default_rng(2)
  obs = rng.random((G, D)).astype(np.float32)
  noise, u, temp = rng.dirichlet([0.25] * A, size=G), rng.random(G), np.ones(G)
  fused, pdl = variant
  lib.mz_set_programmatic_launch(pdl)
  fs = FCSearch(cfg, net, G, use_graph=True, num_streams=4, fused=bool(fused))
  fs.search_host(obs, noise, u, temp)
  for _ in range(3):
    fs.run()
  torch.cuda.synchronize()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(moves):
    fs.run()
  e1.record()
  torch.cuda.synchronize()
  ms = e0.elapsed_time(e1) / moves
  lib.mz_set_programmatic_launch(1)
  return ms, G * S / ms / 1e3


if __name__ == "__main__":
  variants = {"per-launch x4 streams": (0, 1), "fused pdl": (1, 1), "fused no-pdl": (1, 0)}
  for name in sys.argv[1:] or list(SHAPES):
    for vn, v in variants.items():
      ms, rate = run(name, v, moves=5 if name == "C4x4" else 20)
      print("%-5s %-26s %8.3f ms/move %8.1f M expansions/s" % (name, vn, ms, rate), flush=True)
