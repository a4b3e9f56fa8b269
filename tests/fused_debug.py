"""Debug: first divergence between the per-launch search and the fused kernel, with the trees of one game."""
import sys, types
import numpy as np
import torch
sys.path.insert(0, ".")
from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict

S, game = int(sys.argv[1]), int(sys.argv[2])
G, A, D = 300, 18, 128
cfg = types.SimpleNamespace(
    num_simulations=S, action_space=A, two_players=False, discount=0.997, pb_c_base=19652, pb_c_init=1.25,
    init_value_score=0.0, known_bounds=[None, None], root_exploration_fraction=0.25,
    value_support=[-15, 15], reward_support=[-15, 15], no_support=False, no_target_transform=False)
net = FCNetwork(D, A, "cuda", cfg)
net.load_weights(random_state_dict(D, A))
rng = np.random.default_rng(1)
obs = rng.random((G, D)).astype(np.float32)
noise, u, temp = rng.dirichlet([0.25] * A, size=G), rng.random(G), np.ones(G)
out = []
for fused in (False, True):
  fs = FCSearch(cfg, net, G, use_graph=False, num_streams=1, fused=fused)
  fs.enable_record()
  fs.search_host(obs, noise, u, temp)
  torch.cuda.synchronize()
  eng = fs.fused if fused else fs.eng
  out.append((fs, eng.export_game(game), [t.cpu().numpy() for t in fs.trace]))
(fa, ta, tra), (fb, tb, trb) = out
for s in range(S):
  a = [int(tra[i][s, game]) for i in range(3)]
  b = [int(trb[i][s, game]) for i in range(3)]
  if a != b:
    print("sim %d: per-launch (parent, action, depth) = %s, fused = %s" % (s, a, b))
for k in ("prior", "child", "vsum", "visit", "reward"):
  x, y = ta[k], tb[k]
  if not np.array_equal(x, y):
    bad = np.argwhere(x != y)
    print(k, "differs at", bad[:6].tolist(), "e.g.", x[tuple(bad[0])], y[tuple(bad[0])])
print("minmax", fa.minmax[game].tolist(), fb.minmax[game].tolist())
print("done")
