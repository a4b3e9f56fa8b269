"""The persistent search kernel's expansion + backup against the per-launch search, bit for bit, on the shapes that
reach each of its paths: every actions-per-lane instantiation, paths deeper than 32 positions (the backup's second
chunk), two players with known bounds, logits outside the exp table's range (the general exp routine), a ragged
last tile and the largest tree the kernel takes per action band."""
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _cfg(S, A, two, bounds):
  return types.SimpleNamespace(
      num_simulations=S, action_space=A, two_players=two, discount=0.997, pb_c_base=19652, pb_c_init=1.25,
      init_value_score=0.0, known_bounds=list(bounds), root_exploration_fraction=0.25, value_support=[-15, 15],
      reward_support=[-15, 15], no_support=False, no_target_transform=False)


def _largest_s(A):
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  return max(S for S in range(1, 64) if lib.mz_fc_search_supported(S, A))


def _compare(G, A, S, D=16, two=False, bounds=(None, None), policy=None, seed=3):
  """Runs one move on both engines and asserts identical network records, traces, results and trees; returns the
  fused engine's (depth trace, recorded logits)."""
  from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict
  cfg = _cfg(S, A, two, bounds)
  net = FCNetwork(D, A, "cuda", cfg)
  sd = random_state_dict(D, A, seed=seed)
  if policy is not None:
    policy(sd)
  net.load_weights(sd)
  rng = np.random.default_rng(seed)
  obs = rng.normal(size=(G, D)).astype(np.float32)
  noise = rng.dirichlet([0.25] * A, size=G)
  to_play = rng.choice([-1, 1], size=G).astype(np.int8) if two else None
  u, temp = rng.random(G), rng.choice([0.0, 1.0], size=G)
  outs = []
  for fused in (False, True):
    fs = FCSearch(cfg, net, G, use_graph=False, num_streams=1, fused=fused)
    assert (fs.fused is not None) == fused
    fs.enable_record()
    r = fs.search_host(obs, noise, u, temp, to_play=to_play)
    torch.cuda.synchronize()
    if fused:
      assert int(fs.fused.error_flag.item()) == 0
    eng = fs.fused if fused else fs.eng
    outs.append(dict(result=[t.clone() for t in r], visits=fs.visits.cpu(), minmax=fs.minmax.cpu(),
                     record=[t.cpu() for t in fs.record], trace=[t.cpu() for t in fs.trace],
                     trees=[eng.export_game(g) for g in (0, G // 2, G - 1)]))
  a, b = outs
  for name, x, y in zip(("value", "reward", "logits"), a["record"], b["record"]):
    assert torch.equal(x, y), "network %s differs" % name
  for name, x, y in zip(("parent", "action", "depth"), a["trace"], b["trace"]):
    assert torch.equal(x, y), "trace %s differs" % name
  for name, x, y in zip(("actions", "root_value", "child_visits", "init_value"), a["result"], b["result"]):
    assert torch.equal(x, y), name
  assert torch.equal(a["visits"], b["visits"]) and torch.equal(a["minmax"], b["minmax"])
  for ta, tb in zip(a["trees"], b["trees"]):
    for k in ("prior", "child", "vsum", "visit", "reward"):
      assert np.array_equal(ta[k], tb[k]), "tree %s differs" % k
  return b["trace"][2], b["record"][2]


@pytest.mark.parametrize("A", [8, 9, 16, 17, 24, 25, 32])
def test_each_actions_per_lane_instantiation(A):
  _compare(G=300, A=A, S=min(30, _largest_s(A)))


@pytest.mark.parametrize("A,two", [(1, False), (1, True), (2, False)])
def test_paths_deeper_than_32_positions(A, two):
  # one action: every simulation extends the same chain, so depth reaches S; two: deep paths of a binary tree
  depth, _ = _compare(G=150, A=A, S=63, two=two, bounds=(-1, 1) if two else (None, None))
  if A == 1:
    assert int(depth.max()) == 63


def test_two_players_known_bounds():
  _compare(G=130, A=9, S=30, two=True, bounds=(-1, 1))


def test_logits_outside_the_exp_table_range():
  def policy(sd):  # logits around -600: |x| >= 512 takes the general exp routine
    sd["policy_head.policy.weight"] = sd["policy_head.policy.weight"] * 100
    sd["policy_head.policy.bias"] = sd["policy_head.policy.bias"] * 0 - 600
  _, logits = _compare(G=200, A=18, S=20, policy=policy)
  assert float(logits.abs().max()) >= 512.0


@pytest.mark.parametrize("A", [4, 8, 13, 16, 18, 24, 32])
def test_largest_tree_per_action_band(A):
  _compare(G=129, A=A, S=_largest_s(A))
