"""GPU parity tests for the tree kernels (run with -m gpu on the B200 box).

Bar (north_star): visit counts, selected actions and the per-simulation (parent, action, depth)
trace are BIT-EXACT against the reference (golden vectors from the unmodified mcts.py) and against
the CPU oracle on larger seeded inputs; root values within 1e-5 relative (they come out bit-exact
whenever the paths agree, because value sums only combine network outputs).
"""
import ctypes as C
import types

import numpy as np
import pytest
import torch

import oracle
from helpers import SEARCH_CASES, load, oracle_search_from_golden, search_case_cfg

pytestmark = pytest.mark.gpu


def _cfg_ns(d):
  return types.SimpleNamespace(**d)


def _engine_from_golden(g, trace=True):
  from model_based_rl_b200.mcts import BatchedMCTS
  cfg = _cfg_ns(search_case_cfg(g))
  G = len(g["root_state"])
  eng = BatchedMCTS(cfg, G, hidden_words=2, prior_sum_mode=int(g["py_sum_mode"]))
  if trace:
    eng.enable_trace()
  return eng, cfg, G


def _hashnet(g):
  from model_based_rl_b200.testing import HashNetwork
  hv = g["hashnet"]
  return HashNetwork(int(g["action_space"]), float(hv[0]), float(hv[1]), float(hv[2]), int(hv[3]),
                     device="cuda")


def _run_golden(g):
  eng, cfg, G = _engine_from_golden(g)
  net = _hashnet(g)
  state = torch.from_numpy(g["root_state"].astype(np.int64)).view(G, 1).cuda()
  noise = g["noise"] if int(g["use_noise"]) else None
  res = eng.search(net, g["root_logits"], state, legal_mask=g["legal"].astype(np.int64), noise=noise,
                   noise_frac=float(g["noise_frac"]), to_play=g["to_play"])
  torch.cuda.synchronize()
  return eng, res


@pytest.fixture(params=["wide", "wide_1_game_per_cta"])
def step_kernel(request):
  """The step kernel runs four games per CTA or one (the choice large launches get,
  mz_tree_set_games_per_block): run the parity tests through both, since the golden batches are too small to
  reach one game per CTA by launch size."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  lib.mz_tree_set_games_per_block(1 if request.param == "wide_1_game_per_cta" else 4)
  yield request.param
  lib.mz_tree_set_games_per_block(0)


@pytest.mark.parametrize("case", SEARCH_CASES)
def test_search_matches_reference_golden(case, step_kernel):
  g = load("search_" + case)
  eng, res = _run_golden(g)
  assert np.array_equal(res.visits.cpu().numpy(), g["visits"])
  assert np.array_equal(res.trace_parent.cpu().numpy().T, g["trace_parent"])
  assert np.array_equal(res.trace_action.cpu().numpy().T, g["trace_action"])
  assert np.array_equal(res.trace_depth.cpu().numpy().T, g["trace_depth"])
  rv = res.root_value.cpu().numpy()
  assert np.allclose(rv, g["root_value"], rtol=1e-5, atol=0)  # stated tolerance
  assert np.array_equal(rv, g["root_value"])                    # and in fact bit-exact
  assert np.array_equal(res.minmax.cpu().numpy(), g["minmax"])
  want_cv = g["visits"] / g["visits"].sum(1, keepdims=True)
  assert np.array_equal(res.child_visits.cpu().numpy(), want_cv)
  # whole tree of every game
  exact = total = 0
  for gi in range(len(g["root_state"])):
    t = eng.export_game(gi)
    child = np.where(g["edge_child"][gi] == -2, -2, g["edge_child"][gi])
    assert np.array_equal(t["child"], child)
    # node-centric stats on the device <-> edge-centric stats in the golden dump
    for n in range(t["child"].shape[0]):
      for a in range(t["child"].shape[1]):
        c = t["child"][n, a]
        if c >= 0:
          assert t["visit"][c] == g["edge_visit"][gi, n, a]
          assert t["vsum"][c] == g["edge_vsum"][gi, n, a]
          assert np.float64(t["reward"][c]) == g["edge_reward"][gi, n, a]
        else:
          assert g["edge_visit"][gi, n, a] == 0
    legal = g["edge_child"][gi] != -2
    p, q = t["prior"][legal], g["edge_prior"][gi][legal]
    # device exp() (csrc/mz_exp_algo.h, the restatement of glibc's algorithm) + Neumaier sum + IEEE division:
    # every prior of every node is bit-identical to what the reference computed with math.exp / sum() / '/'
    assert np.array_equal(p, q), "priors differ in %d of %d entries" % (int((p != q).sum()), p.size)
    exact += int((p == q).sum())
    total += p.size
  print("priors bit-exact: %d / %d" % (exact, total))


def _random_case(G, A, S, two_players, seed, known_bounds=(None, None), legal_subsets=False):
  rng = np.random.default_rng(seed)
  cfg = dict(num_simulations=S, action_space=A, two_players=two_players,
             discount=1.0 if two_players else 0.997, pb_c_base=19652, pb_c_init=1.25,
             init_value_score=0.0, known_bounds=list(known_bounds))
  root_state = rng.integers(0, 2**63 - 1, size=G, dtype=np.int64)
  legal = (rng.integers(1, 2**A, size=G, dtype=np.int64) if legal_subsets else
           np.full(G, (1 << A) - 1, np.int64))
  noise = np.zeros((G, A))
  for i in range(G):
    n = bin(int(legal[i])).count("1")
    noise[i, :n] = rng.dirichlet([0.25] * n)
  to_play = rng.choice([-1, 1], size=G).astype(np.int8) if two_players else np.ones(G, np.int8)
  return cfg, root_state, legal, noise, to_play


def _run_engine_vs_oracle(G, A, S, two_players, seed, fused, **kw):
  from model_based_rl_b200.mcts import BatchedMCTS
  from model_based_rl_b200.testing import HashNetwork
  cfg, root_state, legal, noise, to_play = _random_case(G, A, S, two_players, seed, **kw)
  hk = dict(value_scale=1.0, reward_scale=0.5, logit_scale=2.0, reward_density=3)
  net = HashNetwork(A, device="cuda", **hk)
  state = torch.from_numpy(root_state).view(G, 1).cuda()
  init = net.initial_inference(state)
  eng = BatchedMCTS(_cfg_ns(cfg), G, hidden_words=2)
  eng.enable_trace()
  if not fused:
    res = eng.search(net, init.policy_logits, state, legal_mask=legal, noise=noise, noise_frac=0.25,
                     to_play=to_play)
  else:  # fused step kernel: backup(s) + descent(s+1) in one launch
    eng.set_root(init.policy_logits, legal, noise, 0.25, to_play, state)
    eng.step(-1, gather=True)
    for sim in range(S):
      out = net.recurrent_inference(eng.gathered.view(torch.int64).view(G, 1), eng.leaf_action)
      eng.step(sim, out.value.reshape(G).contiguous(), out.reward.reshape(G).contiguous(),
               out.policy_logits.contiguous(), eng._hidden_words(out.hidden_state), gather=True)
    eng.root_stats()
    from model_based_rl_b200.mcts import SearchResult
    res = SearchResult(eng.visits, eng.child_visits, eng.root_value, eng.minmax, *eng.trace)
  torch.cuda.synchronize()
  ocfg = oracle.make_cfg(**cfg)
  want = oracle.search(ocfg, init.policy_logits.cpu().numpy(), legal_mask=legal.astype(np.uint32),
                       noise=noise, noise_frac=0.25, root_to_play=to_play,
                       hashnet=oracle.HashNet(1.0, 0.5, 2.0, 3), root_state=root_state.astype(np.uint64))
  return res, want


@pytest.mark.parametrize("G,A,S,two,fused,kw", [
    (512, 18, 50, False, False, {}),
    (512, 18, 50, False, True, {}),
    (777, 4, 50, False, True, {}),
    (300, 9, 30, True, False, dict(known_bounds=(-1.0, 1.0), legal_subsets=True)),
    (300, 9, 30, True, True, dict(known_bounds=(-1.0, 1.0), legal_subsets=True)),
    (65, 32, 20, False, True, {}),
    (33, 1, 10, False, True, {}),
    (129, 6, 64, True, True, {}),
    # warp-per-game kernel (17..32 actions): one game, two players + known bounds + legal subsets,
    # long searches (paths deeper than one 32-lane chunk, non-staged fallback for big trees)
    (1, 18, 50, False, True, {}),
    (200, 20, 100, True, True, dict(known_bounds=(-1.0, 1.0), legal_subsets=True)),
    (37, 17, 200, False, True, {}),
    (3, 32, 700, True, True, {}),
])
def test_search_matches_oracle_seeded(G, A, S, two, fused, kw, step_kernel):
  res, want = _run_engine_vs_oracle(G, A, S, two, 1234 + A, fused, **kw)
  assert np.array_equal(res.visits.cpu().numpy(), want["visits"])
  assert np.array_equal(res.trace_parent.cpu().numpy().T, want["trace_parent"])
  assert np.array_equal(res.trace_action.cpu().numpy().T, want["trace_action"])
  assert np.array_equal(res.trace_depth.cpu().numpy().T, want["trace_depth"])
  assert np.array_equal(res.root_value.cpu().numpy(), want["root_value"])
  assert np.array_equal(res.minmax.cpu().numpy(), want["minmax"])


def test_full_size_properties():
  """BASELINE size (4096 games x 50 sims, A=18): size-independent invariants + oracle on a slice."""
  G, A, S = 4096, 18, 50
  res, want = _run_engine_vs_oracle(G, A, S, False, 99, True)
  v = res.visits.cpu().numpy()
  assert (v.sum(1) == S).all()           # every simulation adds exactly one visit below the root
  assert (v >= 0).all()
  depth = res.trace_depth.cpu().numpy()
  assert depth.min() >= 1 and depth.max() <= S
  assert (res.trace_parent.cpu().numpy() <= np.arange(S)[:, None]).all()  # parents precede children
  cv = res.child_visits.cpu().numpy()
  assert np.allclose(cv.sum(1), 1.0, rtol=0, atol=1e-12)
  assert np.array_equal(v, want["visits"])  # the C oracle finishes this size in seconds
  assert np.array_equal(res.root_value.cpu().numpy(), want["root_value"])


def test_select_action_matches_reference_golden():
  from model_based_rl_b200.mcts import BatchedMCTS
  g = load("select_action")
  for A in (4, 9, 18):
    rows = np.where(g["A"] == A)[0]
    cfg = _cfg_ns(dict(num_simulations=2, action_space=A, two_players=False, discount=1.0,
                       pb_c_base=19652, pb_c_init=1.25, init_value_score=0.0,
                       known_bounds=[None, None]))
    eng = BatchedMCTS(cfg, len(rows))
    visits = torch.from_numpy(g["visits"][rows][:, :A].copy()).cuda()
    act = eng.select_action(g["temperature"][rows], g["u"][rows],
                            legal_mask=g["legal"][rows].astype(np.int64), visits=visits)
    torch.cuda.synchronize()
    assert np.array_equal(act.cpu().numpy(), g["action"][rows])


def test_mcts_run_dropin_b1():
  """`MCTS(config).run(root, network)` with a host-built root, as actors.py:132-147 does."""
  from model_based_rl_b200.mcts import MCTS, Node
  g = load("search_ttt")
  cfg = _cfg_ns(search_case_cfg(g))
  net = _hashnet(g)
  for gi in (0, 1, 5):
    state = torch.tensor([[int(g["root_state"][gi])]], dtype=torch.int64, device="cuda")
    init = net.initial_inference(state)
    legal = [a for a in range(cfg.action_space) if (int(g["legal"][gi]) >> a) & 1]
    root = Node(0)
    root.expand(init, int(g["to_play"][gi]), legal)
    real = np.random.dirichlet
    np.random.dirichlet = lambda alpha: g["noise"][gi, :len(alpha)].copy()
    try:
      root.add_exploration_noise(0.25, float(g["noise_frac"]))
    finally:
      np.random.dirichlet = real
    engine = MCTS(cfg)
    paths = engine.run(root, net)
    assert len(paths) == cfg.num_simulations
    assert [len(p) - 1 for p in paths] == list(g["trace_depth"][gi])
    for a in legal:
      assert root.children[a].visit_count == g["visits"][gi, a]
      assert root.children[a].prior == g["edge_prior"][gi, 0, a]  # host expansion: libm exp
    assert root.value() == g["root_value"][gi]
    assert root.visit_count == cfg.num_simulations
    assert (engine.min_max_stats.minimum, engine.min_max_stats.maximum) == tuple(g["minmax"][gi])
    # walking the tree after the search (evaluate.py:306-326)
    s_last = paths[-1]
    assert s_last[0] is root and s_last[-1].expanded() and s_last[-1].visit_count == 1
    node = root
    for step in range(len(s_last) - 1):
      assert s_last[step + 1] in node.children.values()
      node = s_last[step + 1]


def test_fast_division_is_ieee_division():
  """The descent divides by the per-descent constant (max - min) through a reciprocal + two fma
  correction steps; the result must be the correctly rounded quotient, bit for bit."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  cnt = torch.zeros(2, dtype=torch.int64, device="cuda")
  for seed in (1, 2, 3, 4):
    _lib.check(lib.mz_debug_div_check(seed, 148 * 16, 1 << 12, C.c_void_p(cnt.data_ptr()),
                                      C.c_void_p(cnt.data_ptr() + 8), _lib.current_stream()), "div")
  torch.cuda.synchronize()
  bad, tested = cnt.cpu().tolist()
  print("pairs tested", tested, "mismatches", bad)
  assert tested > 3_000_000_000 and bad == 0
