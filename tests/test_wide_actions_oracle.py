"""Search checkers past 32 actions, on the CPU: the C oracle (oracle/mz_oracle.c, written for up to 64 actions)
against the pure-Python port of the reference's search (oracle/search_ref.py) at 33, 50 and 64 actions, bit for bit,
beyond the goldens (which stop at 18 actions); the port on legal subsets that span both mask words; and the
host-side conversion of legal masks into the kernels' word layout."""
import numpy as np
import pytest

import oracle
import wide_ref

HK = dict(value_scale=1.0, reward_scale=0.5, logit_scale=2.0, reward_density=3)
EXACT = ("visits", "trace_parent", "trace_action", "trace_depth", "root_value", "minmax")


def _cfg(S, A, two_players=False, known_bounds=(None, None)):
  return dict(num_simulations=S, action_space=A, two_players=two_players, discount=1.0 if two_players else 0.997,
              pb_c_base=19652, pb_c_init=1.25, init_value_score=0.0, known_bounds=tuple(known_bounds))


def _hash_roots(rng, G, A, hk):
  from model_based_rl_b200.testing import HashNetwork
  import torch
  root_state = rng.integers(0, 2**63 - 1, size=G, dtype=np.int64)
  init = HashNetwork(A, **hk).initial_inference(torch.from_numpy(root_state).view(G, 1))
  return root_state, init.policy_logits.numpy()


@pytest.mark.parametrize("A", [33, 50, 64])
@pytest.mark.parametrize("kind", ["one_player", "two_players_bounds", "zero_policy"])
def test_c_oracle_matches_python_port(A, kind):
  """Every root action legal (the C oracle reads legal masks only up to 32 actions), noise on the roots."""
  rng = np.random.default_rng(A * 7 + len(kind))
  G, S = 6, 40
  two, bounds = kind == "two_players_bounds", ((-1.0, 1.0) if kind == "two_players_bounds" else (None, None))
  hk = dict(HK, logit_scale=0.0) if kind == "zero_policy" else HK
  cfg = _cfg(S, A, two, bounds)
  root_state, logits = _hash_roots(rng, G, A, hk)
  noise = None if kind == "zero_policy" else rng.dirichlet([0.25] * A, size=G)
  to_play = rng.choice([-1, 1], size=G).astype(np.int8) if two else None
  want = oracle.search(oracle.make_cfg(**cfg), logits, noise=noise, root_to_play=to_play,
                       hashnet=oracle.HashNet(*[hk[k] for k in ("value_scale", "reward_scale", "logit_scale",
                                                                  "reward_density")]),
                       root_state=root_state.astype(np.uint64))
  got = wide_ref.port_search(cfg, logits, noise=noise, to_play=to_play, hashnet=hk, root_state=root_state)
  for k in EXACT:
    assert np.array_equal(got[k], want[k]), k
  assert np.array_equal(got["child_visits"], want["visits"] / want["visits"].sum(1, keepdims=True))
  if kind == "zero_policy":  # equal priors everywhere: the first descent takes the largest action
    assert (want["trace_action"][:, 0] == A - 1).all()


@pytest.mark.parametrize("A", [33, 64])
def test_c_oracle_replay_matches_python_port(A):
  """Recorded network outputs replayed by both checkers (how the FCNetwork searches are checked)."""
  rng = np.random.default_rng(A)
  G, S = 5, 30
  cfg = _cfg(S, A)
  logits = rng.normal(size=(G, A)).astype(np.float32)
  rec_value = rng.normal(size=(G, S)).astype(np.float32)
  rec_reward = np.where(rng.random((G, S)) < 0.3, rng.normal(size=(G, S)), 0).astype(np.float32)
  rec_logits = rng.normal(size=(G, S, A)).astype(np.float32)
  want = oracle.search(oracle.make_cfg(**cfg), logits, rec_value=rec_value, rec_reward=rec_reward,
                       rec_logits=rec_logits)
  got = wide_ref.port_search(cfg, logits, rec_value=rec_value, rec_reward=rec_reward, rec_logits=rec_logits)
  for k in EXACT:
    assert np.array_equal(got[k], want[k]), k


@pytest.mark.parametrize("A", [33, 50, 64])
def test_python_port_on_legal_subsets_of_both_words(A):
  """Legal subsets with actions in both mask words, and roots whose legal actions all lie above 32: illegal actions
  are never searched, every simulation lands below a legal root action."""
  rng = np.random.default_rng(100 + A)
  G, S = 6, 30
  legal = wide_ref.random_legal(rng, G, A, only_high_rows=(1, 2))
  root_state, logits = _hash_roots(rng, G, A, HK)
  got = wide_ref.port_search(_cfg(S, A, True, (-1.0, 1.0)), logits, legal, wide_ref.dense_noise(rng, legal),
                             to_play=np.ones(G, np.int8), hashnet=HK, root_state=root_state)
  assert (got["visits"][~legal] == 0).all() and (got["visits"].sum(1) == S).all()
  first = got["trace_action"][got["trace_parent"] == 0]
  assert first.min() >= 0
  for g in (1, 2):
    assert (got["trace_action"][g][got["trace_parent"][g] == 0] >= 32).all()
  # a mask with every action legal is no mask
  full = wide_ref.port_search(_cfg(S, A), logits, np.ones((G, A), bool), hashnet=HK, root_state=root_state)
  none = wide_ref.port_search(_cfg(S, A), logits, None, hashnet=HK, root_state=root_state)
  for k in EXACT:
    assert np.array_equal(full[k], none[k])


@pytest.mark.parametrize("A", [9, 32, 33, 50, 64])
def test_legal_words_layout(A):
  """mcts.legal_words: Python ints, int64 / uint64 arrays (bit 63 = action 63), bool [G, A] and [G, W] words all give
  the kernels' layout (bit b of word w <=> action 32 w + b); up to 32 actions the old int32 conversion."""
  from model_based_rl_b200.mcts import legal_words
  rng = np.random.default_rng(A)
  G, W = 7, (A + 31) // 32
  legal = wide_ref.random_legal(rng, G, A)
  ints = [sum(1 << int(a) for a in np.nonzero(row)[0]) for row in legal]
  want = np.zeros((G, W), np.uint32)
  for g in range(G):
    for w in range(W):
      want[g, w] = (ints[g] >> (32 * w)) & 0xffffffff
  want = want.view(np.int32)
  forms = [ints, np.array(ints, np.uint64), np.array(ints, np.uint64).view(np.int64), legal, legal.tolist(), want]
  for form in forms:
    got = legal_words(form, G, A)
    assert got.dtype == np.int32 and np.array_equal(got, want)
  if A <= 32:
    assert np.array_equal(np.asarray(ints).astype(np.int64).astype(np.int32), want[:, 0])
  with pytest.raises(ValueError):
    legal_words(legal[:, :-1], G, A)
