"""MuZeroNetwork value / reward supports wider than 32 bins: the tensor-core support head
(mz_conv_support_head_tc, csrc/mz_conv_tc.cu) against float64 arithmetic on the kernel's bf16 operands, the
whole network against the float32 oracle (oracle/muzero_ref.py) at the paper's Atari value support
[-300, 300], ConvSearch and the self-play driver on top of it, and the narrow (<= 32 bins) path left as it
was.  Every tolerance is stated next to the largest value measured on a B200."""
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

MZ_ERR_BAD_ARG, MZ_ERR_UNSUPPORTED = -1, -2


def _h_inv(x):  # Config.inverse_transform's h^-1 (config.py:27-33), float64
  eps = 0.001
  return np.sign(x) * (((np.sqrt(1 + 4 * eps * (np.abs(x) + 1 + eps)) - 1) / (2 * eps)) ** 2 - 1)


def _head_ref(hidden, w2, b2, support_min, no_tt):
  """float64 on the kernel's operands: hidden and W2 rounded to bf16, bias float32."""
  h = hidden.to(torch.bfloat16).double().cpu().numpy()
  w = w2.to(torch.bfloat16).double().cpu().numpy()
  logits = h @ w.T + b2.double().cpu().numpy()[None, :]
  p = np.exp(logits - logits.max(axis=1, keepdims=True))
  p /= p.sum(axis=1, keepdims=True)
  x = p @ (support_min + np.arange(w.shape[0], dtype=np.float64))
  return x if no_tt else _h_inv(x)


# (bins, support_min, no_target_transform, games, column offset in the 1536-wide fc buffer): every bin count,
# negative / positive / asymmetric supports, both transforms, ragged tiles and both head columns
HEAD_CASES = [(33, -16, 0, 1, 0), (33, 5, 1, 129, 512), (64, -10, 0, 127, 512), (64, 3, 1, 1000, 0),
              (65, -32, 1, 129, 0), (65, -20, 0, 1000, 512), (257, -128, 0, 1000, 0), (257, -100, 1, 127, 512),
              (601, -300, 0, 1000, 512), (601, -300, 1, 129, 0), (601, 0, 0, 127, 0), (1024, -512, 0, 1000, 0),
              (1024, -300, 1, 1, 512), (1024, 7, 0, 129, 512)]


# float32 softmax sums over up to 1024 terms: at most 1024 * 2^-24 = 6.1e-5 relative in the expectation (worst-case
# accumulation bound), which h^-1 at most doubles
HEAD_BAR = 1e-4


@pytest.mark.parametrize("bins,support_min,no_tt,games,col", HEAD_CASES)
def test_support_head_kernel_matches_float64(bins, support_min, no_tt, games, col):
  """Rows: random ReLU'd hidden layers, plus one row at each end of the support (its hidden vector is a large
  multiple of W2's first / last row, so the softmax is one-hot there) and, in a second launch with a constant
  bias, a zero row whose logits are all equal (expectation = the support's midpoint).  The other columns of
  the fc buffer hold NaN: the kernel reads only its 512.  Relative bar: |got - want| <= HEAD_BAR (|want| + max
  |support|), measured at most 1.1e-5 (at 1024 bins)."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  dev = "cuda"
  torch.manual_seed(bins * 7 + games + col)
  fc = torch.full((games, 1536), float("nan"), device=dev)
  w2 = torch.randn((bins, 512), device=dev) * 0.05
  hid = torch.relu(torch.randn((games, 512), device=dev))
  if games > 1:
    hid[games - 1] = 60.0 * w2[bins - 1]   # expectation at the top of the support
  if games > 2:
    hid[games // 2] = 60.0 * w2[0]         # ... and at the bottom
  hid[0] = 0.0
  fc[:, col:col + 512] = hid
  scale = max(abs(support_min), abs(support_min + bins - 1))
  worst = 0.0
  P = _lib.ptr
  w_bf = w2.to(torch.bfloat16).contiguous()  # the image MuZeroNetwork.load_weights packs
  for const_bias in (False, True):
    b2 = torch.full((bins,), 0.25, device=dev) if const_bias else torch.randn(bins, device=dev) * 0.1
    out = torch.full((games,), float("nan"), device=dev)
    args = (games, fc[:, col:].data_ptr(), 1536, P(w_bf), P(b2), bins, support_min, no_tt)
    _lib.check(lib.mz_conv_support_head_tc(*args, P(out), 1, _lib.current_stream()), "support head")
    again = torch.full_like(out, float("nan"))
    _lib.check(lib.mz_conv_support_head_tc(*args, P(again), 1, _lib.current_stream()), "support head")
    torch.cuda.synchronize()
    assert torch.equal(out, again)  # fixed reduction order: a rerun gives the same bits
    want = _head_ref(hid, w2, b2, support_min, no_tt)
    got = out.double().cpu().numpy()
    rel = np.abs(got - want) / (np.abs(want) + scale)
    worst = max(worst, float(rel.max()))
    ends = [(games - 1, support_min + bins - 1)] if games > 1 else []
    ends += [(games // 2, support_min)] if games > 2 else []
    for row, end in ends:  # one-hot softmax: the expectation is the support's end
      e = end if no_tt else _h_inv(np.float64(end))
      assert abs(got[row] - e) <= 1e-3 * (abs(e) + 1), (row, got[row], e)
    if const_bias:  # all logits equal in row 0
      mid = support_min + (bins - 1) / 2.0
      e = mid if no_tt else _h_inv(np.float64(mid))
      assert abs(got[0] - e) <= HEAD_BAR * (abs(e) + scale), (got[0], e)
  print("bins %d min %d no_tt %d games %d col %d: max relative error %.3g" % (bins, support_min, no_tt, games, col,
                                                                             worst))
  assert worst <= HEAD_BAR


def test_support_head_kernel_refusals():
  """33 to 1024 bins; narrower heads stay on mz_conv_head.  Misaligned hidden rows are rejected."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  dev = "cuda"
  fc = torch.zeros((4, 1536), device=dev)
  w = torch.zeros((1025, 512), dtype=torch.bfloat16, device=dev)
  b = torch.zeros(1025, device=dev)
  out = torch.zeros(4, device=dev)
  P, st = _lib.ptr, _lib.current_stream()
  for bins in (32, 1025):
    assert lib.mz_conv_support_head_tc(4, P(fc), 1536, P(w), P(b), bins, 0, 0, P(out), 1, st) == MZ_ERR_UNSUPPORTED
  assert lib.mz_conv_support_head_tc(4, fc[:, 1:].data_ptr(), 1536, P(w), P(b), 64, 0, 0, P(out), 1, st) == \
      MZ_ERR_BAD_ARG
  assert lib.mz_conv_support_head_tc(4, P(fc), 511, P(w), P(b), 64, 0, 0, P(out), 1, st) == MZ_ERR_BAD_ARG
  assert lib.mz_conv_support_head_tc(0, P(fc), 1536, P(w), P(b), 64, 0, 0, P(out), 1, st) == MZ_ERR_BAD_ARG


def _cfg(value, reward, **kw):
  c = types.SimpleNamespace(value_support=list(value), reward_support=list(reward), no_support=False,
                            no_target_transform=False, num_simulations=8, action_space=18, two_players=False,
                            discount=0.997, pb_c_base=19652, pb_c_init=1.25, init_value_score=0.0,
                            known_bounds=[None, None], root_exploration_fraction=0.25)
  c.__dict__.update(kw)
  return c


def _bins(s):
  return s[1] - s[0] + 1


def _h(v):  # Config.scalar_transform (config.py:51-54), the inverse of h^-1
  return np.sign(v) * (np.sqrt(np.abs(v) + 1) - 1) + 0.001 * v


def _support_err(got, logits, support):
  """Error of network scalars `got` against the float64 softmax expectation of the oracle's head `logits`, taken in
  support space (h(got); h undoes the h^-1 of inverse_transform).  Returned as (error / D, error) per row with
  D = sum_i p_i |s_i - x|, the softmax's mean absolute deviation over the support: a logit error of at most d moves
  the expectation by at most d * D (first order).  So error / D is the logit error the difference amounts to, and it
  is comparable across supports of any width.  A relative bar on the value itself cannot hold near zero: there the
  bf16 towers' logit error (~0.03) times D (~150 for a near-uniform softmax over 601 bins) is ~0.5 in support space
  however small the value."""
  l = logits.double().cpu().numpy()
  p = np.exp(l - l.max(axis=1, keepdims=True))
  p /= p.sum(axis=1, keepdims=True)
  sv = np.arange(support[0], support[1] + 1, dtype=np.float64)
  x = p @ sv
  dev = (p * np.abs(sv[None, :] - x[:, None])).sum(axis=1)
  err = np.abs(_h(got.double().cpu().numpy().ravel()) - x)
  return err / dev, err


def _tilted(sd, value, reward):
  """Seeded weights put both expectations near zero.  A bias ramp of 2 across each support moves the value towards
  the top of its support and the reward towards the bottom of its, so a value / reward mix-up changes signs."""
  sd = dict(sd)
  for key, sup, sign in (("prediction_head.fc_value_o.bias", value, 1.0), ("dynamics_head.fc2.bias", reward, -1.0)):
    sd[key] = sd[key] + sign * 2.0 * torch.linspace(0.0, 1.0, _bins(sup))
  return sd


# value / reward supports: both wide, swapped, and wide next to narrow
ARRANGEMENTS = [((-300, 300), (-20, 20)), ((-20, 20), (-300, 300)), ((-300, 300), (-15, 15))]
SUPPORT_ERR_BAR = 0.05  # in logit units (see _support_err); measured at most 0.0082 on a B200


@pytest.mark.parametrize("value,reward", ARRANGEMENTS)
def test_network_matches_oracle_at_wide_supports(value, reward):
  """initial_inference and recurrent_inference against the float32 oracle on the same seeded (bias-tilted) state
  dict.  Hidden states and logits keep the conv bars of test_gpu_muzero.py (0.06 worst / 0.01 mean, logits 0.15).
  Values and rewards: the support-space error is at most SUPPORT_ERR_BAR times the softmax's spread over the
  support (_support_err), and every value is positive and every reward negative, as in the oracle.  The value is
  also recomputed in float64 from the network's own fc1 output, at the head kernel's bar (HEAD_BAR): what separates it
  from the oracle comes from the bf16 towers, not from the head."""
  from model_based_rl_b200.muzero import MuZeroNetwork
  from oracle import muzero_ref
  C_in, A, B = 4, 18, 6
  sd = _tilted(muzero_ref.seeded_state_dict(C_in, A, 21, value_bins=_bins(value), reward_bins=_bins(reward)),
               value, reward)
  net = MuZeroNetwork(C_in, A, "cuda", _cfg(value, reward))
  net.load_weights(sd)
  sdc = {k: v.cuda() for k, v in sd.items()}
  gen = torch.Generator().manual_seed(8)
  obs = torch.rand((B, C_in, 96, 96), generator=gen)
  init = net.initial_inference(obs)
  torch.cuda.synchronize()
  fc1 = net.buffers(B)["fc"][:, 512:1024].clone()  # the value head's hidden layer of that call
  own = _head_ref(fc1, sd["prediction_head.fc_value_o.weight"], sd["prediction_head.fc_value_o.bias"], value[0], 0)
  own_err = float((np.abs(init.value.double().cpu().numpy().ravel() - own) / (np.abs(own) + max(map(abs, value)))).max())
  print("init_value vs float64 head on the network's own fc1: relative %.3g" % own_err)
  assert own_err <= HEAD_BAR
  with torch.no_grad():
    h0 = muzero_ref.representation(obs.cuda(), sdc)
    pol0, v0 = muzero_ref.prediction_logits(h0, sdc)
  actions = [int(a) for a in torch.randint(0, A, (B,), generator=gen)]
  rec = net.recurrent_inference(h0, actions)
  with torch.no_grad():
    h1, r1 = muzero_ref.dynamics_logits(h0, actions, sdc, A)
    pol1, v1 = muzero_ref.prediction_logits(h1, sdc)
  torch.cuda.synchronize()
  for name, got, want in (("init_hidden", init.hidden_state, h0), ("rec_hidden", rec.hidden_state, h1)):
    err = (got - want).abs()
    print(name, float(err.max()), float(err.mean()))
    assert float(err.max()) < 0.06 and float(err.mean()) < 0.01, name
  for name, got, want in (("init_logits", init.policy_logits, pol0), ("rec_logits", rec.policy_logits, pol1)):
    err = float((got - want).abs().max())
    print(name, err)
    assert err < 0.15, name
  for name, got, logits, sup, sign in (("init_value", init.value, v0, value, 1), ("rec_value", rec.value, v1, value, 1),
                                       ("rec_reward", rec.reward, r1, reward, -1)):
    ratio, err = _support_err(got, logits, sup)
    want = muzero_ref.inverse_transform(logits.double(), *sup)
    print(name, "support-space error %.3g (%.3g logit units), values %s, oracle %s" % (
        err.max(), ratio.max(), np.round(got.cpu().numpy().ravel(), 2), np.round(want.cpu().numpy().ravel(), 2)))
    assert ratio.max() <= SUPPORT_ERR_BAR, (name, ratio.max())
    assert (np.sign(want.cpu().numpy()) == sign).all() and (np.sign(got.cpu().numpy()) == sign).all(), name


class _CallLog(object):
  """Records which C entries a network calls."""

  def __init__(self, lib):
    self._lib, self.called = lib, set()

  def __getattr__(self, name):
    self.called.add(name)
    return getattr(self._lib, name)


@pytest.mark.parametrize("value,reward,wide", [((-15, 15), (-15, 15), False), ((-300, 300), (-15, 15), True),
                                               ((-15, 15), (-20, 20), True)])
def test_head_kernel_selection(value, reward, wide):
  """31-bin heads (the benchmark's C5) never reach the new entry; a head above 32 bins always does."""
  from model_based_rl_b200.muzero import MuZeroNetwork, random_state_dict
  net = MuZeroNetwork(4, 6, "cuda", _cfg(value, reward))
  net.load_weights(random_state_dict(4, 6, value_bins=_bins(value), reward_bins=_bins(reward)))
  net.lib = log = _CallLog(net.lib)
  init = net.initial_inference(torch.rand((2, 4, 96, 96)))
  net.recurrent_inference(init.hidden_state, [1, 2])
  torch.cuda.synchronize()
  assert ("mz_conv_support_head_tc" in log.called) == wide
  assert "mz_conv_head" in log.called  # the policy head, and any narrow support


def test_load_weights_refuses_more_than_1024_bins():
  from model_based_rl_b200.muzero import MuZeroNetwork, random_state_dict
  net = MuZeroNetwork(4, 6, "cuda", _cfg((-512, 512), (-5, 5)))
  with pytest.raises(ValueError, match="1024"):
    net.load_weights(random_state_dict(4, 6, value_bins=1025, reward_bins=11))
  assert net._state is None  # refused before anything was copied or packed


def test_conv_search_wide_value_support_replays_bit_exact_in_oracle():
  """A ConvSearch move with the 601-bin value support (reward [-20, 20]), eager and as a CUDA graph: the oracle
  replays the search from the recorded network outputs and reproduces parents, actions, visit counts and root
  values bit for bit.  The recorded values and rewards along game 0's path are checked against the float32 oracle
  network (same bar as test_network_matches_oracle_at_wide_supports)."""
  import oracle
  from oracle import muzero_ref
  from model_based_rl_b200.muzero import ConvSearch, MuZeroNetwork, from_padded
  C_in, A, G, S = 4, 18, 7, 12
  value, reward = (-300, 300), (-20, 20)
  cfg = _cfg(value, reward, num_simulations=S)
  sd = muzero_ref.seeded_state_dict(C_in, A, 99, value_bins=601, reward_bins=41)
  net = MuZeroNetwork(C_in, A, "cuda", cfg)
  net.load_weights(sd)
  rng = np.random.default_rng(3)
  obs = torch.from_numpy(rng.random((G, C_in, 96, 96)).astype(np.float32))
  noise = rng.dirichlet([0.25] * A, size=G)
  u, temp = rng.random(G), rng.choice([0.0, 1.0], size=G)
  for use_graph in (False, True):
    cs = ConvSearch(cfg, net, G, use_graph=use_graph)
    cs.enable_record()
    actions, root_value, child_visits, init_value = cs.search(obs, noise, u, temp)
    torch.cuda.synchronize()
    ocfg = oracle.make_cfg(S, A, False, 0.997)
    want = oracle.search(ocfg, cs.root_logits.cpu().numpy(), noise=noise, noise_frac=0.25,
                         rec_value=cs.record[0].cpu().numpy().T, rec_reward=cs.record[1].cpu().numpy().T,
                         rec_logits=cs.record[2].cpu().numpy().transpose(1, 0, 2))
    assert np.array_equal(cs.trace[0].cpu().numpy().T, want["trace_parent"])
    assert np.array_equal(cs.trace[1].cpu().numpy().T, want["trace_action"])
    assert np.array_equal(cs.eng.visits.cpu().numpy(), want["visits"])
    assert np.array_equal(root_value.cpu().numpy(), want["root_value"])
    for i in range(G):
      assert int(actions[i]) == oracle.select_action(want["visits"][i], temp[i], u[i])
  sdc = {k: v.cuda() for k, v in sd.items()}
  pool = cs.pool.view(G, S + 1, 49, 128)
  parents, acts = cs.trace[0].cpu().numpy()[:, 0], cs.trace[1].cpu().numpy()[:, 0]
  worst = [0.0, 0.0]
  for sim in range(S):
    h = from_padded(pool[0, int(parents[sim])].reshape(49, 128), 1)
    with torch.no_grad():
      h2, r = muzero_ref.dynamics_logits(h, [int(acts[sim])], sdc, A)
      _, v = muzero_ref.prediction_logits(h2, sdc)
    for k, (got, logits, sup) in enumerate(((cs.record[0][sim, :1], v, value), (cs.record[1][sim, :1], r, reward))):
      worst[k] = max(worst[k], float(_support_err(got, logits, sup)[0].max()))
  print("recorded value / reward vs oracle, support-space error in logit units:", worst)
  assert max(worst) <= SUPPORT_ERR_BAR


def test_selfplay_driver_through_conv_search_at_wide_supports():
  """One BatchedActor(search=ConvSearch) move at value [-300, 300] / reward [-20, 20]: what the actor returns is
  what the engine searched, and the oracle replays that search bit for bit."""
  import oracle
  from oracle import muzero_ref
  from model_based_rl_b200.environments import SyntheticFrames
  from model_based_rl_b200.muzero import ConvSearch, MuZeroNetwork
  from model_based_rl_b200.selfplay import BatchedActor
  C_in, A, G, S = 4, 6, 5, 6
  cfg = _cfg((-300, 300), (-20, 20), num_simulations=S, action_space=A, root_dirichlet_alpha=0.25,
             num_unroll_steps=2, td_steps=2, max_history_length=3, max_steps=100, norm_obs=False)
  net = MuZeroNetwork(C_in, A, "cuda", cfg)
  net.load_weights(muzero_ref.seeded_state_dict(C_in, A, 7, value_bins=601, reward_bins=41))
  cs = ConvSearch(cfg, net, G)
  cs.enable_record()
  actor = BatchedActor(cfg, net, SyntheticFrames(G, A, (C_in, 96, 96), episode_length=4, seed=11), search=cs)
  rng = np.random.default_rng(5)
  noise, u = rng.dirichlet([0.25] * A, size=G), rng.random(G)
  actions, root_value, child_visits, _, _ = actor.play_move(noise=noise, uniforms=u)
  want = oracle.search(oracle.make_cfg(S, A, False, 0.997), cs.root_logits.cpu().numpy(), noise=noise,
                       noise_frac=0.25, rec_value=cs.record[0].cpu().numpy().T,
                       rec_reward=cs.record[1].cpu().numpy().T,
                       rec_logits=cs.record[2].cpu().numpy().transpose(1, 0, 2))
  assert np.array_equal(cs.eng.visits.cpu().numpy(), want["visits"])
  assert np.array_equal(root_value, want["root_value"])
  for i in range(G):
    assert int(actions[i]) == oracle.select_action(want["visits"][i], 1.0, u[i])
  assert np.allclose(child_visits.sum(1), 1.0)
  assert actor.experiences_collected == G


def test_conv_search_after_load_weights_at_wide_supports():
  """At 601-bin value and reward supports, a second load_weights changes the next move's outputs: the captured
  graph (which holds the wide head's packed W2) is re-captured, and the move equals an engine built after the
  load."""
  from model_based_rl_b200.muzero import ConvSearch, MuZeroNetwork, random_state_dict
  G, A, S, C_in = 8, 6, 4, 4
  cfg = _cfg((-300, 300), (-300, 300), num_simulations=S, action_space=A)
  rng = np.random.default_rng(4)
  obs = torch.from_numpy(rng.random((G, C_in, 96, 96), dtype=np.float32))
  noise, u, temp = rng.dirichlet([0.25] * A, size=G), rng.random(G), np.ones(G)
  net = MuZeroNetwork(C_in, A, "cuda", cfg)
  net.load_weights(random_state_dict(C_in, A, value_bins=601, reward_bins=601, seed=1))
  cs = ConvSearch(cfg, net, G, use_graph=True)
  first = [t.clone() for t in cs.search(obs, noise, u, temp)]
  sd2 = random_state_dict(C_in, A, value_bins=601, reward_bins=601, seed=2)
  net.load_weights(sd2)
  second = [t.clone() for t in cs.search(obs, noise, u, temp)]
  fresh = MuZeroNetwork(C_in, A, "cuda", cfg)
  fresh.load_weights(sd2)
  want = [t.clone() for t in ConvSearch(cfg, fresh, G, use_graph=False).search(obs, noise, u, temp)]
  torch.cuda.synchronize()
  assert not torch.equal(first[3], second[3])
  assert not torch.equal(first[1], second[1])
  for x, y in zip(second, want):
    assert torch.equal(x, y)
