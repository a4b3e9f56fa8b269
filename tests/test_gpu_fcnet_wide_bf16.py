"""The bf16 FCNetwork kernels' wide head geometry: more than 32 actions or supports of more than 32 bins, up to 64.

Kernels against the float64 reference's bf16 emulation at the bar of tests/test_gpu_fcnet_shapes.py (2e-3 of the
largest entry of each output; value and reward in support space), with both recurrent modes bit for bit; negative
controls in the upper half of the widened heads; the sizing entry point and the C ABI's limits (without a GPU); and
the layers above the kernel -- search, self-play and the learner's weight hand-off -- at 64 actions in bf16.
Measured on a B200 (1000 W power limit), against the bar of 2e-3: the largest error is 8.6e-4 of the largest entry
(a46_obs1 recurrent value, h' forced) and 4.7e-4 for h' and reward.  The float64 emulation run end to end differs
from the same emulation fed the kernel's h' by up to 5.8e-3 (a33 initial value): the rounding flips `_rows` removes.
"""
import ctypes as C
import functools
import types

import numpy as np
import pytest
import torch

import oracle
from model_based_rl_b200 import _lib
from test_gpu_fcnet_shapes import (Cfg, _expected_initial_kernel, _failures, _initial, _initial_kernel_name, _inputs,
                                   _network, _recurrent, _recurrent_both_splits, _ref, _refs, _report, _state_dict, h64)
from test_gpu_wide_actions import (_cfg, _ns, test_device_actor_64_actions_fills_the_replay_like_the_list_path as
                                   _device_actor_64, test_fc_search_64_actions_replays_bit_exact as _search_64,
                                   _learner_case)

BF16 = ("bf16",)
# k1 (the dynamics layer's padded K) is 96 for A 30..45, 112 for A 46..61 and 128 for A 62..64; the logits staging
# area outgrows the h' staging from A = 52 on
WIDE = {
    "a33": Cfg(16, 33, (-15, 15), (-10, 10), False, BF16),
    "a45_nott": Cfg(8, 45, (-20, 12), (-31, 31), True, BF16),
    "a46_obs1": Cfg(1, 46, (-31, 32), (-16, 16), False, BF16),
    "a50": Cfg(40, 50, (-15, 15), (-31, 32), False, BF16),
    "a61_obs192": Cfg(192, 61, (-16, 16), (-12, 12), True, BF16),
    "a62_one_bin": Cfg(24, 62, (0, 0), (-31, 32), False, BF16),
    "a64_obs191": Cfg(191, 64, (-31, 32), (-31, 31), False, BF16),
    "a1_wide": Cfg(4, 1, (-31, 32), (-16, 16), False, BF16),
    "a4_wide_nott": Cfg(191, 4, (-20, 12), (-31, 31), True, BF16),
    "a32_wide": Cfg(12, 32, (-16, 16), (-3, 3), False, BF16),
}
MZ_ERR_UNSUPPORTED = -2


@functools.lru_cache(maxsize=None)
def _wide(name):
  c = WIDE[name]
  sd = _state_dict(c)
  return c, sd, _network(c, "bf16", sd)


def _rows(c, sd, got, tag, **inputs):
  """_report rows of one bf16 kernel call: h' and reward against the float64 emulation of the whole call; value and
  policy logits against the emulation's prediction heads fed the kernel's own h'.  The kernel and the emulation
  round h' to bf16 from float32 and float64 values, and where they round an element to different neighbours, one
  such flip moves a 64-bin value by up to ~0.07 in support space at these logit spreads (measured) -- more than
  the bar.  Feeding both the same h' takes that luck out; h' itself is held to the bar on its own."""
  truth, ref32 = _refs(c, sd, True, **inputs)
  chain = {q: truth[q] for q in truth if q in ("hidden", "reward")}
  rows = _report({q: got[q] for q in chain}, chain, {q: ref32[q] for q in chain}, True, c.no_tt, tag)
  emu = _ref(c, sd, torch.float64, True)
  with torch.no_grad():
    logits, value = emu._predict(torch.from_numpy(got["hidden"]))
  forced = {"logits": logits.numpy(), "value": value.numpy().reshape(-1, 1)}
  _report({q: truth[q] for q in forced}, forced, forced, True, c.no_tt, tag + " (whole-chain emulation)")
  return rows + _report({q: got[q] for q in forced}, forced, forced, True, c.no_tt, tag + " (h' forced)")


@pytest.mark.gpu
@pytest.mark.parametrize("batch", (1, 127, 129, 293))
@pytest.mark.parametrize("name", list(WIDE))
def test_wide_kernels_match_float64_reference(name, batch):
  """initial_inference (tensor cores up to 191 observation features, the float32 kernel at 192) and
  recurrent_inference in both of its modes, which agree bit for bit, at 2e-3 of the largest entry of each output."""
  c, sd, net = _wide(name)
  obs, hidden, actions = _inputs(c, batch, seed=batch + c.A)
  tag = "%s/B=%d" % (name, batch)
  init_kernel = _initial_kernel_name(net, batch)
  assert init_kernel == _expected_initial_kernel(c, "bf16")
  got = _initial(net, obs)
  if init_kernel == "mz_fc_initial_tc":
    rows = _rows(c, sd, got, tag + " initial", obs=obs)
  else:
    truth, ref32 = _refs(c, sd, False, obs=obs)
    rows = _report(got, truth, ref32, False, c.no_tt, tag + " initial")
  assert not _failures(rows), "initial_inference (%s): %s" % (init_kernel, _failures(rows))
  got = _recurrent_both_splits(net, hidden, actions)
  rows = _rows(c, sd, got, tag + " recurrent", hidden=hidden, actions=actions)
  assert not _failures(rows), "recurrent_inference: %s" % _failures(rows)


@pytest.mark.gpu
def test_comparison_rejects_faults_in_the_upper_half_of_the_heads():
  """At A = 64 with a 64-bin value support: a policy bias moved at column 40, a value bias moved at bin 50 (each by
  what moves its output ~5x the bar) and actions shifted by 32 (the one-hot in the other half) are rejected."""
  c, sd, net = _wide("a64_obs191")
  _, hidden, actions = _inputs(c, 129, seed=5)
  got = _recurrent(net, hidden, actions)
  rows = {r[0]: r for r in _rows(c, sd, got, "wide control real", hidden=hidden, actions=actions)}
  assert not _failures(rows.values())
  truth = _refs(c, sd, True, hidden=hidden, actions=actions)[0]

  def moved(key, index, delta):
    w = dict(sd)
    w[key] = sd[key].clone()
    w[key][index] += delta
    return w

  d0 = 1e-3
  shift = np.abs(h64(_refs(c, moved("value_head.value.bias", 50, d0), True, hidden=hidden, actions=actions)[0]["value"])
                 - h64(truth["value"])).max()
  controls = {
      "policy b2[40] moved": (moved("policy_head.policy.bias", 40, 5.0 * rows["logits"][2]), actions),
      "value b2[50] moved": (moved("value_head.value.bias", 50, d0 * 5.0 * rows["value"][2] / shift), actions),
      "actions + 32": (sd, (actions + 32) % c.A),
  }
  for label, (w, acts) in controls.items():
    assert _failures(_rows(c, w, got, "wide control " + label, hidden=hidden, actions=acts)), label


def _weights(obs_dim, A, vb, rb, no_support=0):
  return _lib.FcWeights(obs_dim, A, vb, rb, 0, 0, 0, no_support, *([None] * len(_lib.FcWeights._names)))


def _sizes(lib, w):
  rec, init, tail = C.c_int64(), C.c_int64(), C.c_int32()
  rc = lib.mz_fc_tc_sizes(C.byref(w), C.byref(rec), C.byref(init), C.byref(tail))
  return rc, rec.value, init.value, tail.value


def _wide_image_bytes(k, n2):
  """bytes of the four chunks of one head: [128 features x K] W1 + [N2 x 128] W2, bf16"""
  return 4 * (128 * k * 2 + n2 * 128 * 2)


def test_sizes_of_narrow_and_wide_images_without_a_gpu():
  """mz_fc_tc_sizes: for narrow weights exactly what mz_fc_tc_packed_bytes, mz_fc_tc_initial_packed_bytes and
  mz_fc_tc_tail_floats return; for wide weights the N = 64 heads and the 384-float tail, with observations up to 191
  features on the tensor cores at A = 64."""
  lib = _lib.load()
  for A in (1, 4, 18, 31, 32):
    for vb, rb in ((1, 32), (31, 31), (32, 1)):
      for obs_dim in (1, 8, 191, 192, 1000):
        assert _sizes(lib, _weights(obs_dim, A, vb, rb)) == (
            0, lib.mz_fc_tc_packed_bytes(A), lib.mz_fc_tc_initial_packed_bytes(obs_dim), lib.mz_fc_tc_tail_floats())
  assert lib.mz_fc_tc_tail_floats() == 288
  for A, vb, rb in ((33, 31, 31), (64, 64, 64), (1, 64, 1), (32, 1, 33), (50, 63, 2)):
    k1 = (50 + A + 1 + 15) // 16 * 16
    for obs_dim in (1, 191, 192):
      rc, rec, init, tail = _sizes(lib, _weights(obs_dim, A, vb, rb))
      k1i = (obs_dim + 1 + 15) // 16 * 16
      assert (rc, tail) == (0, 384)
      assert rec == 2 * _wide_image_bytes(k1, 64) + 2 * _wide_image_bytes(64, 64)
      assert init == (MZ_ERR_UNSUPPORTED if obs_dim > 191 else _wide_image_bytes(k1i, 64) + 2 * _wide_image_bytes(64, 64))


def test_c_abi_refuses_more_than_64_actions_or_bins_and_no_support_without_a_gpu():
  lib = _lib.load()
  buf = C.c_void_p(256)  # never dereferenced: the shape is refused first
  for w in (_weights(8, 65, 31, 31), _weights(8, 4, 65, 31), _weights(8, 4, 31, 65), _weights(8, 64, 64, 64, 1),
            _weights(8, 4, 31, 31, 1), _weights(8, 0, 31, 31)):
    assert _sizes(lib, w)[0] == MZ_ERR_UNSUPPORTED
    assert lib.mz_fc_tc_pack(w, buf, buf, None) == MZ_ERR_UNSUPPORTED
    assert lib.mz_fc_tc_pack_initial(w, buf, buf, None) == MZ_ERR_UNSUPPORTED
    assert lib.mz_fc_recurrent_tc(w, buf, buf, 1, buf, 50, None, buf, buf, 50, 0, buf, buf, buf, None) == \
        MZ_ERR_UNSUPPORTED
    assert lib.mz_fc_initial_tc(w, buf, buf, 1, buf, buf, 50, buf, buf, None) == MZ_ERR_UNSUPPORTED
  assert lib.mz_fc_tc_packed_bytes(33) == MZ_ERR_UNSUPPORTED  # the narrow image's size stays narrow


@pytest.mark.gpu
def test_bf16_network_refuses_65_actions_or_bins():
  from model_based_rl_b200.networks import FCNetwork, random_state_dict
  for A, vs in ((65, (-15, 15)), (4, (-32, 32))):
    net = FCNetwork(8, A, "cuda", types.SimpleNamespace(value_support=list(vs), reward_support=[-15, 15]))
    with pytest.raises(NotImplementedError, match="64"):
      net.load_weights(random_state_dict(8, A, vs[1] - vs[0] + 1, 31))


@pytest.mark.gpu
def test_fc_search_64_actions_bf16_replays_bit_exact():
  """tests/test_gpu_wide_actions.py's replay check (per-launch path, graphed, one and three slices, legal subsets of
  both mask words in the reference port, every action legal in the C oracle) with a bf16 network."""
  _search_64("bf16")


@pytest.mark.gpu
def test_fc_search_18_actions_with_63_bin_support_runs_per_launch_and_replays():
  """A bf16 network with a 63-bin value support at A = 18: the persistent search kernel reads only the narrow image,
  so fused=None takes the per-launch path and fused=True is refused; the search replays bit for bit in the C
  oracle."""
  from model_based_rl_b200.networks import FCNetwork, FCSearch
  G, A, S, D = 200, 18, 30, 24
  cfg = _ns(_cfg(S, A), value_support=[-31, 31])
  c = Cfg(D, A, (-31, 31), (-15, 15), False, BF16)
  net = FCNetwork(D, A, "cuda", cfg)
  net.load_weights(_state_dict(c))
  assert net.precision == "bf16" and net._tc_tail.numel() == 384
  with pytest.raises(ValueError, match="32 bins"):
    FCSearch(cfg, net, G, fused=True)
  fs = FCSearch(cfg, net, G)
  assert fs.fused is None
  fs.enable_record()
  rng = np.random.default_rng(2)
  obs = rng.normal(size=(G, D)).astype(np.float32)
  noise = rng.dirichlet([0.25] * A, size=G)
  u, temp = rng.random(G), np.ones(G)
  actions, root_value, child_visits, _ = fs.search_host(obs, noise, u, temp)
  rec = [r.cpu().numpy() for r in fs.record]
  want = oracle.search(oracle.make_cfg(**_cfg(S, A)), fs.root_logits.cpu().numpy(), noise=noise, noise_frac=0.25,
                       rec_value=rec[0].T, rec_reward=rec[1].T, rec_logits=rec[2].transpose(1, 0, 2))
  assert np.array_equal(fs.trace[0].cpu().numpy().T, want["trace_parent"])
  assert np.array_equal(fs.trace[1].cpu().numpy().T, want["trace_action"])
  assert np.array_equal(fs.visits.cpu().numpy(), want["visits"])
  assert np.array_equal(root_value.numpy(), want["root_value"])
  assert np.array_equal(child_visits.numpy(), want["visits"] / want["visits"].sum(1, keepdims=True))
  for g in range(G):
    assert int(actions[g]) == oracle.select_action(want["visits"][g], temp[g], u[g])


@pytest.mark.gpu
def test_device_actor_64_actions_bf16_fills_the_replay_like_the_list_path(monkeypatch):
  """tests/test_gpu_wide_actions.py's self-play check (DeviceActor against BatchedActor on FillBoard64, every live
  replay slot bit for bit) with the network that test builds made a bf16 one."""
  from model_based_rl_b200 import networks
  made = []

  class Bf16FCNetwork(networks.FCNetwork):
    def __init__(self, *args, precision=None, **kwargs):
      super().__init__(*args, precision="bf16", **kwargs)
      made.append(self)

  monkeypatch.setattr(networks, "FCNetwork", Bf16FCNetwork)
  _device_actor_64()
  assert made and all(n.precision == "bf16" and n._tc_packed is not None for n in made)


@pytest.mark.gpu
def test_bf16_learner_hands_64_action_64_bin_weights_to_a_bf16_search_network():
  """FusedLearner(precision='bf16') at A = 64 with a (-31, 32) value support and a bf16 search network: after a step
  and send_weights the search network computes bit for bit what a fresh bf16 FCNetwork loaded from the learner's
  state dict computes, and an FCSearch move runs on it."""
  from model_based_rl_b200 import fused_learner
  from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict
  A, G, S = 64, 256, 16
  cfg, batch, D = _learner_case(A=A)
  cfg.value_support = [-31, 32]
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  net.load_weights(random_state_dict(D, A, 64, 31, seed=21))
  search_net = FCNetwork(D, A, "cuda", cfg)
  search_net.load_weights(net.state_dict())
  learner = fused_learner.FusedLearner(cfg, net, search_network=search_net, use_graph=False, precision="bf16")
  learner.update_weights(batch)
  learner.send_weights()
  fresh = FCNetwork(D, A, "cuda", cfg)
  fresh.load_weights({k: v.detach().cpu() for k, v in net.state_dict().items()})
  assert search_net.precision == fresh.precision == "bf16" and search_net._tc_tail.numel() == 384
  assert torch.equal(search_net._tc_packed, fresh._tc_packed) and torch.equal(search_net._tc_tail, fresh._tc_tail)
  rng = np.random.default_rng(8)
  obs = torch.from_numpy(rng.normal(size=(G, D)).astype(np.float32)).cuda()
  hidden = torch.from_numpy(np.maximum(rng.normal(0.3, 1.0, size=(G, 50)), 0).astype(np.float32)).cuda()
  acts = torch.from_numpy(rng.integers(0, A, size=G).astype(np.int32)).cuda()
  for a, b in ((search_net.initial_inference(obs), fresh.initial_inference(obs)),
               (search_net.recurrent_inference(hidden, acts), fresh.recurrent_inference(hidden, acts))):
    for x, y in zip(a, b):
      if torch.is_tensor(x):
        assert torch.equal(x, y)
  fs = FCSearch(_ns(_cfg(S, A), value_support=[-31, 32]), search_net, G)
  actions, root_value, _, _ = fs.search_host(obs.cpu().numpy(), rng.dirichlet([0.25] * A, size=G), rng.random(G),
                                             np.ones(G))
  assert fs.fused is None and np.isfinite(root_value.numpy()).all()
  assert ((actions.numpy() >= 0) & (actions.numpy() < A)).all()
