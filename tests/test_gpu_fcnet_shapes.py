"""The FCNetwork inference kernels against a float64 reference over the shapes their C ABI accepts.

Three kernel families evaluate FCNetwork: `mz_fc_*_f32` (float32, CUDA cores), `mz_fc_*_tf32x3` (float32-accurate,
split-TF32 tensor-core products) and `mz_fc_*_tc` (bf16 tcgen05, recurrent and initial).  Each configuration below
has unequal value / reward supports or a shape at an edge of some kernel: 32 bins (the bf16 kernels' only case
without a -inf padding column), one bin, one action, supports that do not straddle zero, raw expectations
(no_target_transform), more than 32 actions or bins (the tf32x3 `second_stage<4, 8>` / `<8, 8>` paths), and
observation widths at the limits of the initial-inference kernels (bf16: 191 on the tensor cores, 192 on the
float32 fallback; tf32x3: 1, 7, 448, and 449 on the fallback).  Batches cross the row tiles of all three kernels
(8 rows f32, 32 tf32x3, 128 bf16).

Truth is `FCNetworkRef(...).double()` (oracle/fcnet_ref.py), or for the bf16 kernels `TcEmulation` of it, which
rounds to bf16 exactly where the kernels do.  Value and reward are compared in support space: the kernel's scalar
is mapped back through h (config.py:51-54) in float64, which undoes h^-1 without the float32 cancellation of
h^-1 itself; with no_target_transform the scalars are the expectations already.

Bars.  The float32 kernels' error is measured against the error that FCNetworkRef in float32 on the CPU makes on
the same inputs against the same truth: err <= K * max(err_torch32, floor) with K = 8.  The floor keeps a lucky
zero error of torch (one row, one bin) from making the bar zero: 1e-6 of the largest entry, or for scalars that
went through h^-1 in float32, 1e-4 -- the resolution of float32 h^-1 mapped back to support space (its
sqrt(d) - 1 with d in [1, 2) moves in steps of 2^-23, i.e. 6e-5 of the expectation).  Measured on a B200
(1000 W power limit): the largest ratio is 4.7, tf32x3 values at obs_dim 448.

The bf16 kernels are held to 2e-3 of the largest entry of each output, the bar of the learner's bf16 test at the
same rounding points.  A ratio to torch does not work there: where a float32 value lies within float32 rounding of
a bf16 rounding midpoint, the kernel and the emulation round it to different neighbours.  One such flip in h'
(the prediction heads' bf16 input) moves a row's value by up to ~1e-2 in support space at these logit spreads,
and whether the float32 emulation happens to flip the same element is luck.  Measured: 5.4e-4 of the largest
entry at most.
"""
import collections
import ctypes as C
import functools
import types

import numpy as np
import pytest
import torch

from oracle.fcnet_ref import FCNetworkRef, TcEmulation

H = 50
ALL, FLOAT32 = ("f32", "tf32x3", "bf16"), ("f32", "tf32x3")
Cfg = collections.namedtuple("Cfg", "obs_dim A vs rs no_tt precisions")
CONFIGS = {
    "asym32": Cfg(8, 4, (-5, 26), (-3, 3), False, ALL),
    "offset_nott": Cfg(15, 1, (0, 20), (-31, 0), True, ALL),
    "one_bin": Cfg(16, 32, (3, 3), (-15, 15), False, ALL),
    "bf16_widest": Cfg(191, 32, (-15, 15), (-10, 10), False, ALL),
    "pol_wide": Cfg(1, 40, (-15, 15), (-40, 23), False, FLOAT32),
    "all_wide": Cfg(448, 64, (-31, 32), (-20, 20), True, FLOAT32),
    "obs7": Cfg(7, 6, (-8, 8), (-6, 6), False, ("tf32x3",)),
    "obs192": Cfg(192, 8, (-15, 15), (-12, 12), False, ("bf16",)),
    "obs449": Cfg(449, 10, (-12, 12), (-15, 15), False, ("tf32x3",)),
}
BATCHES = (1, 31, 33, 127, 129, 293)
CASES = [(name, p, b) for name, c in CONFIGS.items() for p in c.precisions
         for b in (BATCHES if name == "asym32" else (1, 129))]

SPREAD = 16.0  # value / reward second layers x16: support logits with a spread of ~2.7 instead of ~0.17
K, BF16_FRAC = 8.0, 2e-3  # see the module docstring
FLOOR_REL, FLOOR_HINV = 1e-6, 1e-4


def h64(x):
  """config.py:51-54, h(x) = sign(x) (sqrt(|x| + 1) - 1) + 0.001 x, in float64."""
  x = np.asarray(x, np.float64)
  return np.sign(x) * (np.sqrt(np.abs(x) + 1.0) - 1.0) + 0.001 * x


def _bins(s):
  return s[1] - s[0] + 1


def _state_dict(c, seed=7):
  """random_state_dict with a random LayerNorm affine and spread-out support logits."""
  from model_based_rl_b200.networks import random_state_dict
  sd = random_state_dict(c.obs_dim, c.A, _bins(c.vs), _bins(c.rs), seed=seed)
  g = torch.Generator().manual_seed(seed)
  sd["LN.weight"] = 0.5 + torch.rand(H, generator=g)
  sd["LN.bias"] = 0.3 * torch.randn(H, generator=g)
  for k in ("value_head.value", "reward_head.reward"):
    sd[k + ".weight"] = sd[k + ".weight"] * SPREAD
    sd[k + ".bias"] = sd[k + ".bias"] * SPREAD
  return sd


def _ref(c, sd, dtype, bf16):
  net = FCNetworkRef(c.obs_dim, c.A, c.vs, c.rs, c.no_tt)
  net.load_state_dict(sd)
  net = net.to(dtype)
  return TcEmulation(net) if bf16 else net


def _run_ref(model, dtype, obs=None, hidden=None, actions=None):
  """outputs of a reference model as float64 arrays: hidden, logits, value (and reward for recurrent)."""
  with torch.no_grad():
    if obs is not None:
      o = model.initial_inference(torch.from_numpy(obs).to(dtype))
    else:
      o = model.recurrent_inference(torch.from_numpy(hidden).to(dtype), actions.tolist())
  out = dict(hidden=o.hidden_state, logits=o.policy_logits, value=o.value)
  if obs is None:
    out["reward"] = o.reward
  return {k: v.double().numpy().reshape(v.shape[0], -1) for k, v in out.items()}


def _refs(c, sd, bf16, **inputs):
  """(float64 truth, torch float32 result) of one call."""
  return (_run_ref(_ref(c, sd, torch.float64, bf16), torch.float64, **inputs),
          _run_ref(_ref(c, sd, torch.float32, bf16), torch.float32, **inputs))


def _gpu(out):
  torch.cuda.synchronize()
  d = dict(hidden=out.hidden_state, logits=out.policy_logits, value=out.value)
  if not isinstance(out.reward, int):
    d["reward"] = out.reward
  return {k: v.double().cpu().numpy().reshape(v.shape[0], -1) for k, v in d.items()}


def _initial(net, obs):
  return _gpu(net.initial_inference(torch.from_numpy(obs).cuda()))


def _recurrent(net, hidden, actions):
  return _gpu(net.recurrent_inference(torch.from_numpy(hidden).cuda(), torch.from_numpy(actions).cuda()))


def _report(got, truth, ref32, bf16, no_tt, tag=""):
  """[(quantity, err, bar, ratio)] for every output; value / reward in support space.  One helper for the
  real comparisons and the negative controls."""
  rows = []
  for q in truth:
    space = (lambda x: x) if no_tt or q not in ("value", "reward") else h64
    t = space(truth[q])
    scale = max(1.0, float(np.abs(t).max()))
    g = space(got[q])
    err = float(np.abs(g - t).max()) if np.isfinite(g).all() else float("inf")
    err32 = float(np.abs(space(ref32[q]) - t).max())
    floor = FLOOR_REL * scale if space is not h64 else FLOOR_HINV
    bar = BF16_FRAC * scale if bf16 else K * max(err32, floor)
    ratio = err / max(err32, floor)
    rows.append((q, err, bar, ratio))
    if tag:
      print("%-34s %-7s err %.3g  torch32 %.3g  ratio %6.2f  bar %.3g  (scale %.3g)" % (tag, q, err, err32, ratio,
                                                                                        bar, scale))
  return rows


def _failures(rows):
  return [r for r in rows if not r[1] <= r[2]]


def _expected_initial_kernel(c, precision):
  if precision == "bf16":
    return "mz_fc_initial_tc" if c.obs_dim <= 191 else "mz_fc_initial_f32"
  if precision == "tf32x3":
    return "mz_fc_initial_tf32x3" if c.obs_dim <= 448 else "mz_fc_initial_f32"
  return "mz_fc_initial_f32"


def _network(c, precision, sd):
  from model_based_rl_b200.networks import FCNetwork
  cfg = types.SimpleNamespace(value_support=list(c.vs), reward_support=list(c.rs), no_support=False,
                              no_target_transform=c.no_tt)
  net = FCNetwork(c.obs_dim, c.A, "cuda", cfg, precision=precision)
  net.load_weights(sd)
  return net


@functools.lru_cache(maxsize=None)
def _cached(name, precision):
  c = CONFIGS[name]
  sd = _state_dict(c)
  return c, sd, _network(c, precision, sd)


def _inputs(c, batch, seed):
  rng = np.random.default_rng(seed)
  obs = rng.normal(size=(batch, c.obs_dim)).astype(np.float32)
  hidden = np.maximum(rng.normal(0.3, 1.0, size=(batch, H)), 0.0).astype(np.float32)
  actions = rng.integers(0, c.A, size=batch).astype(np.int32)
  return obs, hidden, actions


def _initial_kernel_name(net, batch):
  dev = torch.empty((batch, max(H, net.action_space)), device="cuda")
  obs = torch.empty((batch, net.input_dim), device="cuda")
  return net.initial_call(batch, obs, dev, H, dev, dev, None)[0].__name__


def _recurrent_both_splits(net, hidden, actions):
  """bf16 recurrent kernel as two-CTA clusters (the default) and as one CTA per 128 rows: every head runs the
  same MMA sequence on the same operands in both modes, so the outputs must agree bit for bit."""
  lib = net.lib
  two = _recurrent(net, hidden, actions)
  try:
    assert lib.mz_fc_tc_set_split(0) == 0
    one = _recurrent(net, hidden, actions)
  finally:
    lib.mz_fc_tc_set_split(1)
  for q in two:
    assert np.array_equal(two[q], one[q]), "split and one-CTA recurrent kernels differ in %s" % q
  return two


def _check_network(c, sd, net, precision, obs, hidden, actions, tag):
  """Run initial and recurrent inference, compare both with their references; returns the recurrent outputs."""
  B = obs.shape[0]
  init_kernel = _initial_kernel_name(net, B)
  assert init_kernel == _expected_initial_kernel(c, precision)
  init_bf16 = init_kernel == "mz_fc_initial_tc"
  got = _initial(net, obs)
  truth, ref32 = _refs(c, sd, init_bf16, obs=obs)
  bad = _failures(_report(got, truth, ref32, init_bf16, c.no_tt, tag + " initial"))
  assert not bad, "initial_inference (%s): %s" % (init_kernel, bad)
  bf16 = precision == "bf16"
  got = _recurrent_both_splits(net, hidden, actions) if bf16 else _recurrent(net, hidden, actions)
  truth, ref32 = _refs(c, sd, bf16, hidden=hidden, actions=actions)
  rows = _report(got, truth, ref32, bf16, c.no_tt, tag + " recurrent")
  assert not _failures(rows), "recurrent_inference: %s" % _failures(rows)
  return got


@pytest.mark.gpu
@pytest.mark.parametrize("name,precision,batch", CASES)
def test_kernels_match_float64_reference(name, precision, batch):
  """Hidden states, policy logits, value and reward of initial_inference and recurrent_inference against the
  float64 reference (bf16 kernels: its bf16 emulation), at the bars of the module docstring.  The bf16 recurrent
  kernel runs in both of its modes, which must agree bit for bit."""
  c, sd, net = _cached(name, precision)
  obs, hidden, actions = _inputs(c, batch, seed=batch)
  _check_network(c, sd, net, precision, obs, hidden, actions, "%s/%s/B=%d" % (name, precision, batch))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ALL)
def test_comparison_rejects_a_subtly_wrong_reference(precision):
  """Negative controls: the comparison above, with the kernel's real outputs, against references that are wrong
  in the ways a kernel could be -- one value-head b2 entry moved so that the values move by ~5x the bar, the
  value and reward support offsets swapped, the actions shifted by one.  Each must be rejected."""
  c, sd, net = _cached("asym32", precision)
  B, bf16 = 129, precision == "bf16"
  _, hidden, actions = _inputs(c, B, seed=3)
  got = _recurrent(net, hidden, actions)
  truth, ref32 = _refs(c, sd, bf16, hidden=hidden, actions=actions)
  rows = {r[0]: r for r in _report(got, truth, ref32, bf16, c.no_tt, "control %s real" % precision)}
  assert not _failures(rows.values())

  def wrong_refs(cfg=c, weights=sd, acts=actions):  # (float64, float32) of the wrong reference: its own bar
    return _refs(cfg, weights, bf16, hidden=hidden, actions=acts)

  def value_bias_moved(delta):  # b2 is added unrounded in every kernel: the change is not quantised by bf16
    w = dict(sd)
    w["value_head.value.bias"] = sd["value_head.value.bias"].clone()
    w["value_head.value.bias"][row] += delta
    return w

  # move the bias of the bin that most rows' expectations round to, by what moves the values ~5x their bar
  row = int(np.argmax(np.bincount(np.round(h64(truth["value"][:, 0])).astype(int) - c.vs[0], minlength=_bins(c.vs))))
  d0 = 1e-3
  moved = np.abs(h64(wrong_refs(weights=value_bias_moved(d0))[0]["value"]) - h64(truth["value"])).max()
  delta = d0 * 5.0 * rows["value"][2] / moved
  swapped = c._replace(vs=(c.rs[0], c.rs[0] + _bins(c.vs) - 1), rs=(c.vs[0], c.vs[0] + _bins(c.rs) - 1))
  controls = {"value b2[%d] + %.3g" % (row, delta): wrong_refs(weights=value_bias_moved(delta)),
              "supports swapped": wrong_refs(cfg=swapped),
              "action + 1": wrong_refs(acts=(actions + 1) % c.A)}
  for label, (wrong, wrong32) in controls.items():
    bad = _failures(_report(got, wrong, wrong32, bf16, c.no_tt, "control %s %s" % (precision, label)))
    assert bad, "the comparison accepts a reference with %s" % label


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ALL)
def test_recurrent_into_gathers_and_writes_only_its_rows(precision):
  """The raw form the search engine calls: rows gathered through in_index from a three-slot pool, h' scattered
  into the same pool at an odd column offset, output buffers longer than the batch.  The results equal the plain
  call on the gathered rows bit for bit; nothing outside the B rows x 50 columns and the B value / reward /
  logit rows is written (NaN sentinels), and the source slots are untouched."""
  c, sd, net = _cached("asym32", precision)
  B, stride, off, extra = 129, 224, 151, 5  # even input stride: the bf16 kernel reads hidden rows as float2
  rng = np.random.default_rng(17)
  pool = torch.full((B + extra, stride), float("nan"), device="cuda")
  pool[:, :3 * H] = torch.from_numpy(np.maximum(rng.normal(0.3, 1.0, size=(B + extra, 3 * H)), 0)).float().cuda()
  idx = torch.from_numpy(rng.integers(0, 3, size=B).astype(np.int32)).cuda()
  act = torch.from_numpy(rng.integers(0, c.A, size=B).astype(np.int32)).cuda()
  before = pool.clone()
  value, reward = (torch.full((B + extra, 1), float("nan"), device="cuda") for _ in range(2))
  logits = torch.full((B + extra, c.A), float("nan"), device="cuda")
  net.recurrent_into(pool, stride, idx, act, pool, stride, off, value, reward, logits)
  torch.cuda.synchronize()
  rows = torch.arange(B, device="cuda")
  gathered = before[:B, :3 * H].reshape(B, 3, H)[rows, idx.long()].contiguous()
  want = net.recurrent_inference(gathered, act)
  torch.cuda.synchronize()
  assert torch.equal(pool[:B, off:off + H], want.hidden_state)
  assert torch.equal(value[:B], want.value) and torch.equal(reward[:B], want.reward)
  assert torch.equal(logits[:B], want.policy_logits)
  untouched = torch.ones_like(pool, dtype=torch.bool)
  untouched[:B, off:off + H] = False
  assert torch.equal(pool.view(torch.int32)[untouched], before.view(torch.int32)[untouched])
  for t in (value, reward, logits):
    assert t[B:].isnan().all()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ALL)
def test_constant_pre_layernorm_rows_and_extreme_support_logits(precision):
  """Degenerate rows.  A transition head with zero W2 and a constant bias makes every pre-LayerNorm row constant:
  zero variance, so h' = relu(LN.bias) exactly up to the last bit of the mean (the bias 0.5 sums exactly).  Value
  and reward logits scaled to span about +-100: exp overflows float32 unless the maximum is subtracted first,
  in every support-to-scalar path.  The rest of the outputs go through the comparison above."""
  c = CONFIGS["asym32"]
  sd = _state_dict(c, seed=5)
  sd["transition_head.out.weight"] = torch.zeros_like(sd["transition_head.out.weight"])
  sd["transition_head.out.bias"] = torch.full((H,), 0.5)
  obs, hidden, actions = _inputs(c, 129, seed=9)
  ref = _ref(c, sd, torch.float64, False)
  with torch.no_grad():
    h = ref.initial_inference(torch.from_numpy(obs).double()).hidden_state
    span = max(ref.value_head(h).abs().max().item(),
               ref.reward_head(ref._attach_action(torch.from_numpy(hidden).double(), actions).double()).abs().max().item())
  for k in ("value_head.value", "reward_head.reward"):
    sd[k + ".weight"] = sd[k + ".weight"] * (100.0 / span)
    sd[k + ".bias"] = sd[k + ".bias"] * (100.0 / span)
  net = _network(c, precision, sd)
  got = _check_network(c, sd, net, precision, obs, hidden, actions, "degenerate/%s" % precision)
  want = np.maximum(sd["LN.bias"].double().numpy(), 0.0)
  assert np.abs(got["hidden"] - want).max() <= 1e-5


# ---- without a GPU: the references themselves, and the bf16 kernel's argument check --------------------------------
@pytest.mark.parametrize("name,obs_dim,A,no_support", [("atari18", 128, 18, False), ("ttt", 9, 9, False),
                                                       ("nosupport", 8, 4, True)])
def test_float64_reference_reproduces_reference_golden(name, obs_dim, A, no_support):
  """The float64 evaluation of FCNetworkRef against the outputs of the unmodified reference module (torch
  float32 on the CPU): hidden states and logits within 2e-6 of their largest entry (float32 rounding through
  four layers), support scalars within 1e-4 in support space (float32 h^-1 resolution, see the module
  docstring; the no_support scalars are raw outputs and held to 2e-6)."""
  from helpers import load
  g = load("fcnet_" + name)
  net = FCNetworkRef(obs_dim, A, no_support=no_support)
  net.load_state_dict({k[2:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("w_")})
  got = {"init": _run_ref(net.double(), torch.float64, obs=g["obs"]),
         "rec": _run_ref(net, torch.float64, hidden=g["init_hidden"], actions=g["actions"])}
  for pre, outs in got.items():
    for q, v in outs.items():
      want = g["%s_%s" % (pre, q)].astype(np.float64).reshape(v.shape)
      if q in ("value", "reward") and not no_support:
        err, bar = np.abs(h64(v) - h64(want)).max(), FLOOR_HINV
      else:
        err, bar = np.abs(v - want).max(), 2e-6 * max(1.0, np.abs(want).max())
      assert err <= bar, "%s_%s: %g > %g" % (pre, q, err, bar)


@pytest.mark.parametrize("name", ["asym32", "offset_nott", "all_wide"])
def test_emulation_without_rounding_is_the_float64_reference(name):
  """TcEmulation(bf16=False) restates the network with the first-layer bias folded into the weights; in float64
  that is the reference module's result up to float64 rounding.  With the rounding on it moves by bf16 amounts."""
  c = CONFIGS[name]
  sd = _state_dict(c)
  obs, hidden, actions = _inputs(c, 40, seed=1)
  net = _ref(c, sd, torch.float64, False)
  for inputs in (dict(obs=obs), dict(hidden=hidden, actions=actions)):
    want = _run_ref(net, torch.float64, **inputs)
    exact = _run_ref(TcEmulation(net, bf16=False), torch.float64, **inputs)
    rounded = _run_ref(TcEmulation(net, bf16=True), torch.float64, **inputs)
    for q in want:
      scale = max(1.0, np.abs(want[q]).max())
      assert np.abs(exact[q] - want[q]).max() <= 1e-12 * scale, q
      assert 1e-5 * scale < np.abs(rounded[q] - want[q]).max() < 5e-2 * scale, q


def test_recurrent_tc_rejects_misaligned_hidden_rows():
  """mz_fc_recurrent_tc reads hidden rows as float2: an odd in_row_stride or a hidden_in that is not 8-byte aligned
  is MZ_ERR_BAD_ARG, answered before anything is launched (host pointers here, no device needed)."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  w = _lib.FcWeights(8, 4, 31, 31, -15, -15, 0, 0, *([0] * len(_lib.FcWeights._names)))
  buf = np.zeros(4096, np.float64)
  p = buf.ctypes.data
  def call(hidden_in, in_row_stride):
    return lib.mz_fc_recurrent_tc(C.byref(w), p, p, 1, hidden_in, in_row_stride, None, p, p, 50, 0, p, p, p, None)
  assert call(p, 51) == -1
  assert call(p + 4, 50) == -1
  assert call(p + 4, 51) == -1
