"""The MuZeroNetwork kernels (csrc/mz_conv_tc.cu) against float64 arithmetic on their own operands, at the batch
sizes of the C5 benchmark (4096 games), where every persistent loop runs several work items per CTA.

The references below are test helpers, not oracle changes.  Each takes what the kernel takes -- bf16 activations
and residuals, the packed bf16 weights (`_Conv.w` with BatchNorm folded, `_StridedConv.w`, `_pack_fc`), float32
bias and action-plane term -- and evaluates one launch in float64.  `test_reference_helpers_compose_to_the_oracle`
pins them without a GPU: composed into representation, dynamics and prediction they equal oracle/muzero_ref.py in
float64, which catches a misread packed layout (tap order, the padded rows of `_pack_fc`).

Bars, derived from the arithmetic and stated as err / bar <= 1 per element (the worst ratio is printed):
  - float32 accumulation of K products and their epilogue: K_eff * 2^-24 * sum|terms|, K_eff = K + the float32
    epilogue operations.  K = 1152 (3x3 conv, 128 channels; 576 at 64), 9 * cin_pad (strided conv), 6272 (Linear
    over the padded state), 16 + 5 (conv_head_kernel: 16 fmaf per lane, then a 5-step butterfly).  The tensor
    cores round once per block of products rather than per product, so the count K covers their truncating
    accumulator (unit 2^-23) as well;
  - one bf16 output rounding: 2^-8 relative to the float32 value (8 significant bits, round to nearest even: the
    unit roundoff is 2^-8; values just above a power of two reach 2^-8 / (1 + 2^-8), so 2^-9 would not hold);
  - the scaled state: both kernels (EPI_SCALE in conv_gemm_tc_kernel and conv_pair_tc_kernel) take min / max over
    the float32 epilogue values x of a pixel -- not the bf16 output -- and write bf16((x - min) / (max - min)).
    With |x - y| <= E on every channel of the pixel, numerator and denominator move by at most 2E each, so the
    scaled value moves by at most 4E / (den - 2E) (s in [0, 1]); plus three float32 roundings and the bf16 one;
  - the support heads: see `ref_head`.

Measured on a B200 (1000 W power limit): worst err / bar 0.996 for the bf16 outputs (average pool and strided
conv; the 2^-8 of a single bf16 rounding is nearly the whole bar there), 0.70 for the scaled state, 0.002 for the
float32 Linear heads, 0.31 for mz_conv_head.  The whole file took 8 to 25 s (two runs) with a peak of 27.3 GB of
device memory (the ConvSearch move at 4096 games).

Work items.  conv_gemm_tc_kernel (single CTA, also the Linear heads and the strided-conv GEMM) runs min(tiles, SMs)
CTAs over tiles of 128 rows; conv_pair_tc_kernel runs min(ceil(tiles / 2), SMs / 2) clusters over pairs of tiles.
Every case prints what its busiest CTA or cluster gets (from the SM count the device reports), and the largest
case of each kernel asserts that this is at least 3 -- the first count at which a CTA reuses an accumulator buffer
at the flipped mbarrier parity.
"""
import math
import time
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from model_based_rl_b200 import muzero
from oracle import muzero_ref

U = 2.0 ** -24    # float32 unit roundoff
BF = 2.0 ** -8    # bf16 unit roundoff (8-bit significand)
RELU, RESIDUAL, ACTION, SCALE = muzero.RELU, muzero.RESIDUAL, muzero.ACTION, muzero.SCALE
CFG = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=False,
                            no_target_transform=False)
SENTINEL = 7.0    # bf16 sentinel of rows a kernel must not write
gpu = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _time_and_peak_memory(request):
  """Prints each GPU test's wall time and peak device memory, and frees the cached blocks afterwards."""
  on_gpu = request.node.get_closest_marker("gpu") is not None and torch.cuda.is_available()
  if on_gpu:
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
  t0 = time.time()
  yield
  if on_gpu:
    torch.cuda.synchronize()
    print("[%s] %.1f s, peak device memory %.2f GB" % (request.node.name, time.time() - t0,
                                                      torch.cuda.max_memory_allocated() / 1e9))
    torch.cuda.empty_cache()


# ---- float64 references on the kernels' operands ---------------------------------------------------------------
def _pad64(x):
  """[B, C, W, W] -> [B, (W + 1)^2 * C]: muzero.to_padded's layout in float64, without the bf16 cast."""
  b, c, w = x.shape[0], x.shape[1], x.shape[-1]
  return F.pad(x.permute(0, 2, 3, 1), (0, 0, 0, 1, 1, 0)).reshape(b, (w + 1) * (w + 1) * c)


def conv_weight64(conv):
  """_Conv.w [C][9 C] bf16, k = (ky * 3 + kx) * C + c  ->  [C, C, 3, 3] float64."""
  c = conv.channels
  return conv.w.double().reshape(c, 3, 3, c).permute(0, 3, 1, 2)


def ref_conv(x, conv, flags, residual=None, actions=None, num_actions=18, weight=None):
  """One mz_conv3x3_tc launch: x [B, C, W, W] float64 holding bf16 values, residual likewise.  Returns (y, mag): the
  epilogue's value before the bf16 output rounding (bias, a / A * plane, residual, ReLU) and the sum of |terms|
  that float32 adds up for it.  `weight` replaces the unpacked weights (negative controls)."""
  w = conv_weight64(conv) if weight is None else weight
  bias = conv.bias.double()[None, :, None, None]
  y = F.conv2d(x, w, None, 1, 1) + bias
  mag = F.conv2d(x.abs(), w.abs(), None, 1, 1) + bias.abs()
  if flags & ACTION:
    width = x.shape[-1]
    a = (actions.to(x.device, torch.float32) / num_actions).double()  # the kernel's float32 a / A
    plane = conv.plane.double().to(x.device).reshape(width, width, -1).permute(2, 0, 1)
    term = a[:, None, None, None] * plane[None]
    y, mag = y + term, mag + term.abs()
  if flags & RESIDUAL:
    y, mag = y + residual, mag + residual.abs()
  if flags & RELU:
    y = y.clamp_min(0.0)
  return y, mag


def conv_bar(y, mag, k):
  """bf16 rounding of the float32 epilogue value, whose error is (K + 4) 2^-24 sum|terms| (K products; bias,
  action fma, residual add)."""
  return BF * y.abs() + (1 + BF) * (k + 4) * U * mag


def ref_scale(y, mag=None, k=None):
  """scale_state per pixel over the channel dimension (networks.py:543-547); with (mag, k) also the bar of the
  kernel's scaled output (module docstring)."""
  mn, mx = y.amin(dim=1, keepdim=True), y.amax(dim=1, keepdim=True)
  den = mx - mn
  s = (y - mn) / den
  if mag is None:
    return s
  e = ((k + 4) * U * mag).amax(dim=1, keepdim=True)
  assert bool((den > 2 * e).all()), "a pixel whose channels are all within rounding of each other"
  return s, BF * s + (1 + BF) * (4 * e / (den - 2 * e) + 3 * U)


def strided_weight64(conv):
  """_StridedConv.w [Cout][k_pad] bf16, k = (ky * 3 + kx) * cin_pad + c  ->  [Cout, cin_pad, 3, 3] float64."""
  return conv.w.double()[:, :9 * conv.cin_pad].reshape(conv.cout, 3, 3, conv.cin_pad).permute(0, 3, 1, 2)


def ref_strided(x, conv):
  """im2col + mz_conv_gemm_to_padded: x [B, cin_pad, W, W] -> (y before bf16 rounding, sum|terms|)."""
  w, b = strided_weight64(conv), conv.bias.double()
  return F.conv2d(x, w, b, 2, 1), F.conv2d(x.abs(), w.abs(), b.abs(), 2, 1)


def strided_bar(y, mag, conv):
  return BF * y.abs() + (1 + BF) * (9 * conv.cin_pad + 2) * U * mag


def ref_pool(x):
  """AvgPool2d(3, 2, 1), count_include_pad: (y, sum|x| over the window)."""
  return F.avg_pool2d(x, 3, 2, 1), 9.0 * F.avg_pool2d(x.abs(), 3, 2, 1)


def pool_bar(y, mag):
  """conv_avgpool_kernel: nine float32 adds from zero (eight round), times float32(1/9) (two roundings), bf16."""
  return BF * y.abs() + (1 + BF) * (8 * U * mag / 9 + 2 * U * y.abs())


def ref_fc(state, w_packed, bias, relu=True):
  """mz_conv_fc_tc: state [B, 128, 6, 6] (bf16 values) in the padded flat layout the packed weights [n][6272]
  index.  Returns (y, sum|terms|); the output is float32, bar (6272 + 2) 2^-24 sum|terms|."""
  a, w, b = _pad64(state), w_packed.double().to(state.device), bias.double().to(state.device)
  y = a @ w.T + b
  mag = a.abs() @ w.abs().T + b.abs()
  return (y.clamp_min(0.0) if relu else y), mag


FC_K = muzero.K_FC + 2


def _h_inv(x):  # config.py:27-33, float64
  eps = 0.001
  return torch.sign(x) * (((torch.sqrt(1 + 4 * eps * (x.abs() + 1 + eps)) - 1) / (2 * eps)) ** 2 - 1)


def ref_head(hidden, w2, b2, outs, to_scalar, support_min=0, no_tt=0):
  """mz_conv_head on its float32 operands (hidden [B, >= 512], W2 [outs][512], b2).  Returns (out, bar).
  Logits: every product passes at most 16 fmaf + 5 butterfly adds + the bias add: 22 roundings,
  dl = 23 * 2^-24 * sum|terms|.  Scalars: expf(l - max) of computed logits is off by a factor exp(2 dl + the
  subtraction's rounding) and expf's 2 ulp; a per-term factor within 1 +- eta moves the softmax expectation by at
  most eta / (1 - eta) * sum_i p_i |s_i - x|.  The butterfly sums and the division add 6 * 2^-24 (sum p|s| + |x|).
  h^-1 in float32: u = 1 + 4 eps (|x| + 1 + eps) within 5 roundings, sqrtf correctly rounded, the subtraction of 1
  exact, division by 0.002f (two roundings) -> t within 2 t 2^-24 + 3.5 2^-24 sqrt(u) / 0.002, t * t - 1 within
  2 t dt + 2 * 2^-24 t^2; the expectation's own error enters through the slope 2 t / sqrt(u) at |x| + dx."""
  h = hidden[:, :512].double()
  w, b = w2[:outs].double().to(h.device), b2[:outs].double().to(h.device)
  logits = h @ w.T + b
  dl = 23 * U * (h.abs() @ w.abs().T + b.abs())
  if not to_scalar:
    return logits, dl
  sv = support_min + torch.arange(outs, dtype=torch.float64, device=h.device)
  m = logits.amax(dim=1, keepdim=True)
  p = torch.softmax(logits, dim=1)
  x = (p * sv).sum(dim=1)
  arg = 2 * dl.amax(dim=1) + U * (logits - m).abs().amax(dim=1)
  eta = torch.exp(arg) * (1 + 4 * U) - 1
  dx = eta / (1 - eta) * (p * (sv[None, :] - x[:, None]).abs()).sum(dim=1) + 6 * U * ((p * sv.abs()).sum(dim=1) + x.abs())
  if no_tt:
    return x, dx
  eps = 0.001

  def t_of(v):
    u = 1 + 4 * eps * (v + 1 + eps)
    return (torch.sqrt(u) - 1) / (2 * eps), u
  t, u = t_of(x.abs())
  e_h = 2 * t * (2 * U * t + 3.5 * U * torch.sqrt(u) / 0.002) + 2 * U * t * t
  t_hi, u_hi = t_of(x.abs() + dx)
  return _h_inv(x), 2 * t_hi / torch.sqrt(u_hi) * dx + e_h


def _ratio(got, want, bar):
  """max over entries of |got - want| / bar (inf when got holds a non-finite value)."""
  got = got.double().to(want.device)
  if not bool(torch.isfinite(got).all()):
    return math.inf
  return float(((got - want).abs() / bar.clamp_min(1e-300)).max())


# ---- composition of the helpers (the CPU pin) ------------------------------------------------------------------
def ref_tower(convs, x):
  for i in range(len(convs) // 2):
    t = ref_conv(x, convs[2 * i], RELU)[0]
    x = ref_conv(t, convs[2 * i + 1], RELU | RESIDUAL, residual=x)[0]
  return x


def ref_representation(net, obs):
  c1 = net.rep_conv1
  x = F.pad(obs, (0, 0, 0, 0, 0, c1.cin_pad - obs.shape[1]))
  x = ref_tower(net.rep_blocks1, ref_strided(x, c1)[0])
  x = ref_tower(net.rep_blocks2, ref_strided(x, net.rep_conv2)[0])
  x = ref_tower(net.rep_blocks3, ref_pool(x)[0])
  return ref_scale(ref_tower(net.rep_tower, ref_pool(x)[0]))


def ref_prediction(net, state):
  hid = ref_fc(ref_tower(net.pred_tower, state), net.vp_fc1_w, net.vp_fc1_b)[0]
  value = ref_head(hid[:, :512], net.val_fc2_w, net.val_fc2_b, net.value_bins, 1, net.value_min,
                   net.no_target_transform)[0]
  logits = ref_head(hid[:, 512:], net.pol_fc2_w, net.pol_fc2_b, net.action_space, 0)[0]
  return value, logits


def ref_dynamics(net, state, actions):
  x = ref_conv(state, net.dyn_conv, RELU | ACTION, actions=actions, num_actions=net.action_space)[0]
  x = ref_tower(net.dyn_tower, x)
  hid = ref_fc(x, net.rew_fc1_w, net.rew_fc1_b)[0]
  reward = ref_head(hid, net.rew_fc2_w, net.rew_fc2_b, net.reward_bins, 1, net.reward_min,
                    net.no_target_transform)[0]
  return ref_scale(x), reward


def _exact_state_dict(C_in, A, seed, value_bins, reward_bins):
  """seeded_state_dict with every parameter on a grid that packing keeps exact: weights and biases multiples of
  2^-10 rounded to bf16; BatchNorm with running_var = 2^40 (var + 1e-5 rounds to 2^40 in float32 and in float64, so
  the fold divides by exactly 2^20), running_mean = 0 and gamma = 2^20 * (1/2 or 1): the folded weights are the
  bf16 weights times a power of two."""
  sd = muzero_ref.seeded_state_dict(C_in, A, seed, value_bins, reward_bins)
  g = torch.Generator().manual_seed(seed + 1)
  out = {}
  for k, v in sd.items():
    if k.endswith("num_batches_tracked"):
      out[k] = v
    elif k.endswith("running_var"):
      out[k] = torch.full_like(v, 2.0 ** 40)
    elif k.endswith("running_mean"):
      out[k] = torch.zeros_like(v)
    elif ".bn" in k and k.endswith(".weight"):
      out[k] = 2.0 ** 20 * (0.5 + 0.5 * (torch.rand(v.shape, generator=g) < 0.5).float())
    else:
      out[k] = (torch.round(v * 1024) / 1024).to(torch.bfloat16).float()
  return out


def _cpu_network(sd, C_in, A, value_support, reward_support, no_tt):
  """MuZeroNetwork's packing (load_weights) on the CPU, without the CUDA library."""
  net = muzero.MuZeroNetwork.__new__(muzero.MuZeroNetwork)
  net.device = torch.device("cpu")
  net.input_channels, net.action_space = C_in, A
  net.value_min, net.value_max = value_support
  net.reward_min, net.reward_max = reward_support
  net.value_bins, net.reward_bins = value_support[1] - value_support[0] + 1, reward_support[1] - reward_support[0] + 1
  net.no_target_transform = no_tt
  muzero.MuZeroNetwork.load_weights.__wrapped__(net, sd)
  return net


def test_reference_helpers_compose_to_the_oracle():
  """Without a GPU: the float64 layer references, composed over MuZeroNetwork's packed weights into
  initial_inference and recurrent_inference, equal oracle/muzero_ref.py run in float64, for both no_target_transform
  settings and asymmetric supports.  Weights are chosen so that packing is exact (_exact_state_dict), so the only
  difference left is the order of float64 sums through ~40 layers: measured at most 7e-13 (a value after h^-1),
  bar 1e-10 of the largest entry.  A misread layout (tap order, the padded rows of _pack_fc, value / policy halves) moves outputs by
  O(1e-2) or more."""
  C_in, A, B = 4, 18, 2
  vs, rs = (-12, 18), (-20, 10)
  sd = _exact_state_dict(C_in, A, 5, 31, 31)
  sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
  g = torch.Generator().manual_seed(11)
  obs = torch.rand((B, C_in, 96, 96), generator=g, dtype=torch.float64)
  hidden = torch.rand((B, 128, 6, 6), generator=g, dtype=torch.float64)
  actions = torch.tensor([3, 17], dtype=torch.int32)

  def close(name, got, want):
    err = float((got - want).abs().max())
    bar = 1e-10 * max(1.0, float(want.abs().max()))
    print("%-22s max |helpers - oracle| %.3g (bar %.3g)" % (name, err, bar))
    assert err <= bar, name

  with torch.no_grad():
    want_h0 = muzero_ref.representation(obs, sd64)
    want_pol0, want_v0 = muzero_ref.prediction_logits(want_h0, sd64)
    want_h1, want_r1 = muzero_ref.dynamics_logits(hidden, actions.tolist(), sd64, A)
    want_pol1, want_v1 = muzero_ref.prediction_logits(want_h1, sd64)
    for no_tt in (False, True):
      net = _cpu_network(sd, C_in, A, vs, rs, no_tt)
      h0 = ref_representation(net, obs)
      v0, pol0 = ref_prediction(net, h0)
      h1, r1 = ref_dynamics(net, hidden, actions)
      v1, pol1 = ref_prediction(net, h1)
      tag = "no_tt=%d " % no_tt
      close(tag + "initial hidden", h0, want_h0)
      close(tag + "initial logits", pol0, want_pol0)
      close(tag + "initial value", v0, muzero_ref.inverse_transform(want_v0, *vs, no_tt).flatten())
      close(tag + "recurrent hidden", h1, want_h1)
      close(tag + "recurrent logits", pol1, want_pol1)
      close(tag + "recurrent value", v1, muzero_ref.inverse_transform(want_v1, *vs, no_tt).flatten())
      close(tag + "recurrent reward", r1, muzero_ref.inverse_transform(want_r1, *rs, no_tt).flatten())


def test_head_bar_covers_float32_evaluation():
  """Without a GPU: ref_head's bar holds for the same head evaluated in float32 by torch (a different summation
  order than the kernel's, but the same count of roundings or fewer), and is not loose by orders of magnitude."""
  g = torch.Generator().manual_seed(2)
  hid = torch.relu(torch.randn((300, 512), generator=g))
  for outs, smin in ((1, 3), (18, -5), (31, -20), (32, 0)):
    w2, b2 = torch.randn((outs, 512), generator=g) * 0.1, torch.randn(outs, generator=g) * 0.5
    l32 = hid @ w2.T + b2
    for no_tt in (0, 1):
      want, bar = ref_head(hid, w2, b2, outs, 1, smin, no_tt)
      got = muzero_ref.inverse_transform(l32, smin, smin + outs - 1, bool(no_tt)).flatten()
      assert _ratio(got, want, bar) <= 1.0, (outs, no_tt)
    want, bar = ref_head(hid, w2, b2, outs, 0)
    assert _ratio(l32, want, bar) <= 1.0
    assert float(bar.max()) < 1e-3


# ---- work items per CTA ----------------------------------------------------------------------------------------
def _sms():
  return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def single_items(rows, n_tiles=1):
  """Work items of the busiest CTA of conv_gemm_tc_kernel (launch_conv: grid = min(tiles, SMs))."""
  tiles = -(-rows // 128) * n_tiles
  return -(-tiles // min(tiles, _sms()))


def pair_items(rows):
  """Work items of the busiest cluster of conv_pair_tc_kernel (launch_conv_pair: min(ceil(tiles / 2), SMs / 2))."""
  pairs = -(-(-(-rows // 128)) // 2)
  return -(-pairs // min(pairs, _sms() // 2))


def stride_items(total):
  """Iterations of the busiest thread of the grid-stride kernels (im2col, average pool: 148 * 16 blocks of 256)."""
  return -(-total // (148 * 16 * 256))


def conv_items(rows, mode, channels=128):
  return pair_items(rows) if channels == 128 and mode else single_items(rows)


# ---- layer cases ----------------------------------------------------------------------------------------------
def _lib():
  from model_based_rl_b200 import _lib as lib_mod
  return lib_mod, lib_mod.load()


def _rand_conv(ch, dev, action=False):
  cin = ch + 1 if action else ch
  w = (torch.rand((ch, cin, 3, 3), device=dev) * 2 - 1) * (3.0 / (9 * cin)) ** 0.5
  if action:
    w[:, ch] = (torch.rand((ch, 3, 3), device=dev) * 2 - 1) * 0.5  # a plane term of O(1): a / A visibly matters
  return muzero._Conv(w, torch.randn(ch, device=dev) * 0.1, None, dev)


def _launch_conv(lib_mod, lib, games, width, conv, flags, x, out, residual=None, actions=None, scaled=None,
                 pool=None, pool_base=None):
  P = lib_mod.ptr
  lib_mod.check(lib.mz_conv3x3_tc(games, width, conv.channels, P(x), P(conv.w), P(conv.bias), flags,
                                  P(conv.plane) if flags & ACTION else None, P(actions), 18, P(residual), P(out),
                                  P(scaled), P(pool), P(pool_base), lib_mod.current_stream()), "mz_conv3x3_tc")


def _check_padding(rows, games, width, tag):
  """Padding rows of the first `games` games exactly zero, rows past them still the sentinel."""
  n = games * (width + 1) ** 2
  assert float(muzero.padding_rows(rows[:n], games, width).float().abs().max()) == 0, tag + ": padding written"
  assert bool((rows[n:] == SENTINEL).all()), tag + ": rows past the last game written"


CONV6_GAMES = (1, 3, 386, 387, 1000, 4096, 4097)
CONV6_EPILOGUES = {"relu": (RELU, False), "relu_res": (RELU | RESIDUAL, False), "relu_action": (RELU | ACTION, False),
                   "scale": (RELU | RESIDUAL | SCALE, False), "scale_pool": (RELU | RESIDUAL | SCALE, True)}


@gpu
@pytest.mark.parametrize("epi", list(CONV6_EPILOGUES))
@pytest.mark.parametrize("games", CONV6_GAMES)
def test_conv6_matches_float64_in_every_pair_mode(games, epi):
  """The 6 x 6, 128-channel convolution in pair modes 0 (single CTA), 1 (CTA pair, per-tap loads) and 2 (CTA pair,
  row windows), each against float64 and each bit-identical to mode 0.  Games 386 / 387: the last count without /
  the first with a CTA's second tile; 1000 and up: accumulator buffers reused at the flipped parity.  With a pool,
  game g's scaled rows also land in slot dst[g] of a [games][slots][49][128] pool (51 slots from 4096 games on:
  the last slots lie past 2 GiB); every other pool row keeps its sentinel."""
  lib_mod, lib = _lib()
  flags, with_pool = CONV6_EPILOGUES[epi]
  dev = "cuda"
  torch.manual_seed(games * 32 + flags + with_pool)
  conv = _rand_conv(128, dev, action=bool(flags & ACTION))
  x = muzero.to_padded(torch.rand((games, 128, 6, 6), device=dev))
  res = muzero.to_padded(torch.rand((games, 128, 6, 6), device=dev)) if flags & RESIDUAL else None
  actions = torch.randint(0, 18, (games,), device=dev, dtype=torch.int32) if flags & ACTION else None
  rows = (games + 1) * 49
  out = torch.full((rows, 128), SENTINEL, dtype=torch.bfloat16, device=dev)
  scaled = torch.full_like(out, SENTINEL) if flags & SCALE else None
  pool = pool_base = None
  if with_pool:
    slots = 51 if games >= 4096 else 3
    pool = torch.full((games * slots * 49, 128), SENTINEL, dtype=torch.bfloat16, device=dev)
    dst = torch.randint(0, slots, (games,), device=dev)
    dst[::97] = slots - 1
    dst[-1] = slots - 1
    pool_base = ((torch.arange(games, device=dev) * slots + dst) * 49).to(torch.int32)
    if games >= 4096:
      assert (int(pool_base.max()) + 48) * 128 * 2 > 2 ** 31  # the last slots' byte offsets need 64 bits
  y, mag = ref_conv(muzero.from_padded(x, games).double(), conv, flags,
                    residual=muzero.from_padded(res, games).double() if res is not None else None,
                    actions=actions)
  bar = conv_bar(y, mag, 1152)
  if flags & SCALE:
    s, bar_s = ref_scale(y, mag, 1152)
  first = None
  try:
    for mode in (0, 1, 2):
      assert lib.mz_conv_set_pair(mode) == 0
      out.fill_(SENTINEL)
      if scaled is not None:
        scaled.fill_(SENTINEL)
      _launch_conv(lib_mod, lib, games, 6, conv, flags, x, out, residual=res, actions=actions, scaled=scaled,
                   pool=pool, pool_base=pool_base)
      torch.cuda.synchronize()
      r = _ratio(muzero.from_padded(out[:games * 49], games), y, bar)
      msg = "conv6 %-11s games %4d mode %d: work items on the busiest CTA/cluster %2d, worst err/bar %.3g" % (
          epi, games, mode, conv_items(games * 49, mode), r)
      if scaled is not None:
        rs = _ratio(muzero.from_padded(scaled[:games * 49], games), s, bar_s)
        msg += ", scaled %.3g" % rs
        assert rs <= 1.0, (mode, rs)
        _check_padding(scaled, games, 6, "scaled mode %d" % mode)
      print(msg)
      assert r <= 1.0, (mode, r)
      _check_padding(out, games, 6, "mode %d" % mode)
      if with_pool:
        pv = pool.view(games, slots, 49, 128)
        ar = torch.arange(games, device=dev)
        assert torch.equal(pv[ar, dst].reshape(-1, 128), scaled[:games * 49]), mode
        pv[ar, dst] = SENTINEL  # ... and nothing else of the pool was written: all sentinel again
        assert bool((pool == SENTINEL).all()), mode
      if first is None:
        first = (out.clone(), None if scaled is None else scaled.clone())
      else:
        assert torch.equal(out, first[0]), "mode %d differs from the single-CTA kernel" % mode
        if scaled is not None:
          assert torch.equal(scaled, first[1]), mode
      if games == max(CONV6_GAMES):
        assert conv_items(games * 49, mode) >= 3
  finally:
    lib.mz_conv_set_pair(2)


@gpu
@pytest.mark.parametrize("width,games,ch", [(12, 400, 128), (24, 100, 128), (48, 256, 64)])
def test_conv_representation_widths_match_float64(width, games, ch):
  """The representation tower's 12 x 12 and 24 x 24 (128 channels: single CTA and CTA pair -- mode 2 falls back to
  per-tap loads at these widths) and 48 x 48 (64 channels, always single CTA) residual convolutions, each at >= 3
  tiles on the busiest CTA or cluster, against float64."""
  lib_mod, lib = _lib()
  dev = "cuda"
  torch.manual_seed(width)
  conv = _rand_conv(ch, dev)
  x = muzero.to_padded(torch.rand((games, ch, width, width), device=dev))
  res = muzero.to_padded(torch.rand((games, ch, width, width), device=dev))
  n = games * (width + 1) ** 2
  out = torch.full((n + (width + 1) ** 2, ch), SENTINEL, dtype=torch.bfloat16, device=dev)
  y, mag = ref_conv(muzero.from_padded(x, games, width).double(), conv, RELU | RESIDUAL,
                    residual=muzero.from_padded(res, games, width).double())
  bar = conv_bar(y, mag, 9 * ch)
  try:
    for mode in ((0, 2) if ch == 128 else (2,)):
      assert lib.mz_conv_set_pair(mode) == 0
      out.fill_(SENTINEL)
      _launch_conv(lib_mod, lib, games, width, conv, RELU | RESIDUAL, x, out, residual=res)
      torch.cuda.synchronize()
      items = conv_items(n, mode, ch)
      r = _ratio(muzero.from_padded(out[:n], games, width), y, bar)
      print("conv %d px %d ch games %d mode %d: work items on the busiest CTA/cluster %d, worst err/bar %.3g" % (
          width, ch, games, mode, items, r))
      assert r <= 1.0
      assert items >= 3
      _check_padding(out, games, width, "mode %d" % mode)
  finally:
    lib.mz_conv_set_pair(2)


FC_GAMES = (1, 127, 128, 129, 4096, 9601)


@gpu
@pytest.mark.parametrize("n_out,col", [(1024, 512), (512, 0)])
@pytest.mark.parametrize("games", FC_GAMES)
def test_fc_matches_float64(games, n_out, col):
  """mz_conv_fc_tc as the network calls it: value + policy (1024 outputs at column 512 of the 1536-wide head buffer)
  and reward (512 at column 0), over the padded state.  9601 games: 5 (1024) and 3 (512) work items on the busiest
  CTA.  Columns outside the kernel's range and the row past the last game keep their NaN sentinels."""
  lib_mod, lib = _lib()
  dev = "cuda"
  torch.manual_seed(games + n_out)
  x = muzero.to_padded(torch.relu(torch.randn((games, 128, 6, 6), device=dev)))
  w = muzero._pack_fc((torch.rand((n_out, 4608), device=dev) * 2 - 1) * 4608 ** -0.5, dev)
  bias = torch.randn(n_out, device=dev) * 0.5
  fc = torch.full((games + 1, 1536), float("nan"), device=dev)
  P = lib_mod.ptr
  lib_mod.check(lib.mz_conv_fc_tc(games, P(x), P(w), P(bias), n_out, 1, muzero.C_ptr(fc[:, col:]), 1536,
                                  lib_mod.current_stream()), "mz_conv_fc_tc")
  torch.cuda.synchronize()
  y, mag = ref_fc(muzero.from_padded(x, games).double(), w, bias)
  items = single_items(games, n_out // 128)
  r = _ratio(fc[:games, col:col + n_out], y, FC_K * U * mag)
  print("fc n_out %4d col %3d games %4d: work items on the busiest CTA %d, worst err/bar %.3g" % (n_out, col, games,
                                                                                                  items, r))
  assert r <= 1.0
  outside = torch.ones_like(fc, dtype=torch.bool)
  outside[:games, col:col + n_out] = False
  assert bool(fc[outside].isnan().all())
  if games == max(FC_GAMES):
    assert items >= 3


HEAD_SUPPORT_MIN = {1: 3, 18: -5, 31: -20, 32: 0}


@gpu
@pytest.mark.parametrize("games", [1, 4097])
@pytest.mark.parametrize("outs", [1, 18, 31, 32])
def test_head_matches_float64(outs, games):
  """mz_conv_head: policy logits (to_scalar = 0), and support scalars with and without h^-1 over asymmetric
  supports [support_min, support_min + outs), reading 512 columns at offset 1024 of a 1536-wide buffer whose other
  columns are NaN.  Bars: ref_head."""
  lib_mod, lib = _lib()
  dev = "cuda"
  torch.manual_seed(outs * 7 + games)
  fc = torch.full((games, 1536), float("nan"), device=dev)
  fc[:, 1024:] = torch.relu(torch.randn((games, 512), device=dev))
  w2, b2 = torch.randn((outs, 512), device=dev) * 0.1, torch.randn(outs, device=dev) * 0.5
  P, smin = lib_mod.ptr, HEAD_SUPPORT_MIN[outs]
  for to_scalar, no_tt in ((0, 0), (1, 0), (1, 1)):
    out = torch.full((games + 1, 1 if to_scalar else outs), float("nan"), device=dev)
    lib_mod.check(lib.mz_conv_head(games, muzero.C_ptr(fc[:, 1024:]), 1536, P(w2), P(b2), outs, to_scalar, smin,
                                   no_tt, P(out), out.shape[1], lib_mod.current_stream()), "mz_conv_head")
    torch.cuda.synchronize()
    want, bar = ref_head(fc[:, 1024:], w2, b2, outs, to_scalar, smin, no_tt)
    r = _ratio(out[:games].reshape(want.shape), want, bar)
    print("head outs %2d games %4d to_scalar %d no_tt %d support_min %3d: worst err/bar %.3g" % (
        outs, games, to_scalar, no_tt, smin, r))
    assert r <= 1.0
    assert bool(out[games].isnan().all())


@gpu
def test_gather_4096_games_of_51_nodes():
  """mz_conv_gather over the C5 hidden pool ([4096][51][49][128] bf16, 2.6 GB): picks include the last slot (game
  4095's lies past 2 GiB).  Exact; the rows past the last game keep their sentinel."""
  lib_mod, lib = _lib()
  dev = "cuda"
  G, S1 = 4096, 51
  torch.manual_seed(3)
  pool = torch.randn((G * S1 * 49, 128), device=dev).to(torch.bfloat16)
  node = torch.randint(0, S1, (G,), device=dev, dtype=torch.int32)
  node[::50] = S1 - 1
  node[-1] = S1 - 1
  out = torch.full(((G + 1) * 49, 128), SENTINEL, dtype=torch.bfloat16, device=dev)
  lib_mod.check(lib.mz_conv_gather(G, S1, lib_mod.ptr(node), lib_mod.ptr(pool), lib_mod.ptr(out),
                                   lib_mod.current_stream()), "mz_conv_gather")
  torch.cuda.synchronize()
  want = pool.view(G, S1, 49, 128)[torch.arange(G, device=dev), node.long()].reshape(-1, 128)
  assert torch.equal(out[:G * 49], want)
  assert bool((out[G * 49:] == SENTINEL).all())


# (C_in, C_out, input width, games, im2col budget in games or None): real chunk sizes -- 3 and 4 channels: 682 games
# per chunk; 32: 273; 64 at 96 px: 151; 64 at 48 px (conv2): 606 -- each with a last chunk of one game, and 8 games in
# chunks of 3 / 3 / 2
STRIDED = [(3, 64, 96, 683, None), (4, 64, 96, 8, 3), (32, 64, 96, 274, None), (64, 64, 96, 152, None),
           (64, 128, 48, 607, None)]


@gpu
@pytest.mark.parametrize("cin,cout,w_in,games,budget", STRIDED)
def test_strided_conv_chunks_match_float64_and_one_chunk(cin, cout, w_in, games, budget):
  """MuZeroNetwork._strided (im2col + GEMM into the padded layout, a chunk of games at a time) against float64, and
  bit for bit against the same call with a budget large enough for a single chunk: chunk seams change no row."""
  from model_based_rl_b200.muzero import MuZeroNetwork
  dev = "cuda"
  torch.manual_seed(cin + w_in + games)
  net = MuZeroNetwork(cin, 18, dev, CFG)
  w = (torch.rand((cout, cin, 3, 3), device=dev) * 2 - 1) * (3.0 / (9 * cin)) ** 0.5
  conv = muzero._StridedConv(w, torch.randn(cout, device=dev) * 0.1, dev)
  xin = F.pad(torch.rand((games, cin, w_in, w_in), device=dev), (0, 0, 0, 0, 0, conv.cin_pad - cin))
  x = muzero.to_padded(xin)
  w_out = w_in // 2
  per_game = w_out * w_out * conv.k_pad * 2
  if budget is not None:
    net.IM2COL_BYTES = budget * per_game
  chunk = max(1, min(games, net.IM2COL_BYTES // per_game))
  chunks = [min(chunk, games - g0) for g0 in range(0, games, chunk)]
  assert len(chunks) >= 2
  n = games * (w_out + 1) ** 2
  outs = []
  for budget_bytes in (net.IM2COL_BYTES, games * per_game):
    net.IM2COL_BYTES = budget_bytes
    out = torch.zeros((n + (w_out + 1) ** 2, cout), dtype=torch.bfloat16, device=dev)
    out[n:] = SENTINEL
    net._strided(games, conv, x, w_in, out)
    torch.cuda.synchronize()
    outs.append(out)
  assert torch.equal(outs[0], outs[1]), "chunked and single-chunk results differ"
  y, mag = ref_strided(muzero.from_padded(x, games, w_in).double(), conv)
  r = _ratio(muzero.from_padded(outs[0][:n], games, w_out), y, strided_bar(y, mag, conv))
  items, im2col_items = single_items(chunk * w_out * w_out), stride_items(chunk * w_out * w_out * conv.k_pad // 8)
  print("strided C_in %2d -> %3d at %d px, games %d in chunks %s: work items on the busiest CTA %d (im2col: %d per "
        "thread), worst err/bar %.3g" % (cin, cout, w_in, games, chunks, items, im2col_items, r))
  assert r <= 1.0
  _check_padding(outs[0], games, w_out, "strided")
  if budget is None:
    assert items >= 3 and im2col_items >= 3


@gpu
@pytest.mark.parametrize("w_in", [24, 12])
def test_avgpool_matches_float64(w_in):
  """MuZeroNetwork._pool (AvgPool2d(3, 2, 1)) at 24 -> 12 and 12 -> 6 pixels over 1001 games."""
  from model_based_rl_b200.muzero import MuZeroNetwork
  dev, games = "cuda", 1001
  torch.manual_seed(w_in)
  net = MuZeroNetwork(4, 18, dev, CFG)
  x = muzero.to_padded(torch.rand((games, 128, w_in, w_in), device=dev) * 4 - 1)
  w_out = w_in // 2
  n = games * (w_out + 1) ** 2
  out = torch.zeros((n + (w_out + 1) ** 2, 128), dtype=torch.bfloat16, device=dev)
  out[n:] = SENTINEL
  net._pool(games, x, w_in, out)
  torch.cuda.synchronize()
  y, mag = ref_pool(muzero.from_padded(x, games, w_in).double())
  r = _ratio(muzero.from_padded(out[:n], games, w_out), y, pool_bar(y, mag))
  items = stride_items(games * w_out * w_out * 128 // 8)
  print("avgpool %d -> %d px, %d games: %d items per thread, worst err/bar %.3g" % (w_in, w_out, games, items, r))
  assert r <= 1.0
  if w_in == 24:
    assert items >= 3
  _check_padding(out, games, w_out, "avgpool")


@gpu
def test_comparison_rejects_subtly_wrong_references():
  """Negative controls: the comparisons above, on the kernels' real outputs, against references wrong in ways a
  kernel could be -- one tap's second block of 64 input channels dropped, action + 1 in the action plane, the
  residual taken from the neighbouring game, the value and policy halves of the 1024-wide fc bias swapped.  The
  real reference passes and every wrong one is rejected."""
  lib_mod, lib = _lib()
  dev, games = "cuda", 387
  torch.manual_seed(1)
  flags = RELU | RESIDUAL | ACTION
  conv = _rand_conv(128, dev, action=True)
  x = muzero.to_padded(torch.rand((games, 128, 6, 6), device=dev))
  res = muzero.to_padded(torch.rand((games, 128, 6, 6), device=dev))
  actions = torch.randint(0, 17, (games,), device=dev, dtype=torch.int32)
  out = torch.full(((games + 1) * 49, 128), SENTINEL, dtype=torch.bfloat16, device=dev)
  _launch_conv(lib_mod, lib, games, 6, conv, flags, x, out, residual=res, actions=actions)
  torch.cuda.synchronize()
  got = muzero.from_padded(out[:games * 49], games)
  x64, res64 = muzero.from_padded(x, games).double(), muzero.from_padded(res, games).double()
  dropped = conv_weight64(conv).clone()
  dropped[:, 64:, 1, 2] = 0.0  # tap (ky, kx) = (1, 2), input channels 64..127
  refs = {"real": dict(),
          "tap 5 channels 64-127 dropped": dict(weight=dropped),
          "action + 1": dict(actions=actions + 1),
          "residual of the neighbouring game": dict(residual=torch.roll(res64, 1, dims=0))}
  for label, kw in refs.items():
    args = dict(residual=res64, actions=actions)
    args.update(kw)
    y, mag = ref_conv(x64, conv, flags, **args)
    r = _ratio(got, y, conv_bar(y, mag, 1152))
    print("control conv6 %-34s worst err/bar %.3g -> %s" % (label, r, "accepted" if r <= 1 else "rejected"))
    assert (r <= 1.0) == (label == "real"), label
  # fc, 1024 outputs
  fgames = 300
  xs = muzero.to_padded(torch.relu(torch.randn((fgames, 128, 6, 6), device=dev)))
  w = muzero._pack_fc((torch.rand((1024, 4608), device=dev) * 2 - 1) * 4608 ** -0.5, dev)
  bias = torch.randn(1024, device=dev) * 0.5
  fc = torch.full((fgames, 1536), float("nan"), device=dev)
  P = lib_mod.ptr
  lib_mod.check(lib.mz_conv_fc_tc(fgames, P(xs), P(w), P(bias), 1024, 1, muzero.C_ptr(fc[:, 512:]), 1536,
                                  lib_mod.current_stream()), "mz_conv_fc_tc")
  torch.cuda.synchronize()
  state = muzero.from_padded(xs, fgames).double()
  for label, b in (("real", bias), ("value / policy bias halves swapped", torch.cat((bias[512:], bias[:512])))):
    y, mag = ref_fc(state, w, b)
    r = _ratio(fc[:, 512:], y, FC_K * U * mag)
    print("control fc   %-34s worst err/bar %.3g -> %s" % (label, r, "accepted" if r <= 1 else "rejected"))
    assert (r <= 1.0) == (label == "real"), label


# ---- whole network: batch invariance ---------------------------------------------------------------------------
def _net_outputs(o):
  d = dict(value=o.value, logits=o.policy_logits, hidden=o.hidden_state)
  if not isinstance(o.reward, int):
    d["reward"] = o.reward
  return {k: v.clone() for k, v in d.items()}


def _picked_games(net, G, seed):
  """Games whose rows sit where a layout or loop bug would show: 0 and 2 (game 2 straddles the 6 x 6 convolutions'
  tiles 0 and 1), the games holding the first rows of tiles 148, 149, 296 and 297 (a CTA's second and third tile,
  the pair kernel's second work item), the first and last seams of each strided convolution's im2col chunks, the
  last game, and random ones up to 20."""
  picks = [0, 2, G - 1] + [t * 128 // muzero.ROWS for t in (148, 149, 296, 297)]
  for conv, w_in in ((net.rep_conv1, 96), (net.rep_conv2, 48)):
    chunk = net.IM2COL_BYTES // ((w_in // 2) ** 2 * conv.k_pad * 2)
    if chunk < G:
      last = (G - 1) // chunk * chunk
      picks += [chunk - 1, chunk, last - 1, last]
  picks = sorted(set(p for p in picks if p < G))
  rng = np.random.default_rng(seed)
  while len(picks) < 20:
    p = int(rng.integers(0, G))
    if p not in picks:
      picks.append(p)
  return picks


def _oracle_bars(tag, got, want):
  """The whole-network bars of test_gpu_muzero.test_network_matches_reference_golden: hidden 0.06 worst / 0.01
  mean, logits 0.15, scalars 0.1 worst / 0.05 mean in h space and 0.45 in value space."""
  h = lambda v: np.sign(v) * (np.sqrt(np.abs(v) + 1) - 1) + 0.001 * v
  for k, g in got.items():
    w = want[k].double().cpu().numpy().reshape(g.shape[0], -1)
    g = g.double().cpu().numpy().reshape(g.shape[0], -1)
    err = np.abs(g - w)
    if k == "hidden":
      assert err.max() < 0.06 and err.mean() < 0.01, (tag, k, err.max(), err.mean())
    elif k == "logits":
      assert err.max() < 0.15, (tag, k, err.max())
    else:
      dh = np.abs(h(g) - h(w))
      assert dh.max() < 0.1 and dh.mean() < 0.05 and err.max() < 0.45, (tag, k, dh.max(), err.max())


@gpu
@pytest.mark.parametrize("C_in,G", [(32, 4096), (64, 1000)])
def test_outputs_do_not_depend_on_the_batch(C_in, G):
  """initial_inference and recurrent_inference at G games, then about 20 of those games again in calls of 1 and of
  5 games (other neighbours, other positions in the tiles).  Every row's K order and epilogue are independent of
  where the row sits in a tile, so value, reward, logits and hidden state must be bit-identical; a tile-loop,
  parity, halo, chunk-seam or padding-hygiene bug breaks this exactly.  The big call twice gives the same bits.
  The small calls are checked against the float64 oracle at the whole-network bars, which ties the chain to a
  reference."""
  from model_based_rl_b200.muzero import MuZeroNetwork
  A, dev = 18, "cuda"
  sd = muzero_ref.seeded_state_dict(C_in, A, 40 + C_in)
  net = MuZeroNetwork(C_in, A, dev, CFG)
  net.load_weights(sd)
  gen = torch.Generator(device=dev).manual_seed(C_in)
  obs = torch.rand((G, C_in, 96, 96), device=dev, generator=gen)
  actions = torch.randint(0, A, (G,), device=dev, generator=gen, dtype=torch.int32)
  big_init = _net_outputs(net.initial_inference(obs))
  assert all(torch.equal(v, big_init[k]) for k, v in _net_outputs(net.initial_inference(obs)).items())
  hidden = big_init["hidden"]
  big_rec = _net_outputs(net.recurrent_inference(hidden, actions))
  assert all(torch.equal(v, big_rec[k]) for k, v in _net_outputs(net.recurrent_inference(hidden, actions)).items())
  picks = _picked_games(net, G, seed=C_in)
  print("C_in %d, %d games: recomputed games %s" % (C_in, G, picks))
  rng = np.random.default_rng(C_in)
  groups = [[p] for p in picks]
  order = list(rng.permutation(picks))
  groups += [[int(g) for g in order[i:i + 5]] for i in range(0, len(order), 5)]
  for grp in groups:
    idx = torch.tensor(grp, device=dev)
    small_init = _net_outputs(net.initial_inference(obs[idx]))
    small_rec = _net_outputs(net.recurrent_inference(hidden[idx], actions[idx]))
    for name, small, big in (("initial", small_init, big_init), ("recurrent", small_rec, big_rec)):
      for k, v in small.items():
        if not torch.equal(v, big[k][idx]):
          bad = (v != big[k][idx]).reshape(len(grp), -1).any(dim=1)
          raise AssertionError("%s %s of games %s differs between a call of %d and the call of %d games" % (
              name, k, [g for g, b in zip(grp, bad.tolist()) if b], len(grp), G))
  # the small calls against the float64 oracle
  idx = torch.tensor(picks, device=dev)
  sd64 = {k: (v.double() if v.is_floating_point() else v).to(dev) for k, v in sd.items()}
  with torch.no_grad():
    v0, pol0, h0 = muzero_ref.initial_inference(obs[idx].double(), sd64)
    v1, r1, pol1, h1 = muzero_ref.recurrent_inference(hidden[idx].double(), actions[idx].tolist(), sd64, A)
  _oracle_bars("initial", {k: v[idx] for k, v in big_init.items()}, dict(value=v0, logits=pol0, hidden=h0))
  _oracle_bars("recurrent", {k: v[idx] for k, v in big_rec.items()},
               dict(value=v1, reward=r1, logits=pol1, hidden=h1))


@gpu
def test_conv_search_at_c5_size_replays_in_oracle_and_matches_a_small_engine():
  """One ConvSearch move at the C5 benchmark's size (4096 games, 50 simulations, 18 actions, 32 input planes) as a
  CUDA graph with the hidden pool of 2.6 GB: the oracle replays the search from the recorded network outputs and
  reproduces parents, actions, visit counts, root values and the selected actions bit for bit for every game.  A
  5-game engine fed the same observation, noise, uniform and temperature rows of 5 of those games returns the same
  actions, visits and root values (batch invariance of the whole search)."""
  import oracle
  from model_based_rl_b200.muzero import ConvSearch, MuZeroNetwork
  C_in, A, G, S, dev = 32, 18, 4096, 50, "cuda"
  cfg = types.SimpleNamespace(num_simulations=S, action_space=A, two_players=False, discount=0.997,
                              pb_c_base=19652, pb_c_init=1.25, init_value_score=0.0, known_bounds=[None, None],
                              root_exploration_fraction=0.25)
  net = MuZeroNetwork(C_in, A, dev, CFG)
  net.load_weights(muzero_ref.seeded_state_dict(C_in, A, 99))
  obs = torch.rand((G, C_in, 96, 96), device=dev, generator=torch.Generator(device=dev).manual_seed(5))
  rng = np.random.default_rng(3)
  noise = rng.dirichlet([0.25] * A, size=G)
  u, temp = rng.random(G), rng.choice([0.0, 1.0], size=G)
  cs = ConvSearch(cfg, net, G, use_graph=True)
  cs.enable_record()
  big = [t.clone() for t in cs.search(obs, noise, u, temp)]
  torch.cuda.synchronize()
  assert cs.graph_move is not None
  want = oracle.search(oracle.make_cfg(S, A, False, 0.997), cs.root_logits.cpu().numpy(), noise=noise,
                       noise_frac=0.25, rec_value=cs.record[0].cpu().numpy().T,
                       rec_reward=cs.record[1].cpu().numpy().T,
                       rec_logits=cs.record[2].cpu().numpy().transpose(1, 0, 2))
  assert np.array_equal(cs.trace[0].cpu().numpy().T, want["trace_parent"])
  assert np.array_equal(cs.trace[1].cpu().numpy().T, want["trace_action"])
  visits = cs.eng.visits.cpu().numpy()
  assert np.array_equal(visits, want["visits"])
  assert np.array_equal(big[1].cpu().numpy(), want["root_value"])
  acts = big[0].cpu().numpy()
  assert all(int(acts[i]) == oracle.select_action(want["visits"][i], temp[i], u[i]) for i in range(G))
  print("ConvSearch %d games x %d simulations: oracle replay bit-exact" % (G, S))
  idx = [0, 389, 2047, 3001, G - 1]
  small = ConvSearch(cfg, net, len(idx), use_graph=True)
  got = [t.clone() for t in small.search(obs[idx], noise[idx], u[idx], temp[idx])]
  torch.cuda.synchronize()
  ti = torch.tensor(idx, device=dev)
  for name, a, b in zip(("actions", "root_value", "child_visits", "initial value"), got, big):
    assert torch.equal(a, b[ti]), name
  assert np.array_equal(small.eng.visits.cpu().numpy(), visits[idx])
