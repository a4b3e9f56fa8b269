"""Inference side of the reference's MuZeroNetwork (networks.py:372-554) on tcgen05 tensor cores.

`MuZeroNetwork` keeps the reference's constructor, `initial_inference` / `recurrent_inference`
(NetworkOutput(value, reward, policy_logits, hidden_state), eval mode: scalars after the
softmax-expectation + h^-1 of config.py:27-33) and `load_weights` / `get_weights` with the
reference's state-dict keys.  Underneath, every dense layer of `recurrent_inference` -- 65 3x3
convolutions with BatchNorm folded, the three Linear(4608 -> 512) heads -- is one launch of the
implicit-GEMM kernel in csrc/mz_conv_tc.cu on bf16 activations in a flat padded channels-last layout
(49 rows x 128 channels per game: a zero row of 7, then 6 image rows of 6 pixels + 1 zero); the
hidden-state pool of the search holds states in the same layout, is gathered by one small copy
kernel per simulation and written in place by the last dynamics convolution.

Representation tower (`initial_inference`, once per move): the residual blocks at 48 x 48 (64
channels), 24 x 24, 12 x 12 and 6 x 6 pixels run on the same implicit-GEMM kernel, the two strided
convolutions as im2col + the kernel's plain-GEMM mode, the two average pools as a small kernel; the
only torch operation left is the layout change of the raw observation.
"""
import numpy as np
import torch
import torch.nn.functional as F

from . import _lib
from .networks import NetworkOutput

CH = 128          # channels of the hidden state
ROWS = 49         # rows per game: 7 zero | 6 x (6 pixels + 1 zero)
K_FC = ROWS * CH  # 6272: flattened padded state
RELU, RESIDUAL, ACTION, SCALE = 1, 2, 4, 8
BN_EPS = 1e-5
NARROW_HEAD_BINS = 32    # value / reward supports up to this width: mz_conv_head (one warp per game)
MAX_SUPPORT_BINS = 1024  # wider ones: mz_conv_support_head_tc, which takes up to this many bins


def to_padded(state):
  """[B, 128, W, W] float -> [B * (W + 1)^2, 128] bf16 rows: channels last, one zero row on top and one
  zero pixel after every image row (the zero padding neighbouring games share)."""
  b, c, w = state.shape[0], state.shape[1], state.shape[-1]
  x = F.pad(state.permute(0, 2, 3, 1), (0, 0, 0, 1, 1, 0))    # [B, W + 1, W + 1, C]
  return x.reshape(b * (w + 1) * (w + 1), c).to(torch.bfloat16).contiguous()


def from_padded(rows, b, width=6):
  """[B * (W + 1)^2, C] bf16 rows -> [B, C, W, W] float32."""
  x = rows.reshape(b, width + 1, width + 1, rows.shape[-1])[:, 1:, :width, :]
  return x.permute(0, 3, 1, 2).float().contiguous()


def padding_rows(rows, b, width=6):
  """The padding rows of every game (must stay zero)."""
  x = rows.reshape(b, width + 1, width + 1, rows.shape[-1])
  return torch.cat((x[:, 0], x[:, 1:, width]), dim=1)


class _Conv(object):
  """One folded convolution: packed bf16 weights [C][9 C] (C = 64 or 128), float32 bias (+ action-plane
  term of MuZeroDynamics.conv)."""

  def __init__(self, weight, conv_bias, bn, device):
    w = weight.to(device, torch.float32)
    if bn is not None:
      gamma, beta, mean, var = [t.to(device, torch.float32) for t in bn]
      scale = gamma / torch.sqrt(var + BN_EPS)
      w = w * scale[:, None, None, None]
      bias = beta - mean * scale
      if conv_bias is not None:
        bias = bias + conv_bias.to(device, torch.float32) * scale
    else:
      bias = (conv_bias.to(device, torch.float32) if conv_bias is not None
              else torch.zeros(w.shape[0], device=device))
    self.channels = c = int(w.shape[0])
    self.plane = None
    if w.shape[1] == CH + 1:  # MuZeroDynamics.conv: the 129th input channel is the action plane
      ones = torch.ones((1, 1, 6, 6), device=device)
      # what a constant plane of ones contributes at each interior pixel (zero padding outside)
      self.plane = F.conv2d(ones, w[:, CH:], None, 1, 1)[0].permute(1, 2, 0).reshape(36, CH).contiguous()
      w = w[:, :CH]
    self.w = w.permute(0, 2, 3, 1).reshape(c, 9 * c).to(torch.bfloat16).contiguous()
    self.bias = bias.contiguous()


class _StridedConv(object):
  """Conv2d(Cin -> Cout, 3x3, stride 2, padding 1, bias) as im2col + GEMM: weights [Cout][k_pad] bf16
  with k = (ky * 3 + kx) * Cin_pad + c (input channels padded to a multiple of 8, K to one of 64)."""

  def __init__(self, weight, bias, device):
    w = weight.to(device, torch.float32)
    cout, cin = int(w.shape[0]), int(w.shape[1])
    self.cin_pad = (cin + 7) // 8 * 8
    self.cout = cout
    self.k_pad = (9 * self.cin_pad + 63) // 64 * 64
    wp = torch.zeros((cout, 3, 3, self.cin_pad), dtype=torch.float32, device=device)
    wp[..., :cin] = w.permute(0, 2, 3, 1)
    full = torch.zeros((cout, self.k_pad), dtype=torch.float32, device=device)
    full[:, :9 * self.cin_pad] = wp.reshape(cout, 9 * self.cin_pad)
    self.w = full.to(torch.bfloat16).contiguous()
    self.bias = bias.to(device, torch.float32).contiguous()


def _pack_support_head(weight, bias, device):
  """Second layer Linear(512 -> bins) of a value or reward head: float32 [bins][512] for mz_conv_head up to
  NARROW_HEAD_BINS bins, above that the bf16 [bins][512] B operand of mz_conv_support_head_tc (rounded here,
  once).  The bias stays float32."""
  w = weight.to(device, torch.float32)
  if w.shape[0] > NARROW_HEAD_BINS:
    w = w.to(torch.bfloat16)
  return w.contiguous(), bias.to(device, torch.float32).contiguous()


def _pack_fc(weight, device):
  """Linear(128*6*6 -> n) weight [n, c*36 + y*6 + x] -> [n, (7 + y*7 + x)*128 + c] bf16."""
  n = weight.shape[0]
  w = weight.to(device, torch.float32).reshape(n, CH, 6, 6).permute(0, 2, 3, 1)
  out = torch.zeros((n, ROWS, CH), dtype=torch.float32, device=device)
  out[:, 7:].view(n, 6, 7, CH)[:, :, :6, :] = w
  return out.reshape(n, K_FC).to(torch.bfloat16).contiguous()


class MuZeroNetwork(object):

  accepts_device_actions = True
  training = False

  def __init__(self, input_channels, action_space, device, config):
    _lib.require_cuda()
    if getattr(config, 'no_support', False):
      raise NotImplementedError("no_support is implemented for the FCNetwork family (networks.FCNetwork, "
                                "learners.FCNetworkTrain), not for the conv network")
    self.lib = _lib.load()
    self.device = _lib.normalize_device(device)
    self.input_channels = int(input_channels)
    self.action_space = int(action_space)
    if self.action_space > 32:
      raise NotImplementedError("the head kernel supports action_space <= 32")
    self.value_min, self.value_max = [int(v) for v in config.value_support]
    self.reward_min, self.reward_max = [int(v) for v in config.reward_support]
    self.value_bins = self.value_max - self.value_min + 1
    self.reward_bins = self.reward_max - self.reward_min + 1
    self.no_target_transform = bool(getattr(config, 'no_target_transform', False))
    self._state = None
    self._bufs = {}
    self.launches = 0  # kernels of csrc/mz_conv_tc.cu launched so far

  # -- weights -----------------------------------------------------------------------------------
  @_lib.on_device
  def load_weights(self, weights):
    """Accepts the reference's state dict (networks.py:549-550); folds BatchNorm (eval statistics)
    into the convolutions and packs everything for the tensor-core kernels."""
    for name, bins in (('value', self.value_bins), ('reward', self.reward_bins)):
      if bins > MAX_SUPPORT_BINS:
        raise ValueError("the %s support has %d bins; MuZeroNetwork's support heads take at most %d"
                         % (name, bins, MAX_SUPPORT_BINS))
    dev = self.device
    sd = {k: torch.as_tensor(v).detach() for k, v in weights.items()}
    # a snapshot (the reference hands weights over as `.cpu()` copies, networks.py:36-40): later in-place
    # changes of the caller's tensors must not reach the search network
    self._state = {k: v.to(dev, copy=True) for k, v in sd.items()}
    # the packed tensors below are rebuilt: anything that captured their addresses (ConvSearch's CUDA graph)
    # must be re-captured -- engines compare this counter before every move
    self.weights_version = getattr(self, 'weights_version', 0) + 1

    def bn(p):
      return (sd[p + '.weight'], sd[p + '.bias'], sd[p + '.running_mean'], sd[p + '.running_var'])

    def tower(p):
      convs = []
      for i in range(16):
        b = '%s.resblocks.%d' % (p, i)
        convs.append(_Conv(sd[b + '.conv1.weight'], None, bn(b + '.bn1'), dev))
        convs.append(_Conv(sd[b + '.conv2.weight'], None, bn(b + '.bn2'), dev))
      return convs

    # representation tower: every layer runs on this library's kernels (strided convolutions as
    # im2col + GEMM, residual blocks on the implicit-GEMM kernel, average pools)
    r = 'representation_head'

    def blocks(p, n):
      convs = []
      for i in range(n):
        b = '%s.%d' % (p, i)
        convs.append(_Conv(sd[b + '.conv1.weight'], None, bn(b + '.bn1'), dev))
        convs.append(_Conv(sd[b + '.conv2.weight'], None, bn(b + '.bn2'), dev))
      return convs

    self.rep_conv1 = _StridedConv(sd[r + '.conv1.weight'], sd[r + '.conv1.bias'], dev)
    self.rep_blocks1 = blocks(r + '.resblocks1', 2)   # 64 channels at 48 x 48
    self.rep_conv2 = _StridedConv(sd[r + '.conv2.weight'], sd[r + '.conv2.bias'], dev)
    self.rep_blocks2 = blocks(r + '.resblocks2', 3)
    self.rep_blocks3 = blocks(r + '.resblocks3', 3)
    self.rep_tower = blocks(r + '.resblocks', 16)
    d, q = 'dynamics_head', 'prediction_head'
    if sd[d + '.conv.weight'].shape != (CH, CH + 1, 3, 3):
      raise ValueError("dynamics_head.conv.weight has shape %s" % (tuple(sd[d + '.conv.weight'].shape),))
    self.dyn_conv = _Conv(sd[d + '.conv.weight'], sd[d + '.conv.bias'], bn(d + '.bn'), dev)
    self.dyn_tower = tower(d)
    self.pred_tower = tower(q)
    f32 = lambda k: sd[k].to(dev, torch.float32).contiguous()
    self.rew_fc1_w = _pack_fc(sd[d + '.fc1.weight'], dev)
    self.rew_fc1_b = f32(d + '.fc1.bias')
    self.rew_fc2_w, self.rew_fc2_b = _pack_support_head(sd[d + '.fc2.weight'], sd[d + '.fc2.bias'], dev)
    # value and policy heads read the same state: one GEMM with 1024 outputs
    self.vp_fc1_w = torch.cat((_pack_fc(sd[q + '.fc_value.weight'], dev),
                               _pack_fc(sd[q + '.fc_policy.weight'], dev)), dim=0).contiguous()
    self.vp_fc1_b = torch.cat((f32(q + '.fc_value.bias'), f32(q + '.fc_policy.bias'))).contiguous()
    self.val_fc2_w, self.val_fc2_b = _pack_support_head(sd[q + '.fc_value_o.weight'], sd[q + '.fc_value_o.bias'], dev)
    self.pol_fc2_w, self.pol_fc2_b = f32(q + '.fc_policy_o.weight'), f32(q + '.fc_policy_o.bias')
    if self.rew_fc2_w.shape[0] != self.reward_bins or self.val_fc2_w.shape[0] != self.value_bins or \
        self.pol_fc2_w.shape[0] != self.action_space:
      raise ValueError("head widths do not match config supports / action_space")

  load_state_dict = load_weights

  def get_weights(self):
    return {k: v.cpu() for k, v in self._state.items()}

  def state_dict(self):
    return dict(self._state)

  def to(self, device):
    if torch.device(device).type != 'cuda':
      raise RuntimeError("the B200 MuZeroNetwork only runs on CUDA devices")
    return self

  def eval(self):
    return self

  def train(self, mode=True):
    if mode:
      raise NotImplementedError("training stays with the reference's torch module; this class is "
                                "the inference path (load_weights moves parameters across)")
    return self

  # -- buffers ---------------------------------------------------------------------------------------
  def buffers(self, games, width=6, channels=CH):
    """Scratch activations for `games` games of width x width pixels: three flat padded bf16 buffers
    (+ one for the scaled state) and the head hidden layer [games][reward 512 | value 512 | policy
    512] float32."""
    b = self._bufs.get((games, width, channels))
    if b is None:
      dev = self.device
      rows = games * (width + 1) * (width + 1)
      b = dict(x=[torch.zeros((rows, channels), dtype=torch.bfloat16, device=dev) for _ in range(3)])
      if width == 6:
        b['scaled'] = torch.zeros((rows, CH), dtype=torch.bfloat16, device=dev)
        b['fc'] = torch.zeros((games, 1536), dtype=torch.float32, device=dev)
      self._bufs[(games, width, channels)] = b
    return b

  # -- launches --------------------------------------------------------------------------------------
  def _conv(self, games, conv, x, flags, out, residual=None, actions=None, out_scaled=None, pool_out=None,
            pool_base=None, width=6):
    P = _lib.ptr
    _lib.check(self.lib.mz_conv3x3_tc(games, width, conv.channels, P(x), P(conv.w), P(conv.bias), flags,
                                      P(conv.plane) if flags & ACTION else None, P(actions),
                                      self.action_space, P(residual), P(out), P(out_scaled), P(pool_out),
                                      P(pool_base), _lib.current_stream()), "mz_conv3x3_tc")
    self.launches += 1

  def _tower(self, games, convs, x, bufs, last_flags=0, out_scaled=None, pool_out=None, pool_base=None,
             width=6):
    """len(convs) / 2 ResidualBlocks (networks.py:372-391) starting from the flat tensor `x`.  Returns
    the scratch buffer holding the (unscaled) output."""
    cur, n = x, len(convs) // 2
    for i in range(n):
      t, o = [b for b in bufs if b.data_ptr() != cur.data_ptr()][:2]
      self._conv(games, convs[2 * i], cur, RELU, t, width=width)
      extra = last_flags if i == n - 1 else 0
      self._conv(games, convs[2 * i + 1], t, RELU | RESIDUAL | extra, o, residual=cur,
                 out_scaled=out_scaled if extra else None, pool_out=pool_out if extra else None,
                 pool_base=pool_base if extra else None, width=width)
      cur = o
    return cur

  def _support_head(self, games, hidden, w2, b2, bins, support_min, out):
    """Linear(512 -> bins) of the value or reward head over `hidden` (a view of the fc buffer, row stride 1536)
    + softmax expectation + h^-1 -> out [games] f32.  Supports of up to NARROW_HEAD_BINS bins run on
    mz_conv_head, wider ones on the tensor-core kernel."""
    P, st, ntt = _lib.ptr, _lib.current_stream(), int(self.no_target_transform)
    if bins <= NARROW_HEAD_BINS:
      _lib.check(self.lib.mz_conv_head(games, C_ptr(hidden), 1536, P(w2), P(b2), bins, 1, support_min, ntt,
                                       P(out), 1, st), "mz_conv_head")
    else:
      _lib.check(self.lib.mz_conv_support_head_tc(games, C_ptr(hidden), 1536, P(w2), P(b2), bins, support_min, ntt,
                                                  P(out), 1, st), "mz_conv_support_head_tc")

  def run_recurrent(self, games, state, actions, value, reward, logits, pool_out=None, pool_base=None):
    """recurrent_inference (networks.py:31-34) for `games` games on the current stream.
      state      [games * 49][128] bf16 (flat padded layout)
      actions    [games] int32 (device)
      value, reward [games] f32, logits [games][A] f32 (device)
      pool_out / pool_base: also write game g's scaled next state at rows pool_base[g].. of pool_out
    Returns the flat scaled next state (a scratch buffer owned by the network)."""
    b = self.buffers(games)
    X, scaled = b['x'], b['scaled']
    P = _lib.ptr
    st = _lib.current_stream()
    # dynamics: conv(129 -> 128) + bn + relu, 16 blocks, scale_state; reward head on the unscaled state
    self._conv(games, self.dyn_conv, state, RELU | ACTION, X[0], actions=actions)
    raw = self._tower(games, self.dyn_tower, X[0], X, last_flags=SCALE, out_scaled=scaled,
                      pool_out=pool_out, pool_base=pool_base)
    _lib.check(self.lib.mz_conv_fc_tc(games, P(raw), P(self.rew_fc1_w), P(self.rew_fc1_b), 512, 1,
                                      P(b['fc']), 1536, st), "mz_conv_fc_tc")
    self._support_head(games, b['fc'], self.rew_fc2_w, self.rew_fc2_b, self.reward_bins, self.reward_min, reward)
    self.launches += 2
    self.run_prediction(games, scaled, value, logits)  # prediction on the scaled state
    return scaled

  def run_prediction(self, games, state, value, logits):
    """prediction (networks.py:465-480 + inverse value transform) from a flat padded bf16 state."""
    b = self.buffers(games)
    P = _lib.ptr
    st = _lib.current_stream()
    out = self._tower(games, self.pred_tower, state, b['x'])
    fc_vp = b['fc'][:, 512:]
    _lib.check(self.lib.mz_conv_fc_tc(games, P(out), P(self.vp_fc1_w), P(self.vp_fc1_b), 1024, 1,
                                      C_ptr(fc_vp), 1536, st), "mz_conv_fc_tc")
    self._support_head(games, fc_vp, self.val_fc2_w, self.val_fc2_b, self.value_bins, self.value_min, value)
    _lib.check(self.lib.mz_conv_head(games, C_ptr(b['fc'][:, 1024:]), 1536, P(self.pol_fc2_w),
                                     P(self.pol_fc2_b), self.action_space, 0, 0, 0, P(logits),
                                     self.action_space, st), "mz_conv_head")
    self.launches += 3

  # -- reference interface ---------------------------------------------------------------------------
  IM2COL_BYTES = 384 << 20  # scratch budget for the patch matrix of a strided convolution

  def _strided(self, games, conv, x, w_in, out):
    """Conv2d(stride 2) over `games` padded images x [games * (w_in + 1)^2][Cin_pad] -> rows of the
    padded (w_in / 2)-pixel layout `out` (im2col + GEMM, a chunk of games at a time)."""
    P, st = _lib.ptr, _lib.current_stream()
    w_out, cin = w_in // 2, conv.cin_pad
    per_game = w_out * w_out * conv.k_pad * 2
    chunk = max(1, min(games, self.IM2COL_BYTES // per_game))
    cols = self._bufs.get(('im2col', chunk * per_game))
    if cols is None:
      cols = torch.empty(chunk * per_game, dtype=torch.uint8, device=self.device)
      self._bufs[('im2col', chunk * per_game)] = cols
    in_rows, out_rows = (w_in + 1) * (w_in + 1), (w_out + 1) * (w_out + 1)
    for g0 in range(0, games, chunk):
      n = min(chunk, games - g0)
      _lib.check(self.lib.mz_conv_im2col_s2(n, w_in, cin, conv.k_pad, C_ptr(x[g0 * in_rows:]), P(cols), st),
                 "mz_conv_im2col_s2")
      _lib.check(self.lib.mz_conv_gemm_to_padded(n, w_out, conv.k_pad, conv.cout, P(cols), P(conv.w),
                                                 P(conv.bias), 0, C_ptr(out[g0 * out_rows:]), st),
                 "mz_conv_gemm_to_padded")
    self.launches += 2 * ((games + chunk - 1) // chunk)

  def _pool(self, games, x, w_in, out):
    _lib.check(self.lib.mz_conv_avgpool(games, w_in, CH, _lib.ptr(x), _lib.ptr(out), _lib.current_stream()),
               "mz_conv_avgpool")
    self.launches += 1

  def representation_rows(self, observation):
    """MuZeroRepresentation + scale_state (networks.py:412-426, 500-503) -> the scaled 6 x 6 state in
    the flat padded bf16 layout (a scratch buffer owned by the network).  Only the layout change of
    the raw observation (NCHW float -> padded channels-last bf16) is a torch operation."""
    obs = torch.as_tensor(observation).to(self.device, torch.float32)
    g, cin, w0 = obs.shape[0], obs.shape[1], obs.shape[-1]
    if w0 != 96 or obs.shape[-2] != 96:
      raise ValueError("MuZeroRepresentation expects 96 x 96 observations")
    c1 = self.rep_conv1
    if cin < c1.cin_pad:
      obs = F.pad(obs, (0, 0, 0, 0, 0, c1.cin_pad - cin))
    x = to_padded(obs)                                          # [g * 97^2][cin_pad]
    b48 = self.buffers(g, 48, 64)['x']
    self._strided(g, c1, x, 96, b48[0])                         # conv1: 96 -> 48, 64 channels
    s1 = self._tower(g, self.rep_blocks1, b48[0], b48, width=48)
    b24 = self.buffers(g, 24)['x']
    self._strided(g, self.rep_conv2, s1, 48, b24[0])            # conv2: 48 -> 24, 128 channels
    s2 = self._tower(g, self.rep_blocks2, b24[0], b24, width=24)
    b12 = self.buffers(g, 12)['x']
    self._pool(g, s2, 24, b12[0])
    s3 = self._tower(g, self.rep_blocks3, b12[0], b12, width=12)
    b = self.buffers(g)
    self._pool(g, s3, 12, b['x'][0])
    self._tower(g, self.rep_tower, b['x'][0], b['x'], last_flags=SCALE, out_scaled=b['scaled'])
    return b['scaled']

  def representation(self, observation):
    """networks.py:500-503: [B, C, 96, 96] -> scaled hidden state [B, 128, 6, 6] float32."""
    with torch.inference_mode():
      rows = self.representation_rows(observation)
      return from_padded(rows, rows.shape[0] // ROWS)

  def initial_inference(self, observation):
    """networks.py:26-29 (eval mode)."""
    with torch.inference_mode():
      rows = self.representation_rows(observation).clone()  # the scratch buffer is reused below
      b = rows.shape[0] // ROWS
      value = torch.zeros(b, dtype=torch.float32, device=self.device)
      logits = torch.zeros((b, self.action_space), dtype=torch.float32, device=self.device)
      self.run_prediction(b, rows, value, logits)
    return NetworkOutput(value.reshape(b, 1), 0, logits, from_padded(rows, b))

  def recurrent_inference(self, hidden_state, action):
    """networks.py:31-34 (eval mode): hidden_state [B, 128, 6, 6], action: B ints (or an int32 CUDA
    tensor)."""
    with torch.inference_mode():
      b = hidden_state.shape[0]
      dev = self.device
      rows = to_padded(hidden_state.to(dev, torch.float32))
      acts = torch.as_tensor(action, dtype=torch.int32).to(dev).reshape(-1).contiguous()
      value = torch.zeros(b, dtype=torch.float32, device=dev)
      reward = torch.zeros(b, dtype=torch.float32, device=dev)
      logits = torch.zeros((b, self.action_space), dtype=torch.float32, device=dev)
      nxt = self.run_recurrent(b, rows, acts, value, reward, logits)
      hidden = from_padded(nxt, b)
    return NetworkOutput(value.reshape(b, 1), reward.reshape(b, 1), logits, hidden)


class ConvSearch(object):
  """The per-move body of Actor.play_game (actors.py:131-153) for G games with MuZeroNetwork.

  Hidden states live in a bf16 pool [G][S+1][49 rows][128] (the padded layout the kernels read):
  one copy kernel per simulation gathers `search_path[-2].hidden_state` into the flat activation
  buffer and the last dynamics convolution writes the scaled next state straight into slot sim+1.
  The search part of a move (72 launches per simulation) is captured in one CUDA graph."""

  def __init__(self, config, net, num_games, noise_frac=None, use_graph=True):
    from .mcts import BatchedMCTS
    G, A, dev = int(num_games), int(config.action_space), net.device
    self.net, self.G, self.A, self.S = net, G, A, int(config.num_simulations)
    self.noise_frac = float(getattr(config, 'root_exploration_fraction', 0.25)
                            if noise_frac is None else noise_frac)
    self.eng = BatchedMCTS(config, G, hidden_words=0, device=dev)
    S = self.S
    self.pool = torch.zeros((G * (S + 1) * ROWS, CH), dtype=torch.bfloat16, device=dev)
    slot0 = torch.arange(G, device=dev, dtype=torch.int64) * (S + 1)
    self.out_base = ((slot0[None, :] + torch.arange(1, S + 1, device=dev)[:, None]) * ROWS).to(torch.int32)
    self.root_base = (slot0 * ROWS).to(torch.int32)
    self.gathered = torch.zeros((G * ROWS, CH), dtype=torch.bfloat16, device=dev)
    self.noise = torch.zeros((G, A), dtype=torch.float64, device=dev)
    self.legal = torch.full((G,), (1 << A) - 1, dtype=torch.int64, device=dev).to(torch.int32)
    self.to_play = torch.ones(G, dtype=torch.int8, device=dev)
    self.temperature = torch.ones(G, dtype=torch.float64, device=dev)
    self.uniforms = torch.zeros(G, dtype=torch.float64, device=dev)
    self.root_logits = torch.zeros((G, A), dtype=torch.float32, device=dev)
    self.init_value = torch.zeros(G, dtype=torch.float32, device=dev)
    self.value = torch.zeros(G, dtype=torch.float32, device=dev)
    self.reward = torch.zeros(G, dtype=torch.float32, device=dev)
    self.logits = torch.zeros((G, A), dtype=torch.float32, device=dev)
    self.use_graph, self.graph, self.use_noise = use_graph, None, True
    self.record = None
    self.launches_per_move = 0

  def enable_record(self):
    dev, G, S, A = self.net.device, self.G, self.S, self.A
    self.record = (torch.zeros((S, G), dtype=torch.float32, device=dev),
                   torch.zeros((S, G), dtype=torch.float32, device=dev),
                   torch.zeros((S, G, A), dtype=torch.float32, device=dev))
    self.eng.enable_trace()
    self.graph = self.graph_move = None

  @property
  def trace(self):
    return self.eng.trace

  def set_roots(self, observation):
    """initial_inference for every game: representation (torch operators, float32) -> pool slot 0,
    prediction on the tensor cores -> root logits / value."""
    with torch.inference_mode():
      rows = self.net.representation_rows(observation)
      self.pool.view(self.G, self.S + 1, ROWS, CH)[:, 0] = rows.view(self.G, ROWS, CH)
      self.net.run_prediction(self.G, self.pool_root(), self.init_value, self.root_logits)

  def pool_root(self):
    """Flat copy of the roots' states (slot 0 of every game)."""
    self.gathered.view(self.G, ROWS, CH).copy_(self.pool.view(self.G, self.S + 1, ROWS, CH)[:, 0])
    return self.gathered

  def _enqueue(self):
    eng, net, lib, P = self.eng, self.net, self.net.lib, _lib.ptr
    st = _lib.current_stream()
    tree = eng.tree
    n0 = net.launches
    _lib.check(lib.mz_tree_set_root(tree, P(self.root_logits), P(self.legal),
                                    P(self.noise) if self.use_noise else None, self.noise_frac,
                                    P(self.to_play), None, st), "mz_tree_set_root")
    _lib.check(lib.mz_tree_step(tree, -1, None, None, None, None, None, *eng._trace_ptrs(0), st),
               "mz_tree_step")
    for sim in range(self.S):
      if self.record is not None:
        v, r, l = self.record[0][sim], self.record[1][sim], self.record[2][sim]
      else:
        v, r, l = self.value, self.reward, self.logits
      _lib.check(lib.mz_conv_gather(self.G, self.S + 1, P(eng.leaf_parent), P(self.pool), P(self.gathered),
                                    st), "mz_conv_gather")
      net.run_recurrent(self.G, self.gathered, eng.leaf_action, v, r, l, pool_out=self.pool,
                        pool_base=self.out_base[sim])
      _lib.check(lib.mz_tree_step(tree, sim, P(v), P(r), P(l), None, None, *eng._trace_ptrs(sim + 1), st),
                 "mz_tree_step")
    _lib.check(lib.mz_tree_root_stats(tree, P(eng.visits), P(eng.child_visits), P(eng.root_value),
                                      P(eng.minmax), st), "mz_tree_root_stats")
    _lib.check(lib.mz_select_action(self.G, self.A, P(eng.visits), P(self.legal), P(self.temperature),
                                    P(self.uniforms), P(eng.actions), st), "mz_select_action")
    self.launches_per_move = net.launches - n0 + 4 + 2 * self.S

  def run(self):
    """The search of one move (roots already set) on the current stream."""
    if not self.use_graph:
      self._enqueue()
      return
    if getattr(self, '_graph_weights', None) != getattr(self.net, 'weights_version', 0):
      self.graph = None  # load_weights rebuilt the packed weights: the captured addresses are stale
      self._graph_weights = getattr(self.net, 'weights_version', 0)
    if self.graph is None:
      self._enqueue()  # warm-up outside capture (cudaFuncSetAttribute, lazy module loading)
      torch.cuda.synchronize()
      self.graph = torch.cuda.CUDAGraph()
      with torch.cuda.graph(self.graph):
        self._enqueue()
    self.graph.replay()

  def run_move(self, observation):
    """initial_inference (representation tower + prediction) AND the search of one move as ONE CUDA graph over a
    static observation buffer: the ~190 launches of the representation join the 3 604 of the search, no eager
    launch is left in a move."""
    obs = torch.as_tensor(observation)
    if not self.use_graph:
      self.set_roots(obs.to(self.net.device, non_blocking=True))
      self._enqueue()
      return
    st = getattr(self, '_obs_static', None)
    if st is None or st.shape != obs.shape:
      st = self._obs_static = torch.empty(obs.shape, dtype=torch.float32, device=self.net.device)
      self.graph_move = None
    st.copy_(obs, non_blocking=True)
    if getattr(self, '_graph_move_weights', None) != getattr(self.net, 'weights_version', 0):
      self.graph_move = None  # load_weights rebuilt the packed weights: the captured addresses are stale
      self._graph_move_weights = getattr(self.net, 'weights_version', 0)
    if getattr(self, 'graph_move', None) is None:
      self.set_roots(st)  # warm-up outside capture (scratch buffers, cudaFuncSetAttribute, lazy module loading)
      self._enqueue()
      torch.cuda.synchronize()
      self.graph_move = torch.cuda.CUDAGraph()
      with torch.cuda.graph(self.graph_move):
        self.set_roots(st)
        self._enqueue()
    self.graph_move.replay()

  @_lib.on_device
  def search(self, observation, noise=None, uniforms=None, temperature=None):
    """observation [G, C, 96, 96] (device or host); returns device tensors (actions [G] i32,
    root_value [G] f64, child_visits [G, A] f64, initial value [G] f32)."""
    if noise is not None:
      self.noise.copy_(torch.as_tensor(noise), non_blocking=True)
    if uniforms is not None:
      self.uniforms.copy_(torch.as_tensor(uniforms), non_blocking=True)
    if temperature is not None:
      self.temperature.copy_(torch.as_tensor(temperature), non_blocking=True)
    self.run_move(observation)
    eng = self.eng
    return eng.actions, eng.root_value, eng.child_visits, self.init_value


  @_lib.on_device
  def search_host(self, obs, noise=None, uniforms=None, temperature=None, legal=None, to_play=None):
    """Same call as `FCSearch.search_host` (networks.py), so `selfplay.BatchedActor(search=...)` drives either
    engine: HOST arrays in -- frames [G, C, 96, 96] float32, Dirichlet noise [G, A] float64 (row g: one value
    per legal action of game g), uniforms / temperature [G] float64, optional legal-action bit masks [G] and
    to_play [G] -- and pinned host tensors out: actions [G] i32, root_value [G] f64, child_visits [G, A] f64,
    initial-inference value [G] f32 (actors.py:131-153).  Both copies are part of the call."""
    dev = self.net.device
    if getattr(self, '_host_out', None) is None:
      G, A = self.G, self.A
      self._host_out = (torch.zeros(G, dtype=torch.int32).pin_memory(), torch.zeros(G, dtype=torch.float64).pin_memory(),
                        torch.zeros((G, A), dtype=torch.float64).pin_memory(), torch.zeros(G, dtype=torch.float32).pin_memory())
    if legal is not None:
      self.legal.copy_(torch.from_numpy(np.ascontiguousarray(np.asarray(legal).astype(np.int64).astype(np.int32))),
                       non_blocking=True)
    if to_play is not None:
      self.to_play.copy_(torch.from_numpy(np.ascontiguousarray(np.asarray(to_play, dtype=np.int8))), non_blocking=True)
    self.use_noise = noise is not None or self.use_noise
    obs = torch.as_tensor(obs)
    if obs.dtype != torch.float32:
      raise TypeError("search_host expects float32 frames")
    outs = self.search(obs, noise, uniforms, temperature)
    for h, d in zip(self._host_out, outs):
      h.copy_(d, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return self._host_out


def C_ptr(t):
  """Pointer of a (possibly offset) view."""
  import ctypes
  return ctypes.c_void_p(t.data_ptr())


def random_state_dict(input_channels, action_space, value_bins=31, reward_bins=31, seed=1234):
  """Random-init weights of the MuZeroNetwork architecture under the reference's state-dict keys
  (torch's default Conv2d / Linear initialisation, BatchNorm at its initial statistics)."""
  import math
  g = torch.Generator().manual_seed(seed)
  sd = {}

  def uniform(shape, bound):
    return (torch.rand(shape, generator=g) * 2 - 1) * bound

  def conv(p, cin, cout, bias):
    bound = 1.0 / math.sqrt(cin * 9)
    sd[p + '.weight'] = uniform((cout, cin, 3, 3), bound)
    if bias:
      sd[p + '.bias'] = uniform((cout,), bound)

  def bn(p, c):
    sd[p + '.weight'], sd[p + '.bias'] = torch.ones(c), torch.zeros(c)
    sd[p + '.running_mean'], sd[p + '.running_var'] = torch.zeros(c), torch.ones(c)
    sd[p + '.num_batches_tracked'] = torch.tensor(0, dtype=torch.int64)

  def blocks(p, n, c):
    for i in range(n):
      b = '%s.%d' % (p, i)
      conv(b + '.conv1', c, c, False)
      bn(b + '.bn1', c)
      conv(b + '.conv2', c, c, False)
      bn(b + '.bn2', c)

  def linear(p, i, o):
    bound = 1.0 / math.sqrt(i)
    sd[p + '.weight'], sd[p + '.bias'] = uniform((o, i), bound), uniform((o,), bound)

  r, q, d = 'representation_head', 'prediction_head', 'dynamics_head'
  conv(r + '.conv1', input_channels, 64, True)
  blocks(r + '.resblocks1', 2, 64)
  conv(r + '.conv2', 64, 128, True)
  blocks(r + '.resblocks2', 3, 128)
  blocks(r + '.resblocks3', 3, 128)
  blocks(r + '.resblocks', 16, 128)
  blocks(q + '.resblocks', 16, 128)
  linear(q + '.fc_value', 4608, 512)
  linear(q + '.fc_value_o', 512, value_bins)
  linear(q + '.fc_policy', 4608, 512)
  linear(q + '.fc_policy_o', 512, action_space)
  conv(d + '.conv', 129, 128, True)
  bn(d + '.bn', 128)
  blocks(d + '.resblocks', 16, 128)
  linear(d + '.fc1', 4608, 512)
  linear(d + '.fc2', 512, reward_bins)
  return sd
