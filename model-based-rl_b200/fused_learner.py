"""Learner.update_weights (learners.py:164-230) for FCNetwork with the network forward and backward on this
library's own kernels instead of torch modules on library GEMMs.

`FusedFCNetwork` keeps every parameter of the reference's FCNetwork (networks.py:122-174) in ONE flat float32 buffer;
its state dict is a set of views with the reference's keys and shapes, so checkpoints, `Learner.send_weights` and the
search kernels' `FCNetwork.load_weights` see the usual tensors.  `FusedLearner(precision=...)` runs a step as

  precision='bf16' (default; csrc/mz_learner_tc.cu: tensor cores, bf16 operands, float32 accumulation, float32 master
  weights / gradients / optimiser state)
    mz_learner_pack           the 20 weight images as bf16 mma B fragments + clears     1 launch
    mz_chain_forward_tc       representation -> LN -> K x (dynamics -> LN)               1 launch
    mz_heads_forward_tc       value / policy / reward heads over all K + 1 steps         1 launch
    mz_unroll_loss            fused loss + logit gradients (csrc/mz_unroll_loss.cu)      2 launches
                              (mz_scalar_unroll_loss for --no_support networks)
    mz_heads_backward_tc      the three output heads                                     1 launch
    mz_chain_backward_tc      the serial part: LN backward -> dH -> dX per step          1 launch
    mz_heads_backward_tc      parameter gradients of dynamics + representation           1 launch
    mz_adam_step              AdamW / Adam over the flat buffer                          2 launches
  -- 10 kernels per step, 128 us at B = 512, K = 5 (7 800 steps/s on a B200; the torch-module step in a
  CUDA graph: 1 100 us).

  precision='f32' (csrc/mz_learner.cu: float32 CUDA-core kernels, one launch per head evaluation; the parity baseline
  against the reference's goldens at float32 bars)
    transposes, 2 (K + 1) forward launches, 3 head launches, loss, 3 + 2 (K + 1) backward launches, optimiser.

Both are captured in CUDA graphs.  SGD / RMSprop use the torch optimiser over the flat buffer (elementwise, the
reference's arithmetic).  Observations of up to 1024 features (MAX_INPUT_DIM) train in both precisions: the
representation head's input goes through the kernels' 128-feature input tiles in slices.  `--no_support` networks
(one-unit value / reward heads, `config.scalar_loss` MSE or Huber, utils.py:61-70) run the same launches with
d_out = 1 heads and the scalar loss kernel.  `save_state` writes the checkpoint dictionary of learners.py:72-83;
`load_state` / `FusedLearner(state=...)` resume from it (weights, optimiser state, training_step, replay throughput), and a
graph captured later keeps the restored optimiser state.  They take a `learners.Learner` checkpoint too: its
per-parameter optimiser state is mapped onto the flat buffer by name (checkpoints.py), and `learners.Learner` resumes
from a FusedLearner checkpoint the same way.  With torch.distributed initialised the gradients of the three output
heads are all-reduced on a side stream while the recurrent part of the backward still runs; the rest follows before the optimiser step.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib, checkpoints, learners, parallel
from .networks import HIDDEN

WIDTH = _lib.FC_WIDTH
MAX_SUPPORT_BINS = 64  # widest value / reward head: LMAXOUT in csrc/mz_learner.cu, head_ok in csrc/mz_learner_tc.cu
MAX_INPUT_DIM = 1024   # widest observation: LMAXD in csrc/mz_learner.cu, MAXIN in csrc/mz_learner_tc.cu
SLICE = 128            # input features per pass of the kernels' X tile: a wider (representation) head has no dX image
_P = lambda t: C.c_void_p(t.data_ptr())


class _Head(object):
  """Views of one head's parameters / gradients / k-major copies inside the flat buffers."""

  def __init__(self, name, out_name, d_in, d_out):
    self.name, self.out_name, self.d_in, self.d_out = name, out_name, d_in, d_out
    self.keys = [k for k, _ in checkpoints.head_params(name, out_name, d_in, d_out)]


class FusedFCNetwork(object):
  """The reference's FCNetwork in train mode (support logits, or one-unit value / reward heads with
  config.no_support) with flat parameter storage.  Heads in buffer order:
  value, policy, reward (the gradient bucket that is complete first), transition, representation, LN."""

  def __init__(self, input_dim, action_space, device, config):
    vmin, vmax = [int(v) for v in config.value_support]
    rmin, rmax = [int(v) for v in config.reward_support]
    no_support = bool(getattr(config, 'no_support', False))  # networks.py:135-136: one-unit scalar heads
    if not 1 <= int(input_dim) <= MAX_INPUT_DIM:  # before the library or the device is touched
      raise ValueError("input_dim %d: the fused learner's kernels take observations of 1 to %d features "
                       "(learners.Learner trains wider ones)" % (int(input_dim), MAX_INPUT_DIM))
    if not no_support:  # before the library or the device is touched: the first step would fail with MZ_ERR_BAD_ARG
      for name, lo, hi in (('value_support', vmin, vmax), ('reward_support', rmin, rmax)):
        if hi < lo or hi - lo + 1 > MAX_SUPPORT_BINS:
          raise ValueError("%s [%d, %d]: the fused learner's head kernels take supports of 1 to %d bins "
                           "(learners.Learner trains wider ones)" % (name, lo, hi, MAX_SUPPORT_BINS))
    self.device = _lib.normalize_device(device)
    self.lib = _lib.load()
    self.input_dim, self.action_space = int(input_dim), int(action_space)
    A = self.action_space
    if HIDDEN + A > SLICE:  # the dynamics / reward heads' input [hidden | one-hot action] needs a dX
      raise ValueError("action_space %d: the fused learner kernels take at most %d actions" % (A, SLICE - HIDDEN))
    self.heads = {h[0]: _Head(*h) for h in checkpoints.fc_heads(self.input_dim, A, config)}
    # every tensor starts on a 16-byte boundary of the flat buffers (the tensor-core backward adds weight gradients
    # with 16-byte vector reductions); the padding floats stay zero in parameters, gradients and optimiser state
    layout, n = checkpoints.flat_layout(self.input_dim, A, config)
    self.flat = torch.zeros(n, dtype=torch.float32, device=self.device)
    self.grad = torch.zeros(n, dtype=torch.float32, device=self.device)
    self.views, self.grads = {}, {}
    for k, s, off in layout:
      m = int(np.prod(s))
      self.views[k] = self.flat[off:off + m].view(s)
      self.grads[k] = self.grad[off:off + m].view(s)
      if k == 'reward_head.reward.bias':
        self.bucket_split = off + checkpoints.pad4(m)  # value, policy and reward heads: the bucket that is complete first
    # k-major copies of the weight matrices (refreshed every step)
    nt = sum(WIDTH * h.d_in + WIDTH * h.d_out for h in self.heads.values())
    self.t_flat = torch.zeros(nt, dtype=torch.float32, device=self.device)
    off = 0
    for h in self.heads.values():
      h.w1t = self.t_flat[off:off + WIDTH * h.d_in].view(h.d_in, WIDTH)
      off += WIDTH * h.d_in
      h.w2t = self.t_flat[off:off + WIDTH * h.d_out].view(WIDTH, h.d_out)
      off += WIDTH * h.d_out
      h.p = [self.views[k] for k in h.keys]
      h.g = [self.grads[k] for k in h.keys]
    # bf16 mma B-operand images of the same matrices for the tensor-core kernels (csrc/mz_learner_tc.cu), refreshed
    # every step from the float32 master weights by ONE launch.  w1tp only feeds dX, which a head wider than SLICE
    # (the representation head, whose input is the observation) never needs: no image for it.
    words = lambda n, k: int(self.lib.mz_learner_packed_words(n, k))
    # (N, K) of w1p w2p w2tp w1tp
    shapes = lambda h: [(WIDTH, h.d_in), (h.d_out, WIDTH), (WIDTH, h.d_out), (h.d_in, WIDTH)][:4 if h.d_in <= SLICE else 3]
    self.packed = torch.zeros(sum(words(n, k) for h in self.heads.values() for n, k in shapes(h)), dtype=torch.int32,
                              device=self.device)
    jobs, off = [], 0
    for h in self.heads.values():
      w1, w2 = h.p[0], h.p[2]
      h.images = []
      for (n, k), (src, sn, sk) in zip(shapes(h), [(w1, h.d_in, 1), (w2, WIDTH, 1), (w2, 1, WIDTH), (w1, 1, h.d_in)]):
        dst = self.packed[off:off + words(n, k)]
        off += words(n, k)
        h.images.append(dst)
        jobs.append(_lib.PackJob(src.data_ptr(), dst.data_ptr(), n, k, sn, sk))
    self._pack_list = jobs
    self._pack_jobs = (_lib.PackJob * len(jobs))(*jobs)
    # the reference's initialisation: torch's defaults for nn.Linear / nn.LayerNorm
    ref = learners.FCNetworkTrain(self.input_dim, A, 'cpu', config)
    self.load_weights(ref.state_dict())

  # -- the reference's network interface ------------------------------------------------------------
  def load_weights(self, weights):
    missing = set(self.views) - set(weights)
    if missing:
      raise KeyError("missing weights: %s" % sorted(missing))
    srcs = {k: torch.as_tensor(weights[k]) for k in self.views}
    for k, v in self.views.items():  # every shape before the first copy: refused weights leave the network as it was
      if tuple(srcs[k].shape) != tuple(v.shape):
        raise ValueError("%s has shape %s, expected %s" % (k, tuple(srcs[k].shape), tuple(v.shape)))
    for k, v in self.views.items():
      v.copy_(srcs[k].to(self.device, torch.float32))

  def load_state_dict(self, weights):
    self.load_weights(weights)

  def state_dict(self):
    return dict(self.views)

  def get_weights(self):
    return {k: v.cpu() for k, v in self.views.items()}

  def parameters(self):
    return [self.flat]

  def train(self, mode=True):
    return self

  def tc_head(self, name):
    """struct mz_tc_head of one head: packed images, float32 biases, gradient views."""
    h = self.heads[name]
    w1tp = h.images[3].data_ptr() if len(h.images) > 3 else None
    return _lib.TcHead(h.images[0].data_ptr(), h.images[1].data_ptr(), h.images[2].data_ptr(), w1tp,
                       h.p[1].data_ptr(), h.p[3].data_ptr(), h.g[0].data_ptr(), h.g[1].data_ptr(), h.g[2].data_ptr(),
                       h.g[3].data_ptr(), h.d_in, h.d_out)

  @_lib.on_device
  def refresh_packed(self):
    _lib.check(self.lib.mz_learner_pack(len(self._pack_jobs), self._pack_jobs, _lib.current_stream()), "mz_learner_pack")

  @_lib.on_device
  def refresh_transposes(self):
    st = _lib.current_stream()
    for h in self.heads.values():
      _lib.check(self.lib.mz_learner_transpose(WIDTH, h.d_in, _P(h.p[0]), _P(h.w1t), st), "mz_learner_transpose")
      _lib.check(self.lib.mz_learner_transpose(h.d_out, WIDTH, _P(h.p[2]), _P(h.w2t), st), "mz_learner_transpose")


class FusedLearner(object):
  """`learners.Learner` with the step on this library's kernels.  Same `update_weights(batch)` on the tuple
  `PrioritizedReplay.sample_batch()` / `sample_batch_device()` returns, priority feedback, weight hand-off,
  schedules, checkpoints (`save_state` / `load_state`, `state=`) and `--no_support` networks (MSE or Huber scalar
  loss, config.scalar_loss)."""

  def __init__(self, config, network, replay_buffer=None, search_network=None, use_graph=True, precision='bf16',
               state=None):
    _lib.require_cuda()
    if not isinstance(network, FusedFCNetwork):
      raise TypeError("FusedLearner trains a FusedFCNetwork")
    if precision not in ('bf16', 'f32'):
      raise ValueError("precision is 'bf16' (tensor cores, float32 accumulation and master weights) or 'f32'")
    self.precision = precision
    self.config, self.network, self.lib = config, network, _lib.load()
    self.device = network.device
    self.replay_buffer, self.search_network = replay_buffer, search_network
    self.use_graph = bool(use_graph)
    self.K, self.A = int(config.num_unroll_steps), network.action_space
    self.loss_cfg = learners.loss_cfg(config)
    self.scalar_loss = None  # support heads: mz_unroll_loss; no_support: 0 = MSE, 1 = Huber (mz_scalar_unroll_loss)
    if getattr(config, 'no_support', False):
      kind = getattr(config, 'scalar_loss', 'MSE')
      if kind not in ('MSE', 'Huber'):
        raise NotImplementedError("scalar_loss %r: the scalar loss kernel computes 'MSE' or 'Huber'" % (kind,))
      self.scalar_loss = int(kind == 'Huber')
    self.training_step = 0
    self.losses_to_log = {'reward': 0., 'value': 0., 'policy': 0.}
    self.last_losses = self.last_errors = None
    self.clip = float(getattr(config, 'clip_grad', 0) or 0)
    name = config.optimizer
    n = network.flat.numel()
    dev = self.device
    self.own_optimizer = name in ('AdamW', 'Adam')
    if self.own_optimizer:
      self.exp_avg = torch.zeros(n, dtype=torch.float32, device=dev)
      self.exp_avg_sq = torch.zeros(n, dtype=torch.float32, device=dev)
      self.opt_state = torch.tensor([0.0, float(config.lr_init), 0.0], dtype=torch.float32, device=dev)
      self.optimizer = _LrHandle(self.opt_state, float(config.lr_init))
    else:  # SGD / RMSprop: elementwise, so the torch optimiser over the flat buffer does the reference's arithmetic
      network.flat.grad = network.grad
      scheduled = getattr(config, 'lr_scheduler', None) is not None
      cap = self.use_graph and name != 'SGD'
      lr = torch.tensor(float(config.lr_init), device=dev) if (cap and scheduled) else None
      self.optimizer = learners.get_optimizer(config, [network.flat], capturable=cap, lr=lr)
      self._graph_opt = self.use_graph and not (name == 'SGD' and scheduled)
    if self.own_optimizer and getattr(config, 'lr_scheduler', None) == 'ExponentialLR':
      self.lr_scheduler = _ExponentialLR(self.optimizer, float(config.lr_init), float(config.lr_decay_rate))
    else:
      self.lr_scheduler = learners.get_lr_scheduler(config, self.optimizer)
    if getattr(config, 'norm_obs', False):
      lo = torch.tensor(config.obs_range[::2], dtype=torch.float32, device=dev)
      hi = torch.tensor(config.obs_range[1::2], dtype=torch.float32, device=dev)
      self.obs_min, self.obs_range = lo, hi - lo
    self._shape = None
    self._graphs = None
    self._comm = None
    if state is not None:
      self.load_state(state)

  # -- buffers of one batch shape ----------------------------------------------------------------------
  def _alloc(self, B):
    K, A, dev, net = self.K, self.A, self.device, self.network
    f = lambda *s: torch.zeros(s, dtype=torch.float32, device=dev)
    V, R = net.heads['value_head'].d_out, net.heads['reward_head'].d_out
    self.B, self.ldx = B, HIDDEN + A
    self.s_obs = f(B, net.input_dim)
    self.s_actions = torch.zeros((B, max(K, 1)), dtype=torch.int32, device=dev)
    self.s_tv, self.s_tr, self.s_tp = f(B, K + 1), f(B, K + 1), f(B, K + 1, A)
    self.s_isw = torch.ones(B, dtype=torch.float64, device=dev)
    self.xs = f((K + 1) * B, self.ldx)       # [h_k | one-hot(a_k)] rows of every unroll step
    self.dxs = f((K + 1) * B, self.ldx)
    self.yall = f(K + 1, B, HIDDEN)          # pre-LayerNorm outputs of the representation / dynamics heads
    self.mean, self.rstd = f(K + 1, B), f(K + 1, B)
    self.dy = f(B, HIDDEN)
    self.v, self.r, self.p = f(K + 1, B, V), f(max(K, 1), B, R), f(K + 1, B, A)
    self.dv, self.dr, self.dp = torch.empty_like(self.v), torch.empty_like(self.r), torch.empty_like(self.p)
    self.rows = torch.zeros((3, B), dtype=torch.float64, device=dev)
    self.losses = torch.zeros(3, dtype=torch.float64, device=dev)
    self.new_errors = f(B)
    self.c_loss = _lib.LossCfg(B, K, A, self.loss_cfg['value_min'], self.loss_cfg['value_max'], self.loss_cfg['reward_min'],
                               self.loss_cfg['reward_max'], int(self.loss_cfg['no_target_transform']))
    self._shape, self._graphs = B, None
    if self.precision == 'bf16':
      self._alloc_tc()

  def _alloc_tc(self):
    """Argument structs of the four tensor-core launches (pointers into the buffers of this batch shape)."""
    net, K, B, A, ldx = self.network, self.K, self.B, self.A, self.ldx
    P = lambda t: t.data_ptr()
    self.relu_mask = torch.zeros(int(self.lib.mz_chain_mask_words(B, K + 1)), dtype=torch.int32, device=self.device)
    self.dyall = torch.zeros((K + 1, B, HIDDEN), dtype=torch.float32, device=self.device)
    self.tc_chain = _lib.TcChain(net.tc_head('representation_head'), net.tc_head('transition_head'), B, K + 1, HIDDEN, A,
                                 P(self.s_obs), net.input_dim, P(self.s_actions), max(K, 1), K, P(net.views['LN.weight']),
                                 P(net.views['LN.bias']), P(self.xs), ldx, P(self.yall), P(self.mean), P(self.rstd),
                                 P(self.relu_mask), P(self.dxs), 0.5, P(net.grads['LN.weight']), P(net.grads['LN.bias']),
                                 P(self.dyall))
    # parameter gradients of the recurrent heads, off the chain: all K B + B rows in one launch
    rec = [_lib.TcJob(net.tc_head('representation_head'), B, net.input_dim, HIDDEN, 0, P(self.s_obs), None, P(self.dyall[0]),
                      None)]
    if K > 0:
      rec.append(_lib.TcJob(net.tc_head('transition_head'), K * B, ldx, HIDDEN, 0, P(self.xs), None, P(self.dyall[1]), None))
    self.tc_rec_jobs = (_lib.TcJob * len(rec))(*rec)
    # the step's first launch packs the weight images AND clears the two accumulation buffers (src NULL = zero n words)
    first = list(net._pack_list) + [_lib.PackJob(None, P(net.grad), net.grad.numel(), 0, 0, 0),
                                    _lib.PackJob(None, P(self.dxs), self.dxs.numel(), 0, 0, 0)]
    self.tc_first_jobs = (_lib.PackJob * len(first))(*first)
    V, R = self.v.shape[2], self.r.shape[2]
    jobs = [_lib.TcJob(net.tc_head('value_head'), (K + 1) * B, ldx, V, ldx, P(self.xs), P(self.v), P(self.dv), P(self.dxs)),
            _lib.TcJob(net.tc_head('policy_head'), (K + 1) * B, ldx, A, ldx, P(self.xs), P(self.p), P(self.dp), P(self.dxs))]
    if K > 0:
      jobs.append(_lib.TcJob(net.tc_head('reward_head'), K * B, ldx, R, ldx, P(self.xs), P(self.r), P(self.dr), P(self.dxs)))
    self.tc_jobs = (_lib.TcJob * len(jobs))(*jobs)

  # -- launch sequences --------------------------------------------------------------------------------
  def _fwd(self, head, rows, x, ldx, y, ldy, st):
    h = self.network.heads[head]
    _lib.check(self.lib.mz_mlp2_forward(rows, h.d_in, ldx, _P(x), _P(h.w1t), _P(h.p[1]), _P(h.w2t), _P(h.p[3]), h.d_out,
                                        _P(y), ldy, st), "mz_mlp2_forward")

  def _bwd(self, head, rows, x, ldx, dy, ldy, dx, lddx, st):
    h = self.network.heads[head]
    _lib.check(self.lib.mz_mlp2_backward(rows, h.d_in, ldx, _P(x), _P(h.w1t), _P(h.p[1]), _P(h.p[0]), _P(h.p[2]), h.d_out,
                                         _P(dy), ldy, None if dx is None else _P(dx), lddx, _P(h.g[0]), _P(h.g[1]),
                                         _P(h.g[2]), _P(h.g[3]), st), "mz_mlp2_backward")

  def _loss(self, st):
    """The loss and the gradient of every head output: support logits (mz_unroll_loss) or the scalar heads of a
    no_support network (mz_scalar_unroll_loss)."""
    args = (_P(self.v), _P(self.r), _P(self.p), _P(self.s_tv), _P(self.s_tr), _P(self.s_tp), _P(self.s_isw), _P(self.dv),
            _P(self.dr), _P(self.dp), _P(self.rows), _P(self.losses), _P(self.new_errors), st)
    if self.scalar_loss is None:
      _lib.check(self.lib.mz_unroll_loss(self.c_loss, *args), "mz_unroll_loss")
    else:
      _lib.check(self.lib.mz_scalar_unroll_loss(self.c_loss, self.scalar_loss, *args), "mz_scalar_unroll_loss")

  def _forward_and_heads_backward(self):
    """Transposes, the K + 1 network evaluations (learners.py:175-206), the loss, and the backward of the three
    output heads (whose parameter gradients are then complete)."""
    net, lib, K, B, A, ldx = self.network, self.lib, self.K, self.B, self.A, self.ldx
    st = _lib.current_stream()
    if self.precision == 'bf16':
      _lib.check(lib.mz_learner_pack(len(self.tc_first_jobs), self.tc_first_jobs, st), "mz_learner_pack")
      _lib.check(lib.mz_chain_forward_tc(self.tc_chain, st), "mz_chain_forward_tc")
      _lib.check(lib.mz_heads_forward_tc(len(self.tc_jobs), self.tc_jobs, st), "mz_heads_forward_tc")
      self._loss(st)
      _lib.check(lib.mz_heads_backward_tc(len(self.tc_jobs), self.tc_jobs, st), "mz_heads_backward_tc")
      return
    ln_w, ln_b = net.views['LN.weight'], net.views['LN.bias']
    net.refresh_transposes()
    net.grad.zero_()
    self.dxs.zero_()
    xs = self.xs.view(K + 1, B, ldx)
    self._fwd('representation_head', B, self.s_obs, net.input_dim, self.yall[0], HIDDEN, st)
    for k in range(K + 1):
      if k > 0:
        self._fwd('transition_head', B, xs[k - 1], ldx, self.yall[k], HIDDEN, st)
      acts = C.c_void_p(self.s_actions.data_ptr() + 4 * k) if k < K else None
      _lib.check(lib.mz_ln_relu_forward(B, HIDDEN, _P(self.yall[k]), _P(ln_w), _P(ln_b), acts, max(K, 1), A, _P(xs[k]), ldx,
                                        _P(self.mean[k]), _P(self.rstd[k]), st), "mz_ln_relu_forward")
    self._fwd('value_head', (K + 1) * B, self.xs, ldx, self.v, self.v.shape[2], st)
    self._fwd('policy_head', (K + 1) * B, self.xs, ldx, self.p, A, st)
    if K > 0:
      self._fwd('reward_head', K * B, self.xs, ldx, self.r, self.r.shape[2], st)
    self._loss(st)
    self._bwd('value_head', (K + 1) * B, self.xs, ldx, self.dv, self.v.shape[2], self.dxs, ldx, st)
    self._bwd('policy_head', (K + 1) * B, self.xs, ldx, self.dp, A, self.dxs, ldx, st)
    if K > 0:
      self._bwd('reward_head', K * B, self.xs, ldx, self.dr, self.r.shape[2], self.dxs, ldx, st)

  def _recurrent_backward(self):
    """Back through the dynamics chain and the representation; the 0.5 hook of learners.py:201 scales the gradient
    of every hidden state the dynamics produced."""
    net, lib, K, B, ldx = self.network, self.lib, self.K, self.B, self.ldx
    st = _lib.current_stream()
    if self.precision == 'bf16':
      _lib.check(lib.mz_chain_backward_tc(self.tc_chain, st), "mz_chain_backward_tc")
      _lib.check(lib.mz_heads_backward_tc(len(self.tc_rec_jobs), self.tc_rec_jobs, st), "mz_heads_backward_tc")
      return
    ln_w = net.views['LN.weight']
    g_w, g_b = net.grads['LN.weight'], net.grads['LN.bias']
    xs, dxs = self.xs.view(K + 1, B, ldx), self.dxs.view(K + 1, B, ldx)
    for k in range(K, -1, -1):
      _lib.check(lib.mz_ln_relu_backward(B, HIDDEN, _P(dxs[k]), ldx, 0.5 if k > 0 else 1.0, _P(self.yall[k]), _P(xs[k]), ldx,
                                         _P(self.mean[k]), _P(self.rstd[k]), _P(ln_w), _P(self.dy), _P(g_w), _P(g_b), st),
                 "mz_ln_relu_backward")
      if k > 0:
        self._bwd('transition_head', B, xs[k - 1], ldx, self.dy, HIDDEN, dxs[k - 1], ldx, st)
      else:
        self._bwd('representation_head', B, self.s_obs, net.input_dim, self.dy, HIDDEN, None, 0, st)

  def _apply(self, world):
    if self.own_optimizer:
      cfg = self.config
      eps = 0.00015  # utils.py:78-80
      _lib.check(self.lib.mz_adam_step(self.network.flat.numel(), _P(self.network.flat), _P(self.network.grad),
                                       _P(self.exp_avg), _P(self.exp_avg_sq), _P(self.opt_state), 0.9, 0.999, eps,
                                       float(cfg.weight_decay), int(cfg.optimizer == 'AdamW'), 1.0 / world, self.clip,
                                       _lib.current_stream()), "mz_adam_step")
      return
    if world > 1:
      self.network.grad.div_(world)
    if self.clip:
      torch.nn.utils.clip_grad_norm_([self.network.flat], self.clip)
    self.optimizer.step()

  # -- one step (learners.py:164-230) --------------------------------------------------------------------
  def _stage(self, batch):
    batch, idxs, is_weights = batch
    if len(batch) == 3:   # sample_batch(): (observations, actions, (target_rewards, target_values, target_policies))
      observations, actions, (t_rewards, t_values, t_policies) = batch
    else:                 # sample_batch_device(): the same five arrays, flat (+ the fused supports, unused here)
      observations, actions, t_rewards, t_values, t_policies = batch[:5]
    dev = self.device
    to = lambda x, dt: (x if torch.is_tensor(x) else torch.as_tensor(np.asarray(x))).to(dev, dt, non_blocking=True)
    obs = to(observations, torch.float32)
    B = int(obs.shape[0])
    if self._shape != B:
      self._alloc(B)
    obs = obs.reshape(B, -1)
    if getattr(self.config, 'norm_obs', False):
      obs = (obs - self.obs_min) / self.obs_range
    self.s_obs.copy_(obs)
    if self.K:
      self.s_actions.copy_(to(actions, torch.int32).reshape(B, self.K))
    self.s_tv.copy_(to(t_values, torch.float32))
    self.s_tr.copy_(to(t_rewards, torch.float32))
    self.s_tp.copy_(to(t_policies, torch.float32))
    if is_weights is None:
      self.s_isw.fill_(1.0)
    else:
      self.s_isw.copy_(to(is_weights, torch.float64))
    return idxs

  @_lib.on_device
  def update_weights(self, batch):
    idxs = self._stage(batch)
    _, world = parallel.world()
    if not self.use_graph:
      self._forward_and_heads_backward()
      self._reduce_and_finish(world, self._recurrent_backward, lambda: self._apply(world))
    else:
      if self._graphs is None:
        self._capture(world)
      g1, g2, g3 = self._graphs
      g1.replay()
      self._reduce_and_finish(world, g2.replay, (g3.replay if g3 is not None else (lambda: self._apply(world))))
    if self.replay_buffer is not None:  # learners.py:182-184
      if torch.is_tensor(idxs) and idxs.is_cuda:
        self.replay_buffer.update(idxs, self.new_errors)
      else:
        self.replay_buffer.update(idxs, self.new_errors.cpu().numpy())
    if self.lr_scheduler is not None:
      self.lr_scheduler.step()
    self.last_losses, self.last_errors = self.losses, self.new_errors
    return self.last_losses

  def _reduce_and_finish(self, world, recurrent_backward, apply):
    """Gradient all-reduce in two buckets: the output heads' gradients travel on a side stream while the recurrent
    backward still runs."""
    if world == 1:
      recurrent_backward()
      apply()
      return
    import torch.distributed as dist
    net = self.network
    main = torch.cuda.current_stream()
    if self._comm is None:
      self._comm = torch.cuda.Stream(device=self.device)
    self._comm.wait_stream(main)
    with torch.cuda.stream(self._comm):
      dist.all_reduce(net.grad[:net.bucket_split])
    recurrent_backward()
    dist.all_reduce(net.grad[net.bucket_split:])
    main.wait_stream(self._comm)
    apply()

  def _optimizer_tensors(self):
    if self.own_optimizer:
      return [self.exp_avg, self.exp_avg_sq, self.opt_state]
    return [v for st in self.optimizer.state.values() for v in st.values() if torch.is_tensor(v)]

  def _capture(self, world):
    # the optimiser state as it stands (fresh, or restored by load_state): the warm-up step below changes it
    saved = {id(t): t.clone() for t in self._optimizer_tensors()}
    # warm-up outside capture: kernel attributes, lazy module loading, optimiser state
    self._forward_and_heads_backward()
    self._recurrent_backward()
    torch.cuda.synchronize()
    snapshot = self.network.flat.clone()
    g1 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g1):
      self._forward_and_heads_backward()
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2, pool=g1.pool()):
      self._recurrent_backward()
    g3 = None
    if self.own_optimizer or self._graph_opt:
      if not self.own_optimizer:
        # the torch optimiser initialises its state on the first step: take one with zero gradients (restored below)
        self.network.grad.zero_()
        self.optimizer.step()
      g3 = torch.cuda.CUDAGraph()
      with torch.cuda.graph(g3, pool=g1.pool()):
        self._apply(world)
    # in place, so that the captured step reads it: the state from before, zeros for state the warm-up step created
    for t in self._optimizer_tensors():
      if id(t) in saved:
        t.copy_(saved[id(t)])
      else:
        t.zero_()
    self.network.flat.copy_(snapshot)
    torch.cuda.synchronize()
    self._graphs = (g1, g2, g3)

  # -- the rest of the reference's learner --------------------------------------------------------------
  def send_weights(self):
    """learners.py:84-85 / actors.py:81-85."""
    weights = {k: v.detach() for k, v in self.network.views.items()}
    parallel.broadcast_weights(weights, src=0)
    if self.search_network is not None:
      self.search_network.load_weights(weights)
    return weights

  def log_losses(self):
    r, v, p = self.last_losses.cpu().tolist()
    self.losses_to_log['reward'] += r
    self.losses_to_log['value'] += v
    self.losses_to_log['policy'] += p
    return r, v, p

  def learn(self, training_steps=None):
    """The loop of learners.py:116-148 for `training_steps` steps (default config.training_steps)."""
    steps = self.config.training_steps if training_steps is None else training_steps
    self.send_weights()
    need = int(getattr(self.config, 'stored_before_train', 0) or 0)
    if self.replay_buffer.size() < need:
      raise RuntimeError("replay buffer holds %d memories, config.stored_before_train is %d" %
                         (self.replay_buffer.size(), need))
    save_every = int(getattr(self.config, 'save_state_frequency', 0) or 0)
    end = self.training_step + steps
    while self.training_step < end:
      self.update_weights(self.replay_buffer.sample_batch_device(False, ring=4))
      self.training_step += 1
      if self.training_step % self.config.send_weights_frequency == 0:
        self.send_weights()
      if save_every and self.training_step % save_every == 0:  # learners.py:135-136
        saves = (getattr(self, 'dirs', None) or {}).get('saves')
        self.save_state(os.path.join(saves, str(self.training_step)) if saves else None)
    return self.training_step

  def save_state(self, path=None, actor_games=None, dirs=None):
    """The checkpoint dictionary of learners.py:72-83 (see learners.Learner.save_state); the optimiser entry is
    {'exp_avg', 'exp_avg_sq', 'state' = (step, learning rate, scratch)} for the library's Adam / AdamW, else the torch
    optimiser's state_dict.  `dirs` / `actor_games` default to the attributes of the same names."""
    tp = self.replay_buffer.get_throughput() if self.replay_buffer is not None else {'frames': 0, 'games': 0}
    if self.own_optimizer:
      opt = {'exp_avg': self.exp_avg.cpu(), 'exp_avg_sq': self.exp_avg_sq.cpu(), 'state': self.opt_state.cpu()}
    else:
      opt = self.optimizer.state_dict()
    state = {'dirs': dict(dirs if dirs is not None else getattr(self, 'dirs', {}) or {}),
             'config': self.config, 'weights': self.network.get_weights(), 'optimizer': opt,
             'training_step': self.training_step, 'total_games': tp['games'], 'total_frames': tp['frames'],
             'actor_games': dict(actor_games if actor_games is not None else getattr(self, 'actor_games', {}) or {})}
    if path is not None:
      torch.save(state, path)
    self.last_saved_state = state
    return state

  def load_state(self, state):
    """Resumes from a `save_state` checkpoint of a FusedLearner or of a `learners.Learner` with the same optimiser and
    network (learners.py:59-70, learners.Learner.load_state): weights, optimiser state, training_step and the replay
    throughput.  A learners.Learner checkpoint's per-parameter optimiser state is mapped onto the flat buffer first
    (checkpoints.module_to_flat).  Every check runs before anything is written: a refused checkpoint raises ValueError
    and leaves the learner as it was.  The library's Adam state is copied in place (captured graphs stay valid); a
    torch optimiser's load_state_dict replaces its tensors, so the step is captured again."""
    opt, n, net = state['optimizer'], self.network.flat.numel(), self.network
    module_form = checkpoints.is_module_form(opt, net.input_dim, net.action_space, self.config)
    saved_kind = getattr(state.get('config'), 'optimizer', self.config.optimizer)
    if saved_kind != self.config.optimizer:
      raise ValueError("the checkpoint of a %s holds %s optimiser state, this learner runs %s" % (
          'learners.Learner' if module_form else 'FusedLearner', saved_kind, self.config.optimizer))
    if module_form:
      opt = checkpoints.module_to_flat(opt, self.config, net.input_dim, net.action_space)
    own = isinstance(opt, dict) and 'exp_avg' in opt
    if own != self.own_optimizer:
      raise ValueError("the checkpoint holds %s optimiser state, this learner runs %s" % (
          'the library Adam kernel\'s' if own else 'torch optimiser', self.config.optimizer))
    if own:
      sizes = {opt['exp_avg'].numel(), opt['exp_avg_sq'].numel()}
    else:
      sizes = {v.numel() for st in opt['state'].values() for v in st.values() if torch.is_tensor(v) and v.dim() > 0}
    if sizes - {n}:
      raise ValueError("the checkpoint's optimiser state has %s elements per tensor, the flat buffer %d" % (sorted(sizes), n))
    self.network.load_weights(state['weights'])
    if own:
      self.exp_avg.copy_(opt['exp_avg'])
      self.exp_avg_sq.copy_(opt['exp_avg_sq'])
      self.opt_state.copy_(opt['state'])
      if isinstance(self.lr_scheduler, _ExponentialLR):  # the decay continues from the restored rate
        self.lr_scheduler.lr = float(self.opt_state[1])
    else:
      learners.load_optimizer_state(self.optimizer, opt, self.device)
      self._graphs = None
    self.training_step = state['training_step']
    if self.replay_buffer is not None and 'total_frames' in state:
      self.replay_buffer.add_initial_throughput(state['total_frames'], state['total_games'])


class _LrHandle(object):
  """What the schedules of learners.py need from an optimiser (`param_groups[..]['lr']`), backed by the device scalar
  the Adam kernel reads."""

  def __init__(self, opt_state, lr):
    self.param_groups = [{'lr': opt_state[1:2]}]
    self.param_groups[0]['lr'].fill_(lr)


class _ExponentialLR(object):
  """torch.optim.lr_scheduler.ExponentialLR (utils.py:122-123) for the device-side learning rate."""

  def __init__(self, handle, lr, gamma):
    self.handle, self.lr, self.gamma = handle, lr, gamma

  def step(self):
    self.lr *= self.gamma
    learners._set_lr(self.handle, self.lr)
