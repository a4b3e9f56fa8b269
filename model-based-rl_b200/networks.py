"""Inference side of the reference's FCNetwork (networks.py:55-174) on hand-written kernels.

`FCNetwork` here keeps the reference's interface -- initial_inference / recurrent_inference
returning NetworkOutput(value, reward, policy_logits, hidden_state), load_weights / get_weights with
the reference's state-dict keys -- but evaluates the whole network in one fused CUDA kernel per
call (eval mode: value / reward are scalars after softmax-expectation + h^-1, config.py:27-33).
Training (backward, train-mode support logits) stays with the reference's torch module; weights
move between the two through the state dict.
"""
import ctypes as C
import os
from collections import OrderedDict, namedtuple

import numpy as np
import torch

from . import _lib

NetworkOutput = namedtuple('network_output', ('value', 'reward', 'policy_logits', 'hidden_state'))

HIDDEN = _lib.FC_HIDDEN

# reference state-dict keys (networks.py:137-144) -> (struct field, transposed?)
_KEYS = OrderedDict([
    ('representation_head.fc1.weight', ('rep_w1', True)), ('representation_head.fc1.bias', ('rep_b1', False)),
    ('representation_head.out.weight', ('rep_w2', False)), ('representation_head.out.bias', ('rep_b2', False)),
    ('value_head.fc1.weight', ('val_w1', True)), ('value_head.fc1.bias', ('val_b1', False)),
    ('value_head.value.weight', ('val_w2', False)), ('value_head.value.bias', ('val_b2', False)),
    ('policy_head.fc1.weight', ('pol_w1', True)), ('policy_head.fc1.bias', ('pol_b1', False)),
    ('policy_head.policy.weight', ('pol_w2', False)), ('policy_head.policy.bias', ('pol_b2', False)),
    ('reward_head.fc1.weight', ('rew_w1', True)), ('reward_head.fc1.bias', ('rew_b1', False)),
    ('reward_head.reward.weight', ('rew_w2', False)), ('reward_head.reward.bias', ('rew_b2', False)),
    ('transition_head.fc1.weight', ('dyn_w1', True)), ('transition_head.fc1.bias', ('dyn_b1', False)),
    ('transition_head.out.weight', ('dyn_w2', False)), ('transition_head.out.bias', ('dyn_b2', False)),
    ('LN.weight', ('ln_w', False)), ('LN.bias', ('ln_b', False)),
])


class FCNetwork(object):
  """Fused-kernel FCNetwork (inference).  `config` supplies value_support / reward_support /
  no_support / no_target_transform exactly like the reference's Config (config.py:9-19)."""

  accepts_device_actions = True
  training = False

  def __init__(self, input_dim, action_space, device, config, precision='bf16'):
    """precision: 'bf16' = tcgen05 tensor-core kernel for recurrent_inference (bf16 operands, fp32
    accumulation; A <= 64 and supports of at most 64 bins); 'f32' = CUDA-core float32 kernel (reference precision, used for parity); 'tf32x3' =
    reference precision on the tensor cores (three TF32 instructions per product on split operands,
    float32 accumulation: the results of 'f32' within float32 rounding)."""
    _lib.require_cuda()
    if precision not in ('bf16', 'f32', 'tf32x3'):
      raise ValueError("precision must be 'bf16', 'f32' or 'tf32x3'")
    # --no_support (config.py:95; networks.py:135-136, 153, 161): one-unit value / reward heads, their raw outputs
    # are the scalars.  The float32-accurate kernels evaluate it; the bf16 kernels (and with them the persistent
    # search kernel) are built around the support heads, so the default precision becomes 'tf32x3' here.
    self.no_support = bool(getattr(config, 'no_support', False))
    if self.no_support and precision == 'bf16':
      precision = 'tf32x3'
    self.precision = precision
    self.lib = _lib.load()
    self.device = _lib.normalize_device(device)
    self.input_dim = int(input_dim)
    self.action_space = int(action_space)
    self.value_min, self.value_max = [int(v) for v in config.value_support]
    self.reward_min, self.reward_max = [int(v) for v in config.reward_support]
    self.value_bins = 1 if self.no_support else self.value_max - self.value_min + 1
    self.reward_bins = 1 if self.no_support else self.reward_max - self.reward_min + 1
    self.no_target_transform = bool(getattr(config, 'no_target_transform', False))
    self._state = None    # reference-layout float32 tensors (device)
    self._packed = None   # kernel-layout tensors, kept alive for the struct
    self.weights = None   # _lib.FcWeights

  # -- weights -----------------------------------------------------------------------------------
  @_lib.on_device
  def load_weights(self, weights):
    """Accepts the reference's state dict (networks.py:176-177).

    The network holds a SNAPSHOT (the reference copies through `.cpu()` state dicts, networks.py:36-40):
    every tensor is copied into storage allocated on the first call, so the device pointers inside
    `self.weights`, the packed tensor-core images and anything that captured them (the search engines'
    launch plans and CUDA graphs) stay valid across weight hand-offs (Learner.send_weights)."""
    missing = [k for k in _KEYS if k not in weights]
    if missing:
      raise KeyError("state dict is missing %s" % missing)
    new = {k: torch.as_tensor(weights[k]).detach().to(self.device, torch.float32) for k in _KEYS}
    shapes = {
        'representation_head.fc1.weight': (512, self.input_dim),
        'transition_head.fc1.weight': (512, HIDDEN + self.action_space),
        'reward_head.fc1.weight': (512, HIDDEN + self.action_space),
        'value_head.fc1.weight': (512, HIDDEN), 'policy_head.fc1.weight': (512, HIDDEN),
        'representation_head.out.weight': (HIDDEN, 512), 'transition_head.out.weight': (HIDDEN, 512),
        'reward_head.reward.weight': (self.reward_bins, 512),
        'value_head.value.weight': (self.value_bins, 512),
        'policy_head.policy.weight': (self.action_space, 512), 'LN.weight': (HIDDEN,)}
    for k, shp in shapes.items():
      if tuple(new[k].shape) != shp:
        raise ValueError("%s has shape %s, expected %s" % (k, tuple(new[k].shape), shp))
    if self._state is None:
      self._state = {k: v.clone().contiguous() for k, v in new.items()}
      self._packed = {}
      fields = {}
      for k, (name, transposed) in _KEYS.items():
        t = self._state[k].t().contiguous() if transposed else self._state[k]
        self._packed[name] = t
        fields[name] = t.data_ptr()
      self.weights = _lib.FcWeights(self.input_dim, self.action_space, self.value_bins,
                                    self.reward_bins, self.value_min, self.reward_min,
                                    int(self.no_target_transform), int(self.no_support),
                                    *[fields[n] for n in _lib.FcWeights._names])
      self._tc_packed = self._tc_tail = None
      self._tc_init_packed = self._tc_init_tail = None
      if self.precision == 'bf16':
        if self.action_space > 64 or self.value_bins > 64 or self.reward_bins > 64:
          raise NotImplementedError("the tensor-core kernel supports A <= 64 and supports <= 64 bins; "
                                    "use precision='f32'")
        rec, init, tail = C.c_int64(), C.c_int64(), C.c_int32()
        _lib.check(self.lib.mz_fc_tc_sizes(self.weights, C.byref(rec), C.byref(init), C.byref(tail)),
                   "mz_fc_tc_sizes")
        self._tc_packed = torch.zeros(rec.value, dtype=torch.uint8, device=self.device)
        self._tc_tail = torch.zeros(tail.value, dtype=torch.float32, device=self.device)
        # initial_inference image (representation + prediction heads); observations too wide for
        # the kernel's shared-memory budget stay on the float32 kernel
        nbytes = init.value
        if nbytes > 0:
          self._tc_init_packed = torch.zeros(nbytes, dtype=torch.uint8, device=self.device)
          self._tc_init_tail = torch.zeros_like(self._tc_tail)
    else:
      for k, (name, transposed) in _KEYS.items():
        self._state[k].copy_(new[k])
        if transposed:
          self._packed[name].copy_(self._state[k].t())
    self.weights_version = getattr(self, 'weights_version', 0) + 1
    if self.precision == 'bf16':
      with torch.cuda.device(self.device):
        _lib.check(self.lib.mz_fc_tc_pack(self.weights, _lib.ptr(self._tc_packed),
                                          _lib.ptr(self._tc_tail), _lib.current_stream()),
                   "mz_fc_tc_pack")
        if self._tc_init_packed is not None:
          _lib.check(self.lib.mz_fc_tc_pack_initial(self.weights, _lib.ptr(self._tc_init_packed),
                                                    _lib.ptr(self._tc_init_tail), _lib.current_stream()),
                     "mz_fc_tc_pack_initial")

  load_state_dict = load_weights

  def get_weights(self):
    return {k: v.cpu() for k, v in self._state.items()}

  def state_dict(self):
    return dict(self._state)

  def to(self, device):
    if torch.device(device).type != 'cuda':
      raise RuntimeError("the B200 FCNetwork only runs on CUDA devices")
    return self

  def eval(self):
    return self

  # -- inference ---------------------------------------------------------------------------------
  @_lib.on_device
  def initial_inference(self, observation, hidden_out=None, hidden_stride=None):
    """BaseNetwork.initial_inference (networks.py:26-29).  observation [B, input_dim] float32."""
    obs = observation.to(self.device, torch.float32).reshape(observation.shape[0], -1).contiguous()
    B = obs.shape[0]
    if hidden_out is None:
      hidden_out = torch.empty((B, HIDDEN), dtype=torch.float32, device=self.device)
      hidden_stride = HIDDEN
    value = torch.empty((B, 1), dtype=torch.float32, device=self.device)
    logits = torch.empty((B, self.action_space), dtype=torch.float32, device=self.device)
    fn, args = self.initial_call(B, obs, hidden_out, hidden_stride, value, logits, _lib.current_stream())
    _lib.check(fn(*args), fn.__name__)
    return NetworkOutput(value, 0, logits, hidden_out)

  def initial_call(self, B, obs, hidden_out, hidden_stride, value, logits, stream):
    """(C function, arguments) of initial_inference: the tensor-core kernel when the network runs
    in bf16 and the observation fits it, else the float32 CUDA-core kernel."""
    P = _lib.ptr
    if self.precision == 'bf16' and getattr(self, '_tc_init_packed', None) is not None:
      return self.lib.mz_fc_initial_tc, (self.weights, P(self._tc_init_packed), P(self._tc_init_tail), B,
                                         P(obs), P(hidden_out), int(hidden_stride), P(value), P(logits),
                                         stream)
    fn = self.lib.mz_fc_initial_tf32x3 if self.precision == 'tf32x3' and self.input_dim <= 448 \
        else self.lib.mz_fc_initial_f32
    return fn, (self.weights, B, P(obs), P(hidden_out), int(hidden_stride), P(value), P(logits), stream)

  @_lib.on_device
  def recurrent_inference(self, hidden_state, action):
    """BaseNetwork.recurrent_inference (networks.py:31-34).  `action`: B ints (list or tensor)."""
    h = hidden_state.to(self.device, torch.float32).contiguous()
    B = h.shape[0]
    a = torch.as_tensor(action, device=self.device).to(torch.int32).reshape(B).contiguous()
    out = self._buffers(B)
    self.recurrent_into(h, HIDDEN, None, a, out[3], HIDDEN, 0, out[0], out[1], out[2])
    return NetworkOutput(out[0], out[1], out[2], out[3])

  def recurrent_into(self, hidden_in, in_row_stride, in_index, actions, hidden_out, out_row_stride,
                     out_offset, value, reward, logits):
    """Raw form used by the search engine: gathers from / scatters into the tree's hidden pool."""
    B = actions.shape[0]
    if self.precision == 'bf16':
      _lib.check(self.lib.mz_fc_recurrent_tc(
          self.weights, _lib.ptr(self._tc_packed), _lib.ptr(self._tc_tail), B, _lib.ptr(hidden_in),
          int(in_row_stride), _lib.ptr(in_index), _lib.ptr(actions), _lib.ptr(hidden_out),
          int(out_row_stride), int(out_offset), _lib.ptr(value), _lib.ptr(reward), _lib.ptr(logits),
          _lib.current_stream()), "mz_fc_recurrent_tc")
      return
    fn = self.recurrent_f32_fn()
    _lib.check(fn(self.weights, B, _lib.ptr(hidden_in), int(in_row_stride), _lib.ptr(in_index),
                  _lib.ptr(actions), _lib.ptr(hidden_out), int(out_row_stride), int(out_offset),
                  _lib.ptr(value), _lib.ptr(reward), _lib.ptr(logits), _lib.current_stream()), fn.__name__)

  def recurrent_f32_fn(self):
    """The float32-accurate recurrent_inference entry point: CUDA cores ('f32') or tensor cores ('tf32x3')."""
    return self.lib.mz_fc_recurrent_tf32x3 if self.precision == 'tf32x3' else self.lib.mz_fc_recurrent_f32

  def _buffers(self, B):
    dev = self.device
    return (torch.empty((B, 1), dtype=torch.float32, device=dev),
            torch.empty((B, 1), dtype=torch.float32, device=dev),
            torch.empty((B, self.action_space), dtype=torch.float32, device=dev),
            torch.empty((B, HIDDEN), dtype=torch.float32, device=dev))


class _Lane(object):
  """One slice of the games with its own tree engine, network output buffers and CUDA stream."""

  def __init__(self, config, fcnet, lo, hi, parent, stream):
    from .mcts import BatchedMCTS
    self.lo, self.hi, self.stream = lo, hi, stream
    self.net = fcnet
    self.eng = BatchedMCTS(config, hi - lo, hidden_words=HIDDEN, device=fcnet.device)
    G, A, dev = hi - lo, self.eng.A, fcnet.device
    # inputs / outputs are views into the parent's whole-batch staging tensors
    for name in ('obs', 'noise', 'legal', 'to_play', 'temperature', 'uniforms', 'root_logits',
                 'init_value'):
      setattr(self, name, getattr(parent, name)[lo:hi])
    self.eng.visits = parent.visits[lo:hi]
    self.eng.child_visits = parent.child_visits[lo:hi]
    self.eng.root_value = parent.root_value[lo:hi]
    self.eng.minmax = parent.minmax[lo:hi]
    self.eng.actions = parent.actions[lo:hi]
    self.value = torch.zeros(G, dtype=torch.float32, device=dev)
    self.reward = torch.zeros(G, dtype=torch.float32, device=dev)
    self.logits = torch.zeros((G, A), dtype=torch.float32, device=dev)
    self.hidden_f32 = self.eng.hidden.view(torch.float32)
    self.record = None

  def _plan(self, use_noise, noise_frac, stream_ptr):
    """The launch list of one move as (C function, ctypes args) pairs, built once per (stream,
    noise setting): at ~100 launches per move the Python-side argument marshalling would
    otherwise dominate the un-graphed path."""
    key = (bool(use_noise), float(noise_frac), stream_ptr, self.record is not None)
    if getattr(self, '_plan_key', None) == key:
      return self._plan_list
    eng, net, S, G = self.eng, self.net, self.eng.S, self.hi - self.lo
    lib, P, st = net.lib, _lib.ptr, C.c_void_p(stream_ptr)
    stride = (S + 1) * HIDDEN
    tree = C.byref(eng.tree)
    plan = [net.initial_call(G, self.obs, self.hidden_f32, stride, self.init_value, self.root_logits, st),
            (lib.mz_tree_set_root, (tree, P(self.root_logits), P(self.legal),
                                    P(self.noise) if use_noise else None, float(noise_frac),
                                    P(self.to_play), None, st)),
            (lib.mz_tree_step, (tree, -1, None, None, None, None, None) + eng._trace_ptrs(0) + (st,))]
    bf16 = net.precision == 'bf16'
    for sim in range(S):
      if self.record is not None:
        v, r, l = self.record[0][sim], self.record[1][sim], self.record[2][sim]
      else:
        v, r, l = self.value, self.reward, self.logits
      tail = (G, P(self.hidden_f32), stride, P(eng.leaf_parent), P(eng.leaf_action),
              P(self.hidden_f32), stride, (sim + 1) * HIDDEN, P(v), P(r), P(l), st)
      if bf16:
        plan.append((lib.mz_fc_recurrent_tc, (net.weights, P(net._tc_packed), P(net._tc_tail)) + tail))
      else:
        plan.append((net.recurrent_f32_fn(), (net.weights,) + tail))
      plan.append((lib.mz_tree_step, (tree, sim, P(v), P(r), P(l), None, None) +
                   eng._trace_ptrs(sim + 1) + (st,)))
    plan.append((lib.mz_tree_root_stats, (tree, P(eng.visits), P(eng.child_visits), P(eng.root_value),
                                          P(eng.minmax), st)))
    plan.append((lib.mz_select_action, (G, eng.A, P(eng.visits), P(self.legal), P(self.temperature),
                                        P(self.uniforms), P(eng.actions), st)))
    self._plan_key, self._plan_list = key, plan
    return plan

  def enqueue(self, use_noise, noise_frac):
    plan = self._plan(use_noise, noise_frac, torch.cuda.current_stream().cuda_stream)
    for fn, args in plan:
      rc = fn(*args)
      if rc:
        _lib.check(rc, fn.__name__)
    return len(plan)


class _FusedEngine(object):
  """The whole move in one persistent kernel (`mz_fc_search`): root set-up, S x {descent, network,
  expand + backup} and the root statistics for all games, one launch.  Owns the tree blocks (the fused
  kernel's layout), the bf16 hidden pool and the argument struct; inputs / outputs are the parent's
  whole-batch staging tensors."""

  def __init__(self, config, fcnet, parent):
    from .mcts import pb_c_table, default_prior_sum_mode
    import math
    self.net, self.lib = fcnet, fcnet.lib
    G, S, A, dev = parent.G, parent.S, parent.A, fcnet.device
    self.G, self.S, self.A = G, S, A
    self.game_bytes = int(self.lib.mz_fc_search_game_bytes(S, A))
    self.games = torch.zeros(G * self.game_bytes, dtype=torch.uint8, device=dev)
    self.pool = torch.zeros((G, S + 1, int(self.lib.mz_fc_search_pool_row())), dtype=torch.bfloat16, device=dev)
    self.pb_c = torch.from_numpy(pb_c_table(S, config.pb_c_base, config.pb_c_init)).to(dev)
    self.root_hidden = torch.zeros((G, HIDDEN), dtype=torch.float32, device=dev)
    self.error_flag = torch.zeros(1, dtype=torch.int32, device=dev)
    self.trace = None
    self.record = None
    self.timeline = None
    kb = list(config.known_bounds)
    self.args = _lib.FcSearchArgs()
    a = self.args
    a.num_games, a.num_simulations, a.two_players = G, S, int(bool(config.two_players))
    a.prior_sum_mode = default_prior_sum_mode()
    a.game_bytes = self.game_bytes
    a.discount, a.init_value_score = float(config.discount), float(config.init_value_score)
    a.min_bound = math.inf if kb[0] is None else float(kb[0])
    a.max_bound = -math.inf if kb[1] is None else float(kb[1])
    a.games, a.pb_c_table, a.pool = self.games.data_ptr(), self.pb_c.data_ptr(), self.pool.data_ptr()
    a.root_logits, a.root_hidden = parent.root_logits.data_ptr(), self.root_hidden.data_ptr()
    a.legal_mask, a.root_to_play = parent.legal.data_ptr(), parent.to_play.data_ptr()
    a.visits, a.child_visits = parent.visits.data_ptr(), parent.child_visits.data_ptr()
    a.root_value, a.minmax = parent.root_value.data_ptr(), parent.minmax.data_ptr()
    a.error_flag = self.error_flag.data_ptr()
    self._bind_weights()

  def _bind_weights(self):
    net, a = self.net, self.args
    a.weights = C.pointer(net.weights)
    a.packed, a.tail = net._tc_packed.data_ptr(), net._tc_tail.data_ptr()

  def enable_trace(self):
    self.trace = tuple(torch.zeros((self.S, self.G), dtype=torch.int32, device=self.net.device) for _ in range(3))
    a = self.args
    a.trace_parent, a.trace_action, a.trace_depth = (t.data_ptr() for t in self.trace)

  def enable_record(self):
    dev = self.net.device
    self.record = (torch.zeros((self.S, self.G), dtype=torch.float32, device=dev),
                   torch.zeros((self.S, self.G), dtype=torch.float32, device=dev),
                   torch.zeros((self.S, self.G, self.A), dtype=torch.float32, device=dev))
    a = self.args
    a.rec_value, a.rec_reward, a.rec_logits = (t.data_ptr() for t in self.record)

  def enable_timeline(self):
    """clock64 stamps of tile 0's phases, [S, 32] int64 (diagnostics; see csrc/mz_fcsearch.cu FS_STAMP)."""
    self.timeline = torch.zeros((self.S, 32), dtype=torch.int64, device=self.net.device)
    self.args.timeline = self.timeline.data_ptr()

  def export_game(self, game):
    """Dense copy of one game's tree in the layout of BatchedMCTS.export_game (+ the cached child q)."""
    S, A, dev = self.S, self.A, self.net.device
    prior = torch.zeros((S + 1, A), dtype=torch.float64, device=dev)
    q = torch.zeros((S + 1, A), dtype=torch.float64, device=dev)
    child = torch.zeros((S + 1, A), dtype=torch.int32, device=dev)
    vsum = torch.zeros(S + 1, dtype=torch.float64, device=dev)
    visit = torch.zeros(S + 1, dtype=torch.int32, device=dev)
    reward = torch.zeros(S + 1, dtype=torch.float32, device=dev)
    _lib.check(self.lib.mz_fc_search_export(self.args, int(game), _lib.ptr(prior), _lib.ptr(child), _lib.ptr(vsum),
                                            _lib.ptr(visit), _lib.ptr(reward), _lib.ptr(q), _lib.current_stream()),
               "mz_fc_search_export")
    return dict(prior=prior.cpu().numpy(), child=child.cpu().numpy(), vsum=vsum.cpu().numpy(),
                visit=visit.cpu().numpy(), reward=reward.cpu().numpy(), q=q.cpu().numpy())

  def plan(self, parent, use_noise, noise_frac, st):
    net, lib, P = self.net, self.lib, _lib.ptr
    a = self.args
    a.noise = parent.noise.data_ptr() if use_noise else None
    a.noise_frac = float(noise_frac)
    return [net.initial_call(self.G, parent.obs, self.root_hidden, HIDDEN, parent.init_value, parent.root_logits, st),
            (lib.mz_fc_search, (C.byref(a), st)),
            (lib.mz_select_action, (self.G, self.A, P(parent.visits), P(parent.legal), P(parent.temperature),
                                    P(parent.uniforms), P(parent.actions), st))]


class FCSearch(object):
  """The per-move body of Actor.play_game (actors.py:131-153) for G games with FCNetwork.

  The network kernel reads parent hidden states straight from the tree's hidden pool and writes the
  new state into it.  The games are split into `num_streams` slices that run the same launch
  sequence on their own CUDA streams, so one slice's tree kernel overlaps another slice's network
  kernel (the network kernel only occupies G/128 SMs); every launch of one move is captured in one
  CUDA graph, and inputs / outputs are staged through pinned host buffers for the end-to-end
  (host buffers in, host buffers out) call."""

  def __init__(self, config, fcnet, num_games, noise_frac=None, use_graph=True, num_streams=1, fused=None):
    """fused: True = the whole move in one persistent kernel (`mz_fc_search`, csrc/mz_fcsearch.cu), False =
    one tree launch + one network launch per simulation on `num_streams` slices, None = fused whenever the
    network runs in bf16 with supports of at most 32 bins, at most 8192 games play and the shape fits the kernel:
    S <= 63 and (S, A) within its shared-memory plan, as `mz_fc_search_supported` reports (S <= 63 for A <= 13, S <= 55 for A <= 20, S <= 53 for
    A <= 29, S <= 19 for A <= 32).  Every other shape runs the per-launch path; MZ_FUSED=0 in the environment turns
    the default off.  Both give bit-identical searches (tests/test_gpu_fcnet.py)."""
    self.net = fcnet
    G, A, dev = int(num_games), int(config.action_space), fcnet.device
    self.G, self.A, self.S = G, A, int(config.num_simulations)
    self.noise_frac = float(getattr(config, 'root_exploration_fraction', 0.25)
                            if noise_frac is None else noise_frac)
    self.use_graph = use_graph
    self.graph = None
    self._e2e_key = None
    self.use_noise = True
    self.launches_per_move = 0
    self.obs = torch.zeros((G, fcnet.input_dim), dtype=torch.float32, device=dev)
    # host-visible inputs / outputs live in two blobs so that the end-to-end call moves each with ONE copy
    self._in_specs = [('noise', torch.float64, (G, A)), ('uniforms', torch.float64, (G,)),
                      ('temperature', torch.float64, (G,)), ('legal', torch.int32, _legal_shape(G, A)),
                      ('to_play', torch.int8, (G,)), ('obs_u8', torch.uint8, (G, fcnet.input_dim))]
    self._out_specs = [('root_value', torch.float64, (G,)), ('child_visits', torch.float64, (G, A)),
                       ('actions', torch.int32, (G,)), ('init_value', torch.float32, (G,))]
    self._in_dev, views = _carve(self._in_specs, device=dev)
    self.__dict__.update(views)
    self._out_dev, views = _carve(self._out_specs, device=dev)
    self.__dict__.update(views)
    _fill_all_legal(self.legal, A)
    self.to_play.fill_(1)
    self.temperature.fill_(1.0)
    self.root_logits = torch.zeros((G, A), dtype=torch.float32, device=dev)
    self.visits = torch.zeros((G, A), dtype=torch.int32, device=dev)
    self.minmax = torch.zeros((G, 2), dtype=torch.float64, device=dev)
    # the persistent kernel reads the narrow bf16 image only: supports of at most 32 bins
    can_fuse = (fcnet.precision == 'bf16' and fcnet.weights is not None and
                fcnet.value_bins <= 32 and fcnet.reward_bins <= 32 and
                int(fcnet.lib.mz_fc_search_supported(self.S, A)) == 1)
    if fused is None:
      # measured (profiles/r02l_fused_sweep.log): the persistent kernel wins wherever one wave of clusters holds
      # the games (C4 204 vs 140, C1 254 vs 199, C3 253 vs 196 M expansions/s), ties at 1024 games and loses a
      # few per cent from 16 384 games on, where the per-launch path has more games in flight per SM
      fused = can_fuse and os.environ.get("MZ_FUSED", "1") != "0" and G <= 8192
    elif fused and not can_fuse:
      raise ValueError("the fused search kernel needs a bf16 FCNetwork with loaded weights, A <= 32, value and "
                       "reward supports of at most 32 bins, S <= 63 and a tree that fits its shared-memory plan")
    self.fused = _FusedEngine(config, fcnet, self) if fused else None
    self.lanes = []
    self.eng = None
    if self.fused is not None:
      return
    ns = max(1, min(int(num_streams), G))
    bounds = [(G * i) // ns for i in range(ns + 1)]
    self.lanes = []
    for i in range(ns):
      stream = None if ns == 1 else torch.cuda.Stream(device=dev)
      self.lanes.append(_Lane(config, fcnet, bounds[i], bounds[i + 1], self, stream))
    self.eng = self.lanes[0].eng  # single-lane convenience (tests, kernel breakdown)

  # -- recording for parity checks -----------------------------------------------------------------
  def enable_record(self):
    """Keep every simulation's network outputs (and the engines' parent/action/depth traces) so
    that a checker can replay the search with identical network outputs."""
    dev = self.net.device
    if self.fused is not None:
      self.fused.enable_record()
      self.fused.enable_trace()
      self.graph = None
      self._e2e_key = None
      self._fused_plan_key = None
      return
    for lane in self.lanes:
      g = lane.hi - lane.lo
      lane.record = (torch.zeros((self.S, g), dtype=torch.float32, device=dev),
                     torch.zeros((self.S, g), dtype=torch.float32, device=dev),
                     torch.zeros((self.S, g, self.A), dtype=torch.float32, device=dev))
      lane.eng.enable_trace()
    self.graph = None
    self._e2e_key = None

  @property
  def record(self):
    if self.fused is not None:
      return self.fused.record
    if self.lanes[0].record is None:
      return None
    return tuple(torch.cat([lane.record[i] for lane in self.lanes], dim=1) for i in range(3))

  @property
  def trace(self):
    if self.fused is not None:
      return self.fused.trace
    return tuple(torch.cat([lane.eng.trace[i] for lane in self.lanes], dim=1) for i in range(3))

  # -- launch sequence -----------------------------------------------------------------------------
  def _enqueue(self):
    """All launches of one move; lanes fork from / join back into the current stream."""
    if self.fused is not None:
      stream_ptr = torch.cuda.current_stream().cuda_stream
      key = (bool(self.use_noise), float(self.noise_frac), stream_ptr)
      if getattr(self, '_fused_plan_key', None) != key:
        self._fused_plan = self.fused.plan(self, self.use_noise, self.noise_frac, C.c_void_p(stream_ptr))
        self._fused_plan_key = key
      for fn, args in self._fused_plan:
        rc = fn(*args)
        if rc:
          _lib.check(rc, fn.__name__)
      self.launches_per_move = len(self._fused_plan)
      return
    if len(self.lanes) == 1:
      self.launches_per_move = self.lanes[0].enqueue(self.use_noise, self.noise_frac)
      return
    main = torch.cuda.current_stream()
    fork = torch.cuda.Event()
    fork.record(main)
    n = 0
    for lane in self.lanes:
      lane.stream.wait_event(fork)
      with torch.cuda.stream(lane.stream):
        n += lane.enqueue(self.use_noise, self.noise_frac)
        done = torch.cuda.Event()
        done.record(lane.stream)
      main.wait_event(done)
    self.launches_per_move = n

  @_lib.on_device
  def run(self):
    """One move for all games with inputs already in the device staging buffers."""
    if not self.use_graph:
      self._enqueue()
      return
    if self.graph is None:
      # warm up once outside capture (lazy module loading, cudaFuncSetAttribute)
      self._enqueue()
      torch.cuda.synchronize()
      self.graph = torch.cuda.CUDAGraph()
      with torch.cuda.graph(self.graph):
        self._enqueue()
    self.graph.replay()

  # -- end-to-end call: host buffers in, host buffers out ----------------------------------------
  def _pinned(self):
    if getattr(self, '_h', None) is None:
      self._in_host, h = _carve(self._in_specs, pin_memory=True)
      self._out_host, out = _carve(self._out_specs, pin_memory=True)
      h.update(out)
      h['obs'] = torch.zeros((self.G, self.net.input_dim), dtype=torch.float32, pin_memory=True)
      _fill_all_legal(h['legal'], self.A)
      h['to_play'].fill_(1)
      h['temperature'].fill_(1.0)
      self._h = h
    return self._h

  def pinned_inputs(self):
    """Pinned host views of the per-move inputs (one contiguous blob): 'obs_u8' [G, input_dim] uint8,
    'noise' [G, A] f64, 'uniforms' [G] f64, 'temperature' [G] f64, 'legal' [G] i32 bit masks ([G, W] words when
    A > 32, layout of mcts.legal_words), 'to_play' [G] i8.  Write the move's inputs here and call `search_pinned()`: no host-side staging copy."""
    h = self._pinned()
    return {name: h[name] for name, _, _ in self._in_specs}

  @_lib.on_device
  def search_pinned(self):
    """search_host for inputs already written into `pinned_inputs()` (byte observations): ONE
    host->device copy of the input blob, normalisation + the move's graph, ONE device->host copy of the
    output blob.  Returns the pinned (actions, root_value, child_visits, init_value)."""
    h = self._pinned()
    mn, rg = getattr(self, '_obs_norm', (None, None))
    if self.fused is not None and self.use_graph:
      # ONE graph launch for the whole call: the observation bytes cross first and the initial inference starts on
      # them while the rest of the blob (noise, uniforms, temperatures, masks) crosses on a second branch that joins
      # in front of the search kernel; the output blob's copy is the graph's last node
      key = (bool(self.use_noise), float(self.noise_frac), None if mn is None else mn.data_ptr(),
             None if rg is None else rg.data_ptr())
      if getattr(self, '_e2e_key', None) != key:
        self._e2e_graph, self._e2e_key = self._capture_e2e(mn, rg), key
      self._e2e_graph.replay()
      torch.cuda.current_stream().synchronize()
      return h['actions'], h['root_value'], h['child_visits'], h['init_value']
    self._in_dev.copy_(self._in_host, non_blocking=True)
    _lib.check(self.net.lib.mz_obs_normalize_u8(self.G, self.net.input_dim, _lib.ptr(self.obs_u8), _lib.ptr(mn),
                                                _lib.ptr(rg), _lib.ptr(self.obs), _lib.current_stream()),
               "mz_obs_normalize_u8")
    self.run()
    self._out_host.copy_(self._out_dev, non_blocking=True)
    torch.cuda.current_stream().synchronize()
    return h['actions'], h['root_value'], h['child_visits'], h['init_value']

  def _capture_e2e(self, mn, rg):
    """The CUDA graph behind `search_pinned` (fused path)."""
    def body():
      self._in_dev.copy_(self._in_host, non_blocking=True)
      _lib.check(self.net.lib.mz_obs_normalize_u8(self.G, self.net.input_dim, _lib.ptr(self.obs_u8), _lib.ptr(mn),
                                                  _lib.ptr(rg), _lib.ptr(self.obs), _lib.current_stream()),
                 "mz_obs_normalize_u8")
      self._enqueue()
      self._out_host.copy_(self._out_dev, non_blocking=True)

    body()  # warm up once outside capture (lazy module loading, cudaFuncSetAttribute)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
      body()
    return graph

  def draw_noise(self, alpha):
    """Node.add_exploration_noise's Dirichlet draw (mcts.py:59) for every root, made on the device from the legal
    masks already staged there (`mz_dirichlet_noise`): same distribution as np.random.dirichlet, another stream.
    The seed comes from np.random at first use, so `np.random.seed` still fixes a run."""
    if getattr(self, '_noise_seed', None) is None:
      self._noise_seed, self._noise_move = int(np.random.randint(1 << 62)), 0
    _lib.check(self.net.lib.mz_dirichlet_noise(self.G, self.A, float(alpha), _lib.ptr(self.legal), self._noise_seed,
                                               self._noise_move, _lib.ptr(self.noise), _lib.current_stream()),
               "mz_dirichlet_noise")
    self._noise_move += 1
    self.use_noise = True

  @_lib.on_device
  def search_host(self, obs, noise=None, uniforms=None, temperature=None, legal=None, to_play=None,
                  dirichlet_alpha=None, wait=True):
    """The per-move body of Actor.play_game (actors.py:131-153) for G games.

    Inputs are HOST arrays (numpy or CPU tensors): obs [G, input_dim] float32 -- or uint8, in which
    case only the bytes cross PCIe and `(obs - obs_min) / obs_range` (actors.py:127-129, set with
    `set_obs_normalization`, default 0 / 255) runs on the device in the same float32 arithmetic --, Dirichlet noise
    [G, A] float64 (row g: one value per legal action of game g, in action order), uniforms [G]
    float64 (action sampling), temperature [G] float64, and optionally the roots' legal-action bit
    masks (actors.py:141-142; any form mcts.legal_words takes: [G] integers with bit a = action a, a bool [G, A]
    array, or [G, W] words) and to_play [G] (+1 / -1).  Returns
    pinned host tensors: actions [G] i32, root_value [G] f64, child_visits [G, A] f64, and the
    initial-inference value [G] f32 (the priority seed `error = root.value() - value`,
    actors.py:147).  Host->device and device->host copies are part of the call.  With `dirichlet_alpha` set and no
    `noise` buffer the root noise is drawn on the device instead (`draw_noise`).
    wait=False: the call returns once everything is enqueued; `search_result()` waits for the move and returns the
    outputs (the host side of another actor's move then runs under this search: selfplay.PipelinedActors).
    """
    h = self._pinned()
    def stage(name, src, dst):
      if src is None:
        return
      t = src if torch.is_tensor(src) else torch.from_numpy(src)
      if not t.is_pinned():
        h[name].copy_(t)
        t = h[name]
      dst.copy_(t, non_blocking=True)
    t_obs = obs if torch.is_tensor(obs) else torch.from_numpy(obs)
    if t_obs.dtype == torch.uint8:
      stage('obs_u8', t_obs, self.obs_u8)
      mn, rg = getattr(self, '_obs_norm', (None, None))
      _lib.check(self.net.lib.mz_obs_normalize_u8(self.G, self.net.input_dim, _lib.ptr(self.obs_u8), _lib.ptr(mn),
                                                  _lib.ptr(rg), _lib.ptr(self.obs), _lib.current_stream()),
                 "mz_obs_normalize_u8")
    else:
      stage('obs', t_obs, self.obs)
    stage('noise', noise, self.noise)
    stage('uniforms', uniforms, self.uniforms)
    stage('temperature', temperature, self.temperature)
    if legal is not None:
      from .mcts import legal_words
      stage('legal', legal_words(legal, self.G, self.A).reshape(self.legal.shape), self.legal)
    if to_play is not None:
      stage('to_play', np.ascontiguousarray(np.asarray(to_play, dtype=np.int8)), self.to_play)
    self.use_noise = noise is not None or self.use_noise
    if noise is None and dirichlet_alpha is not None:
      self.draw_noise(dirichlet_alpha)
    self.run()
    self._out_host.copy_(self._out_dev, non_blocking=True)  # the four outputs share one blob
    if not wait:
      if getattr(self, '_done', None) is None:
        self._done = torch.cuda.Event()
      self._done.record()
      return None
    torch.cuda.current_stream().synchronize()
    return h['actions'], h['root_value'], h['child_visits'], h['init_value']

  def search_result(self):
    """The outputs of the move a `search_host(..., wait=False)` call enqueued (pinned host tensors)."""
    self._done.synchronize()
    h = self._pinned()
    return h['actions'], h['root_value'], h['child_visits'], h['init_value']

  def set_obs_normalization(self, obs_min, obs_range):
    """Per-feature float32 obs_min / obs_range (config.obs_range[::2], max - min: actors.py:60-63) for
    uint8 observations handed to `search_host`."""
    dev = self.obs.device
    self._obs_norm = (torch.as_tensor(obs_min, dtype=torch.float32).to(dev).contiguous(),
                      torch.as_tensor(obs_range, dtype=torch.float32).to(dev).contiguous())

  def h2d_bytes(self, obs_bytes_per_element=4):
    return (self.obs.numel() * obs_bytes_per_element + self.noise.numel() * 8 + self.uniforms.numel() * 8 +
            self.temperature.numel() * 8)

  def d2h_bytes(self):
    return self._out_dev.numel()

  def h2d_blob_bytes(self):
    return self._in_dev.numel()


def _all_legal(A):
  """int32 legal-mask words with the low A bits set (a full word: all ones = -1 as a signed word)."""
  return [-1 if A >= 32 * (w + 1) else (1 << (A - 32 * w)) - 1 for w in range((A + 31) // 32)]


def _legal_shape(G, A):
  """Legal masks of the per-launch path: one int32 word per game up to 32 actions, [G, W] words above."""
  return (G,) if A <= 32 else (G, (A + 31) // 32)


def _fill_all_legal(legal, A):
  legal.view(legal.shape[0], -1).copy_(torch.tensor(_all_legal(A), dtype=torch.int32).expand(legal.shape[0], -1))


def _carve(specs, **alloc):
  """One uint8 blob + typed views into it, every view 8-byte aligned."""
  offs, off = [], 0
  for _, dtype, shape in specs:
    off = (off + 7) // 8 * 8
    offs.append(off)
    n = 1
    for d in shape:
      n *= d
    off += n * torch.empty((), dtype=dtype).element_size()
  blob = torch.zeros((off + 7) // 8 * 8, dtype=torch.uint8, **alloc)
  views = {}
  for (name, dtype, shape), o in zip(specs, offs):
    n = 1
    for d in shape:
      n *= d
    nbytes = n * torch.empty((), dtype=dtype).element_size()
    views[name] = blob[o:o + nbytes].view(dtype).view(shape)
  return blob, views


def random_state_dict(input_dim, action_space, value_bins=31, reward_bins=31, seed=1234):
  """Random-init weights of the FCNetwork architecture under the reference's state-dict keys
  (torch's default nn.Linear initialisation, LayerNorm = identity affine).  For benchmarks and
  smoke tests: there is no network access for checkpoints."""
  import torch.nn as nn
  gen_state = torch.random.get_rng_state()
  torch.manual_seed(seed)
  dims = [('representation_head', 'out', input_dim, HIDDEN), ('value_head', 'value', HIDDEN, value_bins),
          ('policy_head', 'policy', HIDDEN, action_space),
          ('reward_head', 'reward', HIDDEN + action_space, reward_bins),
          ('transition_head', 'out', HIDDEN + action_space, HIDDEN)]
  sd = {}
  for head, out_name, d_in, d_out in dims:
    fc1, out = nn.Linear(d_in, _lib.FC_WIDTH), nn.Linear(_lib.FC_WIDTH, d_out)
    sd[head + '.fc1.weight'], sd[head + '.fc1.bias'] = fc1.weight.detach(), fc1.bias.detach()
    sd['%s.%s.weight' % (head, out_name)] = out.weight.detach()
    sd['%s.%s.bias' % (head, out_name)] = out.bias.detach()
  sd['LN.weight'], sd['LN.bias'] = torch.ones(HIDDEN), torch.zeros(HIDDEN)
  torch.random.set_rng_state(gen_state)
  return sd
