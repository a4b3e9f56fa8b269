"""Learner step of the reference (Learner.update_weights / learn, learners.py:116-230) around the
fused unroll-loss kernel.

What runs where:
  * the train-mode network (support logits, backward) is a plain torch module with the reference's
    state-dict keys (`FCNetworkTrain`, networks.py:55-174) -- library GEMMs, as SURVEY.md section 8
    f-4 prescribes;
  * everything between the logits and the scalar losses -- h(x) of the targets (config.py:51-54),
    the two-hot projection (config.py:56-68), the three cross-entropies (utils.py:53-56), the
    float64 importance weighting and means (learners.py:208-210), the 1/K gradient scale
    (learners.py:213), the priority errors (learners.py:182-183) and the gradient with respect to
    every logit -- is ONE launch of `mz_unroll_loss` (csrc/mz_unroll_loss.cu) wrapped in
    `UnrollLoss`, a torch.autograd.Function;
  * with torch.distributed initialised, the gradients are averaged over the ranks through one flat
    all-reduce (parallel.allreduce_gradients) before clipping and the optimiser step, and
    `send_weights` hands the new weights to the search network (and to the other ranks).

There is no CPU fallback: the loss needs the CUDA library.
"""
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, parallel
from .networks import HIDDEN, NetworkOutput

WIDTH = _lib.FC_WIDTH


# ------------------------------------------------------------------------------------------------
# train-mode network
# ------------------------------------------------------------------------------------------------
class _Head(nn.Module):
  """Linear(d_in, 512) -> ReLU -> Linear(512, d_out); the reference names the second layer after the
  head (networks.py:55-119)."""

  def __init__(self, d_in, d_out, out_name):
    super().__init__()
    self.fc1 = nn.Linear(d_in, WIDTH)
    self.add_module(out_name, nn.Linear(WIDTH, d_out))
    self._out = out_name

  def forward(self, x):
    return getattr(self, self._out)(F.relu(self.fc1(x)))


class FCNetworkTrain(nn.Module):
  """The reference's FCNetwork (networks.py:122-174) in train mode: value / reward are support
  logits.  Same parameter names, so `get_weights()` feeds `networks.FCNetwork.load_weights` (the
  search kernels) and reference checkpoints load unchanged."""

  def __init__(self, input_dim, action_space, device, config):
    super().__init__()
    self.action_space = int(action_space)
    vmin, vmax = [int(v) for v in config.value_support]
    rmin, rmax = [int(v) for v in config.reward_support]
    no_support = bool(getattr(config, 'no_support', False))  # networks.py:135-136: one-unit scalar heads
    self.representation_head = _Head(input_dim, HIDDEN, 'out')
    self.value_head = _Head(HIDDEN, 1 if no_support else vmax - vmin + 1, 'value')
    self.policy_head = _Head(HIDDEN, self.action_space, 'policy')
    self.reward_head = _Head(HIDDEN + self.action_space, 1 if no_support else rmax - rmin + 1, 'reward')
    self.transition_head = _Head(HIDDEN + self.action_space, HIDDEN, 'out')
    self.LN = nn.LayerNorm([HIDDEN], elementwise_affine=True)
    self.device = torch.device(device)
    self.to(self.device)
    self.train()

  def initial_inference(self, observation):
    h = F.relu(self.LN(self.representation_head(observation.reshape(observation.shape[0], -1))))
    return NetworkOutput(self.value_head(h), 0, self.policy_head(h), h)

  def recurrent_inference(self, hidden_state, action):
    a = torch.as_tensor(action, dtype=torch.int64, device=hidden_state.device).reshape(-1, 1)
    one_hot = torch.zeros((a.shape[0], self.action_space), dtype=torch.float32, device=hidden_state.device)
    one_hot.scatter_(1, a, 1.0)
    x = torch.cat((hidden_state, one_hot), dim=1)
    reward = self.reward_head(x)
    h = F.relu(self.LN(self.transition_head(x)))
    return NetworkOutput(self.value_head(h), reward, self.policy_head(h), h)

  def unroll(self, observation, actions):
    """The K+1 network evaluations of one learner step (learners.py:175-206) with the heads batched:
    only the transition head is a recurrence; value / policy (and reward) logits of all unroll steps
    come from ONE head evaluation over the stacked hidden states, which cuts the step's launch count by
    ~40 %.  Every hidden state produced by the dynamics carries the reference's 0.5 gradient hook
    (learners.py:201), which sees the sum of the gradients from its heads and from the next step, as in
    the reference.  actions: [B, K] int64.  Returns stacked logits (value [K+1, B, V], reward [K, B, R],
    policy [K+1, B, A])."""
    B, K = actions.shape
    h = F.relu(self.LN(self.representation_head(observation.reshape(B, -1))))
    one_hot = torch.zeros((K, B, self.action_space), dtype=torch.float32, device=h.device)
    one_hot.scatter_(2, actions.t().reshape(K, B, 1), 1.0)
    hs, xs = [h], []
    for i in range(K):
      x = torch.cat((h, one_hot[i]), dim=1)
      h = F.relu(self.LN(self.transition_head(x)))
      h.register_hook(lambda grad: grad * 0.5)
      xs.append(x)
      hs.append(h)
    hs = torch.cat(hs, dim=0)
    value = self.value_head(hs).reshape(K + 1, B, -1)
    policy = self.policy_head(hs).reshape(K + 1, B, -1)
    reward = self.reward_head(torch.cat(xs, dim=0)).reshape(K, B, -1)
    return value, reward, policy

  def load_weights(self, weights):
    self.load_state_dict(weights)

  def get_weights(self):
    return {key: value.cpu() for key, value in self.state_dict().items()}


# ------------------------------------------------------------------------------------------------
# fused loss
# ------------------------------------------------------------------------------------------------
class UnrollLoss(torch.autograd.Function):
  """losses[3] (reward, value, policy; float64) and new_errors[B] from the stacked logits.  The
  gradient the kernel stores already carries the 1/K of learners.py:213; backward only multiplies by
  the incoming gradient of each loss."""

  @staticmethod
  def forward(ctx, value_logits, reward_logits, policy_logits, t_values, t_rewards, t_policies, is_weights,
              cfg):
    for t in (value_logits, reward_logits, policy_logits, t_values, t_rewards, t_policies):
      if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
        raise RuntimeError("unroll_loss takes contiguous float32 CUDA tensors (there is no CPU fallback)")
    K1, B, V = value_logits.shape
    K, A = K1 - 1, policy_logits.shape[2]
    if tuple(reward_logits.shape[:2]) != (K, B) or tuple(policy_logits.shape[:2]) != (K1, B):
      raise ValueError("logits must be stacked [steps][batch][bins]")
    if tuple(t_values.shape) != (B, K1) or tuple(t_rewards.shape) != (B, K1) or \
       tuple(t_policies.shape) != (B, K1, A):
      raise ValueError("targets must be [batch][K+1](, [A]) as sample_batch returns them")
    c = _lib.LossCfg(B, K, A, cfg['value_min'], cfg['value_max'], cfg['reward_min'], cfg['reward_max'],
                     int(cfg['no_target_transform']))
    if V != c.value_max - c.value_min + 1 or reward_logits.shape[2] != c.reward_max - c.reward_min + 1:
      raise ValueError("logit widths do not match the supports")
    if is_weights is not None:
      is_weights = is_weights.to(value_logits.device, torch.float64).contiguous()
    dev = value_logits.device
    d_v, d_r, d_p = torch.empty_like(value_logits), torch.empty_like(reward_logits), torch.empty_like(policy_logits)
    rows = torch.empty((3, B), dtype=torch.float64, device=dev)
    losses = torch.empty(3, dtype=torch.float64, device=dev)
    new_errors = torch.empty(B, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):  # the launch goes to the logits' GPU, whatever the caller's current device is
      _lib.check(_lib.load().mz_unroll_loss(
          c, _lib.ptr(value_logits), _lib.ptr(reward_logits), _lib.ptr(policy_logits), _lib.ptr(t_values),
          _lib.ptr(t_rewards), _lib.ptr(t_policies), _lib.ptr(is_weights), _lib.ptr(d_v), _lib.ptr(d_r),
          _lib.ptr(d_p), _lib.ptr(rows), _lib.ptr(losses), _lib.ptr(new_errors), _lib.current_stream()),
                 "mz_unroll_loss")
    ctx.save_for_backward(d_v, d_r, d_p)
    ctx.mark_non_differentiable(new_errors)
    return losses, new_errors

  @staticmethod
  def backward(ctx, g_losses, _g_errors):
    d_v, d_r, d_p = ctx.saved_tensors
    g = g_losses.to(torch.float32)
    return d_v * g[1], d_r * g[0], d_p * g[2], None, None, None, None, None


def loss_cfg(config):
  vmin, vmax = [int(v) for v in config.value_support]
  rmin, rmax = [int(v) for v in config.reward_support]
  return dict(value_min=vmin, value_max=vmax, reward_min=rmin, reward_max=rmax,
              no_target_transform=bool(getattr(config, 'no_target_transform', False)))


def unroll_loss(config, values, rewards, policies, t_values, t_rewards, t_policies, is_weights):
  """values / policies: the K+1 per-step logits [B, bins] as lists or stacked [K+1, B, bins] tensors;
  rewards: the K logits of steps 1..K.  Returns (losses[3] float64 = reward, value, policy;
  new_errors[B] float32)."""
  stacked = [t.contiguous() if torch.is_tensor(t) else torch.stack(t, 0) for t in (values, rewards, policies)]
  return UnrollLoss.apply(stacked[0], stacked[1], stacked[2], t_values, t_rewards, t_policies, is_weights,
                          loss_cfg(config))


def scalar_unroll_loss(config, values, rewards, policies, t_values, t_rewards, t_policies, is_weights):
  """The loss half of Learner.update_weights for `--no_support` networks (learners.py:182-213 with utils.py:61-70):
  the value / reward heads emit one scalar, compared with the (h-transformed unless no_target_transform) targets by
  `--scalar_loss` MSE or Huber (SmoothL1), the policy by cross entropy; importance weights in float64, the 1/K
  gradient scale of learners.py:213 inside.  Same signature and results layout as `unroll_loss`; plain torch
  (this configuration is outside the benchmarked ones -- the fused CUDA loss covers the support heads)."""
  v, r, p = [t if torch.is_tensor(t) else torch.stack(t, 0) for t in (values, rewards, policies)]
  K = r.shape[0]
  with torch.no_grad():
    new_errors = v[0].squeeze(-1) - t_values[:, 0]  # learners.py:182-183: no inverse transform
    if not getattr(config, 'no_target_transform', False):  # config.py:51-54
      h = lambda x: torch.sign(x) * (torch.sqrt(torch.abs(x) + 1) - 1) + 0.001 * x
      t_values, t_rewards = h(t_values), h(t_rewards)
  kind = getattr(config, 'scalar_loss', 'MSE')
  if kind == 'MSE':
    scalar = torch.nn.MSELoss(reduction='none')
  elif kind == 'Huber':
    scalar = torch.nn.SmoothL1Loss(reduction='none')
  else:
    raise NotImplementedError(kind)
  value_loss = sum(scalar(v[i].squeeze(-1), t_values[:, i]) for i in range(K + 1))
  reward_loss = sum(scalar(r[i - 1].squeeze(-1), t_rewards[:, i]) for i in range(1, K + 1)) if K else torch.zeros_like(value_loss)
  policy_loss = sum((-t_policies[:, i] * F.log_softmax(p[i], dim=1)).sum(1) for i in range(K + 1))
  losses = torch.stack([(is_weights * reward_loss).mean(), (is_weights * value_loss).mean(),
                        (is_weights * policy_loss).mean()])
  if losses.requires_grad:
    losses.register_hook(lambda grad: grad * (1.0 / max(K, 1)))
  return losses, new_errors


# ------------------------------------------------------------------------------------------------
# optimisers / schedules (utils.py:72-128)
# ------------------------------------------------------------------------------------------------
def get_optimizer(config, parameters, capturable=False, lr=None):
  """utils.py:72-83.  capturable: optimiser state (step counters) lives on the device so that the
  step can sit inside a CUDA graph; lr may then be a device tensor a schedule updates in place."""
  name = config.optimizer
  lr = config.lr_init if lr is None else lr
  cap = dict(capturable=True) if capturable else {}
  if name == 'RMSprop':
    return torch.optim.RMSprop(parameters, lr=lr, momentum=config.momentum, eps=0.01,
                               weight_decay=config.weight_decay, **cap)
  if name == 'Adam':
    return torch.optim.Adam(parameters, lr=lr, weight_decay=config.weight_decay, eps=0.00015, **cap)
  if name == 'AdamW':
    return torch.optim.AdamW(parameters, lr=lr, weight_decay=config.weight_decay, eps=0.00015, **cap)
  if name == 'SGD':
    return torch.optim.SGD(parameters, lr=lr, momentum=config.momentum, weight_decay=config.weight_decay)
  raise NotImplementedError(name)


def load_optimizer_state(optimizer, state_dict, device):
  """optimizer.load_state_dict(state_dict), keeping how this optimiser runs its step: a learning rate held in a device
  scalar (which a captured step reads) stays that scalar, and `capturable` with it the place of the step counters
  (on `device` when capturable, on the host otherwise) -- neither is the checkpoint's to decide."""
  group = dict(optimizer.param_groups[0])
  optimizer.load_state_dict(state_dict)
  g = optimizer.param_groups[0]
  if torch.is_tensor(group['lr']):
    group['lr'].fill_(float(g['lr']))
    g['lr'] = group['lr']
  if 'capturable' in group:
    g['capturable'] = group['capturable']
    for st in optimizer.state.values():
      if torch.is_tensor(st.get('step')):
        st['step'] = st['step'].to(device if g['capturable'] else 'cpu', torch.float32)


def _set_lr(optimizer, lr):
  for group in optimizer.param_groups:
    if torch.is_tensor(group["lr"]):
      group["lr"].fill_(lr)  # read by the captured optimiser step
    else:
      group["lr"] = lr


class MuZeroLR(object):
  """lr_init * decay_rate ** (step / decay_steps)  (utils.py:87-101)."""

  def __init__(self, optimizer, config):
    self.optimizer, self.lr_init = optimizer, config.lr_init
    self.lr_decay_steps, self.lr_decay_rate = config.lr_decay_steps, config.lr_decay_rate
    self.lr_step, self.lr = 0, config.lr_init

  def step(self):
    self.lr_step += 1
    self.lr = self.lr_init * self.lr_decay_rate ** (self.lr_step / self.lr_decay_steps)
    _set_lr(self.optimizer, self.lr)


class WarmUpLR(object):
  """Linear warm-up over 5000 steps (utils.py:104-120)."""

  def __init__(self, optimizer, config):
    self.optimizer, self.max_lr, self.warm_up_steps, self.lr_step = optimizer, config.lr_init, 5000, 0
    self.lr = (1 / self.warm_up_steps) * self.max_lr
    _set_lr(self.optimizer, self.lr)

  def step(self):
    self.lr_step += 1
    if self.lr_step <= self.warm_up_steps:
      self.lr = (self.lr_step / self.warm_up_steps) * self.max_lr
      _set_lr(self.optimizer, self.lr)


def get_lr_scheduler(config, optimizer):
  kind = getattr(config, 'lr_scheduler', None)
  if kind is None:
    return None
  if kind == 'ExponentialLR':
    return torch.optim.lr_scheduler.ExponentialLR(optimizer, config.lr_decay_rate)
  if kind == 'MuZeroLR':
    return MuZeroLR(optimizer, config)
  if kind == 'WarmUpLR':
    return WarmUpLR(optimizer, config)
  raise NotImplementedError(kind)


# ------------------------------------------------------------------------------------------------
# the learner
# ------------------------------------------------------------------------------------------------
class Learner(object):
  """Learner (learners.py:16-230) without the Ray / logging plumbing: same `update_weights(batch)`
  on the tuple `PrioritizedReplay.sample_batch()` returns, same optimisers, schedules, gradient
  clipping, priority feedback (`replay_buffer.update(idxs, new_errors)`) and weight hand-off.

  network: a train-mode module with the reference's interface (default `FCNetworkTrain`);
  search_network: optional `networks.FCNetwork` that `send_weights()` refreshes;
  loss_fn(config, values, rewards, policies, t_values, t_rewards, t_policies, is_weights) ->
  (losses[3], new_errors): defaults to the CUDA kernel (`unroll_loss`); the gloo tests of the
  data-parallel step pass the oracle's torch restatement because they run without a GPU.

  use_graph: the step's ~400 small launches (5 MLPs x (K+1) steps forward and backward, the loss, the
  optimiser) are captured once in CUDA graphs and replayed on static input buffers: graph 1 = forward
  + fused loss + backward, graph 2 = gradient clipping + optimiser step (device-side step counters,
  learning rate in a device scalar the schedule updates in place); between them, at N > 1, the eager
  gradient all-reduce.  The first step runs eagerly (it initialises the optimiser state)."""

  def __init__(self, config, network, replay_buffer=None, search_network=None, state=None, loss_fn=None,
               use_graph=False, batched_heads=True):
    self.batched_heads = bool(batched_heads)  # network.unroll (heads over all steps at once) when offered
    self.config = config
    self.network = network
    self.network.train()
    self.device = next(network.parameters()).device
    if loss_fn is None:
      _lib.require_cuda()
      if self.device.type != 'cuda':
        raise RuntimeError("the B200 learner only runs on CUDA devices, got %s" % self.device)
      loss_fn = scalar_unroll_loss if getattr(config, 'no_support', False) else unroll_loss
    self.loss_fn = loss_fn
    self.replay_buffer = replay_buffer
    self.search_network = search_network
    self.use_graph = bool(use_graph)
    if self.use_graph and self.device.type != 'cuda':
      raise RuntimeError("use_graph needs a CUDA device")
    # SGD has no capturable mode: its step is graph-safe only while lr is a constant
    scheduled = getattr(config, 'lr_scheduler', None) is not None
    self._graph_opt = self.use_graph and not (config.optimizer == 'SGD' and scheduled)
    lr = torch.tensor(float(config.lr_init), device=self.device) if (self._graph_opt and scheduled) else None
    self.optimizer = get_optimizer(config, self.network.parameters(),
                                   capturable=self._graph_opt and config.optimizer != 'SGD', lr=lr)
    self.lr_scheduler = get_lr_scheduler(config, self.optimizer)
    self._graphs = None
    self.training_step = 0
    self.losses_to_log = {'reward': 0., 'value': 0., 'policy': 0.}
    self.last_losses = self.last_errors = None
    if getattr(config, 'norm_obs', False):
      lo = torch.tensor(config.obs_range[::2], dtype=torch.float32, device=self.device)
      hi = torch.tensor(config.obs_range[1::2], dtype=torch.float32, device=self.device)
      self.obs_min, self.obs_range = lo, hi - lo
    if state is not None:
      self.load_state(state)

  # -- checkpoint (learners.py:59-82) ------------------------------------------------------------
  def load_state(self, state):
    """Resumes from a `save_state` checkpoint, or from a `fused_learner.FusedLearner` one: its flat optimiser state is
    mapped onto FCNetworkTrain's parameters by name (checkpoints.flat_to_module), checked before anything is written,
    and loaded the way this learner runs its step (capturable or not, learning rate in a device scalar or not)."""
    from . import checkpoints  # checkpoints builds FCNetworkTrain: imported here, where learners is complete
    opt = state['optimizer']
    if checkpoints.is_flat_form(opt) and ('exp_avg' in opt or len(list(self.network.parameters())) != 1):
      opt = self._module_state(checkpoints, state)
      self.network.load_state_dict(state['weights'])
      load_optimizer_state(self.optimizer, opt, self.device)
      self._graphs = None  # the captured optimiser step read the replaced state tensors
    else:
      self.network.load_state_dict(state['weights'])
      self.optimizer.load_state_dict(opt)
    self.training_step = state['training_step']
    if self.replay_buffer is not None and 'total_frames' in state:
      self.replay_buffer.add_initial_throughput(state['total_frames'], state['total_games'])

  def _module_state(self, checkpoints, state):
    """A FusedLearner checkpoint's optimiser state as this learner's, after every check that can refuse it."""
    shapes = [(name, tuple(p.shape)) for name, p in self.network.named_parameters()]
    geometry = dict(shapes)
    try:
      input_dim = geometry['representation_head.fc1.weight'][1]
      action_space = geometry['policy_head.policy.weight'][0]
    except KeyError:
      input_dim = action_space = None
    if input_dim is None or shapes != checkpoints.module_params(input_dim, action_space, self.config):
      raise ValueError("flat optimiser state maps only onto the FCNetwork parameters (learners.FCNetworkTrain), "
                       "this learner's network has others")
    saved_kind = getattr(state.get('config'), 'optimizer', self.config.optimizer)
    if saved_kind != self.config.optimizer:
      raise ValueError("the checkpoint of a FusedLearner holds %s optimiser state, this learner runs %s" %
                       (saved_kind, self.config.optimizer))
    opt = checkpoints.flat_to_module(state['optimizer'], self.config, input_dim, action_space)
    weights = state['weights']
    for name, shape in shapes:
      if name not in weights or tuple(weights[name].shape) != shape:
        raise ValueError("the checkpoint's weight %s has shape %s, this network's %s" % (
            name, tuple(weights[name].shape) if name in weights else None, shape))
    return opt

  def save_state(self, path=None, actor_games=None, dirs=None):
    """The checkpoint dictionary of learners.py:72-83 with every key the reference's tooling reads
    (evaluate.py: `config`, `weights`; actors.py:75-79: `actor_games[actor_key]`; learners.py:62-70:
    `optimizer`, `training_step`, `total_frames`, `total_games`).  `actor_games` is the per-actor game counter
    SharedStorage keeps in the reference (default: the attribute set by the self-play driver, else empty);
    `dirs` the logger's directory table.  Written with torch.save when `path` is given (the reference saves to
    dirs['saves']/<training_step>)."""
    tp = self.replay_buffer.get_throughput() if self.replay_buffer is not None else {'frames': 0, 'games': 0}
    state = {'dirs': dict(dirs if dirs is not None else getattr(self, 'dirs', {}) or {}),
             'config': self.config,
             'weights': self.network.get_weights(), 'optimizer': self.optimizer.state_dict(),
             'training_step': self.training_step, 'total_games': tp['games'], 'total_frames': tp['frames'],
             'actor_games': dict(actor_games if actor_games is not None else getattr(self, 'actor_games', {}) or {})}
    if path is not None:
      torch.save(state, path)
    self.last_saved_state = state
    return state

  def send_weights(self):
    """learners.py:84-85 / actors.py:81-85: learner -> self-play weight hand-off; rank 0's weights
    win when several ranks run (each rank's search network is refreshed from the broadcast)."""
    weights = {k: v.detach() for k, v in self.network.state_dict().items()}
    parallel.broadcast_weights(weights, src=0)
    if self.search_network is not None:
      self.search_network.load_weights(weights)
    return weights

  # -- one step (learners.py:164-230) ------------------------------------------------------------
  def _dev(self, x, dtype):
    if isinstance(x, torch.Tensor):
      return x.to(self.device, dtype).contiguous()
    return torch.as_tensor(x, dtype=dtype).to(self.device).contiguous()

  def _forward_backward(self, observations, actions, target_values, target_rewards, target_policies, is_weights):
    if self.batched_heads and hasattr(self.network, 'unroll'):
      values, rewards, policies = self.network.unroll(observations, actions)
      losses, new_errors = self.loss_fn(self.config, values, rewards, policies, target_values, target_rewards,
                                        target_policies, is_weights)
      losses.sum().backward()
      return losses.detach(), new_errors.detach()
    out = self.network.initial_inference(observations)
    values, rewards, policies = [out.value], [], [out.policy_logits]
    hidden_state = out.hidden_state
    for i in range(actions.shape[1]):
      out = self.network.recurrent_inference(hidden_state, actions[:, i])
      hidden_state = out.hidden_state
      hidden_state.register_hook(lambda grad: grad * 0.5)
      values.append(out.value)
      rewards.append(out.reward)
      policies.append(out.policy_logits)
    losses, new_errors = self.loss_fn(self.config, values, rewards, policies, target_values, target_rewards,
                                      target_policies, is_weights)
    full_weighted_loss = losses.sum()  # the 1/K hook of learners.py:213 lives inside the loss
    full_weighted_loss.backward()
    return losses.detach(), new_errors.detach()

  def _apply_gradients(self):
    if getattr(self.config, 'clip_grad', 0):
      torch.nn.utils.clip_grad_norm_(self.network.parameters(), self.config.clip_grad)
    self.optimizer.step()

  def update_weights(self, batch):
    batch, idxs, is_weights = batch
    observations, actions, targets = batch
    target_rewards, target_values, target_policies = targets

    observations = self._dev(observations, torch.float32)
    if getattr(self.config, 'norm_obs', False):
      observations = (observations - self.obs_min) / self.obs_range
    inputs = (observations, self._dev(actions, torch.int64), self._dev(target_values, torch.float32),
              self._dev(target_rewards, torch.float32), self._dev(target_policies, torch.float32),
              self._dev(is_weights, torch.float64))

    if not self.use_graph or self._graphs is None and not self._warm:
      # eager step (always the first one: it creates the optimiser state the graphs reuse)
      self.optimizer.zero_grad(set_to_none=self.use_graph)
      losses, new_errors = self._forward_backward(*inputs)
      self._feed_back(idxs, new_errors)
      parallel.allreduce_gradients(list(self.network.parameters()), average=True)
      self._apply_gradients()
      self._warm = True
    else:
      if self._graphs is None or any(a.shape != b.shape for a, b in zip(self._static, inputs)):
        self._capture(inputs)
      for dst, src in zip(self._static, inputs):
        dst.copy_(src, non_blocking=True)
      fwd_bwd, apply = self._graphs
      fwd_bwd.replay()
      losses, new_errors = self._static_out
      self._feed_back(idxs, new_errors)
      parallel.allreduce_gradients(list(self.network.parameters()), average=True)
      if apply is not None:
        apply.replay()
      else:
        self._apply_gradients()
    if self.lr_scheduler is not None:
      self.lr_scheduler.step()
    self.last_losses, self.last_errors = losses, new_errors
    return self.last_losses

  _warm = False

  def _feed_back(self, idxs, new_errors):
    if self.replay_buffer is not None:  # learners.py:182-184
      if torch.is_tensor(idxs) and idxs.is_cuda:  # a device-resident batch: nothing crosses to the host
        self.replay_buffer.update(idxs, new_errors)
      else:
        self.replay_buffer.update(idxs, new_errors.cpu().numpy())

  def _capture(self, inputs):
    """Captures the step for this batch shape.  Gradients are released first so that the captured
    backward allocates them inside the graph's pool: every replay rewrites the same .grad storage,
    which the (captured or eager) optimiser step then reads."""
    self._static = tuple(torch.empty_like(t).copy_(t) for t in inputs)
    self.optimizer.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    fwd_bwd = torch.cuda.CUDAGraph()
    with torch.cuda.graph(fwd_bwd):
      self._static_out = self._forward_backward(*self._static)
    apply = None
    if self._graph_opt:
      apply = torch.cuda.CUDAGraph()
      with torch.cuda.graph(apply, pool=fwd_bwd.pool()):
        self._apply_gradients()
    self._graphs = (fwd_bwd, apply)

  def log_losses(self):
    """Host read of the last step's losses into the running sums (learners.py:226-228); kept out of
    update_weights so the step itself never synchronises."""
    r, v, p = self.last_losses.cpu().tolist()
    self.losses_to_log['reward'] += r
    self.losses_to_log['value'] += v
    self.losses_to_log['policy'] += p
    return r, v, p

  def learn(self, training_steps=None):
    """The loop of learners.py:116-148 for `training_steps` steps (default config.training_steps)."""
    steps = self.config.training_steps if training_steps is None else training_steps
    self.send_weights()
    # learners.py:119-120: training starts once the replay buffer holds `stored_before_train` memories.  The
    # reference polls a buffer that actor processes fill concurrently; here the caller fills it (or runs the
    # self-play driver between calls), so an under-filled buffer is an error, not a wait that cannot end
    need = int(getattr(self.config, 'stored_before_train', 0) or 0)
    if self.replay_buffer.size() < need:
      raise RuntimeError("replay buffer holds %d memories, config.stored_before_train is %d" %
                         (self.replay_buffer.size(), need))
    save_every = int(getattr(self.config, 'save_state_frequency', 0) or 0)
    end = self.training_step + steps
    while self.training_step < end:
      self.update_weights(self.replay_buffer.sample_batch())
      self.training_step += 1
      if self.training_step % self.config.send_weights_frequency == 0:
        self.send_weights()
      if save_every and self.training_step % save_every == 0:  # learners.py:135-136
        saves = (getattr(self, 'dirs', None) or {}).get('saves')
        self.save_state(os.path.join(saves, str(self.training_step)) if saves else None)
    return self.training_step
