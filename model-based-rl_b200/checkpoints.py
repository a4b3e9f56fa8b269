"""The two optimiser-state forms of an FCNetwork checkpoint and the exact mapping between them.

`learners.Learner.save_state` writes the reference's form (learners.py:72-83): a torch optimiser state_dict over the 22
parameters of `learners.FCNetworkTrain`, one state dict per parameter, keyed by its position in `parameters()` (heads in
the order representation, value, policy, reward, transition, LN).  `fused_learner.FusedLearner.save_state` keeps every
parameter in ONE flat float32 buffer (heads in the order value, policy, reward, transition, representation, LN, every
tensor padded to a multiple of four floats) and writes

  * Adam / AdamW (the library's `mz_adam_step`): {'exp_avg', 'exp_avg_sq': [n], 'state': [step, lr, scratch]};
  * SGD / RMSprop: the torch optimiser's state_dict over the single flat parameter, every tensor of length n.

`module_to_flat` and `flat_to_module` convert the 'optimizer' entry of one into the other by parameter NAME (the names of
FCNetworkTrain.named_parameters(), the offsets of `flat_layout`, which FusedFCNetwork allocates from), so a run moves
between the learners with its optimiser state.  Tensors are copied, never computed: a round trip gives back the same
bits.  The converted state keeps the step counter on the host and the learning rate as a Python float (capturable
False); the learner that loads it moves them to where its own step needs them.
"""
import numpy as np
import torch

from . import _lib, learners
from .networks import HIDDEN

WIDTH = _lib.FC_WIDTH
pad4 = lambda m: (m + 3) & ~3  # every tensor of the flat buffers starts on a 16-byte boundary


# ------------------------------------------------------------------------------------------------
# the two layouts
# ------------------------------------------------------------------------------------------------
def fc_heads(input_dim, action_space, config):
  """(head, output layer, d_in, d_out) of FCNetwork's five heads in flat-buffer order: value, policy, reward (the
  gradient bucket that is complete first), transition, representation."""
  vmin, vmax = [int(v) for v in config.value_support]
  rmin, rmax = [int(v) for v in config.reward_support]
  no_support = bool(getattr(config, 'no_support', False))  # networks.py:135-136: one-unit scalar heads
  A = int(action_space)
  return [('value_head', 'value', HIDDEN, 1 if no_support else vmax - vmin + 1),
          ('policy_head', 'policy', HIDDEN, A),
          ('reward_head', 'reward', HIDDEN + A, 1 if no_support else rmax - rmin + 1),
          ('transition_head', 'out', HIDDEN + A, HIDDEN),
          ('representation_head', 'out', int(input_dim), HIDDEN)]


def head_params(name, out_name, d_in, d_out):
  """(key, shape) of one head's four tensors, with the reference's state-dict keys."""
  return [("%s.fc1.weight" % name, (WIDTH, d_in)), ("%s.fc1.bias" % name, (WIDTH,)),
          ("%s.%s.weight" % (name, out_name), (d_out, WIDTH)), ("%s.%s.bias" % (name, out_name), (d_out,))]


def flat_layout(input_dim, action_space, config):
  """[(key, shape, offset)] of FusedFCNetwork's flat buffer in buffer order, and the buffer's length in floats.  The
  floats between one tensor's end and the next offset are padding: zero in parameters, gradients and optimiser state."""
  specs = [p for h in fc_heads(input_dim, action_space, config) for p in head_params(*h)]
  specs += [('LN.weight', (HIDDEN,)), ('LN.bias', (HIDDEN,))]
  layout, off = [], 0
  for key, shape in specs:
    layout.append((key, shape, off))
    off += pad4(int(np.prod(shape)))
  return layout, off


def module_params(input_dim, action_space, config):
  """[(name, shape)] of FCNetworkTrain.named_parameters(): the order of a module-form optimiser state."""
  with torch.device('meta'):
    net = learners.FCNetworkTrain(input_dim, action_space, 'meta', config)
  return [(name, tuple(p.shape)) for name, p in net.named_parameters()]


def is_module_form(opt, input_dim, action_space, config):
  """A torch optimiser state_dict over FCNetworkTrain's parameters (what learners.Learner saves)."""
  return (isinstance(opt, dict) and 'param_groups' in opt and len(opt['param_groups']) == 1 and
          len(opt['param_groups'][0]['params']) == len(module_params(input_dim, action_space, config)))


def is_flat_form(opt):
  """The library's Adam state or a torch optimiser state_dict over one parameter (what FusedLearner saves)."""
  if not isinstance(opt, dict):
    return False
  return 'exp_avg' in opt or ('param_groups' in opt and len(opt['param_groups']) == 1 and
                              len(opt['param_groups'][0]['params']) == 1)


# ------------------------------------------------------------------------------------------------
# per-parameter entries of the library's optimisers
# ------------------------------------------------------------------------------------------------
def _own(config):
  return config.optimizer in ('Adam', 'AdamW')


def _entries(config):
  """(required, allowed) per-parameter tensor entries besides 'step', and whether there is a 'step'."""
  name, momentum = config.optimizer, float(getattr(config, 'momentum', 0) or 0)
  if name in ('Adam', 'AdamW'):
    return {'exp_avg', 'exp_avg_sq'}, {'exp_avg', 'exp_avg_sq'}, True
  if name == 'RMSprop':
    need = {'square_avg'} | ({'momentum_buffer'} if momentum else set())
    return need, need, True
  if name == 'SGD':  # torch creates the momentum buffer on the first step, and only with momentum
    return set(), ({'momentum_buffer'} if momentum else set()), False
  raise NotImplementedError(name)


def _check_entries(where, st, config):
  need, allowed, has_step = _entries(config)
  keys = set(st) - {'step'}
  if keys - allowed:
    raise ValueError("%s holds optimiser state %s, which %s never creates" % (where, sorted(keys - allowed), config.optimizer))
  if need - keys:
    raise ValueError("%s lacks optimiser state %s of %s" % (where, sorted(need - keys), config.optimizer))
  if has_step != ('step' in st):
    raise ValueError("%s %s a step counter, %s %s one" % (where, 'holds' if 'step' in st else 'lacks', config.optimizer,
                                                          'keeps' if has_step else 'has no'))


def _host_step(step):
  return step.detach().to('cpu', copy=True) if torch.is_tensor(step) else torch.tensor(float(step), dtype=torch.float32)


def _group(group, n_params):
  """The param group with a plain learning rate, host-side step counters and n_params parameters."""
  g = dict(group, params=list(range(n_params)))
  g['lr'] = float(g['lr'])
  if 'capturable' in g:
    g['capturable'] = False
  if torch.is_tensor(g.get('initial_lr')):
    g['initial_lr'] = float(g['initial_lr'])
  return g


# ------------------------------------------------------------------------------------------------
# the mapping
# ------------------------------------------------------------------------------------------------
def module_to_flat(opt, config, input_dim, action_space):
  """learners.Learner's 'optimizer' entry -> FusedLearner's for config.optimizer.  Raises ValueError (naming the key)
  for a state of another geometry, an entry the library's optimisers never create, or per-parameter step counters
  that differ."""
  params = module_params(input_dim, action_space, config)
  layout, n = flat_layout(input_dim, action_space, config)
  offset = {key: off for key, _, off in layout}
  if not is_module_form(opt, input_dim, action_space, config):
    raise ValueError("the optimiser state is not a torch state_dict over the %d FCNetwork parameters" % len(params))
  group, state = opt['param_groups'][0], opt['state']
  index = {p: i for i, p in enumerate(group['params'])}
  per_param = {}
  for p, st in state.items():
    if p not in index:
      raise ValueError("optimiser state of parameter %r, which the param group does not list" % (p,))
    name, shape = params[index[p]]
    _check_entries("optimiser state of %s" % name, st, config)
    for k, v in st.items():
      if k != 'step' and tuple(v.shape) != shape:
        raise ValueError("optimiser state %s of %s has shape %s, expected %s" % (k, name, tuple(v.shape), shape))
    per_param[name] = st
  if per_param and len(per_param) != len(params):
    raise ValueError("optimiser state for %d of the %d FCNetwork parameters" % (len(per_param), len(params)))
  steps = {float(st['step']) for st in per_param.values() if 'step' in st}
  if len(steps) > 1:
    raise ValueError("the parameters' step counters differ (%s): the flat buffer keeps one" % sorted(steps))
  flat = {}
  for name, shape in params:
    for k, v in per_param.get(name, {}).items():
      if k != 'step':
        dst = flat.setdefault(k, torch.zeros(n, dtype=v.dtype))
        dst[offset[name]:offset[name] + v.numel()] = v.detach().reshape(-1).cpu()
  if _own(config):
    for k in ('exp_avg', 'exp_avg_sq'):
      flat.setdefault(k, torch.zeros(n, dtype=torch.float32))
    # state[2] is the clipping kernel's scratch, cleared before every read: 0, as in a fresh learner
    step = steps.pop() if steps else 0.0
    flat['state'] = torch.tensor([step, float(group['lr']), 0.0], dtype=torch.float32)
    return flat
  out = {'state': {}, 'param_groups': [_group(group, 1)]}
  if per_param:
    st = dict(flat)
    if 'step' in next(iter(per_param.values())):
      st['step'] = _host_step(per_param[params[0][0]]['step'])
    out['state'][0] = st
  return out


def flat_to_module(opt, config, input_dim, action_space):
  """FusedLearner's 'optimizer' entry -> learners.Learner's (a torch state_dict over FCNetworkTrain's parameters) for
  config.optimizer.  Raises ValueError for state of another optimiser kind or flat length, or an entry the library's
  optimisers never create."""
  params = module_params(input_dim, action_space, config)
  layout, n = flat_layout(input_dim, action_space, config)
  offset = {key: off for key, _, off in layout}
  own = isinstance(opt, dict) and 'exp_avg' in opt
  if own != _own(config) or not is_flat_form(opt):
    raise ValueError("the optimiser state is not FusedLearner's %s state" % config.optimizer)
  if own:
    if set(opt) != {'exp_avg', 'exp_avg_sq', 'state'} or opt['state'].numel() != 3:
      raise ValueError("the library's Adam state is {'exp_avg', 'exp_avg_sq', 'state' = [step, lr, scratch]}, got %s"
                       % sorted(opt))
    st = {'exp_avg': opt['exp_avg'], 'exp_avg_sq': opt['exp_avg_sq'], 'step': opt['state'][0]}
    group = learners.get_optimizer(config, [torch.zeros(1, requires_grad=True)]).state_dict()['param_groups'][0]
    group['lr'] = float(opt['state'][1])
    if getattr(config, 'lr_scheduler', None) == 'ExponentialLR':
      group['initial_lr'] = float(config.lr_init)  # what torch's ExponentialLR sets when it is built
  else:
    if len(opt['state']) > 1 or (opt['state'] and 0 not in opt['state']):
      raise ValueError("a flat optimiser state_dict holds the state of one parameter, got %s" % sorted(opt['state']))
    st, group = opt['state'].get(0, {}), opt['param_groups'][0]
  if st:
    _check_entries("the flat optimiser state", st, config)
  for k, v in st.items():
    if k != 'step' and v.numel() != n:
      raise ValueError("optimiser state %s has %d elements, the flat buffer of this network %d" % (k, v.numel(), n))
  state = {}
  if st:
    for i, (name, shape) in enumerate(params):
      m = int(np.prod(shape))
      state[i] = {k: (_host_step(v) if k == 'step' else
                      v.detach().reshape(-1)[offset[name]:offset[name] + m].cpu().clone().view(shape))
                  for k, v in st.items()}
  return {'state': state, 'param_groups': [_group(group, len(params))]}
