"""torch (CPU, float32) restatement of the reference's FCNetwork inference -- TEST INFRASTRUCTURE /
CPU BASELINE only.  Same layer shapes and state-dict keys as networks.py:55-174, eval-mode outputs
(scalars after Config.inverse_transform, config.py:27-33).  Pinned against golden outputs of the
unmodified reference module in tests/test_oracle_golden.py and tests/test_gpu_fcnet_shapes.py.

The module evaluates in the dtype of its parameters: `FCNetworkRef(...).double()` with float64 inputs is
the float64 reference the kernel tests measure errors against.  `TcEmulation` evaluates the same network
with the bf16 rounding points of the tensor-core kernels (csrc/mz_fcnet_tc.cu)."""
from collections import namedtuple

import torch
import torch.nn as nn
import torch.nn.functional as F

NetworkOutput = namedtuple('network_output', ('value', 'reward', 'policy_logits', 'hidden_state'))

HIDDEN, WIDTH = 50, 512


class _Head(nn.Module):
  """Linear(d_in, 512) + ReLU + Linear(512, d_out); the second layer's attribute name varies."""

  def __init__(self, d_in, d_out, out_name):
    super().__init__()
    self.fc1 = nn.Linear(d_in, WIDTH)
    setattr(self, out_name, nn.Linear(WIDTH, d_out))
    self._out_name = out_name

  def forward(self, x):
    return getattr(self, self._out_name)(F.relu(self.fc1(x)))


def support_to_scalar(logits, support_min, support_max, no_target_transform=False):
  p = torch.softmax(logits, dim=1)
  support = torch.arange(support_min, support_max + 1, dtype=logits.dtype).expand(p.shape)
  v = torch.sum(support * p, dim=1, keepdim=True)
  if not no_target_transform:
    v = torch.sign(v) * (((torch.sqrt(1 + 4 * 0.001 * (torch.abs(v) + 1 + 0.001)) - 1) / (2 * 0.001)) ** 2 - 1)
  return v


class FCNetworkRef(nn.Module):

  def __init__(self, input_dim, action_space, value_support=(-15, 15), reward_support=(-15, 15),
               no_target_transform=False, no_support=False):
    """no_support: one-unit value / reward heads whose raw outputs are the scalars (networks.py:135-136,
    153, 161)."""
    super().__init__()
    self.action_space = action_space
    self.vs, self.rs, self.no_tt = tuple(value_support), tuple(reward_support), no_target_transform
    self.no_support = no_support
    self.representation_head = _Head(input_dim, HIDDEN, 'out')
    self.value_head = _Head(HIDDEN, 1 if no_support else self.vs[1] - self.vs[0] + 1, 'value')
    self.policy_head = _Head(HIDDEN, action_space, 'policy')
    self.reward_head = _Head(HIDDEN + action_space, 1 if no_support else self.rs[1] - self.rs[0] + 1, 'reward')
    self.transition_head = _Head(HIDDEN + action_space, HIDDEN, 'out')
    self.LN = nn.LayerNorm([HIDDEN])
    self.eval()

  def _predict(self, h):
    value = self.value_head(h)
    if not self.training and not self.no_support:  # train mode keeps the support logits (networks.py:151-154)
      value = support_to_scalar(value, *self.vs, self.no_tt)
    return self.policy_head(h), value

  def initial_inference(self, observation):
    h = F.relu(self.LN(self.representation_head(observation.reshape(observation.shape[0], -1))))
    logits, value = self._predict(h)
    return NetworkOutput(value, 0, logits, h)

  def _attach_action(self, hidden_state, action):
    a = torch.as_tensor(action, dtype=torch.int64).reshape(-1, 1)
    onehot = torch.zeros((a.shape[0], self.action_space), dtype=torch.float32).scatter_(1, a, 1.0)
    return torch.cat((hidden_state, onehot), dim=1)

  def recurrent_inference(self, hidden_state, action):
    x = self._attach_action(hidden_state, action)
    reward = self.reward_head(x)
    if not self.training and not self.no_support:
      reward = support_to_scalar(reward, *self.rs, self.no_tt)
    h = F.relu(self.LN(self.transition_head(x)))
    logits, value = self._predict(h)
    return NetworkOutput(value, reward, logits, h)


def bf16_round(x):
  """x rounded to the nearest bfloat16 (ties to even), in x's dtype."""
  return x.to(torch.bfloat16).to(x.dtype)


class TcEmulation(object):
  """The network of an FCNetworkRef evaluated in its parameters' dtype (float64 after `.double()`), with
  values rounded to bf16 exactly where the tensor-core kernels round them (fc_tc_pack_kernel and the
  epilogues of csrc/mz_fcnet_tc.cu):

  - the first-layer A operand of every head: [h | onehot(a) | 1] (reward, transition), [obs | 1]
    (representation) or [h' | 1] (value, policy), where the constant-1 column feeds the first-layer bias;
  - the first-layer weights W1 with the bias b1 folded in as the weight row of that constant column;
  - the ReLU output of the first layer (the A operand of the second layer);
  - the second-layer weights W2.  The second-layer bias b2 is added unrounded (float32 in the kernel);
  - nothing else: LayerNorm + ReLU and softmax-expectation + h^-1 take the unrounded values, and the
    hidden state the kernels return is h' before its bf16 rounding (only the prediction heads read the
    rounded copy).

  The kernels accumulate in float32, the emulation in the parameters' dtype.  With bf16=False every
  rounding is the identity and the evaluation is the reference module's own, restated with the bias folding.
  """

  def __init__(self, net, bf16=True):
    self.net = net
    self.round = bf16_round if bf16 else (lambda x: x)

  def _head(self, head, x):
    r = self.round
    fc1, fc2 = head.fc1, getattr(head, head._out_name)
    a = r(torch.cat((x, torch.ones((x.shape[0], 1), dtype=x.dtype)), dim=1))
    w1 = r(torch.cat((fc1.weight, fc1.bias[:, None]), dim=1))
    return r(F.relu(a @ w1.t())) @ r(fc2.weight).t() + fc2.bias

  def _predict(self, h):
    net = self.net
    value = self._head(net.value_head, h)
    if not net.no_support:
      value = support_to_scalar(value, *net.vs, net.no_tt)
    return self._head(net.policy_head, h), value

  def _state(self, x):
    return F.relu(self.net.LN(x))

  def initial_inference(self, observation):
    net = self.net
    with torch.no_grad():
      h = self._state(self._head(net.representation_head, observation.reshape(observation.shape[0], -1)))
      logits, value = self._predict(h)
    return NetworkOutput(value, 0, logits, h)

  def recurrent_inference(self, hidden_state, action):
    net = self.net
    with torch.no_grad():
      x = net._attach_action(hidden_state, action).to(hidden_state.dtype)
      reward = self._head(net.reward_head, x)
      if not net.no_support:
        reward = support_to_scalar(reward, *net.rs, net.no_tt)
      h = self._state(self._head(net.transition_head, x))
      logits, value = self._predict(h)
    return NetworkOutput(value, reward, logits, h)


def random_state_dict(input_dim, action_space, seed=1234):
  """Random-init weights of the FCNetwork architecture with the reference's keys (torch default
  nn.Linear / LayerNorm initialisation)."""
  g = torch.random.get_rng_state()
  torch.manual_seed(seed)
  net = FCNetworkRef(input_dim, action_space)
  torch.random.set_rng_state(g)
  return {k: v.detach().clone() for k, v in net.state_dict().items()}
