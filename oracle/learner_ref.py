"""torch (CPU) restatement of the reference's learner step -- TEST INFRASTRUCTURE only.

Follows Learner.update_weights (learners.py:164-230) with the loss closures of
utils.get_loss_functions (utils.py:53-56) and the transforms of config.py:51-68, on the oracle's
FCNetworkRef in train mode.  Pinned against tests/golden/learner_*.npz, which were produced by the
reference's own FCNetwork / Config around the same lines (tests/golden/make_golden.py gen_learner).
"""
import torch


def scalar_transform(x):
  """config.py:51-54"""
  return torch.sign(x) * (torch.sqrt(torch.abs(x) + 1) - 1) + 0.001 * x


def scalar_to_support(x, mn, mx):
  """config.py:56-68 (clamp, p_high at ceil, then p_low at floor).  The support has x's dtype and device, so that
  float64 targets give a float64 reference."""
  x = x.clamp(mn, mx)
  floor, ceil = x.floor(), x.ceil()
  p_high = x - floor
  p_low = 1 - p_high
  support = torch.zeros(x.shape[0], x.shape[1], mx - mn + 1, dtype=x.dtype, device=x.device)
  support.scatter_(2, (ceil - mn).long().unsqueeze(-1), p_high.unsqueeze(-1))
  support.scatter_(2, (floor - mn).long().unsqueeze(-1), p_low.unsqueeze(-1))
  return support


def cross_entropy(logits, target):
  """utils.py:54-55"""
  return (-target * torch.nn.LogSoftmax(dim=1)(logits)).sum(1)


def unroll_loss_ref(config, values, rewards, policies, t_values, t_rewards, t_policies, is_weights):
  """Same signature as model_based_rl_b200.learners.unroll_loss: (losses[3] float64 = reward, value,
  policy; new_errors[B]).  The 1/K gradient hook of learners.py:213 is folded into the returned
  losses' gradient the same way the CUDA loss does (losses.sum().backward() gives the reference's
  gradients)."""
  from .fcnet_ref import support_to_scalar
  vmin, vmax = [int(v) for v in config.value_support]
  rmin, rmax = [int(v) for v in config.reward_support]
  no_tt = bool(getattr(config, 'no_target_transform', False))
  K = len(rewards)  # lists of per-step logits or stacked [steps, B, bins] tensors
  with torch.no_grad():
    init_value = support_to_scalar(values[0], vmin, vmax, no_tt)
    new_errors = init_value.squeeze(1) - t_values[:, 0]
    if not no_tt:
      t_values, t_rewards = scalar_transform(t_values), scalar_transform(t_rewards)
    t_values = scalar_to_support(t_values, vmin, vmax)
    t_rewards = scalar_to_support(t_rewards, rmin, rmax)
  reward_loss = 0
  value_loss = cross_entropy(values[0], t_values[:, 0])
  policy_loss = cross_entropy(policies[0], t_policies[:, 0])
  for i in range(1, K + 1):
    reward_loss = reward_loss + cross_entropy(rewards[i - 1], t_rewards[:, i])
    value_loss = value_loss + cross_entropy(values[i], t_values[:, i])
    policy_loss = policy_loss + cross_entropy(policies[i], t_policies[:, i])
  losses = torch.stack([(is_weights * reward_loss).mean(), (is_weights * value_loss).mean(),
                        (is_weights * policy_loss).mean()])
  losses.register_hook(lambda grad: grad * (1 / K))
  return losses, new_errors
