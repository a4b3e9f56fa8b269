"""Checkpoints across the two FCNetwork learners: a run saved by learners.Learner (per-parameter torch optimiser state)
resumes on fused_learner.FusedLearner (optimiser state over one flat buffer) and the reverse.

CPU part: the mapping of checkpoints.py -- exact round trips in both directions for every optimiser, head kind, action
count and observation width the fused learner takes, the flat offsets and padding, its refusals -- and
learners.Learner resuming from flat optimiser state on the CPU (the oracle's torch loss stands in for the CUDA kernel).
GPU part: a resumed learner of the other kind continues the run at the bars of the FusedLearner-vs-Learner step
comparisons, where the same weights with a fresh optimiser visibly do not."""
import types

import numpy as np
import pytest
import torch

import helpers
from oracle import learner_ref

BAR = 2e-5  # one step of FusedLearner(precision='f32') against learners.Learner from the same weights and state


# -- config and batch helpers of tests/test_learner.py and tests/test_fused_learner_checkpoint.py ---------------------
def _config(g):
  return types.SimpleNamespace(
      value_support=[-15, 15], reward_support=[-15, 15], no_support=False,
      no_target_transform=bool(g["no_target_transform"]), num_unroll_steps=int(g["K"]),
      optimizer=str(g["optimizer"]), lr_init=float(g["lr"]), momentum=float(g["momentum"]),
      weight_decay=float(g["weight_decay"]), clip_grad=int(g["clip_grad"]), lr_scheduler=None,
      norm_obs=False, send_weights_frequency=500, training_steps=2)


def _batch(g, step):
  s = "s%d_" % step
  actions = [list(map(int, row)) for row in g[s + "actions"]]
  return ((g[s + "obs"], actions, (g[s + "t_rewards"].copy(), g[s + "t_values"].copy(), g[s + "t_policies"].copy())),
          None, g[s + "is_weights"])


def _weights(g, prefix="w0_"):
  return {k[len(prefix):]: torch.from_numpy(v.copy()) for k, v in g.items() if k.startswith(prefix)}


def _cfg(case, optimizer):
  g = helpers.load("learner_" + case)
  cfg = _config(g)
  if "scalar_loss" in g:
    cfg.no_support, cfg.scalar_loss = True, str(g["scalar_loss"])
  cfg.optimizer = optimizer
  return g, cfg


# -- runs: golden cases, and synthetic ones at 64 actions / 512 features -------------------------------------------------
SYNTHETIC = {"a64": (24, 64), "d512": (512, 18)}  # (input_dim, action_space)


def _case(case, optimizer, scheduler=None):
  """(config, input_dim, action_space, initial weights, the two batches of the run)."""
  if case in SYNTHETIC:
    D, A = SYNTHETIC[case]
    B, K = 48, 3
    cfg = types.SimpleNamespace(
        value_support=[-15, 15], reward_support=[-15, 15], no_support=False, no_target_transform=False,
        num_unroll_steps=K, optimizer=optimizer, lr_init=0.0008, momentum=0.9, weight_decay=1e-4, clip_grad=0,
        lr_scheduler=None, norm_obs=False, send_weights_frequency=500, training_steps=2)
    rng = np.random.default_rng(D + A)
    batches = []
    for _ in range(2):
      batches.append(((rng.normal(size=(B, D)).astype(np.float32), rng.integers(0, A, size=(B, K)).tolist(),
                       (rng.normal(size=(B, K + 1)).astype(np.float32),
                        rng.normal(scale=3.0, size=(B, K + 1)).astype(np.float32),
                        rng.dirichlet([0.3] * A, size=(B, K + 1)).astype(np.float32))), None, rng.uniform(0.5, 1.0, size=B)))
    from model_based_rl_b200 import learners
    torch.manual_seed(D + A)
    weights = learners.FCNetworkTrain(D, A, "cpu", cfg).get_weights()
  else:
    g, cfg = _cfg(case, optimizer)
    D, A = int(g["obs_dim"]), int(g["action_space"])
    weights, batches = _weights(g), [_batch(g, 0), _batch(g, 1)]
  cfg.lr_scheduler, cfg.lr_decay_rate, cfg.lr_decay_steps = scheduler, 0.9, 3
  return cfg, D, A, weights, batches


def _torch_learner(cfg, D, A, weights, graph=False, state=None, device="cuda", loss_fn=None):
  from model_based_rl_b200 import learners
  net = learners.FCNetworkTrain(D, A, device, cfg)
  net.load_weights(weights)
  return learners.Learner(cfg, net, use_graph=graph, state=state, loss_fn=loss_fn)


def _fused_learner(cfg, D, A, weights, graph=False, state=None, precision="f32"):
  from model_based_rl_b200 import fused_learner
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  net.load_weights(weights)
  return fused_learner.FusedLearner(cfg, net, use_graph=graph, precision=precision, state=state)


def _flat_weights(learner):
  """Every weight of either learner in FCNetworkTrain's parameter order, on the host."""
  sd = learner.network.state_dict()
  return torch.cat([sd[k].detach().reshape(-1).cpu() for k in sorted(sd)])


def _lr(learner):
  if getattr(learner, "own_optimizer", False):
    return float(learner.opt_state[1])
  return float(learner.optimizer.param_groups[0]["lr"])


def _opt_tensors(learner):
  if getattr(learner, "own_optimizer", False):
    return {"exp_avg": learner.exp_avg, "exp_avg_sq": learner.exp_avg_sq, "state": learner.opt_state}
  return {"%s.%s" % (i, k): v for i, st in enumerate(learner.optimizer.state.values()) for k, v in st.items()
          if torch.is_tensor(v)}


def _snapshot(learner):
  out = {"weights": _flat_weights(learner)}
  out.update({k: v.detach().cpu().clone() for k, v in _opt_tensors(learner).items()})
  return out


def _assert_untouched(learner, before):
  after = _snapshot(learner)
  assert sorted(after) == sorted(before)
  for k in before:
    assert torch.equal(after[k], before[k]), k


# ======================================================================================================================
# CPU: the mapping
# ======================================================================================================================
def _ns(D, A, optimizer, no_support=False, momentum=0.9):
  return types.SimpleNamespace(value_support=[-15, 15], reward_support=[-10, 12], no_support=no_support,
                               optimizer=optimizer, lr_init=0.003, momentum=momentum, weight_decay=1e-4,
                               lr_scheduler=None)


def _pad4(m):
  return (m + 3) // 4 * 4


def _reference_offsets(D, A, cfg):
  """FusedFCNetwork's buffer order restated: heads value, policy, reward, transition, representation, then LN; every
  tensor padded to a multiple of four floats."""
  V = 1 if cfg.no_support else cfg.value_support[1] - cfg.value_support[0] + 1
  R = 1 if cfg.no_support else cfg.reward_support[1] - cfg.reward_support[0] + 1
  heads = [("value_head", "value", 50, V), ("policy_head", "policy", 50, A), ("reward_head", "reward", 50 + A, R),
           ("transition_head", "out", 50 + A, 50), ("representation_head", "out", D, 50)]
  out, off = {}, 0
  for name, o, d_in, d_out in heads:
    for key, m in (("fc1.weight", 512 * d_in), ("fc1.bias", 512), ("%s.weight" % o, d_out * 512), ("%s.bias" % o, d_out)):
      out["%s.%s" % (name, key)] = (off, m)
      off += _pad4(m)
  for key in ("LN.weight", "LN.bias"):
    out[key] = (off, 50)
    off += _pad4(50)
  return out, off


def _module_state(cfg, D, A, seed=0, fill=None):
  """A torch optimiser state_dict over FCNetworkTrain's parameters as learners.Learner saves it after a step, every
  state tensor replaced: distinct random values, or fill(index of the parameter)."""
  from model_based_rl_b200 import learners
  net = learners.FCNetworkTrain(D, A, "cpu", cfg)
  opt = learners.get_optimizer(cfg, net.parameters())
  for p in net.parameters():
    p.grad = torch.ones_like(p)
  opt.step()
  sd = opt.state_dict()
  gen = torch.Generator().manual_seed(seed)
  state = {}
  for i, st in sd["state"].items():
    state[i] = {k: (v.clone() if k == "step" else
                    torch.full_like(v, float(fill(i))) if fill else torch.randn(v.shape, generator=gen))
                for k, v in st.items()}
    if "step" in st:
      state[i]["step"] = torch.tensor(7.0)
  return {"state": state, "param_groups": sd["param_groups"]}


def _flat_state(cfg, D, A, seed=0):
  """FusedLearner's optimiser entry with distinct random values in every state tensor and zero padding."""
  from model_based_rl_b200 import learners
  offsets, n = _reference_offsets(D, A, cfg)
  gen = torch.Generator().manual_seed(seed)

  def rand():
    t = torch.zeros(n)
    for off, m in offsets.values():
      t[off:off + m] = torch.randn(m, generator=gen)
    return t
  if cfg.optimizer in ("Adam", "AdamW"):
    return {"exp_avg": rand(), "exp_avg_sq": rand(), "state": torch.tensor([5.0, 0.0021, 0.0])}
  flat = torch.zeros(n, requires_grad=True)
  opt = learners.get_optimizer(cfg, [flat])
  flat.grad = torch.ones(n)
  opt.step()
  sd = opt.state_dict()
  for st in sd["state"].values():
    for k in list(st):
      st[k] = torch.tensor(5.0) if k == "step" else rand()
  return sd


OPTIMISERS = [("AdamW", 0.9), ("Adam", 0.9), ("RMSprop", 0.9), ("SGD", 0.9), ("SGD", 0.0)]
GEOMETRIES = [(8, 9, False), (128, 18, True), (147, 64, False), (1024, 18, False), (1024, 64, True), (147, 9, True)]


@pytest.mark.parametrize("D,A,no_support", GEOMETRIES, ids=["d%d-a%d-%s" % (d, a, "nosup" if n else "sup") for d, a, n in GEOMETRIES])
@pytest.mark.parametrize("optimizer,momentum", OPTIMISERS, ids=["%s-m%g" % o for o in OPTIMISERS])
def test_round_trips_are_bit_exact(optimizer, momentum, D, A, no_support):
  from model_based_rl_b200 import checkpoints
  cfg = _ns(D, A, optimizer, no_support, momentum)
  # module -> flat -> module
  sd = _module_state(cfg, D, A, seed=D + A)
  flat = checkpoints.module_to_flat(sd, cfg, D, A)
  back = checkpoints.flat_to_module(flat, cfg, D, A)
  assert sorted(back["state"]) == sorted(sd["state"])
  assert len(sd["state"]) == (0 if (optimizer, momentum) == ("SGD", 0.0) else 22)
  for i, st in sd["state"].items():
    assert sorted(back["state"][i]) == sorted(st), i
    for k, v in st.items():
      assert back["state"][i][k].dtype == v.dtype and torch.equal(back["state"][i][k], v), (i, k)
  assert len(back["param_groups"][0]["params"]) == 22
  assert np.float32(back["param_groups"][0]["lr"]) == np.float32(sd["param_groups"][0]["lr"])
  # flat -> module -> flat
  fs = _flat_state(cfg, D, A, seed=D * A)
  again = checkpoints.module_to_flat(checkpoints.flat_to_module(fs, cfg, D, A), cfg, D, A)
  if optimizer in ("Adam", "AdamW"):
    assert sorted(again) == ["exp_avg", "exp_avg_sq", "state"]
    for k in again:
      assert torch.equal(again[k], fs[k]), k
  else:
    assert sorted(again["state"]) == sorted(fs["state"])
    for k, v in fs["state"].get(0, {}).items():
      assert torch.equal(again["state"][0][k], v), k
    assert again["param_groups"][0]["params"] == [0]
    assert again["param_groups"][0]["lr"] == fs["param_groups"][0]["lr"]


@pytest.mark.parametrize("D,A,no_support", GEOMETRIES, ids=["d%d-a%d-%s" % (d, a, "nosup" if n else "sup") for d, a, n in GEOMETRIES])
@pytest.mark.parametrize("optimizer", ["AdamW", "RMSprop"])
def test_each_parameter_lands_at_its_flat_offset_with_zero_padding(optimizer, D, A, no_support):
  """Parameter i's state (written as i + 1) at FusedFCNetwork's offset of its name; every padding float zero."""
  from model_based_rl_b200 import checkpoints, learners
  cfg = _ns(D, A, optimizer, no_support)
  names = [n for n, _ in learners.FCNetworkTrain(D, A, "cpu", cfg).named_parameters()]
  offsets, n = _reference_offsets(D, A, cfg)
  assert sorted(names) == sorted(offsets)
  assert checkpoints.flat_layout(D, A, cfg)[1] == n
  flat = checkpoints.module_to_flat(_module_state(cfg, D, A, fill=lambda i: i + 1), cfg, D, A)
  tensors = [flat["exp_avg"], flat["exp_avg_sq"]] if optimizer == "AdamW" else [flat["state"][0]["square_avg"],
                                                                                 flat["state"][0]["momentum_buffer"]]
  for t in tensors:
    assert t.numel() == n
    covered = torch.zeros(n, dtype=torch.bool)
    for i, name in enumerate(names):
      off, m = offsets[name]
      assert torch.equal(t[off:off + m], torch.full((m,), float(i + 1))), name
      covered[off:off + m] = True
    assert not t[~covered].any()
  if optimizer == "AdamW":
    assert flat["state"].tolist() == [7.0, float(np.float32(0.003)), 0.0]
  else:
    assert float(flat["state"][0]["step"]) == 7.0


def test_unequal_steps_are_refused():
  from model_based_rl_b200 import checkpoints
  for optimizer in ("AdamW", "RMSprop"):
    cfg = _ns(9, 9, optimizer)
    sd = _module_state(cfg, 9, 9)
    sd["state"][3]["step"] = torch.tensor(8.0)
    with pytest.raises(ValueError, match="step"):
      checkpoints.module_to_flat(sd, cfg, 9, 9)


@pytest.mark.parametrize("optimizer,entry", [("AdamW", "max_exp_avg_sq"), ("RMSprop", "grad_avg"),
                                             ("SGD", "square_avg")])
def test_unknown_state_entries_are_refused(optimizer, entry):
  from model_based_rl_b200 import checkpoints
  cfg = _ns(9, 9, optimizer)
  sd = _module_state(cfg, 9, 9)
  sd["state"][5][entry] = torch.zeros_like(sd["state"][5]["momentum_buffer" if optimizer == "SGD" else
                                                          "exp_avg" if optimizer == "AdamW" else "square_avg"])
  with pytest.raises(ValueError, match=entry):
    checkpoints.module_to_flat(sd, cfg, 9, 9)
  fs = _flat_state(cfg, 9, 9)
  if optimizer == "AdamW":
    fs[entry] = torch.zeros_like(fs["exp_avg"])
  else:
    fs["state"][0][entry] = torch.zeros_like(fs["state"][0]["momentum_buffer"])
  with pytest.raises(ValueError, match=entry):
    checkpoints.flat_to_module(fs, cfg, 9, 9)


@pytest.mark.parametrize("other", ["actions", "input_dim", "supports", "no_support"])
def test_state_of_another_geometry_is_refused(other):
  from model_based_rl_b200 import checkpoints
  cfg = _ns(9, 9, "AdamW")
  D, A = (9, 8) if other == "actions" else (10, 9) if other == "input_dim" else (9, 9)
  src = _ns(D, A, "AdamW", no_support=other == "no_support")
  if other == "supports":
    src.value_support = [-10, 10]
  with pytest.raises(ValueError):
    checkpoints.module_to_flat(_module_state(src, D, A), cfg, 9, 9)
  with pytest.raises(ValueError):
    checkpoints.flat_to_module(_flat_state(src, D, A), cfg, 9, 9)


def test_state_of_another_optimiser_kind_is_refused():
  from model_based_rl_b200 import checkpoints
  with pytest.raises(ValueError):
    checkpoints.module_to_flat(_module_state(_ns(9, 9, "RMSprop"), 9, 9), _ns(9, 9, "AdamW"), 9, 9)
  with pytest.raises(ValueError):
    checkpoints.flat_to_module(_flat_state(_ns(9, 9, "AdamW"), 9, 9), _ns(9, 9, "RMSprop"), 9, 9)
  with pytest.raises(ValueError):
    checkpoints.flat_to_module(_flat_state(_ns(9, 9, "RMSprop"), 9, 9), _ns(9, 9, "SGD"), 9, 9)


# ======================================================================================================================
# CPU: learners.Learner resumes from flat optimiser state
# ======================================================================================================================
def _cpu_learner(cfg, D, A, weights, state=None):
  return _torch_learner(cfg, D, A, weights, state=state, device="cpu", loss_fn=learner_ref.unroll_loss_ref)


def _as_fused_checkpoint(state, cfg, D, A):
  from model_based_rl_b200 import checkpoints
  return dict(state, optimizer=checkpoints.module_to_flat(state["optimizer"], cfg, D, A))


@pytest.mark.parametrize("case,optimizer,scheduler", [("ttt", "AdamW", None), ("ttt", "Adam", "ExponentialLR"),
                                                      ("breakout", "RMSprop", None), ("lunar_raw", "SGD", "ExponentialLR")])
def test_cpu_learner_resumes_from_flat_state_bit_exact(case, optimizer, scheduler):
  """Two CPU steps, the checkpoint's optimiser state put into the flat form, a new Learner from it: its third step is
  the uninterrupted learner's, bit for bit; the same weights with a fresh optimiser step elsewhere."""
  cfg, D, A, weights, batches = _case(case, optimizer, scheduler)
  l1 = _cpu_learner(cfg, D, A, weights)
  for b in batches:
    l1.update_weights(b)
  l1.training_step = 2
  state = _as_fused_checkpoint(l1.save_state(), cfg, D, A)
  fresh = {k: v + 1.0 for k, v in weights.items()}
  l2 = _cpu_learner(cfg, D, A, fresh, state=state)
  control = _cpu_learner(cfg, D, A, {k: v.clone() for k, v in l1.network.get_weights().items()})
  assert l2.training_step == 2 and torch.equal(_flat_weights(l2), _flat_weights(l1))
  assert np.float32(_lr(l2)) == np.float32(_lr(l1))
  for learner in (l1, l2, control):
    learner.update_weights(batches[0])
  assert torch.equal(_flat_weights(l2), _flat_weights(l1))
  o1, o2 = _opt_tensors(l1), _opt_tensors(l2)
  assert sorted(o1) == sorted(o2)
  for k in o1:
    assert torch.equal(o1[k], o2[k]), k
  assert float((_flat_weights(control) - _flat_weights(l1)).abs().max()) > 10 * BAR


def test_cpu_learner_refuses_flat_state_it_cannot_take():
  """Another optimiser kind, another geometry, or a network that is not FCNetworkTrain: ValueError, learner untouched."""
  import torch.nn as nn
  from model_based_rl_b200 import learners
  cfg, D, A, weights, batches = _case("ttt", "AdamW")
  learner = _cpu_learner(cfg, D, A, weights)
  learner.update_weights(batches[0])
  before = _snapshot(learner)
  # another optimiser kind
  cfg_r = _case("ttt", "RMSprop")[0]
  src = _cpu_learner(cfg_r, D, A, weights)
  src.update_weights(batches[0])
  with pytest.raises(ValueError, match="FusedLearner"):
    learner.load_state(_as_fused_checkpoint(src.save_state(), cfg_r, D, A))
  _assert_untouched(learner, before)
  # another action count / input width
  for D2, A2 in ((D, A - 1), (D + 3, A)):
    src = _cpu_learner(cfg, D2, A2, learners.FCNetworkTrain(D2, A2, "cpu", cfg).get_weights())
    with pytest.raises(ValueError):
      learner.load_state(_as_fused_checkpoint(src.save_state(), cfg, D2, A2))
    _assert_untouched(learner, before)
  # a network with other parameters
  other = learners.Learner(cfg, nn.Linear(3, 2), loss_fn=learner_ref.unroll_loss_ref)
  with pytest.raises(ValueError, match="FCNetwork parameters"):
    other.load_state(_as_fused_checkpoint(learner.save_state(), cfg, D, A))


# ======================================================================================================================
# GPU: a run continued on the other learner
# ======================================================================================================================
# (case, optimizer, schedule, graph for the saving learner, graph for the resuming learner)
RUNS = [("ttt", "AdamW", None, False, False), ("ttt", "AdamW", "ExponentialLR", True, True),
        ("breakout", "Adam", None, True, False), ("breakout", "RMSprop", "ExponentialLR", False, True),
        ("breakout", "RMSprop", None, True, True), ("lunar_raw", "SGD", None, True, True),
        ("lunar_raw", "SGD", "ExponentialLR", False, True), ("nosupport_mse", "AdamW", None, True, False),
        ("a64", "Adam", "ExponentialLR", False, True), ("d512", "RMSprop", None, True, False)]
RUN_IDS = ["-".join(map(str, r)) for r in RUNS]


def _run_two_steps(make, cfg, D, A, weights, batches, graph, path):
  learner = make(cfg, D, A, weights, graph)
  for b in batches:
    learner.update_weights(b)
  learner.training_step = 2  # what learn() would have counted
  learner.save_state(str(path))
  torch.cuda.synchronize()
  return learner, torch.load(path, weights_only=False)


def _continue(source, resumed, control, batch, bar=BAR, name=""):
  assert torch.equal(_flat_weights(resumed), _flat_weights(source))
  for learner in (source, resumed, control):
    learner.update_weights(batch)
  torch.cuda.synchronize()
  diff = float((_flat_weights(resumed) - _flat_weights(source)).abs().max())
  off = float((_flat_weights(control) - _flat_weights(source)).abs().max())
  print(name, "resumed vs uninterrupted %.3g, fresh optimiser vs uninterrupted %.3g" % (diff, off))
  assert diff <= bar, diff
  assert off > 10 * bar, off


@pytest.mark.gpu
@pytest.mark.parametrize("run", RUNS, ids=RUN_IDS)
def test_learner_checkpoint_resumes_on_fused_learner(run, tmp_path):
  torch.backends.cuda.matmul.allow_tf32 = False
  case, optimizer, scheduler, graph_save, graph_load = run
  cfg, D, A, weights, batches = _case(case, optimizer, scheduler)
  l1, state = _run_two_steps(_torch_learner, cfg, D, A, weights, batches, graph_save, tmp_path / "ckpt")
  fresh = {k: v + 1.0 for k, v in weights.items()}  # the checkpoint's weights must replace these
  l2 = _fused_learner(cfg, D, A, fresh, graph_load, state=state)
  assert l2.training_step == 2
  assert np.float32(_lr(l2)) == np.float32(_lr(l1))
  if l2.own_optimizer:
    assert float(l2.opt_state[0]) == 2.0
  control = _fused_learner(cfg, D, A, l1.network.get_weights(), graph_load)
  _continue(l1, l2, control, batches[0], name=run)
  assert abs(_lr(l2) - _lr(l1)) <= 1e-6 * _lr(l1)  # ExponentialLR: one decay in float32 or float64


@pytest.mark.gpu
@pytest.mark.parametrize("run", RUNS, ids=RUN_IDS)
def test_fused_learner_checkpoint_resumes_on_learner(run, tmp_path):
  torch.backends.cuda.matmul.allow_tf32 = False
  case, optimizer, scheduler, graph_save, graph_load = run
  cfg, D, A, weights, batches = _case(case, optimizer, scheduler)
  l1, state = _run_two_steps(_fused_learner, cfg, D, A, weights, batches, graph_save, tmp_path / "ckpt")
  fresh = {k: v + 1.0 for k, v in weights.items()}
  l2 = _torch_learner(cfg, D, A, fresh, graph_load, state=state)
  assert l2.training_step == 2
  assert np.float32(_lr(l2)) == np.float32(_lr(l1))
  steps = {float(st["step"]) for st in l2.optimizer.state.values() if "step" in st}
  assert steps == ({2.0} if optimizer != "SGD" else set())
  control = _torch_learner(cfg, D, A, l1.network.get_weights(), graph_load)
  _continue(l1, l2, control, batches[0], name=run)
  assert abs(_lr(l2) - _lr(l1)) <= 1e-6 * _lr(l1)  # ExponentialLR: one decay in float32 or float64


@pytest.mark.gpu
@pytest.mark.parametrize("case,optimizer,graph", [("ttt", "AdamW", True), ("breakout", "RMSprop", False),
                                                  ("a64", "Adam", True)])
def test_bf16_fused_learner_resumes_from_learner_checkpoint(case, optimizer, graph, tmp_path):
  """The bf16 learner keeps float32 master weights and optimiser state: the same converted state as the f32 one.  Its
  third step lies within one step's bar of tests/test_fused_learner.py (2.5 learning rates; SGD 2e-3) of the f32
  resume, and its fresh-optimiser control outside ten times the f32 bar."""
  torch.backends.cuda.matmul.allow_tf32 = False
  cfg, D, A, weights, batches = _case(case, optimizer)
  l1, state = _run_two_steps(_torch_learner, cfg, D, A, weights, batches, False, tmp_path / "ckpt")
  f32 = _fused_learner(cfg, D, A, weights, False, state=state)
  bf = _fused_learner(cfg, D, A, weights, graph, state=state, precision="bf16")
  control = _fused_learner(cfg, D, A, l1.network.get_weights(), graph, precision="bf16")
  assert bf.training_step == 2
  want_lr = float(state["optimizer"]["param_groups"][0]["lr"])
  assert np.float32(_lr(bf)) == np.float32(want_lr)
  steps = {float(st["step"]) for st in state["optimizer"]["state"].values()}
  if bf.own_optimizer:
    assert {float(bf.opt_state[0])} == steps
  else:
    assert {float(st["step"]) for st in bf.optimizer.state.values()} == steps
  for learner in (f32, bf, control):
    learner.update_weights(batches[0])
  torch.cuda.synchronize()
  bar = 2e-3 if optimizer == "SGD" else 2.5 * cfg.lr_init
  diff = float((_flat_weights(bf) - _flat_weights(f32)).abs().max())
  off = float((_flat_weights(control) - _flat_weights(bf)).abs().max())
  print(case, optimizer, "bf16 vs f32 resume %.3g, fresh optimiser vs bf16 resume %.3g" % (diff, off))
  assert diff <= bar, diff
  assert off > 10 * BAR, off


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["AdamW", "RMSprop"])
@pytest.mark.parametrize("scheduler", ["MuZeroLR", "WarmUpLR"])
@pytest.mark.parametrize("target", ["fused", "learner"])
def test_schedule_after_a_switch_matches_a_resume_of_the_same_kind(target, scheduler, optimizer, tmp_path):
  """Neither checkpoint holds a schedule's counter (as in the reference): MuZeroLR / WarmUpLR restart theirs on any
  resume.  After a switch the next step runs at the learning rate, and the schedule continues with the one, that the
  target learner has after resuming from its own kind's checkpoint of the same run."""
  torch.backends.cuda.matmul.allow_tf32 = False
  cfg, D, A, weights, batches = _case("ttt", optimizer, scheduler)
  own_make, other_make = (_fused_learner, _torch_learner) if target == "fused" else (_torch_learner, _fused_learner)
  _, own_state = _run_two_steps(own_make, cfg, D, A, weights, batches, True, tmp_path / "own")
  _, other_state = _run_two_steps(other_make, cfg, D, A, weights, batches, True, tmp_path / "other")
  same = own_make(cfg, D, A, weights, True, state=own_state)
  switched = own_make(cfg, D, A, weights, True, state=other_state)
  assert _lr(switched) == _lr(same)
  for learner in (same, switched):
    learner.update_weights(batches[0])
  torch.cuda.synchronize()
  assert _lr(switched) == _lr(same)
  assert switched.lr_scheduler.lr_step == same.lr_scheduler.lr_step == 1


def _learner_checkpoint(cfg, D, A):
  """A learners.Learner checkpoint after a step: reference keys, per-parameter optimiser state."""
  from model_based_rl_b200 import learners
  weights = learners.FCNetworkTrain(D, A, "cpu", cfg).get_weights()
  return {"config": cfg, "weights": weights, "optimizer": _module_state(cfg, D, A), "training_step": 1}


@pytest.mark.gpu
@pytest.mark.parametrize("other", ["optimizer", "actions", "input_dim", "supports", "no_support"])
@pytest.mark.parametrize("optimizer", ["AdamW", "RMSprop"])
def test_fused_learner_refuses_learner_checkpoint_untouched(other, optimizer):
  """A learners.Learner checkpoint of another optimiser kind or network geometry: ValueError, and the FusedLearner's
  flat weights and optimiser tensors are what they were."""
  cfg, D, A, weights, batches = _case("ttt", optimizer)
  src = _case("ttt", {"AdamW": "RMSprop", "RMSprop": "AdamW"}[optimizer] if other == "optimizer" else optimizer)[0]
  D2, A2 = (D, A - 1) if other == "actions" else (D + 7, A) if other == "input_dim" else (D, A)
  if other == "supports":
    src.value_support = [-10, 10]
  if other == "no_support":
    src.no_support, src.scalar_loss = True, "MSE"
  learner = _fused_learner(cfg, D, A, weights, graph=optimizer == "AdamW")
  learner.update_weights(batches[0])
  torch.cuda.synchronize()
  before = _snapshot(learner)
  with pytest.raises(ValueError) as err:
    learner.load_state(_learner_checkpoint(src, D2, A2))
  _assert_untouched(learner, before)
  if other == "optimizer":
    assert "learners.Learner" in str(err.value)


@pytest.mark.gpu
def test_flat_layout_is_the_fused_networks():
  """checkpoints.flat_layout -- the offsets the mapping uses -- against the views FusedFCNetwork allocates."""
  from model_based_rl_b200 import checkpoints, fused_learner
  for D, A, no_support in GEOMETRIES:
    cfg = _ns(D, A, "AdamW", no_support)
    net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
    layout, n = checkpoints.flat_layout(D, A, cfg)
    assert net.flat.numel() == n and sorted(k for k, _, _ in layout) == sorted(net.views)
    for key, shape, off in layout:
      v = net.views[key]
      assert tuple(v.shape) == shape and (v.data_ptr() - net.flat.data_ptr()) // 4 == off, key
