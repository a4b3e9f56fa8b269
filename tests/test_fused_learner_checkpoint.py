"""FusedLearner checkpoints: save_state -> FusedLearner(state=...) / load_state resumes the run where it stopped (weights,
optimiser state, step counter, learning rate), in eager and graphed modes, and learn() writes checkpoints every
config.save_state_frequency steps."""
import types

import numpy as np
import pytest
import torch

import helpers
from test_learner import _batch, _config, _weights

pytestmark = pytest.mark.gpu

# (optimizer, graph for the saving learner, graph for the resuming learner)
RUNS = [("AdamW", True, True), ("AdamW", False, False), ("RMSprop", True, True), ("SGD", False, False),
        ("RMSprop", False, True)]
BAR = 1e-6  # the resumed and the uninterrupted step differ only in the order of the gradient atomics


def _cfg(case, optimizer):
  g = helpers.load("learner_" + case)
  cfg = _config(g)
  if "scalar_loss" in g:
    cfg.no_support, cfg.scalar_loss = True, str(g["scalar_loss"])
  cfg.optimizer = optimizer
  return g, cfg


def _learner(g, cfg, graph, state=None, weights=None):
  from model_based_rl_b200 import fused_learner
  net = fused_learner.FusedFCNetwork(int(g["obs_dim"]), int(g["action_space"]), "cuda", cfg)
  net.load_weights(_weights(g) if weights is None else weights)
  return fused_learner.FusedLearner(cfg, net, use_graph=graph, state=state)


def _opt_tensors(learner):
  if learner.own_optimizer:
    return {"exp_avg": learner.exp_avg, "exp_avg_sq": learner.exp_avg_sq, "state": learner.opt_state}
  return {"%s.%s" % (i, k): v for i, st in enumerate(learner.optimizer.state.values()) for k, v in st.items()
          if torch.is_tensor(v)}


def _lr(learner):
  return float(learner.opt_state[1]) if learner.own_optimizer else float(learner.optimizer.param_groups[0]["lr"])


@pytest.mark.parametrize("run", RUNS, ids=["-".join(map(str, r)) for r in RUNS])
@pytest.mark.parametrize("case", ["ttt", "nosupport_mse"])
def test_resumed_learner_continues_the_run(case, run, tmp_path):
  optimizer, graph_save, graph_load = run
  g, cfg = _cfg(case, optimizer)
  l1 = _learner(g, cfg, graph_save)
  for step in range(2):
    l1.update_weights(_batch(g, step))
  l1.training_step = 2  # what learn() would have counted
  path = str(tmp_path / "ckpt")
  l1.save_state(path)
  torch.cuda.synchronize()
  fresh = {k: v + 1.0 for k, v in _weights(g).items()}  # the checkpoint's weights must replace these
  l2 = _learner(g, cfg, graph_load, state=torch.load(path, weights_only=False), weights=fresh)
  assert torch.equal(l2.network.flat, l1.network.flat)
  assert l2.training_step == 2
  o1, o2 = _opt_tensors(l1), _opt_tensors(l2)
  assert sorted(o1) == sorted(o2) and o1
  for k in o1:
    assert torch.equal(o1[k].cpu(), o2[k].cpu()), k
  assert _lr(l1) == _lr(l2)
  # one more step on the same batch from both
  control = _learner(g, cfg, graph_load, weights={k: v.clone() for k, v in l1.network.get_weights().items()})
  batch = _batch(g, 0)
  for learner in (l1, l2, control):
    learner.update_weights(batch)
  torch.cuda.synchronize()
  diff = float((l2.network.flat - l1.network.flat).abs().max())
  assert diff <= BAR, diff
  o1, o2 = _opt_tensors(l1), _opt_tensors(l2)
  if l1.own_optimizer:
    assert float(o1["state"][0]) == float(o2["state"][0]) == 3.0
  for k in o1:
    if k.endswith(".step"):
      assert float(o1[k]) == float(o2[k]) == 3.0, k
  # negative control: the same weights with a fresh optimiser take a visibly different step
  off = float((control.network.flat - l1.network.flat).abs().max())
  print(case, run, "resumed vs uninterrupted %.3g, fresh optimiser vs uninterrupted %.3g" % (diff, off))
  assert off > 10 * BAR, off


def test_checkpoint_of_another_optimiser_or_size_is_refused(tmp_path):
  g, cfg = _cfg("ttt", "AdamW")
  state = _learner(g, cfg, False).save_state()
  g2, cfg2 = _cfg("ttt", "RMSprop")
  with pytest.raises(ValueError):
    _learner(g2, cfg2, False, state=state)
  gs, cfgs = _cfg("nosupport_huber", "AdamW")  # same observation / action sizes, one-unit heads: a smaller flat buffer
  with pytest.raises(ValueError):
    _learner(gs, cfgs, False, state=state)


def _replay(cfg, seed):
  from model_based_rl_b200.replay_buffer import PrioritizedReplay
  from model_based_rl_b200.selfplay import HistorySlice
  D, A = cfg.obs_space[0], cfg.action_space
  rb = PrioritizedReplay(cfg)
  r2 = np.random.default_rng(seed)
  for _ in range(8):
    n = int(r2.integers(50, 300))
    rb.save_history(HistorySlice(list(r2.normal(size=(n, D)).astype(np.float32)), r2.random((n, A)).tolist(),
                                 r2.normal(size=n).tolist(), r2.integers(0, A, size=n).tolist(), r2.normal(size=n).tolist(),
                                 np.abs(r2.normal(size=n)).tolist(), [False] * n, list(range(n)), [None] * n, [1] * n),
                    ignore=None, terminal=True)
  return rb


@pytest.mark.parametrize("no_support", [False, True], ids=["support", "no_support"])
def test_learn_saves_every_save_state_frequency_and_resumes_the_schedule(no_support, tmp_path):
  """learn() writes dirs['saves']/<training_step> every save_state_frequency steps; a learner built from the last
  checkpoint starts at its training_step and replay throughput, and its ExponentialLR continues: after resuming,
  lr = lr_init * gamma ** (total steps)."""
  from model_based_rl_b200 import fused_learner
  D, A, K = 8, 4, 3
  cfg = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=no_support, scalar_loss="MSE",
                              no_target_transform=False, num_unroll_steps=K, td_steps=5, optimizer="AdamW", lr_init=0.001,
                              momentum=0.9, weight_decay=1e-4, clip_grad=0, lr_scheduler="ExponentialLR",
                              lr_decay_rate=0.9, norm_obs=False, batch_size=64, beta_increment_per_sampling=0.001,
                              epsilon=0.01, alpha=1.0, beta=0.5, discount=0.997, action_space=A, obs_space=(D,),
                              window_size=2000, window_step=None, seed=None, send_weights_frequency=3, training_steps=7,
                              stored_before_train=100, save_state_frequency=3)
  rb = _replay(cfg, 7)
  learner = fused_learner.FusedLearner(cfg, fused_learner.FusedFCNetwork(D, A, "cuda", cfg), replay_buffer=rb)
  learner.dirs = {"saves": str(tmp_path)}
  learner.actor_games = {"actor_0": 5}
  assert learner.learn() == 7
  assert sorted(p.name for p in tmp_path.iterdir()) == ["3", "6"]
  state = torch.load(str(tmp_path / "6"), weights_only=False)
  assert state["training_step"] == 6 and state["dirs"] == {"saves": str(tmp_path)} and state["actor_games"] == {"actor_0": 5}
  assert learner.last_saved_state["training_step"] == 6
  rb2 = _replay(cfg, 8)
  frames = rb2.get_throughput()["frames"]
  resumed = fused_learner.FusedLearner(cfg, fused_learner.FusedFCNetwork(D, A, "cuda", cfg), replay_buffer=rb2,
                                       state=state)
  assert resumed.training_step == 6
  assert rb2.get_throughput()["frames"] == frames + state["total_frames"]
  assert resumed.learn(2) == 8
  want = 0.001 * 0.9 ** 8
  assert abs(resumed.lr_scheduler.lr - want) <= 1e-6 * want
  assert abs(float(resumed.opt_state[1]) - want) <= 1e-6 * want
