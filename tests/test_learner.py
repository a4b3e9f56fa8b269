"""Learner step (SURVEY.md section 8 f-4; learners.py:164-230).

CPU part: the oracle restatement (oracle/learner_ref.py + FCNetworkRef in train mode) and the host
logic of model_based_rl_b200.learners.Learner (unroll, hidden-gradient hook, optimisers, clipping)
against goldens produced by the reference's own FCNetwork / Config (tests/golden/learner_*.npz),
plus a world-size-2 gloo run of the data-parallel step.
GPU part: the fused CUDA loss against the oracle and the goldens, and the whole step on the device.
"""
import os
import socket
import types

import numpy as np
import pytest
import torch

import helpers
from oracle import learner_ref
from oracle.fcnet_ref import FCNetworkRef

CASES = ["breakout", "ttt", "lunar_raw"]


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


def _sub(v):
  v = v.reshape(-1) if v.numel() > 2048 else v
  return v[::max(1, v.numel() // 1024)] if v.numel() > 2048 else v


def _check_against_golden(g, learner, net, tol, exact_first_step=None):
  """exact_first_step: (losses, errors) the first step must reproduce bit for bit."""
  from model_based_rl_b200 import learners  # noqa: F401  (imported by the caller; keeps flake quiet)
  for step in range(2):
    losses = learner.update_weights(_batch(g, step))
    if step == 0 and exact_first_step is not None:
      np.testing.assert_array_equal(losses.cpu().numpy(), exact_first_step[0])
      np.testing.assert_array_equal(learner.last_errors.cpu().numpy(), exact_first_step[1])
    np.testing.assert_allclose(losses.cpu().numpy(), g["s%d_losses" % step], rtol=tol, atol=0)
    np.testing.assert_allclose(learner.last_errors.cpu().numpy(), g["s%d_new_errors" % step], rtol=0,
                               atol=max(tol * 40, 5e-4))  # h^-1 cancels in float32 (DESIGN.md section 2)
    for k, v in net.state_dict().items():
      np.testing.assert_allclose(_sub(v.detach().cpu()).numpy(), g["s%d_w_%s" % (step, k)], rtol=0, atol=tol,
                                 err_msg="step %d %s" % (step, k))


@pytest.mark.parametrize("case", CASES)
def test_oracle_learner_step_matches_reference_golden(case):
  """Oracle network + oracle loss inside the product's Learner host logic, on the CPU."""
  from model_based_rl_b200 import learners
  g = helpers.load("learner_" + case)
  cfg = _config(g)
  net = FCNetworkRef(int(g["obs_dim"]), int(g["action_space"]), no_target_transform=cfg.no_target_transform)
  net.load_state_dict(_weights(g))
  net.get_weights = lambda: {k: v.cpu() for k, v in net.state_dict().items()}
  learner = learners.Learner(cfg, net, loss_fn=learner_ref.unroll_loss_ref)
  # gradients of the first step, before the optimiser touches anything
  net.train()
  batch = _batch(g, 0)
  (obs, actions, (t_r, t_v, t_p)), _, is_w = batch
  out = net.initial_inference(torch.from_numpy(obs))
  values, rewards, policies, h = [out.value], [], [out.policy_logits], out.hidden_state
  for i in range(cfg.num_unroll_steps):
    out = net.recurrent_inference(h, [a[i] for a in actions])
    h = out.hidden_state
    h.register_hook(lambda grad: grad * 0.5)
    values.append(out.value), rewards.append(out.reward), policies.append(out.policy_logits)
  losses, errs = learner_ref.unroll_loss_ref(cfg, values, rewards, policies, torch.from_numpy(t_v),
                                             torch.from_numpy(t_r), torch.from_numpy(t_p), torch.from_numpy(is_w))
  net.zero_grad()
  losses.sum().backward()
  # torch's CPU kernels (MKL GEMM, ATen's vectorised loops) are picked by the CPU's instruction set, and another kernel
  # groups the float32 sums differently: the reference's run is reproduced bit for bit only on a CPU that picks the
  # same kernels, elsewhere to float32 rounding (losses up to 3e-8 relative; h^-1 amplifies it in the priorities).
  np.testing.assert_allclose(losses.detach().numpy(), g["s0_losses"], rtol=1e-7)
  np.testing.assert_allclose(errs.numpy(), g["s0_new_errors"], rtol=0, atol=5e-4)
  for k, p in net.named_parameters():
    gr = p.grad
    np.testing.assert_allclose(float(gr.double().pow(2).sum().sqrt()), float(g["s0_gnorm_" + k]), rtol=1e-6)
    np.testing.assert_allclose(_sub(gr).numpy(), g["s0_g_" + k], rtol=0, atol=1e-7, err_msg=k)
  net.zero_grad()
  # on the same CPU the Learner's first step is the restatement above, bit for bit
  _check_against_golden(g, learner, net, tol=1e-6, exact_first_step=(losses.detach().numpy(), errs.numpy()))


@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("batched", [True, False])
def test_product_network_unroll_matches_reference_golden(case, batched):
  """The product's torch module through Learner on the CPU with the oracle loss: the batched-heads unroll
  (FCNetworkTrain.unroll: one head evaluation over all K+1 hidden states) and the step-by-step path both
  reproduce the reference's two steps (losses 1e-6 relative, weights 1e-6 absolute: GEMM row blocking
  differs with the batch shape)."""
  from model_based_rl_b200 import learners
  g = helpers.load("learner_" + case)
  cfg = _config(g)
  net = learners.FCNetworkTrain(int(g["obs_dim"]), int(g["action_space"]), "cpu", cfg)
  net.load_weights(_weights(g))
  learner = learners.Learner(cfg, net, loss_fn=learner_ref.unroll_loss_ref, batched_heads=batched)
  _check_against_golden(g, learner, net, tol=1e-6)


@pytest.mark.parametrize("case", ["nosupport_mse", "nosupport_huber"])
@pytest.mark.parametrize("batched", [True, False])
def test_no_support_learner_matches_reference_golden(case, batched):
  """`--no_support` training (config.py:95-96; utils.py:61-70; learners.py:182, 190): one-unit value / reward heads,
  MSE or Huber against the scalar targets.  The product's FCNetworkTrain + scalar_unroll_loss through Learner
  reproduce two steps of the reference's FCNetwork(no_support=True) around the restated update_weights body."""
  from model_based_rl_b200 import learners
  g = helpers.load("learner_" + case)
  cfg = _config(g)
  cfg.no_support, cfg.scalar_loss = True, str(g["scalar_loss"])
  net = learners.FCNetworkTrain(int(g["obs_dim"]), int(g["action_space"]), "cpu", cfg)
  assert net.value_head.value.weight.shape == (1, 512) and net.reward_head.reward.weight.shape == (1, 512)
  net.load_weights(_weights(g))
  learner = learners.Learner(cfg, net, loss_fn=learners.scalar_unroll_loss, batched_heads=batched)
  _check_against_golden(g, learner, net, tol=1e-6)


def test_product_train_network_has_reference_keys_and_outputs():
  """FCNetworkTrain (torch module of the product) == the oracle network on the golden weights."""
  from model_based_rl_b200 import learners
  g = helpers.load("learner_breakout")
  cfg = _config(g)
  w = _weights(g)
  net = learners.FCNetworkTrain(int(g["obs_dim"]), int(g["action_space"]), "cpu", cfg)
  assert sorted(net.state_dict().keys()) == sorted(w.keys())
  net.load_weights(w)
  ref = FCNetworkRef(int(g["obs_dim"]), int(g["action_space"]))
  ref.load_state_dict(w)
  ref.train()
  obs = torch.from_numpy(g["s0_obs"])
  a, b = net.initial_inference(obs), ref.initial_inference(obs)
  assert torch.equal(a.value, b.value) and torch.equal(a.policy_logits, b.policy_logits)
  acts = g["s0_actions"][:, 0]
  a2, b2 = net.recurrent_inference(a.hidden_state, torch.from_numpy(acts)), ref.recurrent_inference(b.hidden_state, list(acts))
  for x, y in zip(a2, b2):
    assert torch.equal(x, y)


def test_learner_without_cuda_raises_like_the_reference():
  from model_based_rl_b200 import learners
  if torch.cuda.is_available():
    pytest.skip("CUDA present")
  g = helpers.load("learner_ttt")
  net = learners.FCNetworkTrain(9, 9, "cpu", _config(g))
  with pytest.raises(RuntimeError, match="GPU was requested"):
    learners.Learner(_config(g), net)


def test_lr_schedules():
  from model_based_rl_b200 import learners
  p = [torch.nn.Parameter(torch.zeros(2))]
  cfg = types.SimpleNamespace(optimizer="SGD", lr_init=0.1, momentum=0.9, weight_decay=0.0, lr_scheduler="MuZeroLR",
                              lr_decay_rate=0.1, lr_decay_steps=10)
  opt = learners.get_optimizer(cfg, p)
  sch = learners.get_lr_scheduler(cfg, opt)
  for _ in range(10):
    sch.step()
  assert abs(opt.param_groups[0]["lr"] - 0.01) < 1e-12
  cfg.lr_scheduler = "WarmUpLR"
  opt = learners.get_optimizer(cfg, p)
  sch = learners.get_lr_scheduler(cfg, opt)
  assert abs(opt.param_groups[0]["lr"] - 0.1 / 5000) < 1e-15
  sch.step()
  assert abs(opt.param_groups[0]["lr"] - 0.1 / 5000) < 1e-15
  sch.step()
  assert abs(opt.param_groups[0]["lr"] - 0.2 / 5000) < 1e-15
  with pytest.raises(NotImplementedError):
    learners.get_optimizer(types.SimpleNamespace(optimizer="LBFGS", lr_init=0.1), p)


# -- world size 2 (gloo, CPU): data-parallel learner step ---------------------------------------
def _dp_worker(rank, world_size, port, out):
  import torch.distributed as dist
  os.environ["MASTER_ADDR"] = "127.0.0.1"
  os.environ["MASTER_PORT"] = str(port)
  dist.init_process_group("gloo", rank=rank, world_size=world_size)
  try:
    from model_based_rl_b200 import learners
    torch.set_num_threads(1)
    g = helpers.load("learner_ttt")
    cfg = _config(g)
    cfg.optimizer, cfg.clip_grad = "SGD", 0
    net = learners.FCNetworkTrain(9, 9, "cpu", cfg)
    torch.manual_seed(100 + rank)  # ranks start from different weights: send_weights must align them
    for p in net.parameters():
      p.data.add_(0.01 * torch.randn_like(p))
    if rank == 0:
      net.load_weights(_weights(g))
    learner = learners.Learner(cfg, net, loss_fn=learner_ref.unroll_loss_ref)
    learner.send_weights()
    for k, v in net.state_dict().items():
      assert torch.equal(v, _weights(g)[k]), k
    learner.update_weights(_batch(g, rank))  # rank r trains on the golden batch of step r
    mine = {k: v.clone() for k, v in net.state_dict().items()}
    # single-process restatement: gradients of both batches averaged, one SGD step
    solo = learners.FCNetworkTrain(9, 9, "cpu", cfg)
    solo.load_weights(_weights(g))
    grads = []
    for r in range(world_size):
      solo.zero_grad()
      l2 = learners.Learner(cfg, solo, loss_fn=learner_ref.unroll_loss_ref)
      l2.optimizer = types.SimpleNamespace(zero_grad=solo.zero_grad, step=lambda: None)
      _solo_grads(l2, _batch(g, r))
      grads.append([p.grad.clone() for p in solo.parameters()])
    opt = learners.get_optimizer(cfg, solo.parameters())
    for p, g0, g1 in zip(solo.parameters(), *grads):
      p.grad = (g0 + g1) / 2
    opt.step()
    for k, v in solo.state_dict().items():
      assert torch.allclose(v, mine[k], rtol=0, atol=1e-7), k
    gathered = [None] * world_size
    dist.all_gather_object(gathered, {k: v.numpy() for k, v in mine.items()})
    for k in mine:
      assert np.array_equal(gathered[0][k], gathered[1][k]), k
    out.put((rank, "ok"))
  except Exception as e:  # pragma: no cover
    import traceback
    out.put((rank, traceback.format_exc()))
  finally:
    dist.destroy_process_group()


def _solo_grads(learner, batch):
  """update_weights without the all-reduce and the optimiser: leaves .grad of this batch alone."""
  from model_based_rl_b200 import parallel
  real = parallel.allreduce_gradients
  parallel.allreduce_gradients = lambda *a, **k: None
  try:
    learner.update_weights(batch)
  finally:
    parallel.allreduce_gradients = real


def test_data_parallel_learner_two_ranks_gloo():
  import torch.multiprocessing as mp
  ctx = mp.get_context("spawn")
  out = ctx.Queue()
  s = socket.socket()
  s.bind(("127.0.0.1", 0))
  port = s.getsockname()[1]
  s.close()
  procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, out)) for r in range(2)]
  for p in procs:
    p.start()
  res = [out.get(timeout=180) for _ in procs]
  for p in procs:
    p.join(timeout=60)
  assert sorted(res) == [(0, "ok"), (1, "ok")], res


# -- GPU: the fused loss kernel and the whole step ----------------------------------------------
def _forward_logits(net, cfg, obs, actions):
  out = net.initial_inference(obs)
  values, rewards, policies, h = [out.value], [], [out.policy_logits], out.hidden_state
  for i in range(cfg.num_unroll_steps):
    out = net.recurrent_inference(h, actions[:, i])
    h = out.hidden_state
    values.append(out.value), rewards.append(out.reward), policies.append(out.policy_logits)
  return values, rewards, policies


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_gpu_unroll_loss_matches_oracle(case):
  """mz_unroll_loss on the golden batch's logits: losses, priority errors and the gradient with
  respect to every logit against the oracle's autograd (float32 arithmetic: 1e-5 relative for the
  losses as north_star states, 1e-7 absolute for the gradients, which are O(1/(B K)))."""
  from model_based_rl_b200 import learners
  g = helpers.load("learner_" + case)
  cfg = _config(g)
  net = learners.FCNetworkTrain(int(g["obs_dim"]), int(g["action_space"]), "cpu", cfg)
  net.load_weights(_weights(g))
  (obs, actions, (t_r, t_v, t_p)), _, is_w = _batch(g, 0)
  with torch.no_grad():
    values, rewards, policies = _forward_logits(net, cfg, torch.from_numpy(obs), torch.tensor(actions))
  cpu = [[t.clone().requires_grad_(True) for t in lst] for lst in (values, rewards, policies)]
  ref_losses, ref_errs = learner_ref.unroll_loss_ref(cfg, cpu[0], cpu[1], cpu[2], torch.from_numpy(t_v),
                                                     torch.from_numpy(t_r), torch.from_numpy(t_p),
                                                     torch.from_numpy(is_w))
  ref_losses.sum().backward()
  dev = [[t.clone().cuda().requires_grad_(True) for t in lst] for lst in (values, rewards, policies)]
  losses, errs = learners.unroll_loss(cfg, dev[0], dev[1], dev[2], torch.from_numpy(t_v).cuda(),
                                      torch.from_numpy(t_r).cuda(), torch.from_numpy(t_p).cuda(),
                                      torch.from_numpy(is_w).cuda())
  losses.sum().backward()
  np.testing.assert_allclose(losses.detach().cpu().numpy(), ref_losses.detach().numpy(), rtol=1e-5)
  np.testing.assert_allclose(losses.detach().cpu().numpy(), g["s0_losses"], rtol=1e-5)
  np.testing.assert_allclose(errs.cpu().numpy(), ref_errs.numpy(), rtol=0, atol=5e-4)
  assert np.mean(np.abs(errs.cpu().numpy() - ref_errs.numpy()) <= 1e-5 * np.maximum(1, np.abs(ref_errs.numpy()))) > 0.9
  for a, b in zip(sum(dev, []), sum(cpu, [])):
    np.testing.assert_allclose(a.grad.cpu().numpy(), b.grad.numpy(), rtol=0, atol=1e-7)


@pytest.mark.gpu
def test_gpu_unroll_loss_edge_rows():
  """Integer targets (one-hot), clamped targets, all-zero policy rows (positions past the end of the
  episode) and no importance weights; wide supports (601 bins)."""
  from model_based_rl_b200 import learners
  rng = np.random.default_rng(5)
  B, K, A = 7, 2, 3
  cfg = types.SimpleNamespace(value_support=[-300, 300], reward_support=[-1, 1], no_target_transform=True,
                              num_unroll_steps=K)
  values = [torch.from_numpy(rng.normal(size=(B, 601)).astype(np.float32)) for _ in range(K + 1)]
  rewards = [torch.from_numpy(rng.normal(size=(B, 3)).astype(np.float32)) for _ in range(K)]
  policies = [torch.from_numpy(rng.normal(size=(B, A)).astype(np.float32)) for _ in range(K + 1)]
  t_v = torch.tensor(rng.uniform(-350, 350, size=(B, K + 1)).astype(np.float32))
  t_v[0, 0], t_v[1, 1], t_v[2, 2] = 300.0, -300.0, 17.0
  t_r = torch.tensor(rng.integers(-2, 3, size=(B, K + 1)).astype(np.float32))
  t_p = torch.zeros(B, K + 1, A)
  t_p[:4] = torch.softmax(torch.from_numpy(rng.normal(size=(4, K + 1, A)).astype(np.float32)), -1)
  ones = torch.ones(B, dtype=torch.float64)
  cpu = [[t.clone().requires_grad_(True) for t in lst] for lst in (values, rewards, policies)]
  ref_losses, _ = learner_ref.unroll_loss_ref(cfg, cpu[0], cpu[1], cpu[2], t_v, t_r, t_p, ones)
  ref_losses.sum().backward()
  dev = [[t.clone().cuda().requires_grad_(True) for t in lst] for lst in (values, rewards, policies)]
  losses, _ = learners.unroll_loss(cfg, dev[0], dev[1], dev[2], t_v.cuda(), t_r.cuda(), t_p.cuda(), None)
  (2.0 * losses.sum()).backward()  # backward scales with the incoming gradient
  np.testing.assert_allclose(losses.detach().cpu().numpy(), ref_losses.detach().numpy(), rtol=1e-5)
  for a, b in zip(sum(dev, []), sum(cpu, [])):
    np.testing.assert_allclose(a.grad.cpu().numpy(), 2.0 * b.grad.numpy(), rtol=0, atol=2e-7)
  with pytest.raises(RuntimeError):
    learners.unroll_loss(cfg, cpu[0], cpu[1], cpu[2], t_v, t_r, t_p, None)  # CPU tensors: no fallback


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_gpu_learner_two_steps_match_reference_golden(case):
  """Whole step on the device (cuBLAS float32 GEMMs + the fused loss + torch optimiser) against the
  reference's losses / updated weights after two steps.  GEMM summation order differs from the CPU's:
  1e-4 relative on the losses, 2e-5 absolute on the weights."""
  from model_based_rl_b200 import learners
  torch.backends.cuda.matmul.allow_tf32 = False
  g = helpers.load("learner_" + case)
  cfg = _config(g)
  net = learners.FCNetworkTrain(int(g["obs_dim"]), int(g["action_space"]), "cuda", cfg)
  net.load_weights(_weights(g))
  learner = learners.Learner(cfg, net)
  for step in range(2):
    losses = learner.update_weights(_batch(g, step))
    np.testing.assert_allclose(losses.cpu().numpy(), g["s%d_losses" % step], rtol=1e-4)
    np.testing.assert_allclose(learner.last_errors.cpu().numpy(), g["s%d_new_errors" % step], rtol=0, atol=2e-3)
    for k, v in net.state_dict().items():
      np.testing.assert_allclose(_sub(v.detach().cpu()).numpy(), g["s%d_w_%s" % (step, k)], rtol=0, atol=2e-5,
                                 err_msg="step %d %s" % (step, k))
  assert learner.log_losses()[1] > 0


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["nosupport_mse", "nosupport_huber"])
def test_gpu_no_support_learner_and_weight_handoff(case):
  """`--no_support` on the device: Learner picks the scalar loss by itself, two steps against the reference's golden,
  then the weight hand-off into the search kernels' FCNetwork (which takes the float32-accurate tensor-core kernels
  for such networks): its value / reward are the train network's raw head outputs."""
  from model_based_rl_b200 import learners, networks
  torch.backends.cuda.matmul.allow_tf32 = False
  g = helpers.load("learner_" + case)
  cfg = _config(g)
  cfg.no_support, cfg.scalar_loss = True, str(g["scalar_loss"])
  D, A = int(g["obs_dim"]), int(g["action_space"])
  net = learners.FCNetworkTrain(D, A, "cuda", cfg)
  net.load_weights(_weights(g))
  search_net = networks.FCNetwork(D, A, "cuda", cfg)
  assert search_net.precision == "tf32x3"
  learner = learners.Learner(cfg, net, search_network=search_net)
  assert learner.loss_fn is learners.scalar_unroll_loss
  for step in range(2):
    losses = learner.update_weights(_batch(g, step))
    np.testing.assert_allclose(losses.cpu().numpy(), g["s%d_losses" % step], rtol=1e-4)
    np.testing.assert_allclose(learner.last_errors.cpu().numpy(), g["s%d_new_errors" % step], rtol=0, atol=1e-4)
    for k, v in net.state_dict().items():
      np.testing.assert_allclose(_sub(v.detach().cpu()).numpy(), g["s%d_w_%s" % (step, k)], rtol=0, atol=2e-5,
                                 err_msg="step %d %s" % (step, k))
  learner.send_weights()
  obs = torch.from_numpy(g["s0_obs"]).cuda()
  acts = torch.from_numpy(g["s0_actions"][:, 0].astype(np.int64)).cuda()
  with torch.no_grad():
    t0 = net.initial_inference(obs)
    t1 = net.recurrent_inference(t0.hidden_state, acts)
  s0 = search_net.initial_inference(obs)
  s1 = search_net.recurrent_inference(t0.hidden_state, acts.to(torch.int32))
  torch.cuda.synchronize()
  for a, b in ((t0.value, s0.value), (t0.policy_logits, s0.policy_logits), (t1.value, s1.value), (t1.reward, s1.reward),
               (t1.hidden_state, s1.hidden_state)):
    assert a.shape == b.shape
    assert torch.allclose(a, b, rtol=1e-4, atol=2e-5), (a - b).abs().max().item()


@pytest.mark.gpu
def test_gpu_learner_loop_with_replay_and_search_network():
  """learn(): PrioritizedReplay.sample_batch -> update_weights -> replay.update, and the weight
  hand-off into the search kernels' FCNetwork (learners.py:116-135, 84-85)."""
  import random
  from model_based_rl_b200 import learners, networks
  import test_gpu_replay as tr
  g = helpers.load("replay_breakout")
  random.seed(3)
  np.random.seed(3)
  rb = tr._filled(g)
  cfg = tr._config(g, optimizer="AdamW", lr_init=0.0008, momentum=0.9, weight_decay=1e-4, clip_grad=0,
                   lr_scheduler="MuZeroLR", lr_decay_rate=0.1, lr_decay_steps=1000, norm_obs=False,
                   send_weights_frequency=2, training_steps=4, no_support=False)
  A, D = int(g["action_space"]), int(g["obs_dim"])
  net = learners.FCNetworkTrain(D, A, "cuda", cfg)
  search_net = networks.FCNetwork(D, A, "cuda", cfg, precision="f32")
  learner = learners.Learner(cfg, net, replay_buffer=rb, search_network=search_net)
  tree_before = rb.index.tree.clone()
  assert learner.learn() == 4
  assert torch.isfinite(learner.last_losses).all()
  assert not torch.equal(tree_before, rb.index.tree)  # priorities were fed back
  assert abs(learner.optimizer.param_groups[0]["lr"] - 0.0008 * 0.1 ** (4 / 1000)) < 1e-12
  # the search network now evaluates the learner's weights: eval-mode scalars of the torch module
  obs = torch.from_numpy(np.stack(g["h0_obs"][:8]).astype(np.float32)).cuda()
  out = search_net.initial_inference(obs)
  with torch.no_grad():
    ref = net.initial_inference(obs)
  np.testing.assert_allclose(out.policy_logits.cpu().numpy(), ref.policy_logits.cpu().numpy(), rtol=0, atol=1e-4)
  state = learner.save_state()
  again = learners.Learner(cfg, learners.FCNetworkTrain(D, A, "cuda", cfg), replay_buffer=rb, state=state)
  assert again.training_step == 4
  for a, b in zip(again.network.state_dict().values(), net.state_dict().values()):
    assert torch.equal(a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("case,scheduler", [("breakout", None), ("ttt", "MuZeroLR"), ("lunar_raw", None),
                                            ("lunar_raw", "WarmUpLR")])
def test_gpu_learner_cuda_graph_step_equals_eager_step(case, scheduler):
  """use_graph=True (forward + loss + backward in one CUDA graph, clipping + optimiser in a second)
  follows the eager learner over five steps on alternating batches, and the reference's golden after
  the first two.  Capturable Adam / RMSprop evaluate their bias corrections in float32 on the device:
  1e-6 absolute on the weights."""
  from model_based_rl_b200 import learners
  torch.backends.cuda.matmul.allow_tf32 = False
  g = helpers.load("learner_" + case)
  nets, ls = [], []
  for use_graph in (False, True):
    cfg = _config(g)
    cfg.lr_scheduler, cfg.lr_decay_rate, cfg.lr_decay_steps = scheduler, 0.1, 3
    net = learners.FCNetworkTrain(int(g["obs_dim"]), int(g["action_space"]), "cuda", cfg)
    net.load_weights(_weights(g))
    nets.append(net)
    ls.append(learners.Learner(cfg, net, use_graph=use_graph))
  for step in range(5):
    la = ls[0].update_weights(_batch(g, step % 2))
    lb = ls[1].update_weights(_batch(g, step % 2))
    np.testing.assert_allclose(lb.cpu().numpy(), la.cpu().numpy(), rtol=1e-5)
    np.testing.assert_allclose(ls[1].last_errors.cpu().numpy(), ls[0].last_errors.cpu().numpy(), rtol=0, atol=2e-3)
    if scheduler is None and step < 2:
      np.testing.assert_allclose(lb.cpu().numpy(), g["s%d_losses" % step], rtol=1e-4)
    for (k, a), b in zip(nets[0].state_dict().items(), nets[1].state_dict().values()):
      np.testing.assert_allclose(b.cpu().numpy(), a.cpu().numpy(), rtol=0, atol=1e-6, err_msg="step %d %s" % (step, k))
  assert ls[1]._graphs is not None
  if scheduler is not None:
    assert abs(float(ls[1].optimizer.param_groups[0]["lr"]) - float(ls[0].optimizer.param_groups[0]["lr"])) < 1e-9
