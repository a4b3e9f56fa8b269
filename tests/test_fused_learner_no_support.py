"""`--no_support` networks (one-unit value / reward heads, MSE or Huber scalar loss) on the fused learner: the scalar
unroll loss kernel (mz_scalar_unroll_loss) against learners.scalar_unroll_loss + autograd, the head kernels at one
output column, and FusedLearner in both precisions against the reference's goldens (tests/golden/learner_nosupport_*)."""
import ctypes as C
import itertools
import types

import numpy as np
import pytest
import torch

import helpers
from test_fused_learner import _rel, _teacher_forced_check
from test_learner import _batch, _config, _sub, _weights

CASES = ["nosupport_mse", "nosupport_huber"]


def _ns_config(g):
  cfg = _config(g)
  cfg.no_support, cfg.scalar_loss = True, str(g["scalar_loss"])
  return cfg


def _nets(g, cfg):
  from model_based_rl_b200 import fused_learner, learners
  D, A = int(g["obs_dim"]), int(g["action_space"])
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  net.load_weights(_weights(g))
  ref = learners.FCNetworkTrain(D, A, "cuda", cfg)
  ref.load_weights(_weights(g))
  return net, ref


def test_scalar_unroll_loss_rejects_bad_arguments_without_a_gpu():
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  ok = lambda: _lib.LossCfg(4, 3, 5, -15, 15, -15, 15, 0)
  dummy = [C.c_void_p(16 * (i + 1)) for i in range(13)]  # never dereferenced: every check comes before a launch
  call = lambda c, kind, ptrs: lib.mz_scalar_unroll_loss(c, kind, *ptrs, None)
  for field, value in (("num_unroll_steps", 0), ("num_unroll_steps", 32), ("num_actions", 0), ("batch", 0),
                       ("batch", -1)):
    c = ok()
    setattr(c, field, value)
    assert call(C.byref(c), 0, dummy) == -1, (field, value)
  for kind in (-1, 2):
    assert call(C.byref(ok()), kind, dummy) == -1, kind
  assert lib.mz_scalar_unroll_loss(None, 0, *dummy, None) == -1
  # required: value, reward, policy, the three targets, row_losses, losses; is_weights, the gradients and new_errors may be NULL
  for i in (0, 1, 2, 3, 4, 5, 10, 11):
    ptrs = list(dummy)
    ptrs[i] = None
    assert call(C.byref(ok()), 1, ptrs) == -2, i


def _h(x):
  return torch.sign(x) * (torch.sqrt(torch.abs(x) + 1) - 1) + 0.001 * x


@pytest.mark.gpu
@pytest.mark.parametrize("weighted", [False, True], ids=["no_is_weights", "is_weights"])
@pytest.mark.parametrize("ntt", [False, True], ids=["h", "no_target_transform"])
@pytest.mark.parametrize("kind", ["MSE", "Huber"])
def test_scalar_unroll_loss_kernel_matches_torch_autograd(kind, ntt, weighted):
  """Losses (rtol 1e-6), priority errors (bit for bit: one subtraction) and the gradient of every value, reward and
  policy output (within 1e-6 of each tensor's largest entry) against learners.scalar_unroll_loss and torch autograd
  on the device, over K in {1, 3, 5}, B in {1, 24, 300}, A in {4, 9, 18}.  Targets include 0, negative and large
  values; where the target is 0 the output sits exactly at, or one float32 step either side of, the Huber kinks +-1."""
  from model_based_rl_b200 import _lib, learners
  lib = _lib.load()
  cfg = types.SimpleNamespace(no_target_transform=ntt, scalar_loss=kind)
  P = lambda t: None if t is None else C.c_void_p(t.data_ptr())
  one = np.float32(1.0)
  kinks = torch.tensor([-1.0, 1.0, np.nextafter(one, 2), np.nextafter(one, 0), -np.nextafter(one, 2),
                        -np.nextafter(one, 0), 0.0, 0.4, -2.5, 7.0], dtype=torch.float32, device="cuda")
  worst = {}
  for K, B, A in itertools.product((1, 3, 5), (1, 24, 300), (4, 9, 18)):
    gen = torch.Generator(device="cuda").manual_seed(1000 * K + 10 * B + A)
    rnd = lambda *s: torch.rand(*s, device="cuda", generator=gen)
    pick = lambda n, vals: vals[torch.randint(0, len(vals), (n,), device="cuda", generator=gen)]
    raw = torch.tensor([0.0, 0.0, -3.0, 0.5, -0.25, 250.0, -1e4, 1e4, 2.0, -17.5], device="cuda")
    tv = torch.where(rnd(B, K + 1) < 0.5, pick(B * (K + 1), raw).view(B, K + 1), 8 * torch.randn(B, K + 1, device="cuda",
                                                                                                generator=gen))
    tr = torch.where(rnd(B, K + 1) < 0.5, pick(B * (K + 1), raw).view(B, K + 1), 3 * torch.randn(B, K + 1, device="cuda",
                                                                                                generator=gen))
    tgt = lambda t: t if ntt else _h(t)
    # outputs = target + an offset from the list above (exact differences where the target is 0)
    v = (tgt(tv).t() + pick(B * (K + 1), kinks).view(K + 1, B)).reshape(K + 1, B, 1).contiguous()
    r = (tgt(tr)[:, 1:].t() + pick(B * K, kinks).view(K, B)).reshape(K, B, 1).contiguous()
    p = 3 * torch.randn(K + 1, B, A, device="cuda", generator=gen)
    tp = rnd(B, K + 1, A)
    tp = tp / tp.sum(-1, keepdim=True)
    isw = (0.2 + rnd(B)).double() if weighted else None
    # the kernel
    dv, dr, dp = torch.empty_like(v), torch.empty_like(r), torch.empty_like(p)
    rows = torch.empty((3, B), dtype=torch.float64, device="cuda")
    losses = torch.empty(3, dtype=torch.float64, device="cuda")
    errs = torch.empty(B, dtype=torch.float32, device="cuda")
    c = _lib.LossCfg(B, K, A, -15, 15, -15, 15, int(ntt))
    _lib.check(lib.mz_scalar_unroll_loss(C.byref(c), int(kind == "Huber"), P(v), P(r), P(p), P(tv), P(tr), P(tp), P(isw),
                                         P(dv), P(dr), P(dp), P(rows), P(losses), P(errs), None), "mz_scalar_unroll_loss")
    # torch
    vv, rr, pp = [t.clone().requires_grad_(True) for t in (v, r, p)]
    w = isw if weighted else torch.ones(B, dtype=torch.float64, device="cuda")
    want, want_errs = learners.scalar_unroll_loss(cfg, vv, rr, pp, tv, tr, tp, w)
    want.sum().backward()
    torch.cuda.synchronize()
    shape = (K, B, A)
    np.testing.assert_allclose(losses.cpu().numpy(), want.detach().cpu().numpy(), rtol=1e-6, err_msg=str(shape))
    assert torch.equal(errs, want_errs), shape
    for name, got, ref in (("value", dv, vv.grad), ("reward", dr, rr.grad), ("policy", dp, pp.grad)):
      err = _rel(got, ref)
      assert err <= 1e-6, (shape, name, err)
      if err >= worst.get(name, (-1,))[0]:
        worst[name] = (err, shape)
  print(kind, "ntt" if ntt else "h", "weighted" if weighted else "unweighted", "worst gradient error / scale:", worst)


def _pack_head(lib, _lib, W1, W2, d_in, d_out):
  imgs, pj = [], []
  for (n, k), (src, sn, sk) in zip([(512, d_in), (d_out, 512), (512, d_out), (d_in, 512)],
                                   [(W1, d_in, 1), (W2, 512, 1), (W2, 1, 512), (W1, 1, d_in)]):
    img = torch.zeros(int(lib.mz_learner_packed_words(n, k)), dtype=torch.int32, device="cuda")
    imgs.append(img)
    pj.append(_lib.PackJob(src.data_ptr(), img.data_ptr(), n, k, sn, sk))
  _lib.check(lib.mz_learner_pack(4, (_lib.PackJob * 4)(*pj), None), "pack")
  return imgs


@pytest.mark.gpu
def test_tc_head_kernels_one_output_column():
  """mz_heads_forward_tc / mz_heads_backward_tc for a one-unit head (d_out = 1, ldy = 1: the scalar value / reward
  heads) on ragged row counts, padded input widths and strided rows, two jobs per launch: against the head in float64
  on the bf16-rounded operands, with the bars of test_tc_head_kernels_ragged_rows_match_torch."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  rng = torch.Generator(device="cuda").manual_seed(12)
  bf = lambda t: t.to(torch.bfloat16).double()
  jobs, keep = [], []
  for rows, d_in, ldx in ((1, 9, 9), (45, 54, 54), (100, 128, 130), (33, 68, 70)):
    X = torch.randn(rows, ldx, device="cuda", generator=rng)
    W1, b1 = torch.randn(512, d_in, device="cuda", generator=rng) * 0.1, torch.randn(512, device="cuda", generator=rng) * 0.1
    W2, b2 = torch.randn(1, 512, device="cuda", generator=rng) * 0.1, torch.randn(1, device="cuda", generator=rng)
    dY = torch.randn(rows, 1, device="cuda", generator=rng)
    Y = torch.full((rows, 1), 7.0, device="cuda")
    dX = torch.ones(rows, ldx, device="cuda")
    grads = [torch.zeros_like(t) for t in (W1, b1, W2, b2)]
    imgs = _pack_head(lib, _lib, W1, W2, d_in, 1)
    head = _lib.TcHead(*[i.data_ptr() for i in imgs], b1.data_ptr(), b2.data_ptr(), *[t.data_ptr() for t in grads], d_in, 1)
    jobs.append(_lib.TcJob(head, rows, ldx, 1, ldx, X.data_ptr(), Y.data_ptr(), dY.data_ptr(), dX.data_ptr()))
    keep.append((rows, d_in, X, W1, b1, W2, b2, dY, Y, dX, grads, imgs))
  for first in (0, 2):
    arr = (_lib.TcJob * 2)(*jobs[first:first + 2])
    _lib.check(lib.mz_heads_forward_tc(2, arr, None), "fwd")
    _lib.check(lib.mz_heads_backward_tc(2, arr, None), "bwd")
  torch.cuda.synchronize()
  for rows, d_in, X, W1, b1, W2, b2, dY, Y, dX, grads, _ in keep:
    x64 = bf(X[:, :d_in]).requires_grad_(True)
    w1, w2 = bf(W1).requires_grad_(True), bf(W2).requires_grad_(True)
    bb1, bb2 = b1.double().requires_grad_(True), b2.double().requires_grad_(True)
    y64 = torch.relu(x64 @ w1.t() + bb1) @ w2.t() + bb2
    y64.backward(bf(dY))
    assert _rel(Y, y64) <= 1e-2, (rows, d_in, _rel(Y, y64))
    for got, want, name in ((dX[:, :d_in] - 1.0, x64.grad, "dX"), (grads[0], w1.grad, "gW1"), (grads[1], bb1.grad, "gb1"),
                            (grads[2], w2.grad, "gW2"), (grads[3], bb2.grad, "gb2")):
      assert _rel(got, want) <= 1.5e-2, (rows, d_in, name, _rel(got, want))
    assert (dX[:, d_in:] == 1.0).all()


@pytest.mark.gpu
def test_mlp2_kernels_one_output_column():
  """mz_mlp2_forward / mz_mlp2_backward for a one-unit head (d_out = 1, ldy = 1) on ragged row counts, wide inputs and
  strided rows: against the float64 head, with the bars of test_mlp2_kernels_ragged_rows_match_torch."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  P = lambda t: C.c_void_p(t.data_ptr())
  rng = torch.Generator(device="cuda").manual_seed(6)
  for rows, d_in, ldx in ((1, 9, 9), (45, 54, 54), (100, 128, 130), (33, 50, 59)):
    X = torch.randn(rows, ldx, device="cuda", generator=rng)
    W1, b1 = torch.randn(512, d_in, device="cuda", generator=rng) * 0.1, torch.randn(512, device="cuda", generator=rng) * 0.1
    W2, b2 = torch.randn(1, 512, device="cuda", generator=rng) * 0.1, torch.randn(1, device="cuda", generator=rng)
    W1T, W2T = W1.t().contiguous(), W2.t().contiguous()
    Y = torch.full((rows, 1), 7.0, device="cuda")
    _lib.check(lib.mz_mlp2_forward(rows, d_in, ldx, P(X), P(W1T), P(b1), P(W2T), P(b2), 1, P(Y), 1, None), "fwd")
    x64 = X[:, :d_in].double().requires_grad_(True)
    w1, bb1, w2, bb2 = [t.double().requires_grad_(True) for t in (W1, b1, W2, b2)]
    y64 = torch.relu(x64 @ w1.t() + bb1) @ w2.t() + bb2
    torch.cuda.synchronize()
    assert torch.allclose(Y.double(), y64, rtol=1e-4, atol=1e-4), (rows, d_in)
    dY = torch.randn(rows, 1, device="cuda", generator=rng)
    y64.backward(dY.double())
    dX = torch.ones(rows, ldx, device="cuda")
    gW1, gb1, gW2, gb2 = torch.zeros_like(W1), torch.zeros_like(b1), torch.zeros_like(W2), torch.zeros_like(b2)
    _lib.check(lib.mz_mlp2_backward(rows, d_in, ldx, P(X), P(W1T), P(b1), P(W1), P(W2), 1, P(dY), 1, P(dX), ldx,
                                    P(gW1), P(gb1), P(gW2), P(gb2), None), "bwd")
    torch.cuda.synchronize()
    for got, want, name in ((dX[:, :d_in] - 1.0, x64.grad, "dX"), (gW1, w1.grad, "gW1"), (gb1, bb1.grad, "gb1"),
                            (gW2, w2.grad, "gW2"), (gb2, bb2.grad, "gb2")):
      scale = want.abs().max().item() + 1e-12
      assert (got.double() - want).abs().max().item() <= 1e-4 * scale, (rows, d_in, name)
    assert (dX[:, d_in:] == 1.0).all()


@pytest.mark.gpu
def test_fused_network_has_the_reference_no_support_state_dict():
  from model_based_rl_b200 import learners
  g = helpers.load("learner_nosupport_mse")
  cfg = _ns_config(g)
  net, _ = _nets(g, cfg)
  ref = learners.FCNetworkTrain(int(g["obs_dim"]), int(g["action_space"]), "cpu", cfg)
  assert {k: tuple(v.shape) for k, v in net.state_dict().items()} == {k: tuple(v.shape) for k, v in ref.state_dict().items()}
  assert tuple(net.state_dict()["value_head.value.weight"].shape) == (1, 512)


@pytest.mark.gpu
def test_fused_learner_rejects_unknown_scalar_loss():
  from model_based_rl_b200 import fused_learner
  g = helpers.load("learner_nosupport_mse")
  cfg = _ns_config(g)
  net, _ = _nets(g, cfg)
  cfg.scalar_loss = "L1"
  with pytest.raises(NotImplementedError):
    fused_learner.FusedLearner(cfg, net)


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True], ids=["eager", "cuda_graph"])
@pytest.mark.parametrize("case", CASES)
def test_f32_no_support_learner_two_steps_match_reference_golden(case, graph):
  """precision='f32', two steps against the reference's FCNetwork(no_support=True) run: losses 1e-4 relative, priority
  errors 1e-4 absolute, every weight 2e-5 absolute (AdamW with the h-transform; RMSprop with clipping and
  no_target_transform)."""
  from model_based_rl_b200 import fused_learner
  g = helpers.load("learner_" + case)
  cfg = _ns_config(g)
  net, _ = _nets(g, cfg)
  learner = fused_learner.FusedLearner(cfg, net, use_graph=graph, precision="f32")
  for step in range(2):
    losses = learner.update_weights(_batch(g, step))
    np.testing.assert_allclose(losses.cpu().numpy(), g["s%d_losses" % step], rtol=1e-4)
    np.testing.assert_allclose(learner.last_errors.cpu().numpy(), g["s%d_new_errors" % step], rtol=0, atol=1e-4)
    for k, v in net.state_dict().items():
      np.testing.assert_allclose(_sub(v.detach().cpu()).numpy(), g["s%d_w_%s" % (step, k)], rtol=0, atol=2e-5,
                                 err_msg="step %d %s" % (step, k))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_f32_no_support_gradients_match_autograd(case):
  """Every parameter gradient of one f32 step against autograd through FCNetworkTrain + scalar_unroll_loss: 2e-4 of
  each tensor's scale."""
  from model_based_rl_b200 import fused_learner, learners
  torch.backends.cuda.matmul.allow_tf32 = False
  g = helpers.load("learner_" + case)
  cfg = _ns_config(g)
  net, ref = _nets(g, cfg)
  fused = fused_learner.FusedLearner(cfg, net, use_graph=False, precision="f32")
  fused._stage(_batch(g, 0))
  fused._forward_and_heads_backward()
  fused._recurrent_backward()
  torch_learner = learners.Learner(cfg, ref)
  assert torch_learner.loss_fn is learners.scalar_unroll_loss
  inputs = (fused.s_obs, fused.s_actions.long(), fused.s_tv, fused.s_tr, fused.s_tp, fused.s_isw)
  losses, errs = torch_learner._forward_backward(*inputs)
  torch.cuda.synchronize()
  np.testing.assert_allclose(fused.losses.cpu().numpy(), losses.cpu().numpy(), rtol=1e-5)
  np.testing.assert_allclose(fused.new_errors.cpu().numpy(), errs.cpu().numpy(), rtol=0, atol=1e-4)
  for name, p in ref.named_parameters():
    want, got = p.grad.cpu().numpy(), net.grads[name].cpu().numpy()
    scale = np.abs(want).max() + 1e-12
    assert np.abs(got - want).max() <= 2e-4 * scale, (name, np.abs(got - want).max(), scale)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_bf16_no_support_step_equals_autograd_with_the_same_rounding_points(case):
  """The tensor-core launches of a no_support step against float64 autograd through heads that round to bf16 where
  the kernels do (test_fused_learner._teacher_forced_check): outputs within 2e-3, gradients within 3e-3."""
  from model_based_rl_b200 import fused_learner
  g = helpers.load("learner_" + case)
  cfg = _ns_config(g)
  net, _ = _nets(g, cfg)
  fused = fused_learner.FusedLearner(cfg, net, use_graph=False)
  fused._stage(_batch(g, 0))
  fused._forward_and_heads_backward()
  fused._recurrent_backward()
  torch.cuda.synchronize()
  worst = _teacher_forced_check(fused, net, 2e-3, 3e-3)
  print(case, "vs emulation", {k: round(x, 5) for k, x in worst.items()})


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_bf16_no_support_gradients_point_like_the_f32_step(case):
  """Parameter gradients of the bf16 step against the f32 step on the same weights and batch: cosine >= 0.98 per
  tensor."""
  from model_based_rl_b200 import fused_learner
  g = helpers.load("learner_" + case)
  cfg = _ns_config(g)
  out = {}
  for prec in ("f32", "bf16"):
    net, _ = _nets(g, cfg)
    fused = fused_learner.FusedLearner(cfg, net, use_graph=False, precision=prec)
    fused._stage(_batch(g, 0))
    fused._forward_and_heads_backward()
    fused._recurrent_backward()
    torch.cuda.synchronize()
    out[prec] = net
  cos = {}
  for k, want in out["f32"].grads.items():
    a, b = out["bf16"].grads[k].double().flatten(), want.double().flatten()
    cos[k] = float((a @ b) / (a.norm() * b.norm() + 1e-300))
  print(case, "cosine vs f32", {k: round(x, 4) for k, x in cos.items()})
  assert min(cos.values()) >= 0.98, cos


@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True], ids=["eager", "cuda_graph"])
@pytest.mark.parametrize("case", CASES)
def test_bf16_no_support_learner_two_steps_against_reference_golden(case, graph):
  """Two steps of the bf16 learner against the golden run: losses 2e-2 relative, weights within 2.5 learning rates
  per step taken."""
  from model_based_rl_b200 import fused_learner
  g = helpers.load("learner_" + case)
  cfg = _ns_config(g)
  net, _ = _nets(g, cfg)
  learner = fused_learner.FusedLearner(cfg, net, use_graph=graph)
  assert learner.precision == "bf16"
  for step in range(2):
    losses = learner.update_weights(_batch(g, step))
    np.testing.assert_allclose(losses.cpu().numpy(), g["s%d_losses" % step], rtol=2e-2)
    bar = 2.5 * cfg.lr_init * (step + 1)
    for k, v in net.state_dict().items():
      np.testing.assert_allclose(_sub(v.detach().cpu()).numpy(), g["s%d_w_%s" % (step, k)], rtol=0, atol=bar,
                                 err_msg="step %d %s" % (step, k))


@pytest.mark.gpu
@pytest.mark.parametrize("precision,scalar_loss", [("bf16", "MSE"), ("f32", "Huber")])
def test_no_support_learn_with_replay_feedback_and_search_hand_off(precision, scalar_loss):
  """learn() on a no_support config: priorities come back from the device, the weights handed to the search
  network (tf32x3 for such networks) equal the learner's, and that network's outputs equal FCNetworkTrain's on the
  same weights (rtol 1e-4, atol 2e-5)."""
  from model_based_rl_b200 import fused_learner, learners
  from model_based_rl_b200.networks import FCNetwork
  from model_based_rl_b200.replay_buffer import PrioritizedReplay
  from model_based_rl_b200.selfplay import HistorySlice
  torch.backends.cuda.matmul.allow_tf32 = False
  D, A, K = 8, 4, 3
  cfg = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=True, scalar_loss=scalar_loss,
                              no_target_transform=False, num_unroll_steps=K, td_steps=5, optimizer="AdamW", lr_init=0.001,
                              momentum=0.9, weight_decay=1e-4, clip_grad=0, lr_scheduler="ExponentialLR",
                              lr_decay_rate=0.99, norm_obs=False, batch_size=64, beta_increment_per_sampling=0.001,
                              epsilon=0.01, alpha=1.0, beta=0.5, discount=0.997, action_space=A, obs_space=(D,),
                              window_size=2000, window_step=None, seed=None, send_weights_frequency=3, training_steps=7,
                              stored_before_train=100)
  rb = PrioritizedReplay(cfg)
  r2 = np.random.default_rng(6)
  for _ in range(8):
    n = int(r2.integers(50, 300))
    rb.save_history(HistorySlice(list(r2.normal(size=(n, D)).astype(np.float32)), r2.random((n, A)).tolist(),
                                 r2.normal(size=n).tolist(), r2.integers(0, A, size=n).tolist(), r2.normal(size=n).tolist(),
                                 np.abs(r2.normal(size=n)).tolist(), [False] * n, list(range(n)), [None] * n, [1] * n),
                    ignore=None, terminal=True)
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  search_net = FCNetwork(D, A, "cuda", cfg)
  assert search_net.precision == "tf32x3"
  learner = fused_learner.FusedLearner(cfg, net, replay_buffer=rb, search_network=search_net, precision=precision)
  before = rb.index.tree.clone()
  w0 = net.flat.clone()
  assert learner.learn() == 7
  torch.cuda.synchronize()
  assert not torch.equal(rb.index.tree, before)
  assert not torch.equal(net.flat, w0) and torch.isfinite(net.flat).all()
  learner.send_weights()  # the last hand-off of learn() was at step 6
  handed = search_net.get_weights()
  for k, v in net.state_dict().items():
    assert torch.equal(handed[k].cpu(), v.cpu()), k
  train = learners.FCNetworkTrain(D, A, "cuda", cfg)
  train.load_weights({k: v.clone() for k, v in net.state_dict().items()})
  obs = torch.from_numpy(r2.normal(size=(37, D)).astype(np.float32)).cuda()
  acts = torch.from_numpy(r2.integers(0, A, size=37)).cuda()
  with torch.no_grad():
    t0 = train.initial_inference(obs)
    t1 = train.recurrent_inference(t0.hidden_state, acts)
  s0 = search_net.initial_inference(obs)
  s1 = search_net.recurrent_inference(t0.hidden_state, acts.to(torch.int32))
  torch.cuda.synchronize()
  for a, b in ((t0.value, s0.value), (t0.policy_logits, s0.policy_logits), (t1.value, s1.value), (t1.reward, s1.reward),
               (t1.hidden_state, s1.hidden_state)):
    assert a.shape == b.shape
    assert torch.allclose(a, b, rtol=1e-4, atol=2e-5), (a - b).abs().max().item()
