"""FusedLearner(precision='tf32x3'): the learner step on the tensor cores at float32 accuracy (csrc/mz_learner_tf32.cu,
three TF32 products on split operands per contraction).  Held to the bars of the float32 path: the reference goldens,
torch autograd, float64 per head kernel, the per-phase float32 chain kernels, learners.Learner step for step,
checkpoints across all three precisions and learners.Learner, learn() with a tf32x3 search network, and two
data-parallel ranks."""
import ctypes as C
import io
import os
import re
import subprocess
import tempfile
import types

import numpy as np
import pytest
import torch

import helpers
from test_fused_learner import _rel
from test_fused_learner_wide_obs import CSRC, _batch as _rand_batch, _cfg as _rand_cfg, _ptxas
from test_learner import CASES, _batch, _config, _sub, _weights

NS_CASES = ["nosupport_mse", "nosupport_huber"]
MZ_ERR_BAD_ARG, MZ_ERR_UNSUPPORTED = -1, -2


def _golden_config(case):
  g = helpers.load("learner_" + case)
  cfg = _config(g)
  if "scalar_loss" in g:
    cfg.no_support, cfg.scalar_loss = True, str(g["scalar_loss"])
  return g, cfg


def _nets(g, cfg):
  from model_based_rl_b200 import fused_learner, learners
  D, A = int(g["obs_dim"]), int(g["action_space"])
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  net.load_weights(_weights(g))
  ref = learners.FCNetworkTrain(D, A, "cuda", cfg)
  ref.load_weights(_weights(g))
  return net, ref


def _close(got, want, bar):
  """All but one element in a thousand within `bar` of the largest entry, every element within 20 x bar (a hidden unit
  whose pre-activation is within float32 rounding of zero is gated differently by a float32 and a float64 sum)."""
  err = (got.detach().double() - want.detach().double()).abs().flatten() / (want.detach().double().abs().max() + 1e-12)
  k = max(1, int(err.numel() * 0.999))
  return float(err.kthvalue(k).values) <= bar and float(err.max()) <= 20 * bar


# -- without a GPU ----------------------------------------------------------------------------------------------
def test_tf32x3_learner_kernels_compile_without_spills_on_tf32_mma():
  """Every kernel of mz_learner_tf32.cu compiles for sm_100a without spills, and its SASS multiplies on the TF32
  tensor-core path only (no bf16 MMA)."""
  from model_based_rl_b200 import _lib
  kernels = _ptxas("mz_learner_tf32.cu")
  assert len(kernels) == 11, sorted(kernels)  # pack, heads_fwd x 2, heads_bwd x 2, chain_fwd x 4, chain_bwd x 2
  assert all(v == 0 for v in kernels.values()), kernels
  nvcc = _lib.nvcc_path()
  cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")
  with tempfile.TemporaryDirectory() as d:
    obj = os.path.join(d, "k.o")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                    "-I" + os.path.join(CSRC, "..", "..", "include"), "-I" + CSRC, "-DMZ_BUILDING", "-c",
                    os.path.join(CSRC, "mz_learner_tf32.cu"), "-o", obj], check=True, capture_output=True)
    sass = subprocess.run([cuobjdump, "-sass", obj], check=True, capture_output=True, text=True).stdout
  mma = set(re.findall(r"HMMA\.[0-9A-Z.]+", sass))
  assert mma and all(m.endswith(".F32.TF32") for m in mma), mma


def _head(_lib, d_in, d_out):
  p = [256 * (i + 1) for i in range(10)]  # never dereferenced: the shape is refused first
  return _lib.TcHead(*p, d_in, d_out)


def test_tf32x3_c_abi_refuses_unsupported_shapes_and_bad_arguments_without_a_gpu():
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  assert lib.mz_learner_packed_words_tf32x3(512, 68) == 64 * 9 * 128
  assert lib.mz_learner_packed_words_tf32x3(1, 512) == 64 * 128
  assert lib.mz_learner_packed_words_tf32x3(0, 8) == 0
  for d_in, d_out, dx, want in ((1025, 50, None, MZ_ERR_UNSUPPORTED), (50, 65, None, MZ_ERR_UNSUPPORTED),
                                (200, 50, 8192, MZ_ERR_BAD_ARG), (0, 50, None, MZ_ERR_BAD_ARG)):
    job = _lib.TcJob(_head(_lib, d_in, d_out), 1, max(d_in, 1), d_out, max(d_in, 1), 4096, 4096, 4096, dx)
    arr = (_lib.TcJob * 1)(job)
    if dx is None:
      assert lib.mz_heads_forward_tf32x3(1, arr, None) == want, (d_in, d_out)
    assert lib.mz_heads_backward_tf32x3(1, arr, None) == want, (d_in, d_out)
  assert lib.mz_heads_forward_tf32x3(4, arr, None) == MZ_ERR_BAD_ARG  # at most three jobs
  assert lib.mz_learner_pack_tf32x3(0, None, None) == MZ_ERR_BAD_ARG
  for first_in, A, want in ((1025, 18, MZ_ERR_UNSUPPORTED), (8, 79, MZ_ERR_UNSUPPORTED), (8, 18, MZ_ERR_BAD_ARG)):
    chain = _lib.TcChain(_head(_lib, first_in, 50), _head(_lib, 50 + A, 50), 16, 2, 50, A, 4096, first_in, None, 1, 1,
                         4096, 4096, None, 50 + A, 4096, 4096, 4096, None, None, 0.5, None, None, None)  # xs NULL
    assert lib.mz_chain_forward_tf32x3(C.byref(chain), None) == want, (first_in, A)


# -- on the GPU: the reference goldens and autograd --------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("graph", [False, True], ids=["eager", "cuda_graph"])
@pytest.mark.parametrize("case", CASES + NS_CASES)
def test_tf32x3_learner_two_steps_match_reference_golden(case, graph):
  """The f32 path's bars, two steps: losses 1e-4 relative, priority errors 2e-3 absolute (1e-4 for the --no_support
  cases, as there), every weight 2e-5 absolute -- RMSprop (breakout), AdamW with clipping on the library's Adam kernel
  (ttt), SGD without target transform (lunar_raw), and the MSE / Huber --no_support networks."""
  from model_based_rl_b200 import fused_learner
  g, cfg = _golden_config(case)
  net, _ = _nets(g, cfg)
  learner = fused_learner.FusedLearner(cfg, net, use_graph=graph, precision="tf32x3")
  err_bar = 1e-4 if case in NS_CASES else 2e-3
  for step in range(2):
    losses = learner.update_weights(_batch(g, step))
    np.testing.assert_allclose(losses.cpu().numpy(), g["s%d_losses" % step], rtol=1e-4)
    np.testing.assert_allclose(learner.last_errors.cpu().numpy(), g["s%d_new_errors" % step], rtol=0, atol=err_bar)
    for k, v in net.state_dict().items():
      np.testing.assert_allclose(_sub(v.detach().cpu()).numpy(), g["s%d_w_%s" % (step, k)], rtol=0, atol=2e-5,
                                 err_msg="step %d %s" % (step, k))


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES + NS_CASES)
def test_tf32x3_gradients_match_autograd(case):
  """Every parameter gradient of one step against torch autograd in float32 (allow_tf32 off) through
  FCNetworkTrain.unroll and the same loss: 2e-4 of each tensor's largest entry, the bar of the f32 step; losses 1e-5
  relative; priority errors within the golden bar of 2e-3 (they pass the value through the inverse h-transform, which
  turns float32 sums in another order into up to 1.7e-4 at a value of 10)."""
  from model_based_rl_b200 import fused_learner, learners
  torch.backends.cuda.matmul.allow_tf32 = False
  g, cfg = _golden_config(case)
  net, ref = _nets(g, cfg)
  fused = fused_learner.FusedLearner(cfg, net, use_graph=False, precision="tf32x3")
  fused._stage(_batch(g, 0))
  fused._forward_and_heads_backward()
  fused._recurrent_backward()
  torch_learner = learners.Learner(cfg, ref)
  inputs = (fused.s_obs, fused.s_actions.long(), fused.s_tv, fused.s_tr, fused.s_tp, fused.s_isw)
  losses, errs = torch_learner._forward_backward(*inputs)
  torch.cuda.synchronize()
  np.testing.assert_allclose(fused.losses.cpu().numpy(), losses.cpu().numpy(), rtol=1e-5)
  np.testing.assert_allclose(fused.new_errors.cpu().numpy(), errs.cpu().numpy(), rtol=0, atol=2e-3)
  for name, p in ref.named_parameters():
    want, got = p.grad.cpu().numpy(), net.grads[name].cpu().numpy()
    scale = np.abs(want).max() + 1e-12
    assert np.abs(got - want).max() <= 2e-4 * scale, (name, np.abs(got - want).max(), scale)


# -- on the GPU: the kernels -------------------------------------------------------------------------------------
HEADS = [(50, 31), (50, 64), (50, 1), (68, 50), (68, 31), (114, 50), (128, 64), (129, 50), (512, 50), (1024, 50)]


@pytest.mark.gpu
@pytest.mark.parametrize("d_in,d_out", HEADS, ids=["%dx%d" % s for s in HEADS])
def test_tf32x3_head_kernels_match_float64(d_in, d_out):
  """mz_heads_forward_tf32x3 / mz_heads_backward_tf32x3 at 1, 33, 100 and 513 rows (strided rows at odd counts), with
  dX wherever the head has one, against float64 autograd on the float32 operands: outputs within 1e-5 of their largest
  entry, dX and the four parameter gradients within 1e-5 for 99.9 % of the elements and 2e-4 for all."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  rng = torch.Generator(device="cuda").manual_seed(d_in * 100 + d_out)
  for rows in (1, 33, 100, 513):
    ldx = d_in + (3 if rows % 2 else 0)
    X = torch.randn(rows, ldx, device="cuda", generator=rng)
    W1, b1 = torch.randn(512, d_in, device="cuda", generator=rng) * 0.1, torch.randn(512, device="cuda", generator=rng) * 0.1
    W2, b2 = torch.randn(d_out, 512, device="cuda", generator=rng) * 0.1, torch.randn(d_out, device="cuda", generator=rng)
    dY = torch.randn(rows, d_out, device="cuda", generator=rng)
    Y = torch.full((rows, d_out), 7.0, device="cuda")
    with_dx = d_in <= 128
    dX = torch.ones(rows, ldx, device="cuda") if with_dx else None
    grads = [torch.zeros_like(t) for t in (W1, b1, W2, b2)]
    shapes = [(512, d_in), (d_out, 512), (512, d_out), (d_in, 512)][:4 if with_dx else 3]
    srcs = [(W1, d_in, 1), (W2, 512, 1), (W2, 1, 512), (W1, 1, d_in)]
    imgs, pj = [], []
    for (n, k), (src, sn, sk) in zip(shapes, srcs):
      img = torch.zeros(int(lib.mz_learner_packed_words_tf32x3(n, k)), dtype=torch.int32, device="cuda")
      imgs.append(img)
      pj.append(_lib.PackJob(src.data_ptr(), img.data_ptr(), n, k, sn, sk))
    _lib.check(lib.mz_learner_pack_tf32x3(len(pj), (_lib.PackJob * len(pj))(*pj), None), "pack")
    ptrs = [i.data_ptr() for i in imgs] + ([] if with_dx else [None])
    head = _lib.TcHead(*ptrs, b1.data_ptr(), b2.data_ptr(), *[t.data_ptr() for t in grads], d_in, d_out)
    arr = (_lib.TcJob * 1)(_lib.TcJob(head, rows, ldx, d_out, ldx, X.data_ptr(), Y.data_ptr(), dY.data_ptr(),
                                      dX.data_ptr() if with_dx else None))
    _lib.check(lib.mz_heads_forward_tf32x3(1, arr, None), "fwd")
    _lib.check(lib.mz_heads_backward_tf32x3(1, arr, None), "bwd")
    torch.cuda.synchronize()
    x64 = X[:, :d_in].double().requires_grad_(True)
    w1, bb1, w2, bb2 = [t.double().requires_grad_(True) for t in (W1, b1, W2, b2)]
    y64 = torch.relu(x64 @ w1.t() + bb1) @ w2.t() + bb2
    y64.backward(dY.double())
    assert _rel(Y, y64) <= 1e-5, (rows, _rel(Y, y64))
    checks = [(grads[0], w1.grad, "gW1"), (grads[1], bb1.grad, "gb1"), (grads[2], w2.grad, "gW2"), (grads[3], bb2.grad, "gb2")]
    if with_dx:
      checks.append((dX[:, :d_in] - 1.0, x64.grad, "dX"))
      assert (dX[:, d_in:] == 1.0).all()  # columns behind d_in untouched
    for got, want, name in checks:
      assert _close(got, want, 1e-5), (rows, name, _rel(got, want))


def _near_zero_rows(fused, net, tol=1e-5):
  """Batch rows in which some head's 512-wide pre-activation is within tol of its largest magnitude of zero (float64
  on the kernels' own inputs): where a float32 sum may gate the unit the other way than a float64 one."""
  K, B = fused.K, fused.B
  W = {k: v.detach().double() for k, v in net.state_dict().items()}
  xs = fused.xs.double().view(K + 1, B, -1)
  inputs = [("representation_head", fused.s_obs.double()[None])]
  if K > 0:
    inputs.append(("transition_head", xs[:K]))
    inputs.append(("reward_head", xs[:K]))
  inputs += [("value_head", xs[..., :50]), ("policy_head", xs[..., :50])]
  rows = torch.zeros(B, dtype=torch.bool, device=xs.device)
  for name, x in inputs:
    pre = (x @ W[name + ".fc1.weight"].t() + W[name + ".fc1.bias"]).abs()
    rows |= (pre < tol * pre.max()).any(-1).any(0)
  return rows


def _learners(B, K, A, D, precisions, optimizer="SGD", no_support=False, seed=0):
  """FusedLearners of the given precisions on the same weights, staged with the same batch, one step's forward and
  backward run (no optimiser step).  In the tf32x3 run the logit gradients of the _near_zero_rows are zeroed after the
  loss, so that a float64 reference of its backward does not hinge on gating ties."""
  from model_based_rl_b200 import fused_learner
  cfg = _rand_cfg(K, optimizer, 0.01, no_support)
  torch.manual_seed(seed)
  w = None
  out = {}
  dlogits = None
  for prec in precisions:
    net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
    if w is None:
      w = {k: v.clone() for k, v in net.state_dict().items()}
    net.load_weights(w)
    fused = fused_learner.FusedLearner(cfg, net, use_graph=False, precision=prec)
    fused._stage(_rand_batch(B, K, A, D, seed))
    if K == 0:  # mz_unroll_loss takes K >= 1: the same fixed logit gradients for every precision instead
      if dlogits is None:
        gen = torch.Generator(device="cuda").manual_seed(seed)
        dlogits = [torch.randn(t.shape, device="cuda", generator=gen) * 1e-2 for t in (fused.dv, fused.dp)]
      fused._loss = lambda st, f=fused: (f.dv.copy_(dlogits[0]), f.dp.copy_(dlogits[1]))
    if prec == "tf32x3":
      loss = fused._loss

      def masked_loss(st, f=fused, n=net, loss=loss):
        loss(st)
        keep = (~_near_zero_rows(f, n)).float()
        for t in (f.dv, f.dp, f.dr):
          t.mul_(keep[None, :, None])
      fused._loss = masked_loss
    fused._forward_and_heads_backward()
    fused._recurrent_backward()
    torch.cuda.synchronize()
    out[prec] = (fused, net)
  return out


@pytest.mark.gpu
@pytest.mark.parametrize("B,K,A,D", [(45, 3, 4, 8), (64, 5, 18, 128), (7, 1, 9, 27), (100, 5, 64, 1024), (33, 0, 4, 16),
                                     (2500, 2, 18, 16)])
def test_tf32x3_chain_kernels_match_the_per_phase_float32_kernels(B, K, A, D):
  """mz_chain_forward_tf32x3 / mz_chain_backward_tf32x3 and the head launches around them on ragged batches, K = 0
  (fixed logit gradients: the loss kernel takes K >= 1) and 1, 64 actions with 1024 features, and 32-row chain CTAs
  (B = 2500).  The forward against the float32 per-phase launches (mz_mlp2_*, mz_ln_relu_*): pre-LayerNorm rows,
  hidden states, LayerNorm statistics, head outputs, losses.  The backward against float64 autograd teacher-forced on
  the kernels' own hidden states and logit gradients (as _teacher_forced_check does for bf16, without rounding): the
  output heads' dX (dxs), every step's LayerNorm input gradient (dyall) and every parameter gradient, LayerNorm's
  included.  All within 1e-5 of scale (99.9 % of the elements; all within 2e-4), with the batch rows that hold a
  gating tie in float64 left out of the backward (_learners).  (Against the f32 path the backward
  differs where one of the two float32 sums gates a ReLU unit the other way: a unit moves a whole row of gW1, and the
  f32 path's step-0 dy leaves the float64 chain by up to 1e-2 of scale in a few rows at B = 45 and 2500 while the
  tf32x3 one stays within 2e-6, measured on a B200.)"""
  import torch.nn.functional as F
  out = _learners(B, K, A, D, ("f32", "tf32x3"), seed=B + K)
  f32, tf = out["f32"][0], out["tf32x3"][0]
  assert torch.equal(tf.xs[:, 50:], f32.xs[:, 50:])  # one-hot actions
  for name in ("yall", "xs", "rstd", "v", "p"):
    assert _close(getattr(tf, name), getattr(f32, name), 1e-5), (name, _rel(getattr(tf, name), getattr(f32, name)))
  np.testing.assert_allclose(tf.losses.cpu().numpy(), f32.losses.cpu().numpy(), rtol=1e-5)
  net = out["tf32x3"][1]
  W = {k: v.detach().double().clone().requires_grad_(True) for k, v in net.state_dict().items()}
  head = lambda x, name, o: F.linear(torch.relu(F.linear(x, W[name + ".fc1.weight"], W[name + ".fc1.bias"])),
                                     W["%s.%s.weight" % (name, o)], W["%s.%s.bias" % (name, o)])
  x_all = tf.xs.double().clone().requires_grad_(True)
  outs = [head(x_all[:, :50], "value_head", "value"), head(x_all[:, :50], "policy_head", "policy")]
  grads = [tf.dv.view(outs[0].shape).double(), tf.dp.view(outs[1].shape).double()]
  if K > 0:
    outs.append(head(x_all[:K * B], "reward_head", "reward"))
    grads.append(tf.dr.view(-1, outs[2].shape[1]).double())
  torch.autograd.backward(outs, grads)
  assert _close(tf.dxs, x_all.grad, 1e-5), _rel(tf.dxs, x_all.grad)
  xs, dxs = tf.xs.double().view(K + 1, B, -1), tf.dxs.double().view(K + 1, B, -1)
  up = None
  for k in range(K, -1, -1):
    x_in = (xs[k - 1] if k else tf.s_obs.double()).clone().requires_grad_(True)
    y = head(x_in, "transition_head" if k else "representation_head", "out")
    y.retain_grad()
    h = torch.relu(F.layer_norm(y, (50,), W["LN.weight"], W["LN.bias"], 1e-5))
    h.backward((dxs[k][:, :50] + (up if up is not None else 0.0)) * (0.5 if k else 1.0))
    up = x_in.grad[:, :50]
    assert _close(tf.dyall[k], y.grad, 1e-5), (k, _rel(tf.dyall[k], y.grad))
  for k, w in W.items():
    if w.grad is None:  # K = 0: no dynamics step
      assert not net.grads[k].any(), k
    else:
      assert _close(net.grads[k], w.grad, 1e-5), (k, _rel(net.grads[k], w.grad))


def _against_torch(D, A, optimizer, no_support, steps=2, B=128, K=5):
  from model_based_rl_b200 import fused_learner, learners
  cfg = _rand_cfg(K, optimizer, 0.0008, no_support)
  torch.manual_seed(D + A)
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  ref = learners.FCNetworkTrain(D, A, "cuda", cfg)
  ref.load_weights({k: v.detach().cpu() for k, v in net.state_dict().items()})
  fused = fused_learner.FusedLearner(cfg, net, use_graph=True, precision="tf32x3")
  torch_learner = learners.Learner(cfg, ref)
  for step in range(steps):
    batch = _rand_batch(B, K, A, D, 100 * D + step)
    got = fused.update_weights(batch).cpu().numpy()
    want = torch_learner.update_weights(batch)
    want = want.cpu().numpy() if torch.is_tensor(want) else np.asarray(want)
    np.testing.assert_allclose(got, want, rtol=1e-4, err_msg="step %d losses" % step)
    torch.cuda.synchronize()
    wref = ref.state_dict()
    for k, v in net.state_dict().items():
      np.testing.assert_allclose(v.detach().cpu().numpy(), wref[k].detach().cpu().numpy(), rtol=0, atol=2e-5,
                                 err_msg="step %d %s" % (step, k))


@pytest.mark.gpu
@pytest.mark.parametrize("D,A,optimizer,no_support", [(1024, 64, "SGD", False), (147, 18, "SGD", True)],
                         ids=["a64_d1024_sgd", "d147_sgd_no_support"])
def test_tf32x3_learner_two_steps_match_torch_learner(D, A, optimizer, no_support):
  """Two captured steps against learners.Learner (torch modules, float32) from the same weights and batches: losses
  1e-4 relative, every weight 2e-5 absolute -- 64 actions on 1024-feature observations, and a --no_support network.
  Both step with SGD, as test_f32_learner_wide_obs_two_steps_match_torch_learner does for --no_support: Adam divides
  by sqrt(v) + 1.5e-4, which turns the last float32 bits of a near-zero gradient (summed in another order than torch's)
  into up to 5.3 times as much weight change -- at A = 64 with AdamW, 23 of the reward head's 58 368 first-layer
  weights land between 2e-5 and 6.2e-5 after the second step (measured on a B200).  The reference goldens hold the
  Adam path (ttt) at 2e-5."""
  _against_torch(D, A, optimizer, no_support)


# -- on the GPU: the learner around the kernels ------------------------------------------------------------------
@pytest.mark.gpu
def test_tf32x3_images_only_for_a_tf32x3_learner():
  """FusedFCNetwork keeps its bf16 images as they were and allocates the hi / lo TF32 images when the first tf32x3
  learner is built; an unknown precision is refused with the three names."""
  from model_based_rl_b200 import fused_learner
  cfg = _rand_cfg(3)
  net = fused_learner.FusedFCNetwork(24, 18, "cuda", cfg)
  bf16_words = net.packed.numel()
  fused_learner.FusedLearner(cfg, net, precision="bf16")
  assert net.packed_tf32x3 is None
  fused_learner.FusedLearner(cfg, net, precision="tf32x3")
  assert net.packed.numel() == bf16_words and net.packed_tf32x3 is not None
  assert len(net.heads["value_head"].images_tf32x3) == 4
  with pytest.raises(ValueError, match="tf32x3"):
    fused_learner.FusedLearner(cfg, net, precision="fp16")


def _run(learner, batches):
  for b in batches:
    learner.update_weights(b)
  torch.cuda.synchronize()
  return {k: v.detach().cpu().clone() for k, v in learner.network.state_dict().items()}


@pytest.mark.gpu
@pytest.mark.parametrize("case,optimizer", [("ttt", "AdamW"), ("breakout", "RMSprop")])
def test_tf32x3_checkpoints_resume_on_every_learner_and_back(case, optimizer):
  """Two tf32x3 steps, save_state, then the run resumes on FusedLearner bf16 / f32 and (AdamW) on learners.Learner;
  the f32 and torch continuations agree with a tf32x3 continuation within 2e-5, the bf16 one's losses within 2e-2 (the bf16
  learner's bar against the goldens).  The other way
  round: after resuming from an f32 checkpoint the next tf32x3 step equals the f32 learner's next step within 2e-5."""
  from model_based_rl_b200 import fused_learner, learners
  g, cfg = _golden_config(case)
  cfg.optimizer = optimizer
  D, A = int(g["obs_dim"]), int(g["action_space"])
  b0, b1 = _batch(g, 0), _batch(g, 1)

  def fused(prec, state=None, graph=True):
    net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
    net.load_weights(_weights(g))
    return fused_learner.FusedLearner(cfg, net, use_graph=graph, precision=prec, state=state)

  def saved(learner):  # through bytes, as a file would: save_state hands out the torch optimiser's live tensors
    buf = io.BytesIO()
    torch.save(learner.save_state(), buf)
    buf.seek(0)
    return torch.load(buf, weights_only=False)

  tf = fused("tf32x3")
  _run(tf, [b0, b1])
  state = saved(tf)
  assert state["training_step"] == tf.training_step
  want = _run(tf, [b0])  # the tf32x3 run continued
  got = _run(fused("f32", state=state), [b0])
  for k in want:
    np.testing.assert_allclose(got[k].numpy(), want[k].numpy(), rtol=0, atol=2e-5, err_msg="f32 %s" % k)
  bf = fused("bf16", state=state)
  _run(bf, [b0])
  assert bf.training_step == state["training_step"]
  np.testing.assert_allclose(bf.last_losses.cpu().numpy(), tf.last_losses.cpu().numpy(), rtol=2e-2)
  if optimizer == "AdamW":  # (learners.Learner resuming torch RMSprop state is the checkpoint interop tests' subject)
    ref = learners.FCNetworkTrain(D, A, "cuda", cfg)
    ref.load_weights(_weights(g))
    torch.backends.cuda.matmul.allow_tf32 = False
    torch_learner = learners.Learner(cfg, ref, state=state)
    torch_learner.update_weights(b0)
    torch.cuda.synchronize()
    for k, v in ref.state_dict().items():
      np.testing.assert_allclose(v.detach().cpu().numpy(), want[k].numpy(), rtol=0, atol=2e-5, err_msg="torch %s" % k)
  # and back: an f32 run resumed at tf32x3
  f32 = fused("f32")
  _run(f32, [b0, b1])
  state = saved(f32)
  want = _run(f32, [b1])
  got = _run(fused("tf32x3", state=state), [b1])
  for k in want:
    np.testing.assert_allclose(got[k].numpy(), want[k].numpy(), rtol=0, atol=2e-5, err_msg="f32 -> tf32x3 %s" % k)


@pytest.mark.gpu
def test_tf32x3_learn_with_replay_feedback_and_a_tf32x3_search_network():
  """learn(): sample_batch_device(ring) -> tf32x3 update_weights -> priorities fed back on the device, and the weight
  hand-off into FCNetwork(precision='tf32x3'), whose initial inference then gives the learner's representation."""
  import torch.nn.functional as F
  from model_based_rl_b200 import fused_learner
  from model_based_rl_b200.networks import FCNetwork
  from model_based_rl_b200.replay_buffer import PrioritizedReplay
  from model_based_rl_b200.selfplay import HistorySlice
  D, A, K = 8, 4, 3
  cfg = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=False, no_target_transform=False,
                              num_unroll_steps=K, td_steps=5, optimizer="AdamW", lr_init=0.001, momentum=0.9,
                              weight_decay=1e-4, clip_grad=0, lr_scheduler="ExponentialLR", lr_decay_rate=0.99, norm_obs=False,
                              batch_size=64, beta_increment_per_sampling=0.001, epsilon=0.01, alpha=1.0, beta=0.5, discount=0.997,
                              action_space=A, obs_space=(D,), window_size=2000, window_step=None, seed=None,
                              send_weights_frequency=3, training_steps=7, stored_before_train=100)
  rb = PrioritizedReplay(cfg)
  r2 = np.random.default_rng(5)
  for _ in range(8):
    n = int(r2.integers(50, 300))
    rb.save_history(HistorySlice(list(r2.normal(size=(n, D)).astype(np.float32)), r2.random((n, A)).tolist(),
                                 r2.normal(size=n).tolist(), r2.integers(0, A, size=n).tolist(), r2.normal(size=n).tolist(),
                                 np.abs(r2.normal(size=n)).tolist(), [False] * n, list(range(n)), [None] * n, [1] * n),
                    ignore=None, terminal=True)
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  search_net = FCNetwork(D, A, "cuda", cfg, precision="tf32x3")
  learner = fused_learner.FusedLearner(cfg, net, replay_buffer=rb, search_network=search_net, precision="tf32x3")
  assert learner.use_graph
  before = rb.index.tree.clone()
  w0 = net.flat.clone()
  assert learner.learn() == 7
  torch.cuda.synchronize()
  assert not torch.equal(rb.index.tree, before)          # priorities came back
  assert not torch.equal(net.flat, w0) and torch.isfinite(net.flat).all()
  assert abs(learner.lr_scheduler.lr - 0.001 * 0.99 ** 7) < 1e-12
  learner.send_weights()
  for k, v in net.state_dict().items():
    assert torch.equal(search_net.get_weights()[k].cpu(), v.cpu()), k
  obs = torch.from_numpy(r2.normal(size=(64, D)).astype(np.float32)).cuda()
  hidden = search_net.initial_inference(obs).hidden_state
  W = net.state_dict()
  y = F.linear(F.relu(F.linear(obs, W["representation_head.fc1.weight"], W["representation_head.fc1.bias"])),
               W["representation_head.out.weight"], W["representation_head.out.bias"])
  want = F.relu(F.layer_norm(y, (50,), W["LN.weight"], W["LN.bias"], 1e-5))
  assert _rel(hidden, want) <= 1e-4


def _dp_worker(rank, world_size, port, out):
  """One of two data-parallel tf32x3 FusedLearner ranks (both on cuda:0, gloo): rank r trains on the golden batch of
  step r with AdamW, captured in CUDA graphs."""
  import torch.distributed as dist
  os.environ["MASTER_ADDR"] = "127.0.0.1"
  os.environ["MASTER_PORT"] = str(port)
  dist.init_process_group("gloo", rank=rank, world_size=world_size)
  try:
    from model_based_rl_b200 import fused_learner
    g, cfg = _golden_config("ttt")
    cfg.optimizer, cfg.clip_grad = "AdamW", 0
    net, _ = _nets(g, cfg)
    if rank == 1:  # ranks start from different weights: send_weights must align them
      net.flat.add_(0.01)
    learner = fused_learner.FusedLearner(cfg, net, use_graph=True, precision="tf32x3")
    learner.send_weights()
    learner.update_weights(_batch(g, rank))
    torch.cuda.synchronize()
    mine = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
    # single-process restatement: the gradients of both batches summed, the same optimiser step with scale 1 / 2
    solo_net, _ = _nets(g, cfg)
    solo = fused_learner.FusedLearner(cfg, solo_net, use_graph=False, precision="tf32x3")
    total = torch.zeros_like(solo_net.grad)
    for r in range(world_size):
      solo._stage(_batch(g, r))
      solo._forward_and_heads_backward()
      solo._recurrent_backward()
      total += solo_net.grad
    solo_net.grad.copy_(total)
    solo._apply(world_size)
    torch.cuda.synchronize()
    for k, v in solo_net.state_dict().items():
      assert torch.allclose(v.cpu(), mine[k], rtol=0, atol=2e-5), (k, float((v.cpu() - mine[k]).abs().max()))
    gathered = [None] * world_size
    dist.all_gather_object(gathered, {k: v.numpy() for k, v in mine.items()})
    for k in mine:
      assert np.array_equal(gathered[0][k], gathered[1][k]), k  # every rank holds the same weights, bit for bit
    out.put((rank, "ok"))
  except Exception:  # pragma: no cover
    import traceback
    out.put((rank, traceback.format_exc()))
  finally:
    dist.destroy_process_group()


@pytest.mark.gpu
def test_tf32x3_learner_data_parallel_two_ranks():
  """Two tf32x3 ranks with the bucketed all-reduce: the same weights on both ranks bit for bit, equal within 2e-5 to
  one process applying the summed gradients of both batches (float32 sums in another order; Adam normalises)."""
  import socket
  import torch.multiprocessing as mp
  ctx = mp.get_context("spawn")
  out = ctx.Queue()
  sk = socket.socket()
  sk.bind(("127.0.0.1", 0))
  port = sk.getsockname()[1]
  sk.close()
  procs = [ctx.Process(target=_dp_worker, args=(r, 2, port, out)) for r in range(2)]
  for p in procs:
    p.start()
  res = [out.get(timeout=300) for _ in procs]
  for p in procs:
    p.join(timeout=60)
  assert sorted(res) == [(0, "ok"), (1, "ok")], res
