"""The fused learner on observations wider than one 128-feature input tile (up to 1024 features): the representation
head's layer 1 and weight gradient run over K slices of X in both precisions (csrc/mz_learner_tc.cu,
csrc/mz_learner.cu).  Kernel parity against float64, the chain, whole steps against learners.Learner, and learn()
with a replay buffer of 512-byte observations."""
import ctypes as C
import os
import re
import subprocess
import tempfile
import types

import numpy as np
import pytest
import torch

from test_fused_learner import _rel, _teacher_forced_check

MZ_ERR_BAD_ARG, MZ_ERR_UNSUPPORTED = -1, -2
WIDE = (129, 136, 147, 200, 256, 512, 1000, 1024)
ROWS = (1, 33, 100, 513)
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "model-based-rl_b200", "csrc")


def _cfg(K=5, optimizer="AdamW", lr=0.0008, no_support=False, **kw):
  c = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=no_support,
                            no_target_transform=False, num_unroll_steps=K, optimizer=optimizer, lr_init=lr, momentum=0.9,
                            weight_decay=1e-4, clip_grad=0, lr_scheduler=None, norm_obs=False, send_weights_frequency=500,
                            training_steps=2)
  if no_support:
    c.scalar_loss = "MSE"
  for k, v in kw.items():
    setattr(c, k, v)
  return c


def _batch(B, K, A, D, seed):
  r = np.random.default_rng(seed)
  pol = r.random((B, K + 1, A)).astype(np.float32)
  return ((r.normal(size=(B, D)).astype(np.float32), r.integers(0, A, size=(B, K)).tolist(),
           ((r.random((B, K + 1)) < 0.2).astype(np.float32), (3 * r.normal(size=(B, K + 1))).astype(np.float32),
            pol / pol.sum(-1, keepdims=True))), None, r.random(B))


# -- without a GPU ----------------------------------------------------------------------------------------------
def _head(lib, _lib, d_in, d_out=50):
  p = [256 * (i + 1) for i in range(10)]  # never dereferenced: the shape is refused first (16-byte aligned gradients)
  return _lib.TcHead(*p, d_in, d_out)


def test_c_abi_refuses_inputs_wider_than_1024_as_unsupported_and_dx_of_wide_heads_as_bad_arg_without_a_gpu():
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  buf = C.c_void_p(4096)
  for d_in, dx, want in ((1025, None, MZ_ERR_UNSUPPORTED), (200, 8192, MZ_ERR_BAD_ARG)):
    job = _lib.TcJob(_head(lib, _lib, d_in), 1, d_in, 50, d_in, 4096, 4096, 4096, dx)
    arr = (_lib.TcJob * 1)(job)
    if dx is None:
      assert lib.mz_heads_forward_tc(1, arr, None) == want
    assert lib.mz_heads_backward_tc(1, arr, None) == want, d_in
    # mz_mlp2_backward(rows, d_in, ldx, X, W1T, b1, W1, W2, d_out, dY, ldy, dX, lddx, gW1, gb1, gW2, gb2, stream)
    assert lib.mz_mlp2_backward(1, d_in, d_in, buf, buf, buf, buf, buf, 50, buf, 50, None if dx is None else C.c_void_p(dx),
                                d_in, buf, buf, buf, buf, None) == MZ_ERR_BAD_ARG, d_in
  assert lib.mz_mlp2_forward(1, 1025, 1025, buf, buf, buf, buf, buf, 50, buf, 50, None) == MZ_ERR_BAD_ARG
  chain = _lib.TcChain(_head(lib, _lib, 1025), _head(lib, _lib, 68), 16, 2, 50, 18, 4096, 1025, None, 1, 1, 4096, 4096,
                       4096, 68, 4096, 4096, 4096, None, None, 0.5, None, None, None)
  assert lib.mz_chain_forward_tc(C.byref(chain), None) == MZ_ERR_UNSUPPORTED


def test_fused_network_refuses_more_than_1024_features_before_touching_the_device():
  from model_based_rl_b200 import fused_learner
  with pytest.raises(ValueError, match=r"1024.*learners\.Learner"):
    fused_learner.FusedFCNetwork(1025, 18, "cuda", _cfg())


def _ptxas(src):
  from model_based_rl_b200 import _lib
  with tempfile.TemporaryDirectory() as d:
    out = subprocess.run([_lib.nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17",
                          "-I" + os.path.join(CSRC, "..", "..", "include"), "-I" + CSRC, "-DMZ_BUILDING", "-Xptxas", "-v",
                          "-c", os.path.join(CSRC, src), "-o", os.path.join(d, "k.o")],
                         capture_output=True, text=True, check=True).stderr
  kernels, cur = {}, None
  for line in out.splitlines():
    m = re.search(r"Compiling entry function '(\S+)'", line)
    if m:
      cur = m.group(1)
    m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
    if m and cur:
      kernels[cur] = int(m.group(1)) + int(m.group(2))
  return kernels


def test_learner_kernels_compile_for_sm100a_without_spills():
  """Every learner kernel that reads a wide head -- the float32 head kernels and the wide (Lb1) tensor-core
  instantiations -- compiles without spills.  heads_bwd_kernel<2, false>, the narrow two-tile backward, keeps the
  32-byte spill it has had since it was written (its SASS is unchanged by the wide instantiations)."""
  f32 = _ptxas("mz_learner.cu")
  tc = _ptxas("mz_learner_tc.cu")
  assert any("mlp2_backward" in k for k in f32) and any("mlp2_forward" in k for k in f32)
  assert all(v == 0 for k, v in f32.items()), f32
  wide = {k: v for k, v in tc.items() if "Lb1E" in k}
  assert len(wide) == 5, sorted(tc)  # heads_fwd, heads_bwd x 2, chain_fwd x 2
  assert all(v == 0 for v in wide.values()), wide
  assert all(v == 0 for k, v in tc.items() if "heads_bwd_kernelILi2ELb0" not in k), tc


# -- on the GPU -------------------------------------------------------------------------------------------------
def _tc_job(lib, _lib, rng, rows, d_in, d_out, ldx, with_dx, keep):
  X = torch.randn(rows, ldx, device="cuda", generator=rng)
  W1, b1 = torch.randn(512, d_in, device="cuda", generator=rng) * 0.1, torch.randn(512, device="cuda", generator=rng) * 0.1
  W2, b2 = torch.randn(d_out, 512, device="cuda", generator=rng) * 0.1, torch.randn(d_out, device="cuda", generator=rng)
  dY = torch.randn(rows, d_out, device="cuda", generator=rng)
  Y = torch.full((rows, d_out), 7.0, device="cuda")
  dX = torch.ones(rows, ldx, device="cuda") if with_dx else None
  grads = [torch.zeros_like(t) for t in (W1, b1, W2, b2)]
  shapes = [(512, d_in), (d_out, 512), (512, d_out), (d_in, 512)]
  srcs = [(W1, d_in, 1), (W2, 512, 1), (W2, 1, 512), (W1, 1, d_in)]
  if d_in > 128:  # no dX image for a wide head
    shapes, srcs = shapes[:3], srcs[:3]
  imgs, pj = [], []
  for (n, k), (src, sn, sk) in zip(shapes, srcs):
    img = torch.zeros(int(lib.mz_learner_packed_words(n, k)), dtype=torch.int32, device="cuda")
    imgs.append(img)
    pj.append(_lib.PackJob(src.data_ptr(), img.data_ptr(), n, k, sn, sk))
  _lib.check(lib.mz_learner_pack(len(pj), (_lib.PackJob * len(pj))(*pj), None), "pack")
  ptrs = [i.data_ptr() for i in imgs] + ([None] if len(imgs) == 3 else [])
  head = _lib.TcHead(*ptrs, b1.data_ptr(), b2.data_ptr(), *[t.data_ptr() for t in grads], d_in, d_out)
  keep.append((rows, d_in, d_out, X, W1, b1, W2, b2, dY, Y, dX, grads, imgs))
  return _lib.TcJob(head, rows, ldx, d_out, ldx, X.data_ptr(), Y.data_ptr(), dY.data_ptr(), dX.data_ptr() if with_dx else None)


def _check_tc(keep):
  bf = lambda t: t.to(torch.bfloat16).double()
  for rows, d_in, d_out, X, W1, b1, W2, b2, dY, Y, dX, grads, _ in keep:
    x64 = bf(X[:, :d_in]).requires_grad_(True)
    w1, w2 = bf(W1).requires_grad_(True), bf(W2).requires_grad_(True)
    bb1, bb2 = b1.double().requires_grad_(True), b2.double().requires_grad_(True)
    y64 = torch.relu(x64 @ w1.t() + bb1) @ w2.t() + bb2
    y64.backward(bf(dY))
    assert _rel(Y, y64) <= 1e-2, (rows, d_in, d_out, _rel(Y, y64))
    checks = [(grads[0], w1.grad, "gW1"), (grads[1], bb1.grad, "gb1"), (grads[2], w2.grad, "gW2"), (grads[3], bb2.grad, "gb2")]
    if dX is not None:
      checks.append((dX[:, :d_in] - 1.0, x64.grad, "dX"))
      assert (dX[:, d_in:] == 1.0).all()
    for got, want, name in checks:
      assert _rel(got, want) <= 1.5e-2, (rows, d_in, d_out, name, _rel(got, want))


@pytest.mark.gpu
@pytest.mark.parametrize("d_in", WIDE)
def test_tc_head_kernels_wide_inputs_match_float64(d_in):
  """mz_heads_forward_tc / mz_heads_backward_tc (dx NULL) at every width and row count, each launch also carrying a
  narrow head with dX (a wide launch serves both), strided rows (ldx > d_in), and a job of 4800 rows (two 32-row tiles
  per CTA) -- against float64 on the bf16-rounded operands, the bars of the narrow head test."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  rng = torch.Generator(device="cuda").manual_seed(d_in)
  for rows in ROWS + (4800,):
    if rows == 4800 and d_in not in (147, 1024):
      continue
    keep = []
    ldx = d_in + (5 if rows % 2 else 0)
    jobs = [_tc_job(lib, _lib, rng, rows, d_in, 50, ldx, False, keep), _tc_job(lib, _lib, rng, 45, 68, 31, 70, True, keep)]
    arr = (_lib.TcJob * 2)(*jobs)
    _lib.check(lib.mz_heads_forward_tc(2, arr, None), "fwd")
    _lib.check(lib.mz_heads_backward_tc(2, arr, None), "bwd")
    torch.cuda.synchronize()
    _check_tc(keep)


@pytest.mark.gpu
@pytest.mark.parametrize("d_in", WIDE)
def test_mlp2_kernels_wide_inputs_match_float64(d_in):
  """mz_mlp2_forward / mz_mlp2_backward (dX NULL) at every width and row count, strided rows: 1e-4 of scale."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  P = lambda t: C.c_void_p(t.data_ptr())
  rng = torch.Generator(device="cuda").manual_seed(d_in + 1)
  d_out = 50
  for rows in ROWS:
    ldx = d_in + (3 if rows % 2 else 0)
    X = torch.randn(rows, ldx, device="cuda", generator=rng)
    W1, b1 = torch.randn(512, d_in, device="cuda", generator=rng) * 0.1, torch.randn(512, device="cuda", generator=rng) * 0.1
    W2, b2 = torch.randn(d_out, 512, device="cuda", generator=rng) * 0.1, torch.randn(d_out, device="cuda", generator=rng)
    W1T, W2T = torch.empty(d_in, 512, device="cuda"), torch.empty(512, d_out, device="cuda")
    _lib.check(lib.mz_learner_transpose(512, d_in, P(W1), P(W1T), None), "transpose")
    _lib.check(lib.mz_learner_transpose(d_out, 512, P(W2), P(W2T), None), "transpose")
    Y = torch.full((rows, d_out), 7.0, device="cuda")
    _lib.check(lib.mz_mlp2_forward(rows, d_in, ldx, P(X), P(W1T), P(b1), P(W2T), P(b2), d_out, P(Y), d_out, None), "fwd")
    x64 = X[:, :d_in].double()
    w1, bb1, w2, bb2 = [t.double().requires_grad_(True) for t in (W1, b1, W2, b2)]
    y64 = torch.relu(x64 @ w1.t() + bb1) @ w2.t() + bb2
    torch.cuda.synchronize()
    assert torch.equal(W1T, W1.t()) and torch.equal(W2T, W2.t())
    assert (Y.double() - y64).abs().max().item() <= 1e-4 * (y64.abs().max().item() + 1e-12), (rows, d_in)
    dY = torch.randn(rows, d_out, device="cuda", generator=rng)
    y64.backward(dY.double())
    gW1, gb1, gW2, gb2 = torch.zeros_like(W1), torch.zeros_like(b1), torch.zeros_like(W2), torch.zeros_like(b2)
    _lib.check(lib.mz_mlp2_backward(rows, d_in, ldx, P(X), P(W1T), P(b1), P(W1), P(W2), d_out, P(dY), d_out, None, 0,
                                    P(gW1), P(gb1), P(gW2), P(gb2), None), "bwd")
    torch.cuda.synchronize()
    for got, want, name in ((gW1, w1.grad, "gW1"), (gb1, bb1.grad, "gb1"), (gW2, w2.grad, "gW2"), (gb2, bb2.grad, "gb2")):
      scale = want.abs().max().item() + 1e-12
      assert (got.double() - want).abs().max().item() <= 1e-4 * scale, (rows, d_in, name)


@pytest.mark.gpu
@pytest.mark.parametrize("B,D", [(45, 147), (100, 1024), (2500, 512)])
def test_bf16_chain_with_a_wide_representation_head(B, D):
  """The tensor-core step with a wide first head at K = 5 (16-row chain CTAs at B <= 2368, 32-row CTAs above): every
  head evaluation -- the representation head's output yall[0] and the saved xs included -- and every parameter
  gradient against float64 autograd with the kernels' rounding points, on the kernels' own inputs; the saved LayerNorm
  statistics against float64 from the saved pre-LayerNorm rows."""
  from model_based_rl_b200 import fused_learner
  A, K = 18, 5
  cfg = _cfg(K)
  torch.manual_seed(D)
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  assert len(net.heads['representation_head'].images) == 3  # no dX image for the observation
  fused = fused_learner.FusedLearner(cfg, net, use_graph=False)
  fused._stage(_batch(B, K, A, D, D))
  fused._forward_and_heads_backward()
  fused._recurrent_backward()
  torch.cuda.synchronize()
  y = fused.yall.double()
  mean, var = y.mean(-1), y.var(-1, unbiased=False)
  assert (fused.mean.double() - mean).abs().max() <= 1e-5 * (y.abs().max() + 1)
  assert _rel(fused.rstd, 1.0 / torch.sqrt(var + 1e-5)) <= 1e-5
  _teacher_forced_check(fused, net, 2e-3, 3e-3)


def _f32_against_torch(D, optimizer, no_support, steps=2):
  from model_based_rl_b200 import fused_learner, learners
  A, K, B = 18, 5, 128
  cfg = _cfg(K, optimizer, 0.0008, no_support)
  torch.manual_seed(D)
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  ref = learners.FCNetworkTrain(D, A, "cuda", cfg)
  ref.load_weights({k: v.detach().cpu() for k, v in net.state_dict().items()})
  fused = fused_learner.FusedLearner(cfg, net, use_graph=True, precision="f32")
  torch_learner = learners.Learner(cfg, ref)
  for step in range(steps):
    batch = _batch(B, K, A, D, 100 * D + step)
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
@pytest.mark.parametrize("D", [147, 512, 1024])
@pytest.mark.parametrize("optimizer,no_support", [("AdamW", False), ("RMSprop", False), ("SGD", True)],
                         ids=["adamw", "rmsprop", "sgd_no_support"])
def test_f32_learner_wide_obs_two_steps_match_torch_learner(D, optimizer, no_support):
  """Two captured f32 steps against learners.Learner (torch modules, float32) from the same weights and batches:
  losses 1e-4 relative, every weight 2e-5 absolute.  The no_support case steps with SGD: Adam divides by
  sqrt(v) + 1.5e-4, which turns the last float32 bits of a near-zero gradient (summed in another order than torch's)
  into up to 5.3 times as much weight change, and the scalar value head of these random batches has such gradients
  (up to 1e-4 on 10 of its 25 600 first-layer weights under AdamW) -- in a head this change does not touch."""
  _f32_against_torch(D, optimizer, no_support)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [147, 512, 1024])
def test_bf16_learner_wide_obs_against_f32_learner(D):
  """One step: every parameter gradient of the tensor-core step at cosine >= 0.98 against the f32 step.  Two
  captured steps: losses within 2e-2 and weights within 2.5 learning rates per step of the f32 learner's."""
  from model_based_rl_b200 import fused_learner
  A, K, B = 18, 5, 256
  cfg = _cfg(K)
  torch.manual_seed(D)
  w = {k: v.clone() for k, v in fused_learner.FusedFCNetwork(D, A, "cuda", cfg).state_dict().items()}
  grads, nets, learners_ = {}, {}, {}
  for prec in ("f32", "bf16"):
    net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
    net.load_weights(w)
    fused = fused_learner.FusedLearner(cfg, net, use_graph=False, precision=prec)
    fused._stage(_batch(B, K, A, D, 7))
    fused._forward_and_heads_backward()
    fused._recurrent_backward()
    torch.cuda.synchronize()
    grads[prec] = {k: g.clone() for k, g in net.grads.items()}
  cos = {}
  for k, want in grads["f32"].items():
    a, b = grads["bf16"][k].double().flatten(), want.double().flatten()
    cos[k] = float((a @ b) / (a.norm() * b.norm() + 1e-300))
  assert min(cos.values()) >= 0.98, cos
  for prec in ("f32", "bf16"):
    nets[prec] = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
    nets[prec].load_weights(w)
    learners_[prec] = fused_learner.FusedLearner(cfg, nets[prec], use_graph=True, precision=prec)
  for step in range(2):
    batch = _batch(B, K, A, D, 11 + step)
    lf = learners_["f32"].update_weights(batch).cpu().numpy()
    lb = learners_["bf16"].update_weights(batch).cpu().numpy()
    np.testing.assert_allclose(lb, lf, rtol=2e-2)
    bar = 2.5 * cfg.lr_init * (step + 1)
    for k, v in nets["bf16"].state_dict().items():
      np.testing.assert_allclose(v.cpu().numpy(), nets["f32"].state_dict()[k].cpu().numpy(), rtol=0, atol=bar,
                                 err_msg="step %d %s" % (step, k))


@pytest.mark.gpu
def test_learn_with_512_byte_observations_feeds_priorities_and_hands_weights_to_a_bf16_network():
  """learn() with graphs on over a PrioritizedReplay of uint8 observations (512 features, norm_obs): priorities come
  back from the device, send_weights() hands the weights to a bf16 FCNetwork, and that network's initial_inference
  (the float32 kernel above 191 features) gives the learner's representation."""
  import torch.nn.functional as F
  from model_based_rl_b200 import fused_learner
  from model_based_rl_b200.networks import FCNetwork
  from model_based_rl_b200.replay_buffer import PrioritizedReplay
  from model_based_rl_b200.selfplay import HistorySlice
  D, A, K = 512, 18, 5
  cfg = _cfg(K, norm_obs=True, obs_range=[0, 255] * D, td_steps=5, batch_size=64, beta_increment_per_sampling=0.001,
             epsilon=0.01, alpha=1.0, beta=0.5, discount=0.997, action_space=A, obs_space=(D,), window_size=2000,
             window_step=None, seed=None, send_weights_frequency=3, training_steps=5, stored_before_train=100)
  rb = PrioritizedReplay(cfg)
  r2 = np.random.default_rng(9)
  for _ in range(6):
    n = int(r2.integers(50, 200))
    rb.save_history(HistorySlice(list(r2.integers(0, 256, size=(n, D)).astype(np.uint8)), r2.random((n, A)).tolist(),
                                 r2.normal(size=n).tolist(), r2.integers(0, A, size=n).tolist(), r2.normal(size=n).tolist(),
                                 np.abs(r2.normal(size=n)).tolist(), [False] * n, list(range(n)), [None] * n, [1] * n),
                    ignore=None, terminal=True)
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  search_net = FCNetwork(D, A, "cuda", cfg)
  learner = fused_learner.FusedLearner(cfg, net, replay_buffer=rb, search_network=search_net)
  assert learner.use_graph and learner.precision == "bf16"
  before = rb.index.tree.clone()
  w0 = net.flat.clone()
  assert learner.learn() == 5
  torch.cuda.synchronize()
  assert not torch.equal(rb.index.tree, before)
  assert not torch.equal(net.flat, w0) and torch.isfinite(net.flat).all()
  learner.send_weights()
  assert search_net.precision == "bf16"
  for k, v in net.state_dict().items():
    assert torch.equal(search_net.get_weights()[k].cpu(), v.cpu()), k
  obs = torch.from_numpy(r2.integers(0, 256, size=(64, D)).astype(np.float32)).cuda() / 255.0
  hidden = search_net.initial_inference(obs).hidden_state
  W = net.state_dict()
  y = F.linear(F.relu(F.linear(obs, W["representation_head.fc1.weight"], W["representation_head.fc1.bias"])),
               W["representation_head.out.weight"], W["representation_head.out.bias"])
  want = F.relu(F.layer_norm(y, (50,), W["LN.weight"], W["LN.bias"], 1e-5))
  assert _rel(hidden, want) <= 3e-2
