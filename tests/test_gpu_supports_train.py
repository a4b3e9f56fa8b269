"""The training side at value and reward supports other than [-15, 15]: the scalar transforms, target construction
with fused supports (all three kernels behind mz_build_targets and the replay's device sampling), the unroll loss
and the fused learner, each against a float64 (or exact float32) reference.

With value support == reward support a kernel that reads the value support's minimum or bin count for the reward
head (or the other way round) gives the right answer; every configuration below has V != R, and their widths cross
the 32-lane loops, the 32-column tiles and the fused learner's 64-bin limit.  Every configuration runs with the
target transform h and with no_target_transform.  Each tolerance is stated next to the largest value measured on a
B200 at its default clocks (power limit not recorded); the tests print what they measure."""
import types

import numpy as np
import pytest
import torch

import helpers
import oracle
from oracle import learner_ref
from oracle.fcnet_ref import FCNetworkRef, support_to_scalar

# id: (value support, reward support)
SUPPORTS = {
    "S0": ((-15, 15), (-15, 15)),   # control: the supports every other test uses
    "S1": ((-4, 27), (-1, 1)),      # 32 / 3 bins: clipped-reward Atari shape, asymmetric value support
    "S2": ((-16, 16), (-8, 31)),    # 33 / 40 bins: both cross the 32-lane loops and the 32-column tile
    "S3": ((-30, 33), (-2, 6)),     # 64 / 9 bins: the fused learner's widest head
    "S4": ((3, 9), (0, 0)),         # 7 bins without 0 (every zero target clamps) / one bin: CE 0, gradient 0
    "S5": ((-300, 300), (-1, 1)),   # 601 / 3 bins: targets, transforms, the torch-module loss; the fused learner refuses it
}
FUSED = ["S0", "S1", "S2", "S3", "S4"]
H_MODES = [False, True]  # no_target_transform
H_IDS = ["h", "no_h"]


def _bins(s):
  return s[1] - s[0] + 1


def _h64(x):
  """Config.scalar_transform (config.py:51-54) in binary64."""
  x = np.asarray(x, np.float64)
  return np.sign(x) * (np.sqrt(np.abs(x) + 1) - 1) + 0.001 * x


def _emulated_support(t, s, no_tt):
  """The kernels' two-hot of float32 targets t: h in float32 (oracle.scalar_transform_f32), then the float32 two-hot
  (oracle.two_hot_f64(..., float32=True))."""
  x = np.asarray(t, np.float32) if no_tt else oracle.scalar_transform_f32(t)
  return oracle.two_hot_f64(x, s[0], s[1], float32=True)[1]


def _spread(rng, n, s, no_tt):
  """Scalars whose (transformed) values land inside the support, on both clamps and near zero."""
  m = max(abs(s[0]), abs(s[1])) + 2
  top = 1.3 * (m * m if not no_tt else m)
  return rng.choice([-1.0, 1.0], size=n) * 10.0 ** rng.uniform(-2, np.log10(top), size=n)


def _cfg(sup, no_tt, K=5, **kw):
  vs, rs = SUPPORTS[sup]
  d = dict(value_support=list(vs), reward_support=list(rs), no_support=False, no_target_transform=no_tt,
           num_unroll_steps=K, optimizer="AdamW", lr_init=1e-3, momentum=0.9, weight_decay=1e-4, clip_grad=0,
           lr_scheduler=None, norm_obs=False, send_weights_frequency=500, training_steps=2)
  d.update(kw)
  return types.SimpleNamespace(**d)


# -- 6. the fused learner refuses supports its head kernels cannot run (CPU) --------------------------------------
@pytest.mark.parametrize("vs,rs", [((-300, 300), (-1, 1)), ((-15, 15), (-40, 40)), ((5, 4), (-1, 1)),
                                   ((-15, 15), (1, -1))], ids=["S5_value_601", "reward_81", "value_max_lt_min",
                                                               "reward_max_lt_min"])
def test_fused_network_refuses_supports_wider_than_64_bins(vs, rs, monkeypatch):
  """FusedFCNetwork raises ValueError naming the 64-bin limit before it loads the library or touches a device (the
  kernels would refuse the first step with a bare MZ_ERR_BAD_ARG).  64 bins and no_support networks pass the check."""
  from model_based_rl_b200 import _lib, fused_learner

  def untouched(*a, **k):
    raise AssertionError("the support check must come before the library and the device")
  monkeypatch.setattr(_lib, "load", untouched)
  monkeypatch.setattr(_lib, "normalize_device", untouched)
  cfg = types.SimpleNamespace(value_support=list(vs), reward_support=list(rs), no_support=False)
  with pytest.raises(ValueError, match="64 bins"):
    fused_learner.FusedFCNetwork(16, 4, "cuda", cfg)
  for ok in (types.SimpleNamespace(value_support=[-30, 33], reward_support=[-1, 1], no_support=False),
             types.SimpleNamespace(value_support=list(vs), reward_support=list(rs), no_support=True)):
    with pytest.raises(AssertionError, match="support check must come before"):
      fused_learner.FusedFCNetwork(16, 4, "cuda", ok)


# -- 2. standalone transforms --------------------------------------------------------------------------------------
def _transform_inputs(rng, s):
  ints = np.arange(s[0] - 1, s[1] + 2, dtype=np.float32)
  big = np.float32(np.finfo(np.float32).max)
  return np.concatenate([ints, np.nextafter(ints, np.float32(np.inf)), np.nextafter(ints, np.float32(-np.inf)),
                         np.array([big, -big, 0.5, -0.5, 1e-30, -1e-30], np.float32),
                         rng.uniform(s[0] - 3, s[1] + 3, size=997).astype(np.float32)]).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("no_tt", H_MODES, ids=H_IDS)
@pytest.mark.parametrize("sup", list(SUPPORTS))
def test_scalar_to_support_and_back(sup, no_tt):
  """mz_scalar_to_support (Config.value_phi / reward_phi) bit for bit against the binary64 two-hot with each weight
  rounded to float32 where the float32 operations round it (oracle.two_hot_f64), with x clamped in place;
  mz_support_to_scalar (inverse_*_transform) against binary64 (oracle.inverse_transform_f64), no further from it than
  2x torch's float32 pipeline (FCNetworkRef's support_to_scalar) plus 1e-7 of max(1, |v|).
  Measured on the B200: kernel / torch ratio of the largest errors 1.0 with h, <= 1.5 without."""
  from model_based_rl_b200.config import Config
  vs, rs = SUPPORTS[sup]
  cfg = Config(dict(value_support=list(vs), reward_support=list(rs), no_target_transform=no_tt))
  rng = np.random.default_rng(_bins(vs) * 7 + _bins(rs))
  for s, phi, inv in ((vs, cfg.value_phi, cfg.inverse_value_transform), (rs, cfg.reward_phi, cfg.inverse_reward_transform)):
    x0 = _transform_inputs(rng, s)
    x = torch.from_numpy(x0.copy()).cuda()
    sup_dev = phi(x.view(-1, 1))
    torch.cuda.synchronize()
    clamped, want = oracle.two_hot_f64(x0, s[0], s[1], float32=True)
    assert np.array_equal(sup_dev.cpu().numpy().reshape(len(x0), -1), want)
    assert np.array_equal(x.cpu().numpy(), clamped.astype(np.float32))  # x.clamp_ in place
    # support -> scalar: random logits with a peak at a random bin, so the expectation covers the support
    n = 2048
    logits = rng.normal(0, 2, size=(n, _bins(s))).astype(np.float32)
    logits[np.arange(n), rng.integers(0, _bins(s), size=n)] += rng.uniform(0, 12, size=n).astype(np.float32)
    got = inv(torch.from_numpy(logits).cuda()).cpu().numpy().reshape(-1).astype(np.float64)
    truth = oracle.inverse_transform_f64(logits, s[0], s[1], no_tt)
    cpu32 = support_to_scalar(torch.from_numpy(logits), s[0], s[1], no_tt).numpy().reshape(-1).astype(np.float64)
    scale = np.maximum(np.abs(truth), 1.0)
    ek, et = np.abs(got - truth) / scale, np.abs(cpu32 - truth) / scale
    print("%s %s bins %d: support_to_scalar max err kernel %.3g torch %.3g" % (sup, H_IDS[no_tt], _bins(s), ek.max(),
                                                                              et.max()))
    assert ek.max() <= 2.0 * et.max() + 1e-7
    assert ek.mean() <= 2.0 * et.mean() + 1e-8


# -- 3. mz_build_targets with fused supports ----------------------------------------------------------------------
@pytest.fixture(params=[0, 1, 2], ids=["kernel_by_shape", "warp_per_row_kernel", "lane_per_position_kernel"])
def targets_kernel(request):
  """The three kernels behind mz_build_targets (include/mzb200.h: TMA-staged by shape, warp per row, lane per
  position).  By shape, S0-S4 at K = 5 fit the TMA-staged kernel's 96 KB shared-memory plan (S2: 8 rows x 6
  positions x 73 bins x 4 B = 14 KB of supports); S5 (8 x 6 x 604 x 4 B = 116 KB) falls back to lane per position."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  lib.mz_debug_set_targets_kernel(request.param)
  yield request.param
  lib.mz_debug_set_targets_kernel(0)


GUARD = 67  # NaN floats behind each support buffer


def _guarded(n):
  buf = torch.full((n + GUARD,), float("nan"), device="cuda")
  buf[:n] = -7.0  # sentinel: every element must be written
  return buf


TARGET_CASES = [(s, h, False) for s in SUPPORTS for h in H_MODES] + [("S1", False, True)]


@pytest.mark.gpu
@pytest.mark.parametrize("sup,no_tt,clip", TARGET_CASES,
                         ids=["%s-%s%s" % (s, H_IDS[h], "-clip" if c else "") for s, h, c in TARGET_CASES])
def test_build_targets_fused_supports(sup, no_tt, clip, targets_kernel):
  """B = 45 rows (the last CTA of the TMA-staged kernel holds five: the non-bulk flush), K = 5, td_steps 10, rewards in
  +-5 (clipped on the fly in the clip case), bootstrap values spread over the support and past both ends.
  Targets against oracle.insert_target; supports bit for bit against h in float32 + two-hot on the kernel's own
  targets; and in binary64 against the oracle's targets: sum_j p_j (min + j) == clamp(h(t)) within 1e-6 of max(1, |.|)
  (measured on the B200: <= 1.4e-7; n-step values may differ from the oracle's by 1e-5 relative), at most two adjacent
  non-zero bins, row mass 1 within 1e-6.  No element of either support is left unwritten; nothing is written past it."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  vs, rs = SUPPORTS[sup]
  V, R = _bins(vs), _bins(rs)
  A, K, T, B, E = 4, 5, 10, 45, 16
  rng = np.random.default_rng(V * 1000 + R * 10 + int(no_tt) + 2 * int(clip))
  lens = rng.integers(1, 60, size=40).astype(np.int32)
  lens[:3] = [1, 2, K + T + 5]
  starts = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
  P = int(lens.sum())
  obs_np = rng.normal(size=(P, E)).astype(np.float32)
  rewards = (rng.uniform(-5, 5, size=P) * (rng.random(P) < 0.7)).astype(np.float32)
  rewards[::3] = np.round(rewards[::3])
  to_play = rng.choice([-1, 1], size=P).astype(np.int8)
  root_values = _spread(rng, P, vs, no_tt)
  cv = rng.random((P, A)).astype(np.float32)
  cv /= cv.sum(1, keepdims=True)
  actions = rng.integers(0, A, size=P, dtype=np.int32)
  disc = 0.997
  ci = rng.integers(0, len(lens), size=B)
  ci[:3] = [0, 1, 2]
  step = (rng.random(B) * lens[ci]).astype(np.int64)
  step[-1] = lens[ci[-1]] - 1
  d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
  t_obs, t_act, t_rew, t_tp, t_rv, t_cv = d(obs_np), d(actions), d(rewards), d(to_play), d(root_values), d(cv)
  discounts = d(np.array([disc**n for n in range(K + T)], np.float32))
  win = _lib.Window(A, E, 0, int(clip), t_obs.data_ptr(), t_act.data_ptr(), t_rew.data_ptr(), t_tp.data_ptr(),
                    t_rv.data_ptr(), t_cv.data_ptr())
  tc = _lib.TargetCfg(B, K, T, 1, vs[0], vs[1], rs[0], rs[1], int(no_tt), 0, disc**T, discounts.data_ptr(), None, None)
  pos, cs, cl = d(starts[ci] + step), d(starts[ci]), d(lens[ci])
  pads = d(rng.integers(0, A, size=(B, K), dtype=np.int32))
  out = [torch.full((B, E), -7.0, device="cuda"), torch.full((B, K), -7, dtype=torch.int32, device="cuda"),
         torch.full((B, K + 1), -7.0, device="cuda"), torch.full((B, K + 1), -7.0, device="cuda"),
         torch.full((B, K + 1, A), -7.0, device="cuda")]
  nv, nr = B * (K + 1) * V, B * (K + 1) * R
  vbuf, rbuf = _guarded(nv), _guarded(nr)
  _lib.check(lib.mz_build_targets(win, tc, _lib.ptr(pos), _lib.ptr(cs), _lib.ptr(cl), _lib.ptr(pads),
                                  *[_lib.ptr(o) for o in out], _lib.ptr(vbuf), _lib.ptr(rbuf), _lib.current_stream()),
             "mz_build_targets")
  torch.cuda.synchronize()
  tr, tv = out[2].cpu().numpy(), out[3].cpu().numpy()
  vbuf, rbuf = vbuf.cpu().numpy(), rbuf.cpu().numpy()
  assert np.isnan(vbuf[nv:]).all() and np.isnan(rbuf[nr:]).all()
  vsup, rsup = vbuf[:nv].reshape(B, K + 1, V), rbuf[:nr].reshape(B, K + 1, R)
  assert not (vsup == -7.0).any() and not (rsup == -7.0).any()
  seen_r = rewards if not clip else oracle.clip_reward(rewards).astype(np.float32)
  want_v, want_r = np.zeros((B, K + 1), np.float32), np.zeros((B, K + 1), np.float32)
  for b in range(B):
    lo, n, s = int(starts[ci[b]]), int(lens[ci[b]]), int(step[b])
    sl = slice(lo, lo + n)
    wr, wv, _ = oracle.insert_target(seen_r[sl], to_play[sl], root_values[sl], cv[sl], K, T, disc, s)
    assert np.array_equal(tr[b], wr), (b, tr[b], wr)
    assert np.max(np.abs(tv[b] - wv) / np.maximum(np.abs(wv), 1.0)) <= 1e-5
    want_v[b], want_r[b] = wv, wr
  assert np.array_equal(vsup, _emulated_support(tv, vs, no_tt))
  assert np.array_equal(rsup, _emulated_support(tr, rs, no_tt))
  worst = 0.0
  for sup_, t, s in ((vsup, want_v, vs), (rsup, want_r, rs)):
    p = sup_.astype(np.float64)
    h = np.clip(t.astype(np.float64) if no_tt else _h64(t), s[0], s[1])
    mean = (p * np.arange(s[0], s[1] + 1, dtype=np.float64)).sum(-1)
    err = np.abs(mean - h) / np.maximum(np.abs(h), 1.0)
    worst = max(worst, float(err.max()))
    assert err.max() <= 1e-6
    assert np.abs(p.sum(-1) - 1.0).max() <= 1e-6
    nz = p != 0
    first, last = nz.argmax(-1), nz.shape[-1] - 1 - nz[..., ::-1].argmax(-1)
    assert (nz.sum(-1) <= 2).all() and (last - first <= 1).all()  # one bin, or two adjacent ones
  print("%s %s clip=%d kernel %d: support mean vs binary64 h(t) max rel err %.3g" % (sup, H_IDS[no_tt], clip,
                                                                                    targets_kernel, worst))


@pytest.mark.gpu
@pytest.mark.parametrize("ring", [0, 2], ids=["fresh_outputs", "ring_of_2"])
@pytest.mark.parametrize("sup,no_tt", [("S1", False), ("S1", True), ("S3", False), ("S3", True)],
                         ids=["S1-h", "S1-no_h", "S3-h", "S3-no_h"])
def test_replay_device_sampling_fuses_the_configured_supports(sup, no_tt, ring):
  """PrioritizedReplay.sample_batch_device(fuse_supports=True) on a replay built with these supports: [B, K+1, V] and
  [B, K+1, R] supports equal to h in float32 + two-hot of the returned targets, over three batches (the ring wraps)."""
  import random
  import test_gpu_replay as tgr
  from model_based_rl_b200.replay_buffer import PrioritizedReplay
  g = helpers.load("replay_breakout")
  vs, rs = SUPPORTS[sup]
  rb = PrioritizedReplay(tgr._config(g, value_support=vs, reward_support=rs, no_target_transform=no_tt))
  for h in range(int(g["n_hist"])):
    ign = int(g["ignores"][h])
    rb.save_history(tgr._history(g, h), ignore=None if ign < 0 else ign, terminal=ign < 0)
  random.seed(7)
  np.random.seed(7)
  B, K = int(g["batch_size"]), int(g["num_unroll_steps"])
  for _ in range(3):
    out, idxs, is_w = rb.sample_batch_device(fuse_supports=True, ring=ring)
    assert len(out) == 7
    t_r, t_v, vsup, rsup = out[2], out[3], out[5], out[6]
    assert tuple(vsup.shape) == (B, K + 1, _bins(vs)) and tuple(rsup.shape) == (B, K + 1, _bins(rs))
    torch.cuda.synchronize()
    assert np.array_equal(vsup.cpu().numpy(), _emulated_support(t_v.cpu().numpy(), vs, no_tt))
    assert np.array_equal(rsup.cpu().numpy(), _emulated_support(t_r.cpu().numpy(), rs, no_tt))


# -- 4. mz_unroll_loss ---------------------------------------------------------------------------------------------
def _loss_inputs(rng, sup, no_tt, K, B, A):
  vs, rs = SUPPORTS[sup]
  values = rng.normal(0, 2, size=(K + 1, B, _bins(vs))).astype(np.float32)
  rewards = rng.normal(0, 2, size=(K, B, _bins(rs))).astype(np.float32)
  policies = rng.normal(0, 2, size=(K + 1, B, A)).astype(np.float32)
  t_v = _spread(rng, B * (K + 1), vs, no_tt).astype(np.float32).reshape(B, K + 1)
  t_v[0, 0], t_v[1, 0] = vs[1], vs[0]  # exactly on the ends (and integers)
  t_r = (rng.uniform(-5, 5, size=(B, K + 1)) * (rng.random((B, K + 1)) < 0.8)).astype(np.float32)
  t_r[::4] = np.round(t_r[::4])
  t_p = rng.random((B, K + 1, A)).astype(np.float32)
  t_p /= t_p.sum(-1, keepdims=True)
  t_p[-3:, -2:] = 0.0  # positions past the end of the episode
  is_w = rng.uniform(0.1, 1.0, size=B)
  return values, rewards, policies, t_v, t_r, t_p, is_w


def _ref_loss(cfg, values, rewards, policies, t_v, t_r, t_p, is_w, dtype):
  """unroll_loss_ref in `dtype` with autograd: (losses, errors, [value, reward, policy logit gradients])."""
  lg = [torch.from_numpy(x).to(dtype).requires_grad_(True) for x in (values, rewards, policies)]
  t = lambda x: torch.from_numpy(x).to(dtype)
  losses, errs = learner_ref.unroll_loss_ref(cfg, lg[0], lg[1], lg[2], t(t_v), t(t_r), t(t_p),
                                             torch.from_numpy(is_w))
  losses.sum().backward()
  return losses.detach().numpy(), errs.numpy().astype(np.float64), [x.grad.numpy() for x in lg]


LOSS_BAR = 1e-6   # losses, relative (measured on the B200: <= 3.1e-8)
GRAD_BAR = 2e-6   # logit gradients, of each tensor's largest entry (measured: <= 2.3e-7)
# priority errors: the kernel's largest error against binary64 <= ERR_MULT x torch's float32 one.  Measured: 1.0 with h
# (h^-1's cancellation dominates both alike), <= 3.9 without (S5, K = 5: the float32 expectation over 601 bins summed in
# another order; the largest of 37 row errors is a noisy statistic -- over 2048 rows the ratio is <= 1.5, see above)
ERR_MULT = 6.0


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 5])
@pytest.mark.parametrize("no_tt", H_MODES, ids=H_IDS)
@pytest.mark.parametrize("sup", list(SUPPORTS))
def test_unroll_loss_against_float64(sup, no_tt, K):
  """mz_unroll_loss through learners.unroll_loss on [K+1][B][V] logits (FusedLearner's layout), B = 37, against
  float64 autograd through unroll_loss_ref on the same float32 logits: losses within LOSS_BAR relative, every logit
  gradient within GRAD_BAR of its tensor's largest entry, priority errors against binary64 no further than ERR_MULT x
  torch's float32 pipeline (h^-1 magnifies float32 rounding at wide supports).  S4's one-bin reward support gives a
  reward loss of exactly 0 and a reward gradient of exactly 0.

  The float64 reference starts from the targets' float32 h(t) (oracle.scalar_transform_f32, which the kernels
  reproduce bit for bit, test_build_targets_fused_supports): h is rounded to float32 in the reference's pipeline too,
  and at 601 bins one float32 ulp of h(t) ~ 300 moves a two-hot weight, and with it a gradient, by 3e-5."""
  from model_based_rl_b200 import learners
  B, A = 37, 5
  rng = np.random.default_rng(_bins(SUPPORTS[sup][0]) + 100 * K + int(no_tt))
  cfg = _cfg(sup, no_tt, K)
  args = _loss_inputs(rng, sup, no_tt, K, B, A)
  values, rewards, policies, t_v, t_r, t_p, is_w = args
  h32 = (lambda t: t) if no_tt else oracle.scalar_transform_f32
  want, _, want_g = _ref_loss(_cfg(sup, True, K), values, rewards, policies, h32(t_v), h32(t_r), t_p, is_w,
                              torch.float64)
  _, cpu32_err, _ = _ref_loss(cfg, *args, torch.float32)
  dev = [torch.from_numpy(x).cuda().requires_grad_(True) for x in (values, rewards, policies)]
  losses, errs = learners.unroll_loss(cfg, dev[0], dev[1], dev[2], torch.from_numpy(t_v).cuda(),
                                      torch.from_numpy(t_r).cuda(), torch.from_numpy(t_p).cuda(),
                                      torch.from_numpy(is_w).cuda())
  losses.sum().backward()
  got = losses.detach().cpu().numpy()
  rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-30)
  grads = [x.grad.cpu().numpy() for x in dev]
  grel = [float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30)) for a, b in zip(grads, want_g)]
  truth = oracle.inverse_transform_f64(values[0], *SUPPORTS[sup][0], no_tt) - t_v[:, 0]
  scale = np.maximum(np.abs(truth), 1.0)
  ek = np.abs(errs.cpu().numpy().astype(np.float64) - truth) / scale
  et = np.abs(cpu32_err - truth) / scale
  print("%s %s K=%d: loss rel %s, grad rel %s, errors max kernel %.3g torch %.3g" % (
      sup, H_IDS[no_tt], K, np.array2string(rel, precision=2), ["%.2g" % x for x in grel], ek.max(), et.max()))
  if SUPPORTS[sup][1] == (0, 0):
    assert got[0] == 0.0 and (grads[1] == 0.0).all()
    assert want[0] == 0.0
    rel[0] = 0.0
    grel[1] = 0.0
  assert rel.max() <= LOSS_BAR, rel
  assert max(grel) <= GRAD_BAR, grel
  assert ek.max() <= ERR_MULT * et.max() + 1e-7


@pytest.mark.gpu
@pytest.mark.parametrize("no_tt", H_MODES, ids=H_IDS)
def test_torch_module_learner_trains_601_bins(no_tt):
  """learners.Learner (cuBLAS GEMMs + mz_unroll_loss) keeps training supports the fused learner refuses: one step at
  S5 against float64 autograd through FCNetworkRef + unroll_loss_ref, losses within 1e-6 relative (measured on the
  B200: <= 2.1e-8)."""
  from model_based_rl_b200 import learners
  torch.backends.cuda.matmul.allow_tf32 = False
  K, B, D, A = 3, 24, 16, 4
  cfg = _cfg("S5", no_tt, K)
  rng = np.random.default_rng(601 + int(no_tt))
  net = learners.FCNetworkTrain(D, A, "cuda", cfg)
  batch = _learner_batch(rng, "S5", no_tt, K, B, D, A)
  want, _, _ = _float64_step(cfg, net.get_weights(), batch, D, A)
  learner = learners.Learner(cfg, net)
  losses = learner.update_weights(batch).cpu().numpy()
  rel = np.abs(losses - want) / np.abs(want)
  print("S5 %s Learner losses rel %s" % (H_IDS[no_tt], rel))
  assert rel.max() <= 1e-6


# -- 5. FusedLearner -----------------------------------------------------------------------------------------------
def _learner_batch(rng, sup, no_tt, K, B, D, A):
  vs, _ = SUPPORTS[sup]
  obs = rng.normal(size=(B, D)).astype(np.float32)
  actions = rng.integers(0, A, size=(B, K)).astype(np.int64)
  t_v = _spread(rng, B * (K + 1), vs, no_tt).astype(np.float32).reshape(B, K + 1)
  t_r = (rng.uniform(-5, 5, size=(B, K + 1)) * (rng.random((B, K + 1)) < 0.8)).astype(np.float32)
  t_p = rng.random((B, K + 1, A)).astype(np.float32)
  t_p /= t_p.sum(-1, keepdims=True)
  t_p[-2:, -1] = 0.0
  is_w = rng.uniform(0.2, 1.0, size=B)
  return (obs, actions, (t_r, t_v, t_p)), None, is_w


def _float64_step(cfg, weights, batch, D, A):
  """Losses, priority errors and parameter gradients of one step in float64 autograd: FCNetworkRef in train mode
  (the 0.5 gradient hook on every hidden state of the dynamics, learners.py:201) + unroll_loss_ref."""
  (obs, actions, (t_r, t_v, t_p)), _, is_w = batch
  net = FCNetworkRef(D, A, cfg.value_support, cfg.reward_support, cfg.no_target_transform).double()
  net.load_state_dict({k: torch.as_tensor(v).double() for k, v in weights.items()})
  net.train()
  out = net.initial_inference(torch.from_numpy(obs).double())
  values, rewards, policies, h = [out.value], [], [out.policy_logits], out.hidden_state
  for i in range(cfg.num_unroll_steps):
    out = net.recurrent_inference(h, actions[:, i])
    h = out.hidden_state
    h.register_hook(lambda grad: grad * 0.5)
    values.append(out.value), rewards.append(out.reward), policies.append(out.policy_logits)
  t = lambda x: torch.from_numpy(x).double()
  losses, errs = learner_ref.unroll_loss_ref(cfg, values, rewards, policies, t(t_v), t(t_r), t(t_p), t(is_w))
  losses.sum().backward()
  return losses.detach().numpy(), errs.numpy(), {k: p.grad for k, p in net.named_parameters()}


# (K, A, no_target_transform): each support sees both h modes, both K and both action counts
LEARNER_SHAPES = [(1, 4, False), (5, 18, False), (1, 18, True), (5, 4, True)]
F32_LOSS_BAR = 1e-6   # relative (measured on the B200: <= 2.8e-8)
F32_GRAD_BAR = 1e-5   # of each gradient tensor's largest entry (measured: <= 8.3e-7)
F32_ERR_BAR = 1e-3    # priority errors, of max(1, |error|): float32 logits through h^-1 (measured: <= 4.2e-4)


def _fused(sup, no_tt, K, A, precision, graph=False, search_network=None, seed=0):
  from model_based_rl_b200 import fused_learner
  cfg = _cfg(sup, no_tt, K)
  torch.manual_seed(seed)
  net = fused_learner.FusedFCNetwork(16, A, "cuda", cfg)
  return cfg, net, fused_learner.FusedLearner(cfg, net, use_graph=graph, precision=precision,
                                              search_network=search_network)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", LEARNER_SHAPES, ids=["K%d-A%d-%s" % (k, a, H_IDS[h]) for k, a, h in LEARNER_SHAPES])
@pytest.mark.parametrize("sup", FUSED[1:])
def test_fused_learner_f32_step_against_float64(sup, shape):
  """One f32 step (forward, mz_unroll_loss, backward) against float64 autograd on the same weights and batch: the
  three losses within F32_LOSS_BAR relative, every parameter gradient within F32_GRAD_BAR of its largest entry, the
  priority errors within F32_ERR_BAR."""
  K, A, no_tt = shape
  B, D = 29, 16
  cfg, net, fused = _fused(sup, no_tt, K, A, "f32")
  rng = np.random.default_rng(K * 100 + A + int(no_tt))
  batch = _learner_batch(rng, sup, no_tt, K, B, D, A)
  want, want_err, want_g = _float64_step(cfg, net.get_weights(), batch, D, A)
  fused._stage(batch)
  fused._forward_and_heads_backward()
  fused._recurrent_backward()
  torch.cuda.synchronize()
  assert fused.v.shape[2] == _bins(SUPPORTS[sup][0]) and fused.r.shape[2] == _bins(SUPPORTS[sup][1])
  got = fused.losses.cpu().numpy()
  rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-30)
  if SUPPORTS[sup][1] == (0, 0):
    assert got[0] == 0.0 and (net.grads["reward_head.reward.weight"] == 0).all()
    rel[0] = 0.0
  grel = {}
  for k, w in want_g.items():
    if float(w.abs().max()) == 0.0:
      assert float(net.grads[k].abs().max()) == 0.0, k
      continue
    grel[k] = float((net.grads[k].cpu().double() - w).abs().max() / w.abs().max())
  err = np.abs(fused.new_errors.cpu().numpy() - want_err) / np.maximum(np.abs(want_err), 1.0)
  print("%s K=%d A=%d %s: loss rel %s, worst grad %s %.2g, errors %.2g" % (
      sup, K, A, H_IDS[no_tt], rel, max(grel, key=grel.get), max(grel.values()), err.max()))
  assert rel.max() <= F32_LOSS_BAR, rel
  assert max(grel.values()) <= F32_GRAD_BAR, grel
  assert err.max() <= F32_ERR_BAR


@pytest.mark.gpu
@pytest.mark.parametrize("shape", LEARNER_SHAPES, ids=["K%d-A%d-%s" % (k, a, H_IDS[h]) for k, a, h in LEARNER_SHAPES])
@pytest.mark.parametrize("sup", FUSED[1:])
def test_fused_learner_bf16_step_against_emulation(sup, shape):
  """The tensor-core step (value heads of 32, 33, 64 and 7 columns, reward heads of 3, 40, 9 and 1) against float64
  autograd with the kernels' bf16 rounding points (test_fused_learner._teacher_forced_check), at that test's bars:
  outputs within 2e-3, parameter gradients within 3e-3 of their largest entry (measured on the B200: <= 1.6e-3)."""
  from test_fused_learner import _teacher_forced_check
  K, A, no_tt = shape
  cfg, net, fused = _fused(sup, no_tt, K, A, "bf16")
  rng = np.random.default_rng(K * 100 + A + int(no_tt))
  fused._stage(_learner_batch(rng, sup, no_tt, K, 29, 16, A))
  fused._forward_and_heads_backward()
  fused._recurrent_backward()
  torch.cuda.synchronize()
  if SUPPORTS[sup][1] == (0, 0):
    assert float(fused.losses[0]) == 0.0 and (fused.dr == 0).all()
  worst = _teacher_forced_check(fused, net, 2e-3, 3e-3)
  print(sup, shape, "vs emulation", max(worst.values()))


GRAPH_BAR = 1e-6  # eager and graphed steps differ only in the order of the gradient atomics (measured: <= 3.2e-7)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["f32", "bf16"])
@pytest.mark.parametrize("sup", FUSED[1:])
def test_fused_learner_graph_equals_eager_and_hands_weights_to_search(sup, precision):
  """Two AdamW steps in eager mode and in CUDA-graph mode from the same weights on the same batches: the same weights
  (within GRAPH_BAR, atomics order the gradient sums differently).  Then send_weights into a search FCNetwork built
  with the same supports: it holds the learner's weights bit for bit, and its value / reward scalars match FCNetworkRef
  in float64 eval mode on those weights within 5e-4 of max(1, |v|) (measured on the B200: <= 9.8e-5, at S3 with h,
  where h^-1 maps the 64-bin expectation to values near 1000)."""
  from model_based_rl_b200 import networks
  K, A, no_tt = 5, 4, sup in ("S2", "S4")
  rng = np.random.default_rng(3)
  batches = [_learner_batch(rng, sup, no_tt, K, 40, 16, A) for _ in range(2)]
  search = networks.FCNetwork(16, A, "cuda", _cfg(sup, no_tt, K), precision="f32")
  _, net_e, eager = _fused(sup, no_tt, K, A, precision, graph=False, search_network=search, seed=5)
  cfg, net_g, graph = _fused(sup, no_tt, K, A, precision, graph=True, seed=5)
  assert torch.equal(net_e.flat, net_g.flat)
  w0 = net_e.flat.clone()
  for b in batches:
    eager.update_weights(b)
    graph.update_weights(b)
  torch.cuda.synchronize()
  assert not torch.equal(net_e.flat, w0) and torch.isfinite(net_e.flat).all()
  diff = float((net_e.flat - net_g.flat).abs().max())
  print("%s %s graph vs eager max weight difference %.3g" % (sup, precision, diff))
  assert diff <= GRAPH_BAR, diff
  weights = eager.send_weights()
  torch.cuda.synchronize()
  for k, v in search.get_weights().items():
    assert torch.equal(v, weights[k].cpu()), k
  obs = torch.from_numpy(batches[0][0][0]).cuda()
  acts = torch.from_numpy(batches[0][0][1][:, 0]).cuda()
  s0 = search.initial_inference(obs)
  s1 = search.recurrent_inference(s0.hidden_state, acts.to(torch.int32))
  ref = FCNetworkRef(16, A, cfg.value_support, cfg.reward_support, no_tt).double()
  ref.load_state_dict({k: v.double() for k, v in search.get_weights().items()})
  with torch.no_grad():
    r0 = ref.initial_inference(obs.cpu().double())
    r1 = ref.recurrent_inference(r0.hidden_state, acts.cpu())
  torch.cuda.synchronize()
  for got, want in ((s0.value, r0.value), (s1.value, r1.value), (s1.reward, r1.reward)):
    got, want = got.cpu().double().reshape(-1), want.reshape(-1)
    e = float(((got - want).abs() / want.abs().clamp(min=1.0)).max())
    print("%s %s search network vs float64: %.3g" % (sup, precision, e))
    assert e <= 5e-4
