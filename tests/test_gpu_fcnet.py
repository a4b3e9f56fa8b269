"""GPU tests of the fused FCNetwork kernels against the reference's torch module (golden outputs
from networks.FCNetwork on CPU, float32) and of the FC-specialised search against the oracle."""
import types

import numpy as np
import pytest
import torch

import oracle
from helpers import load

pytestmark = pytest.mark.gpu

# float32 kernels vs torch float32 (different summation order): stated tolerance
RTOL, ATOL = 1e-4, 2e-5


def _net_from_golden(g, obs_dim, A, precision="f32"):
  from model_based_rl_b200.networks import FCNetwork
  cfg = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=False,
                              no_target_transform=False)
  net = FCNetwork(obs_dim, A, "cuda", cfg, precision=precision)
  net.load_weights({k[2:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("w_")})
  return net


@pytest.mark.parametrize("precision", ["f32", "tf32x3"])
@pytest.mark.parametrize("name,obs_dim,A", [("atari18", 128, 18), ("ttt", 9, 9)])
def test_fc_f32_matches_torch_reference(name, obs_dim, A, precision):
  """Both float32-accurate paths (CUDA cores; tensor cores with three TF32 products per multiply) against the
  outputs of the reference's torch module, at the same bars."""
  g = load("fcnet_" + name)
  net = _net_from_golden(g, obs_dim, A, precision)
  obs = torch.from_numpy(g["obs"]).cuda()
  init = net.initial_inference(obs)
  torch.cuda.synchronize()
  assert init.reward == 0
  assert np.allclose(init.hidden_state.cpu().numpy(), g["init_hidden"], rtol=RTOL, atol=ATOL)
  assert np.allclose(init.policy_logits.cpu().numpy(), g["init_logits"], rtol=RTOL, atol=ATOL)
  # value goes through h^-1 in float32, which amplifies 1-ulp differences to ~1e-4 (see DESIGN.md)
  assert np.allclose(init.value.cpu().numpy(), g["init_value"], rtol=1e-3, atol=1e-3)
  rec = net.recurrent_inference(torch.from_numpy(g["init_hidden"]).cuda(), g["actions"].tolist())
  torch.cuda.synchronize()
  assert np.allclose(rec.hidden_state.cpu().numpy(), g["rec_hidden"], rtol=RTOL, atol=ATOL)
  assert np.allclose(rec.policy_logits.cpu().numpy(), g["rec_logits"], rtol=RTOL, atol=ATOL)
  assert np.allclose(rec.value.cpu().numpy(), g["rec_value"], rtol=1e-3, atol=1e-3)
  assert np.allclose(rec.reward.cpu().numpy(), g["rec_reward"], rtol=1e-3, atol=1e-3)
  # state dict round trip keeps the reference's keys
  sd = net.get_weights()
  assert set(sd) == {k[2:] for k in g if k.startswith("w_")}
  assert np.array_equal(sd["LN.weight"].numpy(), g["w_LN.weight"])


@pytest.mark.parametrize("precision", ["f32", "tf32x3", "bf16"])
def test_fc_no_support_matches_torch_reference(precision):
  """`--no_support` networks (config.py:95; networks.py:135-136, 153, 161): one-unit value / reward heads whose raw
  outputs are the scalars, against outputs of the reference's FCNetwork(no_support=True).  Asking for the default
  bf16 precision gives the float32-accurate tensor-core kernels (the bf16 kernels are built around the support heads
  and refuse such weights)."""
  from model_based_rl_b200.networks import FCNetwork, FCSearch
  g = load("fcnet_nosupport")
  cfg = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=True,
                              no_target_transform=False)
  net = FCNetwork(8, 4, "cuda", cfg, precision=precision)
  assert net.precision == ("tf32x3" if precision == "bf16" else precision)
  net.load_weights({k[2:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("w_")})
  init = net.initial_inference(torch.from_numpy(g["obs"]).cuda())
  rec = net.recurrent_inference(torch.from_numpy(g["init_hidden"]).cuda(), g["actions"].tolist())
  torch.cuda.synchronize()
  for got, want in ((init.hidden_state, "init_hidden"), (init.policy_logits, "init_logits"), (init.value, "init_value"),
                    (rec.hidden_state, "rec_hidden"), (rec.policy_logits, "rec_logits"), (rec.value, "rec_value"),
                    (rec.reward, "rec_reward")):
    assert got.shape == g[want].shape
    assert np.allclose(got.cpu().numpy(), g[want], rtol=RTOL, atol=ATOL), want
  # and a search on it: per-launch path, tree bit-exact against the oracle's replay of the recorded outputs
  G, A, S = 96, 4, 20
  scfg = types.SimpleNamespace(num_simulations=S, action_space=A, two_players=False, discount=0.997,
                               pb_c_base=19652, pb_c_init=1.25, init_value_score=0.0, known_bounds=[None, None],
                               root_exploration_fraction=0.25)
  rng = np.random.default_rng(3)
  noise, u = rng.dirichlet([0.25] * A, size=G), rng.random(G)
  fs = FCSearch(scfg, net, G, use_graph=True, num_streams=2)
  assert fs.fused is None
  fs.enable_record()
  actions, root_value, child_visits, init_value = fs.search_host(rng.normal(size=(G, 8)).astype(np.float32), noise, u,
                                                                 np.ones(G))
  want = oracle.search(oracle.make_cfg(S, A, False, 0.997), fs.root_logits.cpu().numpy(), noise=noise, noise_frac=0.25,
                       rec_value=fs.record[0].cpu().numpy().T, rec_reward=fs.record[1].cpu().numpy().T,
                       rec_logits=fs.record[2].cpu().numpy().transpose(1, 0, 2))
  assert np.array_equal(fs.visits.cpu().numpy(), want["visits"])
  assert np.array_equal(root_value.numpy(), want["root_value"])


def test_bf16_kernels_refuse_no_support_weights():
  """The C ABI of the bf16 kernels answers MZ_ERR_UNSUPPORTED for a weights struct with no_support set."""
  from model_based_rl_b200 import _lib
  from model_based_rl_b200.networks import FCNetwork
  cfg = types.SimpleNamespace(value_support=[-15, 15], reward_support=[-15, 15], no_support=True,
                              no_target_transform=False)
  g = load("fcnet_nosupport")
  net = FCNetwork(8, 4, "cuda", cfg)
  net.load_weights({k[2:]: torch.from_numpy(v) for k, v in g.items() if k.startswith("w_")})
  buf = torch.zeros(1 << 20, dtype=torch.uint8, device="cuda")
  tail = torch.zeros(512, dtype=torch.float32, device="cuda")
  rc = net.lib.mz_fc_tc_pack(net.weights, _lib.ptr(buf), _lib.ptr(tail), _lib.current_stream())
  assert rc == -2  # MZ_ERR_UNSUPPORTED


@pytest.mark.parametrize("name,obs_dim,A", [("atari18", 128, 18), ("ttt", 9, 9)])
@pytest.mark.parametrize("batch", [1, 31, 129, 1000])
def test_fc_tf32x3_matches_f32_kernel(name, obs_dim, A, batch):
  """mz_fc_*_tf32x3 (split-TF32 tensor-core products) against the CUDA-core float32 kernels on the same weights:
  float32 rounding level (different summation order only) -- 2e-5 on hidden states and logits; the scalars go
  through softmax + h^-1, which amplifies last-bit differences (same bar as against torch).  Ragged last CTAs,
  gather through in_index / scatter at an offset like the search engine's calls."""
  g = load("fcnet_" + name)
  tc = _net_from_golden(g, obs_dim, A, "tf32x3")
  f32 = _net_from_golden(g, obs_dim, A, "f32")
  gen = torch.Generator(device="cuda").manual_seed(11 + batch)
  obs = torch.rand((batch, obs_dim), device="cuda", generator=gen)
  a, b = f32.initial_inference(obs), tc.initial_inference(obs)
  torch.cuda.synchronize()
  for x, y, tol in ((a.hidden_state, b.hidden_state, 2e-5), (a.policy_logits, b.policy_logits, 2e-5),
                    (a.value, b.value, 1e-3)):
    assert torch.allclose(x, y, rtol=tol, atol=tol), (x - y).abs().max().item()
  # raw form: three candidate parent rows per game, the kernel picks in_index[b]; output at slot 3
  pool = torch.rand((batch, 4, 50), device="cuda", generator=gen) * 2.0
  idx = torch.randint(0, 3, (batch,), device="cuda", generator=gen, dtype=torch.int32)
  act = torch.randint(0, A, (batch,), device="cuda", generator=gen, dtype=torch.int32)
  outs = []
  for net in (f32, tc):
    p = pool.clone()
    v, r = torch.empty((batch, 1), device="cuda"), torch.empty((batch, 1), device="cuda")
    l = torch.empty((batch, A), device="cuda")
    net.recurrent_into(p, 200, idx, act, p, 200, 150, v, r, l)
    torch.cuda.synchronize()
    assert torch.equal(p[:, :3], pool[:, :3])
    outs.append((p[:, 3].clone(), l, v, r))
  for x, y, tol in zip(outs[0], outs[1], (2e-5, 2e-5, 1e-3, 1e-3)):
    assert torch.allclose(x, y, rtol=tol, atol=tol), (x - y).abs().max().item()


@pytest.mark.parametrize("name,obs_dim,A", [("atari18", 128, 18), ("ttt", 9, 9)])
@pytest.mark.parametrize("batch", [64, 129, 1000])
def test_fc_tensor_core_matches_f32(name, obs_dim, A, batch):
  """tcgen05 bf16 kernel vs the float32 kernel (and, at B=64, torch's float32 golden).
  Tolerance: bf16 operands (8-bit mantissa) through four layers, fp32 accumulation."""
  g = load("fcnet_" + name)
  f32 = _net_from_golden(g, obs_dim, A, "f32")
  tc = _net_from_golden(g, obs_dim, A, "bf16")
  rng = np.random.default_rng(batch)
  if batch == 64:
    hidden = torch.from_numpy(g["init_hidden"]).cuda()
    actions = torch.from_numpy(g["actions"]).cuda()
  else:
    hidden = torch.from_numpy(np.maximum(rng.normal(0.3, 0.7, size=(batch, 50)), 0).astype(np.float32)).cuda()
    actions = torch.from_numpy(rng.integers(0, A, size=batch, dtype=np.int32)).cuda()
  a = f32.recurrent_inference(hidden, actions)
  b = tc.recurrent_inference(hidden, actions)
  torch.cuda.synchronize()
  for name_, x, y in (("hidden", a.hidden_state, b.hidden_state), ("logits", a.policy_logits, b.policy_logits),
                      ("value", a.value, b.value), ("reward", a.reward, b.reward)):
    x, y = x.cpu().numpy(), y.cpu().numpy()
    assert np.isfinite(y).all(), name_
    err = np.abs(x - y).max()
    scale = max(1.0, np.abs(x).max())
    assert err <= 3e-2 * scale, "%s: max abs err %g (scale %g)" % (name_, err, scale)
  if batch == 64:
    # the bf16 kernel against the REFERENCE's own outputs (torch float32 FCNetwork, eval mode) directly:
    # logits / hidden within 3e-2 absolute, the value / reward scalars (after softmax expectation + h^-1,
    # which stretches support-space errors by up to |dh^-1/dx| ~ 2 + 0.1 |v|) within 5e-2 absolute
    assert np.allclose(b.policy_logits.cpu().numpy(), g["rec_logits"], rtol=0, atol=3e-2)
    assert np.allclose(b.hidden_state.cpu().numpy(), g["rec_hidden"], rtol=0, atol=3e-2)
    for name_, got, want in (("value", b.value, g["rec_value"]), ("reward", b.reward, g["rec_reward"])):
      err = np.abs(got.cpu().numpy().reshape(-1) - want.reshape(-1))
      print("bf16 %s vs reference golden: max abs err %.4g (|scalar| up to %.3g)" % (name_, err.max(), np.abs(want).max()))
      assert err.max() <= 5e-2, name_


@pytest.mark.parametrize("name,obs_dim,A", [("atari18", 128, 18), ("ttt", 9, 9)])
@pytest.mark.parametrize("batch", [64, 300])
def test_fc_initial_tensor_core_matches_f32(name, obs_dim, A, batch):
  """initial_inference on the tcgen05 kernel (representation + prediction heads) vs the float32
  kernel and, at B=64, the reference golden.  Same bf16 tolerance as the recurrent kernel."""
  g = load("fcnet_" + name)
  f32 = _net_from_golden(g, obs_dim, A, "f32")
  tc = _net_from_golden(g, obs_dim, A, "bf16")
  assert tc._tc_init_packed is not None
  rng = np.random.default_rng(batch)
  obs = (torch.from_numpy(g["obs"]) if batch == 64 else
         torch.from_numpy(rng.random((batch, obs_dim)).astype(np.float32))).cuda()
  a = f32.initial_inference(obs)
  b = tc.initial_inference(obs)
  torch.cuda.synchronize()
  assert b.reward == 0
  for name_, x, y in (("hidden", a.hidden_state, b.hidden_state), ("logits", a.policy_logits, b.policy_logits),
                      ("value", a.value, b.value)):
    x, y = x.cpu().numpy(), y.cpu().numpy()
    assert np.isfinite(y).all(), name_
    err = np.abs(x - y).max()
    assert err <= 3e-2 * max(1.0, np.abs(x).max()), "%s: max abs err %g" % (name_, err)
  if batch == 64:
    assert np.allclose(b.hidden_state.cpu().numpy(), g["init_hidden"], rtol=0, atol=3e-2)
    assert np.allclose(b.policy_logits.cpu().numpy(), g["init_logits"], rtol=0, atol=3e-2)
    err = np.abs(b.value.cpu().numpy().reshape(-1) - g["init_value"].reshape(-1))
    print("bf16 initial value vs reference golden: max abs err %.4g" % err.max())
    assert err.max() <= 5e-2


def test_fc_search_replays_bit_exact_in_oracle():
  """Full move with the real FC network (C4 shape, fewer games): the engine records what the
  network returned for every simulation; the oracle replays the search with those outputs."""
  from model_based_rl_b200.networks import FCSearch
  g = load("fcnet_atari18")
  net = _net_from_golden(g, 128, 18, "bf16")
  G, A, S = 256, 18, 50
  cfg = types.SimpleNamespace(num_simulations=S, action_space=A, two_players=False, discount=0.997,
                              pb_c_base=19652, pb_c_init=1.25, init_value_score=0.0,
                              known_bounds=[None, None], root_exploration_fraction=0.25)
  rng = np.random.default_rng(7)
  obs = rng.normal(size=(G, 128)).astype(np.float32)
  noise = rng.dirichlet([0.25] * A, size=G)
  u = rng.random(G)
  temp = rng.choice([0.0, 0.25, 1.0], size=G)
  for use_graph, streams, fused in ((False, 1, False), (True, 1, False), (True, 3, False), (False, 1, True),
                                    (True, 1, True)):
    fs = FCSearch(cfg, net, G, use_graph=use_graph, num_streams=streams, fused=fused)
    fs.enable_record()
    actions, root_value, child_visits, init_value = fs.search_host(obs, noise, u, temp)
    if use_graph:  # replay the captured graph once more: results must be identical
      a2 = actions.clone()
      actions, root_value, child_visits, init_value = fs.search_host(obs, noise, u, temp)
      assert torch.equal(a2, actions)
    ocfg = oracle.make_cfg(S, A, False, 0.997)
    want = oracle.search(ocfg, fs.root_logits.cpu().numpy(), noise=noise, noise_frac=0.25,
                         rec_value=fs.record[0].cpu().numpy().T, rec_reward=fs.record[1].cpu().numpy().T,
                         rec_logits=fs.record[2].cpu().numpy().transpose(1, 0, 2))
    assert np.array_equal(fs.trace[0].cpu().numpy().T, want["trace_parent"])
    assert np.array_equal(fs.trace[1].cpu().numpy().T, want["trace_action"])
    assert np.array_equal(fs.visits.cpu().numpy(), want["visits"])
    assert np.array_equal(root_value.numpy(), want["root_value"])
    cv = want["visits"] / want["visits"].sum(1, keepdims=True)
    assert np.array_equal(child_visits.numpy(), cv)
    for i in range(G):
      assert int(actions[i]) == oracle.select_action(want["visits"][i], temp[i], u[i])
    assert fs.launches_per_move == (3 if fused else streams * (2 * S + 5))


def test_fc_search_tf32x3_replays_bit_exact_in_oracle():
  """The same move with the float32-accurate tensor-core network (per-launch path, graph + three slices): the tree
  the engine builds from the kernel's outputs is the oracle's, bit for bit; and its root values stay within the
  float32 kernels' distance of the CUDA-core float32 network's (the search amplifies nothing here: same visits
  for nearly every game)."""
  from model_based_rl_b200.networks import FCSearch
  g = load("fcnet_atari18")
  G, A, S = 200, 18, 50
  cfg = types.SimpleNamespace(num_simulations=S, action_space=A, two_players=False, discount=0.997,
                              pb_c_base=19652, pb_c_init=1.25, init_value_score=0.0,
                              known_bounds=[None, None], root_exploration_fraction=0.25)
  rng = np.random.default_rng(17)
  obs = rng.random(size=(G, 128)).astype(np.float32)
  noise = rng.dirichlet([0.25] * A, size=G)
  u = rng.random(G)
  temp = np.ones(G)
  visits = {}
  for precision in ("tf32x3", "f32"):
    net = _net_from_golden(g, 128, 18, precision)
    fs = FCSearch(cfg, net, G, use_graph=True, num_streams=3)
    assert fs.fused is None
    fs.enable_record()
    actions, root_value, child_visits, init_value = fs.search_host(obs, noise, u, temp)
    ocfg = oracle.make_cfg(S, A, False, 0.997)
    want = oracle.search(ocfg, fs.root_logits.cpu().numpy(), noise=noise, noise_frac=0.25,
                         rec_value=fs.record[0].cpu().numpy().T, rec_reward=fs.record[1].cpu().numpy().T,
                         rec_logits=fs.record[2].cpu().numpy().transpose(1, 0, 2))
    assert np.array_equal(fs.trace[0].cpu().numpy().T, want["trace_parent"])
    assert np.array_equal(fs.visits.cpu().numpy(), want["visits"])
    assert np.array_equal(root_value.numpy(), want["root_value"])
    visits[precision] = (fs.visits.cpu().numpy().copy(), root_value.numpy().copy())
  same = (visits["tf32x3"][0] == visits["f32"][0]).all(axis=1)
  print("games with identical visit counts under both float32 networks: %d / %d" % (same.sum(), G))
  assert same.mean() >= 0.9
  assert np.allclose(visits["tf32x3"][1][same], visits["f32"][1][same], rtol=1e-3, atol=1e-3)


def _search_cfg(S, A, two_players=False, discount=0.997, known_bounds=(None, None), value_support=(-15, 15),
                reward_support=(-15, 15), no_target_transform=False):
  return types.SimpleNamespace(
      num_simulations=S, action_space=A, two_players=two_players, discount=discount, pb_c_base=19652,
      pb_c_init=1.25, init_value_score=0.0, known_bounds=list(known_bounds), root_exploration_fraction=0.25,
      value_support=list(value_support), reward_support=list(reward_support), no_support=False,
      no_target_transform=no_target_transform)


@pytest.mark.parametrize("shape", ["atari18", "ttt9", "lunar4", "wide32", "ties6", "asym5_nott", "edge13"])
def test_fused_search_equals_per_launch_search(shape):
  """mz_fc_search (the whole move in one persistent kernel, clusters of 4 CTAs) against the
  per-simulation launches of mz_tree_step + mz_fc_recurrent_tc on the same inputs: identical network
  outputs at every simulation (same MMA sequence on the same bf16 operands), identical (parent, action,
  depth) traces, visit counts, root values, MinMax bounds, child-visit distributions and selected
  actions -- bit for bit -- and the same trees (priors, children, value sums, visit counts, rewards).
  Game counts are not multiples of the 128-game tile (absent rows), TTT has legal masks, two players
  and known bounds; `ties6` runs a network whose policy head is zero (all priors equal at every node: every
  unexpanded-child choice is a tie broken by the action index); `asym5_nott` has a 32-bin value support
  [-4, 27], a 9-bin reward support [-2, 6] and raw expectations (no_target_transform), with support logits
  spread x16.  `wide32` (S = 19) and `edge13` (S = 63) are the largest trees the kernel takes at A = 32 and at
  A = 13: `edge13` has the largest shared-memory plan of all shapes (217 248 of 232 448 bytes)."""
  from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict
  G, A, S, D, two, disc, kb = {"atari18": (300, 18, 50, 128, False, 0.997, (None, None)),
                               "ttt9": (130, 9, 30, 9, True, 1.0, (-1, 1)),
                               "lunar4": (257, 4, 30, 8, False, 0.997, (None, None)),
                               "wide32": (100, 32, 19, 16, False, 0.99, (None, None)),
                               "ties6": (140, 6, 40, 12, False, 0.997, (None, None)),
                               "asym5_nott": (150, 5, 25, 10, False, 0.997, (None, None)),
                               "edge13": (200, 13, 63, 24, False, 0.997, (None, None))}[shape]
  vs, rs, nott = ((-4, 27), (-2, 6), True) if shape == "asym5_nott" else ((-15, 15), (-15, 15), False)
  cfg = _search_cfg(S, A, two, disc, kb, vs, rs, nott)
  net = FCNetwork(D, A, "cuda", cfg)
  sd = random_state_dict(D, A, vs[1] - vs[0] + 1, rs[1] - rs[0] + 1, seed=11)
  if shape == "asym5_nott":
    for k in ("value_head.value", "reward_head.reward"):
      sd[k + ".weight"], sd[k + ".bias"] = sd[k + ".weight"] * 16, sd[k + ".bias"] * 16
  if shape == "ties6":
    sd["policy_head.policy.weight"] = torch.zeros_like(sd["policy_head.policy.weight"])
    sd["policy_head.policy.bias"] = torch.zeros_like(sd["policy_head.policy.bias"])
  net.load_weights(sd)
  rng = np.random.default_rng(5)
  obs = rng.normal(size=(G, D)).astype(np.float32)
  legal = to_play = None
  noise = rng.dirichlet([0.25] * A, size=G)
  if shape == "ttt9":
    legal = rng.integers(1, 1 << A, size=G).astype(np.int32)
    to_play = rng.choice([-1, 1], size=G).astype(np.int8)
    noise = np.zeros((G, A))
    for i in range(G):
      n = bin(int(legal[i])).count("1")
      noise[i, :n] = rng.dirichlet([0.25] * n)
  u, temp = rng.random(G), rng.choice([0.0, 0.5, 1.0], size=G)
  outs = []
  for fused in (False, True):
    fs = FCSearch(cfg, net, G, use_graph=False, num_streams=1, fused=fused)
    fs.enable_record()
    r = fs.search_host(obs, noise, u, temp, legal=legal, to_play=to_play)
    torch.cuda.synchronize()
    if fused:
      assert int(fs.fused.error_flag.item()) == 0
    eng = fs.fused if fused else fs.eng
    trees = [eng.export_game(g) for g in (0, G // 2, G - 1)]
    outs.append(dict(actions=r[0].clone(), root_value=r[1].clone(), child_visits=r[2].clone(),
                     init_value=r[3].clone(), visits=fs.visits.cpu(), minmax=fs.minmax.cpu(),
                     record=[t.cpu() for t in fs.record], trace=[t.cpu() for t in fs.trace], trees=trees))
  a, b = outs
  for i, name in enumerate(("value", "reward", "logits")):
    assert torch.equal(a["record"][i], b["record"][i]), "network %s differs" % name
  for i, name in enumerate(("parent", "action", "depth")):
    assert torch.equal(a["trace"][i], b["trace"][i]), "trace %s differs" % name
  for k in ("visits", "root_value", "child_visits", "minmax", "actions", "init_value"):
    assert torch.equal(a[k], b[k]), k
  for ta, tb in zip(a["trees"], b["trees"]):
    for k in ("prior", "child", "vsum", "visit", "reward"):
      assert np.array_equal(ta[k], tb[k]), "tree %s differs" % k


def test_search_outside_fused_plan_runs_per_launch():
  """A = 18, S = 60 lies outside the persistent kernel's plan (S <= 55 at 18 actions): the default engine is the
  per-launch path, and asking for the fused kernel is an error."""
  from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict
  G, A, S, D = 130, 18, 60, 32
  cfg = _search_cfg(S, A)
  net = FCNetwork(D, A, "cuda", cfg)
  net.load_weights(random_state_dict(D, A, seed=3))
  fs = FCSearch(cfg, net, G, fused=None)
  assert fs.fused is None and len(fs.lanes) == 1
  with pytest.raises(ValueError):
    FCSearch(cfg, net, G, fused=True)


def test_search_after_load_weights_uses_new_weights():
  """Weight hand-off (Learner.send_weights -> network.load_weights): launch plans and CUDA graphs captured
  before the hand-off hold device pointers; load_weights refills the same storage, so the next search runs
  on the new weights -- same result as an engine built after the load -- and the network holds a snapshot
  (later in-place changes of the source tensors do not leak in)."""
  from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict
  G, A, S, D = 192, 6, 16, 32
  cfg = _search_cfg(S, A)
  rng = np.random.default_rng(21)
  obs = rng.normal(size=(G, D)).astype(np.float32)
  noise, u, temp = rng.dirichlet([0.25] * A, size=G), rng.random(G), np.ones(G)
  sd1 = random_state_dict(D, A, seed=1)
  sd2 = random_state_dict(D, A, seed=2)
  for fused in (False, True):
    net = FCNetwork(D, A, "cuda", cfg)
    net.load_weights(sd1)
    fs = FCSearch(cfg, net, G, use_graph=True, num_streams=2, fused=fused)
    first = [t.clone() for t in fs.search_host(obs, noise, u, temp)]
    live = {k: v.clone().cuda() for k, v in sd2.items()}
    net.load_weights(live)
    for v in live.values():
      v.add_(1.0)  # the caller's tensors change after the hand-off (an optimiser step): no effect
    second = [t.clone() for t in fs.search_host(obs, noise, u, temp)]
    fresh_net = FCNetwork(D, A, "cuda", cfg)
    fresh_net.load_weights(sd2)
    fresh = FCSearch(cfg, fresh_net, G, use_graph=False, num_streams=1, fused=fused)
    want = [t.clone() for t in fresh.search_host(obs, noise, u, temp)]
    assert not torch.equal(first[2], second[2])
    for x, y in zip(second, want):
      assert torch.equal(x, y)


@pytest.mark.gpu
def test_search_host_uint8_observations_equal_float_observations():
  """Byte observations normalised on the device ((x - min) / range in float32, actors.py:127-129) give
  the same search, bit for bit, as the host-normalised float32 observations -- default 0 / 255 and an
  explicit per-feature range."""
  import types
  import numpy as np
  import torch
  from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict
  G, A, S, D = 200, 4, 12, 128
  cfg = types.SimpleNamespace(
      num_simulations=S, action_space=A, two_players=False, discount=0.997, pb_c_base=19652, pb_c_init=1.25,
      init_value_score=0.0, known_bounds=[None, None], root_exploration_fraction=0.25,
      value_support=[-15, 15], reward_support=[-15, 15], no_support=False, no_target_transform=False)
  net = FCNetwork(D, A, "cuda", cfg)
  net.load_weights(random_state_dict(D, A))
  fs = FCSearch(cfg, net, G, num_streams=2)
  rng = np.random.default_rng(3)
  obs_u8 = rng.integers(0, 256, size=(G, D)).astype(np.uint8)
  noise, u, temp = rng.dirichlet([0.25] * A, size=G), rng.random(G), np.ones(G)
  for mn, rg in ((None, None), (rng.integers(0, 4, D).astype(np.float32), rng.integers(200, 256, D).astype(np.float32))):
    if mn is None:
      want_obs = obs_u8.astype(np.float32) / np.float32(255)
    else:
      fs.set_obs_normalization(mn, rg)
      want_obs = (obs_u8.astype(np.float32) - mn) / rg
    a = [t.clone() for t in fs.search_host(want_obs, noise, u, temp)]
    visits_a = fs.visits.clone()
    b = [t.clone() for t in fs.search_host(obs_u8, noise, u, temp)]
    assert np.array_equal(fs.obs.cpu().numpy(), want_obs)
    assert torch.equal(visits_a, fs.visits)
    for x, y in zip(a, b):
      assert torch.equal(x, y)


@pytest.mark.gpu
def test_search_pinned_equals_search_host():
  """Inputs written into the engine's pinned blob views + one copy per direction give what the per-array
  call gives (legal masks and to_play included)."""
  import types
  import numpy as np
  import torch
  from model_based_rl_b200.networks import FCNetwork, FCSearch, random_state_dict
  G, A, S, D = 130, 9, 10, 9
  cfg = types.SimpleNamespace(
      num_simulations=S, action_space=A, two_players=True, discount=1.0, pb_c_base=19652, pb_c_init=1.25,
      init_value_score=0.0, known_bounds=[-1, 1], root_exploration_fraction=0.25,
      value_support=[-15, 15], reward_support=[-15, 15], no_support=False, no_target_transform=False)
  net = FCNetwork(D, A, "cuda", cfg, precision="f32")
  net.load_weights(random_state_dict(D, A))
  rng = np.random.default_rng(9)
  obs_u8 = rng.integers(0, 3, size=(G, D)).astype(np.uint8)
  legal = rng.integers(1, 1 << A, size=G).astype(np.int32)
  to_play = rng.choice([-1, 1], size=G).astype(np.int8)
  noise = np.zeros((G, A))
  for i in range(G):
    n = bin(int(legal[i])).count("1")
    noise[i, :n] = rng.dirichlet([0.25] * n)
  u, temp = rng.random(G), rng.choice([0.0, 0.5, 1.0], size=G)
  outs = []
  for mode in ("host", "pinned"):
    fs = FCSearch(cfg, net, G, num_streams=2)
    fs.set_obs_normalization(np.ones(D, np.float32), np.full(D, 2.0, np.float32))
    if mode == "host":
      r = fs.search_host(obs_u8, noise, u, temp, legal=legal, to_play=to_play)
    else:
      pin = fs.pinned_inputs()
      for name, src in (("obs_u8", obs_u8), ("noise", noise), ("uniforms", u), ("temperature", temp),
                        ("legal", legal), ("to_play", to_play)):
        pin[name].copy_(torch.from_numpy(src))
      r = fs.search_pinned()
    outs.append([t.clone() for t in r] + [fs.visits.cpu()])
    for g in range(G):
      assert (int(legal[g]) >> int(r[0][g])) & 1  # only legal actions are played
  for x, y in zip(*outs):
    assert torch.equal(x, y)
