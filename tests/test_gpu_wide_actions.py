"""Search, self-play and learning with 33 to 64 actions on the B200 (the tree kernels' two-actions-per-lane
instantiation and the [G][W] legal-mask words).  Searches are checked bit for bit against the pure-Python port of the
reference's search (tests/wide_ref.py: legal subsets of any width) and against the C oracle where every root action
is legal; the rest against the same bars as the existing tests at fewer actions."""
import types

import numpy as np
import pytest
import torch

import oracle
import wide_ref

pytestmark = pytest.mark.gpu

HK = dict(value_scale=1.0, reward_scale=0.5, logit_scale=2.0, reward_density=3)


def _cfg(S, A, two_players=False, known_bounds=(None, None)):
  return dict(num_simulations=S, action_space=A, two_players=two_players, discount=1.0 if two_players else 0.997,
              pb_c_base=19652, pb_c_init=1.25, init_value_score=0.0, known_bounds=tuple(known_bounds))


def _ns(cfg, **extra):
  d = dict(cfg, known_bounds=list(cfg["known_bounds"]), root_exploration_fraction=0.25, value_support=[-15, 15],
           reward_support=[-15, 15], no_support=False, no_target_transform=False)
  d.update(extra)
  return types.SimpleNamespace(**d)


@pytest.fixture(params=["staged_4_games_per_cta", "staged_1_game_per_cta", "global_memory"])
def tree_mode(request):
  """The step kernel on a shared-memory image (four games per CTA or one) and on the global blocks directly."""
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  lib.mz_tree_set_games_per_block(1 if request.param == "staged_1_game_per_cta" else 4)
  lib.mz_debug_set_tree_staging(1 if request.param == "global_memory" else 0)
  yield request.param
  lib.mz_tree_set_games_per_block(0)
  lib.mz_debug_set_tree_staging(0)


# (G, A, S, players, bounds, legal kind, logit scale); G is never a multiple of the four games of a CTA
HASH_CASES = {
    "a33_subsets": (37, 33, 50, False, (None, None), "subsets", 2.0),
    "a50_two_players": (45, 50, 40, True, (-1.0, 1.0), "subsets", 2.0),
    "a64_zero_policy": (29, 64, 50, False, (None, None), "subsets", 0.0),
    "a64_all_legal": (515, 64, 50, False, (None, None), "all", 2.0),
}
_PORT = {}


def _hash_case(name):
  G, A, S, two, bounds, kind, scale = HASH_CASES[name]
  rng = np.random.default_rng(len(name) * 1000 + A)
  legal = wide_ref.random_legal(rng, G, A, only_high_rows=(1, 2)) if kind == "subsets" else np.ones((G, A), bool)
  root_state = rng.integers(0, 2**63 - 1, size=G, dtype=np.int64)
  noise = wide_ref.dense_noise(rng, legal)
  to_play = rng.choice([-1, 1], size=G).astype(np.int8) if two else np.ones(G, np.int8)
  return _cfg(S, A, two, bounds), dict(HK, logit_scale=scale), legal, root_state, noise, to_play, kind


def _engine_search(cfg, hk, legal_mask, root_state, noise, to_play):
  """BatchedMCTS through mz_tree_step: expand + backup of simulation s fused with the descent of s + 1."""
  from model_based_rl_b200.mcts import BatchedMCTS
  from model_based_rl_b200.testing import HashNetwork
  G, A, S = len(root_state), cfg["action_space"], cfg["num_simulations"]
  net = HashNetwork(A, device="cuda", **hk)
  state = torch.from_numpy(root_state).view(G, 1).cuda()
  init = net.initial_inference(state)
  eng = BatchedMCTS(_ns(cfg), G, hidden_words=2)
  eng.enable_trace()
  eng.set_root(init.policy_logits, legal_mask, noise, 0.25, to_play, state)
  eng.step(-1, gather=True)
  for sim in range(S):
    out = net.recurrent_inference(eng.gathered.view(torch.int64).view(G, 1), eng.leaf_action)
    eng.step(sim, out.value.reshape(G).contiguous(), out.reward.reshape(G).contiguous(), out.policy_logits.contiguous(),
             eng._hidden_words(out.hidden_state), gather=True)
  eng.root_stats()
  torch.cuda.synchronize()
  return eng, init.policy_logits.cpu().numpy()


@pytest.mark.parametrize("case", sorted(HASH_CASES))
def test_hash_search_matches_reference_port(case, tree_mode):
  cfg, hk, legal, root_state, noise, to_play, kind = _hash_case(case)
  G, A = legal.shape
  # the same masks in three host forms and the kernels' device words
  ints = [sum(1 << int(a) for a in np.nonzero(row)[0]) for row in legal]
  forms = {"all": None, "subsets": [legal, np.array(ints, np.uint64), ints][len(case) % 3]}
  eng, logits = _engine_search(cfg, hk, forms[kind], root_state, noise, to_play)
  if case not in _PORT:
    if kind == "all":  # every root action legal: the C oracle, which reads masks only up to 32 actions
      want = oracle.search(oracle.make_cfg(**cfg), logits, noise=noise, root_to_play=to_play,
                           hashnet=oracle.HashNet(hk["value_scale"], hk["reward_scale"], hk["logit_scale"],
                                                  hk["reward_density"]), root_state=root_state.astype(np.uint64))
      want["child_visits"] = want["visits"] / want["visits"].sum(1, keepdims=True)
    else:
      want = wide_ref.port_search(cfg, logits, legal, noise, to_play=to_play, hashnet=hk, root_state=root_state)
    _PORT[case] = want
  want = _PORT[case]
  assert np.array_equal(eng.trace[0].cpu().numpy().T, want["trace_parent"])
  assert np.array_equal(eng.trace[1].cpu().numpy().T, want["trace_action"])
  assert np.array_equal(eng.trace[2].cpu().numpy().T, want["trace_depth"])
  assert np.array_equal(eng.visits.cpu().numpy(), want["visits"])
  assert np.array_equal(eng.root_value.cpu().numpy(), want["root_value"])
  assert np.array_equal(eng.minmax.cpu().numpy(), want["minmax"])
  assert np.array_equal(eng.child_visits.cpu().numpy(), want["child_visits"])
  # Config.select_action at three temperatures, masks in the kernels' own word form
  rng = np.random.default_rng(5)
  lists = wide_ref.legal_lists(legal)
  words = torch.from_numpy(eng_words(legal)).cuda()
  for T in (0.0, 0.5, 1.0):
    u = rng.random(G)
    got = eng.select_action(np.full(G, T), u, words).cpu().numpy()
    for g in range(G):
      dense = want["visits"][g][lists[g]]
      assert got[g] == lists[g][oracle.select_action(dense, T, u[g])], (T, g)
  if kind == "subsets":
    assert (want["trace_action"][1:3][want["trace_parent"][1:3] == 0] >= 32).all()


def eng_words(legal):
  """bool [G, A] -> the kernels' int32 [G, W] mask words."""
  from model_based_rl_b200.mcts import legal_words
  return legal_words(legal, *legal.shape)


def _bits(legal_mask, G, A):
  """Any legal-mask form -> bool [G, A]."""
  from model_based_rl_b200.mcts import legal_words
  words = legal_words(legal_mask, G, A).view(np.uint32)
  return ((words[:, :, None] >> np.arange(32, dtype=np.uint32)) & 1).reshape(G, -1)[:, :A].astype(bool)


def _fc_net(D, A, precision, seed=3):
  from model_based_rl_b200.networks import FCNetwork, random_state_dict
  net = FCNetwork(D, A, "cuda", _ns(_cfg(1, A)), precision=precision)
  net.load_weights(random_state_dict(D, A, seed=seed))
  return net


@pytest.mark.parametrize("precision", ["tf32x3", "f32"])
def test_fc_search_64_actions_replays_bit_exact(precision):
  """FCSearch at 64 actions (per-launch path, CUDA graph, one and three slices): the recorded network outputs
  replayed by the reference port on legal subsets of both words, and by the C oracle with every action legal."""
  from model_based_rl_b200.networks import FCSearch
  G, A, S, D = 96, 64, 50, 32
  cfg = _cfg(S, A)
  net = _fc_net(D, A, precision)
  rng = np.random.default_rng(11)
  obs = rng.normal(size=(G, D)).astype(np.float32)
  legal = wide_ref.random_legal(rng, G, A, only_high_rows=(3,))
  legal[5] = True
  u, temp = rng.random(G), rng.choice([0.0, 0.5, 1.0], size=G)
  with pytest.raises(ValueError):
    FCSearch(_ns(cfg), net, G, fused=True)
  for streams, mask in ((1, "subsets"), (3, "subsets"), (3, "all")):
    fs = FCSearch(_ns(cfg), net, G, use_graph=True, num_streams=streams)
    assert fs.fused is None
    fs.enable_record()
    lg = legal if mask == "subsets" else np.ones((G, A), bool)
    noise = wide_ref.dense_noise(rng, lg)
    actions, root_value, child_visits, _ = fs.search_host(obs, noise, u, temp,
                                                          legal=(eng_words(lg) if mask == "subsets" else None))
    rec = [r.cpu().numpy() for r in fs.record]
    kw = dict(rec_value=rec[0].T, rec_reward=rec[1].T, rec_logits=rec[2].transpose(1, 0, 2))
    logits = fs.root_logits.cpu().numpy()
    if mask == "subsets":
      want = wide_ref.port_search(cfg, logits, lg, noise, **kw)
    else:
      want = oracle.search(oracle.make_cfg(**cfg), logits, noise=noise, **kw)
      want["child_visits"] = want["visits"] / want["visits"].sum(1, keepdims=True)
    assert np.array_equal(fs.trace[0].cpu().numpy().T, want["trace_parent"])
    assert np.array_equal(fs.trace[1].cpu().numpy().T, want["trace_action"])
    assert np.array_equal(fs.visits.cpu().numpy(), want["visits"])
    assert np.array_equal(root_value.numpy(), want["root_value"])
    assert np.array_equal(child_visits.numpy(), want["child_visits"])
    lists = wide_ref.legal_lists(lg)
    for g in range(G):
      assert int(actions[g]) == lists[g][oracle.select_action(want["visits"][g][lists[g]], temp[g], u[g])]


def test_mcts_run_b1_with_action_63_legal():
  """`MCTS(config).run(root, network)` at 64 actions with action 63 among the root's children."""
  from model_based_rl_b200.mcts import MCTS, Node
  from model_based_rl_b200.testing import HashNetwork
  A, S = 64, 40
  cfg = _cfg(S, A, True, (-1.0, 1.0))
  net = HashNetwork(A, device="cuda", **HK)
  rng = np.random.default_rng(63)
  for trial in range(3):
    legal = sorted(set(rng.choice(A, size=20, replace=False).tolist()) | {63})
    state = int(rng.integers(0, 2**62))
    init = net.initial_inference(torch.tensor([[state]], dtype=torch.int64, device="cuda"))
    root = Node(0)
    root.expand(init, 1, legal)
    paths = MCTS(_ns(cfg)).run(root, net)
    lb = np.zeros((1, A), bool)
    lb[0, legal] = True
    want = wide_ref.port_search(cfg, init.policy_logits.cpu().numpy(), lb, to_play=[1], hashnet=HK,
                                root_state=np.array([state]))
    assert [len(p) - 1 for p in paths] == list(want["trace_depth"][0])
    assert [root.children[a].visit_count for a in legal] == list(want["visits"][0][legal])
    assert root.value() == want["root_value"][0]


def test_dirichlet_noise_64_actions():
  """mz_dirichlet_noise with two mask words: rows dense over the legal actions, zeros behind their count,
  components Beta(alpha, (n - 1) alpha) (Kolmogorov-Smirnov against scipy and numpy), correlation -1 / (n - 1)."""
  from scipy import stats
  from model_based_rl_b200 import _lib
  lib = _lib.load()
  G, A, alpha = 20000, 64, 0.25
  rng = np.random.default_rng(0)
  legal = np.ones((G, A), bool)
  legal[G // 2:] = rng.random((G - G // 2, A)) < 0.5
  legal[G // 2:G // 2 + 500, :32] = False  # only high-word actions
  legal[legal.sum(1) == 0, 40] = True
  n = legal.sum(1)
  d_legal = torch.from_numpy(eng_words(legal)).cuda()
  out = torch.full((G, A), -1.0, dtype=torch.float64, device="cuda")

  def draw(seed, move):
    _lib.check(lib.mz_dirichlet_noise(G, A, alpha, _lib.ptr(d_legal), seed, move, _lib.ptr(out), None), "noise")
    torch.cuda.synchronize()
    return out.cpu().numpy().copy()
  x = draw(7, 0)
  assert np.allclose(x.sum(1), 1.0, atol=1e-12) and (x >= 0).all()
  assert all((x[g, n[g]:] == 0).all() and (x[g, :n[g]] > 0).all() for g in range(G // 2, G, 37))
  full = x[:G // 2]
  for col in (0, 31, 32, 63):
    assert stats.kstest(full[:, col], stats.beta(alpha, (A - 1) * alpha).cdf).pvalue > 1e-3
    assert stats.ks_2samp(full[:, col], rng.dirichlet([alpha] * A, size=G // 2)[:, col]).pvalue > 1e-3
  assert abs(np.corrcoef(full[:, 0], full[:, 40])[0, 1] + 1.0 / (A - 1)) < 0.03
  for k in (30, 32, 34):
    rows = np.nonzero((n == k) & (np.arange(G) >= G // 2))[0]
    if len(rows) > 300:
      assert stats.kstest(x[rows, k - 1], stats.beta(alpha, (k - 1) * alpha).cdf).pvalue > 1e-3
  assert np.array_equal(draw(7, 0), x) and not np.array_equal(draw(7, 1), x)
  assert lib.mz_dirichlet_noise(G, 65, alpha, None, 1, 0, _lib.ptr(out), None) == -1


class FillBoard64(object):
  """Test environment: G one-player games on 64 cells; a move fills an empty cell, the legal set shrinks every move
  (bit 63 included), reward +1 / -1 / 0 from a fixed pattern of cells, 24 moves per game."""
  num_actions = 64

  def __init__(self, num_games):
    self.num_games = int(num_games)
    self.board = np.zeros((self.num_games, 64), np.uint8)
    self.elapsed = np.zeros(self.num_games, np.int32)
    self.pattern = (np.arange(64) * 7 % 5).astype(np.int64) - 2

  def reset(self, which=None):
    idx = np.arange(self.num_games) if which is None else np.asarray(which)
    self.board[idx] = 0
    self.elapsed[idx] = 0
    return self.board[idx].copy()

  def legal_mask(self):
    empty = (self.board == 0).astype(np.uint64)
    return (empty << np.arange(64, dtype=np.uint64)).sum(axis=1, dtype=np.uint64)

  def step(self, actions):
    actions = np.asarray(actions, np.int64)
    g = np.arange(self.num_games)
    if (self.board[g, actions] != 0).any():
      raise ValueError("illegal move: the cell is taken")
    self.board[g, actions] = 1 + self.elapsed % 200
    self.elapsed += 1
    reward = np.clip(self.pattern[actions], -1, 1)
    done = self.elapsed >= 24
    return self.board.copy(), reward, done, np.where(done, 2, -1)


def test_device_actor_64_actions_fills_the_replay_like_the_list_path():
  """DeviceActor against BatchedActor + save_history at 64 actions with shrinking legal sets (uint64 masks from the
  environment): same moves, same replay buffer bit for bit; sampled policies are 64 wide."""
  from model_based_rl_b200.networks import FCSearch, FCNetwork, random_state_dict
  from model_based_rl_b200.replay_buffer import PrioritizedReplay
  from model_based_rl_b200.selfplay import BatchedActor, DeviceActor
  A, G, S, D, L, moves = 64, 70, 12, 64, 5, 30
  cfg = _ns(_cfg(S, A), root_dirichlet_alpha=0.25, num_unroll_steps=3, td_steps=4, max_history_length=L,
            max_steps=10 ** 9, batch_size=32, beta_increment_per_sampling=0.001, epsilon=0.01, alpha=0.8, beta=0.5,
            obs_space=(D,), window_size=600, window_step=None, seed=None, clip_rewards=False)
  net = FCNetwork(D, A, "cuda", cfg, precision="tf32x3")
  net.load_weights(random_state_dict(D, A, seed=3))
  temps = np.array([[1.0, 0.5, 0.0, 0.25][i % 4] for i in range(G)])
  rb_a, rb_b = PrioritizedReplay(cfg, window_positions=40000), PrioritizedReplay(cfg, window_positions=40000)
  fs_a, fs_b = FCSearch(cfg, net, G), FCSearch(cfg, net, G)
  assert fs_a.fused is None
  fs_b.set_obs_normalization(np.zeros(D, np.float32), np.ones(D, np.float32))
  list_actor = BatchedActor(cfg, net, FillBoard64(G), replay_buffer=rb_a, device="cuda", temperature=temps, search=fs_a)
  dev_actor = DeviceActor(cfg, FillBoard64(G), rb_b, fs_b, temperature=temps)
  rng = np.random.default_rng(17)
  for move in range(moves):
    legal = list_actor.env.legal_mask()
    assert np.array_equal(legal, dev_actor.env.legal_mask())
    noise = wide_ref.dense_noise(rng, _bits(legal, G, A))
    u = rng.random(G)
    a = list_actor.play_move(noise.copy(), u.copy())
    b = dev_actor.play_move(noise.copy(), u.copy())
    for x, y, name in zip(a, b, ("actions", "root_value", "child_visits", "errors", "done")):
      assert np.array_equal(np.asarray(x), np.asarray(y)), (move, name)
  torch.cuda.synchronize()
  assert dev_actor.games_played == list_actor.games_played > 0
  assert rb_a.size() == rb_b.size() > 0
  assert np.array_equal(rb_a.index.tree.cpu().numpy(), rb_b.index.tree.cpu().numpy())
  ia, ib = rb_a.index, rb_b.index
  live = ia.slot_chunk >= 0
  assert np.array_equal(live, ib.slot_chunk >= 0)
  pa, sa, la = ia.slot_pos.cpu().numpy(), ia.slot_start.cpu().numpy(), ia.slot_len.cpu().numpy()
  pb, sb, lb = ib.slot_pos.cpu().numpy(), ib.slot_start.cpu().numpy(), ib.slot_len.cpu().numpy()
  assert np.array_equal((pa - sa)[live], (pb - sb)[live]) and np.array_equal(la[live], lb[live])
  for k in ("w_obs", "w_actions", "w_rewards", "w_to_play", "w_root_values", "w_child_visits"):
    wa, wb = getattr(rb_a, k).cpu().numpy(), getattr(rb_b, k).cpu().numpy()
    for slot in np.nonzero(live)[0]:
      n = int(la[slot])
      assert np.array_equal(wa[sa[slot]:sa[slot] + n], wb[sb[slot]:sb[slot] + n]), (k, slot)
  (obs, actions, t_rewards, t_values, t_policies, *_), idxs, isw = rb_b.sample_batch_device()
  assert t_policies.shape[-1] == A and actions.shape[0] == cfg.batch_size
  assert torch.allclose(t_policies[:, 0].sum(-1).double(), torch.ones(cfg.batch_size, dtype=torch.float64,
                                                                      device="cuda"), atol=1e-5)


def _learner_case(A=64, D=24, B=48, K=3, seed=9):
  rng = np.random.default_rng(seed)
  cfg = types.SimpleNamespace(
      value_support=[-15, 15], reward_support=[-15, 15], no_support=False, no_target_transform=False,
      num_unroll_steps=K, optimizer="SGD", lr_init=0.0008, momentum=0.9, weight_decay=1e-4, clip_grad=0,
      lr_scheduler=None, norm_obs=False, send_weights_frequency=500, training_steps=2)
  obs = rng.normal(size=(B, D)).astype(np.float32)
  actions = rng.integers(0, A, size=(B, K))
  actions[0] = [63, 32, 31]
  t_rewards = rng.normal(size=(B, K + 1)).astype(np.float32)
  t_values = rng.normal(scale=3.0, size=(B, K + 1)).astype(np.float32)
  t_policies = rng.dirichlet([0.3] * A, size=(B, K + 1)).astype(np.float32)
  batch = ((obs, [list(map(int, r)) for r in actions], (t_rewards, t_values, t_policies)), None,
           rng.uniform(0.5, 1.0, size=B))
  return cfg, batch, D


def _learner_nets(cfg, D, A=64):
  from model_based_rl_b200 import fused_learner, learners
  from model_based_rl_b200.networks import random_state_dict
  w = random_state_dict(D, A, seed=21)
  net = fused_learner.FusedFCNetwork(D, A, "cuda", cfg)
  net.load_weights(w)
  ref = learners.FCNetworkTrain(D, A, "cuda", cfg)
  ref.load_weights(w)
  return net, ref


def test_fused_learner_f32_gradients_64_actions_match_autograd():
  """FusedLearner(precision='f32') at 64 actions (one-hot columns 32..63 in the recurrent inputs): losses, priority
  errors and every parameter gradient against torch autograd through FCNetworkTrain, at the bars of
  tests/test_fused_learner.py."""
  from model_based_rl_b200 import fused_learner, learners
  torch.backends.cuda.matmul.allow_tf32 = False
  cfg, batch, D = _learner_case()
  net, ref = _learner_nets(cfg, D)
  fused = fused_learner.FusedLearner(cfg, net, use_graph=False, precision="f32")
  fused._stage(batch)
  fused._forward_and_heads_backward()
  fused._recurrent_backward()
  torch_learner = learners.Learner(cfg, ref)
  losses, errs = torch_learner._forward_backward(fused.s_obs, fused.s_actions.long(), fused.s_tv, fused.s_tr,
                                                 fused.s_tp, fused.s_isw)
  torch.cuda.synchronize()
  np.testing.assert_allclose(fused.losses.cpu().numpy(), losses.cpu().numpy(), rtol=1e-5)
  np.testing.assert_allclose(fused.new_errors.cpu().numpy(), errs.cpu().numpy(), rtol=0, atol=1e-4)
  for name, p in ref.named_parameters():
    want, got = p.grad.cpu().numpy(), net.grads[name].cpu().numpy()
    assert np.abs(got - want).max() <= 2e-4 * (np.abs(want).max() + 1e-12), name
  # the one-hot block of the recurrent inputs: column d + a set for the step's action a
  xs = fused.xs.view(cfg.num_unroll_steps + 1, fused.B, -1)[0].cpu().numpy()
  assert xs[0, 50 + 63] == 1.0 and xs[0, 50:].sum() == 1.0


def test_bf16_learner_64_actions_against_f32_and_autograd_emulation():
  """precision='bf16' at 64 actions (d + A = 114 <= 128): the teacher-forced float64 emulation of the tensor-core
  rounding points at the bars of tests/test_fused_learner.py, and gradients as directions against the float32 step
  (cosine >= 0.98)."""
  from model_based_rl_b200 import fused_learner
  from test_fused_learner import _teacher_forced_check
  cfg, batch, D = _learner_case()
  out = {}
  for prec in ("f32", "bf16"):
    net, _ = _learner_nets(cfg, D)
    fused = fused_learner.FusedLearner(cfg, net, use_graph=False, precision=prec)
    fused._stage(batch)
    fused._forward_and_heads_backward()
    fused._recurrent_backward()
    torch.cuda.synchronize()
    out[prec] = (fused, net)
  _teacher_forced_check(out["bf16"][0], out["bf16"][1], 2e-3, 3e-3)
  np.testing.assert_allclose(out["bf16"][0].losses.cpu().numpy(), out["f32"][0].losses.cpu().numpy(), rtol=1e-2)
  for k, want in out["f32"][1].grads.items():
    a, b = out["bf16"][1].grads[k].double().flatten(), want.double().flatten()
    assert float((a @ b) / (a.norm() * b.norm() + 1e-300)) >= 0.98, k


def test_learner_step_64_actions():
  """One step of learners.Learner (torch modules) and of FusedLearner(precision='f32') from the same weights:
  losses within 1e-4 relative, weights within 2e-5."""
  from model_based_rl_b200 import fused_learner, learners
  torch.backends.cuda.matmul.allow_tf32 = False
  cfg, batch, D = _learner_case(seed=4)
  net, ref = _learner_nets(cfg, D)
  l_ref = learners.Learner(cfg, ref)
  l_fused = fused_learner.FusedLearner(cfg, net, use_graph=False, precision="f32")
  as_np = lambda x: x.detach().cpu().numpy() if torch.is_tensor(x) else np.asarray(x)
  a = l_ref.update_weights(batch)
  b = l_fused.update_weights(batch)
  np.testing.assert_allclose(as_np(b), as_np(a), rtol=1e-4)
  sd = net.state_dict()
  for k, v in ref.state_dict().items():
    np.testing.assert_allclose(sd[k].detach().cpu().numpy(), v.detach().cpu().numpy(), rtol=0, atol=2e-5, err_msg=k)


def test_more_than_64_actions_is_refused():
  from model_based_rl_b200 import _lib
  from model_based_rl_b200.mcts import BatchedMCTS
  with pytest.raises(ValueError):
    BatchedMCTS(_ns(_cfg(10, 65)), 4)
  lib = _lib.load()
  eng = BatchedMCTS(_ns(_cfg(10, 64)), 4)
  tree = _lib.Tree.from_buffer_copy(eng.tree)
  tree.num_actions = 65
  assert lib.mz_tree_set_root(tree, _lib.ptr(eng.root_value), None, None, 0.0, None, None, None) == -1
  assert lib.mz_tree_step(tree, -1, None, None, None, None, None, None, None, None, None) == -1
  visits = torch.zeros((4, 65), dtype=torch.int32, device="cuda")
  t = torch.zeros(4, dtype=torch.float64, device="cuda")
  assert lib.mz_select_action(4, 65, _lib.ptr(visits), None, _lib.ptr(t), _lib.ptr(t), _lib.ptr(eng.actions),
                              None) == -1
