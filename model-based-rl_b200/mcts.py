"""Search API of the reference (mcts.py) on top of the B200 tree kernels.

Mirrors the reference names and call shapes (SURVEY.md section 8b):

  MinMaxStats, Node, MCTS(config).run(root, network) -> search_paths       (mcts.py:6-145)

plus the batched engine those are built on:

  BatchedMCTS(config, num_games, ...).search(...)  -- thousands of independent games per call.

The tree lives in HBM as one contiguous block per game (layout: include/mzb200.h); every
simulation is: descent kernel -> one batched recurrent_inference -> expand+backup kernel.  There is
no CPU implementation of the search here: without a CUDA device this module raises.
"""
import math
import sys
from collections import namedtuple

import numpy as np
import torch

from . import _lib

NetworkOutput = namedtuple('network_output', ('value', 'reward', 'policy_logits', 'hidden_state'))


def default_prior_sum_mode():
  """mcts.py:53 uses builtin sum(); CPython >= 3.12 compensates (Neumaier), older ones do not."""
  return 1 if sys.version_info >= (3, 12) else 0


class MinMaxStats(object):
  """Running bounds of the Q values seen in one search (mcts.py:6-25)."""

  def __init__(self, minimum_bound=None, maximum_bound=None):
    self.reset(minimum_bound, maximum_bound)

  def reset(self, minimum_bound=None, maximum_bound=None):
    self.minimum = math.inf if minimum_bound is None else minimum_bound
    self.maximum = -math.inf if maximum_bound is None else maximum_bound

  def update(self, value):
    if value < self.minimum:
      self.minimum = value
    if value > self.maximum:
      self.maximum = value

  def normalize(self, value):
    if self.maximum > self.minimum:
      return (value - self.minimum) / (self.maximum - self.minimum)
    if self.maximum == self.minimum:
      return 1.0
    return value


class Node(object):
  """Host view of one tree node with the reference's attributes (mcts.py:28-61).

  Callers build the root exactly as with the reference (Node(0); root.expand(...);
  root.add_exploration_noise(...)); MCTS.run then fills visit counts, value sums, rewards and the
  expanded children back in from the device tree.
  """

  __slots__ = ('hidden_state', 'visit_count', 'value_sum', 'reward', 'children', 'prior', 'to_play')

  def __init__(self, prior):
    self.hidden_state = None
    self.visit_count = 0
    self.value_sum = 0
    self.reward = 0
    self.children = {}
    self.prior = prior
    self.to_play = 1

  def expanded(self):
    return len(self.children) > 0

  def value(self):
    if self.visit_count == 0:
      return 0
    return self.value_sum / self.visit_count

  def expand(self, network_output, to_play, actions):
    """Host-side expansion of a root (actors.py:142); float64 softmax over `actions` only."""
    self.to_play = to_play
    self.hidden_state = network_output.hidden_state
    reward = network_output.reward
    if torch.is_tensor(reward):
      reward = reward.item()
    if reward:
      self.reward = reward
    logits = network_output.policy_logits[0]
    weights = {int(a): math.exp(logits[int(a)].item()) for a in actions}
    total = sum(weights.values())
    self.children = {a: Node(w / total) for a, w in weights.items()}

  def add_exploration_noise(self, dirichlet_alpha, frac):
    actions = list(self.children.keys())
    noise = np.random.dirichlet([dirichlet_alpha] * len(actions))
    for a, n in zip(actions, noise):
      child = self.children[a]
      child.prior = child.prior * (1 - frac) + n * frac


SearchResult = namedtuple('SearchResult', ('visits', 'child_visits', 'root_value', 'minmax',
                                           'trace_parent', 'trace_action', 'trace_depth'))


def legal_words(legal_mask, num_games, num_actions):
  """Host legal masks -> the kernels' layout (include/mzb200.h): int32 [G, W], W = ceil(A / 32), bit b of word w
  set <=> action 32 w + b is legal.

  Accepts one mask per game as integers (Python ints, or an int64 / uint64 / uint32 array [G]: bit a <=> action a;
  at A = 64 action 63 is the sign bit of an int64), a bool array [G, A], or integer words [G, W] already in the
  kernels' layout.  Bits at or beyond A are passed on; the kernels ignore them."""
  G, A = int(num_games), int(num_actions)
  W = (A + 31) // 32
  if torch.is_tensor(legal_mask):
    m = legal_mask.cpu().numpy()
  elif isinstance(legal_mask, np.ndarray):
    m = legal_mask
  else:  # a sequence: Python ints with bit 63 set would become float64 (or fail) under numpy's inference
    m = np.asarray(legal_mask, dtype=object)
    if m.ndim == 1 and not isinstance(m[0], (bool, np.bool_)):
      m = np.array([int(x) & 0xffffffffffffffff for x in m], np.uint64)
    else:
      m = np.array(m.tolist())
  if m.dtype == object:
    m = np.array([int(x) & 0xffffffffffffffff for x in m.ravel()], np.uint64).reshape(m.shape)
  if m.dtype == np.bool_:
    if m.shape != (G, A):
      raise ValueError("expected a bool legal mask of shape %s, got %s" % ((G, A), m.shape))
    bits = np.zeros((G, 32 * W), np.bool_)
    bits[:, :A] = m
    return np.packbits(bits.reshape(G, W, 32), axis=-1, bitorder='little').reshape(G, 4 * W).view('<i4').copy()
  if m.ndim == 2:
    if m.shape != (G, W):
      raise ValueError("expected legal-mask words of shape %s, got %s" % ((G, W), m.shape))
    return np.ascontiguousarray(m.astype(np.int64).astype(np.int32))
  if m.shape != (G,):
    raise ValueError("expected shape %s, got %s" % ((G,), m.shape))
  u = m.astype(np.uint64) if m.dtype.kind == 'u' else m.astype(np.int64).view(np.uint64)
  words = [(u >> np.uint64(32 * w)) & np.uint64(0xffffffff) for w in range(W)]
  return np.ascontiguousarray(np.stack(words, axis=1).astype(np.uint32).view(np.int32))


def pb_c_table(num_simulations, pb_c_base, pb_c_init):
  """[(S+1), (S+1)] float64: entry [N, n] is pb_c after the two statements at mcts.py:116-117,
  evaluated with the interpreter's own math.log / math.sqrt (so it is what the reference computes)."""
  S = int(num_simulations)
  tab = np.empty((S + 1, S + 1), np.float64)
  for N in range(S + 1):
    pb_c = math.log((N + pb_c_base + 1) / pb_c_base) + pb_c_init
    root_n = math.sqrt(N)
    for n in range(S + 1):
      tab[N, n] = pb_c * (root_n / (n + 1))
  return tab


class BatchedMCTS(object):
  """G independent searches in lock step on one GPU.

  config fields read (same names as the reference, mcts.py:66-76): num_simulations, discount,
  pb_c_base, pb_c_init, init_value_score, action_space, two_players, known_bounds.
  """

  def __init__(self, config, num_games, hidden_words=0, device=None, prior_sum_mode=None):
    _lib.require_cuda()
    self.lib = _lib.load()
    self.device = _lib.normalize_device(device)
    self.G = int(num_games)
    self.S = int(config.num_simulations)
    self.A = int(config.action_space)
    if not 1 <= self.A <= _lib.MZ_MAX_ACTIONS:
      raise ValueError("action_space must be in [1, %d]" % _lib.MZ_MAX_ACTIONS)
    self.W = (self.A + 31) // 32  # legal-mask words per game
    self.two_players = bool(config.two_players)
    self.discount = float(config.discount)
    self.init_value_score = float(config.init_value_score)
    kb = list(config.known_bounds)
    self.min_bound = math.inf if kb[0] is None else float(kb[0])
    self.max_bound = -math.inf if kb[1] is None else float(kb[1])
    self.hidden_words = int(hidden_words)
    self.prior_sum_mode = default_prior_sum_mode() if prior_sum_mode is None else int(prior_sum_mode)

    G, S, A, dev = self.G, self.S, self.A, self.device
    self.node_bytes = int(self.lib.mz_tree_node_bytes(A))
    self.game_bytes = int(self.lib.mz_tree_game_bytes(S, A))
    self.games = torch.zeros(G * self.game_bytes, dtype=torch.uint8, device=dev)
    self.pb_c = torch.from_numpy(pb_c_table(S, config.pb_c_base, config.pb_c_init)).to(dev)
    self.hidden = (torch.zeros((G, S + 1, self.hidden_words), dtype=torch.int32, device=dev)
                   if self.hidden_words > 0 else None)
    self.path = torch.zeros((G, S + 2), dtype=torch.int16, device=dev)
    self.path_len = torch.zeros(G, dtype=torch.int32, device=dev)
    self.leaf_parent = torch.zeros(G, dtype=torch.int32, device=dev)
    self.leaf_action = torch.zeros(G, dtype=torch.int32, device=dev)
    self.gathered = (torch.zeros((G, self.hidden_words), dtype=torch.int32, device=dev)
                     if self.hidden_words > 0 else None)
    # root statistics
    self.visits = torch.zeros((G, A), dtype=torch.int32, device=dev)
    self.child_visits = torch.zeros((G, A), dtype=torch.float64, device=dev)
    self.root_value = torch.zeros(G, dtype=torch.float64, device=dev)
    self.minmax = torch.zeros((G, 2), dtype=torch.float64, device=dev)
    self.actions = torch.zeros(G, dtype=torch.int32, device=dev)
    self.trace = None
    self.tree = _lib.Tree(
        G, S, A, int(self.two_players), self.prior_sum_mode, self.hidden_words, self.node_bytes, 0,
        self.game_bytes, self.discount, self.init_value_score, self.min_bound, self.max_bound,
        self.games.data_ptr(), self.pb_c.data_ptr(),
        self.hidden.data_ptr() if self.hidden is not None else None, self.path.data_ptr(),
        self.path_len.data_ptr(), self.leaf_parent.data_ptr(), self.leaf_action.data_ptr())

  # -- building blocks (thin wrappers over the C ABI) --------------------------------------------
  def _stream(self):
    return _lib.current_stream()

  def enable_trace(self):
    G, S, dev = self.G, self.S, self.device
    self.trace = tuple(torch.zeros((S, G), dtype=torch.int32, device=dev) for _ in range(3))

  def _trace_ptrs(self, sim):
    if self.trace is None or sim >= self.S:
      return None, None, None
    return tuple(_lib.ptr(t[sim]) for t in self.trace)

  @_lib.on_device
  def set_root(self, root_logits, legal_mask=None, noise=None, noise_frac=0.25, to_play=None,
               root_hidden=None):
    """Node.expand over legal actions + add_exploration_noise + MinMaxStats.reset for all games."""
    root_logits = self._dev(root_logits, torch.float32, (self.G, self.A))
    legal_mask = self._mask(legal_mask)
    noise = None if noise is None else self._dev(noise, torch.float64, (self.G, self.A))
    to_play = None if to_play is None else self._dev(to_play, torch.int8, (self.G,))
    root_hidden = self._hidden_words(root_hidden)
    self._keep = (root_logits, legal_mask, noise, to_play, root_hidden)
    _lib.check(self.lib.mz_tree_set_root(self.tree, _lib.ptr(root_logits), _lib.ptr(legal_mask),
                                         _lib.ptr(noise), float(noise_frac), _lib.ptr(to_play),
                                         _lib.ptr(root_hidden), self._stream()), "mz_tree_set_root")

  @_lib.on_device
  def set_root_priors(self, root_priors, legal_mask=None, to_play=None, root_hidden=None):
    root_priors = self._dev(root_priors, torch.float64, (self.G, self.A))
    legal_mask = self._mask(legal_mask)
    to_play = None if to_play is None else self._dev(to_play, torch.int8, (self.G,))
    root_hidden = self._hidden_words(root_hidden)
    self._keep = (root_priors, legal_mask, to_play, root_hidden)
    _lib.check(self.lib.mz_tree_set_root_priors(self.tree, _lib.ptr(root_priors),
                                                _lib.ptr(legal_mask), _lib.ptr(to_play),
                                                _lib.ptr(root_hidden), self._stream()),
               "mz_tree_set_root_priors")

  @_lib.on_device
  def select(self, sim, gather=True):
    tp, ta, td = self._trace_ptrs(sim)
    g = self.gathered if gather else None
    _lib.check(self.lib.mz_tree_select(self.tree, int(sim), _lib.ptr(g), tp, ta, td, self._stream()),
               "mz_tree_select")

  @_lib.on_device
  def expand_backup(self, sim, value, reward, logits, new_hidden=None):
    _lib.check(self.lib.mz_tree_expand_backup(self.tree, int(sim), _lib.ptr(value), _lib.ptr(reward),
                                              _lib.ptr(logits), _lib.ptr(new_hidden), self._stream()),
               "mz_tree_expand_backup")

  @_lib.on_device
  def step(self, sim, value=None, reward=None, logits=None, new_hidden=None, gather=False):
    """expand+backup of `sim` fused with the descent of sim + 1 (sim = -1: first descent only)."""
    tp, ta, td = self._trace_ptrs(sim + 1)
    g = self.gathered if gather else None
    _lib.check(self.lib.mz_tree_step(self.tree, int(sim), _lib.ptr(value), _lib.ptr(reward),
                                     _lib.ptr(logits), _lib.ptr(new_hidden), _lib.ptr(g), tp, ta, td,
                                     self._stream()), "mz_tree_step")

  @_lib.on_device
  def root_stats(self):
    """visits [G,A] i32, child_visits [G,A] f64 (game.py:107-110), root_value [G] f64, minmax."""
    _lib.check(self.lib.mz_tree_root_stats(self.tree, _lib.ptr(self.visits),
                                           _lib.ptr(self.child_visits), _lib.ptr(self.root_value),
                                           _lib.ptr(self.minmax), self._stream()),
               "mz_tree_root_stats")
    return self.visits, self.child_visits, self.root_value, self.minmax

  @_lib.on_device
  def select_action(self, temperature, uniforms, legal_mask=None, visits=None):
    """Config.select_action (config.py:70-81) for every game; randomness is host supplied."""
    visits = self.visits if visits is None else visits
    temperature = self._dev(temperature, torch.float64, (self.G,))
    uniforms = self._dev(uniforms, torch.float64, (self.G,))
    legal_mask = self._mask(legal_mask)
    self._keep_sa = (temperature, uniforms, legal_mask)
    _lib.check(self.lib.mz_select_action(self.G, self.A, _lib.ptr(visits), _lib.ptr(legal_mask),
                                         _lib.ptr(temperature), _lib.ptr(uniforms),
                                         _lib.ptr(self.actions), self._stream()), "mz_select_action")
    return self.actions

  @_lib.on_device
  def export_game(self, game):
    """Dense copy of one game's tree (debug / Node façade)."""
    S, A, dev = self.S, self.A, self.device
    prior = torch.zeros((S + 1, A), dtype=torch.float64, device=dev)
    child = torch.zeros((S + 1, A), dtype=torch.int32, device=dev)
    vsum = torch.zeros(S + 1, dtype=torch.float64, device=dev)
    visit = torch.zeros(S + 1, dtype=torch.int32, device=dev)
    reward = torch.zeros(S + 1, dtype=torch.float32, device=dev)
    _lib.check(self.lib.mz_tree_export(self.tree, int(game), _lib.ptr(prior), _lib.ptr(child),
                                       _lib.ptr(vsum), _lib.ptr(visit), _lib.ptr(reward),
                                       self._stream()), "mz_tree_export")
    return dict(prior=prior.cpu().numpy(), child=child.cpu().numpy(), vsum=vsum.cpu().numpy(),
                visit=visit.cpu().numpy(), reward=reward.cpu().numpy())

  # -- generic search loop: any network with the reference interface -----------------------------
  @_lib.on_device
  def search(self, network, root_logits, root_hidden, legal_mask=None, noise=None, noise_frac=0.25,
             to_play=None, root_priors=None):
    """MCTS.run (mcts.py:78-102) for all games, driving `network.recurrent_inference` with batch G.

    root_hidden: tensor [G, ...] (any 4-byte-multiple dtype); the engine keeps hidden states as
    opaque words.  Returns a SearchResult of device tensors.
    """
    hshape, hdtype = tuple(root_hidden.shape[1:]), root_hidden.dtype
    if root_priors is not None:
      self.set_root_priors(root_priors, legal_mask, to_play, root_hidden)
    else:
      self.set_root(root_logits, legal_mask, noise, noise_frac, to_play, root_hidden)
    device_actions = bool(getattr(network, 'accepts_device_actions', False))
    for sim in range(self.S):
      self.select(sim)
      hidden_in = self.gathered.view(hdtype).view((self.G,) + hshape)
      actions = self.leaf_action if device_actions else self.leaf_action.cpu().tolist()
      out = network.recurrent_inference(hidden_in, actions)
      value = out.value.reshape(self.G).to(torch.float32).contiguous()
      reward = out.reward
      if not torch.is_tensor(reward):
        reward = torch.full((self.G,), float(reward), device=self.device)
      reward = reward.reshape(self.G).to(torch.float32).contiguous()
      logits = out.policy_logits.reshape(self.G, self.A).to(torch.float32).contiguous()
      new_hidden = self._hidden_words(out.hidden_state)
      self.expand_backup(sim, value, reward, logits, new_hidden)
    self.root_stats()
    tr = self.trace if self.trace is not None else (None, None, None)
    return SearchResult(self.visits, self.child_visits, self.root_value, self.minmax, *tr)

  # -- helpers -----------------------------------------------------------------------------------
  def _dev(self, x, dtype, shape):
    if not torch.is_tensor(x):
      x = torch.as_tensor(np.asarray(x))
    x = x.to(device=self.device, dtype=dtype).contiguous()
    if tuple(x.shape) != tuple(shape):
      raise ValueError("expected shape %s, got %s" % (tuple(shape), tuple(x.shape)))
    return x

  def _mask(self, legal_mask):
    """Legal masks in the kernels' form: an int32 device tensor [G, W] (`legal_words`; [G] when A <= 32)."""
    if legal_mask is None:
      return None
    kernel_shape = (self.G,) if self.W == 1 else (self.G, self.W)
    if (torch.is_tensor(legal_mask) and legal_mask.dtype == torch.int32 and
        legal_mask.device == self.device and tuple(legal_mask.shape) == kernel_shape):
      return legal_mask.contiguous()  # already in kernel form (bit b of word w set <=> action 32 w + b legal)
    if torch.is_tensor(legal_mask) and legal_mask.dim() == 1 and legal_mask.dtype != torch.bool:
      m = self._dev(legal_mask.to(torch.int64), torch.int64, (self.G,))  # one integer per game
      if self.W == 1:
        return m.to(torch.int32)
      return torch.stack([m & 0xffffffff, (m >> 32) & 0xffffffff], dim=1).to(torch.int32).contiguous()
    words = legal_words(legal_mask, self.G, self.A)
    return self._dev(words.reshape(kernel_shape), torch.int32, kernel_shape)

  def _hidden_words(self, h):
    if h is None or self.hidden_words == 0:
      return None
    h = h.to(self.device).contiguous()
    words = h.reshape(self.G, -1).view(torch.int32)
    if words.shape[1] != self.hidden_words:
      raise ValueError("hidden state has %d words per row, engine was built for %d" %
                       (words.shape[1], self.hidden_words))
    return words


def hidden_words_of(hidden_state):
  """4-byte words per row of a hidden-state tensor [B, ...]."""
  nbytes = hidden_state[0].numel() * hidden_state.element_size()
  if nbytes % 4:
    raise ValueError("hidden state rows must be a multiple of 4 bytes")
  return nbytes // 4


class MCTS(object):
  """Drop-in for the reference's MCTS (mcts.py:64-145): `MCTS(config).run(root, network)`.

  `root` is a Node the caller expanded (and optionally noised) on the host; the search itself runs
  on the GPU with one game in the batch and the result is written back into `root` and its
  descendants, so `root.value()`, `root.children[a].visit_count / prior / reward`,
  `node.expanded()` and the returned search paths behave as with the reference.
  """

  def __init__(self, config):
    self.config = config
    self.num_simulations = config.num_simulations
    self.discount = config.discount
    self.pb_c_base = config.pb_c_base
    self.pb_c_init = config.pb_c_init
    self.init_value_score = config.init_value_score
    self.action_space = range(config.action_space)
    self.two_players = config.two_players
    self.known_bounds = config.known_bounds
    self.min_max_stats = MinMaxStats(*config.known_bounds)
    self._engine = None

  def run(self, root, network):
    _lib.require_cuda()
    hidden = root.hidden_state
    if hidden is None or not root.children:
      raise ValueError("root must be expanded before MCTS.run (root.expand(...))")
    hidden = hidden.to('cuda')
    hw = hidden_words_of(hidden)
    if self._engine is None or self._engine.hidden_words != hw:
      self._engine = BatchedMCTS(self.config, 1, hidden_words=hw, device=hidden.device)
      self._engine.enable_trace()
    eng = self._engine
    A = eng.A
    priors = np.zeros((1, A), np.float64)
    mask = 0
    for a, child in root.children.items():
      priors[0, a] = child.prior
      mask |= 1 << a
    to_play = np.array([root.to_play], np.int8)
    # uint64: at A = 64 bit 63 (action 63) does not fit an int64
    res = eng.search(network, None, hidden, legal_mask=np.array([mask], np.uint64), to_play=to_play,
                     root_priors=priors)
    mm = res.minmax.cpu().numpy()
    self.min_max_stats.minimum, self.min_max_stats.maximum = float(mm[0, 0]), float(mm[0, 1])
    return self._materialise(root, eng, hidden)

  def _materialise(self, root, eng, root_hidden):
    S, A = eng.S, eng.A
    tree = eng.export_game(0)
    parents = eng.trace[0][:, 0].cpu().numpy()
    actions = eng.trace[1][:, 0].cpu().numpy()
    hshape, hdtype = tuple(root_hidden.shape), root_hidden.dtype
    nodes = [None] * (S + 1)
    nodes[0] = root
    depth = [0] * (S + 1)
    parent_of = [0] * (S + 1)
    # nodes are numbered in expansion order, so parents always precede children
    for s in range(S):
      n, p, a = s + 1, int(parents[s]), int(actions[s])
      pnode = nodes[p]
      node = pnode.children.get(a)
      if node is None:
        raise RuntimeError("device tree is inconsistent with the host root")
      nodes[n] = node
      depth[n] = depth[p] + 1
      parent_of[n] = p
      node.to_play = (root.to_play * (-1 if depth[n] % 2 else 1)) if self.two_players else root.to_play
      node.hidden_state = eng.hidden[0, n].view(hdtype).view(hshape)
      node.children = {b: Node(float(tree['prior'][n, b])) for b in range(A)}
    for n in range(S + 1):
      node = nodes[n]
      node.visit_count = int(tree['visit'][n])
      node.value_sum = float(tree['vsum'][n])
      if n > 0:
        r = float(tree['reward'][n])
        node.reward = r if r else 0
    paths = []
    for s in range(S):
      chain = [s + 1]
      while chain[-1] != 0:
        chain.append(parent_of[chain[-1]])
      paths.append([nodes[i] for i in reversed(chain)])
    return paths
