"""Batched self-play: the body of Actor.play_game (actors.py:125-176) for G games in lock step.

Per move: observations -> `initial_inference` -> root expansion over the legal actions + Dirichlet
noise -> batched search on the GPU (`BatchedMCTS.search`, any network with the reference's interface)
-> `select_action` with per-game temperature -> environment step -> `Game.apply` /
`store_search_statistics` bookkeeping (game.py:75-115) -> history slices pushed to the replay buffer
with the reference's chunking rules (`max_history_length`, the `num_unroll_steps + td_steps` overlap,
`ignore` for running games, actors.py:160-169).  A finished game is replaced by a new one at once, so
the batch always holds G live games.

With `search=` an `FCSearch` built on the same network (networks.py), the whole move -- initial
inference, root set-up, the S simulations, root statistics and action selection -- is the engine's
single CUDA-graph replay behind `search_host` (host arrays in, host arrays out) instead of one
`recurrent_inference` call per simulation.

Random draws (Dirichlet noise per root, one uniform per action selection) come from numpy unless the
caller passes them in -- which is how the parity test replays the reference.
"""
import collections

import numpy as np
import torch

from .mcts import BatchedMCTS, legal_words

HistorySlice = collections.namedtuple(
    "HistorySlice", "observations child_visits root_values actions rewards errors dones steps env_states "
    "to_play")  # game.py:5-16


class _Game(object):
  """The per-game bookkeeping of game.Game (game.py:56-126) without the environment."""

  def __init__(self, first_observation):
    self.observations = [first_observation]
    self.child_visits, self.root_values, self.actions, self.rewards = [], [], [], []
    self.errors, self.dones, self.steps, self.to_play_hist = [], [], [], []
    self.previous_collect_to = 0
    self.history_idx = 0
    self.step = 0
    self.to_play = 1
    self.sum_rewards = 0
    self.sum_values = 0.0
    self.max_value = -np.inf

  def slice(self, collect_from):  # History.get_slice + get_history_sequence (game.py:40-51, 123-126)
    s = slice(collect_from, None)
    out = HistorySlice(self.observations[s], self.child_visits[s], self.root_values[s], self.actions[s],
                       self.rewards[s], self.errors[s], self.dones[s], self.steps[s],
                       [None] * len(self.actions[s]), self.to_play_hist[s])
    self.previous_collect_to = self.history_idx
    return out


def _legal_count(legal, i, A):
  """Legal actions of game i in env.legal_mask()'s result: one integer per game, [G, W] words or a bool [G, A]
  array (mcts.legal_words)."""
  if A <= 32 and np.ndim(legal[i]) == 0:
    return bin(int(legal[i])).count("1")
  words = legal_words(np.asarray(legal[i:i + 1]) if isinstance(legal, np.ndarray) else legal[i:i + 1], 1, A)
  return int(np.unpackbits(words.view(np.uint8), bitorder='little')[:A].sum())


class BatchedActor(object):

  def __init__(self, config, network, env, replay_buffer=None, device=None, temperature=1.0, search=None):
    self.config, self.network, self.env, self.replay = config, network, env, replay_buffer
    self.search = search
    if search is not None and search.G != env.num_games:
      raise ValueError("the search engine was built for %d games, the environment has %d" % (search.G, env.num_games))
    self.G, self.A = env.num_games, int(config.action_space)
    self.device = torch.device("cuda" if device is None else device)
    self.eng = None  # built on the first move (the hidden-state width comes from the network)
    self.temperature = np.broadcast_to(np.asarray(temperature, np.float64), (self.G,)).copy()
    self.games = [_Game(o) for o in env.reset()]
    self.experiences_collected = 0
    self.games_played = 0
    self.results = collections.Counter()
    self.saved = []  # (game index, history, ignore, terminal) when no replay buffer is attached

  # -- one move for every game -------------------------------------------------------------------------
  def play_move(self, noise=None, uniforms=None):
    cfg, env, G, A = self.config, self.env, self.G, self.A
    obs = np.stack([np.float32(g.observations[-1]) for g in self.games])      # get_observation(-1)
    if getattr(cfg, "norm_obs", False):
      obs = (obs - cfg.obs_min) / cfg.obs_range
    legal = env.legal_mask()
    to_play = np.array([g.to_play for g in self.games], np.int8)
    if noise is None:  # Node.add_exploration_noise (mcts.py:57-61): one draw per root over its children
      noise = np.zeros((G, A))
      for i in range(G):
        n = _legal_count(legal, i, A)
        noise[i, :n] = np.random.dirichlet([cfg.root_dirichlet_alpha] * n)
    if uniforms is None:
      uniforms = np.random.random(G)
    if self.search is not None:
      actions, root_value, child_visits, init_value = self.search.search_host(
          np.ascontiguousarray(obs, dtype=np.float32), noise, uniforms, self.temperature, legal=legal, to_play=to_play)
      actions, root_value = actions.numpy().copy(), root_value.numpy().copy()
      child_visits, init_value = child_visits.numpy().copy(), init_value.double().numpy()
      return self._advance(actions, root_value, child_visits, root_value - init_value)
    with torch.inference_mode():
      init = self.network.initial_inference(torch.from_numpy(obs).to(self.device))
    hidden = init.hidden_state
    if self.eng is None:
      words = hidden[0].numel() * hidden.element_size() // 4
      self.eng = BatchedMCTS(cfg, G, hidden_words=words, device=self.device)
    eng = self.eng
    eng.search(self.network, init.policy_logits.reshape(G, A).float().contiguous(), hidden, legal_mask=legal,
               noise=noise, noise_frac=cfg.root_exploration_fraction, to_play=to_play)
    actions = eng.select_action(self.temperature, uniforms, legal)
    actions = actions.cpu().numpy()
    root_value = eng.root_value.cpu().numpy()
    child_visits = eng.child_visits.cpu().numpy()
    init_value = init.value.reshape(G).double().cpu().numpy()
    return self._advance(actions, root_value, child_visits, root_value - init_value)  # actors.py:147

  def _advance(self, actions, root_value, child_visits, errors):
    """Environment step and the Game / History bookkeeping of every game (actors.py:150-176)."""
    cfg, env = self.config, self.env
    next_obs, reward, done, result = env.step(actions)
    finished = []
    overlap = cfg.num_unroll_steps + cfg.td_steps
    for i, g in enumerate(self.games):
      g.errors.append(float(errors[i]))
      # Game.apply (game.py:75-104)
      g.steps.append(g.step)
      g.sum_rewards += reward[i].item() if hasattr(reward[i], 'item') else reward[i]  # game.py:85
      g.step = int(env.elapsed[i])
      g.history_idx += 1
      g.observations.append(next_obs[i])
      g.actions.append(int(actions[i]))
      g.dones.append(bool(done[i]))
      g.rewards.append(reward[i].item() if hasattr(reward[i], 'item') else reward[i])  # the raw env reward, game.py:97
      g.to_play_hist.append(g.to_play)
      if cfg.two_players:
        g.to_play *= -1
      # Game.store_search_statistics (game.py:106-115)
      g.child_visits.append(child_visits[i].tolist())
      g.root_values.append(float(root_value[i]))
      g.sum_values += float(root_value[i])
      g.max_value = max(g.max_value, float(root_value[i]))
      self.experiences_collected += 1
      terminal = bool(done[i])  # episode_life is off for the vectorised environments
      # actors.py:160-169
      if (g.history_idx - g.previous_collect_to) == cfg.max_history_length or terminal:
        if not g.dones[g.previous_collect_to - 1]:
          collect_from = max(0, g.previous_collect_to - overlap)
        else:
          collect_from = g.previous_collect_to
        history = g.slice(collect_from)
        ignore = overlap if not done[i] else None
        if self.replay is not None:
          self.replay.save_history(history, ignore=ignore, terminal=terminal)
        else:
          self.saved.append((i, history, ignore, terminal))
      if terminal or g.step >= cfg.max_steps:
        finished.append(i)
        if result[i] >= 0:
          self.results[int(result[i])] += 1
    if finished:  # run_selfplay: a new game replaces the finished one (actors.py:94-97)
      self.games_played += len(finished)
      for i, o in zip(finished, env.reset(finished)):
        self.games[i] = _Game(o)
    return actions, root_value, child_visits, errors, done


class DeviceActor(object):
  """`BatchedActor` with the trajectories resident on the GPU: the body of Actor.play_game (actors.py:125-176) for
  G games in lock step, where a move's record (observation, action, reward, to_play, root value, child-visit
  distribution) goes from the search engine's output buffers straight into the replay window
  (`PrioritizedReplay.append_steps`, one launch per move) instead of per-game Python lists that are re-uploaded as
  HistorySlices.  The host keeps what the reference keeps per game -- counters and the priority seeds
  `error = root.value() - initial value` (actors.py:147) -- as arrays over the games; per-game Python runs only for
  the few games that finish a chunk in a move (max_history_length steps or a terminal, actors.py:160-169).

  Chunking, the num_unroll_steps + td_steps overlap of a running game's chunks, `ignore` and the priorities are the
  reference's; tests/test_selfplay.py checks the resulting replay buffer against the list path's, bit for bit.
  Observations are stored as the environment returns them: uint8 (normalised on the device for the search,
  `FCSearch.set_obs_normalization`) or float32 without `norm_obs`."""

  def __init__(self, config, env, replay_buffer, search, temperature=1.0):
    self.config, self.env, self.replay, self.search = config, env, replay_buffer, search
    if search.G != env.num_games:
      raise ValueError("the search engine was built for %d games, the environment has %d" % (search.G, env.num_games))
    if getattr(config, "norm_obs", False):
      raise ValueError("DeviceActor stores raw observations: use uint8 observations with FCSearch.set_obs_normalization")
    G = self.G = env.num_games
    self.A = int(config.action_space)
    self.L = int(config.max_history_length)
    self.overlap = int(config.num_unroll_steps + config.td_steps)
    self.cap = self.L + self.overlap
    self.temperature = np.broadcast_to(np.asarray(temperature, np.float64), (G,)).copy()
    self.obs = np.ascontiguousarray(env.reset())
    self.obs_u8 = self.obs.dtype == np.uint8
    dev = replay_buffer.device
    self.history_idx = np.zeros(G, np.int64)      # Game.history_idx
    self.prev_collect = np.zeros(G, np.int64)     # Game.previous_collect_to
    self.first = np.zeros(G, np.int64)            # history index of the open chunk's first position
    self.to_play = np.ones(G, np.int8)
    self.sum_rewards = np.zeros(G, np.float64)
    self.errors = np.zeros((G, self.cap), np.float64)
    self.chunk_id = np.zeros(G, np.int64)
    self.chunk_start = np.zeros(G, np.int64)
    odt = torch.uint8 if self.obs_u8 else torch.float32
    for g in range(G):
      self.chunk_id[g], self.chunk_start[g] = replay_buffer.open_chunk(self.cap, odt)
    self._odt = odt
    self.h_pos = torch.zeros(G, dtype=torch.int64).pin_memory()
    self.h_rew = torch.zeros(G, dtype=torch.float32).pin_memory()
    self.d_pos = torch.zeros(G, dtype=torch.int64, device=dev)
    self.d_rew = torch.zeros(G, dtype=torch.float32, device=dev)
    self.experiences_collected = 0
    self.games_played = 0
    self.results = collections.Counter()

  def play_move(self, noise=None, uniforms=None):
    self.begin_move(noise, uniforms)
    return self.finish_move()

  def begin_move(self, noise=None, uniforms=None):
    """First half of a move: the roots' inputs go to the device and the search is enqueued; returns without
    waiting for it (`finish_move` does).  Between the two, the host is free for another actor's move."""
    cfg, env, G, A, fs = self.config, self.env, self.G, self.A, self.search
    legal = env.legal_mask()
    # Node.add_exploration_noise (mcts.py:57-61): one Dirichlet draw per root over its children -- on the device
    # (FCSearch.draw_noise) unless the caller brings the draws (the bit-exact path the tests replay)
    alpha = None
    if noise is None:
      if hasattr(fs, "draw_noise"):
        alpha = cfg.root_dirichlet_alpha
      else:
        noise = np.zeros((G, A))
        for i in range(G):
          n = _legal_count(legal, i, A)
          noise[i, :n] = np.random.dirichlet([cfg.root_dirichlet_alpha] * n)
    if uniforms is None:
      uniforms = np.random.random(G)
    obs_in = self.obs if self.obs_u8 else np.ascontiguousarray(self.obs, dtype=np.float32)
    kw = {} if alpha is None else {"dirichlet_alpha": alpha}
    if hasattr(fs, "search_result"):  # enqueue only: the host goes on while the device searches
      kw["wait"] = False
    self._pending = fs.search_host(obs_in, noise, uniforms, self.temperature, legal=legal, to_play=self.to_play, **kw)

  def finish_move(self):
    """Second half: waits for the search, steps the environments, appends the move's record to the replay window on
    the device and commits the chunks that ended (actors.py:147-169)."""
    cfg, env, G, fs = self.config, self.env, self.G, self.search
    out, self._pending = self._pending, None
    actions, root_value, child_visits, init_value = fs.search_result() if out is None else out
    actions = actions.numpy().copy()
    errors = root_value.numpy() - init_value.numpy().astype(np.float64)  # actors.py:147
    next_obs, reward, done, result = env.step(actions)
    # Game.apply + store_search_statistics for every game: one launch, straight from the engine's device buffers
    idx = self.history_idx - self.first
    self.h_pos.copy_(torch.from_numpy(self.chunk_start + idx))
    self.h_rew.copy_(torch.from_numpy(np.asarray(reward, np.float64).astype(np.float32)))
    self.d_pos.copy_(self.h_pos, non_blocking=True)
    self.d_rew.copy_(self.h_rew, non_blocking=True)
    self.replay.append_steps(self.d_pos, fs.obs_u8 if self.obs_u8 else fs.obs, fs.actions, self.d_rew, fs.to_play,
                             fs.root_value, fs.child_visits)
    self.errors[np.arange(G), idx] = errors
    self.sum_rewards += reward
    self.history_idx += 1
    if cfg.two_players:
      self.to_play = (-self.to_play).astype(np.int8)
    self.experiences_collected += G
    self.obs = np.ascontiguousarray(next_obs)
    # actors.py:160-169: a chunk is complete after max_history_length new steps or at a terminal
    full = ((self.history_idx - self.prev_collect) == self.L) | done
    over = done | (env.elapsed >= cfg.max_steps)
    src, dst, cnt, commits = [], [], [], []
    for g in np.nonzero(full | over)[0]:
      g = int(g)
      if full[g]:
        n = int(self.history_idx[g] - self.first[g])
        commits.append((int(self.chunk_id[g]), int(self.chunk_start[g]), n, self.errors[g, :n].copy(),
                        None if done[g] else self.overlap, bool(done[g])))
        self.prev_collect[g] = self.history_idx[g]
      elif over[g]:
        # cut by max_steps without a terminal: the reference drops the unsent tail with the Game object
        commits.append((int(self.chunk_id[g]), int(self.chunk_start[g]), 0, self.errors[g, :0], None, False))
      old_start, old_first = int(self.chunk_start[g]), int(self.first[g])
      # the finished chunk stays reserved (open) until every new chunk of this move has its place, so a chunk without
      # priorities cannot be recycled under the overlap copy below
      self.chunk_id[g], self.chunk_start[g] = self.replay.open_chunk(self.cap, self._odt)
      if over[g]:  # run_selfplay: a new game replaces the finished one (actors.py:94-97)
        if result[g] >= 0:
          self.results[int(result[g])] += 1
        self.games_played += 1
        self.history_idx[g] = self.prev_collect[g] = self.first[g] = 0
        self.to_play[g] = 1
        self.sum_rewards[g] = 0.0
      else:  # the next chunk of a running game starts with the last `overlap` steps of this one
        first = max(0, int(self.history_idx[g]) - self.overlap)
        keep = int(self.history_idx[g]) - first
        src.append(old_start + (first - old_first))
        dst.append(int(self.chunk_start[g]))
        cnt.append(keep)
        self.errors[g, :keep] = self.errors[g, first - old_first:first - old_first + keep].copy()
        self.first[g] = first
    if src:
      self.replay.copy_positions(src, dst, cnt)
    if commits:  # save_history for every finished chunk of the move: one sum-tree call
      self.replay.commit_chunks(commits)
    fin = np.nonzero(over)[0]
    if len(fin):
      self.obs[fin] = env.reset(fin)
    return actions, root_value, child_visits, errors, done


class PipelinedActors(object):
  """Several `DeviceActor`s (each with its own environments and search engine, one shared replay buffer) taking turns
  on one GPU, the way the reference runs several Ray actors beside each other (train.py: `--num_actors`): while one
  actor's search runs on the device, the host steps the environments, appends the records and stages the next roots
  of the others.  A move costs max(device search, host work) instead of their sum.  Results -- every record, chunk
  commit and random draw -- are those of calling the actors' `play_move` in turn (tests/test_selfplay.py)."""

  def __init__(self, actors, copy_outputs=False):
    """copy_outputs: root values / child-visit distributions of a move are views of the engine's pinned output
    blob, which the actor's NEXT search (enqueued before `play_round` returns) overwrites when it completes; pass
    True to get private copies."""
    self.actors = list(actors)
    self.copy_outputs = bool(copy_outputs)
    self._primed = False
    self._staged, self._events, self._flip = None, None, 0

  def play_round(self):
    """One move of every actor; returns their `play_move` results in order."""
    if not self._primed:
      for a in self.actors:
        a.begin_move()
      self._primed = True
    out = []
    for a in self.actors:
      # the replay buffer's pinned staging areas are shared: the previous actor's append / commit copies (enqueued
      # behind THIS actor's search, so a few microseconds after it) must have read them before they are rewritten
      if self._staged is not None:
        self._staged.synchronize()
      res = a.finish_move()
      if self._events is None:
        self._events = [torch.cuda.Event() for _ in range(2)]
      self._staged = self._events[self._flip]
      self._flip ^= 1
      self._staged.record()
      if self.copy_outputs:
        res = (res[0], res[1].clone(), res[2].clone(), res[3], res[4])
      out.append(res)
      a.begin_move()  # its next search runs under the other actors' host work
    return out

  def drain(self):
    """Finishes the moves in flight (call before reading the actors' counters for the last time)."""
    out = []
    if self._primed:
      for a in self.actors:
        if self._staged is not None:
          self._staged.synchronize()
        out.append(a.finish_move())
        self._staged = self._events[self._flip] if self._events else None
        if self._staged is not None:
          self._flip ^= 1
          self._staged.record()
      self._primed = False
    return out

  @property
  def experiences_collected(self):
    return sum(a.experiences_collected for a in self.actors)
