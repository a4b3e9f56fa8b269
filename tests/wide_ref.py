"""Reference searches past 32 actions for the wide-action tests: the pure-Python port of the reference's search
(oracle/search_ref.py, pinned to the unmodified mcts.py by tests/test_oracle_golden.py) run game by game, with
legal subsets of any width, driven by the hash network or by a network that replays recorded outputs."""
import numpy as np
import torch

from oracle.search_ref import FlatSearch

from model_based_rl_b200.testing import HashNetwork, NetworkOutput


def legal_lists(legal_bool):
  """bool [G, A] -> the root's legal actions of every game, ascending."""
  return [list(np.nonzero(row)[0].astype(int)) for row in legal_bool]


def random_legal(rng, G, A, only_high_rows=()):
  """bool [G, A] legal subsets with at least one legal action; rows in `only_high_rows` only have actions >= 32."""
  legal = rng.random((G, A)) < rng.uniform(0.2, 0.9, size=(G, 1))
  for g in only_high_rows:
    legal[g, :32] = False
  for g in range(G):
    if not legal[g].any():
      legal[g, rng.integers(32 if g in only_high_rows else 0, A)] = True
  legal[0, A - 1] = True  # the highest action legal somewhere
  return legal


def dense_noise(rng, legal_bool, alpha=0.25):
  """Dirichlet draws dense over each root's legal actions (the layout mcts.py:59 produces and the kernels read)."""
  G, A = legal_bool.shape
  noise = np.zeros((G, A))
  for g in range(G):
    n = int(legal_bool[g].sum())
    noise[g, :n] = rng.dirichlet([alpha] * n)
  return noise


class ReplayNetwork(object):
  """recurrent_inference returns the outputs recorded for one game's simulations, in call order."""

  def __init__(self, value, reward, logits):
    self.value, self.reward, self.logits, self.s = value, reward, logits, 0

  def recurrent_inference(self, hidden_state, action):
    s = self.s
    self.s += 1
    return NetworkOutput(torch.tensor([[self.value[s]]], dtype=torch.float32),
                         torch.tensor([[self.reward[s]]], dtype=torch.float32),
                         torch.from_numpy(np.ascontiguousarray(self.logits[s][None], dtype=np.float32)), None)


def port_search(cfg, root_logits, legal_bool=None, noise=None, noise_frac=0.25, to_play=None, hashnet=None,
                root_state=None, rec_value=None, rec_reward=None, rec_logits=None):
  """FlatSearch for G games; returns numpy arrays named like oracle.search's outputs plus child_visits.

  cfg: dict of FlatSearch's keyword arguments.  hashnet: dict of HashNetwork's scales with root_state [G];
  otherwise rec_value [G, S], rec_reward [G, S], rec_logits [G, S, A] are replayed."""
  root_logits = np.asarray(root_logits, np.float32)
  G, A = root_logits.shape
  S = int(cfg["num_simulations"])
  legal = legal_lists(np.ones((G, A), bool) if legal_bool is None else legal_bool)
  out = dict(visits=np.zeros((G, A), np.int32), root_value=np.zeros(G), minmax=np.zeros((G, 2)),
             child_visits=np.zeros((G, A)), trace_parent=np.zeros((G, S), np.int32),
             trace_action=np.zeros((G, S), np.int32), trace_depth=np.zeros((G, S), np.int32))
  net = HashNetwork(A, **hashnet) if hashnet is not None else None
  for g in range(G):
    fs = FlatSearch(**cfg)
    if net is not None:
      hidden, run_net = torch.tensor([[int(root_state[g])]], dtype=torch.int64), net
    else:
      hidden, run_net = None, ReplayNetwork(rec_value[g], rec_reward[g], rec_logits[g])
    init = NetworkOutput(None, 0, torch.from_numpy(root_logits[g:g + 1].copy()), hidden)
    tp = 1 if to_play is None else int(to_play[g])
    fs.setup_root(init, tp, legal[g], None if noise is None else noise[g, :len(legal[g])], noise_frac)
    fs.run(run_net)
    out["visits"][g] = fs.root_visits()
    out["root_value"][g] = fs.root_value()
    out["minmax"][g] = fs.minmax
    out["child_visits"][g] = fs.child_visits()
    out["trace_parent"][g], out["trace_action"][g], out["trace_depth"][g] = np.array(fs.trace).T
  return out
