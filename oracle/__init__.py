"""CPU oracle bindings -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this package; the product path (model-based-rl_b200/) never does.  See oracle/mz_oracle.c.
"""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libmz_oracle.so")


def build(force=False):
  src = os.path.join(_HERE, "mz_oracle.c")
  if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
    subprocess.check_call(["make", "-C", _HERE, "-B", "libmz_oracle.so"], stdout=subprocess.DEVNULL)
  return _LIB_PATH


class SearchCfg(C.Structure):
  _fields_ = [("S", C.c_int32), ("A", C.c_int32), ("two_players", C.c_int32),
              ("sum_mode", C.c_int32), ("discount", C.c_double), ("pb_c_base", C.c_double),
              ("pb_c_init", C.c_double), ("init_value_score", C.c_double),
              ("min_bound", C.c_double), ("max_bound", C.c_double)]


class HashNet(C.Structure):
  _fields_ = [("value_scale", C.c_float), ("reward_scale", C.c_float), ("logit_scale", C.c_float),
              ("reward_density", C.c_int32)]


_lib = None


def lib():
  global _lib
  if _lib is None:
    build()
    _lib = C.CDLL(_LIB_PATH)
    _lib.orc_hashnet_next.restype = C.c_uint64
    _lib.orc_hashnet_next.argtypes = [C.c_uint64, C.c_int32]
    _lib.orc_py_sum.restype = C.c_double
    _lib.orc_py_sum.argtypes = [C.c_void_p, C.c_int, C.c_int]
    _lib.orc_select_action.restype = C.c_int32
    _lib.orc_select_action.argtypes = [C.c_void_p, C.c_int, C.c_double, C.c_double]
    _lib.orc_scalar_transform.restype = C.c_float
    _lib.orc_scalar_transform.argtypes = [C.c_float]
    _lib.orc_inverse_scalar_transform.restype = C.c_float
    _lib.orc_inverse_scalar_transform.argtypes = [C.c_float]
    _lib.orc_inverse_transform.restype = C.c_float
    _lib.orc_inverse_transform.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
    _lib.orc_search.restype = C.c_int
  return _lib


def default_sum_mode():
  """builtin sum() semantics of the interpreter the reference would run under."""
  return 1 if sys.version_info >= (3, 12) else 0


def _p(a):
  return None if a is None else a.ctypes.data_as(C.c_void_p)


def make_cfg(num_simulations, action_space, two_players=False, discount=0.997, pb_c_base=19652,
             pb_c_init=1.25, init_value_score=0.0, known_bounds=(None, None), sum_mode=None):
  mn = math.inf if known_bounds[0] is None else float(known_bounds[0])
  mx = -math.inf if known_bounds[1] is None else float(known_bounds[1])
  return SearchCfg(int(num_simulations), int(action_space), int(bool(two_players)),
                   default_sum_mode() if sum_mode is None else int(sum_mode), float(discount),
                   float(pb_c_base), float(pb_c_init), float(init_value_score), mn, mx)


def search(cfg, root_logits, legal_mask=None, noise=None, noise_frac=0.25, root_to_play=None,
           hashnet=None, root_state=None, rec_value=None, rec_reward=None, rec_logits=None,
           dump_tree=False):
  """Runs the oracle search for G games; returns a dict of numpy arrays."""
  root_logits = np.ascontiguousarray(root_logits, dtype=np.float32)
  G, A = root_logits.shape
  S = cfg.S
  assert A == cfg.A
  if legal_mask is not None:
    legal_mask = np.ascontiguousarray(legal_mask, dtype=np.uint32)
  if noise is not None:
    noise = np.ascontiguousarray(noise, dtype=np.float64)
    assert noise.shape == (G, A)
  if root_to_play is not None:
    root_to_play = np.ascontiguousarray(root_to_play, dtype=np.int8)
  if hashnet is not None:
    net_mode = 0
    root_state = np.ascontiguousarray(root_state, dtype=np.uint64)
    hn = C.byref(hashnet)
  else:
    net_mode = 1
    rec_value = np.ascontiguousarray(rec_value, dtype=np.float32).reshape(G, S)
    rec_reward = np.ascontiguousarray(rec_reward, dtype=np.float32).reshape(G, S)
    rec_logits = np.ascontiguousarray(rec_logits, dtype=np.float32).reshape(G, S, A)
    hn = None
  out = {
      "visits": np.zeros((G, A), np.int32),
      "root_value": np.zeros(G, np.float64),
      "root_vsum": np.zeros(G, np.float64),
      "minmax": np.zeros((G, 2), np.float64),
      "trace_parent": np.zeros((G, S), np.int32),
      "trace_action": np.zeros((G, S), np.int32),
      "trace_depth": np.zeros((G, S), np.int32),
  }
  tree = {}
  if dump_tree:
    tree = {
        "edge_prior": np.zeros((G, S + 1, A), np.float64),
        "edge_vsum": np.zeros((G, S + 1, A), np.float64),
        "edge_visit": np.zeros((G, S + 1, A), np.int32),
        "edge_reward": np.zeros((G, S + 1, A), np.float64),
        "edge_child": np.zeros((G, S + 1, A), np.int32),
    }
  rc = lib().orc_search(
      C.byref(cfg), C.c_int32(G), _p(root_logits), _p(legal_mask), _p(noise),
      C.c_double(noise_frac), _p(root_to_play), C.c_int32(net_mode), hn, _p(root_state),
      _p(rec_value), _p(rec_reward), _p(rec_logits), _p(out["visits"]), _p(out["root_value"]),
      _p(out["root_vsum"]), _p(out["minmax"]), _p(out["trace_parent"]), _p(out["trace_action"]),
      _p(out["trace_depth"]), _p(tree.get("edge_prior")), _p(tree.get("edge_vsum")),
      _p(tree.get("edge_visit")), _p(tree.get("edge_reward")), _p(tree.get("edge_child")))
  if rc != 0:
    raise ValueError("orc_search rejected its arguments (rc=%d)" % rc)
  out.update(tree)
  return out


def py_sum(xs, mode=None):
  xs = np.ascontiguousarray(xs, dtype=np.float64)
  return lib().orc_py_sum(_p(xs), len(xs), default_sum_mode() if mode is None else mode)


def select_action(visits, temperature, u):
  visits = np.ascontiguousarray(visits, dtype=np.int32)
  return int(lib().orc_select_action(_p(visits), len(visits), float(temperature), float(u)))


def child_visits(visits, child=None):
  visits = np.ascontiguousarray(visits, dtype=np.int32)
  out = np.zeros(len(visits), np.float64)
  if child is not None:
    child = np.ascontiguousarray(child, dtype=np.int32)
  lib().orc_child_visits(_p(visits), _p(child), C.c_int(len(visits)), _p(out))
  return out


def clip_reward(reward):
  """ClipRewardEnv.reward (wrappers.py:236-238): np.sign of what the environment returned, applied per
  step before the reward enters the history (Breakout configuration, README.md:56)."""
  return np.sign(reward)


def insert_target(rewards, to_play, root_values, child_visits_, K, T, discount, step):
  """One sampled position -> (t_rewards[K+1], t_values[K+1], t_policies[K+1, A])."""
  rewards = np.ascontiguousarray(rewards, dtype=np.float64)
  to_play = np.ascontiguousarray(to_play, dtype=np.int8)
  root_values = np.ascontiguousarray(root_values, dtype=np.float64)
  cv = np.ascontiguousarray(child_visits_, dtype=np.float64)
  A = cv.shape[1] if cv.ndim == 2 and cv.shape[0] else cv.shape[-1]
  cv = cv.reshape(len(root_values), A)
  discounts = np.array([discount**n for n in range(K + T)], dtype=np.float32)
  tr = np.zeros(K + 1, np.float32)
  tv = np.zeros(K + 1, np.float32)
  tp = np.zeros((K + 1, A), np.float32)
  lib().orc_insert_target(_p(rewards), _p(to_play), C.c_int(len(rewards)), _p(root_values), _p(cv),
                          C.c_int(len(root_values)), C.c_int(A), C.c_int(K), C.c_int(T),
                          C.c_double(discount**T), _p(discounts), C.c_int(step), _p(tr), _p(tv),
                          _p(tp))
  return tr, tv, tp


def scalar_transform(x):
  x = np.asarray(x, dtype=np.float32)
  f = lib().orc_scalar_transform
  return np.array([f(float(v)) for v in x.ravel()], np.float32).reshape(x.shape)


def inverse_scalar_transform(x):
  x = np.asarray(x, dtype=np.float32)
  f = lib().orc_inverse_scalar_transform
  return np.array([f(float(v)) for v in x.ravel()], np.float32).reshape(x.shape)


def scalar_to_support(x, mn, mx):
  x = np.asarray(x, dtype=np.float32)
  size = mx - mn + 1
  out = np.zeros(x.shape + (size,), np.float32)
  flat = out.reshape(-1, size)
  for i, v in enumerate(x.ravel()):
    row = np.zeros(size, np.float32)
    lib().orc_scalar_to_support(C.c_float(float(v)), C.c_int(mn), C.c_int(mx), _p(row))
    flat[i] = row
  return out


def scalar_transform_f32(x):
  """mz_scalar_transform_f (csrc/mz_transforms.cuh) in numpy float32, same operation order: c = sqrt(|x| + 1) - 1,
  then sign(x) * c + 0.001f * x, every operation rounded to float32.  numpy's float32 sqrt is correctly rounded (torch's
  CPU sqrt is not), so this is the kernel's result bit for bit."""
  x = np.asarray(x, dtype=np.float32)
  c = np.sqrt(np.abs(x) + np.float32(1)) - np.float32(1)
  return (np.sign(x) * c + np.float32(0.001) * x).astype(np.float32)


def two_hot_f64(x, mn, mx, float32=False):
  """Config.scalar_to_support (config.py:56-68) in binary64: x clamped to [mn, mx], p_hi = x - floor(x) at ceil(x),
  then 1 - p_hi at floor(x) (1.0 at an integer).  Returns (clamped x, support[..., mx - mn + 1]).

  float32=True gives the float32 two-hot of mz_two_hot (csrc/mz_transforms.cuh) bit for bit, as float32.  For float32
  x both of its subtractions are exact in binary64, but x - floor(x) is not exact in float32 when x is a negative
  non-integer (-0.24 + 1 needs the bits of both), and 1 - p_hi then starts from the rounded p_hi: so p_hi is rounded
  to float32 before 1 - p_hi is formed, and each weight is rounded once, where the float32 operations round it."""
  x = np.clip(np.asarray(x, dtype=np.float64), mn, mx)
  lo = np.floor(x)
  p_hi = x - lo
  if float32:
    p_hi = p_hi.astype(np.float32).astype(np.float64)
  out = np.zeros(x.shape + (mx - mn + 1,), np.float64)
  idx = (lo - mn).astype(np.int64)
  hi = np.minimum(idx + 1, mx - mn)
  np.put_along_axis(out, hi[..., None], p_hi[..., None], axis=-1)
  np.put_along_axis(out, idx[..., None], (1.0 - p_hi)[..., None], axis=-1)  # the low bin wins on integers
  return x, (out.astype(np.float32) if float32 else out)


def inverse_transform(logits, mn, mx, no_target_transform=False):
  logits = np.ascontiguousarray(logits, dtype=np.float32)
  B, size = logits.shape
  assert size == mx - mn + 1
  out = np.zeros((B, 1), np.float32)
  for b in range(B):
    out[b, 0] = lib().orc_inverse_transform(_p(logits[b]), mn, mx, int(no_target_transform))
  return out


def inverse_transform_f64(logits, mn, mx, no_target_transform=False):
  """Config.inverse_transform (config.py:27-33) evaluated in binary64 from the float32 logits: the value the
  float32 pipelines (torch's and the CUDA kernel's) approximate.  h^-1 cancels catastrophically in float32
  (sqrt(1 + 4 eps (|x| + 1 + eps)) - 1 with eps = 0.001), so two correct float32 implementations differ by up to
  ~5e-4; this restatement says which side is closer to the exact result."""
  z = np.asarray(logits, np.float64)
  e = np.exp(z - z.max(axis=1, keepdims=True))
  p = e / e.sum(axis=1, keepdims=True)
  x = (p * np.arange(mn, mx + 1, dtype=np.float64)).sum(axis=1)
  if no_target_transform:
    return x
  eps = 0.001
  return np.sign(x) * (((np.sqrt(1 + 4 * eps * (np.abs(x) + 1 + eps)) - 1) / (2 * eps))**2 - 1)
