"""ctypes binding of libmzb200.so (C ABI declared in include/mzb200.h).

There is no fallback: if the CUDA library is missing or a call fails, this raises.
"""
import ctypes as C
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmzb200.so")
CSRC = os.path.join(_HERE, "csrc")

MZ_MAX_ACTIONS = 64  # one warp per game; lane l owns action l and, when A > 32, action l + 32
CHILD_UNEXPANDED = -1
CHILD_ILLEGAL = -2
GAME_HEADER_BYTES = 32
FC_HIDDEN = 50
FC_WIDTH = 512


class MzError(RuntimeError):
  pass


class Tree(C.Structure):
  """struct mz_tree"""
  _fields_ = [
      ("num_games", C.c_int32), ("num_simulations", C.c_int32), ("num_actions", C.c_int32),
      ("two_players", C.c_int32), ("prior_sum_mode", C.c_int32), ("hidden_words", C.c_int32),
      ("node_bytes", C.c_int32), ("reserved0", C.c_int32), ("game_bytes", C.c_int64),
      ("discount", C.c_double), ("init_value_score", C.c_double), ("min_bound", C.c_double),
      ("max_bound", C.c_double), ("games", C.c_void_p), ("pb_c_table", C.c_void_p),
      ("hidden", C.c_void_p), ("path", C.c_void_p), ("path_len", C.c_void_p),
      ("leaf_parent", C.c_void_p), ("leaf_action", C.c_void_p)]


class FcWeights(C.Structure):
  """struct mz_fc_weights"""
  _names = ["rep_w1", "rep_b1", "rep_w2", "rep_b2", "dyn_w1", "dyn_b1", "dyn_w2", "dyn_b2",
            "rew_w1", "rew_b1", "rew_w2", "rew_b2", "val_w1", "val_b1", "val_w2", "val_b2",
            "pol_w1", "pol_b1", "pol_w2", "pol_b2", "ln_w", "ln_b"]
  _fields_ = [("obs_dim", C.c_int32), ("num_actions", C.c_int32), ("value_bins", C.c_int32),
              ("reward_bins", C.c_int32), ("value_min", C.c_int32), ("reward_min", C.c_int32),
              ("no_target_transform", C.c_int32), ("no_support", C.c_int32)] + \
             [(n, C.c_void_p) for n in _names]


class FcSearchArgs(C.Structure):
  """struct mz_fc_search_args"""
  _fields_ = [("weights", C.POINTER(FcWeights)), ("packed", C.c_void_p), ("tail", C.c_void_p),
              ("num_games", C.c_int32), ("num_simulations", C.c_int32), ("two_players", C.c_int32),
              ("prior_sum_mode", C.c_int32), ("game_bytes", C.c_int64), ("discount", C.c_double),
              ("init_value_score", C.c_double), ("min_bound", C.c_double), ("max_bound", C.c_double), ("noise_frac", C.c_double),
              ("games", C.c_void_p), ("pb_c_table", C.c_void_p), ("pool", C.c_void_p),
              ("root_logits", C.c_void_p), ("legal_mask", C.c_void_p), ("noise", C.c_void_p),
              ("root_to_play", C.c_void_p), ("root_hidden", C.c_void_p), ("visits", C.c_void_p),
              ("child_visits", C.c_void_p), ("root_value", C.c_void_p), ("minmax", C.c_void_p),
              ("trace_parent", C.c_void_p), ("trace_action", C.c_void_p), ("trace_depth", C.c_void_p),
              ("rec_value", C.c_void_p), ("rec_reward", C.c_void_p), ("rec_logits", C.c_void_p),
              ("timeline", C.c_void_p), ("error_flag", C.c_void_p)]


class Window(C.Structure):
  """struct mz_window"""
  _fields_ = [("num_actions", C.c_int32), ("obs_elems", C.c_int32), ("obs_is_u8", C.c_int32),
              ("clip_rewards", C.c_int32), ("obs", C.c_void_p), ("actions", C.c_void_p),
              ("rewards", C.c_void_p), ("to_play", C.c_void_p), ("root_values", C.c_void_p),
              ("child_visits", C.c_void_p)]


class TargetCfg(C.Structure):
  """struct mz_target_cfg"""
  _fields_ = [("batch", C.c_int32), ("num_unroll_steps", C.c_int32), ("td_steps", C.c_int32),
              ("fuse_supports", C.c_int32), ("value_min", C.c_int32), ("value_max", C.c_int32),
              ("reward_min", C.c_int32), ("reward_max", C.c_int32),
              ("no_target_transform", C.c_int32), ("normalize_obs", C.c_int32),
              ("disc_pow_td", C.c_double), ("discounts", C.c_void_p), ("obs_min", C.c_void_p),
              ("obs_range", C.c_void_p)]


class LossCfg(C.Structure):
  """struct mz_loss_cfg"""
  _fields_ = [("batch", C.c_int32), ("num_unroll_steps", C.c_int32), ("num_actions", C.c_int32),
              ("value_min", C.c_int32), ("value_max", C.c_int32), ("reward_min", C.c_int32),
              ("reward_max", C.c_int32), ("no_target_transform", C.c_int32)]


class PackJob(C.Structure):
  """struct mz_pack_job"""
  _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("n", C.c_int32), ("k", C.c_int32), ("stride_n", C.c_int32),
              ("stride_k", C.c_int32)]


class TcHead(C.Structure):
  """struct mz_tc_head"""
  _fields_ = [("w1p", C.c_void_p), ("w2p", C.c_void_p), ("w2tp", C.c_void_p), ("w1tp", C.c_void_p), ("b1", C.c_void_p),
              ("b2", C.c_void_p), ("gw1", C.c_void_p), ("gb1", C.c_void_p), ("gw2", C.c_void_p), ("gb2", C.c_void_p),
              ("d_in", C.c_int32), ("d_out", C.c_int32)]


class TcJob(C.Structure):
  """struct mz_tc_job"""
  _fields_ = [("head", TcHead), ("rows", C.c_int32), ("ldx", C.c_int32), ("ldy", C.c_int32), ("lddx", C.c_int32),
              ("x", C.c_void_p), ("y", C.c_void_p), ("dy", C.c_void_p), ("dx", C.c_void_p)]


class TcChain(C.Structure):
  """struct mz_tc_chain"""
  _fields_ = [("first", TcHead), ("next", TcHead), ("rows", C.c_int32), ("steps", C.c_int32), ("d", C.c_int32),
              ("num_actions", C.c_int32), ("x0", C.c_void_p), ("ldx0", C.c_int32), ("actions", C.c_void_p),
              ("action_stride", C.c_int32), ("action_steps", C.c_int32), ("gamma", C.c_void_p), ("beta", C.c_void_p),
              ("xs", C.c_void_p), ("ldxs", C.c_int32), ("yall", C.c_void_p), ("mean", C.c_void_p), ("rstd", C.c_void_p),
              ("relu_mask", C.c_void_p), ("dxs", C.c_void_p), ("hook_scale", C.c_float), ("ggamma", C.c_void_p),
              ("gbeta", C.c_void_p), ("dyall", C.c_void_p)]


_V = C.c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)
    "mz_tree_node_bytes": (C.c_int32, [C.c_int32]),
    "mz_tree_game_bytes": (C.c_int64, [C.c_int32, C.c_int32]),
    "mz_fill_pb_c_table": (C.c_int, [C.c_int32, C.c_double, C.c_double, _V]),
    "mz_tree_set_root": (C.c_int, [C.POINTER(Tree), _V, _V, _V, C.c_double, _V, _V, _V]),
    "mz_tree_set_root_priors": (C.c_int, [C.POINTER(Tree), _V, _V, _V, _V, _V]),
    "mz_tree_select": (C.c_int, [C.POINTER(Tree), C.c_int32, _V, _V, _V, _V, _V]),
    "mz_tree_expand_backup": (C.c_int, [C.POINTER(Tree), C.c_int32, _V, _V, _V, _V, _V]),
    "mz_tree_step": (C.c_int, [C.POINTER(Tree), C.c_int32, _V, _V, _V, _V, _V, _V, _V, _V, _V]),
    "mz_tree_root_stats": (C.c_int, [C.POINTER(Tree), _V, _V, _V, _V, _V]),
    "mz_select_action": (C.c_int, [C.c_int32, C.c_int32, _V, _V, _V, _V, _V, _V]),
    "mz_exp_f32": (C.c_int, [C.c_int64, _V, _V, _V]),
    "mz_tree_export": (C.c_int, [C.POINTER(Tree), C.c_int32, _V, _V, _V, _V, _V, _V]),
    "mz_obs_normalize_u8": (C.c_int, [C.c_int64, C.c_int32, _V, _V, _V, _V, _V]),
    "mz_fc_initial_f32": (C.c_int, [C.POINTER(FcWeights), C.c_int32, _V, _V, C.c_int64, _V, _V, _V]),
    "mz_fc_recurrent_f32": (C.c_int, [C.POINTER(FcWeights), C.c_int32, _V, C.c_int64, _V, _V, _V,
                                      C.c_int64, C.c_int64, _V, _V, _V, _V]),
    "mz_fc_initial_tf32x3": (C.c_int, [C.POINTER(FcWeights), C.c_int32, _V, _V, C.c_int64, _V, _V, _V]),
    "mz_fc_recurrent_tf32x3": (C.c_int, [C.POINTER(FcWeights), C.c_int32, _V, C.c_int64, _V, _V, _V,
                                         C.c_int64, C.c_int64, _V, _V, _V, _V]),
    "mz_fc_tc_packed_bytes": (C.c_int64, [C.c_int32]),
    "mz_debug_set_tc_trace": (C.c_int, [_V]),
    "mz_debug_set_targets_kernel": (C.c_int, [C.c_int32]),
    "mz_debug_set_targets_tma": (C.c_int, [C.c_int32, C.c_int32]),
    "mz_debug_set_tc_trace_block": (C.c_int, [C.c_int32]),
    "mz_fc_tc_tail_floats": (C.c_int32, []),
    "mz_fc_tc_sizes": (C.c_int, [C.POINTER(FcWeights), C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                 C.POINTER(C.c_int32)]),
    "mz_fc_tc_pack": (C.c_int, [C.POINTER(FcWeights), _V, _V, _V]),
    "mz_fc_recurrent_tc": (C.c_int, [C.POINTER(FcWeights), _V, _V, C.c_int32, _V, C.c_int64, _V, _V, _V,
                                     C.c_int64, C.c_int64, _V, _V, _V, _V]),
    "mz_fc_tc_set_split": (C.c_int, [C.c_int32]),
    "mz_fc_tc_initial_packed_bytes": (C.c_int64, [C.c_int32]),
    "mz_fc_tc_pack_initial": (C.c_int, [C.POINTER(FcWeights), _V, _V, _V]),
    "mz_fc_initial_tc": (C.c_int, [C.POINTER(FcWeights), _V, _V, C.c_int32, _V, _V, C.c_int64, _V, _V, _V]),
    "mz_fc_search_game_bytes": (C.c_int64, [C.c_int32, C.c_int32]),
    "mz_fc_search_pool_row": (C.c_int32, []),
    "mz_fc_search_supported": (C.c_int, [C.c_int32, C.c_int32]),
    "mz_fc_search": (C.c_int, [C.POINTER(FcSearchArgs), _V]),
    "mz_fc_search_export": (C.c_int, [C.POINTER(FcSearchArgs), C.c_int32, _V, _V, _V, _V, _V, _V, _V]),
    "mz_scalar_transform": (C.c_int, [C.c_int64, _V, _V, _V]),
    "mz_scalar_to_support": (C.c_int, [C.c_int64, _V, C.c_int32, C.c_int32, C.c_int32, _V, _V]),
    "mz_support_to_scalar": (C.c_int, [C.c_int64, _V, C.c_int32, C.c_int32, C.c_int32, _V, _V]),
    "mz_build_targets": (C.c_int, [C.POINTER(Window), C.POINTER(TargetCfg), _V, _V, _V, _V, _V, _V,
                                   _V, _V, _V, _V, _V, _V]),
    "mz_window_append": (C.c_int, [C.POINTER(Window), C.c_int32, _V, _V, _V, _V, _V, _V, _V, _V]),
    "mz_window_copy": (C.c_int, [C.POINTER(Window), C.c_int32, _V, _V, _V, _V]),
    "mz_sumtree_update": (C.c_int, [_V, C.c_int64, C.c_int64, _V, _V, _V, _V]),
    "mz_sumtree_add": (C.c_int, [_V, C.c_int64, C.c_int64, _V, _V, C.c_int64, C.c_int32, _V, _V, _V,
                                 _V, _V]),
    "mz_dirichlet_noise": (C.c_int, [C.c_int32, C.c_int32, C.c_double, _V, C.c_uint64, C.c_uint64, _V, _V]),
    "mz_sumtree_add_chunks": (C.c_int, [_V, C.c_int64, C.c_int64, _V, _V, C.c_int32, _V, _V, _V, _V, _V, _V, _V, _V]),
    "mz_replay_sample_targets": (C.c_int, [_V, C.c_int64, _V, C.c_int32, _V, _V, _V, C.c_int64, C.c_double, _V, _V, _V, _V,
                                           _V, _V, C.POINTER(Window), C.POINTER(TargetCfg), _V, C.c_uint64, _V, _V, _V, _V,
                                           _V, _V, _V, _V]),
    "mz_sumtree_sample_mt": (C.c_int, [_V, C.c_int64, C.c_int32, _V, C.c_int32, _V, _V, _V, C.c_int64, C.c_double, _V, _V,
                                       _V, _V, _V, _V, _V]),
    "mz_sumtree_update_errors": (C.c_int, [_V, C.c_int64, C.c_int64, _V, _V, C.c_double, C.c_double, _V, _V, _V]),
    "mz_mlp2_forward": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _V, _V, _V, _V, _V, C.c_int32, _V, C.c_int32, _V]),
    "mz_mlp2_backward": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _V, _V, _V, _V, _V, C.c_int32, _V, C.c_int32, _V,
                                   C.c_int32, _V, _V, _V, _V, _V]),
    "mz_ln_relu_forward": (C.c_int, [C.c_int32, C.c_int32, _V, _V, _V, _V, C.c_int32, C.c_int32, _V, C.c_int32, _V, _V, _V]),
    "mz_ln_relu_backward": (C.c_int, [C.c_int32, C.c_int32, _V, C.c_int32, C.c_float, _V, _V, C.c_int32, _V, _V, _V, _V, _V,
                                      _V, _V]),
    "mz_learner_transpose": (C.c_int, [C.c_int32, C.c_int32, _V, _V, _V]),
    "mz_adam_step": (C.c_int, [C.c_int64, _V, _V, _V, _V, _V, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32,
                               C.c_float, C.c_float, _V]),
    "mz_chain_mask_words": (C.c_int64, [C.c_int32, C.c_int32]),
    "mz_learner_packed_words": (C.c_int64, [C.c_int32, C.c_int32]),
    "mz_learner_pack": (C.c_int, [C.c_int32, C.POINTER(PackJob), _V]),
    "mz_heads_forward_tc": (C.c_int, [C.c_int32, C.POINTER(TcJob), _V]),
    "mz_heads_backward_tc": (C.c_int, [C.c_int32, C.POINTER(TcJob), _V]),
    "mz_chain_forward_tc": (C.c_int, [C.POINTER(TcChain), _V]),
    "mz_chain_backward_tc": (C.c_int, [C.POINTER(TcChain), _V]),
    "mz_learner_packed_words_tf32x3": (C.c_int64, [C.c_int32, C.c_int32]),
    "mz_learner_pack_tf32x3": (C.c_int, [C.c_int32, C.POINTER(PackJob), _V]),
    "mz_heads_forward_tf32x3": (C.c_int, [C.c_int32, C.POINTER(TcJob), _V]),
    "mz_heads_backward_tf32x3": (C.c_int, [C.c_int32, C.POINTER(TcJob), _V]),
    "mz_chain_forward_tf32x3": (C.c_int, [C.POINTER(TcChain), _V]),
    "mz_chain_backward_tf32x3": (C.c_int, [C.POINTER(TcChain), _V]),
    "mz_sumtree_add_from": (C.c_int, [_V, C.c_int64, C.c_int64, _V, _V, C.c_int64, C.c_int32, C.c_int32, _V, _V, _V,
                                      _V, _V]),
    "mz_sumtree_sample": (C.c_int, [_V, C.c_int64, C.c_int32, _V, _V, _V, _V, C.c_int64, C.c_double,
                                    _V, _V, _V, _V, _V, _V, _V]),
    "mz_conv3x3_tc": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _V, _V, _V, C.c_int32, _V, _V, C.c_int32, _V,
                                _V, _V, _V, _V, _V]),
    "mz_conv_set_pair": (C.c_int, [C.c_int32]),
    "mz_conv_im2col_s2": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _V, _V, _V]),
    "mz_conv_gemm_to_padded": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _V, _V, _V, C.c_int32, _V,
                                         _V]),
    "mz_conv_avgpool": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, _V, _V, _V]),
    "mz_conv_gather": (C.c_int, [C.c_int32, C.c_int32, _V, _V, _V, _V]),
    "mz_conv_fc_tc": (C.c_int, [C.c_int32, _V, _V, _V, C.c_int32, C.c_int32, _V, C.c_int32, _V]),
    "mz_conv_head": (C.c_int, [C.c_int32, _V, C.c_int32, _V, _V, C.c_int32, C.c_int32, C.c_int32,
                               C.c_int32, _V, C.c_int32, _V]),
    "mz_conv_support_head_tc": (C.c_int, [C.c_int32, _V, C.c_int32, _V, _V, C.c_int32, C.c_int32, C.c_int32, _V,
                                          C.c_int32, _V]),
    "mz_unroll_loss": (C.c_int, [C.POINTER(LossCfg), _V, _V, _V, _V, _V, _V, _V, _V, _V, _V, _V, _V, _V, _V]),
    "mz_scalar_unroll_loss": (C.c_int, [C.POINTER(LossCfg), C.c_int32, _V, _V, _V, _V, _V, _V, _V, _V, _V, _V, _V, _V,
                                        _V, _V]),
    "mz_debug_div_check": (C.c_int, [C.c_uint64, C.c_int32, C.c_int32, _V, _V, _V]),
    "mz_set_programmatic_launch": (C.c_int, [C.c_int32]),
    "mz_tree_set_games_per_block": (C.c_int, [C.c_int32]),
    "mz_debug_set_tree_staging": (C.c_int, [C.c_int32]),
    "mz_version": (C.c_char_p, []),
    "mz_compiled_arch": (C.c_int32, []),
}

EXPORTED_SYMBOLS = sorted(_SIGNATURES)

_lib = None


def nvcc_path():
  """$NVCC, else nvcc on PATH, else the toolkit under $CUDA_HOME or /usr/local/cuda: a login shell's PATH often
  lacks the CUDA bin directory."""
  found = os.environ.get("NVCC") or shutil.which("nvcc")
  if found:
    return found
  for root in (os.environ.get("CUDA_HOME"), "/usr/local/cuda"):
    if root and os.access(os.path.join(root, "bin", "nvcc"), os.X_OK):
      return os.path.join(root, "bin", "nvcc")
  raise MzError("nvcc not found: put the CUDA toolkit's bin directory on PATH or set CUDA_HOME")


def build(force=False, verbose=False):
  """Compiles csrc/*.cu for sm_100a into libmzb200.so (nvcc cross-compiles without a GPU)."""
  cmd = ["make", "-C", CSRC, "-j8", "NVCC=" + nvcc_path()] + (["-B"] if force else [])
  out = None if verbose else subprocess.DEVNULL
  subprocess.check_call(cmd, stdout=out)
  return LIB_PATH


def load():
  """Loads the library; raises MzError when it is missing (there is no CPU fallback)."""
  global _lib
  if _lib is not None:
    return _lib
  path = os.environ.get("MZB200_LIB", LIB_PATH)  # A/B builds of the same ABI (diagnostics)
  if not os.path.exists(path):
    raise MzError("libmzb200.so is not built (%s); run `python -c 'import __graft_entry__ as g; "
                  "g.build()'` -- this package has no CPU fallback" % path)
  lib = C.CDLL(path)
  for name, (res, args) in _SIGNATURES.items():
    if name.startswith("mz_debug_") and not hasattr(lib, name) and path != LIB_PATH:
      continue
    fn = getattr(lib, name)  # AttributeError if the symbol is not exported
    fn.restype = res
    fn.argtypes = args
  _lib = lib
  return lib


def check(rc, what):
  if rc != 0:
    if rc > 0:
      raise MzError("%s: CUDA error %d" % (what, rc))
    raise MzError("%s: rejected arguments (code %d)" % (what, rc))


def ptr(t):
  """Device (or host) pointer of a tensor, None -> NULL."""
  if t is None:
    return None
  return C.c_void_p(t.data_ptr())


def current_stream():
  import torch
  return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def require_cuda():
  import torch
  if not torch.cuda.is_available():
    # same message as the reference raises when a GPU was requested (actors.py:41, learners.py:35)
    raise RuntimeError("GPU was requested but torch.cuda.is_available() is False.")


def normalize_device(device=None):
  """torch.device with an explicit index (so that comparisons with tensor.device work)."""
  import torch
  dev = torch.device('cuda' if device is None else device)
  if dev.type != 'cuda':
    raise RuntimeError("the B200 engine only runs on CUDA devices, got %s" % dev)
  if dev.index is None:
    dev = torch.device('cuda', torch.cuda.current_device())
  return dev


def on_device(method):
  """Decorator for methods of objects with a `.device` (or `.net.device`): the body runs with that CUDA device
  current, so `current_stream()` and every launch made through the C ABI land on the object's own GPU even when
  the caller's current device is another one."""
  import functools

  @functools.wraps(method)
  def wrapped(self, *args, **kwargs):
    import torch
    dev = getattr(self, "device", None)
    if dev is None:
      dev = self.net.device
    if torch.cuda.current_device() == dev.index:
      return method(self, *args, **kwargs)
    with torch.cuda.device(dev):
      return method(self, *args, **kwargs)
  return wrapped
