"""CPU-side checks of the drop-in boundary: the library builds for sm_100a, loads, exports every
symbol include/mzb200.h declares, and the ctypes mirrors of the structs match the C layout."""
import ctypes as C
import os
import re
import subprocess
import tempfile

import numpy as np

from model_based_rl_b200 import _lib
from model_based_rl_b200.mcts import pb_c_table

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(REPO, "include", "mzb200.h")


def declared_functions():
  src = open(HEADER).read()
  src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
  return sorted(set(re.findall(r"\b(mz_[a-z0-9_]+)\s*\(", src)))


def test_library_builds_and_exports_every_declared_symbol():
  _lib.build()
  lib = _lib.load()
  names = declared_functions()
  assert len(names) >= 15
  for n in names:
    assert hasattr(lib, n), "libmzb200.so does not export %s" % n
  assert sorted(_lib.EXPORTED_SYMBOLS) == names  # the ctypes table covers the whole header
  assert lib.mz_compiled_arch() == 100
  assert b"sm_100a" in lib.mz_version()


def test_struct_layouts_match_c():
  prog = r'''
#include <stdio.h>
#include <stddef.h>
#include "mzb200.h"
int main(void) {
  printf("%zu %zu %zu %zu\n", sizeof(mz_tree), sizeof(mz_fc_weights), sizeof(mz_window), sizeof(mz_target_cfg));
  printf("%zu %zu %zu %zu\n", offsetof(mz_tree, games), offsetof(mz_tree, leaf_action),
         offsetof(mz_fc_weights, rep_w1), offsetof(mz_target_cfg, discounts));
  printf("%zu %zu %zu %zu %zu %zu %zu\n", sizeof(mz_pack_job), sizeof(mz_tc_head), sizeof(mz_tc_job), sizeof(mz_tc_chain),
         offsetof(mz_tc_job, dx), offsetof(mz_tc_chain, hook_scale), offsetof(mz_tc_chain, dyall));
  printf("%zu %zu %zu\n", sizeof(mz_fc_search_args), offsetof(mz_fc_search_args, game_bytes),
         offsetof(mz_fc_search_args, error_flag));
  return 0;
}'''
  with tempfile.TemporaryDirectory() as d:
    open(os.path.join(d, "t.c"), "w").write(prog)
    subprocess.check_call(["gcc", "-I", os.path.join(REPO, "include"), "-o", os.path.join(d, "t"),
                           os.path.join(d, "t.c")])
    out = subprocess.check_output([os.path.join(d, "t")]).decode().split()
  sizes = [int(x) for x in out]
  assert sizes[:4] == [C.sizeof(_lib.Tree), C.sizeof(_lib.FcWeights), C.sizeof(_lib.Window),
                       C.sizeof(_lib.TargetCfg)]
  assert sizes[4:8] == [_lib.Tree.games.offset, _lib.Tree.leaf_action.offset,
                        _lib.FcWeights.rep_w1.offset, _lib.TargetCfg.discounts.offset]
  assert sizes[8:15] == [C.sizeof(_lib.PackJob), C.sizeof(_lib.TcHead), C.sizeof(_lib.TcJob), C.sizeof(_lib.TcChain),
                         _lib.TcJob.dx.offset, _lib.TcChain.hook_scale.offset, _lib.TcChain.dyall.offset]
  assert sizes[15:] == [C.sizeof(_lib.FcSearchArgs), _lib.FcSearchArgs.game_bytes.offset,
                        _lib.FcSearchArgs.error_flag.offset]


def test_fused_search_shape_boundary():
  """The shapes the persistent search kernel takes: S <= 63 and a shared-memory plan within 232 448 bytes.  The
  largest S is 63 up to 13 actions, 55 at 14..20 and 19 at 30..32; every other shape runs the per-launch path."""
  lib = _lib.load()
  for S, A in ((50, 18), (55, 18), (63, 13), (19, 32), (1, 1)):
    assert lib.mz_fc_search_supported(S, A) == 1, (S, A)
    assert lib.mz_fc_search_game_bytes(S, A) > 0, (S, A)
  for S, A in ((56, 18), (64, 4), (20, 32), (253, 1), (0, 4), (10, 0), (10, 33)):
    assert lib.mz_fc_search_supported(S, A) == 0, (S, A)
    assert lib.mz_fc_search_game_bytes(S, A) == -2, (S, A)  # MZ_ERR_UNSUPPORTED


def test_tree_geometry_and_pb_c_table_host_helpers():
  lib = _lib.load()
  for A in (1, 4, 9, 18, 32):
    nb = lib.mz_tree_node_bytes(A)
    assert nb % 16 == 0 and nb >= 16 + 10 * A
    gb = lib.mz_tree_game_bytes(50, A)
    assert gb % 128 == 0 and gb >= 32 + 51 * nb
  # the host helper and the Python table (what the reference's math.log/sqrt give) agree bit for bit
  for S, base, init in ((30, 19652, 1.25), (50, 19652, 1.25), (7, 100, 0.5)):
    tab = np.zeros((S + 1, S + 1))
    assert lib.mz_fill_pb_c_table(S, float(base), float(init), tab.ctypes.data_as(C.c_void_p)) == 0
    assert np.array_equal(tab, pb_c_table(S, base, init))


def test_bad_arguments_are_rejected_without_a_gpu():
  lib = _lib.load()
  t = _lib.Tree()
  assert lib.mz_tree_select(C.byref(t), 0, None, None, None, None, None) == -1
  assert lib.mz_scalar_transform(-1, None, None, None) == -1
  assert lib.mz_select_action(0, 4, None, None, None, None, None, None) == -1
  # host-side switches: accepted values only, and back to their defaults
  assert lib.mz_tree_set_games_per_block(3) == -1 and lib.mz_tree_set_games_per_block(8) == -1
  for games in (1, 2, 4, 0):
    assert lib.mz_tree_set_games_per_block(games) == 0
  assert lib.mz_debug_set_targets_kernel(1) == 0 and lib.mz_debug_set_targets_kernel(0) == 0
  assert lib.mz_learner_packed_words(512, 54) == 64 * 2 * 128 and lib.mz_learner_packed_words(31, 512) == 4 * 16 * 128
  assert lib.mz_learner_pack(0, None, None) == -1 and lib.mz_heads_forward_tc(4, None, None) == -1
  assert lib.mz_chain_forward_tc(C.byref(_lib.TcChain()), None) == -1
  assert lib.mz_chain_backward_tc(C.byref(_lib.TcChain()), None) == -1
  w, c = _lib.Window(), _lib.TargetCfg()
  assert lib.mz_build_targets(C.byref(w), C.byref(c), None, None, None, None, None, None, None, None, None,
                              None, None, None) == -1
