// Tree kernels: root set-up, pUCT descent, expand + backup, root statistics, action selection.
//
// One warp owns one game.  Lane l owns action l, and action l + 32 as well when A > 32: the kernels are
// instantiated for APL (actions per lane) = 1 (A <= 32) and 2 (32 < A <= 64), chosen from A at launch, and every
// sequential pass over the actions (prior sums, argmax ties) runs over ascending action indices, the low half
// (owned as action l) before the high half (action l + 32).  All score arithmetic is IEEE
// binary64 in the reference's operation order (explicit __d*_rn intrinsics; this file is also
// compiled with -fmad=false), so that argmaxes -- and therefore visit counts -- are bit-identical to
// mcts.py executed by CPython.
//
// Reference: mcts.py:6-145, config.py:70-81, game.py:106-111 (JimOhman/model-based-rl).
#include <math.h>

#include <type_traits>

#include "mz_common.cuh"
#include "mz_exp.cuh"

int g_mz_pdl = 1;

namespace {

constexpr int kThreads = 128;

// Actions [32 h, end) of the game are held by the lanes as their action `lane + 32 h`.
template <int APL>
MZ_DEV int half_end(int A, int h) {
  return APL == 1 ? A : min(A, 32 * h + 32);
}

// Node.expand priors mcts.py:52-55 for the lanes of one warp: p_a = exp(logit_a) / sum(p) with the
// sum evaluated like CPython's builtin sum() over the legal actions in ascending order.
template <int APL>
MZ_DEV void legal_priors(const float (&logit)[APL], const bool (&legal)[APL], int sum_mode, int A,
                         double (&prior)[APL]) {
  double p[APL];
  unsigned legal_bits[APL];
#pragma unroll
  for (int h = 0; h < APL; ++h) {
    p[h] = legal[h] ? mz_exp((double)logit[h]) : 0.0;
    legal_bits[h] = __ballot_sync(MZ_FULL, legal[h]);
  }
  double f = 0.0, c = 0.0;
  bool first = true;
#pragma unroll
  for (int h = 0; h < APL; ++h) {
#pragma unroll 1
    for (int a = 32 * h; a < half_end<APL>(A, h); ++a) {
      const double x = shfl_f64<32>(p[h], a - 32 * h);
      if (!((legal_bits[h] >> (a - 32 * h)) & 1u)) continue;
      if (first) {
        f = x;  // int 0 + x
        first = false;
      } else if (sum_mode == 0) {
        f = __dadd_rn(f, x);
      } else {  // Neumaier step, CPython >= 3.12 Python/bltinmodule.c
        const double t = __dadd_rn(f, x);
        if (fabs(f) >= fabs(x)) c = __dadd_rn(c, __dadd_rn(__dsub_rn(f, t), x));
        else c = __dadd_rn(c, __dadd_rn(__dsub_rn(x, t), f));
        f = t;
      }
    }
  }
  if (sum_mode != 0 && c != 0.0 && isfinite(c)) f = __dadd_rn(f, c);
#pragma unroll
  for (int h = 0; h < APL; ++h) prior[h] = legal[h] ? __ddiv_rn(p[h], f) : 0.0;
}

// ================================================================================================
// Descent (while node.expanded(): select_child, mcts.py:87-92, 104-124) and expand + backup of one
// game by a converged warp: every loop bound and branch is warp-uniform, the child's (q, visit,
// reward) arrives in one 16-byte load, MinMax normalisation divides by a per-descent constant, and
// the sequential loops run A / depth iterations.
// ================================================================================================
MZ_DEV unsigned long long sortable_key(double x) {  // monotone map double -> u64 (no NaNs)
  const unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return b ^ ((unsigned long long)((long long)b >> 63) | 0x8000000000000000ull);
}

struct NodeHead {  // first 16 bytes of a node record
  double q;
  int32_t visit;
  float reward;
};
MZ_DEV NodeHead load_head(const uint8_t* rec) {
  const int4 v = *reinterpret_cast<const int4*>(rec);
  NodeHead h;
  h.q = __hiloint2double(v.y, v.x);
  h.visit = v.z;
  h.reward = __int_as_float(v.w);
  return h;
}
MZ_DEV void store_head(uint8_t* rec, double q, int visit, float reward) {
  *reinterpret_cast<int4*>(rec) =
      make_int4(__double2loint(q), __double2hiint(q), visit, __float_as_int(reward));
}

// x / d, correctly rounded, for a divisor whose correctly rounded reciprocal r = RN(1/d) is known:
// q0 = RN(x r) is within 2 ulp, one residual step makes it faithful, and for a faithful q with an
// exact residual (fma) Markstein's theorem gives RN(q + rem r) = RN(x/d).  Valid while nothing
// under/overflows (the caller guards the exponent ranges of d and x); bit-identical to __ddiv_rn,
// checked on the device over 2^33 operand pairs by tests/test_gpu_search.py::test_fast_division.
MZ_DEV double div_by_const(double x, double d, double r) {
  const double q0 = __dmul_rn(x, r);
  const double q1 = __fma_rn(__fma_rn(-q0, d, x), r, q0);
  return __fma_rn(__fma_rn(-q1, d, x), r, q1);
}
MZ_DEV bool exp_in_fast_range(double x) {  // 2^-200 <= |x| <= 2^200
  const unsigned h = (unsigned)__double2hiint(x) & 0x7fffffffu;
  return (h - 0x33700000u) <= 0x19000000u;
}
MZ_DEV bool divisor_ok(double d) {  // exponent in range and significand not all ones
  const unsigned h = (unsigned)__double2hiint(d), l = (unsigned)__double2loint(d);
  return exp_in_fast_range(d) && !(((h & 0xfffffu) == 0xfffffu) && l == 0xffffffffu);
}

MZ_DEV unsigned long long unsortable_key(unsigned long long k) {
  return (k >> 63) ? (k ^ 0x8000000000000000ull) : ~k;
}
// max of the sortable keys of a converged warp (0 = lane does not take part)
MZ_DEV unsigned long long warp_max_key(unsigned long long key) {
  const unsigned hi = (unsigned)(key >> 32);
  const unsigned hi_max = __reduce_max_sync(MZ_FULL, hi);
  const unsigned lo_max = __reduce_max_sync(MZ_FULL, hi == hi_max ? (unsigned)key : 0u);
  return ((unsigned long long)hi_max << 32) | lo_max;
}

// Loads for the descent.  STAGED: `base` is a 32-bit shared-memory address and the loads are
// explicit ld.shared (no generic-address arithmetic in the loop); otherwise a generic pointer.
template <bool STAGED>
struct ImgLoad {
  using Addr = typename std::conditional<STAGED, uint32_t, const uint8_t*>::type;
  static MZ_DEV Addr base(const uint8_t* img) {
    if constexpr (STAGED) return smem_u32(img);
    else return img;
  }
  static MZ_DEV double f64(Addr a) {
    if constexpr (STAGED) {
      double v;
      asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
      return v;
    } else {
      return *reinterpret_cast<const double*>(a);
    }
  }
  static MZ_DEV int s16(Addr a) {
    if constexpr (STAGED) {
      int v;
      asm volatile("ld.shared.s16 %0, [%1];" : "=r"(v) : "r"(a));
      return v;
    } else {
      return *reinterpret_cast<const int16_t*>(a);
    }
  }
  static MZ_DEV NodeHead head(Addr a) {
    int x, y, z, w;
    if constexpr (STAGED) {
      asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(x), "=r"(y), "=r"(z), "=r"(w) : "r"(a));
    } else {
      const int4 v = *reinterpret_cast<const int4*>(a);
      x = v.x; y = v.y; z = v.z; w = v.w;
    }
    NodeHead h;
    h.q = __hiloint2double(y, x);
    h.visit = z;
    h.reward = __int_as_float(w);
    return h;
  }
};

// (score, action) argmax over the actions of a converged warp, ties -> larger action
// (mcts.py:106-112): returns the winning action or -1 when no action is a candidate.
template <int APL>
MZ_DEV int warp_argmax(const double (&score)[APL], const bool (&cand)[APL]) {
  if constexpr (APL == 1) {
    const unsigned long long key = cand[0] ? sortable_key(score[0]) : 0ull;
    const unsigned long long best_key = warp_max_key(key);
    const unsigned winners = __ballot_sync(MZ_FULL, cand[0] && key == best_key);
    return winners ? 31 - __clz(winners) : -1;
  } else {
    // the lane's own pair first (a tie goes to action lane + 32), then the warp; every high-half action is
    // larger than every low-half one, so a high-half winner takes the ties across lanes
    const unsigned long long k0 = cand[0] ? sortable_key(score[0]) : 0ull;
    const unsigned long long k1 = cand[1] ? sortable_key(score[1]) : 0ull;
    const bool hi = cand[1] && k1 >= k0;
    const unsigned long long key = hi ? k1 : k0;  // 0 <=> neither action is a candidate
    const unsigned long long best_key = warp_max_key(key);
    const bool win = key != 0ull && key == best_key;
    const unsigned win_hi = __ballot_sync(MZ_FULL, win && hi), win_lo = __ballot_sync(MZ_FULL, win && !hi);
    if (win_hi) return 63 - __clz(win_hi);
    return win_lo ? 31 - __clz(win_lo) : -1;
  }
}

// MODE: MinMaxStats.normalize (mcts.py:16-21) hoisted out of the loop -- 2 = (v - min) / (max - min)
// through the constant-divisor division, 3 = same through IEEE division, 1 = constant 1.0, 0 = raw.
template <bool STAGED, int MODE, int APL>
MZ_DEV void descend_loop(const mz_tree& t, typename ImgLoad<STAGED>::Addr nodes, int lane, int16_t* path,
                         int N, double mn, double d, double r, int& out_depth, int& out_parent,
                         int& out_action) {
  using L = ImgLoad<STAGED>;
  const int A = t.num_actions, SP1 = t.num_simulations + 1, NB = t.node_bytes;
  const double init_score = t.init_value_score;
  bool lane_ok[APL];
  int prior_off[APL], child_off[APL];
#pragma unroll
  for (int h = 0; h < APL; ++h) {
    lane_ok[h] = lane + 32 * h < A;
    const int sp = lane_ok[h] ? lane + 32 * h : A - 1;
    prior_off[h] = MZ_NODE_STATS_BYTES + 8 * sp;
    child_off[h] = MZ_NODE_STATS_BYTES + 8 * A + 2 * sp;
  }
  const double* table = t.pb_c_table;
  int node = 0, depth = 0, parent, action;
  const double* row = table + N * SP1;  // pb_c[N][.] of the node being expanded (warp-uniform)
  for (;;) {
    const typename L::Addr rec = nodes + node * NB;
    double score[APL];
    bool cand[APL];
    int ch[APL], n[APL];
#pragma unroll
    for (int h = 0; h < APL; ++h) {
      const double prior = L::f64(rec + prior_off[h]);
      ch[h] = L::s16(rec + child_off[h]);
      if (!lane_ok[h]) ch[h] = MZ_CHILD_ILLEGAL;
      const NodeHead c = L::head(nodes + max(ch[h], 0) * NB);
      n[h] = ch[h] >= 0 ? c.visit : 0;
      // ucb_score mcts.py:115-124
      const double pb_c = __ldg(row + n[h]);
      double value_score;
      if (MODE == 0) {
        value_score = c.q;
      } else if (MODE == 1) {
        value_score = 1.0;
      } else if (MODE == 3) {
        value_score = __ddiv_rn(__dsub_rn(c.q, mn), d);
      } else {
        // every lane evaluates the constant-divisor division (lanes without a visited child discard it);
        // only a visited child outside [2^-200, 2^200] (or exactly at the minimum) takes the IEEE path
        const double x = __dsub_rn(c.q, mn);
        value_score = div_by_const(x, d, r);
        const unsigned hx = (unsigned)__double2hiint(x);  // x >= 0 because min <= q
        if (__builtin_expect(n[h] > 0 && hx - 0x33700000u > 0x19000000u, 0))
          value_score = (x == 0.0) ? 0.0 : __ddiv_rn(x, d);
      }
      if (n[h] <= 0) value_score = init_score;
      score[h] = __dadd_rn(__dmul_rn(pb_c, prior), value_score);
      cand[h] = ch[h] != MZ_CHILD_ILLEGAL;
    }
    const int best = warp_argmax<APL>(score, cand);
    const int src = best < 0 ? 0 : (APL == 1 ? best : best & 31);
    const bool high = APL == 2 && best >= 32;  // warp-uniform
    const int ch_b = __shfl_sync(MZ_FULL, high ? ch[APL - 1] : ch[0], src);
    const int n_b = __shfl_sync(MZ_FULL, high ? n[APL - 1] : n[0], src);
    depth++;
    if (ch_b < 0) {  // child not expanded: this is the leaf
      parent = node;
      action = best;
      break;
    }
    node = ch_b;
    row = table + n_b * SP1;
    path[depth] = (int16_t)node;  // every lane stores the same value to the same address
  }
  out_depth = depth;
  out_parent = parent;
  out_action = action;
}

template <bool STAGED, int APL>
MZ_DEV void descend(const mz_tree& t, const uint8_t* img, int lane, int16_t* path, int& out_depth,
                    int& out_parent, int& out_action) {
  using L = ImgLoad<STAGED>;
  const int A = t.num_actions;
  const typename L::Addr base = L::base(img);
  const double mn = L::f64(base), mx = L::f64(base + 8);
  const typename L::Addr nodes = base + MZ_GAME_HEADER_BYTES;
  const int N = L::head(nodes).visit;
  if (lane == 0) path[0] = 0;
  if (N == 0) {
    // mcts.py:105-108: an unvisited root (simulation 0) ranks its children by prior; none of them
    // is expanded yet, so the first step already reaches the leaf
    double prior[APL];
    bool cand[APL];
#pragma unroll
    for (int h = 0; h < APL; ++h) {
      const bool lane_ok = lane + 32 * h < A;
      const int sp = lane_ok ? lane + 32 * h : A - 1;
      prior[h] = L::f64(nodes + MZ_NODE_STATS_BYTES + 8 * sp);
      const int ch = L::s16(nodes + MZ_NODE_STATS_BYTES + 8 * A + 2 * sp);
      cand[h] = lane_ok && ch != MZ_CHILD_ILLEGAL;
    }
    const int best = warp_argmax<APL>(prior, cand);
    out_depth = 1;
    out_parent = 0;
    out_action = best;
    return;
  }
  const double d = __dsub_rn(mx, mn);
  if (mx > mn) {
    if (divisor_ok(d)) descend_loop<STAGED, 2, APL>(t, nodes, lane, path, N, mn, d, __drcp_rn(d), out_depth, out_parent, out_action);
    else descend_loop<STAGED, 3, APL>(t, nodes, lane, path, N, mn, d, 0.0, out_depth, out_parent, out_action);
  } else if (mx == mn) {
    descend_loop<STAGED, 1, APL>(t, nodes, lane, path, N, mn, d, 0.0, out_depth, out_parent, out_action);
  } else {
    descend_loop<STAGED, 0, APL>(t, nodes, lane, path, N, mn, d, 0.0, out_depth, out_parent, out_action);
  }
}

// expand (mcts.py:47-55) + backpropagate (mcts.py:126-143).  `img` is the
// image the warp reads (shared memory when STAGED, else the global block); stores go to the global
// block and, when staged, to the image as well.
template <bool STAGED, int APL>
MZ_DEV void expand_backup(const mz_tree& t, uint8_t* img, uint8_t* gbl, int lane, int sim,
                          float value_f, float reward_f, const float (&logit)[APL], int16_t* path, int depth,
                          int parent, int action) {
  const int A = t.num_actions, NB = t.node_bytes;
  const bool two = t.two_players != 0;
  const double disc = t.discount;
  const int newn = sim + 1;
  const float node_reward_new = (reward_f != 0.0f) ? reward_f : 0.0f;  // `if network_output.reward:`
  uint8_t* nodes_s = img + MZ_GAME_HEADER_BYTES;
  uint8_t* nodes_g = gbl + MZ_GAME_HEADER_BYTES;

  // the path positions this lane owns in the first (deepest) chunk: issue the loads early
  const int top = (depth >> 5) << 5;
  int nid_top = 0;
  if (top + lane < depth) nid_top = path[top + lane];

  // priors: p_a = exp(logit_a) / sum(p), the sum evaluated like CPython's builtin sum()
  // (every action is legal below the root, mcts.py:72, 97)
  double p[APL];
#pragma unroll
  for (int h = 0; h < APL; ++h) p[h] = lane + 32 * h < A ? mz_exp((double)logit[h]) : 0.0;
  double f = shfl_f64<32>(p[0], 0), c = 0.0;
  if (t.prior_sum_mode == 0) {
#pragma unroll
    for (int h = 0; h < APL; ++h) {
#pragma unroll 1
      for (int a = h == 0 ? 1 : 32; a < half_end<APL>(A, h); ++a) f = __dadd_rn(f, shfl_f64<32>(p[h], a - 32 * h));
    }
  } else {  // Neumaier step, CPython >= 3.12 Python/bltinmodule.c
#pragma unroll
    for (int h = 0; h < APL; ++h) {
#pragma unroll 1
      for (int a = h == 0 ? 1 : 32; a < half_end<APL>(A, h); ++a) {
        const double x = shfl_f64<32>(p[h], a - 32 * h);
        const double s = __dadd_rn(f, x);
        const bool big = fabs(f) >= fabs(x);
        const double hi = big ? f : x, lo = big ? x : f;
        c = __dadd_rn(c, __dadd_rn(__dsub_rn(hi, s), lo));
        f = s;
      }
    }
    if (c != 0.0 && isfinite(c)) f = __dadd_rn(f, c);
  }
#pragma unroll
  for (int h = 0; h < APL; ++h) {
    const int a = lane + 32 * h;
    if (a < A) {
      const double prior = __ddiv_rn(p[h], f);
      const int po = newn * NB + MZ_NODE_STATS_BYTES + 8 * a;
      const int co = newn * NB + MZ_NODE_STATS_BYTES + 8 * A + 2 * a;
      *reinterpret_cast<double*>(nodes_g + po) = prior;
      *reinterpret_cast<int16_t*>(nodes_g + co) = (int16_t)MZ_CHILD_UNEXPANDED;
      if (STAGED) {
        *reinterpret_cast<double*>(nodes_s + po) = prior;
        *reinterpret_cast<int16_t*>(nodes_s + co) = (int16_t)MZ_CHILD_UNEXPANDED;
      }
    }
  }
  if (lane == 0) {
    const int co = parent * NB + MZ_NODE_STATS_BYTES + 8 * A + 2 * action;
    *reinterpret_cast<int16_t*>(nodes_g + co) = (int16_t)newn;
    if (STAGED) *reinterpret_cast<int16_t*>(nodes_s + co) = (int16_t)newn;
    path[depth] = (int16_t)newn;
  }

  // backup.  Position k on the path holds node path[k] (k < depth) or the new node (k == depth).
  double value = (double)value_f;
  unsigned long long kmax = 0ull, kmin = 0ull;  // sortable keys of max(q) and of -min ordering
  const unsigned twomask = two ? 0x80000000u : 0u;
  unsigned signmask = twomask;  // position `depth` is the leaf: node.to_play == to_play
  for (int base = top; base >= 0; base -= 32) {
    const int k = base + lane;
    const bool has = k <= depth;
    const int nid = k < depth ? (base == top ? nid_top : (int)path[k]) : newn;
    double vs = 0.0;
    int vc = 0;
    float rw = node_reward_new;
    if (k < depth) {
      const uint8_t* rec = nodes_s + nid * NB;
      const NodeHead h = load_head(rec);
      vc = h.visit;
      rw = h.reward;
      vs = *reinterpret_cast<const double*>(rec + 16);
    }
    double myval = 0.0;
    unsigned mysign = 0u;
#pragma unroll 1
    for (int j = min(31, depth - base); j >= 0; --j) {
      const unsigned rj = __shfl_sync(MZ_FULL, __float_as_uint(rw), j);
      if (lane == j) {
        myval = value;
        mysign = signmask;
      }
      // value = (-reward if two_players and node.to_play == to_play else reward) + discount * value
      value = __dadd_rn((double)__uint_as_float(rj ^ signmask), __dmul_rn(disc, value));
      signmask ^= twomask;
    }
    if (has) {
      // value_sum += value if node.to_play == to_play else -value   (mysign set <=> same player
      // in a two-player game; single player: always the same player)
      const bool same = two ? mysign != 0u : true;
      vs = __dadd_rn(vs, same ? myval : -myval);
      vc += 1;
      double new_q = 0.0;
      if (k > 0) {  // mcts.py:136-141
        const double dq = __dmul_rn(disc, __ddiv_rn(vs, (double)vc));
        new_q = two ? __dsub_rn((double)rw, dq) : __dadd_rn((double)rw, dq);
      }
      store_head(nodes_g + nid * NB, new_q, vc, rw);
      *reinterpret_cast<double*>(nodes_g + nid * NB + 16) = vs;
      if (STAGED) {
        store_head(nodes_s + nid * NB, new_q, vc, rw);
        *reinterpret_cast<double*>(nodes_s + nid * NB + 16) = vs;
      }
      if (k > 0) {
        const unsigned long long key = sortable_key(new_q);
        kmax = key > kmax ? key : kmax;
        kmin = ~key > kmin ? ~key : kmin;
      }
    }
    if (depth > 0) {
      kmax = warp_max_key(kmax);
      kmin = warp_max_key(kmin);
    }
  }
  if (lane == 0 && depth > 0) {  // MinMaxStats.update mcts.py:11-14
    const double lmax = __longlong_as_double((long long)unsortable_key(kmax));
    const double lmin = __longlong_as_double((long long)unsortable_key(~kmin));
    if (lmin < *reinterpret_cast<double*>(img)) {
      *reinterpret_cast<double*>(gbl) = lmin;
      if (STAGED) *reinterpret_cast<double*>(img) = lmin;
    }
    if (lmax > *reinterpret_cast<double*>(img + 8)) {
      *reinterpret_cast<double*>(gbl + 8) = lmax;
      if (STAGED) *reinterpret_cast<double*>(img + 8) = lmax;
    }
  }
}

MZ_DEV void copy_words(uint32_t* dst, const uint32_t* src, int words, int lane) {
  for (int i = lane; i < words; i += 32) dst[i] = src[i];
}

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
template <int APL>
__global__ void __launch_bounds__(kThreads)
set_root_kernel(mz_tree t, const float* __restrict__ root_logits,
                const uint32_t* __restrict__ legal_mask, const double* __restrict__ noise,
                double noise_frac, const int8_t* __restrict__ root_to_play,
                const uint32_t* __restrict__ root_hidden, const double* __restrict__ root_priors) {
  const int gidx = (blockIdx.x * kThreads + threadIdx.x) / 32;
  const int lane = threadIdx.x & 31;
  const bool valid = gidx < t.num_games;
  const int g = valid ? gidx : t.num_games - 1;
  const int A = t.num_actions;
  const MzGame gm{t.games + (size_t)g * t.game_bytes, t.node_bytes, A};
  uint32_t lm[APL];  // legal-mask words of the game (APL = ceil(A / 32))
  bool legal[APL];
  double prior[APL];
#pragma unroll
  for (int h = 0; h < APL; ++h) {
    lm[h] = legal_mask ? legal_mask[(size_t)g * APL + h] : 0xffffffffu;
    legal[h] = lane + 32 * h < A && ((lm[h] >> lane) & 1u);
  }
  if (root_priors) {  // the caller ran Node.expand / add_exploration_noise itself
#pragma unroll
    for (int h = 0; h < APL; ++h) prior[h] = legal[h] ? root_priors[(size_t)g * A + lane + 32 * h] : 0.0;
  } else {
    float logit[APL];
#pragma unroll
    for (int h = 0; h < APL; ++h) logit[h] = lane + 32 * h < A ? root_logits[(size_t)g * A + lane + 32 * h] : 0.0f;
    legal_priors<APL>(logit, legal, t.prior_sum_mode, A, prior);
  }
#pragma unroll
  for (int h = 0; h < APL; ++h) {
    if (noise && legal[h]) {  // add_exploration_noise mcts.py:57-61; noise is dense over children
      // every bit of the low word is an action when A > 32
      const int j = (h ? __popc(lm[0]) : 0) + __popc(lm[h] & ((1u << lane) - 1u));
      const double nz = noise[(size_t)g * A + j];
      prior[h] = __dadd_rn(__dmul_rn(prior[h], __dsub_rn(1.0, noise_frac)), __dmul_rn(nz, noise_frac));
    }
  }
  if (!valid) return;
  const MzNode root = gm.node(0);
#pragma unroll
  for (int h = 0; h < APL; ++h) {
    if (lane + 32 * h < A) {
      root.prior()[lane + 32 * h] = prior[h];
      root.child()[lane + 32 * h] = (int16_t)(legal[h] ? MZ_CHILD_UNEXPANDED : MZ_CHILD_ILLEGAL);
    }
  }
  if (lane == 0) {
    root.vsum() = 0.0;
    root.q() = 0.0;
    root.visit() = 0;
    root.reward() = 0.0f;
    gm.mn() = t.min_bound;  // MinMaxStats.reset mcts.py:79
    gm.mx() = t.max_bound;
    gm.root_to_play() = root_to_play ? (int32_t)root_to_play[g] : 1;
  }
  if (root_hidden && t.hidden_words > 0)
    copy_words(t.hidden + (size_t)g * (t.num_simulations + 1) * t.hidden_words,
               root_hidden + (size_t)g * t.hidden_words, t.hidden_words, lane);
}

// One launch per simulation boundary: [expand + backup of simulation `sim`] then [descent of
// simulation sim + 1].  STAGED: the live part of each game block (header + nodes 0..sim) is brought
// into shared memory with one cp.async.bulk (TMA unit) per game and both phases run on that image.
// blockDim.x = 32 * games_per_block.
template <bool STAGED, int APL>
__global__ void __launch_bounds__(kThreads)
tree_step_w32_kernel(mz_tree t, int sim, int do_backup, int do_select, int live_nodes, int stage_bytes,
                     const float* __restrict__ value, const float* __restrict__ reward,
                     const float* __restrict__ logits, const uint32_t* __restrict__ new_hidden,
                     uint32_t* __restrict__ gathered_hidden, int32_t* __restrict__ trace_parent,
                     int32_t* __restrict__ trace_action, int32_t* __restrict__ trace_depth) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int wpb = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x * wpb + warp;
  const bool valid = g < t.num_games;
  const int A = t.num_actions, SP1 = t.num_simulations + 1, HW = t.hidden_words;
  uint8_t* gbl = t.games + (size_t)(valid ? g : 0) * t.game_bytes;
  uint8_t* img = gbl;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)wpb * stage_bytes);
  if (STAGED) {
    if (threadIdx.x == 0) {
      for (int i = 0; i < wpb; ++i) mbar_init(&bars[i], 1);
      mbar_fence_init();
    }
    __syncthreads();
    if (!valid) return;
    img = smem + (size_t)warp * stage_bytes;
    // nodes 0..live_nodes-1 exist before this launch (a backup creates node `sim + 1` in place)
    const uint32_t live = MZ_GAME_HEADER_BYTES + (uint32_t)live_nodes * (uint32_t)t.node_bytes;
    if (lane == 0) {
      mbar_arrive_expect_tx(&bars[warp], live);
      bulk_copy_g2s(img, gbl, live, &bars[warp]);
    }
  } else if (!valid) {
    return;
  }
  int16_t* path = t.path + (size_t)g * (t.num_simulations + 2);

  if (do_backup) {
    // everything the backup needs from global memory is requested before waiting for the image
    const int depth = t.path_len[g], parent = t.leaf_parent[g], action = t.leaf_action[g];
    pdl_wait();     // the network kernel's outputs (and nothing before this line) depend on it
    pdl_trigger();
    float logit[APL];
#pragma unroll
    for (int h = 0; h < APL; ++h) logit[h] = lane + 32 * h < A ? logits[(size_t)g * A + lane + 32 * h] : 0.0f;
    const float v = value[g], r = reward[g];
    if (STAGED) mbar_wait(&bars[warp], 0);
    expand_backup<STAGED, APL>(t, img, gbl, lane, sim, v, r, logit, path, depth, parent, action);
    if (new_hidden && HW > 0)
      copy_words(t.hidden + ((size_t)g * SP1 + sim + 1) * HW, new_hidden + (size_t)g * HW, HW, lane);
    __syncwarp();
  } else {
    pdl_wait();
    pdl_trigger();
    if (STAGED) mbar_wait(&bars[warp], 0);
  }
  if (do_select) {
    int depth, parent, action;
    descend<STAGED, APL>(t, img, lane, path, depth, parent, action);
    if (lane == 0) {
      t.path_len[g] = depth;
      t.leaf_parent[g] = parent;
      t.leaf_action[g] = action;
      if (trace_parent) trace_parent[g] = parent;
      if (trace_action) trace_action[g] = action;
      if (trace_depth) trace_depth[g] = depth;
    }
    if (gathered_hidden && HW > 0)
      copy_words(gathered_hidden + (size_t)g * HW, t.hidden + ((size_t)g * SP1 + parent) * HW, HW, lane);
  }
}

// game.py:106-111 + Node.value mcts.py:42-45
// One warp per game, a lane per action (two above 32 actions; the per-action loads are two dependent L2
// accesses: child index -> child's visit count; a thread per game serialised 2 A of them).
template <int APL>
__global__ void root_stats_kernel(mz_tree t, int32_t* __restrict__ visits,
                                  double* __restrict__ child_visits, double* __restrict__ root_value,
                                  double* __restrict__ minmax) {
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (g >= t.num_games) return;
  const int A = t.num_actions;
  const MzGame gm{t.games + (size_t)g * t.game_bytes, t.node_bytes, A};
  const MzNode root = gm.node(0);
  int ch[APL], v[APL], mine = 0;
#pragma unroll
  for (int h = 0; h < APL; ++h) {
    ch[h] = MZ_CHILD_ILLEGAL;
    v[h] = 0;
    if (lane + 32 * h < A) {
      ch[h] = root.child()[lane + 32 * h];
      v[h] = ch[h] >= 0 ? gm.node(ch[h]).visit() : 0;
    }
    mine += v[h];
  }
  const int sum = __reduce_add_sync(MZ_FULL, mine);  // integer: order does not matter
#pragma unroll
  for (int h = 0; h < APL; ++h) {
    const int a = lane + 32 * h;
    if (a < A) {
      if (visits) visits[(size_t)g * A + a] = v[h];
      if (child_visits)
        child_visits[(size_t)g * A + a] = ch[h] != MZ_CHILD_ILLEGAL ? __ddiv_rn((double)v[h], (double)sum) : 0.0;
    }
  }
  if (lane == 0) {
    if (root_value) {
      const int n = root.visit();
      root_value[g] = n == 0 ? 0.0 : __ddiv_rn(root.vsum(), (double)n);
    }
    if (minmax) {
      minmax[2 * g] = gm.mn();
      minmax[2 * g + 1] = gm.mx();
    }
  }
}

// numpy's float64 add.reduce over a contiguous row (pairwise sum with 8 accumulators, n <= 128)
__device__ double np_pairwise_sum(const double* a, int n) {
  if (n < 8) {
    double res = 0.0;
    for (int i = 0; i < n; ++i) res = __dadd_rn(res, a[i]);
    return res;
  }
  double r[8];
  for (int j = 0; j < 8; ++j) r[j] = a[j];
  int i;
  for (i = 8; i < n - (n % 8); i += 8)
    for (int j = 0; j < 8; ++j) r[j] = __dadd_rn(r[j], a[i + j]);
  double res = __dadd_rn(__dadd_rn(__dadd_rn(r[0], r[1]), __dadd_rn(r[2], r[3])),
                         __dadd_rn(__dadd_rn(r[4], r[5]), __dadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __dadd_rn(res, a[i]);
  return res;
}

// Config.select_action config.py:70-81.  One warp per game: the legal actions are compacted to
// candidates 0..n-1 (action order, like the dict of children), candidate i on lane i % 32; pow, the two
// divisions and the comparison run per candidate, the two float64 sums keep numpy's order (pairwise
// add.reduce, sequential cumsum).
template <int APL>
__global__ void select_action_kernel(int G, int A, const int32_t* __restrict__ visits,
                                     const uint32_t* __restrict__ legal_mask,
                                     const double* __restrict__ temperature,
                                     const double* __restrict__ uniforms,
                                     int32_t* __restrict__ actions) {
  __shared__ double s_d[4][32 * APL];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x * 4 + w;
  if (g >= G) return;
  uint32_t lm[APL];
#pragma unroll
  for (int h = 0; h < APL; ++h) lm[h] = legal_mask ? legal_mask[(size_t)g * APL + h] : 0xffffffffu;
  if (A < 32 * APL) lm[APL - 1] &= (1u << (A - 32 * (APL - 1))) - 1u;
  const int n0 = __popc(lm[0]);
  const int n = APL == 1 ? n0 : n0 + __popc(lm[APL - 1]);
  if (n == 0) {
    if (lane == 0) actions[g] = -1;
    return;
  }
  // candidate i = lane + 32 h < n is the i-th legal action
  int my_act[APL], cnt[APL];
#pragma unroll
  for (int h = 0; h < APL; ++h) {
    const int i = lane + 32 * h;
    my_act[h] = i >= n ? 0 : (APL == 1 || i < n0) ? __fns(lm[0], 0, i + 1) : 32 + __fns(lm[APL - 1], 0, i - n0 + 1);
    cnt[h] = i < n ? visits[(size_t)g * A + my_act[h]] : 0;
  }
  const double T = temperature[g], u = uniforms[g];
  double* d = s_d[w];
  int idx = 0;
  if (T != 0.0) {
    const double inv_t = __ddiv_rn(1.0, T);
#pragma unroll
    for (int h = 0; h < APL; ++h)
      if (lane + 32 * h < n) d[lane + 32 * h] = pow((double)cnt[h], inv_t);
    __syncwarp();
    double s = 0.0;
    if (lane == 0) s = np_pairwise_sum(d, n);
    s = shfl_f64<32>(s, 0);
    __syncwarp();
#pragma unroll
    for (int h = 0; h < APL; ++h)
      if (lane + 32 * h < n) d[lane + 32 * h] = __ddiv_rn(d[lane + 32 * h], s);  // distribution / sum
    __syncwarp();
    if (lane == 0) {  // cumsum
      double acc = d[0];
      for (int i = 1; i < n; ++i) {
        acc = __dadd_rn(acc, d[i]);
        d[i] = acc;
      }
    }
    __syncwarp();
    const double last = d[n - 1];
    unsigned m[APL];
#pragma unroll
    for (int h = 0; h < APL; ++h) {
      const int i = lane + 32 * h;
      m[h] = __ballot_sync(MZ_FULL, i < n && __ddiv_rn(d[i], last) <= u);  // searchsorted(side='right')
    }
    // (last index with cdf <= u) + 1, as the sequential scan leaves it
    idx = (APL == 2 && m[APL - 1]) ? 64 - __clz(m[APL - 1]) : m[0] ? 32 - __clz(m[0]) : 0;
    if (idx >= n) idx = n - 1;
  } else {
    int c = lane < n ? cnt[0] : -1;
    if (APL == 2) c = max(c, lane + 32 < n ? cnt[APL - 1] : -1);
    const int mx = __reduce_max_sync(MZ_FULL, c);
    unsigned tie[APL];
#pragma unroll
    for (int h = 0; h < APL; ++h) tie[h] = __ballot_sync(MZ_FULL, lane + 32 * h < n && cnt[h] == mx);
    const int t0 = __popc(tie[0]);
    const int ties = APL == 1 ? t0 : t0 + __popc(tie[APL - 1]);
    int pick = (int)floor(__dmul_rn(u, (double)ties));
    if (pick >= ties) pick = ties - 1;
    // the pick-th tie in action order
    idx = (APL == 1 || pick < t0) ? __fns(tie[0], 0, pick + 1) : 32 + __fns(tie[APL - 1], 0, pick - t0 + 1);
  }
  const int chosen = __shfl_sync(MZ_FULL, (APL == 2 && idx >= 32) ? my_act[APL - 1] : my_act[0],
                                   APL == 1 ? idx : idx & 31);
  if (lane == 0) actions[g] = chosen;
}

__global__ void tree_export_kernel(mz_tree t, int game, double* prior, int32_t* child, double* vsum,
                                   int32_t* visit, float* reward) {
  const int A = t.num_actions, SP1 = t.num_simulations + 1;
  const MzGame gm{t.games + (size_t)game * t.game_bytes, t.node_bytes, A};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < SP1 * A; i += gridDim.x * blockDim.x) {
    const int n = i / A, a = i % A;
    const MzNode nd = gm.node(n);
    if (prior) prior[i] = nd.prior()[a];
    if (child) child[i] = nd.child()[a];
    if (a == 0) {
      if (vsum) vsum[n] = nd.vsum();
      if (visit) visit[n] = nd.visit();
      if (reward) reward[n] = nd.reward();
    }
  }
}

__global__ void exp_f32_kernel(long long n, const float* __restrict__ x, double* __restrict__ out) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x)
    out[i] = mz_exp((double)x[i]);
}

// Diagnostics: div_by_const against __ddiv_rn on pseudo-random operand pairs shaped like the
// MinMax normalisation (0 <= x <= d) plus adversarial significands.  Counts mismatches.
MZ_DEV unsigned long long mix64(unsigned long long z) {
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
__global__ void div_check_kernel(unsigned long long seed, int per_thread,
                                 unsigned long long* __restrict__ mismatches,
                                 unsigned long long* __restrict__ tested) {
  unsigned long long state = seed + (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x) * 0x632be59bd9b4e019ull;
  unsigned long long bad = 0, done = 0;
  for (int i = 0; i < per_thread; ++i) {
    const unsigned long long a = mix64(state), b = mix64(state + 1), c = mix64(state + 2);
    state += 3;
    // divisor: random significand (sometimes nearly all ones / all zeros / few bits), exponent 2^-60..2^60
    unsigned long long mant = a & 0xfffffffffffffull;
    const unsigned kind = (unsigned)(c & 7u);
    if (kind == 0) mant |= 0xffffffffff000ull;
    else if (kind == 1) mant &= 0xfffull;
    else if (kind == 2) mant &= 0xfff0000000000ull;
    const long long ed = 1023 + (long long)((a >> 52) % 121) - 60;
    const double d = __longlong_as_double((long long)(((unsigned long long)ed << 52) | mant));
    // dividend: u * d with u in [0, 1], or a small multiple of d, nudged by a few ulps
    double x;
    const unsigned xk = (unsigned)((c >> 3) & 3u);
    if (xk == 0) x = __dmul_rn(d, (double)(b >> 11) * 0x1p-53);
    else if (xk == 1) x = __dmul_rn(d, (double)((b >> 20) & 1023u) * 0x1p-10);
    else if (xk == 2) x = __longlong_as_double((long long)(((unsigned long long)(ed - (long long)((b >> 52) % 40)) << 52) | (b & 0xfffffffffffffull)));
    else x = __dmul_rn(d, (double)(b >> 11) * 0x1p-53 * 0x1p-30);
    long long xb = __double_as_longlong(x) + (long long)((c >> 5) & 7u) - 3;
    if (xb < 0) xb = 0;
    x = __longlong_as_double(xb);
    if (!divisor_ok(d) || !(x == 0.0 || exp_in_fast_range(x))) continue;
    const double want = __ddiv_rn(x, d);
    const double got = div_by_const(x, d, __drcp_rn(d));
    bad += (__double_as_longlong(want) != __double_as_longlong(got));
    ++done;
  }
  if (bad) atomicAdd(mismatches, bad);
  atomicAdd(tested, done);
}

int check_tree(const mz_tree* t) {
  if (!t || !t->games || !t->pb_c_table || !t->path || !t->path_len || !t->leaf_parent ||
      !t->leaf_action)
    return MZ_ERR_BAD_ARG;
  if (t->num_games < 1 || t->num_simulations < 1 || t->num_simulations > 32000) return MZ_ERR_BAD_ARG;
  if (t->num_actions < 1 || t->num_actions > MZ_MAX_ACTIONS) return MZ_ERR_BAD_ARG;
  if (t->node_bytes != mz_tree_node_bytes(t->num_actions)) return MZ_ERR_BAD_ARG;
  if (t->game_bytes < mz_tree_game_bytes(t->num_simulations, t->num_actions)) return MZ_ERR_BAD_ARG;
  if (t->hidden_words < 0 || (t->hidden_words > 0 && !t->hidden)) return MZ_ERR_BAD_ARG;
  return MZ_OK;
}

// Games (= warps) per CTA of the warp-per-game step kernel.  One game per CTA from 512 games per launch on: a CTA
// gives its shared memory back as soon as ITS game's descent ends (a four-game CTA holds 4 images until the
// deepest of them is done), 21 instead of 20 images fit an SM at the last simulation, and a one-game CTA fits
// beside a network-kernel CTA (16 KB of shared memory left there).  Measured on one box, 30 timed moves, 4 / 2 / 1
// games per CTA: C4 136.9-137.3 / 135.9 / 139.1-139.3 M expansions/s, 16 384 games 191.6-194.8 / 196.5 / 209.6 M,
// C3 shape 188.5-189.6 / 186.5 / 205.9-208.7 M; 256-game launches (C2 shape) prefer four: 60.1-60.3 vs 57.6-59.0 M.
// mz_tree_set_games_per_block(1|2|4) forces one value, 0 = by launch size.
int g_w32_gpb = 0;
int w32_games_per_block(int num_games) {
  if (g_w32_gpb) return g_w32_gpb;
  return num_games >= 512 ? 1 : kThreads / 32;
}

constexpr int kMaxStageSmem = 200 * 1024;

// Shared-memory image of the step kernel: 0 = staged whenever the images fit (default), 1 = never staged
// (mz_debug_set_tree_staging; for measurements).
int g_tree_staging = 0;

template <bool STAGED, int APL>
int set_smem_attr_w32_once() {
  static int rc = -1;
  if (rc < 0)
    rc = (int)cudaFuncSetAttribute(tree_step_w32_kernel<STAGED, APL>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxStageSmem + 1024);
  return rc;
}

template <int APL>
int launch_step_apl(const mz_tree* t, int sim, int live_nodes, int do_backup, int do_select, const float* value,
                    const float* reward, const float* logits, const uint32_t* new_hidden,
                    uint32_t* gathered_hidden, int32_t* tp, int32_t* ta, int32_t* td, void* stream) {
  // image: header + nodes 0..sim+1 (the new node is built in place)
  const int nodes = live_nodes + (do_backup ? 1 : 0);
  const int stage_bytes = MZ_GAME_HEADER_BYTES + nodes * t->node_bytes;
  int gpb = w32_games_per_block(t->num_games);
  while (gpb > 1 && (size_t)gpb * stage_bytes > 96 * 1024) gpb >>= 1;
  const bool staged = g_tree_staging == 0 && (size_t)gpb * stage_bytes <= kMaxStageSmem;
  if (!staged) gpb = kThreads / 32;
  const int grid = (t->num_games + gpb - 1) / gpb;
  if (staged) {
    int rc = set_smem_attr_w32_once<true, APL>();
    if (rc) return rc;
    cudaError_t e = mz_launch(tree_step_w32_kernel<true, APL>, dim3(grid), dim3(gpb * 32),
                              (size_t)gpb * stage_bytes + sizeof(uint64_t) * gpb, (cudaStream_t)stream,
                              do_backup != 0, *t, sim, do_backup, do_select, live_nodes, stage_bytes, value,
                              reward, logits, new_hidden, gathered_hidden, tp, ta, td);
    if (e != cudaSuccess) return (int)e;
  } else {  // tree too large for shared memory: run on the global block directly
    cudaError_t e = mz_launch(tree_step_w32_kernel<false, APL>, dim3(grid), dim3(gpb * 32), 0,
                              (cudaStream_t)stream, do_backup != 0, *t, sim, do_backup, do_select,
                              live_nodes, 0, value, reward, logits, new_hidden, gathered_hidden, tp, ta, td);
    if (e != cudaSuccess) return (int)e;
  }
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int launch_step(const mz_tree* t, int sim, int live_nodes, int do_backup, int do_select, const float* value,
                const float* reward, const float* logits, const uint32_t* new_hidden,
                uint32_t* gathered_hidden, int32_t* tp, int32_t* ta, int32_t* td, void* stream) {
  // One warp per game at every action count.  Packing 8 / 4 / 2 games of few actions into a warp makes the games
  // of a warp wait for each other's descents, and the code is not warp-uniform.  Measured (A = 4, 50 simulations):
  // the converged warp-per-game kernel is faster at every batch size -- 13.9 vs 32.0 us per step at 4096 games,
  // 27.8 vs 44.5 us at 16 k, 83 vs 122 us at 64 k.  More than 32 actions: two per lane.
  return t->num_actions > 32
             ? launch_step_apl<2>(t, sim, live_nodes, do_backup, do_select, value, reward, logits, new_hidden,
                                  gathered_hidden, tp, ta, td, stream)
             : launch_step_apl<1>(t, sim, live_nodes, do_backup, do_select, value, reward, logits, new_hidden,
                                  gathered_hidden, tp, ta, td, stream);
}

}  // namespace

extern "C" {

int32_t mz_tree_node_bytes(int32_t A) { return (MZ_NODE_STATS_BYTES + 10 * A + 15) / 16 * 16; }

int64_t mz_tree_game_bytes(int32_t S, int32_t A) {
  int64_t b = MZ_GAME_HEADER_BYTES + (int64_t)(S + 1) * mz_tree_node_bytes(A);
  return (b + 127) / 128 * 128;
}

int mz_fill_pb_c_table(int32_t S, double pb_c_base, double pb_c_init, double* h_table) {
  if (S < 1 || !h_table) return MZ_ERR_BAD_ARG;
  const int SP1 = S + 1;
  for (int N = 0; N < SP1; ++N) {
    // mcts.py:116: math.log((N + base + 1) / base) + init   (host libm log, like CPython)
    volatile double ratio = ((double)N + pb_c_base + 1.0) / pb_c_base;
    volatile double pb_c = log(ratio) + pb_c_init;
    volatile double sq = sqrt((double)N);
    for (int n = 0; n < SP1; ++n) {
      volatile double f = sq / (double)(n + 1);  // mcts.py:117
      volatile double v = pb_c * f;
      h_table[(size_t)N * SP1 + n] = v;
    }
  }
  return MZ_OK;
}

int mz_tree_set_root(const mz_tree* t, const float* root_logits, const uint32_t* legal_mask,
                     const double* noise, double noise_frac, const int8_t* root_to_play,
                     const uint32_t* root_hidden, void* stream) {
  int rc = check_tree(t);
  if (rc) return rc;
  if (!root_logits) return MZ_ERR_BAD_ARG;
  const int grid = (t->num_games + 3) / 4;  // a warp per game
  if (t->num_actions > 32)
    set_root_kernel<2><<<grid, kThreads, 0, (cudaStream_t)stream>>>(*t, root_logits, legal_mask, noise, noise_frac,
                                                                  root_to_play, root_hidden, nullptr);
  else
    set_root_kernel<1><<<grid, kThreads, 0, (cudaStream_t)stream>>>(*t, root_logits, legal_mask, noise, noise_frac,
                                                                  root_to_play, root_hidden, nullptr);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_tree_set_root_priors(const mz_tree* t, const double* root_priors, const uint32_t* legal_mask,
                            const int8_t* root_to_play, const uint32_t* root_hidden, void* stream) {
  int rc = check_tree(t);
  if (rc) return rc;
  if (!root_priors) return MZ_ERR_BAD_ARG;
  const int grid = (t->num_games + 3) / 4;  // a warp per game
  if (t->num_actions > 32)
    set_root_kernel<2><<<grid, kThreads, 0, (cudaStream_t)stream>>>(*t, nullptr, legal_mask, nullptr, 0.0, root_to_play,
                                                                  root_hidden, root_priors);
  else
    set_root_kernel<1><<<grid, kThreads, 0, (cudaStream_t)stream>>>(*t, nullptr, legal_mask, nullptr, 0.0, root_to_play,
                                                                  root_hidden, root_priors);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_tree_select(const mz_tree* t, int32_t sim, uint32_t* gathered_hidden, int32_t* trace_parent,
                   int32_t* trace_action, int32_t* trace_depth, void* stream) {
  int rc = check_tree(t);
  if (rc) return rc;
  if (sim < 0 || sim >= t->num_simulations) return MZ_ERR_BAD_ARG;
  return launch_step(t, sim, sim + 1, 0, 1, nullptr, nullptr, nullptr, nullptr, gathered_hidden,
                     trace_parent, trace_action, trace_depth, stream);
}

int mz_tree_expand_backup(const mz_tree* t, int32_t sim, const float* value, const float* reward,
                          const float* logits, const uint32_t* new_hidden, void* stream) {
  int rc = check_tree(t);
  if (rc) return rc;
  if (sim < 0 || sim >= t->num_simulations || !value || !reward || !logits) return MZ_ERR_BAD_ARG;
  return launch_step(t, sim, sim + 1, 1, 0, value, reward, logits, new_hidden, nullptr, nullptr,
                     nullptr, nullptr, stream);
}

int mz_tree_step(const mz_tree* t, int32_t sim, const float* value, const float* reward,
                 const float* logits, const uint32_t* new_hidden, uint32_t* gathered_hidden,
                 int32_t* trace_parent, int32_t* trace_action, int32_t* trace_depth, void* stream) {
  int rc = check_tree(t);
  if (rc) return rc;
  if (sim < -1 || sim >= t->num_simulations) return MZ_ERR_BAD_ARG;
  const int do_backup = sim >= 0, do_select = sim + 1 < t->num_simulations;
  if (do_backup && (!value || !reward || !logits)) return MZ_ERR_BAD_ARG;
  return launch_step(t, sim, sim + 1 < 1 ? 1 : sim + 1, do_backup, do_select, value, reward, logits,
                     new_hidden, gathered_hidden, trace_parent, trace_action, trace_depth, stream);
}

int mz_tree_root_stats(const mz_tree* t, int32_t* visits, double* child_visits, double* root_value,
                       double* minmax, void* stream) {
  int rc = check_tree(t);
  if (rc) return rc;
  const int threads = 128, grid = (t->num_games + 3) / 4;  // a warp per game
  if (t->num_actions > 32)
    root_stats_kernel<2><<<grid, threads, 0, (cudaStream_t)stream>>>(*t, visits, child_visits, root_value, minmax);
  else
    root_stats_kernel<1><<<grid, threads, 0, (cudaStream_t)stream>>>(*t, visits, child_visits, root_value, minmax);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_select_action(int32_t G, int32_t A, const int32_t* visits, const uint32_t* legal_mask,
                     const double* temperature, const double* uniforms, int32_t* actions,
                     void* stream) {
  if (G < 1 || A < 1 || A > MZ_MAX_ACTIONS || !visits || !temperature || !uniforms || !actions)
    return MZ_ERR_BAD_ARG;
  const int threads = 128, grid = (G + 3) / 4;  // a warp per game
  if (A > 32)
    select_action_kernel<2><<<grid, threads, 0, (cudaStream_t)stream>>>(G, A, visits, legal_mask, temperature,
                                                                       uniforms, actions);
  else
    select_action_kernel<1><<<grid, threads, 0, (cudaStream_t)stream>>>(G, A, visits, legal_mask, temperature,
                                                                       uniforms, actions);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_tree_export(const mz_tree* t, int32_t game, double* prior, int32_t* child, double* vsum,
                   int32_t* visit, float* reward, void* stream) {
  int rc = check_tree(t);
  if (rc) return rc;
  if (game < 0 || game >= t->num_games) return MZ_ERR_BAD_ARG;
  tree_export_kernel<<<4, 128, 0, (cudaStream_t)stream>>>(*t, game, prior, child, vsum, visit, reward);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_exp_f32(int64_t n, const float* x, double* out, void* stream) {
  if (n < 0 || (n > 0 && (!x || !out))) return MZ_ERR_BAD_ARG;
  if (n == 0) return MZ_OK;
  exp_f32_kernel<<<148 * 8, 256, 0, (cudaStream_t)stream>>>(n, x, out);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_debug_div_check(uint64_t seed, int32_t blocks, int32_t per_thread, uint64_t* mismatches,
                       uint64_t* tested, void* stream) {
  if (blocks < 1 || per_thread < 1 || !mismatches || !tested) return MZ_ERR_BAD_ARG;
  div_check_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
      seed, per_thread, (unsigned long long*)mismatches, (unsigned long long*)tested);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_tree_set_games_per_block(int32_t games) {
  if (games != 0 && games != 1 && games != 2 && games != 4) return MZ_ERR_BAD_ARG;
  g_w32_gpb = games;
  return MZ_OK;
}

int mz_debug_set_tree_staging(int32_t mode) {
  if (mode != 0 && mode != 1) return MZ_ERR_BAD_ARG;
  g_tree_staging = mode;
  return MZ_OK;
}

int mz_set_programmatic_launch(int32_t enable) {
  g_mz_pdl = enable ? 1 : 0;
  return MZ_OK;
}

const char* mz_version(void) { return "mzb200 0.1.0 (sm_100a)"; }
int32_t mz_compiled_arch(void) { return 100; }

}  // extern "C"
