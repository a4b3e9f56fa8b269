// Tree engine of the persistent search kernel (mz_fcsearch.cu): sparse and node-parallel.
//
// What bounds the search is the length of ONE game's dependent instruction stream per simulation (a warp
// issues ~1 dependent instruction per 10 cycles), so this engine shortens that stream instead of packing
// more games per warp:
//
//  * select_child (mcts.py:104-113) only has to rank the EXPANDED children of a node plus its best
//    unexpanded child: every unexpanded child scores pb_c(N, 0) * prior + init_value_score, monotone in the
//    prior, so with the priors' maximum known the others cannot win.  (Exactness: the reference breaks score
//    ties towards the larger action.  The stand-in is the largest action among the maximal priors; a smaller
//    prior could only tie after rounding if it lies within 2^-50 relative of the maximum -- such nodes, and
//    every node when init_value_score != 0, are flagged at expansion and ranked densely over all actions.)
//  * the argmax of EVERY expanded node is evaluated each simulation, all nodes in parallel over the eight
//    lanes of a game (two items per node: its best unexpanded child and the edge that leads to it); the
//    descent (mcts.py:87-92) is then a pointer chase through the per-node winners in shared memory --
//    a handful of instructions per level instead of a full score evaluation per level.
//
// Arithmetic per score is the one of mz_tree.cu (IEEE binary64, reference operation order);
// results are bit-identical (tests/test_gpu_fcnet.py::test_fused_search_equals_per_launch_search).
//
// Per-game block in global memory (L2):   S1 = round_up(S + 1, 2) node slots, A2 = round_up(A, 2)
//   header 64 B : f64 min | f64 max
//   own[n]  16 B: f64 value_sum | f32 reward | u32 -
//   edge[n] 32 B: f64 prior of the edge parent(n) -> n | f64 q(n) = reward -/+ discount * value()
//                 | f64 utop(n) = prior of the best unexpanded child of n | -    (one record: an item of the
//                 ranking pass reads 16 bytes at offset 0 (edge) or 16 (best unexpanded child), branch free)
//   meta[n]  8 B: copy of the shared-memory node words at the end of the move (export / tests)
//   pri[n][A2]  : all priors of node n (Node.expand, mcts.py:52-55; the root's include the Dirichlet noise)
// Per-game shared memory: node word  N | action << 8 | uact << 16 | parent << 24 (visit count, action from the
// parent, best unexpanded action with bit 6 = rank densely, 0xff = none, parent id), mask of actions that are not
// unexpanded children (expanded or illegal), and the per-node winners of the current simulation.
#pragma once

namespace fs2 {

constexpr int L = 8;               // lanes per game
constexpr int MAX_S = 63;          // items per lane: ceil((2 S + 1) / 8) <= 16
constexpr int MAX_ITEMS = 16;
constexpr int UACT_NONE = 0xff, UACT_DENSE = 0x40;

struct Smem {
  float* logit;        // [GP][A4]
  float* val;          // [GP]
  float* rew;          // [GP]
  double* mm;          // [GP][2]
  double* sp;          // [GP][row] exp(logit) / signed-reward scratch.  It shares each game's row with best_key
                       //           (the two are used in different phases of the SAME game; rows of different games
                       //           never overlap, so warps in different phases cannot disturb each other)
  unsigned long long* best_key;  // [GP][row]: the order-preserving score key of the edge into every node
  uint16_t* best_ca;   // [GP][S1]  winner of select_child per node: (action << 8) | child id (0xff: unexpanded)
  uint8_t* first;      // [GP][S1]  first expanded child of a node (0 = none: the root is nobody's child)
  uint8_t* next;       // [GP][S1]  next expanded child of the same parent
  uint32_t* node;      // [GP][S1]  N | action << 8 | uact << 16
  uint32_t* xmask;     // [GP][S1]
  uint8_t* path_n;     // [GP][PS]
  uint8_t* path_a;     // [GP][PS]
  uint8_t* depth;      // [GP]
  const unsigned long long* exp_tab;
  const double* rcp;   // [64] correctly rounded reciprocals of the visit counts 1..63
  const double* pbc0;  // [64] pb_c[N][0]: the exploration factor of an unvisited child of a node with N visits
  int ps, a4, s1, row;  // row = doubles per game of the shared scratch row = max(S1, SP_STRIDE)
};

struct Game {
  bool valid;
  int g, gl, sub;
  uint8_t* base;
};

struct Geo {  // byte offsets inside a game block
  int own, edge, utop, meta, pri, a2, s1;
  long long bytes;
};
__host__ __device__ inline Geo geo(int S, int A) {
  Geo g;
  g.s1 = (S + 2) & ~1;
  g.a2 = (A + 1) & ~1;
  g.own = 64;
  g.edge = g.own + 16 * g.s1;   // 32-byte records: {prior of the edge into n, q(n), best unexpanded prior of n, -}
  g.utop = g.edge + 16;         // (same records, third double)
  g.meta = g.edge + 32 * g.s1;
  g.pri = g.meta + 8 * g.s1;
  g.bytes = ((long long)g.pri + (long long)g.s1 * 8 * g.a2 + 127) / 128 * 128;
  return g;
}

MZ_DEV double shfl8_xor_f64(double v, int m) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_xor_sync(MZ_FULL, lo, m, L);
  hi = __shfl_xor_sync(MZ_FULL, hi, m, L);
  return __hiloint2double(hi, lo);
}
MZ_DEV unsigned long long sortable(double x) {  // monotone map double -> u64 (no NaNs); > 0 for every finite x
  const unsigned long long b = (unsigned long long)__double_as_longlong(x);
  return b ^ ((unsigned long long)((long long)b >> 63) | 0x8000000000000000ull);
}

// Best unexpanded child over the priors this lane holds (pv[t] = prior of action 8 t + sub, available iff its
// bit is clear in `xmask`): returns across the eight lanes the maximal prior, the largest action that has it,
// and whether another available child with a LARGER action lies within 2^-50 relative below the maximum (then
// a rounded product could tie and the reference's tie-break would prefer it: the node is ranked densely).
// NS independent sets are reduced side by side (the shuffles of one overlap the compares of the other).
template <int AL, int NS>
MZ_DEV void top_unexpanded(const double (&pv)[NS][AL], const uint32_t (&xmask)[NS], int A, int sub, bool force_dense,
                           double (&ptop)[NS], int (&uact)[NS]) {
  double bp[NS];
  int ba[NS];
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    bp[s] = -1.0;
    ba[s] = -1;
#pragma unroll
    for (int t = 0; t < AL; ++t) {
      const int a = L * t + sub;
      if (a < A && !((xmask[s] >> a) & 1u) && pv[s][t] >= bp[s]) {  // ascending actions: >= keeps the larger one
        bp[s] = pv[s][t];
        ba[s] = a;
      }
    }
  }
#pragma unroll
  for (int m = 1; m < L; m <<= 1) {
    double op[NS];
    int oa[NS];
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      op[s] = shfl8_xor_f64(bp[s], m);
      oa[s] = __shfl_xor_sync(MZ_FULL, ba[s], m, L);
    }
#pragma unroll
    for (int s = 0; s < NS; ++s) {
      const bool take = oa[s] >= 0 && (ba[s] < 0 || op[s] > bp[s] || (op[s] == bp[s] && oa[s] > ba[s]));
      bp[s] = take ? op[s] : bp[s];
      ba[s] = take ? oa[s] : ba[s];
    }
  }
  const unsigned lane = threadIdx.x & 31u;
  const unsigned gmask = 0xffu << (lane & ~7u);
#pragma unroll
  for (int s = 0; s < NS; ++s) {
    bool close = false;
    const double thr = __dmul_rn(bp[s], 1.0 - 0x1p-50);
#pragma unroll
    for (int t = 0; t < AL; ++t) {
      const int a = L * t + sub;
      close = close || (ba[s] >= 0 && a < A && !((xmask[s] >> a) & 1u) && a > ba[s] && pv[s][t] < bp[s] && pv[s][t] >= thr);
    }
    const bool any_close = (__ballot_sync(MZ_FULL, close) & gmask) != 0u;
    ptop[s] = bp[s];
    uact[s] = ba[s] < 0 ? UACT_NONE : (ba[s] | ((any_close || force_dense || bp[s] < 0x1p-900) ? UACT_DENSE : 0));
  }
}

// Node.expand priors (mcts.py:52-55) for the eight lanes of a game: p_a = exp(logit_a) / sum over the legal actions
// in ascending order, the sum evaluated like CPython's builtin sum() (prior_sum_mode 1: Neumaier).  Every lane
// returns the sum; pexp[t] holds exp(logit) of action 8 t + sub (0 where illegal / absent).
template <int AL>
MZ_DEV double prior_sum(const FsParams& p, const Smem& sm, const Game& gm, const float* logits, uint32_t legal_bits,
                        double (&pexp)[AL]) {
  const int A = p.A;
  double* sp = sm.sp + gm.gl * sm.row;
#pragma unroll
  for (int t = 0; t < AL; ++t) {
    const int a = L * t + gm.sub;
    double e = 0.0;
    if (a < A && ((legal_bits >> a) & 1u)) e = fs_exp((double)logits[a], sm.exp_tab);
    pexp[t] = e;
    if (a < A) sp[a] = e;
  }
  __syncwarp();
  double f = 0.0, c = 0.0;
  bool first = true;
#pragma unroll 1
  for (int a = 0; a < A; ++a) {
    if (!((legal_bits >> a) & 1u)) continue;
    const double x = sp[a];
    if (first) {
      f = x;  // int 0 + x
      first = false;
    } else if (p.prior_sum_mode == 0) {
      f = __dadd_rn(f, x);
    } else {  // Neumaier step, CPython >= 3.12 Python/bltinmodule.c
      const double s = __dadd_rn(f, x);
      const bool big = fabs(f) >= fabs(x);
      const double hi = big ? f : x, lo = big ? x : f;
      c = __dadd_rn(c, __dadd_rn(__dsub_rn(hi, s), lo));
      f = s;
    }
  }
  if (p.prior_sum_mode != 0 && c != 0.0 && isfinite(c)) f = __dadd_rn(f, c);
  __syncwarp();
  return f;
}

template <int AL>
MZ_DEV void set_root(const FsParams& p, const Smem& sm, const Game& gm, const Geo& G) {
  const int A = p.A;
  uint32_t lm = 0u;
  if (gm.valid) {
    lm = p.legal ? p.legal[gm.g] : 0xffffffffu;
    if (A < 32) lm &= (1u << A) - 1u;
  }
  double pexp[AL];
  const double f = prior_sum<AL>(p, sm, gm, p.root_logits + (size_t)(gm.valid ? gm.g : 0) * A, lm, pexp);
  double pv[AL];
#pragma unroll
  for (int t = 0; t < AL; ++t) {
    const int a = L * t + gm.sub;
    const bool legal = a < A && ((lm >> a) & 1u);
    double prior = legal ? __ddiv_rn(pexp[t], f) : 0.0;
    if (p.noise && legal) {  // noise is dense over the root's children in action order (mcts.py:57-61)
      const int j = __popc(lm & ((1u << a) - 1u));
      const double nz = p.noise[(size_t)gm.g * A + j];
      prior = __dadd_rn(__dmul_rn(prior, __dsub_rn(1.0, p.noise_frac)), __dmul_rn(nz, p.noise_frac));
    }
    pv[t] = prior;
    if (gm.valid && a < A) *reinterpret_cast<double*>(gm.base + G.pri + 8 * a) = prior;
  }
  double pvs[1][AL], ptops[1];
  int uacts[1];
#pragma unroll
  for (int t = 0; t < AL; ++t) pvs[0][t] = pv[t];
  const uint32_t xms[1] = {~lm};
  top_unexpanded<AL, 1>(pvs, xms, A, gm.sub, p.init_score != 0.0, ptops, uacts);
  const double ptop = ptops[0];
  const int uact = uacts[0];
  if (gm.valid && gm.sub == 0) {
    sm.node[gm.gl * sm.s1] = 0u | (0xffu << 8) | ((uint32_t)uact << 16);
    sm.first[gm.gl * sm.s1] = 0;
    sm.xmask[gm.gl * sm.s1] = ~lm;
    sm.mm[2 * gm.gl] = p.min_bound;
    sm.mm[2 * gm.gl + 1] = p.max_bound;
    *reinterpret_cast<uint4*>(gm.base + G.own) = make_uint4(0u, 0u, 0u, 0u);
    *reinterpret_cast<double*>(gm.base + G.utop) = ptop;
  }
  if (!gm.valid) return;
  // hidden state of the root: float32 [50] -> bf16 [64] (zero padded), pool slot 0: one 16-byte block per lane
  const float* h = p.root_hidden + (size_t)gm.g * H;
  __nv_bfloat16* row = p.pool + (size_t)gm.g * (p.S + 1) * POOL_ROW;
  uint32_t w[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int k = 8 * gm.sub + 2 * j;
    w[j] = pack_bf16(k < H ? h[k] : 0.0f, k + 1 < H ? h[k + 1] : 0.0f);
  }
  *reinterpret_cast<uint4*>(row + 8 * gm.sub) = make_uint4(w[0], w[1], w[2], w[3]);
}

// phase stamps of the instrumented instantiation (TL: FsParams::timeline set); the production one has none, so
// no stamp splits its code into separate basic blocks
#define FS2_STAMP(slot_)                    \
  do {                                      \
    if constexpr (TL) {                     \
      if (tl) tl[(slot_)] = clock64();      \
    }                                       \
  } while (0)

// ------------------------------------------------------------------------------------------------------
// descent = [rank every expanded node's candidates in parallel] + [pointer chase from the root]
//
// Items of simulation `sim` (nodes 0..sim exist): i <= sim -> "U": the best unexpanded child of node i;
// i > sim -> "E": the edge into node j = i - sim.  Lane `sub` of a game owns items sub, sub + 8, ...  The item
// arithmetic is straight-line (no per-item branches), four items per basic block, so that the independent
// dependency chains of a lane's items overlap; the rare cases (a node flagged for dense ranking, a MinMax
// range outside the fast-division guard) are redone exactly in a second pass under a warp vote.
// The per-parent maximum over (score, action) runs on native 32-bit shared-memory atomics: high words of the
// order-preserving keys, then low words among the items that reached the high maximum, then actions.
// ------------------------------------------------------------------------------------------------------
struct Norm {  // MinMaxStats.normalize (mcts.py:16-21) hoisted per game
  int mode;    // 2: (v - min) / (max - min) through the reciprocal, 3: IEEE division, 1: constant 1.0, 0: raw
  double mn, d, r;
};
MZ_DEV Norm make_norm(double mn, double mx) {
  Norm n;
  n.mn = mn;
  n.d = __dsub_rn(mx, mn);
  n.r = 0.0;
  n.mode = 0;
  if (mx > mn) {
    if (fs_divisor_ok(n.d)) {
      n.mode = 2;
      n.r = __drcp_rn(n.d);
    } else {
      n.mode = 3;
    }
  } else if (mx == mn) {
    n.mode = 1;
  }
  return n;
}

template <bool TL>
MZ_DEV void descend(const FsParams& p, const Smem& sm, const Game& gm, const Geo& G, int sim, int& out_parent,
                    int& out_action, long long* tl) {
  const int A = p.A, SP1 = p.S + 1;
  const double init_score = p.init_score;
  const Norm nm = make_norm(sm.mm[2 * gm.gl], sm.mm[2 * gm.gl + 1]);
  uint32_t* node = sm.node + gm.gl * sm.s1;
  const uint32_t* xmask = sm.xmask + gm.gl * sm.s1;
  unsigned long long* ekey = sm.best_key + gm.gl * sm.row;
  uint16_t* best_ca = sm.best_ca + gm.gl * sm.s1;
  const uint8_t* first = sm.first + gm.gl * sm.s1;
  const uint8_t* next = sm.next + gm.gl * sm.s1;
  FS2_STAMP(16);
  // Items: slot t of a lane is node n = 8 t + sub.  [0, NT): "U" = the best unexpanded child of node n (n <= sim);
  // [NT, 2 NT): "E" = the edge into node n (1 <= n <= sim), ranked under its parent.
  constexpr int NT = MAX_ITEMS / 2;
  uint32_t key_hi[MAX_ITEMS], key_lo[MAX_ITEMS], pack[MAX_ITEMS];  // pack: valid << 31 | slow << 30 | parent << 16 | action << 8 | child
  bool any_slow = false;
  const bool fast_norm = __all_sync(MZ_FULL, nm.mode == 2 || !gm.valid);  // the usual case: every game normalises
  // ---- loads: edges first (two dependent shared-memory reads ahead of them), then the unexpanded-child priors ----
  double2 ed[NT];
  double pbc[NT], ut[NT];
  uint32_t we[NT], wu[NT];
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    const int n = L * t + gm.sub;
    ed[t] = make_double2(0.0, 0.0);
    pbc[t] = 0.0;
    we[t] = 0u;
    if (L * t > sim) continue;  // warp uniform
    const bool act = gm.valid && n >= 1 && n <= sim;
    we[t] = node[act ? n : 0];
    const int np_ = (int)(node[we[t] >> 24] & 0xffu), nj = (int)(we[t] & 0xffu);
    // a lane without an edge (a game beyond num_games in the last tile, node 0) reads shared memory nobody
    // initialised: keep its table index inside pb_c
    pbc[t] = __ldg(p.pb_c + (act ? (size_t)np_ * SP1 + nj : (size_t)0));
    ed[t] = *reinterpret_cast<const double2*>(gm.base + G.edge + 32 * (act ? n : 0));
  }
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    const int n = L * t + gm.sub;
    ut[t] = 0.0;
    wu[t] = 0u;
    if (L * t > sim) continue;
    const bool act = gm.valid && n <= sim;
    wu[t] = node[act ? n : 0];
    ut[t] = *reinterpret_cast<const double*>(gm.base + G.utop + 32 * (act ? n : 0));
  }
  // ---- scores of the unexpanded-child items: pb_c(N, 0) * prior + init_value_score (mcts.py:115-124) ----
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    const int n = L * t + gm.sub;
    key_hi[t] = key_lo[t] = pack[t] = 0u;
    if (L * t > sim) continue;
    const int ua = (int)((wu[t] >> 16) & 0xffu);
    const bool live = gm.valid && n <= sim && ua != UACT_NONE;
    double score = __dadd_rn(__dmul_rn(sm.pbc0[wu[t] & 0x3fu], ut[t]), init_score);
    if (sim == 0) score = ut[t];  // mcts.py:105-108: the unvisited root ranks its children by prior
    const bool slow = (ua & UACT_DENSE) != 0;
    any_slow = any_slow || (live && slow);
    const unsigned long long k = sortable(score);
    key_hi[t] = (uint32_t)(k >> 32);
    key_lo[t] = (uint32_t)k;
    pack[t] = live ? (0x80000000u | (slow ? 0x40000000u : 0u) | ((uint32_t)n << 16) | ((uint32_t)(ua & 0x3f) << 8) | 0xffu) : 0u;
  }
  // ---- scores of the edges: pb_c(N_parent, n) * prior + normalize(q) ----
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    const int n = L * t + gm.sub;
    const int it = NT + t;
    key_hi[it] = key_lo[it] = pack[it] = 0u;
    if (L * t > sim) continue;
    const bool live = gm.valid && n >= 1 && n <= sim;
    const double q = ed[t].y;
    const double x = __dsub_rn(q, nm.mn);
    double vs = fs_div_by_const(x, nm.d, nm.r);  // exact for x == 0 too
    const unsigned hx = (unsigned)__double2hiint(x);
    bool slow = x != 0.0 && hx - 0x33700000u > 0x19000000u;
    if (!fast_norm) {  // warp uniform
      slow = nm.mode == 3 || (nm.mode == 2 && slow);
      vs = nm.mode == 1 ? 1.0 : (nm.mode == 0 ? q : vs);
    }
    const double score = __dadd_rn(__dmul_rn(pbc[t], ed[t].x), vs);
    any_slow = any_slow || (live && slow);
    const unsigned long long k = sortable(score);
    key_hi[it] = (uint32_t)(k >> 32);
    key_lo[it] = (uint32_t)k;
    pack[it] = live ? (0x80000000u | (slow ? 0x40000000u : 0u) | ((we[t] >> 24) << 16) | (((we[t] >> 8) & 0xffu) << 8) | (uint32_t)n) : 0u;
  }
  FS2_STAMP(17);
  if (__any_sync(MZ_FULL, any_slow)) {
    // exact redo of the flagged items: IEEE division for the value term, dense ranking of a flagged node
#pragma unroll
    for (int it = 0; it < MAX_ITEMS; ++it) {  // unrolled: the item arrays must stay in registers
      if (!(pack[it] & 0x40000000u)) continue;
      const int n = L * (it < NT ? it : it - NT) + gm.sub;
      const int pn = (int)((pack[it] >> 16) & 0xffu);
      double score;
      uint32_t action = (pack[it] >> 8) & 0xffu;
      if (it < NT) {
        const int N = (int)(node[n] & 0xffu);
        const double pb_c = sm.pbc0[N & 0x3f];
        const uint32_t xm = xmask[n];
        bool have = false;
        score = 0.0;
        for (int a = 0; a < A; ++a) {
          if ((xm >> a) & 1u) continue;
          const double pr = *reinterpret_cast<const double*>(gm.base + G.pri + ((size_t)n * G.a2 + a) * 8);
          const double sc = sim == 0 ? pr : __dadd_rn(__dmul_rn(pb_c, pr), init_score);
          if (!have || sc >= score) {
            score = sc;
            action = (uint32_t)a;
            have = true;
          }
        }
      } else {
        const double2 e = *reinterpret_cast<const double2*>(gm.base + G.edge + 32 * n);
        const double pb_c = __ldg(p.pb_c + (size_t)(node[pn] & 0xffu) * SP1 + (node[n] & 0xffu));
        const double x = __dsub_rn(e.y, nm.mn);
        const double vs = (nm.mode == 2 && x == 0.0) ? 0.0 : __ddiv_rn(x, nm.d);
        score = __dadd_rn(__dmul_rn(pb_c, e.x), vs);
      }
      const unsigned long long k = sortable(score);
      key_hi[it] = (uint32_t)(k >> 32);
      key_lo[it] = (uint32_t)k;
      pack[it] = (pack[it] & 0xffff00ffu) | (action << 8);
    }
  }
  // ---- select_child per node: max over (score, action), ties -> larger action (mcts.py:106-112) ----
  // edge keys go to shared memory, indexed by the child node
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    const int n = L * t + gm.sub;
    if (L * t > sim) continue;
    if (pack[NT + t]) ekey[n] = ((unsigned long long)key_hi[NT + t] << 32) | key_lo[NT + t];
  }
  __syncwarp();
  FS2_STAMP(18);
  // the root (many children): every lane ranks the root's edges it owns, lane 0 adds the root's best unexpanded
  // child, then a butterfly over the eight lanes
  {
    unsigned long long bk = 0ull;
    int bac = -1;  // (action << 8) | child
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      if (L * t > sim) continue;
      const uint32_t pk = pack[NT + t];
      if (pk && ((pk >> 16) & 0xffu) == 0u) {
        const unsigned long long k = ((unsigned long long)key_hi[NT + t] << 32) | key_lo[NT + t];
        const int ac = (int)(pk & 0xffffu);
        if (k > bk || (k == bk && ac > bac)) {
          bk = k;
          bac = ac;
        }
      }
    }
    if (gm.sub == 0 && pack[0]) {
      const unsigned long long k = ((unsigned long long)key_hi[0] << 32) | key_lo[0];
      const int ac = (int)(pack[0] & 0xffffu);
      if (k > bk || (k == bk && ac > bac)) {
        bk = k;
        bac = ac;
      }
    }
#pragma unroll
    for (int m = 1; m < L; m <<= 1) {
      const uint32_t ohi = __shfl_xor_sync(MZ_FULL, (uint32_t)(bk >> 32), m, L);
      const uint32_t olo = __shfl_xor_sync(MZ_FULL, (uint32_t)bk, m, L);
      const int oac = __shfl_xor_sync(MZ_FULL, bac, m, L);
      const unsigned long long ok = ((unsigned long long)ohi << 32) | olo;
      if (ok > bk || (ok == bk && oac > bac)) {
        bk = ok;
        bac = oac;
      }
    }
    if (gm.valid && gm.sub == 0) best_ca[0] = (uint16_t)bac;
  }
  // every other node: its owner lane walks the list of its expanded children
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    const int n = L * t + gm.sub;
    if (L * t > sim) continue;
    const bool act = gm.valid && n >= 1 && n <= sim;
    unsigned long long bk = pack[t] ? (((unsigned long long)key_hi[t] << 32) | key_lo[t]) : 0ull;
    int bac = pack[t] ? (int)(pack[t] & 0xffffu) : -1;
    int c = act ? (int)first[n] : 0;
    while (__any_sync(MZ_FULL, c != 0)) {
      if (c != 0) {
        const unsigned long long k = ekey[c];
        const int ac = (int)(((node[c] >> 8) & 0xffu) << 8) | c;
        const int nx = (int)next[c];
        if (k > bk || (k == bk && ac > bac)) {
          bk = k;
          bac = ac;
        }
        c = nx;
      }
    }
    if (act) best_ca[n] = (uint16_t)bac;
  }
  __syncwarp();
  FS2_STAMP(19);
  // ---- pointer chase: while node.expanded(): node = the winner of select_child (mcts.py:87-92) ----
  uint8_t* pn_ = sm.path_n + gm.gl * sm.ps;
  uint8_t* pa_ = sm.path_a + gm.gl * sm.ps;
  int cur = 0, depth = 0, parent = 0, action = 0;
  bool done = !gm.valid;
  if (gm.valid && gm.sub == 0) pn_[0] = 0;
  for (;;) {
#pragma unroll
    for (int rep = 0; rep < 2; ++rep) {  // finished games idle through the extra level
      const uint32_t ca = (uint32_t)best_ca[cur];
      const int a = (int)(ca >> 8), c = (int)(ca & 0xffu);
      if (!done && gm.sub == 0) {
        pa_[depth] = (uint8_t)a;
        pn_[depth + 1] = (uint8_t)c;  // 0xff after the leaf: never read (positions <= depth only)
      }
      const bool leaf = c == 0xff;
      parent = done ? parent : cur;
      action = done ? action : a;
      depth += done ? 0 : 1;
      cur = (done || leaf) ? cur : c;
      done = done || leaf;
    }
    if (!__any_sync(MZ_FULL, !done)) break;
  }
  FS2_STAMP(20);
  if (gm.valid && gm.sub == 0) {
    sm.depth[gm.gl] = (uint8_t)depth;
    if (p.trace_parent) p.trace_parent[(size_t)sim * p.G + gm.g] = parent;
    if (p.trace_action) p.trace_action[(size_t)sim * p.G + gm.g] = action;
    if (p.trace_depth) p.trace_depth[(size_t)sim * p.G + gm.g] = depth;
  }
  out_parent = parent;
  out_action = action;
}

// exp for arguments inside the table algorithm's range (every finite logit of a network); `bad` reports the rest
MZ_DEV double exp_fast(double x, const unsigned long long* tab, bool& bad) {
  const double ax = fabs(x);
  bad = !(ax >= 0x1p-54 && ax < 512.0);
  const double InvLn2N = 0x1.71547652b82fep7, Shift = 0x1.8p52;
  const double NegLn2hiN = -0x1.62e42fefa0000p-8, NegLn2loN = -0x1.cf79abc9e3b3ap-47;
  const double C2 = 0x1.ffffffffffdbdp-2, C3 = 0x1.555555555543cp-3;
  const double C4 = 0x1.55555cf172b91p-5, C5 = 0x1.1111167a4d017p-7;
  const double z = __dmul_rn(InvLn2N, x);
  double kd = __dadd_rn(z, Shift);
  const unsigned long long ki = (unsigned long long)__double_as_longlong(kd);
  kd = __dsub_rn(kd, Shift);
  const double r = __fma_rn(kd, NegLn2loN, __fma_rn(kd, NegLn2hiN, x));
  const unsigned idx = 2u * ((unsigned)ki & 127u);
  const unsigned long long top = ki << 45;
  const double tail = __longlong_as_double((long long)tab[idx]);
  const unsigned long long sbits = tab[idx + 1] + top;
  const double r2 = __dmul_rn(r, r);
  const double a = __fma_rn(r, C3, C2), b = __fma_rn(r, C5, C4);
  const double tmp = __fma_rn(__dmul_rn(r2, r2), b, __fma_rn(r2, a, __dadd_rn(tail, r)));
  const double scale = __longlong_as_double((long long)sbits);
  return __fma_rn(scale, tmp, scale);
}

// ------------------------------------------------------------------------------------------------------
// expand (mcts.py:47-55) + backpropagate (mcts.py:126-143) of simulation `sim`
// ------------------------------------------------------------------------------------------------------
constexpr int MAXP = (MAX_S + 1 + L) / L;  // path positions per lane (depth <= S)

// What the expansion of a simulation can prepare BEFORE the network outputs arrive (the leaf is known since the
// descent): the path nodes' own records, the parent's next best unexpanded child and the prior of the new edge.
// Runs while the lane would otherwise wait for the prediction heads of the other CTAs.
struct Pre {
  uint4 own[MAXP];
  double ptop_par, edge_prior;
  int uact_par, depth, parent, action, dmax;
  uint32_t xm_par;
};

template <int AL>
MZ_DEV void pre_expand(const FsParams& p, const Smem& sm, const Game& gm, const Geo& G, Pre& pre) {
  const int A = p.A;
  const uint8_t* pn_ = sm.path_n + gm.gl * sm.ps;
  const uint8_t* pa_ = sm.path_a + gm.gl * sm.ps;
  const uint32_t* xmask = sm.xmask + gm.gl * sm.s1;
  const int depth = gm.valid ? (int)sm.depth[gm.gl] : 0;
  const int parent = gm.valid ? (int)pn_[depth - 1] : 0, action = gm.valid ? (int)pa_[depth - 1] : 0;
  int dmax = depth;
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) dmax = max(dmax, __shfl_xor_sync(MZ_FULL, dmax, m));
  double ppv[1][AL];
#pragma unroll
  for (int t = 0; t < AL; ++t) {
    const int a = L * t + gm.sub;
    ppv[0][t] = 0.0;
    if (gm.valid && a < A) ppv[0][t] = *reinterpret_cast<const double*>(gm.base + G.pri + ((size_t)parent * G.a2 + a) * 8);
  }
#pragma unroll
  for (int m = 0; m < MAXP; ++m) {
    const int kk = L * m + gm.sub;
    pre.own[m] = make_uint4(0u, 0u, 0u, 0u);
    if (L * m <= dmax && gm.valid && kk < depth) pre.own[m] = ldg16(gm.base + G.own + 16 * (int)pn_[kk]);
  }
  const uint32_t xm_par = gm.valid ? (xmask[parent] | (1u << action)) : 0xffffffffu;
  const uint32_t xms[1] = {xm_par};
  double ptops[1];
  int uacts[1];
  top_unexpanded<AL, 1>(ppv, xms, A, gm.sub, p.init_score != 0.0, ptops, uacts);
  // the prior of the new edge: the lane that holds the parent's prior of `action` hands it round
  double edge_prior = 0.0;
#pragma unroll
  for (int t = 0; t < AL; ++t) {
    const double v = __hiloint2double(__shfl_sync(MZ_FULL, __double2hiint(ppv[0][t]), action & (L - 1), L),
                                      __shfl_sync(MZ_FULL, __double2loint(ppv[0][t]), action & (L - 1), L));
    if (t == action / L) edge_prior = v;
  }
  pre.ptop_par = ptops[0];
  pre.uact_par = uacts[0];
  pre.edge_prior = edge_prior;
  pre.depth = depth;
  pre.parent = parent;
  pre.action = action;
  pre.dmax = dmax;
  pre.xm_par = xm_par;
}

template <bool TL, int AL>
MZ_DEV void expand_backup(const FsParams& p, const Smem& sm, const Game& gm, const Geo& G, int sim, const Pre& pre,
                          long long* tl) {
  const int A = p.A;
  const bool two = p.two_players != 0;
  const double disc = p.discount;
  const int newn = sim + 1;
  const float* logits = sm.logit + gm.gl * sm.a4;
  const float value_f = sm.val[gm.gl], reward_in = sm.rew[gm.gl];
  const float node_reward_new = (reward_in != 0.0f) ? reward_in : 0.0f;  // `if network_output.reward:`
  const uint8_t* pn_ = sm.path_n + gm.gl * sm.ps;
  uint32_t* node = sm.node + gm.gl * sm.s1;
  uint32_t* xmask = sm.xmask + gm.gl * sm.s1;
  const int depth = pre.depth, parent = pre.parent, action = pre.action, dmax = pre.dmax;
  const uint4 (&own)[MAXP] = pre.own;
  if (gm.valid) {
    if (gm.sub == 0) {
      if (p.rec_value) p.rec_value[(size_t)sim * p.G + gm.g] = value_f;
      if (p.rec_reward) p.rec_reward[(size_t)sim * p.G + gm.g] = reward_in;
    }
    if (p.rec_logits) {
#pragma unroll
      for (int t = 0; t < AL; ++t) {
        const int a = L * t + gm.sub;
        if (a < A) p.rec_logits[((size_t)sim * p.G + gm.g) * A + a] = logits[a];
      }
    }
  }
  FS2_STAMP(22);

  // ---- expand: priors of the new node (every action is legal below the root, mcts.py:72, 97):
  // p_a = exp(logit_a) / sum, the sum evaluated like CPython's builtin sum() over the actions in order ----
  double* sp = sm.sp + gm.gl * sm.row;
  double pexp[AL];
  bool bad = false;
#pragma unroll
  for (int t = 0; t < AL; ++t) {
    const int a = L * t + gm.sub;
    bool b1;
    pexp[t] = exp_fast((double)logits[a < A ? a : 0], sm.exp_tab, b1);
    bad = bad || (a < A && b1);
  }
  if (__any_sync(MZ_FULL, bad)) {  // a logit outside the table algorithm's range: the general routine
#pragma unroll
    for (int t = 0; t < AL; ++t) {
      const int a = L * t + gm.sub;
      if (a < A) pexp[t] = fs_exp((double)logits[a], sm.exp_tab);
    }
  }
#pragma unroll
  for (int t = 0; t < AL; ++t) {
    const int a = L * t + gm.sub;
    if (a < A) sp[a] = pexp[t];
  }
  __syncwarp();
  double f = sp[0], c = 0.0;  // int 0 + x
  if (p.prior_sum_mode == 0) {
#pragma unroll 8
    for (int a = 1; a < A; ++a) f = __dadd_rn(f, sp[a]);
  } else {  // Neumaier steps, CPython >= 3.12 Python/bltinmodule.c
#pragma unroll 8
    for (int a = 1; a < A; ++a) {
      const double x = sp[a];
      const double s = __dadd_rn(f, x);
      const bool big = fabs(f) >= fabs(x);
      const double hi = big ? f : x, lo = big ? x : f;
      c = __dadd_rn(c, __dadd_rn(__dsub_rn(hi, s), lo));
      f = s;
    }
    if (c != 0.0 && isfinite(c)) f = __dadd_rn(f, c);
  }
  __syncwarp();
  FS2_STAMP(23);
  double pv[AL];
#pragma unroll
  for (int t = 0; t < AL; ++t) {
    const int a = L * t + gm.sub;
    pv[t] = __ddiv_rn(pexp[t], f);
    if (gm.valid && a < A) *reinterpret_cast<double*>(gm.base + G.pri + ((size_t)newn * G.a2 + a) * 8) = pv[t];
  }
  FS2_STAMP(24);
  const bool force_dense = p.init_score != 0.0;
  const uint32_t all = A < 32 ? (1u << A) - 1u : 0xffffffffu;
  double pvs[1][AL], ptops[1];
  int uacts[1];
#pragma unroll
  for (int t = 0; t < AL; ++t) pvs[0][t] = pv[t];
  const uint32_t xms[1] = {~all};
  top_unexpanded<AL, 1>(pvs, xms, A, gm.sub, force_dense, ptops, uacts);
  const double ptop_new = ptops[0], ptop_par = pre.ptop_par, edge_prior = pre.edge_prior;
  const int uact_new = uacts[0], uact_par = pre.uact_par;
  const uint32_t xm_par = pre.xm_par;
  if (gm.valid && gm.sub == 0) {
    node[newn] = 0u | ((uint32_t)action << 8) | ((uint32_t)uact_new << 16) | ((uint32_t)parent << 24);
    sm.next[gm.gl * sm.s1 + newn] = sm.first[gm.gl * sm.s1 + parent];
    sm.first[gm.gl * sm.s1 + parent] = (uint8_t)newn;
    sm.first[gm.gl * sm.s1 + newn] = 0;
    xmask[newn] = ~all;
    *reinterpret_cast<double*>(gm.base + G.utop + 32 * newn) = ptop_new;
    node[parent] = (node[parent] & 0xff00ffffu) | ((uint32_t)uact_par << 16);
    xmask[parent] = xm_par;
    if (uact_par != UACT_NONE) *reinterpret_cast<double*>(gm.base + G.utop + 32 * parent) = ptop_par;
  }
  __syncwarp();
  FS2_STAMP(25);

  // ---- backup.  Position k on the path is node path_n[k] (k < depth) or the new node (k == depth); lane `sub`
  // owns positions 8 m + sub.  The value recurrence (mcts.py:142: value = (+/-)reward + discount * value) is
  // serial in binary64; it runs in all lanes from the positions' signed rewards in the scratch row ----
  double value = (double)value_f;
  double lmin = INFINITY, lmax = -INFINITY;
  constexpr int CHP = 32;       // positions per chunk (the scratch row holds >= 33 doubles)
  constexpr int CM = CHP / L;   // position slots of a lane per chunk
  auto chunk = [&](auto m0_tag) {
    constexpr int M0 = decltype(m0_tag)::value;
    constexpr int base = M0 * L;
#pragma unroll
    for (int mm = 0; mm < CM; ++mm) {
      constexpr int dummy = 0;
      (void)dummy;
      const int m = M0 + mm;
      if (m >= MAXP) continue;
      const int kk = L * m + gm.sub;
      const bool on = gm.valid && kk <= depth;
      const float rw = kk < depth ? __uint_as_float(own[m < MAXP ? m : 0].z) : node_reward_new;
      // (-reward if two_players and node.to_play == to_play else reward)
      const bool same = two && (((depth - kk) & 1) == 0);
      if (on) sp[kk - base] = (double)(same ? -rw : rw);
    }
    __syncwarp();
    double myval[CM];
#pragma unroll
    for (int mm = CM - 1; mm >= 0; --mm) {
      myval[mm] = 0.0;
      if (M0 + mm >= MAXP || L * (M0 + mm) > dmax) continue;  // warp uniform
#pragma unroll
      for (int jj = L - 1; jj >= 0; --jj) {
        const int kk = L * (M0 + mm) + jj;
        const bool on = gm.valid && kk <= depth;
        const double rs = sp[on ? kk - base : 0];
        myval[mm] = jj == gm.sub ? value : myval[mm];
        const double nv = __dadd_rn(rs, __dmul_rn(disc, value));
        value = on ? nv : value;
      }
    }
    __syncwarp();
    // per-position updates, straight-line over the lane's slots (their chains overlap); value_sum / visit_count
    // through the reciprocal table: bit-identical to IEEE division inside the guarded range, else redone exactly
    bool on[CM], redo = false;
    double nvs[CM], nq[CM];
    int nid[CM], nvc[CM];
    float rwv[CM];
#pragma unroll
    for (int mm = 0; mm < CM; ++mm) {
      const int m = M0 + mm;
      const int kk = L * m + gm.sub;
      on[mm] = m < MAXP && gm.valid && kk <= depth;
      const uint4 o = own[m < MAXP ? m : 0];
      // value_sum += value if node.to_play == to_play else -value
      const bool same = two ? (((depth - kk) & 1) == 0) : true;
      const double vs0 = kk < depth ? u2d(o.x, o.y) : 0.0;
      rwv[mm] = kk < depth ? __uint_as_float(o.z) : node_reward_new;
      nvs[mm] = __dadd_rn(vs0, same ? myval[mm] : -myval[mm]);
      nid[mm] = on[mm] ? (kk < depth ? (int)pn_[kk] : newn) : 0;
      nvc[mm] = (int)(node[nid[mm]] & 0xffu) + 1;
      const double dn = (double)nvc[mm];
      const double mean = fs_div_by_const(nvs[mm], dn, sm.rcp[nvc[mm] & 63]);
      const unsigned hv = (unsigned)__double2hiint(nvs[mm]) & 0x7fffffffu;
      redo = redo || (on[mm] && nvs[mm] != 0.0 && hv - 0x33700000u > 0x19000000u);
      const double dq = __dmul_rn(disc, mean);  // mcts.py:136-141
      nq[mm] = two ? __dsub_rn((double)rwv[mm], dq) : __dadd_rn((double)rwv[mm], dq);
    }
    if (__any_sync(MZ_FULL, redo)) {
#pragma unroll
      for (int mm = 0; mm < CM; ++mm) {
        const double dq = __dmul_rn(disc, __ddiv_rn(nvs[mm], (double)nvc[mm]));
        nq[mm] = two ? __dsub_rn((double)rwv[mm], dq) : __dadd_rn((double)rwv[mm], dq);
      }
    }
#pragma unroll
    for (int mm = 0; mm < CM; ++mm) {
      const int kk = L * (M0 + mm) + gm.sub;
      if (on[mm]) {
        node[nid[mm]] = (node[nid[mm]] & 0xffffff00u) | (uint32_t)nvc[mm];
        *reinterpret_cast<uint4*>(gm.base + G.own + 16 * nid[mm]) = make_uint4(
            (uint32_t)__double2loint(nvs[mm]), (uint32_t)__double2hiint(nvs[mm]), __float_as_uint(rwv[mm]), 0u);
        if (kk > 0) {
          lmin = fmin(lmin, nq[mm]);
          lmax = fmax(lmax, nq[mm]);
          if (kk == depth) *reinterpret_cast<double2*>(gm.base + G.edge + 32 * nid[mm]) = make_double2(edge_prior, nq[mm]);
          else *reinterpret_cast<double*>(gm.base + G.edge + 32 * nid[mm] + 8) = nq[mm];
        }
      }
    }
    __syncwarp();
  };
  if (dmax >= 2 * CHP) chunk(std::integral_constant<int, 2 * CM>());
  if (dmax >= CHP) chunk(std::integral_constant<int, CM>());
  chunk(std::integral_constant<int, 0>());
  FS2_STAMP(26);
#pragma unroll
  for (int m = 1; m < L; m <<= 1) {
    lmin = fmin(lmin, shfl8_xor_f64(lmin, m));
    lmax = fmax(lmax, shfl8_xor_f64(lmax, m));
  }
  if (gm.valid && gm.sub == 0 && depth > 0) {  // MinMaxStats.update mcts.py:11-14
    if (lmin < sm.mm[2 * gm.gl]) sm.mm[2 * gm.gl] = lmin;
    if (lmax > sm.mm[2 * gm.gl + 1]) sm.mm[2 * gm.gl + 1] = lmax;
  }
  __syncwarp();
}

// game.py:106-111 + Node.value (mcts.py:42-45); also leaves the node words in the block for mz_fc_search_export
MZ_DEV void root_stats(const FsParams& p, const Smem& sm, const Game& gm, const Geo& G) {
  if (!gm.valid) return;
  const int A = p.A, S = p.S;
  const uint32_t* node = sm.node + gm.gl * sm.s1;
  const uint32_t lm = ~sm.xmask[gm.gl * sm.s1] | 0u;  // after the search the root's mask also has its expanded children
  (void)lm;
  uint32_t legal = p.legal ? p.legal[gm.g] : 0xffffffffu;
  if (A < 32) legal &= (1u << A) - 1u;
  for (int a = gm.sub; a < A; a += L) {
    if (p.visits) p.visits[(size_t)gm.g * A + a] = 0;
    if (p.child_visits) p.child_visits[(size_t)gm.g * A + a] = 0.0;
  }
  __syncwarp(0xffu << ((threadIdx.x & 31u) & ~7u));
  int sum = 0;
  for (int j = 1; j <= S; ++j)
    if ((node[j] >> 24) == 0u) sum += (int)(node[j] & 0xffu);
  for (int j = 1 + gm.sub; j <= S; j += L) {
    if ((node[j] >> 24) == 0u) {
      const int a = (int)((node[j] >> 8) & 0xffu), v = (int)(node[j] & 0xffu);
      if (p.visits) p.visits[(size_t)gm.g * A + a] = v;
      if (p.child_visits) p.child_visits[(size_t)gm.g * A + a] = __ddiv_rn((double)v, (double)sum);
    }
  }
  for (int n = gm.sub; n <= S; n += L)
    *reinterpret_cast<uint2*>(gm.base + G.meta + 8 * n) = make_uint2(node[n], sm.xmask[gm.gl * sm.s1 + n]);
  if (gm.sub == 0) {
    const uint4 o = ldg16(gm.base + G.own);
    const int n = (int)(node[0] & 0xffu);
    if (p.root_value) p.root_value[gm.g] = n == 0 ? 0.0 : __ddiv_rn(u2d(o.x, o.y), (double)n);
    if (p.minmax) {
      p.minmax[2 * gm.g] = sm.mm[2 * gm.gl];
      p.minmax[2 * gm.g + 1] = sm.mm[2 * gm.gl + 1];
    }
    *reinterpret_cast<double2*>(gm.base) = make_double2(sm.mm[2 * gm.gl], sm.mm[2 * gm.gl + 1]);
    *reinterpret_cast<uint32_t*>(gm.base + 16) = legal;
  }
}

}  // namespace fs2
