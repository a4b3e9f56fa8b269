/*
 * mzb200.h -- C ABI of libmzb200.so, the B200 (sm_100a) search-and-target engine.
 *
 * This is the drop-in boundary for the hot path of JimOhman/model-based-rl (SURVEY.md section 8b).
 * The reference has no FFI layer -- its boundary is duck-typed Python -- so every entry point below
 * names the reference function (file:line, relative to the reference repo) whose arithmetic it
 * replaces.  The Python mirror of the reference classes (MCTS, Node, MinMaxStats,
 * PrioritizedReplay, FCNetwork ...) in model-based-rl_b200/ binds these symbols with ctypes; see
 * INTEGRATION.md for the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless its name starts
 *     with `h_` (host).  The caller owns all memory; nothing here allocates or synchronises.
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it (CUDA-graph capturable).
 *   - return value: 0 on success, a negative MZ_ERR_* for rejected arguments, or a positive
 *     cudaError_t from the launch.  There is no CPU fallback anywhere.
 *   - search arithmetic is IEEE binary64 in the reference's operation order (no FMA contraction),
 *     so visit counts / selected actions are bit-exact against the reference.
 */
#ifndef MZB200_H_
#define MZB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(MZ_BUILDING) && defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define MZ_OK 0
#define MZ_ERR_BAD_ARG (-1)
#define MZ_ERR_UNSUPPORTED (-2)

#define MZ_MAX_ACTIONS 64      /* one warp per game; lane l owns action l and, when A > 32, action l + 32 */
#define MZ_CHILD_UNEXPANDED (-1)
#define MZ_CHILD_ILLEGAL (-2)  /* action absent from root.children (illegal move) */
#define MZ_GAME_HEADER_BYTES 32
#define MZ_NODE_STATS_BYTES 24

/* ------------------------------------------------------------------------------------------- */
/* Tree: flat fixed-capacity node pools, one contiguous block per game (HBM, L2 resident).       */
/*                                                                                               */
/* game block  = header (32 B) | node record x (S + 1)            node n is expanded by sim n-1   */
/* header      = f64 minimum | f64 maximum | i32 root_to_play | i32 reserved   (MinMaxStats,      */
/*               mcts.py:6-25)                                                                    */
/* node record = f64 q | i32 visit_count | f32 reward | f64 value_sum | f64 prior[A] | i16 child[A]*/
/*               | pad  (mcts.py:28-37; prior[a]/child[a] describe the child reached by action a, */
/*               whose own statistics live in node record child[a]; q = reward -/+ discount *     */
/*               value(), the quantity backpropagate feeds to MinMaxStats (mcts.py:136-141) and   */
/*               ucb_score normalises (mcts.py:120-121), cached at backup time)                   */
/* node_bytes  = round_up(24 + 10 * A, 16);  game_bytes = round_up(32 + (S+1) * node_bytes, 128)  */
/* ------------------------------------------------------------------------------------------- */
/* Legal masks (mz_tree_set_root, mz_tree_set_root_priors, mz_select_action, mz_dirichlet_noise):  */
/* W = ceil(A / 32) u32 words per game, row-major [G][W]; bit b of word w set <=> action 32 w + b  */
/* is legal.  Bits at or beyond A are ignored.  For A <= 32 this is one word per game.             */
/* ------------------------------------------------------------------------------------------- */
typedef struct mz_tree {
  int32_t num_games;        /* G */
  int32_t num_simulations;  /* S  config.num_simulations   mcts.py:66 */
  int32_t num_actions;      /* A  config.action_space      mcts.py:72 */
  int32_t two_players;      /*    config.two_players       mcts.py:73 */
  int32_t prior_sum_mode;   /* builtin sum() semantics of mcts.py:53: 1 = CPython >= 3.12
                               (Neumaier-compensated), 0 = plain left-to-right */
  int32_t hidden_words;     /* 4-byte words per hidden state (0 = no hidden pool) */
  int32_t node_bytes;
  int32_t reserved0;
  int64_t game_bytes;
  double discount;          /* config.discount             mcts.py:67 */
  double init_value_score;  /* config.init_value_score     mcts.py:70 */
  double min_bound;         /* known_bounds[0], +inf when None   mcts.py:9, 24 */
  double max_bound;         /* known_bounds[1], -inf when None */
  uint8_t* games;           /* [G] game blocks */
  const double* pb_c_table; /* [(S+1)*(S+1)]: entry [N*(S+1)+n] =
                               (log((N+pb_c_base+1)/pb_c_base)+pb_c_init) * (sqrt(N)/(n+1)), i.e. the
                               two statements at mcts.py:116-117 evaluated on the host in binary64 */
  uint32_t* hidden;         /* [G][S+1][hidden_words] hidden-state pool (Node.hidden_state) */
  int16_t* path;            /* [G][S+2] node ids of the current search path (root first) */
  int32_t* path_len;        /* [G] edges on the current path (= depth of the leaf) */
  int32_t* leaf_parent;     /* [G] node id of search_path[-2]          mcts.py:94 */
  int32_t* leaf_action;     /* [G] action that leaves it               mcts.py:96 */
} mz_tree;

/* Size helpers (host). */
int32_t mz_tree_node_bytes(int32_t num_actions);
int64_t mz_tree_game_bytes(int32_t num_simulations, int32_t num_actions);

/* Host: fills h_table[(S+1)*(S+1)] for mz_tree.pb_c_table.  MCTS.ucb_score mcts.py:116-117. */
int mz_fill_pb_c_table(int32_t num_simulations, double pb_c_base, double pb_c_init, double* h_table);

/*
 * Root set-up for every game: Node.expand over the legal actions (mcts.py:47-55, called at
 * actors.py:142), Node.add_exploration_noise (mcts.py:57-61, actors.py:143) and
 * MinMaxStats.reset (mcts.py:79).
 *   root_logits [G][A] f32   initial_inference().policy_logits
 *   legal_mask  [G][W] u32   legal-action mask (layout above); NULL = all legal
 *   noise       [G][A] f64   Dirichlet sample, dense over the root's children in action order
 *                            (what np.random.dirichlet returns at mcts.py:59); NULL = no noise
 *   root_to_play[G] i8       game.to_play; NULL = 1
 *   root_hidden [G][hidden_words] initial hidden state copied into pool slot 0; NULL = skip
 */
int mz_tree_set_root(const mz_tree* t, const float* root_logits, const uint32_t* legal_mask,
                     const double* noise, double noise_frac, const int8_t* root_to_play,
                     const uint32_t* root_hidden, void* stream);

/*
 * Node.add_exploration_noise's draw (mcts.py:59: np.random.dirichlet([root_dirichlet_alpha] * len(actions))) for
 * every game of a move, made on the device into the `noise` layout of mz_tree_set_root / mz_fc_search: row g holds
 * one value per legal action of game g (legal_mask [G][W], layout above; NULL = all), dense from column 0,
 * zeros behind.  Same distribution, another stream than numpy's: Philox4x32-10 keyed by (seed, game, action) and
 * advanced by `move`; the host-supplied buffer stays the bit-exact path.
 */
int mz_dirichlet_noise(int32_t num_games, int32_t num_actions, double alpha, const int32_t* legal_mask,
                       uint64_t seed, uint64_t move, double* noise, void* stream);

/*
 * Same, for a root the caller has already expanded on the host (the B=1 drop-in path:
 * root.expand + root.add_exploration_noise were run by the caller, actors.py:142-143):
 *   root_priors [G][A] f64 = root.children[a].prior (ignored where the action is illegal).
 */
int mz_tree_set_root_priors(const mz_tree* t, const double* root_priors, const uint32_t* legal_mask,
                            const int8_t* root_to_play, const uint32_t* root_hidden, void* stream);

/*
 * One descent per game for simulation `sim` (nodes 0..sim exist): the `while node.expanded():
 * select_child` loop of MCTS.run
 * (mcts.py:87-92) with MCTS.select_child / ucb_score (mcts.py:104-124).  Writes path, path_len,
 * leaf_parent, leaf_action.  If gathered_hidden != NULL also copies the parent's hidden state to
 * gathered_hidden[G][hidden_words] (the argument of recurrent_inference, mcts.py:94-96).
 * trace_* (each [G], may be NULL) receive parent / action / depth for parity checks.
 */
int mz_tree_select(const mz_tree* t, int32_t sim, uint32_t* gathered_hidden, int32_t* trace_parent,
                   int32_t* trace_action, int32_t* trace_depth, void* stream);

/*
 * Expansion of the leaf reached by the last mz_tree_select with the network outputs, then backup:
 * Node.expand(network_output, to_play, range(A)) (mcts.py:97, 47-55) and MCTS.backpropagate
 * (mcts.py:99, 126-143).  `sim` is the simulation index (the new node gets id sim + 1).
 *   value [G] f32, reward [G] f32, logits [G][A] f32: recurrent_inference outputs (eval mode)
 *   new_hidden [G][hidden_words]: next hidden state to store in the pool; NULL if the network
 *   kernel already wrote it there.
 */
int mz_tree_expand_backup(const mz_tree* t, int32_t sim, const float* value, const float* reward,
                          const float* logits, const uint32_t* new_hidden, void* stream);

/*
 * Fused simulation boundary: expand + backup of simulation `sim` followed by the descent of
 * simulation sim + 1 (skipped when sim + 1 == S), one launch; the live part of every game block is
 * staged in shared memory by one bulk async copy (cp.async.bulk) and both phases run on that image.
 * sim == -1 runs only the first descent.  Same arguments as the two calls above.
 */
int mz_tree_step(const mz_tree* t, int32_t sim, const float* value, const float* reward,
                 const float* logits, const uint32_t* new_hidden, uint32_t* gathered_hidden,
                 int32_t* trace_parent, int32_t* trace_action, int32_t* trace_depth, void* stream);

/*
 * After the last simulation: what callers read from the root (actors.py:147, config.py:72-73,
 * game.py:106-111).  Any output may be NULL.
 *   visits [G][A] i32 (0 for illegal actions), child_visits [G][A] f64 = visits / sum(visits)
 *   (Game.store_search_statistics game.py:107-110), root_value [G] f64 = Node.value() mcts.py:42-45,
 *   minmax [G][2] f64.
 */
int mz_tree_root_stats(const mz_tree* t, int32_t* visits, double* child_visits, double* root_value,
                       double* minmax, void* stream);

/*
 * Config.select_action (config.py:70-81) for G roots with host-supplied randomness.
 *   visits [G][A] i32, legal_mask [G][W] u32 or NULL, temperature [G] f64, uniforms [G] f64 in [0,1)
 *   T > 0 : p = visits**(1/T) / sum; action = children[searchsorted(cumsum(p)/cumsum(p)[-1], u,
 *           'right')]  (what np.random.choice(len, p=p) does with one uniform draw)
 *   T == 0: uniform over the argmax ties, tie index = floor(u * n_ties)
 */
int mz_select_action(int32_t num_games, int32_t num_actions, const int32_t* visits,
                     const uint32_t* legal_mask, const double* temperature, const double* uniforms,
                     int32_t* actions, void* stream);

/* Diagnostic: out[i] = the device's math.exp restatement applied to (double)x[i] (mcts.py:52).
 * Used by the tests to check bit-compatibility with the host libm. */
int mz_exp_f32(int64_t n, const float* x, double* out, void* stream);

/* Debug / façade support: copy one game's tree into dense arrays (any output may be NULL):
 * prior [S+1][A] f64, child [S+1][A] i32, vsum [S+1] f64, visit [S+1] i32, reward [S+1] f32. */
int mz_tree_export(const mz_tree* t, int32_t game, double* prior, int32_t* child, double* vsum,
                   int32_t* visit, float* reward, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* FCNetwork inference (networks.py:55-174), eval mode: hidden size 50, four 512-wide MLP heads, */
/* LayerNorm+ReLU on the state, softmax-expectation + h^-1 on value/reward (config.py:27-33).    */
/* ------------------------------------------------------------------------------------------- */
#define MZ_FC_HIDDEN 50
#define MZ_FC_WIDTH 512

typedef struct mz_fc_weights { /* device pointers, float32.  First layers (*_w1) are stored
                                  TRANSPOSED, [in][512]; second layers (*_w2) keep the
                                  nn.Linear layout [out][512]. */
  int32_t obs_dim, num_actions, value_bins, reward_bins;
  int32_t value_min, reward_min;    /* support = [min, min + bins - 1]  config.py:12-19 */
  int32_t no_target_transform;      /* config.no_target_transform   config.py:31 */
  int32_t no_support;               /* config.no_support (config.py:95; networks.py:135-136, 153, 161): value_bins =
                                       reward_bins = 1 and the heads' raw outputs are the scalars.  The float32 /
                                       tf32x3 kernels take it; the bf16 kernels and mz_fc_search return
                                       MZ_ERR_UNSUPPORTED. */
  const float *rep_w1, *rep_b1, *rep_w2, *rep_b2;  /* representation_head  networks.py:55-67 */
  const float *dyn_w1, *dyn_b1, *dyn_w2, *dyn_b2;  /* transition_head      networks.py:70-80 */
  const float *rew_w1, *rew_b1, *rew_w2, *rew_b2;  /* reward_head          networks.py:83-93 */
  const float *val_w1, *val_b1, *val_w2, *val_b2;  /* value_head           networks.py:96-106 */
  const float *pol_w1, *pol_b1, *pol_w2, *pol_b2;  /* policy_head          networks.py:109-119 */
  const float *ln_w, *ln_b;                        /* LN                   networks.py:144 */
} mz_fc_weights;

/* Observation ingest for byte observations (Breakout-ram: 128 bytes, README.md:56 `--obs_range 0 255
 * --norm_obs`): out[r][k] = (float(obs[r][k]) - obs_min[k]) / obs_range[k] in float32, the arithmetic of
 * actors.py:127-129 / learners.py:170-171.  obs_min / obs_range [obs_dim] f32; NULL = 0 / 255. */
int mz_obs_normalize_u8(int64_t rows, int32_t obs_dim, const uint8_t* obs, const float* obs_min,
                        const float* obs_range, float* out, void* stream);

/*
 * float32 reference-precision path (CUDA cores).
 * BaseNetwork.initial_inference (networks.py:26-29): obs [B][obs_dim] f32 ->
 *   hidden [B][hidden_stride words] (first 50 used), value [B], logits [B][A].
 */
int mz_fc_initial_f32(const mz_fc_weights* w, int32_t batch, const float* obs, float* hidden,
                      int64_t hidden_stride, float* value, float* logits, void* stream);
/*
 * BaseNetwork.recurrent_inference (networks.py:31-34).  Row b reads its input state from
 *   hidden_in + b * in_row_stride + in_index[b] * 50   (in_index may be NULL = 0)
 * and writes the next state to hidden_out + b * out_row_stride + out_offset, so it can gather from /
 * scatter into the tree's hidden pool directly (in_index = leaf_parent, strides = (S+1)*50).
 */
int mz_fc_recurrent_f32(const mz_fc_weights* w, int32_t batch, const float* hidden_in,
                        int64_t in_row_stride, const int32_t* in_index, const int32_t* actions,
                        float* hidden_out, int64_t out_row_stride, int64_t out_offset, float* value,
                        float* reward, float* logits, void* stream);

/*
 * float32-ACCURATE tensor-core path (csrc/mz_fcnet_tf32.cu): the arguments and the results (within float32
 * rounding) of mz_fc_initial_f32 / mz_fc_recurrent_f32, every Linear layer (networks.py:55-119) on the tensor
 * cores as three TF32 instructions per product on split operands (x_lo*w_hi + x_hi*w_lo + x_hi*w_hi, float32
 * accumulation).  MZ_ERR_UNSUPPORTED when obs_dim is too wide for the shared-memory budget (~450).
 */
int mz_fc_initial_tf32x3(const mz_fc_weights* w, int32_t batch, const float* obs, float* hidden,
                         int64_t hidden_stride, float* value, float* logits, void* stream);
int mz_fc_recurrent_tf32x3(const mz_fc_weights* w, int32_t batch, const float* hidden_in,
                           int64_t in_row_stride, const int32_t* in_index, const int32_t* actions,
                           float* hidden_out, int64_t out_row_stride, int64_t out_offset, float* value,
                           float* reward, float* logits, void* stream);

/*
 * bf16 tensor-core path (tcgen05.mma, accumulators in TMEM, fp32 accumulation) of
 * recurrent_inference.  The weights are first re-packed once per weight update into the
 * shared-memory image the MMA consumes (packed bytes and tail floats caller-allocated).
 * mz_fc_recurrent_tc has the arguments of mz_fc_recurrent_f32 plus the packed buffers; `w` is only
 * read for its integer fields.  Limits: 1 <= A <= 64, value/reward bins 1..64, no no_support
 * (MZ_ERR_UNSUPPORTED otherwise).  Hidden rows are read as float2, so hidden_in must be 8-byte aligned
 * and in_row_stride even (MZ_ERR_BAD_ARG otherwise).
 * Two image geometries: narrow (A <= 32 and both supports <= 32 bins; the image mz_fc_search reads) and
 * wide (anything up to 64).  mz_fc_tc_sizes gives the sizes of both images and of the tail for `w`:
 * recurrent packed bytes, initial-inference packed bytes (MZ_ERR_UNSUPPORTED in that slot when obs_dim is
 * too wide for the kernel: use mz_fc_initial_f32), tail floats.  mz_fc_tc_packed_bytes(A),
 * mz_fc_tc_initial_packed_bytes(obs_dim) and mz_fc_tc_tail_floats() give the narrow image's sizes.
 */
int mz_fc_tc_sizes(const mz_fc_weights* w, int64_t* recurrent_bytes, int64_t* initial_bytes,
                   int32_t* tail_floats);
int64_t mz_fc_tc_packed_bytes(int32_t num_actions);
/* Diagnostics: when set to a device buffer of >= 512 int64, CTA 0 of every following
 * mz_fc_recurrent_tc launch stores clock64() stamps of its pipeline phases there (NULL disables). */
int mz_debug_set_tc_trace_block(int32_t block); /* which CTA writes the stamps (default 0) */
int mz_debug_set_tc_trace(int64_t* device_buffer);
int32_t mz_fc_tc_tail_floats(void);
int mz_fc_tc_pack(const mz_fc_weights* w, void* packed, float* tail, void* stream);
int mz_fc_recurrent_tc(const mz_fc_weights* w, const void* packed, const float* tail, int32_t batch,
                       const float* hidden_in, int64_t in_row_stride, const int32_t* in_index,
                       const int32_t* actions, float* hidden_out, int64_t out_row_stride,
                       int64_t out_offset, float* value, float* reward, float* logits, void* stream);

/* 1 (default): mz_fc_recurrent_tc runs as clusters of two CTAs per 128 rows -- rank 0 evaluates the
 * reward and value heads, rank 1 the transition and policy heads, h' crosses through distributed
 * shared memory; 0: one CTA evaluates all four heads. */
int mz_fc_tc_set_split(int32_t enable);

/* BaseNetwork.initial_inference (networks.py:26-29) on the same tensor-core kernel: representation
 * head (obs [B][obs_dim] f32, K = obs_dim + bias column) -> LayerNorm + ReLU -> prediction heads.
 * Its own packed image / tail (mz_fc_tc_initial_packed_bytes, mz_fc_tc_pack_initial);
 * MZ_ERR_UNSUPPORTED when obs_dim is too wide for the shared-memory budget (use mz_fc_initial_f32).
 * hidden_out row g at hidden_out + g * out_row_stride (the tree's hidden pool, slot 0). */
int64_t mz_fc_tc_initial_packed_bytes(int32_t obs_dim);
int mz_fc_tc_pack_initial(const mz_fc_weights* w, void* packed, float* tail, void* stream);
int mz_fc_initial_tc(const mz_fc_weights* w, const void* packed, const float* tail, int32_t batch,
                     const float* obs, float* hidden_out, int64_t out_row_stride, float* value,
                     float* logits, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Whole move in one persistent kernel: MCTS.run (mcts.py:78-102) with FCNetwork (networks.py:31-34,  */
/* 122-174) in the loop.  A thread-block cluster owns 128 games for all S simulations: root set-up */
/* (Node.expand over the legal actions + add_exploration_noise, mcts.py:47-61), then per simulation  */
/* descent (mcts.py:87-92, 104-124) -> recurrent_inference on tcgen05 tensor cores -> expand +     */
/* backpropagate (mcts.py:47-55, 126-143), handed from phase to phase through mbarriers in          */
/* (distributed) shared memory, and the root statistics of game.py:106-111 at the end.  Same       */
/* arithmetic as mz_tree_step + mz_fc_recurrent_tc (bit-identical results); the tree uses its own    */
/* layout (csrc/mz_fcs_sparse.cuh) and the hidden pool is bf16 [G][S+1][64].                        */
/* Shapes: 1 <= A <= 32, 1 <= S <= 63, and (S, A) within the kernel's shared-memory plan, as        */
/* mz_fc_search_supported reports; mz_fc_search returns MZ_ERR_UNSUPPORTED for any other shape.     */
/* ------------------------------------------------------------------------------------------- */
typedef struct mz_fc_search_args {
  const mz_fc_weights* weights;  /* dims, supports (the float32 pointers are not read) */
  const void* packed;            /* mz_fc_tc_pack image */
  const float* tail;
  int32_t num_games;             /* G */
  int32_t num_simulations;       /* S <= 63    config.num_simulations mcts.py:66 */
  int32_t two_players;           /*            config.two_players     mcts.py:73 */
  int32_t prior_sum_mode;        /* as in mz_tree */
  int64_t game_bytes;            /* >= mz_fc_search_game_bytes(S, A) */
  double discount, init_value_score, min_bound, max_bound;  /* as in mz_tree */
  double noise_frac;             /* config.root_exploration_fraction (used when noise != NULL) */
  uint8_t* games;                /* [G] game blocks (this kernel's layout) */
  const double* pb_c_table;      /* [(S+1)*(S+1)] as in mz_tree */
  void* pool;                    /* [G][S+1][64] bf16 hidden states (Node.hidden_state) */
  const float* root_logits;      /* [G][A]   initial_inference().policy_logits */
  const uint32_t* legal_mask;    /* [G] or NULL */
  const double* noise;           /* [G][A] or NULL */
  const int8_t* root_to_play;    /* [G] or NULL (kept for the caller; the arithmetic is relative) */
  const float* root_hidden;      /* [G][50] initial_inference().hidden_state */
  int32_t* visits;               /* [G][A] */
  double* child_visits;          /* [G][A]   game.py:107-110 */
  double* root_value;            /* [G]      root.value() */
  double* minmax;                /* [G][2] */
  int32_t* trace_parent;         /* [S][G] or NULL: leaf parent / action / depth of every simulation */
  int32_t* trace_action;
  int32_t* trace_depth;
  float* rec_value;              /* [S][G] or NULL: what the network returned (parity replays) */
  float* rec_reward;             /* [S][G] */
  float* rec_logits;             /* [S][G][A] */
  int64_t* timeline;             /* [S][32] clock64 stamps of tile 0 or NULL (diagnostics) */
  int32_t* error_flag;           /* set before the kernel traps on a protocol time-out, or NULL */
} mz_fc_search_args;

int64_t mz_fc_search_game_bytes(int32_t num_simulations, int32_t num_actions);
int32_t mz_fc_search_pool_row(void);                         /* bf16 elements per pool row (64) */
int mz_fc_search_supported(int32_t num_simulations, int32_t num_actions); /* 1: shapes fit the kernel */
int mz_fc_search(const mz_fc_search_args* a, void* stream);
/* one game's tree as the arrays of mz_tree_export (+ the cached child q [S+1][A]) */
int mz_fc_search_export(const mz_fc_search_args* a, int32_t game, double* prior, int32_t* child,
                        double* vsum, int32_t* visit, float* reward, double* q, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Scalar transforms and supports (config.py:27-68), float32 in torch's op order.                */
/* ------------------------------------------------------------------------------------------- */
/* Config.scalar_transform config.py:51-54, elementwise h(x). */
int mz_scalar_transform(int64_t n, const float* x, float* out, void* stream);
/* Config.scalar_to_support config.py:56-68: x [n] -> support [n][bins] (two-hot). x is clamped in
 * place like the reference's x.clamp_ when clamp_in_place != 0. */
int mz_scalar_to_support(int64_t n, float* x, int32_t support_min, int32_t support_max,
                         int32_t clamp_in_place, float* support, void* stream);
/* Config.inverse_transform config.py:27-33: logits [n][bins] -> scalar [n]. */
int mz_support_to_scalar(int64_t n, const float* logits, int32_t support_min, int32_t support_max,
                         int32_t no_target_transform, float* out, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Replay window + fused target construction (replay_buffer.py:124-198, learners.py:186-192).    */
/*                                                                                               */
/* The window is a structure of arrays over "positions"; a chunk (one HistorySlice, game.py:5-16)*/
/* occupies positions [chunk_start, chunk_start + chunk_len).                                    */
/* ------------------------------------------------------------------------------------------- */
typedef struct mz_window {
  int32_t num_actions;      /* A */
  int32_t obs_elems;        /* elements per observation */
  int32_t obs_is_u8;        /* 1: obs stored as uint8, 0: float32 */
  int32_t clip_rewards;     /* 1: every reward is read as np.sign(reward) -- ClipRewardEnv.reward,
                               wrappers.py:236-238 (the Breakout configuration, README.md:56): the window keeps
                               the raw environment rewards and the target kernel clips them on the fly */
  const void* obs;          /* [P][obs_elems] u8 or f32   history.observations */
  const int32_t* actions;   /* [P]                        history.actions */
  const float* rewards;     /* [P] f32(history.rewards): both uses (np.array(.., float32) at
                               replay_buffer.py:187 and the float32 store at :193) round to f32 */
  const int8_t* to_play;    /* [P]                        history.to_play */
  const double* root_values;/* [P]                        history.root_values */
  const float* child_visits;/* [P][A] f32(history.child_visits) */
} mz_window;

typedef struct mz_target_cfg {
  int32_t batch;            /* B   config.batch_size */
  int32_t num_unroll_steps; /* K   config.num_unroll_steps */
  int32_t td_steps;         /* T   config.td_steps */
  int32_t fuse_supports;    /* also emit h(x) + two-hot supports (learners.py:186-192) */
  int32_t value_min, value_max, reward_min, reward_max; /* supports config.py:12-19 */
  int32_t no_target_transform;
  int32_t normalize_obs;    /* apply (obs - obs_min) / obs_range (learners.py:170-171) */
  double disc_pow_td;       /* discount ** td_steps (replay_buffer.py:181) */
  const float* discounts;   /* [K+T] f32(discount ** n) (replay_buffer.py:84) */
  const float* obs_min;     /* [obs_elems] or NULL */
  const float* obs_range;   /* [obs_elems] or NULL */
} mz_target_cfg;

/*
 * For every sampled row b: position pos[b] (absolute window position of (history, step)), its
 * chunk [chunk_start[b], chunk_start[b] + chunk_len[b]) (chunk_len = len(root_values)) and
 * chunk_obs_len[b] is not needed (obs are indexed by position).
 * Outputs: obs_out [B][obs_elems] f32, actions_out [B][K] i32 (padded from pad_actions [B][K]),
 * t_rewards/t_values [B][K+1] f32, t_policies [B][K+1][A] f32, and when fuse_supports:
 * value_support [B][K+1][Vbins], reward_support [B][K+1][Rbins].
 */
int mz_build_targets(const mz_window* w, const mz_target_cfg* c, const int64_t* pos,
                     const int64_t* chunk_start, const int32_t* chunk_len, const int32_t* pad_actions,
                     float* obs_out, int32_t* actions_out, float* t_rewards, float* t_values,
                     float* t_policies, float* value_support, float* reward_support, void* stream);
/*
 * Self-play -> replay hand-off on the device (Game.apply + Game.store_search_statistics, game.py:79-115; the
 * HistorySlice an actor sends, actors.py:160-169): one trajectory step of num_games games written straight into
 * the window arrays.  Game g's record goes to position dst_pos[g] (< 0: skip the game):
 *   obs [G][obs_elems] u8 / f32 (the search input of the move), actions [G] i32, rewards [G] f32, to_play [G] i8,
 *   root_values [G] f64, child_visits [G][A] f64 (stored as float32, like replay_buffer.py:192).
 * mz_window_copy copies `count` runs of positions (src[r] .. src[r] + n[r] - 1 -> dst[r] ..): the
 * num_unroll_steps + td_steps positions a running game's next chunk repeats (actors.py:160-166).
 */
int mz_window_append(const mz_window* w, int32_t num_games, const int64_t* dst_pos, const void* obs,
                     const int32_t* actions, const float* rewards, const int8_t* to_play, const double* root_values,
                     const double* child_visits, void* stream);
int mz_window_copy(const mz_window* w, int32_t count, const int64_t* src, const int64_t* dst, const int32_t* n,
                   void* stream);
/* Three kernels serve mz_build_targets.  For K + 1 <= 16 and td_steps <= 64: the TMA-staged kernel (a CTA stages
 * the observation / child-visit windows of its rows with cp.async.bulk, builds shared-memory images of all seven
 * outputs and hands them to the bulk-copy engine) and, where its images do not fit shared memory, the
 * lane-per-unroll-position kernel (a warp owns 32 / (K + 1) consecutive rows).  Everything else (e.g.
 * td_steps = 1000): warp per row.  which = 1 forces the warp-per-row kernel, 2 the lane-per-position kernel,
 * 3 the TMA-staged kernel (parity tests run all of them on the same inputs), 0 restores the choice by shape. */
int mz_debug_set_targets_kernel(int32_t which);
/* launch shape of the TMA-staged kernel: sampled rows per CTA (4, 8, 16 or 32) and threads per CTA (a power of
 * two, 32 .. 256, at least one per row) */
int mz_debug_set_targets_tma(int32_t rows_per_cta, int32_t threads);

/* ------------------------------------------------------------------------------------------- */
/* Prioritized-replay sum-tree in HBM (SumTree, replay_buffer.py:6-66): float64 array-embedded    */
/* heap of 2*max_capacity-1 sums, leaves at [max_capacity-1, 2*max_capacity-1).  Batches of       */
/* updates run in parallel but every node receives its float64 additions in batch order, so the   */
/* sums are bit-identical to the reference's one-leaf-at-a-time loop.                             */
/* ------------------------------------------------------------------------------------------- */
/* SumTree.update (replay_buffer.py:35-41) applied to n (tree index, priority) pairs in order
 * (PrioritizedReplay.update, replay_buffer.py:200-203).  scratch: [n] f64 workspace. */
int mz_sumtree_update(double* tree, int64_t max_capacity, int64_t n, const int64_t* tree_idx,
                      const double* priority, double* scratch, void* stream);
/* SumTree.add (replay_buffer.py:19-33): update + buffer[slot] = (step, history) for the n sampled
 * steps of one chunk; step i of the chunk sits at window position chunk_start + i.  The ring
 * arithmetic that picks the slots (position / capacity growth) stays on the host.
 *   slot_pos/slot_start [max_capacity] i64, slot_len [max_capacity] i32: where each slot's
 *   (history, step) lives in the replay window (see mz_window). */
int mz_sumtree_add(double* tree, int64_t max_capacity, int64_t n, const int64_t* tree_idx,
                   const double* priority, int64_t chunk_start, int32_t chunk_len, int64_t* slot_pos,
                   int64_t* slot_start, int32_t* slot_len, double* scratch, void* stream);
/* Same for memories first_step .. first_step + n - 1 of the chunk (slot -> chunk_start + first_step + i).  The
 * tree indices of ONE call must be distinct: a history that laps the ring is added in pieces, so that the last
 * write to a slot wins like in the reference's one-memory-at-a-time loop (replay_buffer.py:19-33). */
int mz_sumtree_add_from(double* tree, int64_t max_capacity, int64_t n, const int64_t* tree_idx,
                        const double* priority, int64_t chunk_start, int32_t chunk_len, int32_t first_step,
                        int64_t* slot_pos, int64_t* slot_start, int32_t* slot_len, double* scratch, void* stream);
/* SumTree.add for the memories of several chunks in one call (the histories every game of a self-play move
 * finished, actors.py:160-169 -> replay_buffer.py:113-122): memory i belongs to segment s with
 * seg_begin[s] <= i < seg_begin[s + 1] and is step i - seg_begin[s] of the chunk at window position seg_start[s]
 * (length seg_len[s]).  seg_begin [num_segments + 1] i32, seg_start [num_segments] i64, seg_len [num_segments] i32.
 * The tree indices of one call must be distinct, like mz_sumtree_add_from's. */
int mz_sumtree_add_chunks(double* tree, int64_t max_capacity, int64_t n, const int64_t* tree_idx,
                          const double* priority, int32_t num_segments, const int32_t* seg_begin,
                          const int64_t* seg_start, const int32_t* seg_len, int64_t* slot_pos, int64_t* slot_start,
                          int32_t* slot_len, double* scratch, void* stream);
/* The sampling half of sample_batch (replay_buffer.py:134-145, 160-162) for n rows:
 *   value_b = random.uniform(seg*b, seg*(b+1)) with seg = total/n, computed on the device from the
 *   host-drawn u01[b] = random.random() (same binary64 operations as CPython's uniform());
 *   SumTree.get_leaf (replay_buffer.py:43-62) -> tree_idx[n], priority[n]; when slot_pos != NULL
 *   also the row's window position / chunk start / chunk length (inputs of mz_build_targets);
 *   when is_weights != NULL: (num_memories * priority/total) ** -beta, divided by its maximum. */
int mz_sumtree_sample(const double* tree, int64_t max_capacity, int32_t n, const double* u01,
                      const int64_t* slot_pos, const int64_t* slot_start, const int32_t* slot_len,
                      int64_t num_memories, double beta, int64_t* tree_idx, double* priority,
                      int64_t* pos, int64_t* chunk_start, int32_t* chunk_len, double* is_weights,
                      void* stream);
/* sample_batch in one call (replay_buffer.py:124-163): mz_sumtree_sample followed by mz_build_targets on the rows
 * it drew -- the sampling outputs (pos / chunk_start / chunk_len) stay on the device as the target kernel's inputs.
 * Arguments as in the two functions, plus:
 *   u01_is_mt_words != 0: u01[b] holds the two raw MT19937 outputs CPython's random.random() would consume for
 *     row b (little endian, as random.getrandbits(64 * n).to_bytes(8 * n, "little") lays them out); the kernel forms
 *     ((w0 >> 5) * 2**26 + (w1 >> 6)) / 2**53 itself -- the same float64, without 512 interpreter calls;
 *   pad_seed != 0: the padding actions (np.random.randint(action_space), replay_buffer.py:149-152) are drawn on
 *     the device into pad_actions [B][K] from splitmix64(pad_seed, index) instead of being read from it. */
int mz_replay_sample_targets(const double* tree, int64_t max_capacity, const double* u01, int32_t u01_is_mt_words,
                             const int64_t* slot_pos, const int64_t* slot_start, const int32_t* slot_len,
                             int64_t num_memories, double beta, int64_t* tree_idx, double* priority, int64_t* pos,
                             int64_t* chunk_start, int32_t* chunk_len, double* is_weights, const mz_window* w,
                             const mz_target_cfg* c, int32_t* pad_actions, uint64_t pad_seed, float* obs_out,
                             int32_t* actions_out, float* t_rewards, float* t_values, float* t_policies,
                             float* value_support, float* reward_support, void* stream);
/* mz_sumtree_sample with the u01_is_mt_words switch described above */
int mz_sumtree_sample_mt(const double* tree, int64_t max_capacity, int32_t n, const double* u01, int32_t u01_is_mt_words,
                         const int64_t* slot_pos, const int64_t* slot_start, const int32_t* slot_len,
                         int64_t num_memories, double beta, int64_t* tree_idx, double* priority,
                         int64_t* pos, int64_t* chunk_start, int32_t* chunk_len, double* is_weights,
                         void* stream);
/* PrioritizedReplay.update (replay_buffer.py:200-203) from the learner's float32 errors still on the device
 * (learners.py:183): priority = (|error| + epsilon) ** alpha in numpy's float32 arithmetic (np.abs(float32 array) +
 * python float stays float32, NEP 50), widened to the tree's float64, then mz_sumtree_update.  alpha == 1 is
 * bit-exact; any other alpha goes through pow() and may differ from numpy's powf in the last float32 bit (the
 * Python facade routes those through the host).  priority / scratch: [n] f64 workspaces. */
int mz_sumtree_update_errors(double* tree, int64_t max_capacity, int64_t n, const int64_t* tree_idx,
                             const float* errors, double epsilon, double alpha, double* priority, double* scratch,
                             void* stream);

/* ------------------------------------------------------------------------------------------- */
/* MuZeroNetwork (residual conv tower, networks.py:393-554) on tcgen05 tensor cores, bf16/f32 acc. */
/* Activations: flat [games * 49][128] bf16, channels last, shared zero padding: a game is one zero  */
/* row of 7 followed by 6 image rows of (6 pixels + 1 zero), so every out-of-image 3x3 neighbour     */
/* is a zero row and a tap is a row shift of dy*7 + dx: the implicit GEMM needs no im2col.           */
/* ------------------------------------------------------------------------------------------- */
#define MZ_CONV_ROWS_PER_GAME 49
#define MZ_CONV_RELU 1      /* max(x, 0) */
#define MZ_CONV_RESIDUAL 2  /* += residual before the ReLU            ResidualBlock.forward networks.py:384-391 */
#define MZ_CONV_ACTION 4    /* += actions[g] / A * plane_term[pixel]  MuZeroNetwork.attach_action networks.py:536-541 */
#define MZ_CONV_SCALE 8     /* also emit (x - min_c) / (max_c - min_c) MuZeroNetwork.scale_state networks.py:543-547 */
/* Conv2d(C -> C, 3x3, padding 1), C = channels = 128 (or 64: resblocks1 of the representation,
 * rows of 64 channels, w_packed [64][9*64]) with BatchNorm2d (eval) folded into w_packed / bias, on
 * width x width images (6 for the hidden state; 12 / 24 inside the representation tower) in the same
 * flat padded layout with (width + 1)^2 rows per game.
 *   x, residual, out, out_scaled [games*(width+1)^2][128] bf16 (out may be NULL with MZ_CONV_SCALE)
 *   w_packed   [128][9*128] bf16, k = (ky*3 + kx)*128 + c_in;   bias [128] f32
 *   plane_term [36][128] f32, actions [games] i32 (flags & MZ_CONV_ACTION)
 *   pool_out, pool_row_base [games]: with MZ_CONV_SCALE the scaled rows of game g are also written
 *   to rows pool_row_base[g] .. +49 of pool_out (the hidden-pool slot of the node being expanded). */
int mz_conv3x3_tc(int32_t games, int32_t width, int32_t channels, const void* x, const void* w_packed,
                  const float* bias, int32_t flags,
                  const float* plane_term, const int32_t* actions, int32_t num_actions,
                  const void* residual, void* out, void* out_scaled, void* pool_out,
                  const int32_t* pool_row_base, void* stream);
/* 128-channel convolutions run on clusters of two CTAs (tcgen05.mma.cta_group::2, M = 256, the weight
 * matrix resident in the pair's shared memory).  mode 0 selects the single-CTA kernel, 1 the pair kernel
 * with one activation load per tap, 2 (default) the pair kernel with one activation row window per tile
 * for images of width <= 6 (the taps become row offsets of the A descriptor) and mode 1 for wider ones. */
int mz_conv_set_pair(int32_t mode);
/* Strided convolutions of MuZeroRepresentation (conv1, conv2: networks.py:399, 402) = im2col of the
 * stride-2 patches + GEMM whose output rows land in the padded layout; AvgPool2d(3, 2, 1)
 * (networks.py:406, 409) between padded layouts.  Padding rows of the outputs are never written:
 * zero the buffers once. */
int mz_conv_im2col_s2(int32_t games, int32_t w_in, int32_t channels, int32_t k_pad, const void* in, void* out,
                      void* stream);
int mz_conv_gemm_to_padded(int32_t games, int32_t out_w, int32_t k, int32_t n_out, const void* a, const void* w,
                           const float* bias, int32_t relu, void* out, void* stream);
int mz_conv_avgpool(int32_t games, int32_t w_in, int32_t channels, const void* in, void* out, void* stream);
/* out rows [g*49, g*49+49) = pool slot [g][node[g]] of a pool laid out [G][nodes_per_game][49][128]
 * bf16: the gather of search_path[-2].hidden_state (mcts.py:94-96) into the flat layout. */
int mz_conv_gather(int32_t games, int32_t nodes_per_game, const int32_t* node, const void* pool, void* out,
                   void* stream);
/* Linear(6*6*128 -> n_out) (+ReLU) of the heads over the padded state: x [games][6272] bf16,
 * w_packed [n_out][6272] bf16 in the padded channels-last order, out [games][ldo] f32;
 * n_out % 128 == 0.  networks.py:436-439, 470-478. */
int mz_conv_fc_tc(int32_t games, const void* x, const void* w_packed, const float* bias, int32_t n_out,
                  int32_t relu, float* out, int32_t ldo, void* stream);
/* Second head layer Linear(512 -> outs <= 32) on CUDA cores; to_scalar: Config.inverse_transform
 * (config.py:27-33) -> one float per game. */
int mz_conv_head(int32_t games, const float* hidden, int32_t ldh, const float* w2, const float* b2,
                 int32_t outs, int32_t to_scalar, int32_t support_min, int32_t no_target_transform,
                 float* out, int32_t ldo, void* stream);
/* Value / reward head of more than 32 bins on the tensor cores: the second head Linear(512 -> bins)
 * (networks.py:438-440 fc2, 477-483 fc_value_o) followed by Config.inverse_transform (config.py:27-33:
 * softmax expectation over [support_min, support_min + bins), then h^-1 unless no_target_transform):
 * one float per game at out[g * ldo].
 *   hidden  [games][ldh] f32 (the ReLU'd fc1 rows mz_conv_fc_tc writes), 16-byte aligned, ldh % 4 == 0;
 *           rounded to bf16 (nearest even) inside the kernel
 *   w2      [bins][512] bf16 row-major, 16-byte aligned;  b2 [bins] f32
 * 33 <= bins <= 1024 (MZ_ERR_UNSUPPORTED otherwise; 32 bins and fewer are mz_conv_head's).  Float32
 * accumulation, online softmax in a fixed column order: a given input gives the same bits on every run. */
int mz_conv_support_head_tc(int32_t games, const float* hidden, int32_t ldh, const void* w2, const float* b2,
                            int32_t bins, int32_t support_min, int32_t no_target_transform, float* out, int32_t ldo,
                            void* stream);

/* ------------------------------------------------------------------------------------------- */
/* Learner unroll loss (Learner.update_weights, learners.py:182-213; utils.py:53-56)              */
/* ------------------------------------------------------------------------------------------- */
typedef struct mz_loss_cfg {
  int32_t batch;            /* B */
  int32_t num_unroll_steps; /* K (1..31) */
  int32_t num_actions;      /* A */
  int32_t value_min, value_max, reward_min, reward_max; /* supports (config.py:93-94) */
  int32_t no_target_transform;                          /* skip h(x) (learners.py:185-187) */
} mz_loss_cfg;
/* One fused pass over the logits of all unroll steps (train-mode network outputs):
 *   value_logits [K+1][B][V], reward_logits [K][B][R] (steps 1..K), policy_logits [K+1][B][A] f32;
 *   t_values / t_rewards [B][K+1] f32 raw scalars as sample_batch returns them (h(x), config.py:51-54,
 *   and the two-hot projection, config.py:56-68, happen inside), t_policies [B][K+1][A] f32,
 *   is_weights [B] f64 (NULL = ones).
 * Outputs: losses [3] f64 = (is_weights * loss).mean() for reward, value, policy (learners.py:208-210);
 *   row_losses [3][B] f64 workspace (the weighted per-row losses); new_errors [B] f32 =
 *   inverse_value_transform(value_logits[0]) - t_values[:, 0] (learners.py:182-183; may be NULL);
 *   d_*_logits: gradient of (reward + value + policy loss) * 1/K (the hook of learners.py:213) with
 *   respect to each logit, same shapes as the inputs (each may be NULL). */
int mz_unroll_loss(const mz_loss_cfg* c, const float* value_logits, const float* reward_logits,
                   const float* policy_logits, const float* t_values, const float* t_rewards,
                   const float* t_policies, const double* is_weights, float* d_value_logits,
                   float* d_reward_logits, float* d_policy_logits, double* row_losses, double* losses,
                   float* new_errors, void* stream);
/* The same pass for `--no_support` networks (config.py:95-96; learners.py:182-213 with utils.py:61-70), whose
 * value and reward heads emit one scalar: value_out [K+1][B][1], reward_out [K][B][1] f32, the other inputs as
 * above.  Value loss = sum over steps 0..K, reward loss = sum over steps 1..K of l(out, h(target)) (h skipped with
 * no_target_transform), l = MSELoss (scalar_loss 0) or SmoothL1Loss with beta 1 (scalar_loss 1), reduction 'none';
 * policy loss as above.  new_errors [B] = value_out[0] - t_values[:, 0] (raw output minus raw target, no inverse
 * transform).  Gradients with the 1/K scale of learners.py:213, in the operation order of torch's
 * mse_loss_backward / smooth_l1_loss_backward.  Only batch, num_unroll_steps (1..31), num_actions and
 * no_target_transform of c are read.  -1 for a rejected size or scalar_loss, -2 for a NULL required pointer. */
int mz_scalar_unroll_loss(const mz_loss_cfg* c, int32_t scalar_loss, const float* value_out, const float* reward_out,
                          const float* policy_logits, const float* t_values, const float* t_rewards,
                          const float* t_policies, const double* is_weights, float* d_value_out, float* d_reward_out,
                          float* d_policy_logits, double* row_losses, double* losses, float* new_errors, void* stream);

/* Diagnostics: compares the constant-divisor division used by the descent's MinMax normalisation
 * with IEEE division on blocks*256*per_thread pseudo-random operand pairs; adds the number of
 * differing results to *mismatches and the number of pairs checked to *tested (device u64). */
int mz_debug_div_check(uint64_t seed, int32_t blocks, int32_t per_thread, uint64_t* mismatches,
                       uint64_t* tested, void* stream);

/* Games (= warps) per CTA of the warp-per-game step kernel: 1, 2 or 4; 0 (default) = by launch size (one game per
 * CTA from 512 games per launch on: a CTA frees its staged image as soon as its own descent ends and fits beside a
 * network-kernel CTA; four below that).  Results are identical; the parity tests run both. */
int mz_tree_set_games_per_block(int32_t games);

/* Where the step kernel reads a game's tree: 0 (default) = a shared-memory image of its live part whenever the
 * images fit, 1 = the global block directly.  Results are identical; for measurements. */
int mz_debug_set_tree_staging(int32_t mode);

/* The per-simulation kernels (tree step, recurrent network) are launched as programmatic dependents
 * (their prologues overlap the predecessor's tail; griddepcontrol.wait before the first dependent
 * read).  enable = 0 switches back to plain stream-ordered launches.  Default: enabled. */
int mz_set_programmatic_launch(int32_t enable);

/* Library identification. */
const char* mz_version(void);
int32_t mz_compiled_arch(void); /* 100 for sm_100a */

/* ------------------------------------------------------------------------------------------- */
/* Learner network forward / backward for the FCNetwork architecture (learners.py:164-230,      */
/* networks.py:55-174), float32 like the reference.  Weights: torch layout W1 [512][d_in], W2     */
/* [d_out][512] in the flat parameter buffer, plus k-major copies W1T [d_in][512], W2T            */
/* [512][d_out] (mz_learner_transpose) for the forward.  d_in <= 1024, d_out <= 64; dX only for   */
/* d_in <= 128.  A head wider than 128 inputs is the representation head (networks.py:55-68) on   */
/* a wide observation, whose input needs no gradient: its X goes through the kernels' input tile  */
/* in slices of 128 features.                                                                     */
/* ------------------------------------------------------------------------------------------- */
/* Y[r][0:d_out] = W2 relu(W1 X[r][0:d_in] + b1) + b2 -- one head (networks.py:55-119) over `rows` rows. */
int mz_mlp2_forward(int32_t rows, int32_t d_in, int32_t ldx, const float* X, const float* W1T, const float* b1,
                    const float* W2T, const float* b2, int32_t d_out, float* Y, int32_t ldy, void* stream);
/* Backward of the same head: dX[r][0:d_in] += ... (NULL: not needed; must be NULL for d_in > 128), gW1 / gb1 / gW2 /
 * gb2 += (atomics, torch layouts); the 512-wide activation is recomputed from X. */
int mz_mlp2_backward(int32_t rows, int32_t d_in, int32_t ldx, const float* X, const float* W1T, const float* b1,
                     const float* W1, const float* W2, int32_t d_out, const float* dY, int32_t ldy, float* dX,
                     int32_t lddx, float* gW1, float* gb1, float* gW2, float* gb2, void* stream);
/* X_out[r] = [relu(LayerNorm(Y[r][0:d])) | one_hot(actions[r * action_stride], num_actions)]: the hidden state
 * (networks.py:144, 160, 171) and the next head's input row (networks.py:165-166); actions NULL: zeros. */
int mz_ln_relu_forward(int32_t rows, int32_t d, const float* Y, const float* gamma, const float* beta,
                       const int32_t* actions, int32_t action_stride, int32_t num_actions, float* X_out, int32_t ldx,
                       float* mean, float* rstd, void* stream);
/* dY = backward of relu(LayerNorm(Y)) for the incoming gradient scale * dH (scale 0.5: the gradient hook of
 * learners.py:201); ggamma / gbeta += . */
int mz_ln_relu_backward(int32_t rows, int32_t d, const float* dH, int32_t lddh, float scale, const float* Y,
                        const float* H, int32_t ldh, const float* mean, const float* rstd, const float* gamma, float* dY,
                        float* ggamma, float* gbeta, void* stream);
/* out [cols][rows] = in [rows][cols]^T */
int mz_learner_transpose(int32_t rows, int32_t cols, const float* in, float* out, void* stream);
/* torch.optim.AdamW (decoupled != 0) / Adam step over a flat buffer (utils.py:72-83), gradients first multiplied by
 * grad_scale (1 / ranks after a summing all-reduce) and, with clip_norm > 0, clipped to that global norm
 * (learners.py:217-218).  state [3] f32 on the device: step count (incremented here), learning rate, scratch. */
int mz_adam_step(int64_t n, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* state,
                 float beta1, float beta2, float eps, float weight_decay, int32_t decoupled, float grad_scale,
                 float clip_norm, void* stream);

/* ------------------------------------------------------------------------------------------- */
/* The same forward / backward on the tensor cores (csrc/mz_learner_tc.cu): bf16 operands, f32   */
/* accumulation, f32 master weights and gradients.  A training step is FOUR launches: the chain    */
/* representation -> LN -> K x (dynamics -> LN) (learners.py:175-206), the three output heads      */
/* over the stacked hidden states, their backward, and the chain's backward with the 0.5 gradient  */
/* hook of learners.py:201.                                                                        */
/* ------------------------------------------------------------------------------------------- */
/* One matrix to pack as an mma B operand: B[k][n] = src[n * stride_n + k * stride_k] (n < N, k < K), as bf16
 * fragments of 8 (n) x 32 (k) blocks, mz_learner_packed_words(N, K) 32-bit words (zero padded). */
typedef struct mz_pack_job {
  const float* src;
  uint32_t* dst; /* 16-byte aligned */
  int32_t n, k, stride_n, stride_k;
} mz_pack_job;
int64_t mz_learner_packed_words(int32_t n, int32_t k);
/* Up to 24 jobs per launch (a step packs four images per head from the float32 master weights).  A job with src == NULL
 * clears n 32-bit words at dst instead (the gradient buffers a step accumulates into), so one launch prepares the step. */
int mz_learner_pack(int32_t njobs, const mz_pack_job* jobs, void* stream);

/* One head Linear(d_in, 512) -> ReLU -> Linear(512, d_out) (networks.py:55-119); d_in <= 1024, d_out <= 64.
 * d_in > 128 is the representation head (networks.py:55-68) on a wide observation: layer 1 and gw1 run over slices
 * of 128 input features, and there is no dX (w1tp may be NULL).
 * Packed images of W1 [512][d_in] and W2 [d_out][512] (torch layouts):
 *   w1p  (N = 512, K = d_in;  src W1, stride_n d_in, stride_k 1)    layer 1
 *   w2p  (N = d_out, K = 512; src W2, stride_n 512, stride_k 1)     layer 2
 *   w2tp (N = 512, K = d_out; src W2, stride_n 1, stride_k 512)     dH = dY W2        (backward)
 *   w1tp (N = d_in, K = 512;  src W1, stride_n 1, stride_k d_in)    dX = dH W1        (backward)
 * gw1 / gb1 / gw2 / gb2: float32 gradients in torch layouts, accumulated with atomics (backward). */
typedef struct mz_tc_head {
  const uint32_t *w1p, *w2p, *w2tp, *w1tp;
  const float *b1, *b2;
  float *gw1, *gb1, *gw2, *gb2;
  int32_t d_in, d_out;
} mz_tc_head;
/* One head over `rows` rows.  Forward: y[r][0:d_out] = head(x[r][0:d_in]).  Backward: dy in, parameter gradients
 * accumulated, dx[r][0:d_in] += (atomics: several heads may share the rows; NULL = not needed; a job with
 * head.d_in > 128 must pass NULL, else MZ_ERR_BAD_ARG). */
typedef struct mz_tc_job {
  mz_tc_head head;
  int32_t rows, ldx, ldy, lddx;
  const float* x;
  float* y;
  const float* dy;
  float* dx;
} mz_tc_job;
/* Up to three heads in one launch (the value / policy / reward heads of FCNetwork over all unroll steps). */
int mz_heads_forward_tc(int32_t njobs, const mz_tc_job* jobs, void* stream);
int mz_heads_backward_tc(int32_t njobs, const mz_tc_job* jobs, void* stream);

/* The recurrent part: step 0 = `first` (representation, d_in <= 1024; x0 rows of ldx0 floats) on x0, steps
 * 1..steps-1 = `next` (dynamics, d_in = d + num_actions <= 128) on the row
 * [hidden | one_hot(action)] the step before produced.  Per step s: yall[s] = head output (pre-LayerNorm),
 * mean / rstd[s], xs[s][r] = [relu(LN(yall[s][r])) (d values) | one_hot(actions[r * action_stride + s]) for
 * s < action_steps, zeros after]; relu_mask (NULL in inference): the sign bits of the dynamics heads' 512-wide
 * activations in the kernels' fragment order, mz_chain_mask_words(rows, steps) words, for the backward.
 * Backward (the serial part only): dxs[s][r][0:d] = gradient of xs[s] from the output heads; the states the
 * dynamics produced get hook_scale (learners.py:201); per step LayerNorm backward -> dyall[s] (gradient of yall[s])
 * -> dX of the dynamics head -> the step before.  ggamma / gbeta are accumulated here; the parameter gradients of
 * `first` / `next` follow from mz_heads_backward_tc over (x0, dyall[0]) and (xs[0 .. steps-2], dyall[1 .. steps-1])
 * -- all rows in parallel instead of on the chain. */
typedef struct mz_tc_chain {
  mz_tc_head first, next;
  int32_t rows, steps, d, num_actions;
  const float* x0;
  int32_t ldx0;
  const int32_t* actions;
  int32_t action_stride, action_steps;
  const float *gamma, *beta; /* LayerNorm affine (networks.py:144) */
  float* xs;
  int32_t ldxs; /* >= d + num_actions */
  float *yall, *mean, *rstd;
  uint32_t* relu_mask;
  const float* dxs; /* backward */
  float hook_scale;
  float *ggamma, *gbeta;
  float* dyall; /* [steps][rows][d] */
} mz_tc_chain;
int64_t mz_chain_mask_words(int32_t rows, int32_t steps);
int mz_chain_forward_tc(const mz_tc_chain* chain, void* stream);
int mz_chain_backward_tc(const mz_tc_chain* chain, void* stream);

#if defined(MZ_BUILDING) && defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* MZB200_H_ */
