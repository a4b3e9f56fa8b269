// The whole MCTS move of the FCNetwork engine in ONE persistent kernel (MCTS.run, mcts.py:78-102).
//
// A cluster of four CTAs owns a tile of 128 games for all S simulations of a move:
//
//   per simulation   tree phase  : expand + backpropagate of the previous simulation (mcts.py:47-55,
//                                  126-143), pUCT descent of this one (mcts.py:87-92, 104-124), gather of
//                                  the leaf parents' hidden states into the bf16 A operand of the network
//                    net phase   : FCNetwork.recurrent_inference (networks.py:31-34, 122-174) for the 128
//                                  leaves on tcgen05 tensor cores -- the machinery of mz_fcnet_tc.cu
//
// with every hand-off on mbarriers in (distributed) shared memory instead of kernel boundaries:
//
//   tree lanes --st.async--> A1 images of the CTAs that own the dynamics heads      (a1_full)
//   transition head --st.async--> h' (A3) images of the CTAs that own the prediction heads (a3_full)
//   reward / value / policy epilogues --st.async--> output slots of the CTA that owns the game (out_full)
//   h' rows --> bf16 hidden pool in global memory (L2), released to the cluster with the out_full arrival
//
// One head per CTA (rank 0 reward, 1 transition, 2 value, 3 policy), its packed weights resident in shared
// memory for the whole move.  The eight epilogue warps of a CTA double as the tree engine of the 32 games the
// CTA owns (mz_fcs_sparse.cuh: eight lanes per game, its own tree layout; mz_fc_search_export converts a game
// to the arrays of mz_tree_export).  The two phases of a tile are serial by data dependence, so sharing the
// warps costs nothing.  All score arithmetic is IEEE binary64 in the reference's operation order (explicit
// *_rn intrinsics), bit-identical to mz_tree.cu.
//
// Shapes: A <= 32, S <= 63 (fs2::MAX_S), and the shared-memory plan (fs_layout) within kFsMaxSmem; the
// caller runs every other shape on the per-launch kernels (mz_fc_search_supported).
#include <cuda_bf16.h>
#include <math.h>

#include "mz_common.cuh"
#include "mz_exp.cuh"
#include "mz_fc_tc.cuh"
#include "mz_transforms.cuh"

namespace {

using namespace mzfc;

constexpr int FS_THREADS = TC_THREADS;  // warp 0 producer, 1 layer-1 MMA, 2..9 epilogue + tree, 10 layer-2 MMA, 11 store
constexpr int FS_CL = 4;                // CTAs per cluster: one network head each
constexpr int FS_GP = ROWS / FS_CL;     // games whose tree a CTA runs
constexpr int POOL_ROW = 64;            // bf16 elements per hidden-pool row (128 bytes, one line)
constexpr int SP_STRIDE = 33;           // doubles per game of the expansion scratch (>= 32 actions; odd: conflict free)

struct FsParams {
  // network (same packed image as mz_fc_recurrent_tc)
  const uint8_t* chunks;
  const float* tail;
  int k1, A, value_min, reward_min, no_tt;
  // search
  int G, S, two_players, prior_sum_mode;
  double discount, init_score, min_bound, max_bound, noise_frac;
  const double* pb_c;  // [(S+1)^2]
  uint8_t* games;
  long long game_bytes;
  __nv_bfloat16* pool;  // [G][S+1][64]
  // root
  const float* root_logits;
  const uint32_t* legal;
  const double* noise;
  const int8_t* to_play;
  const float* root_hidden;  // [G][50]
  // outputs
  int32_t* visits;
  double* child_visits;
  double* root_value;
  double* minmax;
  // optional
  int32_t *trace_parent, *trace_action, *trace_depth;  // [S][G]
  float *rec_value, *rec_reward, *rec_logits;          // [S][G], [S][G], [S][G][A]
  long long* timeline;                                 // [S][32] clock64 stamps of tile 0 (diagnostics)
  int* error_flag;
};

// ---- small PTX helpers -------------------------------------------------------------------------------
MZ_DEV void fs_timeout(int* err, int code) {
  if (err) atomicExch(err, code);
  __trap();
}
// bounded waits: a protocol error must end the launch (sticky error), never hang the GPU
MZ_DEV void fs_wait(uint64_t* bar, uint32_t parity, int* err, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity))
    if (clock64() - t0 > 6000000000ll) fs_timeout(err, code);
}
MZ_DEV bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
MZ_DEV void fs_wait_cluster(uint64_t* bar, uint32_t parity, int* err, int code) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait_cluster(bar, parity))
    if (clock64() - t0 > 6000000000ll) fs_timeout(err, code);
}
MZ_DEV uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
MZ_DEV void mbar_arrive_remote_release(uint32_t remote_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote_bar) : "memory");
}
MZ_DEV void st_async_b32(uint32_t addr, uint32_t v, uint32_t remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(addr), "r"(v),
               "r"(remote_bar)
               : "memory");
}
MZ_DEV uint4 ldg16(const void* p) { return *reinterpret_cast<const uint4*>(p); }
MZ_DEV uint4 ldg16_cg(const void* p) {  // L2 only: rows written by another CTA of the cluster
  uint4 v;
  asm volatile("ld.global.cg.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}
MZ_DEV double u2d(uint32_t lo, uint32_t hi) { return __hiloint2double((int)hi, (int)lo); }

// x / d through the correctly rounded reciprocal (see mz_tree.cu: div_by_const, bit-identical to IEEE division
// inside the guarded exponent ranges; tests/test_gpu_search.py::test_fast_division)
MZ_DEV double fs_div_by_const(double x, double d, double r) {
  const double q0 = __dmul_rn(x, r);
  const double q1 = __fma_rn(__fma_rn(-q0, d, x), r, q0);
  return __fma_rn(__fma_rn(-q1, d, x), r, q1);
}
MZ_DEV bool fs_exp_in_fast_range(double x) {
  const unsigned h = (unsigned)__double2hiint(x) & 0x7fffffffu;
  return (h - 0x33700000u) <= 0x19000000u;
}
MZ_DEV bool fs_divisor_ok(double d) {
  const unsigned h = (unsigned)__double2hiint(d), l = (unsigned)__double2loint(d);
  return fs_exp_in_fast_range(d) && !(((h & 0xfffffu) == 0xfffffu) && l == 0xffffffffu);
}

// exp() of mz_exp.cuh with the 2 KB table in shared memory: this kernel's shared-memory footprint leaves almost no
// L1, so the table lookups of the global-memory version are L2 round trips on the expansion's critical path.
// Same algorithm and constants (csrc/mz_exp_algo.h), bit-identical results.
MZ_DEV double fs_exp(double x, const unsigned long long* tab) {
  const double ax = fabs(x);
  if (!(ax >= 0x1p-54 && ax < 512.0)) return mz_exp(x);
  const double InvLn2N = 0x1.71547652b82fep7, Shift = 0x1.8p52;
  const double NegLn2hiN = -0x1.62e42fefa0000p-8, NegLn2loN = -0x1.cf79abc9e3b3ap-47;
  const double C2 = 0x1.ffffffffffdbdp-2, C3 = 0x1.555555555543cp-3;
  const double C4 = 0x1.55555cf172b91p-5, C5 = 0x1.1111167a4d017p-7;
  const double z = __dmul_rn(InvLn2N, x);
  double kd = __dadd_rn(z, Shift);
  const unsigned long long ki = (unsigned long long)__double_as_longlong(kd);
  kd = __dsub_rn(kd, Shift);
  const double r = __fma_rn(kd, NegLn2loN, __fma_rn(kd, NegLn2hiN, x));
  const unsigned long long idx = 2 * (ki % 128), top = ki << 45;
  const double tail = __longlong_as_double((long long)tab[idx]);
  const unsigned long long sbits = tab[idx + 1] + top;
  const double r2 = __dmul_rn(r, r);
  const double a = __fma_rn(r, C3, C2), b = __fma_rn(r, C5, C4);
  const double tmp = __fma_rn(__dmul_rn(r2, r2), b, __fma_rn(r2, a, __dadd_rn(tail, r)));
  const double scale = __longlong_as_double((long long)sbits);
  return __fma_rn(scale, tmp, scale);
}

}  // namespace

#include "mz_fcs_sparse.cuh"

namespace {

// shared-memory plan (bytes).  Everything a peer CTA addresses (barriers, output slots, A1 / A3 images) sits at
// the same offset in every CTA of the cluster.  No CTA owns both a dynamics and a prediction head, so the A3
// image shares the A1 region.
__host__ __device__ inline size_t fs_align16(size_t x) { return (x + 15) & ~(size_t)15; }
struct FsLayout {
  size_t a1, w, bars, tail, sh, logit, val, rew, sp, mm, path_n, path_a, depth, total;
  size_t best_ca, node, xmask, links;
  size_t exp_tab, rcp, pbf;
  int ps, a4, s1;
};
__host__ __device__ inline FsLayout fs_layout(int k1, int A, int S) {
  FsLayout L;
  L.a4 = (A + 3) / 4 * 4;
  L.ps = (S + 2 + 15) / 16 * 16;
  L.s1 = (S + 2) & ~1;
  size_t off = 0;
  L.a1 = off; off += (size_t)ROWS * k1 * 2;
  L.w = off; off += (size_t)4 * stage_bytes_for(k1);  // the four chunks of the CTA's head, resident
  L.bars = off; off += 32 * sizeof(uint64_t);
  L.tail = off; off += TAIL_FLOATS * sizeof(float);
  L.sh = off; off += (size_t)ROWS * 128;
  L.logit = off; off += fs_align16((size_t)FS_GP * L.a4 * 4);
  L.val = off; off += fs_align16((size_t)FS_GP * 4);
  L.rew = off; off += fs_align16((size_t)FS_GP * 4);
  L.mm = off; off += (size_t)FS_GP * 16;
  L.path_n = off; off += (size_t)FS_GP * L.ps;
  L.path_a = off; off += (size_t)FS_GP * L.ps;
  L.depth = off; off += fs_align16((size_t)FS_GP);
  L.exp_tab = off; off += 256 * 8;
  L.rcp = off; off += 64 * 8;
  L.pbf = off; off += 64 * 8;
  // exp / reward scratch and the per-node maxima are used in different phases: one region
  const int row = L.s1 > SP_STRIDE ? L.s1 : SP_STRIDE;  // doubles per game (fs2::Smem::row)
  L.sp = off; off += fs_align16((size_t)FS_GP * row * 8);
  L.best_ca = off; off += (size_t)FS_GP * L.s1 * 2;
  L.links = off; off += fs_align16((size_t)FS_GP * L.s1 * 2);
  L.node = off; off += (size_t)FS_GP * L.s1 * 4;
  L.xmask = off; off += (size_t)FS_GP * L.s1 * 4;
  L.total = off;
  return L;
}

// ======================================================================================================
// AL: actions per lane of the tree engine at expansion (eight lanes per game); TL: the instrumented instantiation
// that writes the clock64 phase stamps of FsParams::timeline (launched only when it is set)
template <int AL, bool TL>
__global__ void __maxnreg__(152) fc_search_kernel(FsParams p) {
  constexpr int LANES = fs2::L;
  extern __shared__ __align__(1024) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k1 = p.k1, S = p.S, A = p.A;
  const int stage_bytes = stage_bytes_for(k1);
  const int rank = (int)cluster_ctarank();
  const int tile = (int)blockIdx.x / FS_CL;
  // games whose tree this CTA runs (FS_GP), read from the launched cluster size rather than folded from the constant:
  // with the constant nvcc schedules the tree engine of the 17..24-action instantiation worse (C4 on a B200 at
  // 1000 W: 198 vs 214 M expansions/s)
  const int GP = ROWS / (int)cluster_nctarank();
  // head -> rank: 0 reward, 1 transition (the dynamics heads), 2 value, 3 policy (the prediction heads)
  constexpr int rank_value = 2, rank_policy = 3;
  const bool has_dyn = rank < 2;
  const bool own_reward = rank == 0, own_trans = rank == 1, own_value = rank == rank_value, own_policy = rank == rank_policy;
  int* const err = p.error_flag;

  if (TL && blockIdx.x == 0 && threadIdx.x == 64) {  // diagnostics: kernel entry (cycles, ns)
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    p.timeline[27] = clock64();
    p.timeline[29] = (long long)ns;
  }
  const FsLayout L = fs_layout(k1, A, S);
  uint8_t* sA1 = smem + L.a1;  // A1 image on the dynamics ranks, A3 (h') image on the prediction ranks
  uint8_t* sW = smem + L.w;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
  uint64_t* w_full = bars;            // [4]
  uint64_t* d1_full = bars + 4;       // [2]
  uint64_t* d1_empty = bars + 6;      // [2]
  uint64_t* a2_full = bars + 8;       // [2]
  uint64_t* a2_empty = bars + 10;     // [2]
  uint64_t* a1_full = bars + 12;      // tx: the tile's A1 rows have arrived (st.async from the tree lanes)
  uint64_t* a1_ready = bars + 13;     // epilogue warps -> layer-1 issuer (after the async-proxy fence)
  uint64_t* a3_full = bars + 14;      // tx: h' rows from the transition head
  uint64_t* a3_ready = bars + 15;
  uint64_t* d2_full = bars + 16;
  uint64_t* h_staged = bars + 17;     // transition rank: h' rows are in the staging area
  uint64_t* out_full = bars + 18;     // tx: value / reward / logits of this CTA's games + the pool rows' release
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 20);
  float* sTail = reinterpret_cast<float*>(smem + L.tail);
  uint8_t* sH = smem + L.sh;  // [128][8 x 16 B], block index XOR (row & 7)
  fs2::Smem sm;
  sm.logit = reinterpret_cast<float*>(smem + L.logit);
  sm.val = reinterpret_cast<float*>(smem + L.val);
  sm.rew = reinterpret_cast<float*>(smem + L.rew);
  sm.mm = reinterpret_cast<double*>(smem + L.mm);
  sm.sp = reinterpret_cast<double*>(smem + L.sp);
  sm.best_key = reinterpret_cast<unsigned long long*>(smem + L.sp);
  sm.best_ca = reinterpret_cast<uint16_t*>(smem + L.best_ca);
  sm.first = smem + L.links;
  sm.next = smem + L.links + (size_t)GP * L.s1;
  sm.node = reinterpret_cast<uint32_t*>(smem + L.node);
  sm.xmask = reinterpret_cast<uint32_t*>(smem + L.xmask);
  sm.path_n = smem + L.path_n;
  sm.path_a = smem + L.path_a;
  sm.depth = smem + L.depth;
  sm.ps = L.ps; sm.a4 = L.a4; sm.s1 = L.s1;
  sm.row = L.s1 > SP_STRIDE ? L.s1 : SP_STRIDE;
  unsigned long long* exp_tab_w = reinterpret_cast<unsigned long long*>(smem + L.exp_tab);
  sm.exp_tab = exp_tab_w;
  for (int i = threadIdx.x; i < 256; i += FS_THREADS) exp_tab_w[i] = mz_exp_tab[i];
  double* rcp_w = reinterpret_cast<double*>(smem + L.rcp);
  sm.rcp = rcp_w;
  for (int i = threadIdx.x; i < 64; i += FS_THREADS) rcp_w[i] = i > 0 ? __drcp_rn((double)i) : 0.0;
  double* pbc0_w = reinterpret_cast<double*>(smem + L.pbf);
  sm.pbc0 = pbc0_w;
  for (int i = threadIdx.x; i < 64; i += FS_THREADS) pbc0_w[i] = i <= S ? p.pb_c[(size_t)i * (S + 1)] : 0.0;
  const fs2::Geo geo = fs2::geo(S, A);

  const uint32_t a1_bytes = (uint32_t)(ROWS * k1 * 2), a3_bytes = (uint32_t)(ROWS * K3 * 2);
  const uint32_t out_bytes = (uint32_t)(GP * (8 + 4 * L.a4));

  for (int i = threadIdx.x; i < TAIL_FLOATS; i += FS_THREADS) sTail[i] = p.tail[i];
  if (threadIdx.x == 0) {
    for (int i = 0; i < 4; ++i) mbar_init(&w_full[i], 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&d1_full[i], 1);
      mbar_init(&d1_empty[i], EPI_THREADS / 32);
      mbar_init(&a2_full[i], EPI_THREADS / 32);
      mbar_init(&a2_empty[i], 1);
    }
    mbar_init(a1_full, 1);
    mbar_init(a1_ready, EPI_THREADS / 32);
    mbar_init(a3_full, 1);
    mbar_init(a3_ready, EPI_THREADS / 64);
    mbar_init(d2_full, 1);
    mbar_init(h_staged, EPI_THREADS / 64);
    mbar_init(out_full, 2);
    mbar_fence_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  cluster_sync_all();  // every CTA's barriers exist before anything is sent to them
  const uint32_t tmem = *tmem_ptr;

  if (warp == 0) {
    // ===== producer: the four weight chunks of the CTA's head, loaded once for the whole move =====
    if (lane == 0) {
      for (int c = 0; c < 4; ++c) {
        const int bytes = chunk_geom(4 * rank + c, k1).bytes;
        mbar_arrive_expect_tx(&w_full[c], (uint32_t)bytes);
        bulk_copy_g2s(sW + c * stage_bytes, p.chunks + chunk_offset(4 * rank + c, k1), (uint32_t)bytes, &w_full[c]);
      }
    }
  } else if (warp == 1) {
    // ===== layer-1 MMA issuer (converged warp, one elected lane issues) =====
    const uint32_t a1_addr = smem_u32(sA1), w_addr = smem_u32(sW);
    const uint32_t idesc1 = make_idesc(CHUNK);
    constexpr uint64_t KSTEP = (uint64_t)((2 * (CHUNK / 8) * 128) >> 4);
    int gc = 0;
    for (int sim = 0; sim < S; ++sim) {
      for (int c = 0; c < 4; ++c, ++gc) {
        if (sim == 0) fs_wait(&w_full[c], 0, err, 2);
        if (c == 0) {
          if (has_dyn) fs_wait(a1_ready, sim & 1, err, 3);
          else fs_wait(a3_ready, sim & 1, err, 4);
        }
        fs_wait(&d1_empty[gc & 1], ((gc >> 1) & 1) ^ 1, err, 5);
        tc_fence_after();
        const uint32_t d1 = tmem + COL_D1 + (gc & 1) * CHUNK;
        const uint64_t ad = make_desc(a1_addr, (ROWS / 8) * 128, 128);
        const uint64_t bd = make_desc(w_addr + c * stage_bytes, (CHUNK / 8) * 128, 128);
        if (elect_one()) {
          umma_ss<false>(d1, ad, bd, idesc1);
          if (has_dyn) {  // dynamics: A = [h | onehot | 1] (K = k1)
#pragma unroll 1
            for (int ks = 1; ks < k1 / 16; ++ks) umma_ss<true>(d1, ad + ks * KSTEP, bd + ks * KSTEP, idesc1);
          } else {        // prediction: A = [h' | 1] (K = 64)
#pragma unroll
            for (int ks = 1; ks < K3 / 16; ++ks) umma_ss<true>(d1, ad + ks * KSTEP, bd + ks * KSTEP, idesc1);
          }
          tc_commit(&d1_full[gc & 1]);
        }
        __syncwarp();
      }
    }
  } else if (warp == MMA2_WARP) {
    // ===== layer-2 MMA issuer =====
    const uint32_t w_addr = smem_u32(sW);
    const uint32_t w1_bytes = has_dyn ? CHUNK * k1 * 2 : CHUNK * K3 * 2;
    int gc = 0;
    for (int sim = 0; sim < S; ++sim) {
      for (int c = 0; c < 4; ++c, ++gc) {
        fs_wait(&a2_full[gc & 1], (gc >> 1) & 1, err, 6);
        tc_fence_after();
        const uint32_t a_tm = tmem + COL_A2 + (gc & 1) * (CHUNK / 2);
        const uint32_t b_addr = w_addr + c * stage_bytes + w1_bytes;
        if (elect_one()) {
          if (own_trans) issue_mma2<N_HID>(tmem + COL_D2B, a_tm, b_addr, c == 0);
          else issue_mma2<32>(tmem + ((rank & 1) ? COL_D2B : COL_D2A), a_tm, b_addr, c == 0);
          tc_commit(&a2_empty[gc & 1]);
          if (c == 3) tc_commit(d2_full);
        }
        __syncwarp();
      }
    }
  } else if (warp == STORE_WARP) {
    // ===== h' rows: staging area -> bf16 hidden pool (slot sim + 1), then release them to the cluster =====
    if (own_trans) {
      const int rows_here = min(ROWS, p.G - tile * ROWS);
      for (int sim = 0; sim < S; ++sim) {
        fs_wait(h_staged, sim & 1, err, 7);
#pragma unroll 4
        for (int it = 0; it < ROWS / 4; ++it) {
          const int r = 4 * it + (lane >> 3), kb = lane & 7;
          if (r < rows_here) {
            const uint4 v = *reinterpret_cast<const uint4*>(sH + r * 128 + ((kb ^ (r & 7)) << 4));
            __nv_bfloat16* dst = p.pool + ((size_t)(tile * ROWS + r) * (S + 1) + sim + 1) * POOL_ROW;
            *reinterpret_cast<uint4*>(dst + 8 * kb) = v;
          }
        }
        __syncwarp();
        if (lane < FS_CL) mbar_arrive_remote_release(map_to_cta(smem_u32(out_full), (uint32_t)lane));
        __syncwarp();
      }
    }
  } else {
    // ===== epilogue warps, doubling as the tree engine of this CTA's games =====
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const int grp = (warp - 2) >> 2;              // 0 or 1
    const int row = quarter * 32 + lane;          // the tile row this thread serves in the epilogues
    const int e = (warp - 2) * 32 + lane;         // 0..255
    const uint32_t lane_addr = tmem + ((uint32_t)(quarter * 32) << 16);
    const bool tree_role = e < LANES * GP;
    fs2::Game gm;
    gm.gl = tree_role ? (e / LANES) : 0;
    gm.sub = e % LANES;
    gm.g = tile * ROWS + rank * GP + gm.gl;
    gm.valid = tree_role && gm.g < p.G;
    gm.base = p.games + (size_t)(gm.valid ? gm.g : 0) * p.game_bytes;
    const int my_row = rank * GP + gm.gl;         // tile row of the game this lane works on
    const bool stamp = TL && blockIdx.x == 0 && e == 0;
#define FS_STAMP(sim_, slot_)                                             \
  do {                                                                    \
    if constexpr (TL) {                                                   \
      if (stamp) p.timeline[(size_t)(sim_) * 32 + (slot_)] = clock64();   \
    }                                                                     \
  } while (0)
    // output slots of the game a ROW belongs to (the epilogues send there)
    const uint32_t owner = (uint32_t)(row / GP);
    const int orow = row % GP;
    const uint32_t out_bar_owner = map_to_cta(smem_u32(out_full), owner);

    auto arm = [&]() {  // one thread arms this simulation's transaction barriers
      if (e == 0) {
        if (has_dyn) mbar_arrive_expect_tx(a1_full, a1_bytes);
        else mbar_arrive_expect_tx(a3_full, a3_bytes);
        mbar_arrive_expect_tx(out_full, out_bytes);
      }
    };
    arm();
    FS_STAMP(0, 13);
    if (tree_role) fs2::set_root<AL>(p, sm, gm, geo);
    __syncwarp();
    FS_STAMP(0, 14);

    uint32_t v[32], v2[32];
    int gc = 0, d2ph = 0;
    auto hidden_epilogue = [&]() {  // D1[gc&1] -> relu -> bf16 -> A2[gc&1] (this group's 64 columns)
      const int b = gc & 1;
      const uint32_t ph = (uint32_t)((gc >> 1) & 1);
      fs_wait(&d1_full[b], ph, err, 8);
      tc_fence_after();
      fs_wait(&a2_empty[b], ph ^ 1, err, 9);
      const uint32_t d1 = lane_addr + COL_D1 + b * CHUNK + grp * 64;
      const uint32_t a2 = lane_addr + COL_A2 + b * (CHUNK / 2) + grp * 32;
      tmem_ld32(d1, v);
      tmem_ld32(d1 + 32, v2);
      tmem_wait_ld();
      uint32_t pk[32];
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        pk[j] = pack_bf16_relu(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
        pk[16 + j] = pack_bf16_relu(__uint_as_float(v2[2 * j]), __uint_as_float(v2[2 * j + 1]));
      }
      tmem_st32(a2, pk);
      tmem_wait_st();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&a2_full[b]);
        mbar_arrive(&d1_empty[b]);
      }
      ++gc;
    };

    for (int sim = 0; sim <= S; ++sim) {
      // ---------------- tree phase ----------------
      FS_STAMP(sim < S ? sim : S - 1, sim < S ? 0 : 12);
      if (sim > 0) {
        if (tree_role) {
          fs2::Pre pre;
          fs2::pre_expand<AL>(p, sm, gm, geo, pre);  // overlaps the wait for the outputs
          fs_wait_cluster(out_full, (sim - 1) & 1, err, 10);
          if (sim < S) arm();
          FS_STAMP(sim - 1, 10);
          fs2::expand_backup<TL, AL>(p, sm, gm, geo, sim - 1, pre, stamp ? p.timeline + (size_t)(sim - 1) * 32 : nullptr);
          FS_STAMP(sim - 1, 11);
        }
      }
      if (sim == S) break;
      if (tree_role) {
        int parent, action;
        fs2::descend<TL>(p, sm, gm, geo, sim, parent, action, stamp ? p.timeline + (size_t)sim * 32 : nullptr);
        FS_STAMP(sim, 1);
        // A1 row of the game: bf16([h (50) | onehot(action) (A) | 1 | 0]) as 16-byte blocks of the canonical
        // K-major image, sent to every CTA that owns a dynamics head (ranks 0 and 1)
        const __nv_bfloat16* hrow = p.pool + ((size_t)(gm.valid ? gm.g : 0) * (S + 1) + parent) * POOL_ROW;
        const int kbias = H + A;
        const uint32_t a1_r0 = map_to_cta(smem_u32(sA1), 0), a1_r1 = map_to_cta(smem_u32(sA1), 1);
        const uint32_t bar_r0 = map_to_cta(smem_u32(a1_full), 0), bar_r1 = map_to_cta(smem_u32(a1_full), 1);
        constexpr int NB = (12 + LANES - 1) / LANES;  // 16-byte blocks of the row per lane (k1 / 8 <= 12)
        uint4 blk[NB];
#pragma unroll
        for (int i = 0; i < NB; ++i) {
          const int kb = gm.sub + LANES * i;
          blk[i] = make_uint4(0u, 0u, 0u, 0u);
          if (kb < k1 / 8 && gm.valid && kb <= 6) blk[i] = ldg16_cg(hrow + 8 * kb);
        }
#pragma unroll
        for (int i = 0; i < NB; ++i) {
          const int kb = gm.sub + LANES * i;
          if (kb >= k1 / 8) continue;
          uint4 q = blk[i];
          if (kb >= 6) {
            uint32_t w[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int k = 8 * kb + 2 * j;
              const uint32_t lo = (k - H) == action || k == kbias ? 0x3f80u : 0u;
              const uint32_t hi = (k + 1 - H) == action || (k + 1) == kbias ? 0x3f80u : 0u;
              w[j] = lo | (hi << 16);
            }
            if (kb == 6) w[0] = blk[i].x;  // k = 48, 49: the last two state features
            q = make_uint4(w[0], w[1], w[2], w[3]);
            if (!gm.valid) q = make_uint4(0u, 0u, 0u, 0u);
          }
          const uint32_t off = (uint32_t)canon_off(my_row, 8 * kb, ROWS);
          st_async_v4(a1_r0 + off, q, bar_r0);
          st_async_v4(a1_r1 + off, q, bar_r1);
        }
        FS_STAMP(sim, 2);
      }
      // ---------------- network phase ----------------
      if (has_dyn) {
        fs_wait_cluster(a1_full, sim & 1, err, 11);
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(a1_ready);
        FS_STAMP(sim, 3);
        for (int c = 0; c < 4; ++c) hidden_epilogue();
        fs_wait(d2_full, d2ph & 1, err, 12);
        ++d2ph;
        tc_fence_after();
        FS_STAMP(sim, 4);
        if (own_reward && grp == 1) {
          tmem_ld32(lane_addr + COL_D2A, v);
          tmem_wait_ld();
          const float rew = support_to_scalar_regs(v, sTail + T_REW_B, p.reward_min, p.no_tt);
          st_async_b32(map_to_cta(smem_u32(sm.rew + orow), owner), __float_as_uint(rew), out_bar_owner);
        }
        if (own_trans && grp == 0) {
          float hbuf[64];
          tmem_ld32(lane_addr + COL_D2B, v);
          tmem_ld32(lane_addr + COL_D2B + 32, v2);
          tmem_wait_ld();
          // LayerNorm over the 50 state features in packed float32x2 arithmetic (same sequence as mz_fcnet_tc.cu)
          float2 h2[H / 2];
          {
            const float4* b4 = reinterpret_cast<const float4*>(sTail + T_DYN_B);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float4 b = b4[k];
              h2[2 * k] = __fadd2_rn(make_float2(__uint_as_float(v[4 * k]), __uint_as_float(v[4 * k + 1])), make_float2(b.x, b.y));
              h2[2 * k + 1] = __fadd2_rn(make_float2(__uint_as_float(v[4 * k + 2]), __uint_as_float(v[4 * k + 3])), make_float2(b.z, b.w));
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const float4 b = b4[8 + k];
              h2[16 + 2 * k] = __fadd2_rn(make_float2(__uint_as_float(v2[4 * k]), __uint_as_float(v2[4 * k + 1])), make_float2(b.x, b.y));
              h2[16 + 2 * k + 1] = __fadd2_rn(make_float2(__uint_as_float(v2[4 * k + 2]), __uint_as_float(v2[4 * k + 3])), make_float2(b.z, b.w));
            }
            const float2 b = *reinterpret_cast<const float2*>(sTail + T_DYN_B + 48);
            h2[24] = __fadd2_rn(make_float2(__uint_as_float(v2[16]), __uint_as_float(v2[17])), b);
          }
          float2 s2[4] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
#pragma unroll
          for (int k = 0; k < H / 2; ++k) s2[k & 3] = __fadd2_rn(s2[k & 3], h2[k]);
          const float2 st2 = __fadd2_rn(__fadd2_rn(s2[0], s2[1]), __fadd2_rn(s2[2], s2[3]));
          const float mean = (st2.x + st2.y) * (1.0f / (float)H);
          const float2 nmean = make_float2(-mean, -mean);
          float2 q2[4] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
#pragma unroll
          for (int k = 0; k < H / 2; ++k) {
            h2[k] = __fadd2_rn(h2[k], nmean);
            q2[k & 3] = __ffma2_rn(h2[k], h2[k], q2[k & 3]);
          }
          const float2 qt = __fadd2_rn(__fadd2_rn(q2[0], q2[1]), __fadd2_rn(q2[2], q2[3]));
          const float rstd = rsqrtf((qt.x + qt.y) * (1.0f / (float)H) + 1e-5f);
          const float2 rstd2 = make_float2(rstd, rstd);
          {
            const float2* w2 = reinterpret_cast<const float2*>(sTail + T_LN_W);
            const float2* b2 = reinterpret_cast<const float2*>(sTail + T_LN_B);
#pragma unroll
            for (int k = 0; k < H / 2; ++k) {
              const float2 y = __ffma2_rn(__fmul2_rn(h2[k], rstd2), w2[k], b2[k]);
              hbuf[2 * k] = fmaxf(y.x, 0.0f);
              hbuf[2 * k + 1] = fmaxf(y.y, 0.0f);
            }
          }
          hbuf[H] = 1.0f;  // column H feeds the folded first-layer bias of the prediction heads
#pragma unroll
          for (int j = H + 1; j < 64; ++j) hbuf[j] = 0.0f;
          // h' as bf16: the A operand of the prediction layer of the CTAs that own those heads, and the pool row
          const uint32_t pr0 = (uint32_t)rank_value, pr1 = (uint32_t)rank_policy;
          const uint32_t a3_p0 = map_to_cta(smem_u32(sA1), pr0), a3_p1 = map_to_cta(smem_u32(sA1), pr1);
          const uint32_t bar_p0 = map_to_cta(smem_u32(a3_full), pr0), bar_p1 = map_to_cta(smem_u32(a3_full), pr1);
          uint4 q[K3 / 8];
#pragma unroll
          for (int kb = 0; kb < K3 / 8; ++kb) {
            q[kb] = make_uint4(pack_bf16(hbuf[8 * kb], hbuf[8 * kb + 1]), pack_bf16(hbuf[8 * kb + 2], hbuf[8 * kb + 3]),
                               pack_bf16(hbuf[8 * kb + 4], hbuf[8 * kb + 5]), pack_bf16(hbuf[8 * kb + 6], hbuf[8 * kb + 7]));
            const uint32_t off = (uint32_t)canon_off(row, 8 * kb, ROWS);
            st_async_v4(a3_p0 + off, q[kb], bar_p0);
            st_async_v4(a3_p1 + off, q[kb], bar_p1);
          }
#pragma unroll
          for (int kb = 0; kb < K3 / 8; ++kb)
            *reinterpret_cast<uint4*>(sH + row * 128 + ((kb ^ (row & 7)) << 4)) = q[kb];
          __syncwarp();
          if (lane == 0) mbar_arrive(h_staged);  // the store warp takes it from here
        }
        FS_STAMP(sim, 5);
      } else {
        if (grp == 0) {
          fs_wait_cluster(a3_full, sim & 1, err, 13);
          fence_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive(a3_ready);
        }
        FS_STAMP(sim, 6);
        for (int c = 0; c < 4; ++c) hidden_epilogue();
        fs_wait(d2_full, d2ph & 1, err, 14);
        ++d2ph;
        tc_fence_after();
        FS_STAMP(sim, 7);
        if (own_value && grp == 0) {
          tmem_ld32(lane_addr + COL_D2A, v);
          tmem_wait_ld();
          const float val = support_to_scalar_regs(v, sTail + T_VAL_B, p.value_min, p.no_tt);
          st_async_b32(map_to_cta(smem_u32(sm.val + orow), owner), __float_as_uint(val), out_bar_owner);
        }
        if (own_policy && grp == 1) {
          tmem_ld32(lane_addr + COL_D2B, v);
          tmem_wait_ld();
          const uint32_t dst = map_to_cta(smem_u32(sm.logit + orow * L.a4), owner);
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            if (4 * j4 < L.a4) {
              const float4 b = *reinterpret_cast<const float4*>(sTail + T_POL_B + 4 * j4);
              const uint4 o = make_uint4(__float_as_uint(__uint_as_float(v[4 * j4]) + b.x),
                                         __float_as_uint(__uint_as_float(v[4 * j4 + 1]) + b.y),
                                         __float_as_uint(__uint_as_float(v[4 * j4 + 2]) + b.z),
                                         __float_as_uint(__uint_as_float(v[4 * j4 + 3]) + b.w));
              st_async_v4(dst + 16 * j4, o, out_bar_owner);
            }
          }
        }
        tc_fence_before();
        FS_STAMP(sim, 8);
      }
    }
    if (tree_role) fs2::root_stats(p, sm, gm, geo);
    FS_STAMP(S - 1, 15);
#undef FS_STAMP
  }

  __syncthreads();
  cluster_sync_all();  // no CTA leaves while a peer may still address its shared memory
  if (TL && blockIdx.x == 0 && threadIdx.x == 64) {  // diagnostics: kernel exit
    unsigned long long ns;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns));
    p.timeline[28] = clock64();
    p.timeline[30] = (long long)ns;
  }
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}

// one game of the fused engine's tree as the arrays of mz_tree_export (tests / the Node facade)
__global__ void fs2_export_kernel(const uint8_t* games, long long game_bytes, int S, int A, int game, double* prior,
                                  int32_t* child, double* vsum, int32_t* visit, float* reward, double* q_out) {
  const fs2::Geo G = fs2::geo(S, A);
  const uint8_t* base = games + (size_t)game * game_bytes;
  const uint32_t legal = *reinterpret_cast<const uint32_t*>(base + 16);
  for (int i = threadIdx.x; i < (S + 1) * A; i += blockDim.x) {
    const int n = i / A, a = i % A;
    if (prior) prior[i] = *reinterpret_cast<const double*>(base + G.pri + ((size_t)n * G.a2 + a) * 8);
    if (child) child[i] = (n == 0 && !((legal >> a) & 1u)) ? MZ_CHILD_ILLEGAL : MZ_CHILD_UNEXPANDED;
    if (q_out) q_out[i] = 0.0;
  }
  __syncthreads();
  for (int n = threadIdx.x; n <= S; n += blockDim.x) {
    const uint2 m = *reinterpret_cast<const uint2*>(base + G.meta + 8 * n);
    const uint4 o = *reinterpret_cast<const uint4*>(base + G.own + 16 * n);
    if (vsum) vsum[n] = u2d(o.x, o.y);
    if (reward) reward[n] = __uint_as_float(o.z);
    if (visit) visit[n] = (int)(m.x & 0xffu);
    if (n > 0 && (m.x & 0xffu) > 0) {
      const int par = (int)(m.x >> 24), act = (int)((m.x >> 8) & 0xffu);
      if (child) child[par * A + act] = n;
      if (q_out) q_out[par * A + act] = *reinterpret_cast<const double*>(base + G.edge + 32 * n + 8);
    }
  }
}

int fs_k1_for(int A) { return (H + A + 1 + 15) / 16 * 16; }
constexpr size_t kFsMaxSmem = 232448;

// the shapes the kernel takes: S <= 63 (fs2::MAX_S) and a shared-memory plan within the opt-in maximum
bool fs_fits(int S, int A) {
  return A >= 1 && A <= 32 && S >= 1 && S <= fs2::MAX_S && fs_layout(fs_k1_for(A), A, S).total <= kFsMaxSmem;
}

template <int AL, bool TL>
int fs_launch(const FsParams& p, size_t smem, void* stream) {
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(fc_search_kernel<AL, TL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kFsMaxSmem);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  const int tiles = (p.G + ROWS - 1) / ROWS;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(tiles * FS_CL);
  cfg.blockDim = dim3(FS_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute lattr[2];
  lattr[0].id = cudaLaunchAttributeClusterDimension;
  lattr[0].val.clusterDim.x = FS_CL;
  lattr[0].val.clusterDim.y = 1;
  lattr[0].val.clusterDim.z = 1;
  lattr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  lattr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = lattr;
  // (launching it as a programmatic dependent of the initial-inference kernel was measured: no gain -- 204.5 vs
  // 203.7 M expansions/s on C4, slightly slower on C1 / C3 -- so it is a plain launch)
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, fc_search_kernel<AL, TL>, p);
  if (e != cudaSuccess) return (int)e;
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

}  // namespace

extern "C" {

int64_t mz_fc_search_game_bytes(int32_t S, int32_t A) {
  if (!fs_fits(S, A)) return MZ_ERR_UNSUPPORTED;
  return fs2::geo(S, A).bytes;
}

int32_t mz_fc_search_pool_row(void) { return POOL_ROW; }

int mz_fc_search_supported(int32_t S, int32_t A) { return fs_fits(S, A) ? 1 : 0; }

int mz_fc_search(const mz_fc_search_args* a, void* stream) {
  if (!a || !a->weights || !a->packed || !a->tail || !a->games || !a->pb_c_table || !a->pool || !a->root_logits ||
      !a->root_hidden)
    return MZ_ERR_BAD_ARG;
  const mz_fc_weights* w = a->weights;
  if (a->num_games < 1 || a->num_simulations < 1) return MZ_ERR_BAD_ARG;
  if (w->value_bins > 32 || w->reward_bins > 32 || w->no_support || !fs_fits(a->num_simulations, w->num_actions))
    return MZ_ERR_UNSUPPORTED;
  if (a->game_bytes < mz_fc_search_game_bytes(a->num_simulations, w->num_actions)) return MZ_ERR_BAD_ARG;
  FsParams p;
  p.chunks = (const uint8_t*)a->packed;
  p.tail = a->tail;
  p.k1 = fs_k1_for(w->num_actions);
  p.A = w->num_actions;
  p.value_min = w->value_min;
  p.reward_min = w->reward_min;
  p.no_tt = w->no_target_transform;
  p.G = a->num_games;
  p.S = a->num_simulations;
  p.two_players = a->two_players;
  p.prior_sum_mode = a->prior_sum_mode;
  p.discount = a->discount;
  p.init_score = a->init_value_score;
  p.min_bound = a->min_bound;
  p.max_bound = a->max_bound;
  p.noise_frac = a->noise_frac;
  p.pb_c = a->pb_c_table;
  p.games = a->games;
  p.game_bytes = a->game_bytes;
  p.pool = (__nv_bfloat16*)a->pool;
  p.root_logits = a->root_logits;
  p.legal = a->legal_mask;
  p.noise = a->noise;
  p.to_play = a->root_to_play;
  p.root_hidden = a->root_hidden;
  p.visits = a->visits;
  p.child_visits = a->child_visits;
  p.root_value = a->root_value;
  p.minmax = a->minmax;
  p.trace_parent = a->trace_parent;
  p.trace_action = a->trace_action;
  p.trace_depth = a->trace_depth;
  p.rec_value = a->rec_value;
  p.rec_reward = a->rec_reward;
  p.rec_logits = a->rec_logits;
  p.timeline = (long long*)a->timeline;
  p.error_flag = a->error_flag;
  const size_t smem = fs_layout(p.k1, p.A, p.S).total;
  const int AL = (p.A + fs2::L - 1) / fs2::L;
  if (p.timeline) {
    if (AL <= 1) return fs_launch<1, true>(p, smem, stream);
    if (AL <= 2) return fs_launch<2, true>(p, smem, stream);
    if (AL <= 3) return fs_launch<3, true>(p, smem, stream);
    return fs_launch<4, true>(p, smem, stream);
  }
  if (AL <= 1) return fs_launch<1, false>(p, smem, stream);
  if (AL <= 2) return fs_launch<2, false>(p, smem, stream);
  if (AL <= 3) return fs_launch<3, false>(p, smem, stream);
  return fs_launch<4, false>(p, smem, stream);
}

int mz_fc_search_export(const mz_fc_search_args* a, int32_t game, double* prior, int32_t* child, double* vsum,
                        int32_t* visit, float* reward, double* q, void* stream) {
  if (!a || !a->games || !a->weights || game < 0 || game >= a->num_games) return MZ_ERR_BAD_ARG;
  fs2_export_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(a->games, a->game_bytes, a->num_simulations,
                                                         a->weights->num_actions, game, prior, child, vsum, visit,
                                                         reward, q);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

}  // extern "C"
