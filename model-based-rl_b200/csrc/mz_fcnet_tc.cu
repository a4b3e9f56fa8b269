// FCNetwork.recurrent_inference on the 5th-generation tensor cores (tcgen05 + TMEM), bf16 operands,
// fp32 accumulation.  One CTA evaluates the whole network for 128 rows (games):
//
//   dynamics   : [h | onehot(a)] (K1) --W1--> 2 x 512 --relu--> W2 --> reward logits (32) , h' (64)
//   LayerNorm + ReLU on h'  (fp32, one thread per row), reward = softmax-expectation + h^-1
//   prediction : h' (K3 = 64) --W3--> 2 x 512 --relu--> W4 --> value logits (32), policy logits (32)
//
// That is the narrow head geometry (A <= 32, supports <= 32 bins).  The wide one (mzfc::WideGeom: more actions or
// bins, up to 64) pads reward, value and policy logits to 64 columns each; the kernel and the packing are
// templated on the geometry, and the host picks it from the weights (tc_geometry).
//
// The 512-wide hidden layers are processed in 16 chunks of 128 features.  Per chunk c:
//   MMA1(c): D1[c&1] (TMEM, 128 lanes x 128 cols) = A(128 x K) * W1c^T          (tcgen05.mma)
//   EPI(c) : D1[c&1] -> registers (tcgen05.ld) -> relu, bf16 -> A2[c&1] back in TMEM (tcgen05.st)
//   MMA2(c): D2 (TMEM) += A2[c&1](128 x 128, TMEM operand) * W2c^T
// Keeping the layer-2 A operand in TMEM matters: with both operands in shared memory every
// M = 128 instruction is bound by the 4 KB A read (~140 cycles measured, independent of N), which
// made the 128 narrow (N = 32 / 64) layer-2 instructions the bottleneck.
// Weight chunks are pre-packed in global memory as the exact shared-memory image the MMA reads
// (UMMA canonical K-major layout, no swizzle) and streamed through a 3-stage ring with one
// cp.async.bulk per chunk; the pipeline is driven by mbarriers (TMA -> MMA -> epilogue -> MMA).
//
// Warp roles (352 threads): warp 0 = TMEM allocation + bulk-copy producer, warp 1 = layer-1 MMA
// issuer, warps 2..9 = two epilogue groups of four warps (TMEM lane quarter = warp % 4), warp 10 =
// layer-2 MMA issuer (each issuer: converged warp, one elected lane issues).
//
// Reference semantics: networks.py:31-34, 122-174 (FCNetwork), config.py:27-33.
#include <cuda_bf16.h>
#include <math.h>
#include <stdlib.h>

#include "mz_common.cuh"
#include "mz_transforms.cuh"

#include "mz_fc_tc.cuh"

namespace {

using namespace mzfc;

struct TcParams {
  const uint8_t* chunks;  // packed weights
  const float* tail;
  int k1, num_actions, value_bins, reward_bins, value_min, reward_min, no_tt;
  int batch;
  const float* hidden_in;
  long long in_row_stride;
  const int32_t* in_index;
  const int32_t* actions;
  float* hidden_out;
  long long out_row_stride, out_offset;
  float *value, *reward, *logits;
  long long* trace;  // optional per-phase clock64() stamps of CTA 0 (diagnostics), or nullptr
  // initial_inference mode (networks.py:26-29): chunk0 = 4 skips the reward head, the first head is
  // the representation (A1 = [obs | 1], K = k1), then LayerNorm / ReLU and the prediction heads
  int chunk0;        // 0: recurrent_inference (16 chunks), 4: initial_inference (12 chunks)
  int stages;        // weight-ring depth actually used (<= MAX_STAGES)
  const float* obs;  // [batch][obs_dim] (initial mode)
  int obs_dim;
  // split != 0: the kernel runs as clusters of two CTAs per 128 rows; rank 0 evaluates the reward and
  // value heads, rank 1 the transition and policy heads (8 chunks each instead of 16) and hands h'
  // to rank 0 through distributed shared memory
  int split;
  int trace_block;   // which CTA writes the diagnostic stamps
};

// trace slots: [0,64) epilogue thread (row 0), [64,192) MMA thread, [192,224) producer
#define TC_STAMP(slot)                                              \
  do {                                                              \
    if (p.trace && blockIdx.x == p.trace_block) p.trace[(slot)] = clock64();    \
  } while (0)


template <class G>
__global__ void __maxnreg__(152) fc_recurrent_tc_kernel(TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (p.trace && threadIdx.x == 0 && blockIdx.x < 64) {  // wall-clock entry time of every CTA (ns)
    unsigned long long tns;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(tns));
    p.trace[256 + 2 * blockIdx.x] = (long long)tns;
  }
  const int k1 = p.k1;
  const int stage_bytes = stage_bytes_for<G>(k1);
  const bool split = p.split != 0;
  const int rank = split ? (int)cluster_ctarank() : 0;
  const int tile = split ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;  // which 128 rows
  // epilogue threads request their row's gather index / action before the set-up barrier
  int pre_idx = 0, pre_act = 0;
  if (warp >= 2 && warp < MMA2_WARP) {
    // everything this kernel reads from its predecessor (gather index, actions, hidden states) is
    // read by the epilogue warps, after this point; weights, barriers and TMEM do not depend on it
    pdl_wait();
    pdl_trigger();
    const int g0 = tile * ROWS + (warp & 3) * 32 + lane;
    const int gc0 = g0 < p.batch ? g0 : p.batch - 1;
    if (!p.obs) {
      pre_idx = p.in_index ? p.in_index[gc0] : 0;
      pre_act = p.actions[gc0];
    }
  }
  // carve shared memory
  uint8_t* sA1 = smem;                                  // [128 x k1] bf16 (A of the dynamics layer)
  uint8_t* sW = sA1 + ROWS * k1 * 2;                    // STAGES x stage_bytes
  const int STAGES = p.stages, c0 = p.chunk0;
  const int nch = split ? NCHUNK / 2 : NCHUNK - c0;  // chunks this CTA runs
  const int c_mid = split ? 4 : 8 - c0;               // first chunk of the prediction phase
  // running chunk index -> canonical chunk id (head = id >> 2: reward, transition, value, policy)
  auto canon = [&](int c) { return split ? (c < 4 ? 4 * rank + c : 8 + 4 * rank + (c - 4)) : c + c0; };
  const bool own_reward = !split || rank == 0, own_hidden = !split || rank == 1;
  const bool own_value = own_reward, own_logits = own_hidden;
  uint8_t* sA3 = sW + STAGES * stage_bytes;             // [128 x 64] bf16: h' (A of the prediction layer)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sA3 + ROWS * K3 * 2);
  uint64_t* w_full = bars;            // [STAGES]
  uint64_t* w_empty = bars + 4;       // [STAGES]
  uint64_t* d1_full = bars + 8;       // [2]
  uint64_t* d1_empty = bars + 10;     // [2]
  uint64_t* a2_full = bars + 12;      // [2]
  uint64_t* a2_empty = bars + 14;     // [2]
  uint64_t* a1_ready = bars + 16;
  uint64_t* a3_ready = bars + 17;
  uint64_t* d2_full = bars + 18;
  uint64_t* h_staged = bars + 19;
  uint64_t* a3_remote = bars + 20;    // rank 0 of a split pair: h' rows have arrived from rank 1
  uint64_t* h_stored = bars + 21;     // the store warp is done with sOut (the logits reuse it)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 22);
  float* sTail = reinterpret_cast<float*>(bars + 24);   // 16-byte aligned: second-layer biases + LayerNorm affine
  float* sOut = sTail + G::TAIL_FLOATS;                 // [128][51]: row-major staging of h'
  float* sLog = sOut;                                   // [128][A]: the logits reuse it at the very end
  for (int i = threadIdx.x; i < G::TAIL_FLOATS; i += TC_THREADS) sTail[i] = p.tail[i];

  if (threadIdx.x == 0) {
    for (int i = 0; i < MAX_STAGES; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1); }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&d1_full[i], 1);
      mbar_init(&d1_empty[i], EPI_THREADS / 32);  // one arrival per epilogue warp (after __syncwarp): 512
      mbar_init(&a2_full[i], EPI_THREADS / 32);   // per-thread arrivals per chunk serialise on the barrier word
      mbar_init(&a2_empty[i], 1);
    }
    mbar_init(a1_ready, EPI_THREADS / 32);
    mbar_init(a3_ready, EPI_THREADS / 64);
    mbar_init(d2_full, 1);
    mbar_init(h_staged, EPI_THREADS / 64);
    mbar_init(a3_remote, 1);
    if (split && rank == 0) mbar_arrive_expect_tx(a3_remote, ROWS * K3 * 2);  // the peer's st.async bytes
    mbar_init(h_stored, 1);
    mbar_fence_init();
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (split) cluster_sync_all();  // the peer's barriers exist before anything is sent to them
  const uint32_t tmem = *tmem_ptr;
  if (threadIdx.x == 32) TC_STAMP(0);

  if (warp == 0) {
    // ===== producer: stream the 16 weight chunks through the ring =====
    if (lane == 0) {
      const size_t base = chunk_offset<G>(c0, k1);
      int st = 0, n = 0;  // ring slot and round, advanced incrementally (STAGES is a run-time value)
      for (int c = 0; c < nch; ++c, st = (st + 1 == STAGES ? 0 : st + 1), n += (st == 0)) {
        const int cc = canon(c);
        const ChunkGeom g = chunk_geom<G>(cc, k1);
        mbar_wait(&w_empty[st], (n & 1) ^ 1);
        TC_STAMP(192 + c);
        mbar_arrive_expect_tx(&w_full[st], (uint32_t)g.bytes);
        bulk_copy_g2s(sW + st * stage_bytes, p.chunks + (chunk_offset<G>(cc, k1) - base), (uint32_t)g.bytes,
                      &w_full[st]);
      }
    }
  } else if (warp == 1) {
    // ===== layer-1 MMA issuer: the whole warp walks the pipeline converged (waits, descriptor
    // arithmetic in uniform registers); one elected lane issues tcgen05.mma / tcgen05.commit =====
    const uint32_t a1_addr = smem_u32(sA1);
    const uint32_t w_addr = smem_u32(sW);
    const uint32_t idesc1 = make_idesc(CHUNK);
    constexpr uint64_t KSTEP = (uint64_t)((2 * (CHUNK / 8) * 128) >> 4);  // two K core-matrix columns
    int st = 0, round = 0;
    for (int c = 0; c < nch; ++c, st = (st + 1 == STAGES ? 0 : st + 1), round += (st == 0)) {
      const int cc = canon(c);
      if (lane == 0) TC_STAMP(64 + 8 * c + 0);
      mbar_wait(&w_full[st], round & 1);
      if (c == 0) mbar_wait(a1_ready, 0);
      if (c == c_mid) mbar_wait(a3_ready, 0);
      mbar_wait(&d1_empty[c & 1], ((c >> 1) & 1) ^ 1);
      tc_fence_after();
      if (lane == 0) TC_STAMP(64 + 8 * c + 1);
      const uint32_t d1 = tmem + COL_D1 + (c & 1) * CHUNK;
      const uint64_t bd = make_desc(w_addr + st * stage_bytes, (CHUNK / 8) * 128, 128);
      if (elect_one()) {
        if (cc < 8) {  // dynamics / representation: A = [h | onehot | 1] or [obs | 1] from shared memory, K = k1
          const uint64_t ad = make_desc(a1_addr, (ROWS / 8) * 128, 128);
          umma_ss<false>(d1, ad, bd, idesc1);
#pragma unroll 1
          for (int ks = 1; ks < k1 / 16; ++ks) umma_ss<true>(d1, ad + ks * KSTEP, bd + ks * KSTEP, idesc1);
        } else {      // prediction: A = [h' | 1] from shared memory (written locally or by the peer CTA), K = 64
          const uint64_t ad = make_desc(smem_u32(sA3), (ROWS / 8) * 128, 128);
          umma_ss<false>(d1, ad, bd, idesc1);
#pragma unroll
          for (int ks = 1; ks < K3 / 16; ++ks) umma_ss<true>(d1, ad + ks * KSTEP, bd + ks * KSTEP, idesc1);
        }
        tc_commit(&d1_full[c & 1]);
      }
      __syncwarp();
      if (lane == 0) TC_STAMP(64 + 8 * c + 3);
    }
  } else if (warp == MMA2_WARP) {
    // ===== layer-2 MMA issuer: D2 += A2[c&1] (TMEM) * W2c^T as soon as the epilogue has produced
    // A2[c&1]; runs concurrently with the layer-1 issuer so neither waits behind the other =====
    const uint32_t w_addr = smem_u32(sW);
    const uint32_t w1_bytes_dyn = CHUNK * k1 * 2, w1_bytes_pred = CHUNK * K3 * 2;
    int st = 0;
    for (int c = 0; c < nch; ++c, st = (st + 1 == STAGES ? 0 : st + 1)) {
      const int cc = canon(c), head = cc >> 2;
      mbar_wait(&a2_full[c & 1], (c >> 1) & 1);
      tc_fence_after();
      if (lane == 0) TC_STAMP(64 + 8 * c + 4);
      const uint32_t a_tm = tmem + COL_A2 + (c & 1) * (CHUNK / 2);
      const uint32_t b_addr = w_addr + st * stage_bytes + (cc < 8 ? w1_bytes_dyn : w1_bytes_pred);
      if (elect_one()) {
        if (head == 1) issue_mma2<N_HID>(tmem + G::COL_D2B, a_tm, b_addr, (cc & 3) == 0);
        else issue_mma2<G::NB>(tmem + ((head & 1) ? G::COL_D2B : G::COL_D2A), a_tm, b_addr, (cc & 3) == 0);
        tc_commit(&w_empty[st]);       // chunk c's weights are no longer needed
        tc_commit(&a2_empty[c & 1]);   // A2 buffer may be overwritten
        if (c == c_mid - 1 || c == nch - 1) tc_commit(d2_full);
      }
      __syncwarp();
      if (lane == 0) TC_STAMP(64 + 8 * c + 6);
    }
  } else if (warp == STORE_WARP) {
    // ===== h' rows: shared-memory staging area -> hidden pool, one contiguous 200-byte row per
    // pair of store instructions (a per-thread row store would touch 32 lines per instruction) =====
    if (own_hidden) {
    mbar_wait(h_staged, 0);
    const int rows_here = min(ROWS, p.batch - tile * ROWS);
#pragma unroll 4
    for (int r = 0; r < rows_here; ++r) {
      float* dst = p.hidden_out + (size_t)(tile * ROWS + r) * p.out_row_stride + p.out_offset;
      dst[lane] = sOut[r * OUT_STRIDE + lane];
      if (lane < H - 32) dst[32 + lane] = sOut[r * OUT_STRIDE + 32 + lane];
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(h_stored);
    }
  } else {
    // ===== epilogue warps: two groups of four warps; within a group one thread per row.
    // Both groups split every chunk's 128 accumulator columns; for the row-wise work group 0 takes
    // the state path (gather, LayerNorm, value), group 1 the action / reward / policy path. =====
    const int quarter = warp & 3;                 // TMEM lane quarter this warp may access
    const int grp = (warp - 2) >> 2;              // 0 or 1
    const int row = quarter * 32 + lane;
    const int g = tile * ROWS + row;
    const bool live = g < p.batch;
    const int gc = live ? g : p.batch - 1;
    const uint32_t lane_addr = tmem + ((uint32_t)(quarter * 32) << 16);
    const bool stamp = (row == 0 && grp == 0);

    if (p.obs) {
      // --- initial_inference: A1 = bf16([obs (obs_dim) | 1 (bias input) | 0]); each warp walks 16 of
      // its quarter's rows, lanes stride over the columns (coalesced row reads) ---
      // Four rows at a time with every load of the batch in flight before the first store: the row-by-row loop
      // this replaces exposed one L2 / HBM round trip per 128-byte segment (80 per warp: 25 of the kernel's 33 us).
      const int r0 = quarter * 32 + grp * 16;
      constexpr int RB = 4, KI = 8;  // rows per batch, 32-column segments per row held in registers (k1 <= 256)
      for (int i0 = 0; i0 < 16; i0 += RB) {
        float x[RB][KI];
#pragma unroll
        for (int ii = 0; ii < RB; ++ii) {
          const int gr = min(tile * ROWS + r0 + i0 + ii, p.batch - 1);
          const float* orow = p.obs + (size_t)gr * p.obs_dim;
#pragma unroll
          for (int j = 0; j < KI; ++j) {
            const int k = lane + 32 * j;
            x[ii][j] = k < p.obs_dim ? __ldg(orow + k) : (k == p.obs_dim ? 1.0f : 0.0f);
          }
        }
#pragma unroll
        for (int ii = 0; ii < RB; ++ii) {
#pragma unroll
          for (int j = 0; j < KI; ++j) {
            const int k = lane + 32 * j;
            if (k < k1) *reinterpret_cast<__nv_bfloat16*>(sA1 + canon_off(r0 + i0 + ii, k, ROWS)) = __float2bfloat16_rn(x[ii][j]);
          }
        }
        for (int ii = 0; ii < RB; ++ii) {  // observations wider than 255 features: the rest, row by row
          const int gr = min(tile * ROWS + r0 + i0 + ii, p.batch - 1);
          const float* orow = p.obs + (size_t)gr * p.obs_dim;
          for (int k = 32 * KI + lane; k < k1; k += 32) {
            const float v = k < p.obs_dim ? __ldg(orow + k) : (k == p.obs_dim ? 1.0f : 0.0f);
            *reinterpret_cast<__nv_bfloat16*>(sA1 + canon_off(r0 + i0 + ii, k, ROWS)) = __float2bfloat16_rn(v);
          }
        }
      }
    } else {
      // --- A1 = bf16([h (50) | onehot(action) (A) | 1 (bias input) | 0]) ---
      // k < 48: both warps of a quarter walk 16 of its 32 rows each, 24 lanes load one float2 per row
      // (coalesced 192 B); all 16 row loads are in flight before the first store (one L2 round trip)
      const float* src = p.hidden_in + (size_t)gc * p.in_row_stride + (size_t)pre_idx * H;
      float2 h4849 = make_float2(0.0f, 0.0f);
      if (grp == 1) h4849 = *reinterpret_cast<const float2*>(src + 48);  // in flight with the row loads below
      {
        const unsigned long long my_src = (unsigned long long)src;
        float2 f2[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const unsigned long long rs = __shfl_sync(MZ_FULL, my_src, grp * 16 + i);
          f2[i] = lane < 24 ? *reinterpret_cast<const float2*>(reinterpret_cast<const float*>(rs) + 2 * lane)
                            : make_float2(0.0f, 0.0f);
        }
        if (lane < 24) {
#pragma unroll
          for (int i = 0; i < 16; ++i)
            *reinterpret_cast<uint32_t*>(sA1 + canon_off(quarter * 32 + grp * 16 + i, 2 * lane, ROWS)) =
                pack_bf16(f2[i].x, f2[i].y);
        }
      }
      if (grp == 1) {
      // k >= 48: the row's own thread (last two state features, one-hot action, constant 1)
      const int act = pre_act;
      const int kbias = H + p.num_actions;
      const int a_off = (row >> 3) * 128 + (row & 7) * 16;
      for (int kb = 6; kb < k1 / 8; ++kb) {
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int k = kb * 8 + j;
          f[j] = k == 48 ? h4849.x : (k == 49 ? h4849.y : (((k - H) == act || k == kbias) ? 1.0f : 0.0f));
        }
        uint4 q = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]),
                             pack_bf16(f[6], f[7]));
        *reinterpret_cast<uint4*>(sA1 + kb * (ROWS / 8) * 128 + a_off) = q;
      }
      }
    }
    if (lane == 0) TC_STAMP(224 + warp);
    fence_async_smem();
    if (lane == 0) TC_STAMP(236 + warp);
    __syncwarp();
    if (lane == 0) mbar_arrive(a1_ready);
    if (stamp) TC_STAMP(1);

    uint32_t v[32], v2[32];
    auto hidden_epilogue = [&](int c) {  // D1[c&1] -> relu -> bf16 -> A2[c&1] (this group's 64 columns)
      mbar_wait(&d1_full[c & 1], (c >> 1) & 1);
      tc_fence_after();
      mbar_wait(&a2_empty[c & 1], ((c >> 1) & 1) ^ 1);
      if (stamp) TC_STAMP(4 + 2 * c);
      const uint32_t d1 = lane_addr + COL_D1 + (c & 1) * CHUNK + grp * 64;
      const uint32_t a2 = lane_addr + COL_A2 + (c & 1) * (CHUNK / 2) + grp * 32;
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
        mbar_arrive(&a2_full[c & 1]);
        mbar_arrive(&d1_empty[c & 1]);
      }
      if (stamp) TC_STAMP(5 + 2 * c);
    };

    for (int c = 0; c < c_mid; ++c) hidden_epilogue(c);

    // --- dynamics outputs: group 1 -> reward scalar, group 0 -> h' = relu(LN(.)) -> pool + A3 ---
    mbar_wait(d2_full, 0);
    tc_fence_after();
    if (stamp) TC_STAMP(40);
    if (grp == 1) {
      if (c0 == 0 && own_reward) {  // initial_inference has no reward (networks.py:29 returns 0)
        float rew;
        tmem_ld32(lane_addr + G::COL_D2A, v);
        if constexpr (G::NB == 64) {
          tmem_ld32(lane_addr + G::COL_D2A + 32, v2);
          tmem_wait_ld();
          rew = support_to_scalar_regs(v, v2, sTail + G::T_REW_B, p.reward_min, p.no_tt);
        } else {
          tmem_wait_ld();
          rew = support_to_scalar_regs(v, sTail + G::T_REW_B, p.reward_min, p.no_tt);
        }
        if (live) p.reward[g] = rew;
      }
    } else if (own_hidden) {
      float hbuf[64];
      tmem_ld32(lane_addr + G::COL_D2B, v);
      tmem_ld32(lane_addr + G::COL_D2B + 32, v2);
      tmem_wait_ld();
      // LayerNorm over the 50 state features in packed float32x2 arithmetic (25 pairs; this thread is one
      // in-order stream on the kernel's critical path, the instruction count is its cost)
      float2 h2[H / 2];
      {
        const float4* b4 = reinterpret_cast<const float4*>(sTail + G::T_DYN_B);
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
        const float2 b = *reinterpret_cast<const float2*>(sTail + G::T_DYN_B + 48);
        h2[24] = __fadd2_rn(make_float2(__uint_as_float(v2[16]), __uint_as_float(v2[17])), b);
      }
      float2 s2[4] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
#pragma unroll
      for (int k = 0; k < H / 2; ++k) s2[k & 3] = __fadd2_rn(s2[k & 3], h2[k]);
      const float2 st = __fadd2_rn(__fadd2_rn(s2[0], s2[1]), __fadd2_rn(s2[2], s2[3]));
      const float mean = (st.x + st.y) * (1.0f / (float)H);
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
        const float2* w2 = reinterpret_cast<const float2*>(sTail + G::T_LN_W);
        const float2* b2 = reinterpret_cast<const float2*>(sTail + G::T_LN_B);
#pragma unroll
        for (int k = 0; k < H / 2; ++k) {
          const float2 y = __ffma2_rn(__fmul2_rn(h2[k], rstd2), w2[k], b2[k]);
          hbuf[2 * k] = fmaxf(y.x, 0.0f);
          hbuf[2 * k + 1] = fmaxf(y.y, 0.0f);
        }
      }
      hbuf[H] = 1.0f;  // column H feeds the folded first-layer bias
#pragma unroll
      for (int j = H + 1; j < 64; ++j) hbuf[j] = 0.0f;
      {
        // h' as the bf16 A operand of the prediction layer: this row of the canonical K-major image,
        // in this CTA's shared memory and -- in a split pair -- in the peer's as well
        uint4 q[K3 / 8];
#pragma unroll
        for (int kb = 0; kb < K3 / 8; ++kb) {
          q[kb] = make_uint4(pack_bf16(hbuf[8 * kb], hbuf[8 * kb + 1]), pack_bf16(hbuf[8 * kb + 2], hbuf[8 * kb + 3]),
                             pack_bf16(hbuf[8 * kb + 4], hbuf[8 * kb + 5]), pack_bf16(hbuf[8 * kb + 6], hbuf[8 * kb + 7]));
          *reinterpret_cast<uint4*>(sA3 + canon_off(row, 8 * kb, ROWS)) = q[kb];
        }
        // release the local prediction layer first, then ship the same rows to the peer
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(a3_ready);
        if (split) {
          const uint32_t a3_peer = map_to_cta(smem_u32(sA3), 0);
          const uint32_t bar_peer = map_to_cta(smem_u32(a3_remote), 0);
#pragma unroll
          for (int kb = 0; kb < K3 / 8; ++kb)
            st_async_v4(a3_peer + (uint32_t)canon_off(row, 8 * kb, ROWS), q[kb], bar_peer);
        }
      }
      if (stamp) TC_STAMP(41);
      // after the hand-off: h' goes to the pool through shared memory so that every store
      // instruction writes one contiguous 200-byte row (a per-thread row store touches 32 lines)
#pragma unroll
      for (int j = 0; j < H; ++j) sOut[row * OUT_STRIDE + j] = hbuf[j];
      __syncwarp();
      if (lane == 0) mbar_arrive(h_staged);  // the store warp takes it from here
    } else {
      // rank 0 of a split pair: wait for the peer's rows (cluster-scope acquire), make them visible
      // to the tensor-core (async) proxy, release the local layer-1 issuer
      mbar_wait_cluster(a3_remote, 0);
      fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(a3_ready);
    }

    for (int c = c_mid; c < nch; ++c) hidden_epilogue(c);

    // --- prediction outputs: group 0 -> value scalar, group 1 -> policy logits ---
    mbar_wait(d2_full, 1);
    tc_fence_after();
    if (stamp) TC_STAMP(42);
    if (grp == 0) {
      if (own_value) {
        float val;
        tmem_ld32(lane_addr + G::COL_D2A, v);
        if constexpr (G::NB == 64) {
          tmem_ld32(lane_addr + G::COL_D2A + 32, v2);
          tmem_wait_ld();
          val = support_to_scalar_regs(v, v2, sTail + G::T_VAL_B, p.value_min, p.no_tt);
        } else {
          tmem_wait_ld();
          val = support_to_scalar_regs(v, sTail + G::T_VAL_B, p.value_min, p.no_tt);
        }
        if (live) p.value[g] = val;
      }
    } else if (own_logits) {
      tmem_ld32(lane_addr + G::COL_D2B, v);
      tmem_wait_ld();
      // logits [rows][A] of this CTA are one contiguous block: stage row-major, store linearly
      const int A = p.num_actions;
      mbar_wait(h_stored, 0);  // the staging area is free again
#pragma unroll
      for (int j = 0; j < 32; ++j)
        if (j < A) sLog[row * A + j] = __uint_as_float(v[j]) + sTail[G::T_POL_B + j];
      if constexpr (G::NB == 64) {  // second half of the 64 policy columns
        tmem_ld32(lane_addr + G::COL_D2B + 32, v);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 32; ++j)
          if (32 + j < A) sLog[row * A + 32 + j] = __uint_as_float(v[j]) + sTail[G::T_POL_B + 32 + j];
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");  // the four warps of this group
      const int rows_here = min(ROWS, p.batch - tile * ROWS);
      float* dl = p.logits + (size_t)tile * ROWS * A;
      for (int i = row; i < rows_here * A; i += ROWS) dl[i] = sLog[i];
    }
    tc_fence_before();
    if (stamp) TC_STAMP(43);
  }

  __syncthreads();
  if (threadIdx.x == 0) TC_STAMP(44);
  if (p.trace && threadIdx.x == 0 && blockIdx.x < 64) {
    unsigned long long tns;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(tns));
    p.trace[256 + 2 * blockIdx.x + 1] = (long long)tns;
  }
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, TMEM_COLS);
  }
}

// ---- packing: f32 reference-layout weights -> bf16 chunk images + tail parameters ---------------
// chunk0 = 0: the recurrent image (reward, transition, value, policy heads); chunk0 = 4: the
// initial-inference image (representation in place of the transition head, then value, policy)
template <class G>
__global__ void fc_tc_pack_kernel(mz_fc_weights w, int k1, int chunk0, uint8_t* chunks, float* tail) {
  const int A = w.num_actions;
  const bool init = chunk0 != 0;
  for (int c = chunk0; c < NCHUNK; ++c) {
    const ChunkGeom g = chunk_geom<G>(c, k1);
    uint8_t* base = chunks + (chunk_offset<G>(c, k1) - chunk_offset<G>(chunk0, k1));
    const int head = c >> 2, f0 = (c & 3) * CHUNK;
    const float* dyn_w1 = init ? w.rep_w1 : w.dyn_w1;
    const float* dyn_b1 = init ? w.rep_b1 : w.dyn_b1;
    const float* dyn_w2 = init ? w.rep_w2 : w.dyn_w2;
    const float* w1t = head == 0 ? w.rew_w1 : (head == 1 ? dyn_w1 : (head == 2 ? w.val_w1 : w.pol_w1));
    const float* b1 = head == 0 ? w.rew_b1 : (head == 1 ? dyn_b1 : (head == 2 ? w.val_b1 : w.pol_b1));
    const float* w2 = head == 0 ? w.rew_w2 : (head == 1 ? dyn_w2 : (head == 2 ? w.val_w2 : w.pol_w2));
    const int kin = head < 2 ? (init ? w.obs_dim : H + A) : H;  // real input width of the first layer
    const int nout = head == 0 ? w.reward_bins : (head == 1 ? H : (head == 2 ? w.value_bins : A));
    // W1 chunk: B operand [CHUNK features x K], element (n, k) = w1t[k][f0 + n]
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < CHUNK * g.k; i += gridDim.x * blockDim.x) {
      const int n = i / g.k, k = i % g.k;
      const float x = k < kin ? w1t[(size_t)k * W + f0 + n] : (k == kin ? b1[f0 + n] : 0.0f);
      *reinterpret_cast<__nv_bfloat16*>(base + canon_off(n, k, CHUNK)) = __float2bfloat16_rn(x);
    }
    // W2 chunk: B operand [n2 outputs x CHUNK], element (o, k) = w2[o][f0 + k]
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < g.n2 * CHUNK; i += gridDim.x * blockDim.x) {
      const int o = i / CHUNK, k = i % CHUNK;
      const float x = o < nout ? w2[(size_t)o * W + f0 + k] : 0.0f;
      *reinterpret_cast<__nv_bfloat16*>(base + g.w1_bytes + canon_off(o, k, g.n2)) = __float2bfloat16_rn(x);
    }
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < G::TAIL_FLOATS; i += gridDim.x * blockDim.x) {
    float x = 0.0f;
    if (i < G::T_DYN_B) x = i < w.reward_bins ? w.rew_b2[i] : -INFINITY;  // padding columns: see support_to_scalar_regs
    else if (i < G::T_LN_W) x = (i - G::T_DYN_B) < H ? (init ? w.rep_b2 : w.dyn_b2)[i - G::T_DYN_B] : 0.0f;
    else if (i < G::T_LN_B) x = (i - G::T_LN_W) < H ? w.ln_w[i - G::T_LN_W] : 0.0f;
    else if (i < G::T_VAL_B) x = (i - G::T_LN_B) < H ? w.ln_b[i - G::T_LN_B] : 0.0f;
    else if (i < G::T_POL_B) x = (i - G::T_VAL_B) < w.value_bins ? w.val_b2[i - G::T_VAL_B] : -INFINITY;
    else x = (i - G::T_POL_B) < A ? w.pol_b2[i - G::T_POL_B] : 0.0f;
    tail[i] = x;
  }
}

int k1_for(int A) { return (H + A + 1 + 15) / 16 * 16; }  // state + one-hot + bias column

long long* g_tc_trace = nullptr;
int g_tc_trace_block = 0;
int g_tc_split = 1;  // recurrent kernel: two-CTA clusters, heads split between the CTAs

// weight-ring depth of the recurrent kernel; MZ_TC_STAGES=2|3|4 overrides it (diagnostics: a shallower ring leaves
// shared memory for tree-step CTAs on the same SM)
int recurrent_stages() {
  static int st = 0;
  if (st == 0) {
    const char* e = getenv("MZ_TC_STAGES");
    const int v = e ? atoi(e) : 0;
    st = (v >= 2 && v <= MAX_STAGES) ? v : MAX_STAGES;
  }
  return st;
}

int k1_obs(int obs_dim) { return (obs_dim + 1 + 15) / 16 * 16; }  // observation + bias column

// the staging area holds h' ([128][51]) and then the logits ([128][A]: larger from A = 52 on)
template <class G>
size_t tc_smem_bytes(int k1, int stages, int A) {
  return (size_t)ROWS * k1 * 2 + (size_t)stages * stage_bytes_for<G>(k1) +
         (size_t)ROWS * K3 * 2 + 24 * sizeof(uint64_t) + G::TAIL_FLOATS * sizeof(float) +
         ROWS * (A > OUT_STRIDE ? A : OUT_STRIDE) * sizeof(float);
}

constexpr size_t kTcMaxSmem = 232448;

// Geometry of a network's bf16 images: 0 = not supported, 1 = narrow, 2 = wide.
int tc_geometry(const mz_fc_weights& w) {
  if (w.num_actions < 1 || w.num_actions > 64 || w.value_bins < 1 || w.value_bins > 64 || w.reward_bins < 1 ||
      w.reward_bins > 64 || w.no_support)
    return 0;
  return (w.num_actions > 32 || w.value_bins > 32 || w.reward_bins > 32) ? 2 : 1;
}

// The wide recurrent kernel runs a three-stage ring at every k1: its larger tail does not leave room for a fourth
// stage at k1 = 96 (A 30..45), and k1 = 112 / 128 (A 46..64) have no room for one with either tail.
template <class G>
int stages_for() { return G::NB == 64 && recurrent_stages() > 3 ? 3 : recurrent_stages(); }

template <class G>
int launch_tc(const TcParams& p, void* stream) {
  const size_t smem = tc_smem_bytes<G>(p.k1, p.stages, p.num_actions);
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(fc_recurrent_tc_kernel<G>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcMaxSmem);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  if (smem > kTcMaxSmem) return MZ_ERR_UNSUPPORTED;
  const int tiles = (p.batch + ROWS - 1) / ROWS;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(p.split ? 2 * tiles : tiles);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute lattr[2];
  int na = 0;
  if (p.split) {
    lattr[na].id = cudaLaunchAttributeClusterDimension;
    lattr[na].val.clusterDim.x = 2;
    lattr[na].val.clusterDim.y = 1;
    lattr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (p.obs == nullptr && g_mz_pdl) {
    lattr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    lattr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = lattr;
  cfg.numAttrs = na;
  cudaError_t e = cudaLaunchKernelEx(&cfg, fc_recurrent_tc_kernel<G>, p);
  if (e != cudaSuccess) return (int)e;
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

}  // namespace

extern "C" {

int mz_fc_tc_set_split(int32_t enable) {
  g_tc_split = enable ? 1 : 0;
  return MZ_OK;
}

int mz_debug_set_tc_trace_block(int32_t block) {
  g_tc_trace_block = block;
  return MZ_OK;
}

int mz_debug_set_tc_trace(int64_t* device_buffer) {
  g_tc_trace = (long long*)device_buffer;
  return MZ_OK;
}

int64_t mz_fc_tc_packed_bytes(int32_t num_actions) {
  if (num_actions < 1 || num_actions > 32) return MZ_ERR_UNSUPPORTED;
  return (int64_t)chunk_offset(NCHUNK, k1_for(num_actions));
}

int mz_fc_tc_sizes(const mz_fc_weights* w, int64_t* recurrent_bytes, int64_t* initial_bytes, int32_t* tail_floats) {
  if (!w || !recurrent_bytes || !initial_bytes || !tail_floats) return MZ_ERR_BAD_ARG;
  const int geom = tc_geometry(*w);
  if (geom == 0) return MZ_ERR_UNSUPPORTED;
  const int k1 = k1_for(w->num_actions), k1i = k1_obs(w->obs_dim);
  if (geom == 1) {
    *recurrent_bytes = (int64_t)chunk_offset<NarrowGeom>(NCHUNK, k1);
    *tail_floats = NarrowGeom::TAIL_FLOATS;
  } else {
    *recurrent_bytes = (int64_t)chunk_offset<WideGeom>(NCHUNK, k1);
    *tail_floats = WideGeom::TAIL_FLOATS;
  }
  if (w->obs_dim < 1)
    *initial_bytes = MZ_ERR_BAD_ARG;
  else if ((geom == 1 ? tc_smem_bytes<NarrowGeom>(k1i, 2, w->num_actions)
                      : tc_smem_bytes<WideGeom>(k1i, 2, w->num_actions)) > kTcMaxSmem)
    *initial_bytes = MZ_ERR_UNSUPPORTED;
  else
    *initial_bytes = (int64_t)(geom == 1 ? chunk_offset<NarrowGeom>(NCHUNK, k1i) - chunk_offset<NarrowGeom>(4, k1i)
                                         : chunk_offset<WideGeom>(NCHUNK, k1i) - chunk_offset<WideGeom>(4, k1i));
  return MZ_OK;
}

int32_t mz_fc_tc_tail_floats(void) { return TAIL_FLOATS; }

int mz_fc_tc_pack(const mz_fc_weights* w, void* packed, float* tail, void* stream) {
  if (!w || !packed || !tail) return MZ_ERR_BAD_ARG;
  const int geom = tc_geometry(*w);
  if (geom == 0) return MZ_ERR_UNSUPPORTED;
  if (geom == 1)
    fc_tc_pack_kernel<NarrowGeom><<<64, 256, 0, (cudaStream_t)stream>>>(*w, k1_for(w->num_actions), 0,
                                                                        (uint8_t*)packed, tail);
  else
    fc_tc_pack_kernel<WideGeom><<<64, 256, 0, (cudaStream_t)stream>>>(*w, k1_for(w->num_actions), 0,
                                                                      (uint8_t*)packed, tail);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_fc_recurrent_tc(const mz_fc_weights* w, const void* packed, const float* tail, int32_t batch,
                       const float* hidden_in, int64_t in_row_stride, const int32_t* in_index,
                       const int32_t* actions, float* hidden_out, int64_t out_row_stride,
                       int64_t out_offset, float* value, float* reward, float* logits, void* stream) {
  if (!w || !packed || !tail || batch < 1 || !hidden_in || !actions || !hidden_out || !value ||
      !reward || !logits)
    return MZ_ERR_BAD_ARG;
  // the epilogue reads hidden rows as float2: every row start must be 8-byte aligned
  if ((in_row_stride & 1) || ((uintptr_t)hidden_in & 7)) return MZ_ERR_BAD_ARG;
  const int geom = tc_geometry(*w);
  if (geom == 0) return MZ_ERR_UNSUPPORTED;
  TcParams p;
  p.chunks = (const uint8_t*)packed;
  p.tail = tail;
  p.k1 = k1_for(w->num_actions);
  p.num_actions = w->num_actions;
  p.value_bins = w->value_bins;
  p.reward_bins = w->reward_bins;
  p.value_min = w->value_min;
  p.reward_min = w->reward_min;
  p.no_tt = w->no_target_transform;
  p.batch = batch;
  p.hidden_in = hidden_in;
  p.in_row_stride = in_row_stride;
  p.in_index = in_index;
  p.actions = actions;
  p.hidden_out = hidden_out;
  p.out_row_stride = out_row_stride;
  p.out_offset = out_offset;
  p.value = value;
  p.reward = reward;
  p.logits = logits;
  p.trace = g_tc_trace;
  p.chunk0 = 0;
  p.stages = geom == 1 ? stages_for<NarrowGeom>() : stages_for<WideGeom>();
  p.obs = nullptr;
  p.obs_dim = 0;
  p.split = g_tc_split;
  p.trace_block = g_tc_trace_block;
  return geom == 1 ? launch_tc<NarrowGeom>(p, stream) : launch_tc<WideGeom>(p, stream);
}

/* Initial-inference image: representation head (K = obs_dim + bias column) + value + policy. */
int64_t mz_fc_tc_initial_packed_bytes(int32_t obs_dim) {
  if (obs_dim < 1) return MZ_ERR_BAD_ARG;
  const int k1 = k1_obs(obs_dim);
  if (tc_smem_bytes<NarrowGeom>(k1, 2, 32) > kTcMaxSmem) return MZ_ERR_UNSUPPORTED;
  return (int64_t)(chunk_offset(NCHUNK, k1) - chunk_offset(4, k1));
}

int mz_fc_tc_pack_initial(const mz_fc_weights* w, void* packed, float* tail, void* stream) {
  if (!w || !packed || !tail) return MZ_ERR_BAD_ARG;
  const int geom = tc_geometry(*w);
  if (geom == 0) return MZ_ERR_UNSUPPORTED;
  const int k1 = k1_obs(w->obs_dim);
  if (geom == 1) {
    if (tc_smem_bytes<NarrowGeom>(k1, 2, w->num_actions) > kTcMaxSmem) return MZ_ERR_UNSUPPORTED;
    fc_tc_pack_kernel<NarrowGeom><<<64, 256, 0, (cudaStream_t)stream>>>(*w, k1, 4, (uint8_t*)packed, tail);
  } else {
    if (tc_smem_bytes<WideGeom>(k1, 2, w->num_actions) > kTcMaxSmem) return MZ_ERR_UNSUPPORTED;
    fc_tc_pack_kernel<WideGeom><<<64, 256, 0, (cudaStream_t)stream>>>(*w, k1, 4, (uint8_t*)packed, tail);
  }
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_fc_initial_tc(const mz_fc_weights* w, const void* packed, const float* tail, int32_t batch,
                     const float* obs, float* hidden_out, int64_t out_row_stride, float* value,
                     float* logits, void* stream) {
  if (!w || !packed || !tail || batch < 1 || !obs || !hidden_out || !value || !logits) return MZ_ERR_BAD_ARG;
  const int geom = tc_geometry(*w);
  if (geom == 0) return MZ_ERR_UNSUPPORTED;
  TcParams p;
  p.chunks = (const uint8_t*)packed;
  p.tail = tail;
  p.k1 = k1_obs(w->obs_dim);
  p.num_actions = w->num_actions;
  p.value_bins = w->value_bins;
  p.reward_bins = w->reward_bins;
  p.value_min = w->value_min;
  p.reward_min = w->reward_min;
  p.no_tt = w->no_target_transform;
  p.batch = batch;
  p.hidden_in = nullptr;
  p.in_row_stride = 0;
  p.in_index = nullptr;
  p.actions = nullptr;
  p.hidden_out = hidden_out;
  p.out_row_stride = out_row_stride;
  p.out_offset = 0;
  p.value = value;
  p.reward = nullptr;
  p.logits = logits;
  p.trace = nullptr;
  p.chunk0 = 4;
  p.stages = 2;
  p.obs = obs;
  p.obs_dim = w->obs_dim;
  p.split = 0;
  p.trace_block = 0;
  return geom == 1 ? launch_tc<NarrowGeom>(p, stream) : launch_tc<WideGeom>(p, stream);
}

}  // extern "C"
