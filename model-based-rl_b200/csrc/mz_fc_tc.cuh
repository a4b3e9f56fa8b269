// tcgen05 / TMEM / cluster helpers and the packed-weight geometry of the FCNetwork tensor-core kernels
// (shared by mz_fcnet_tc.cu: one network evaluation per launch, and mz_fcsearch.cu: the whole search in one
// persistent kernel).  Reference semantics: networks.py:31-34, 122-174 (FCNetwork), config.py:27-33.
#pragma once
#include <cuda_bf16.h>
#include <math.h>

#include "mz_common.cuh"
#include "mz_transforms.cuh"

namespace mzfc {

constexpr int H = MZ_FC_HIDDEN;      // 50
constexpr int W = MZ_FC_WIDTH;       // 512
constexpr int ROWS = 128;            // rows (games) per CTA = UMMA M
constexpr int CHUNK = 128;           // hidden features per chunk = UMMA N of the first layer
constexpr int NCHUNK = 16;           // 4 heads x 4 chunks
constexpr int K3 = 64;               // padded K of the prediction first layer
constexpr int MAX_STAGES = 4;        // weight-ring depth (recurrent: 4; initial inference, larger chunks: 2)
constexpr int EPI_THREADS = 256;       // two groups of four epilogue warps
constexpr int MMA2_WARP = 2 + EPI_THREADS / 32;  // second MMA-issuing warp (layer 2)
constexpr int STORE_WARP = MMA2_WARP + 1;       // writes h' rows to the hidden pool, off the critical path
constexpr int TC_THREADS = 64 + EPI_THREADS + 64;
constexpr int N_REW = 32, N_HID = 64, N_VAL = 32, N_POL = 32;  // padded second-layer widths
constexpr int TMEM_COLS = 512;
// TMEM column map (512 columns x 128 lanes x 32 bit)
constexpr int COL_D1 = 0;            // 2 x 128: first-layer accumulators (double buffered)
constexpr int COL_A2 = 256;          // 2 x 64 : relu(first layer) as packed bf16 = A operand of layer 2
constexpr int COL_D2A = 384;         // 32     : reward / value logits
constexpr int COL_D2B = 416;         // 64     : next hidden / policy logits

// tail parameter block (float): second-layer biases and LayerNorm affine
constexpr int T_REW_B = 0, T_DYN_B = 32, T_LN_W = 96, T_LN_B = 160, T_VAL_B = 224, T_POL_B = 256;
constexpr int TAIL_FLOATS = 288;
constexpr int OUT_STRIDE = 51;        // odd row stride of the output staging area (bank-conflict free)

// Second-layer head geometry.  Narrow: A <= 32 and both supports <= 32 bins, reward / value / policy second
// layers padded to N = 32 (the constants above; the persistent search kernel knows only this one).  Wide: any of
// them above 32 (up to 64), all three padded to N = 64, with the TMEM columns and the tail laid out for 64.
struct NarrowGeom {
  static constexpr int NB = 32;  // padded reward / value / policy width
  static constexpr int COL_D2A = mzfc::COL_D2A, COL_D2B = mzfc::COL_D2B;
  static constexpr int T_REW_B = mzfc::T_REW_B, T_DYN_B = mzfc::T_DYN_B, T_LN_W = mzfc::T_LN_W, T_LN_B = mzfc::T_LN_B,
                       T_VAL_B = mzfc::T_VAL_B, T_POL_B = mzfc::T_POL_B, TAIL_FLOATS = mzfc::TAIL_FLOATS;
};
struct WideGeom {
  static constexpr int NB = 64;
  static constexpr int COL_D2A = 384;  // 64: reward / value logits
  static constexpr int COL_D2B = 448;  // 64: next hidden / policy logits (ends at TMEM_COLS)
  static constexpr int T_REW_B = 0, T_DYN_B = 64, T_LN_W = 128, T_LN_B = 192, T_VAL_B = 256, T_POL_B = 320;
  static constexpr int TAIL_FLOATS = 384;
};
static_assert(WideGeom::COL_D2B + N_HID == TMEM_COLS, "the wide column map fills the allocation");

struct ChunkGeom {  // byte geometry of one packed chunk: [W1 | W2]; the first-layer bias is folded
                    // into W1 as the weight of a constant-1 input column (index kin)
  int k;            // K of the first layer (K1 or K3)
  int n2;           // N of the second layer
  int w1_bytes, w2_bytes, bytes;
};

template <class G = NarrowGeom>
__host__ __device__ inline ChunkGeom chunk_geom(int c, int k1) {
  ChunkGeom g;
  const int head = c >> 2;  // 0 reward, 1 transition, 2 value, 3 policy
  g.k = head < 2 ? k1 : K3;
  g.n2 = head == 0 ? G::NB : (head == 1 ? N_HID : G::NB);
  g.w1_bytes = CHUNK * g.k * 2;
  g.w2_bytes = g.n2 * CHUNK * 2;
  g.bytes = g.w1_bytes + g.w2_bytes;
  return g;
}
template <class G = NarrowGeom>
__host__ __device__ inline size_t chunk_offset(int c, int k1) {
  size_t off = 0;
  for (int i = 0; i < c; ++i) off += chunk_geom<G>(i, k1).bytes;
  return off;
}
template <class G = NarrowGeom>
__host__ __device__ inline int stage_bytes_for(int k1) {  // largest chunk: a k1-wide head or a prediction head
  const int a = chunk_geom<G>(4, k1).bytes, b = chunk_geom<G>(8, k1).bytes;
  return a > b ? a : b;
}

// canonical K-major, no swizzle: 8 x 8 core matrices of 128 contiguous bytes,
// core (row_group, k_block) at ((k_block * row_groups) + row_group) * 128
__host__ __device__ inline int canon_off(int row, int k, int rows) {
  return (((k >> 3) * (rows >> 3)) + (row >> 3)) * 128 + (row & 7) * 16 + (k & 7) * 2;
}

// ---- tcgen05 wrappers --------------------------------------------------------------------------
MZ_DEV void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
MZ_DEV void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
MZ_DEV void tmem_dealloc(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols)
               : "memory");
}
// one lane of a converged warp (elect.sync): lets the compiler keep MMA operands in uniform registers
MZ_DEV bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}" : "=r"(pred));
  return pred != 0;
}
MZ_DEV void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
MZ_DEV void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
MZ_DEV void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
MZ_DEV void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
MZ_DEV void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

MZ_DEV void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
MZ_DEV void tmem_st32(uint32_t addr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(addr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
        "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
        "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread (thread i <-> lane base + i)
MZ_DEV void tmem_ld32(uint32_t addr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]),
        "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]),
        "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]),
        "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
        "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(addr)
      : "memory");
}

// shared-memory matrix descriptor: K-major, SWIZZLE_NONE, version 1 (sm_100)
MZ_DEV uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = (uint64_t)((smem_addr >> 4) & 0x3FFFu);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;
  d |= (uint64_t)1 << 46;
  return d;
}
// instruction descriptor: D = f32, A = B = bf16, both K-major, M = 128, N = n
MZ_DEV uint32_t make_idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(ROWS >> 4) << 24);
}

MZ_DEV uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}

// relu + round-to-nearest bf16 pair in one instruction (F2FP.RELU.BF16.PACK_AB)
MZ_DEV uint32_t pack_bf16_relu(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}

// ---- thread-block cluster helpers (distributed shared memory hand-off of h') --------------------
MZ_DEV uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
MZ_DEV void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
MZ_DEV uint32_t map_to_cta(uint32_t smem_addr, uint32_t rank) {  // same offset in the peer CTA's shared memory
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
// 16 bytes into the peer's shared memory; the store itself reports its bytes to the peer's mbarrier, so the
// sender needs neither a cluster-scope fence (MEMBAR.ALL.GPU + ERRBAR in SASS) nor a separate arrival.
MZ_DEV void st_async_v4(uint32_t addr, uint4 v, uint32_t remote_bar) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
               ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w), "r"(remote_bar)
               : "memory");
}
MZ_DEV void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {  // acquire at cluster scope
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}

MZ_DEV float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// softmax(logits + bias) . support, then h^-1, all in registers (one thread per row).  The thread is one
// in-order instruction stream, so the instruction count is the cost: packed float32x2 arithmetic (FADD2 /
// FFMA2) halves it.  The bias of the padding columns (j >= bins) is -inf (fc_tc_pack_kernel), which drops
// them from the maximum and gives them weight exp2(-inf) = 0 without a per-column predicate.
MZ_DEV float support_to_scalar_regs(const uint32_t (&v)[32], const float* bias, int mn, int no_tt) {
  float2 x[16];
  const float4* b4 = reinterpret_cast<const float4*>(bias);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float4 b = b4[k];
    x[2 * k] = __fadd2_rn(make_float2(__uint_as_float(v[4 * k]), __uint_as_float(v[4 * k + 1])), make_float2(b.x, b.y));
    x[2 * k + 1] = __fadd2_rn(make_float2(__uint_as_float(v[4 * k + 2]), __uint_as_float(v[4 * k + 3])), make_float2(b.z, b.w));
  }
  float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};  // four chains keep dependencies short
#pragma unroll
  for (int k = 0; k < 16; ++k) m4[k & 3] = fmaxf(m4[k & 3], fmaxf(x[k].x, x[k].y));
  const float m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
  const float l2e = 1.4426950408889634f;
  const float2 scale = make_float2(l2e, l2e), shift = make_float2(-m * l2e, -m * l2e);
  float2 den[2] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
  float2 num[2] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    const float2 t = __ffma2_rn(x[k], scale, shift);  // (x - m) * log2(e)
    const float2 e = make_float2(ex2_approx(t.x), ex2_approx(t.y));
    den[k & 1] = __fadd2_rn(den[k & 1], e);
    num[k & 1] = __ffma2_rn(e, make_float2((float)(2 * k), (float)(2 * k + 1)), num[k & 1]);
  }
  const float2 d2 = __fadd2_rn(den[0], den[1]), n2 = __fadd2_rn(num[0], num[1]);
  const float mean = __fdividef(n2.x + n2.y, d2.x + d2.y) + (float)mn;  // sum_j (mn + j) softmax_j
  return no_tt ? mean : mz_inverse_scalar_transform_f(mean);
}

// support_to_scalar_regs over 64 columns (wide geometry): columns 0..31 in v, 32..63 in v2.  At 64 bins there
// is no padding column, as at 32 bins in the narrow geometry.
MZ_DEV float support_to_scalar_regs(const uint32_t (&v)[32], const uint32_t (&v2)[32], const float* bias, int mn,
                                    int no_tt) {
  float2 x[32];
  const float4* b4 = reinterpret_cast<const float4*>(bias);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float4 b = b4[k], c = b4[8 + k];
    x[2 * k] = __fadd2_rn(make_float2(__uint_as_float(v[4 * k]), __uint_as_float(v[4 * k + 1])), make_float2(b.x, b.y));
    x[2 * k + 1] = __fadd2_rn(make_float2(__uint_as_float(v[4 * k + 2]), __uint_as_float(v[4 * k + 3])), make_float2(b.z, b.w));
    x[16 + 2 * k] = __fadd2_rn(make_float2(__uint_as_float(v2[4 * k]), __uint_as_float(v2[4 * k + 1])), make_float2(c.x, c.y));
    x[17 + 2 * k] = __fadd2_rn(make_float2(__uint_as_float(v2[4 * k + 2]), __uint_as_float(v2[4 * k + 3])), make_float2(c.z, c.w));
  }
  float m4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
  for (int k = 0; k < 32; ++k) m4[k & 3] = fmaxf(m4[k & 3], fmaxf(x[k].x, x[k].y));
  const float m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
  const float l2e = 1.4426950408889634f;
  const float2 scale = make_float2(l2e, l2e), shift = make_float2(-m * l2e, -m * l2e);
  float2 den[2] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
  float2 num[2] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
#pragma unroll
  for (int k = 0; k < 32; ++k) {
    const float2 t = __ffma2_rn(x[k], scale, shift);
    const float2 e = make_float2(ex2_approx(t.x), ex2_approx(t.y));
    den[k & 1] = __fadd2_rn(den[k & 1], e);
    num[k & 1] = __ffma2_rn(e, make_float2((float)(2 * k), (float)(2 * k + 1)), num[k & 1]);
  }
  const float2 d2 = __fadd2_rn(den[0], den[1]), n2 = __fadd2_rn(num[0], num[1]);
  const float mean = __fdividef(n2.x + n2.y, d2.x + d2.y) + (float)mn;
  return no_tt ? mean : mz_inverse_scalar_transform_f(mean);
}

// immediate-predicate MMA wrappers: the issuing thread is a single dependent instruction stream
// (~5 cycles per SASS instruction), so the per-MMA instruction count is what bounds the issue rate.
template <bool ACC>
MZ_DEV void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  if (ACC)
    asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, 1, 1;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc) : "memory");
  else
    asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, 1, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc) : "memory");
}
template <bool ACC>
MZ_DEV void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc) {
  if (ACC)
    asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, 1, 1;\ntcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}"
                 ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc) : "memory");
  else
    asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, 1, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n}"
                 ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc) : "memory");
}

// layer 2 of chunk c: D2 (+)= A2 (TMEM) * W2c^T, N2 compile time; descriptors advance by an add
template <int N2>
MZ_DEV void issue_mma2(uint32_t d2, uint32_t a_tm, uint32_t b_addr, bool first_chunk_of_head) {
  constexpr uint32_t LBO = (N2 / 8) * 128;
  const uint32_t idesc = make_idesc(N2);
  const uint64_t bd = make_desc(b_addr, LBO, 128);
  if (first_chunk_of_head) umma_ts<false>(d2, a_tm, bd, idesc);
  else umma_ts<true>(d2, a_tm, bd, idesc);
#pragma unroll
  for (int ks = 1; ks < CHUNK / 16; ++ks)
    umma_ts<true>(d2, a_tm + ks * 8, bd + (uint64_t)((ks * 2 * LBO) >> 4), idesc);
}

}  // namespace mzfc
