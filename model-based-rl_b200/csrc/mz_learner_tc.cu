// The learner's network forward and backward (Learner.update_weights, learners.py:164-230) on the tensor cores:
// bf16 operands, float32 accumulation, float32 master weights and gradients.
//
// The step of the FCNetwork architecture (networks.py:55-174) is 4 GFLOP behind a chain of 2 (K + 1) + 3 dependent
// two-layer heads, 32..3072 rows each: what bounds it is the length of that chain, not tensor throughput.  So the
// kernels (mz_learner_tc.cuh, shared with the 3xTF32 step of mz_learner_tf32.cu) are built to make the chain short
// rather than the tiles big:
//
//   chain_fwd   ONE launch for representation -> LN -> K x (dynamics -> LN): the rows of a batch are independent in
//               the forward, so a CTA keeps its 32 rows for all K + 1 steps; the hidden state of a step goes from the
//               LayerNorm epilogue straight into the next step's A tile in shared memory
//   heads_fwd   ONE launch for the value / policy / reward heads over the stacked hidden states (blockIdx.y = head)
//   heads_bwd   ONE launch for their backward (dX accumulated into the hidden states' gradient rows)
//   chain_bwd   ONE launch back through K x (LN -> dynamics), LN, representation: the gradient of a row's hidden state
//               only depends on the same row's later steps, so again a CTA keeps its rows; the dynamics head's dX tile
//               feeds the next LayerNorm backward through shared memory; the 0.5 gradient hook (learners.py:201) is a
//               scale there
//
// -- 4 launches where the float32 CUDA-core path (mz_learner.cu) needs 30.  Inside a tile every contraction is
// mma.sync.m16n8k16 (bf16 x bf16 -> f32): the tiles are 32 rows x 64 columns per warp and change role five times per
// head (activation, dH, dX, two weight gradients with the batch rows as the K dimension, fed by ldmatrix.trans from the
// same row-major tiles), which warp-level fragments do without a TMEM / descriptor round trip per role.  Weights are
// read as pre-packed B fragments (mz_learner_pack: one 16-byte load per lane covers two k-steps), refreshed once per
// step from the float32 master copy.  Weight gradients leave as float32 atomics (one per weight and CTA).
#include <cuda_bf16.h>

#include "mz_learner_tc.cuh"

namespace {

MZ_DEV void ldsm4(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}
MZ_DEV void ldsm4t(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}
// D (16 x 8, f32) += A (16 x 16, row) * B (16 x 8, col), bf16 operands
MZ_DEV void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
MZ_DEV uint32_t pack2(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}

// Packed B operand of a matrix Bm [N][K] (B[k][n] = Bm[n][k]): 32-bit word ((nt KQ + kq) 32 + lane) 4 + i holds
// (Bm[8 nt + g][kk], Bm[8 nt + g][kk + 1]) with g = lane >> 2, kk = 32 kq + 16 (i >> 1) + 8 (i & 1) + 2 (lane & 3):
// the b0 / b1 registers of k-steps 2 kq and 2 kq + 1 of n-tile nt, one 16-byte load per lane.  Zeros outside N x K.
__global__ void pack_kernel(PackParams p) {
  const mz_pack_job job = p.jobs[blockIdx.y];
  if (job.src == nullptr) {  // a buffer to clear before the step (gradients): n 32-bit words
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < job.n; w += gridDim.x * blockDim.x) job.dst[w] = 0u;
    return;
  }
  const int KQ = (job.k + 31) >> 5, NTl = (job.n + 7) >> 3;
  const int words = NTl * KQ * 128;
  for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < words; w += gridDim.x * blockDim.x) {
    const int i = w & 3, lane = (w >> 2) & 31, rest = w >> 7;
    const int kq = rest % KQ, nt = rest / KQ;
    const int nn = 8 * nt + (lane >> 2), kk = 32 * kq + 16 * (i >> 1) + 8 * (i & 1) + 2 * (lane & 3);
    float lo = 0.0f, hi = 0.0f;
    if (nn < job.n) {
      if (kk < job.k) lo = job.src[(size_t)nn * job.stride_n + (size_t)kk * job.stride_k];
      if (kk + 1 < job.k) hi = job.src[(size_t)nn * job.stride_n + (size_t)(kk + 1) * job.stride_k];
    }
    job.dst[w] = pack2(lo, hi);
  }
}

// The bf16 operand format of mz_learner_tc.cuh's kernels.  Tiles are bf16 (XLD 136: ldmatrix rows 16 B apart mod
// 128); a k unit is the 32 features of two m16n8k16 k-steps.  Two 32-row tiles per heads_bwd CTA fit the shared
// memory (heads_bwd_smem: 112 KB at one tile, 190 KB at two of the 227 KB).
struct Bf16 {
  using T = __nv_bfloat16;
  static constexpr int K = 32;
  static constexpr int MAX_TILES = 2;
  static constexpr bool GAMMA_IN_REGS = true, EARLY_LN_LOAD = true;
  static constexpr int PACK_CTA_WORDS = 1024, CLEAR_CTA_WORDS = 4096, PACK_MAX_CTAS = 96;
  static constexpr void (*pack_kernel)(PackParams) = ::pack_kernel;

  static MZ_DEV T cvt(float x) { return __float2bfloat16_rn(x); }
  using T2 = uint32_t;
  static MZ_DEV T2 pair(float a, float b) { return pack2(a, b); }
  static int64_t packed_words(int32_t n, int32_t k) { return (int64_t)((n + 7) / 8) * ((k + 31) / 32) * 128; }

  // acc[MT][NTW][4] += A (16 MT rows x 32 KQ, row-major bf16 in shared memory) * B (packed; n-tiles nt0 ..
  // nt0 + NTW - 1).  ldq: k-step pairs per n-tile of the packed image (KQ, or more when Bp points at a K slice of a
  // wider image).
  template <int MT>
  static MZ_DEV void gemm_wide(float (&acc)[MT][NTW][4], const T* As, int lda, const uint32_t* __restrict__ Bp, int KQ,
                               int nt0, int lane, int ldq) {
    const int arow = (lane & 7) + ((lane >> 3) & 1) * 8, acol = (lane >> 4) * 8;
    const uint4* bp = reinterpret_cast<const uint4*>(Bp) + (size_t)nt0 * ldq * 32 + lane;
    uint4 b[NTW];
#pragma unroll
    for (int n = 0; n < NTW; ++n) b[n] = __ldg(bp + (size_t)n * ldq * 32);
    for (int kq = 0; kq < KQ; ++kq) {
      uint4 bn[NTW];
      if (kq + 1 < KQ) {
#pragma unroll
        for (int n = 0; n < NTW; ++n) bn[n] = __ldg(bp + ((size_t)n * ldq + kq + 1) * 32);
      }
      uint32_t a[2][MT][4];
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) ldsm4(a[ks][mt], As + (16 * mt + arow) * lda + 32 * kq + 16 * ks + acol);
#pragma unroll
      for (int n = 0; n < NTW; ++n) {
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) mma16816(acc[mt][n], a[0][mt], b[n].x, b[n].y);
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) mma16816(acc[mt][n], a[1][mt], b[n].z, b[n].w);
      }
      if (kq + 1 < KQ) {
#pragma unroll
        for (int n = 0; n < NTW; ++n) b[n] = bn[n];
      }
    }
  }

  // acc[MT][4] = A (16 MT rows x 512, row-major bf16 in shared memory) * B (packed, KQ = 16; n-tile nt)
  template <int MT>
  static MZ_DEV void gemm_tall(float (&acc)[MT][4], const T* As, int lda, const uint32_t* __restrict__ Bp, int nt, int lane) {
    const int arow = (lane & 7) + ((lane >> 3) & 1) * 8, acol = (lane >> 4) * 8;
    const uint4* bp = reinterpret_cast<const uint4*>(Bp) + (size_t)nt * 16 * 32 + lane;
    uint4 b[16];
#pragma unroll
    for (int kq = 0; kq < 16; ++kq) b[kq] = __ldg(bp + kq * 32);
    float acc2[MT][4];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[mt][c] = acc2[mt][c] = 0.0f;
#pragma unroll
    for (int kq = 0; kq < 16; ++kq) {
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
        uint32_t a0[4], a1[4];
        ldsm4(a0, As + (16 * mt + arow) * lda + 32 * kq + acol);
        ldsm4(a1, As + (16 * mt + arow) * lda + 32 * kq + 16 + acol);
        mma16816(acc[mt], a0, b[kq].x, b[kq].y);
        mma16816(acc2[mt], a1, b[kq].z, b[kq].w);
      }
    }
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[mt][c] += acc2[mt][c];
  }

  // gW1[j][k] += sum_r dH[r][j] X[r][k] for columns [0, cols) of the X tiles in Xs, to gw1[j * ld + k]: M = the warp's
  // hidden units, N = input features in chunks of 64, K = the CTA's rows.  One slice of a WIDE head's input; narrow
  // heads run the same loop inline over all of X (as one function it changes their register allocation).
  template <int TILES>
  static MZ_DEV void gw1_phase(float* gw1, int ld, int cols, const T* Xs, const T* dHs, float* stage, int warp, int lane) {
    const int lrow = lane & 7, lsel = lane >> 3;  // ldmatrix.trans: lanes 8 i .. 8 i + 7 address matrix i
    for (int mt = 0; mt < CW / 16; ++mt) {
      for (int chunk = 0; 64 * chunk < cols; ++chunk) {
        float acc[8][4];
#pragma unroll
        for (int n = 0; n < 8; ++n)
#pragma unroll
          for (int c = 0; c < 4; ++c) acc[n][c] = 0.0f;
#pragma unroll
        for (int ks = 0; ks < 2 * TILES; ++ks) {
          uint32_t a[4];
          ldsm4t(a, dHs + (16 * ks + lrow + (lsel >> 1) * 8) * HLD + CW * warp + 16 * mt + (lsel & 1) * 8);
#pragma unroll
          for (int np = 0; np < 4; ++np) {
            if (64 * chunk + 16 * np < cols) {  // warp-uniform; the tile is zero padded to a multiple of 32 columns
              uint32_t b[4];
              ldsm4t(b, Xs + (16 * ks + lrow + (lsel & 1) * 8) * XLD + 64 * chunk + 16 * np + (lsel >> 1) * 8);
              mma16816(acc[2 * np], a, b[0], b[1]);
              mma16816(acc[2 * np + 1], a, b[2], b[3]);
            }
          }
        }
        tile_add<8>(gw1 + (size_t)(CW * warp + 16 * mt) * ld + 64 * chunk, ld, 16, min(64, cols - 64 * chunk), acc, stage,
                    lane);
      }
    }
  }

  // Backward of one head over the CTA's TILES tiles of 32 rows.  In: Xs (input rows), dYs (output gradient, zero padded
  // to a multiple of 32 columns).  Out: the four parameter gradients (vector reductions: one per weight and CTA, so two
  // tiles per CTA halve that traffic), and dX (columns [0, dx_cols)) accumulated into global memory.
  // WIDE (heads up to MAXIN inputs, no dX above SLICE): Xs is not loaded by the caller; the recomputed activation and
  // gW1 each stream X (rows of `ldx` floats) through Xs in slices of SLICE features.
  template <int TILES, bool WIDE>
  static MZ_DEV void backward(const mz_tc_head& h, const float* __restrict__ X, int ldx, T* Xs, const T* dYs, T* Hs, T* dHs,
                              float* __restrict__ dX, int lddx, int dx_cols, int row0, int rows, float* stage, int warp,
                              int lane) {
    const int g = lane >> 2, t = lane & 3;
    TC_T(1, 0, 1);
    float s0[NTW], s1[NTW];  // column sums of the gated dH: gb1
#pragma unroll
    for (int n = 0; n < NTW; ++n) s0[n] = s1[n] = 0.0f;
#pragma unroll 1
    for (int tile = 0; tile < TILES; ++tile) {
      const T* Xt = Xs + tile * RT * XLD;
      const T* dYt = dYs + tile * RT * DYLD;
      T* Ht = Hs + tile * RT * HLD;
      T* dHt = dHs + tile * RT * HLD;
      uint32_t mask[2];
      if (WIDE)
        hidden_phase_sliced<Bf16, 2>(h, X, ldx, row0 + RT * tile, rows, Xs + tile * RT * XLD, Ht, mask, warp, lane);
      else
        hidden_phase<Bf16, 2>(h, Xt, Ht, mask, warp, lane);
      // dH = dY W2 for the warp's hidden units, masked by the ReLU -> dHs
      float acc[2][NTW][4];
      zero<2>(acc);
      const int KQ = kunits<Bf16>(h.d_out);
      gemm_wide<2>(acc, dYt, DYLD, h.w2tp, KQ, NTW * warp, lane, KQ);
#pragma unroll
      for (int n = 0; n < NTW; ++n) {
        const int j = CW * warp + 8 * n + 2 * t;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          const uint32_t m = mask[mt] >> (4 * n);
          const float v0 = (m & 1u) ? acc[mt][n][0] : 0.0f, v1 = (m & 2u) ? acc[mt][n][1] : 0.0f;
          const float v2 = (m & 4u) ? acc[mt][n][2] : 0.0f, v3 = (m & 8u) ? acc[mt][n][3] : 0.0f;
          s0[n] += v0 + v2;
          s1[n] += v1 + v3;
          pair_at<Bf16>(dHt + (16 * mt + g) * HLD + j) = pair(v0, v1);
          pair_at<Bf16>(dHt + (16 * mt + g + 8) * HLD + j) = pair(v2, v3);
        }
      }
    }
#pragma unroll
    for (int n = 0; n < NTW; ++n) {
#pragma unroll
      for (int m = 4; m < 32; m <<= 1) {
        s0[n] += __shfl_xor_sync(MZ_FULL, s0[n], m);
        s1[n] += __shfl_xor_sync(MZ_FULL, s1[n], m);
      }
      if (g == 0) {
        atomicAdd(h.gb1 + CW * warp + 8 * n + 2 * t, s0[n]);
        atomicAdd(h.gb1 + CW * warp + 8 * n + 2 * t + 1, s1[n]);
      }
    }
    TC_T(1, 0, 2);
    __syncthreads();
    TC_T(1, 0, 3);
    // dX = dH W1: (tile, n-tile) pairs over the warps
    if (dx_cols > 0) {
      const int ntl = (dx_cols + 7) >> 3;
      for (int w = warp; w < TILES * ntl; w += NW) {
        const int tile = w / ntl, nt = w - tile * ntl;
        float acc[2][4];
        gemm_tall<2>(acc, dHs + tile * RT * HLD, HLD, h.w1tp, nt, lane);
        const int k = 8 * nt + 2 * t;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            const int r = row0 + RT * tile + 16 * mt + g + 8 * half;
            if (r < rows) {
              if (k < dx_cols) atomicAdd(dX + (size_t)r * lddx + k, acc[mt][2 * half]);
              if (k + 1 < dx_cols) atomicAdd(dX + (size_t)r * lddx + k + 1, acc[mt][2 * half + 1]);
            }
          }
        }
      }
    }
    TC_T(1, 0, 4);
    const int lrow = lane & 7, lsel = lane >> 3;  // ldmatrix.trans: lanes 8 i .. 8 i + 7 address matrix i
    // gW2[o][j] = sum_r dY[r][o] H[r][j]: M = outputs (16 per m-tile), N = the warp's hidden units, K = the CTA's rows
    for (int mt = 0; 16 * mt < h.d_out; ++mt) {
      float acc[NTW][4];
#pragma unroll
      for (int n = 0; n < NTW; ++n)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[n][c] = 0.0f;
#pragma unroll
      for (int ks = 0; ks < 2 * TILES; ++ks) {
        uint32_t a[4];
        ldsm4t(a, dYs + (16 * ks + lrow + (lsel >> 1) * 8) * DYLD + 16 * mt + (lsel & 1) * 8);
#pragma unroll
        for (int np = 0; np < NTW / 2; ++np) {
          uint32_t b[4];
          ldsm4t(b, Hs + (16 * ks + lrow + (lsel & 1) * 8) * HLD + CW * warp + 16 * np + (lsel >> 1) * 8);
          mma16816(acc[2 * np], a, b[0], b[1]);
          mma16816(acc[2 * np + 1], a, b[2], b[3]);
        }
      }
      tile_add<NTW>(h.gw2 + (size_t)(16 * mt) * LW + CW * warp, LW, h.d_out - 16 * mt, CW, acc, stage, lane);
    }
    TC_T(1, 0, 5);
    if (!WIDE) {
      // gW1[j][k] = sum_r dH[r][j] X[r][k]: M = the warp's hidden units, N = input features in chunks of 64, K = rows
      for (int mt = 0; mt < CW / 16; ++mt) {
        for (int chunk = 0; 64 * chunk < h.d_in; ++chunk) {
          float acc[8][4];
#pragma unroll
          for (int n = 0; n < 8; ++n)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[n][c] = 0.0f;
#pragma unroll
          for (int ks = 0; ks < 2 * TILES; ++ks) {
            uint32_t a[4];
            ldsm4t(a, dHs + (16 * ks + lrow + (lsel >> 1) * 8) * HLD + CW * warp + 16 * mt + (lsel & 1) * 8);
#pragma unroll
            for (int np = 0; np < 4; ++np) {
              if (64 * chunk + 16 * np < h.d_in) {  // warp-uniform; the tile is zero padded to a multiple of 32 columns
                uint32_t b[4];
                ldsm4t(b, Xs + (16 * ks + lrow + (lsel & 1) * 8) * XLD + 64 * chunk + 16 * np + (lsel >> 1) * 8);
                mma16816(acc[2 * np], a, b[0], b[1]);
                mma16816(acc[2 * np + 1], a, b[2], b[3]);
              }
            }
          }
          tile_add<8>(h.gw1 + (size_t)(CW * warp + 16 * mt) * h.d_in + 64 * chunk, h.d_in, 16, min(64, h.d_in - 64 * chunk),
                      acc, stage, lane);
        }
      }
    } else {
      for (int k0 = 0; k0 < h.d_in; k0 += SLICE) {
        const int w = min(SLICE, h.d_in - k0);
        if (h.d_in > SLICE) {  // one slice: still in Xs from the hidden phase
          __syncthreads();
#pragma unroll
          for (int tile = 0; tile < TILES; ++tile)
            load_rows<Bf16>(Xs + tile * RT * XLD, XLD, X + k0, ldx, row0 + RT * tile, rows, w, round_up<K>(w));
          __syncthreads();
        }
        gw1_phase<TILES>(h.gw1 + k0, h.d_in, w, Xs, dHs, stage, warp, lane);
      }
    }
    TC_T(1, 0, 6);
  }
};

}  // namespace

extern "C" {

#ifdef MZ_TC_TRACE
__attribute__((visibility("default"))) int mz_debug_tc_trace(long long* host) {
  return (int)cudaMemcpyFromSymbol(host, g_tc_trace, sizeof(long long) * 2 * 2 * 16 * 8);
}
#endif

int64_t mz_chain_mask_words(int32_t rows, int32_t steps) {
  if (rows < 1 || steps < 1) return 0;
  return (int64_t)steps * ((rows + 15) / 16) * NTH * 2;
}

int64_t mz_learner_packed_words(int32_t n, int32_t k) { return n < 1 || k < 1 ? 0 : Bf16::packed_words(n, k); }
int mz_learner_pack(int32_t njobs, const mz_pack_job* jobs, void* stream) { return pack<Bf16>(njobs, jobs, stream); }
int mz_heads_forward_tc(int32_t njobs, const mz_tc_job* jobs, void* stream) { return heads_forward<Bf16>(njobs, jobs, stream); }
int mz_heads_backward_tc(int32_t njobs, const mz_tc_job* jobs, void* stream) { return heads_backward<Bf16>(njobs, jobs, stream); }
int mz_chain_forward_tc(const mz_tc_chain* chain, void* stream) { return chain_forward<Bf16>(chain, stream); }
int mz_chain_backward_tc(const mz_tc_chain* chain, void* stream) { return chain_backward<Bf16>(chain, stream); }

}  // extern "C"
