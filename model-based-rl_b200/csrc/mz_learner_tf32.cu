// The learner's network forward and backward (Learner.update_weights, learners.py:164-230) on the tensor cores at
// float32 accuracy: every contraction is three TF32 mma.sync.m16n8k8 products on split operands (x = x_hi + x_lo,
// w = w_hi + w_lo; x w ~= x_lo w_hi + x_hi w_lo + x_hi w_hi, float32 accumulation, see split_tf32), so there is no
// bf16 rounding point anywhere.  float32 master weights, gradients and optimiser state as in the other two learners.
//
// The step is the four-launch step of mz_learner_tc.cuh (chain_fwd, heads_fwd, heads_bwd, chain_bwd), instantiated
// with the operand format here:
//   weights      mz_learner_pack_tf32x3 writes each image as hi / lo TF32 B fragments of m16n8k8 (one 16-byte load
//                per lane and k-step of 8: {hi(k), hi(k + 1), lo(k), lo(k + 1)}) from the float32 master copy
//   activations  X, H, dY, dH and the LayerNorm tiles stay float32 in shared memory and are split when a fragment is
//                loaded (one LOP3 and one FADD per value)
// The six roles of a head (layer 1, layer 2, dH = dY W2, dX = dH W1, gW2 = dY^T H, gW1 = dH^T X) read the row-major
// tiles two ways.  Row-major A fragments (the batch rows are M) permute k inside a k-step -- MMA k slot j <-> column
// 2 (j mod 4) + j / 4 -- so a lane's a0 / a2 are one 8-byte load; the packed B images use the same permutation.  The
// two weight gradients have the batch rows as K and need the tiles transposed, which ldmatrix.trans cannot do for
// 32-bit elements: those fragments are scalar loads of rows t and t + 4 of a k-step, column g.  Every tile stride is
// 8 (mod 32) floats (XLD 136, HLD 520, DYLD 72), which makes both patterns free of bank conflicts: a half-warp's
// 8-byte loads cover banks 8 g + 2 t + {0, 1} (g < 4), a warp's transposed scalar loads banks 8 t + g.
//
// Shared memory is twice that of the bf16 tiles, so heads_bwd keeps one 32-row tile per CTA (190 KB; the bf16 step's
// two-tile plan would need 354 KB); the chain kernels keep 16 or 32 rows as the bf16 ones do.
#include "mz_learner_tc.cuh"

namespace {

constexpr int KS_TALL = LW / 8;  // k-steps of a contraction over the 512 hidden units

// D (16 x 8, f32) += A (16 x 8, row) * B (8 x 8, col), TF32 operands
MZ_DEV void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// Row-major A fragment of one k-step: rows row0 + g, row0 + g + 8, columns k0 + 2 t, k0 + 2 t + 1 (the permuted k
// slots t, t + 4), split.
MZ_DEV void frag_rows(uint32_t (&ah)[4], uint32_t (&al)[4], const float* As, int lda, int row0, int k0, int lane) {
  const int g = lane >> 2, t = lane & 3;
  const float2 x0 = *reinterpret_cast<const float2*>(As + (row0 + g) * lda + k0 + 2 * t);
  const float2 x1 = *reinterpret_cast<const float2*>(As + (row0 + g + 8) * lda + k0 + 2 * t);
  split_tf32(x0.x, ah[0], al[0]);
  split_tf32(x1.x, ah[1], al[1]);
  split_tf32(x0.y, ah[2], al[2]);
  split_tf32(x1.y, ah[3], al[3]);
}
// Transposed A fragment (M = columns c0 .. c0 + 15 of the tile, K = its rows r0 .. r0 + 7)
MZ_DEV void frag_cols_a(uint32_t (&ah)[4], uint32_t (&al)[4], const float* Ts, int ld, int r0, int c0, int lane) {
  const int g = lane >> 2, t = lane & 3;
  const float* p = Ts + (r0 + t) * ld + c0 + g;
  split_tf32(p[0], ah[0], al[0]);
  split_tf32(p[8], ah[1], al[1]);
  split_tf32(p[4 * ld], ah[2], al[2]);
  split_tf32(p[4 * ld + 8], ah[3], al[3]);
}
// Transposed B fragment (N = columns c0 .. c0 + 7 of the tile, K = its rows r0 .. r0 + 7)
MZ_DEV void frag_cols_b(uint32_t (&bh)[2], uint32_t (&bl)[2], const float* Ts, int ld, int r0, int c0, int lane) {
  const int g = lane >> 2, t = lane & 3;
  const float* p = Ts + (r0 + t) * ld + c0 + g;
  split_tf32(p[0], bh[0], bl[0]);
  split_tf32(p[4 * ld], bh[1], bl[1]);
}

// Packed B operand of a matrix Bm [N][K] (B[k][n] = Bm[n][k]): 32-bit word ((nt KS + ks) 32 + lane) 4 + i holds
// split(Bm[8 nt + g][kk]) with g = lane >> 2, kk = 8 ks + 2 (lane & 3) + (i & 1), its hi part for i < 2 and its lo
// part for i >= 2: b0 / b1 of k-step ks of n-tile nt as hi and lo, one 16-byte load per lane.  Zeros outside N x K.
__global__ void pack_kernel(PackParams p) {
  const mz_pack_job job = p.jobs[blockIdx.y];
  if (job.src == nullptr) {  // a buffer to clear before the step (gradients): n 32-bit words
    for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < job.n; w += gridDim.x * blockDim.x) job.dst[w] = 0u;
    return;
  }
  const int KS = (job.k + 7) >> 3, NTl = (job.n + 7) >> 3;
  const int words = NTl * KS * 128;
  for (int w = blockIdx.x * blockDim.x + threadIdx.x; w < words; w += gridDim.x * blockDim.x) {
    const int i = w & 3, lane = (w >> 2) & 31, rest = w >> 7;
    const int ks = rest % KS, nt = rest / KS;
    const int nn = 8 * nt + (lane >> 2), kk = 8 * ks + 2 * (lane & 3) + (i & 1);
    const float v = (nn < job.n && kk < job.k) ? job.src[(size_t)nn * job.stride_n + (size_t)kk * job.stride_k] : 0.0f;
    uint32_t hi, lo;
    split_tf32(v, hi, lo);
    job.dst[w] = i < 2 ? hi : lo;
  }
}

// The 3xTF32 operand format of mz_learner_tc.cuh's kernels: float32 tiles, a k unit is one m16n8k8 k-step.  The
// chain kernels trade two loads for registers: held across the contractions, gamma / beta (chain_fwd) and the next
// step's LayerNorm inputs during the dH one (chain_bwd) would spill.
struct Tf32x3 {
  using T = float;
  static constexpr int K = 8;
  static constexpr int MAX_TILES = 1;
  static constexpr bool GAMMA_IN_REGS = false, EARLY_LN_LOAD = false;
  static constexpr int PACK_CTA_WORDS = 2048, CLEAR_CTA_WORDS = 2048, PACK_MAX_CTAS = 148;
  static constexpr void (*pack_kernel)(PackParams) = ::pack_kernel;

  static MZ_DEV T cvt(float x) { return x; }
  using T2 = float2;
  static MZ_DEV T2 pair(float a, float b) { return make_float2(a, b); }
  static int64_t packed_words(int32_t n, int32_t k) { return (int64_t)((n + 7) / 8) * ((k + 7) / 8) * 128; }

  // acc[MT][NTW][4] += A (16 MT rows x 8 KS, row-major float32 in shared memory) * B (packed; n-tiles nt0 ..
  // nt0 + NTW - 1).  lds: k-steps per n-tile of the packed image (KS, or more when Bp points at a K slice of a wider
  // image).  The B fragments of the next k-step are in flight while a step computes.
  template <int MT>
  static MZ_DEV void gemm_wide(float (&acc)[MT][NTW][4], const float* As, int lda, const uint32_t* __restrict__ Bp, int KS,
                               int nt0, int lane, int lds) {
    const uint4* bp = reinterpret_cast<const uint4*>(Bp) + (size_t)nt0 * lds * 32 + lane;
    uint4 b[NTW];
#pragma unroll
    for (int n = 0; n < NTW; ++n) b[n] = __ldg(bp + (size_t)n * lds * 32);
    for (int ks = 0; ks < KS; ++ks) {
      uint4 bn[NTW];
      if (ks + 1 < KS) {
#pragma unroll
        for (int n = 0; n < NTW; ++n) bn[n] = __ldg(bp + ((size_t)n * lds + ks + 1) * 32);
      }
      uint32_t ah[MT][4], al[MT][4];
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) frag_rows(ah[mt], al[mt], As, lda, 16 * mt, 8 * ks, lane);
#pragma unroll
      for (int n = 0; n < NTW; ++n)
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) mma_tf32(acc[mt][n], al[mt], b[n].x, b[n].y);
#pragma unroll
      for (int n = 0; n < NTW; ++n)
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) mma_tf32(acc[mt][n], ah[mt], b[n].z, b[n].w);
#pragma unroll
      for (int n = 0; n < NTW; ++n)
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) mma_tf32(acc[mt][n], ah[mt], b[n].x, b[n].y);
      if (ks + 1 < KS) {
#pragma unroll
        for (int n = 0; n < NTW; ++n) b[n] = bn[n];
      }
    }
  }

  // acc[MT][4] = A (16 MT rows x 512, row-major float32 in shared memory) * B (packed, KS = 64; n-tile nt).  The B
  // fragments go in blocks of four k-steps, the next block in flight; the two cross terms and the hi x hi term sum in
  // separate accumulators (two independent mma chains per m-tile), added at the end.
  template <int MT>
  static MZ_DEV void gemm_tall(float (&acc)[MT][4], const float* As, int lda, const uint32_t* __restrict__ Bp, int nt, int lane) {
    constexpr int BLK = 4;
    const uint4* bp = reinterpret_cast<const uint4*>(Bp) + (size_t)nt * KS_TALL * 32 + lane;
    uint4 b[BLK];
#pragma unroll
    for (int i = 0; i < BLK; ++i) b[i] = __ldg(bp + i * 32);
    float acc2[MT][4];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[mt][c] = acc2[mt][c] = 0.0f;
#pragma unroll 1
    for (int kb = 0; kb < KS_TALL / BLK; ++kb) {
      uint4 bn[BLK];
      if (kb + 1 < KS_TALL / BLK) {
#pragma unroll
        for (int i = 0; i < BLK; ++i) bn[i] = __ldg(bp + ((kb + 1) * BLK + i) * 32);
      }
#pragma unroll
      for (int i = 0; i < BLK; ++i) {
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          uint32_t ah[4], al[4];
          frag_rows(ah, al, As, lda, 16 * mt, 8 * (kb * BLK + i), lane);
          mma_tf32(acc2[mt], al, b[i].x, b[i].y);
          mma_tf32(acc2[mt], ah, b[i].z, b[i].w);
          mma_tf32(acc[mt], ah, b[i].x, b[i].y);
        }
      }
      if (kb + 1 < KS_TALL / BLK) {
#pragma unroll
        for (int i = 0; i < BLK; ++i) b[i] = bn[i];
      }
    }
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[mt][c] += acc2[mt][c];
  }

  // gW1[j][k] += sum_r dH[r][j] X[r][k] for columns [0, cols) of the X tile in Xs, to gw1[j * ld + k]: M = the warp's
  // hidden units, N = input features in chunks of 64, K = the CTA's 32 rows (transposed fragments of both tiles)
  static MZ_DEV void gw1_phase(float* gw1, int ld, int cols, const float* Xs, const float* dHs, float* stage, int warp,
                               int lane) {
    for (int mt = 0; mt < CW / 16; ++mt) {
      for (int chunk = 0; 64 * chunk < cols; ++chunk) {
        float acc[8][4];
#pragma unroll
        for (int n = 0; n < 8; ++n)
#pragma unroll
          for (int c = 0; c < 4; ++c) acc[n][c] = 0.0f;
#pragma unroll
        for (int ks = 0; ks < RT / 8; ++ks) {
          uint32_t ah[4], al[4];
          frag_cols_a(ah, al, dHs, HLD, 8 * ks, CW * warp + 16 * mt, lane);
#pragma unroll
          for (int n = 0; n < 8; ++n) {
            if (64 * chunk + 8 * n < cols) {  // warp-uniform; the tile is zero padded to a multiple of 8 columns
              uint32_t bh[2], bl[2];
              frag_cols_b(bh, bl, Xs, XLD, 8 * ks, 64 * chunk + 8 * n, lane);
              mma_tf32(acc[n], al, bh[0], bh[1]);
              mma_tf32(acc[n], ah, bl[0], bl[1]);
              mma_tf32(acc[n], ah, bh[0], bh[1]);
            }
          }
        }
        tile_add<8>(gw1 + (size_t)(CW * warp + 16 * mt) * ld + 64 * chunk, ld, 16, min(64, cols - 64 * chunk), acc, stage,
                    lane);
      }
    }
  }

  // Backward of one head over the CTA's 32 rows.  In: Xs (input rows; not loaded by the caller when WIDE), dYs (output
  // gradient, zero padded to a multiple of 16 columns).  Out: the four parameter gradients and dX (columns
  // [0, dx_cols)) accumulated into global memory.  WIDE (heads up to MAXIN inputs, no dX above SLICE): the recomputed
  // activation and gW1 each stream X through Xs in slices of SLICE features.
  template <int TILES, bool WIDE>
  static MZ_DEV void backward(const mz_tc_head& h, const float* __restrict__ X, int ldx, float* Xs, const float* dYs, float* Hs,
                              float* dHs, float* __restrict__ dX, int lddx, int dx_cols, int row0, int rows, float* stage,
                              int warp, int lane) {
    static_assert(TILES == 1, "one 32-row tile per CTA");
    const int g = lane >> 2, t = lane & 3;
    uint32_t mask[2];
    if (WIDE)
      hidden_phase_sliced<Tf32x3, 2>(h, X, ldx, row0, rows, Xs, Hs, mask, warp, lane);
    else
      hidden_phase<Tf32x3, 2>(h, Xs, Hs, mask, warp, lane);
    {  // dH = dY W2 for the warp's hidden units, masked by the ReLU -> dHs; gb1 = column sums of dH
      float acc[2][NTW][4];
      zero<2>(acc);
      const int KS = kunits<Tf32x3>(h.d_out);
      gemm_wide<2>(acc, dYs, DYLD, h.w2tp, KS, NTW * warp, lane, KS);
#pragma unroll
      for (int n = 0; n < NTW; ++n) {
        const int j = CW * warp + 8 * n + 2 * t;
        float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
          const uint32_t m = mask[mt] >> (4 * n);
          const float v0 = (m & 1u) ? acc[mt][n][0] : 0.0f, v1 = (m & 2u) ? acc[mt][n][1] : 0.0f;
          const float v2 = (m & 4u) ? acc[mt][n][2] : 0.0f, v3 = (m & 8u) ? acc[mt][n][3] : 0.0f;
          s0 += v0 + v2;
          s1 += v1 + v3;
          pair_at<Tf32x3>(dHs + (16 * mt + g) * HLD + j) = pair(v0, v1);
          pair_at<Tf32x3>(dHs + (16 * mt + g + 8) * HLD + j) = pair(v2, v3);
        }
#pragma unroll
        for (int m = 4; m < 32; m <<= 1) {
          s0 += __shfl_xor_sync(MZ_FULL, s0, m);
          s1 += __shfl_xor_sync(MZ_FULL, s1, m);
        }
        if (g == 0) {
          atomicAdd(h.gb1 + j, s0);
          atomicAdd(h.gb1 + j + 1, s1);
        }
      }
    }
    __syncthreads();
    // dX = dH W1: n-tiles over the warps
    for (int nt = warp; 8 * nt < dx_cols; nt += NW) {
      float acc[2][4];
      gemm_tall<2>(acc, dHs, HLD, h.w1tp, nt, lane);
      const int k = 8 * nt + 2 * t;
#pragma unroll
      for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          const int r = row0 + 16 * mt + g + 8 * half;
          if (r < rows) {
            if (k < dx_cols) atomicAdd(dX + (size_t)r * lddx + k, acc[mt][2 * half]);
            if (k + 1 < dx_cols) atomicAdd(dX + (size_t)r * lddx + k + 1, acc[mt][2 * half + 1]);
          }
        }
      }
    }
    // gW2[o][j] = sum_r dY[r][o] H[r][j]: M = outputs (16 per m-tile), N = the warp's hidden units, K = the CTA's rows
    for (int mt = 0; 16 * mt < h.d_out; ++mt) {
      float acc[NTW][4];
#pragma unroll
      for (int n = 0; n < NTW; ++n)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[n][c] = 0.0f;
#pragma unroll
      for (int ks = 0; ks < RT / 8; ++ks) {
        uint32_t ah[4], al[4];
        frag_cols_a(ah, al, dYs, DYLD, 8 * ks, 16 * mt, lane);
#pragma unroll
        for (int n = 0; n < NTW; ++n) {
          uint32_t bh[2], bl[2];
          frag_cols_b(bh, bl, Hs, HLD, 8 * ks, CW * warp + 8 * n, lane);
          mma_tf32(acc[n], al, bh[0], bh[1]);
          mma_tf32(acc[n], ah, bl[0], bl[1]);
          mma_tf32(acc[n], ah, bh[0], bh[1]);
        }
      }
      tile_add<NTW>(h.gw2 + (size_t)(16 * mt) * LW + CW * warp, LW, h.d_out - 16 * mt, CW, acc, stage, lane);
    }
    if (!WIDE) {
      gw1_phase(h.gw1, h.d_in, h.d_in, Xs, dHs, stage, warp, lane);
    } else {
      for (int k0 = 0; k0 < h.d_in; k0 += SLICE) {
        const int w = min(SLICE, h.d_in - k0);
        if (h.d_in > SLICE) {  // one slice: still in Xs from the hidden phase
          __syncthreads();
          load_rows<Tf32x3>(Xs, XLD, X + k0, ldx, row0, rows, w, round_up<K>(w));
          __syncthreads();
        }
        gw1_phase(h.gw1 + k0, h.d_in, w, Xs, dHs, stage, warp, lane);
      }
    }
  }
};

}  // namespace

extern "C" {

int64_t mz_learner_packed_words_tf32x3(int32_t n, int32_t k) { return n < 1 || k < 1 ? 0 : Tf32x3::packed_words(n, k); }
int mz_learner_pack_tf32x3(int32_t njobs, const mz_pack_job* jobs, void* stream) { return pack<Tf32x3>(njobs, jobs, stream); }
int mz_heads_forward_tf32x3(int32_t njobs, const mz_tc_job* jobs, void* stream) { return heads_forward<Tf32x3>(njobs, jobs, stream); }
int mz_heads_backward_tf32x3(int32_t njobs, const mz_tc_job* jobs, void* stream) { return heads_backward<Tf32x3>(njobs, jobs, stream); }
int mz_chain_forward_tf32x3(const mz_tc_chain* chain, void* stream) { return chain_forward<Tf32x3>(chain, stream); }
int mz_chain_backward_tf32x3(const mz_tc_chain* chain, void* stream) { return chain_backward<Tf32x3>(chain, stream); }

}  // extern "C"
