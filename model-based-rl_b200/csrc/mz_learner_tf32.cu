// The learner's network forward and backward (Learner.update_weights, learners.py:164-230) on the tensor cores at
// float32 accuracy: every contraction is three TF32 mma.sync.m16n8k8 products on split operands (x = x_hi + x_lo,
// w = w_hi + w_lo; x w ~= x_lo w_hi + x_hi w_lo + x_hi w_hi, float32 accumulation, see split_tf32), so there is no
// bf16 rounding point anywhere.  float32 master weights, gradients and optimiser state as in the other two learners.
//
// The step has the four-launch structure of mz_learner_tc.cu (chain_fwd, heads_fwd, heads_bwd, chain_bwd) and its
// argument structs; what changes is the operand format:
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
// Shared memory is twice that of the bf16 tiles, so every kernel keeps one 32-row tile per CTA (heads_bwd: 190 KB;
// the bf16 kernel's two-tile plan would need 354 KB); the chain kernels keep 16 or 32 rows as in mz_learner_tc.cu.
#include <math.h>

#include "mz_common.cuh"

namespace {

constexpr int LW = 512;    // hidden width of every head (networks.py:55-119)
constexpr int RT = 32;     // rows per CTA of the head kernels
constexpr int NW = 16;             // warps per CTA
constexpr int NTH = 32 * NW;       // threads per CTA
constexpr int CW = LW / NW;        // hidden units per warp: warp w owns [CW w, CW w + CW)
constexpr int NTW = CW / 8;        // n-tiles per warp
constexpr int XLD = 136;   // floats per row of the input tile (<= 128 features); 8 (mod 32), see the header
constexpr int SLICE = 128;  // features per pass through the input tile: a wider head's input is staged in K slices
constexpr int MAXIN = 1024; // widest head input (the representation head on a wide observation; no dX above SLICE)
constexpr int HLD = 520;   // floats per row of the activation tiles
constexpr int DYLD = 72;   // floats per row of the output-gradient tile (<= 64 outputs)
constexpr int FLD = 68;    // floats per row of the layer-2 output / dX tile of the chain kernels
constexpr int KS_TALL = LW / 8;  // k-steps of a contraction over the 512 hidden units
constexpr int MAXJOBS = 3, MAXPACK = 24;

struct PlainParams {
  mz_tc_job jobs[MAXJOBS];
};
struct PackParams {
  mz_pack_job jobs[MAXPACK];
};

// x = hi + lo: hi = x cut to TF32's 11 significant bits, lo = the exact float32 remainder, of which the tensor core
// reads the top 11 bits.  What a product loses -- lo's own cut and the x_lo * w_lo term -- is below 2^-20 of it
// (the argument of mz_fcnet_tf32.cu).
MZ_DEV void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
// D (16 x 8, f32) += A (16 x 8, row) * B (8 x 8, col), TF32 operands
MZ_DEV void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
MZ_DEV int round_up8(int v) { return (v + 7) & ~7; }

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

// acc[MT][NTW][4] += A (16 MT rows x 8 KS, row-major float32 in shared memory) * B (packed; n-tiles nt0 ..
// nt0 + NTW - 1).  lds: k-steps per n-tile of the packed image (KS, or more when Bp points at a K slice of a wider
// image).  The B fragments of the next k-step are in flight while a step computes.
template <int MT>
MZ_DEV void gemm_wide(float (&acc)[MT][NTW][4], const float* As, int lda, const uint32_t* __restrict__ Bp, int KS, int nt0,
                      int lane, int lds) {
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
// fragments go in blocks of eight k-steps, the next block in flight; the two cross terms and the hi x hi term sum in
// separate accumulators (two independent mma chains per m-tile), added at the end.
template <int MT>
MZ_DEV void gemm_tall(float (&acc)[MT][4], const float* As, int lda, const uint32_t* __restrict__ Bp, int nt, int lane) {
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

// rows [row0, row0 + ROWS) x columns [0, d) of a float32 matrix -> tile, zeros up to column dpad (<= 128) and behind
// `rows`.  A warp moves 32-column segments; all of a thread's loads are in flight before its first store.
template <int ROWS = RT>
MZ_DEV void load_rows(float* Ts, int ld, const float* __restrict__ X, int ldx, int row0, int rows, int d, int dpad) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int spr = (dpad + 31) >> 5, segs = ROWS * spr;  // segments per row (1..4), in all
  constexpr int NI = (4 * ROWS + NW - 1) / NW;
  float v[NI];
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int sg = warp + NW * i, r = sg / spr, c = 32 * (sg - r * spr) + lane;
    v[i] = (sg < segs && row0 + r < rows && c < d) ? X[(size_t)(row0 + r) * ldx + c] : 0.0f;
  }
#pragma unroll
  for (int i = 0; i < NI; ++i) {
    const int sg = warp + NW * i, r = sg / spr, c = 32 * (sg - r * spr) + lane;
    if (sg < segs && c < dpad) Ts[r * ld + c] = v[i];
  }
}

MZ_DEV void red4(float* p, const float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// A warp's 16 x 8 NT accumulator tile (C fragments: rows g, g + 8; columns 8 n + 2 t + {0, 1}) added to global memory:
// element (r, c) -> dst[r * ld + c] for r < rows_ok, c < cols.  Eight rows at a time cross the warp's staging area and
// leave as 16-byte vector reductions where the alignment allows (always when the rows are dense in memory, per row
// when ld and cols are multiples of 4), scalar atomics otherwise.  dst must be 16-byte aligned.
template <int NT>
MZ_DEV void tile_add(float* __restrict__ dst, int ld, int rows_ok, int cols, const float (&acc)[NT][4], float* stage, int lane) {
  const int g = lane >> 2, t = lane & 3;
  const bool dense = cols == ld;
  const int sld = dense ? cols : 68;  // staging row stride (68: 16-byte aligned rows, banks spread)
  for (int half = 0; half < 2; ++half) {
    if (8 * half >= rows_ok) break;  // warp-uniform
    __syncwarp();
#pragma unroll
    for (int n = 0; n < NT; ++n) {
      const int c = 8 * n + 2 * t;
      if (c < cols) stage[g * sld + c] = acc[n][2 * half];
      if (c + 1 < cols) stage[g * sld + c + 1] = acc[n][2 * half + 1];
    }
    __syncwarp();
    float* out = dst + (size_t)(8 * half) * ld;
    const int live = min(8, rows_ok - 8 * half);
    if (dense) {
      const float4* s4 = reinterpret_cast<const float4*>(stage);
      for (int i = lane; i < (live * cols) >> 2; i += 32) red4(out + 4 * i, s4[i]);
      for (int i = ((live * cols) & ~3) + lane; i < live * cols; i += 32) atomicAdd(out + i, stage[i]);
    } else if (((ld | cols) & 3) == 0) {
      const int c4n = cols >> 2;
      for (int i = lane; i < live * c4n; i += 32) {
        const int r = i / c4n, c4 = i - r * c4n;
        red4(out + (size_t)r * ld + 4 * c4, *reinterpret_cast<const float4*>(stage + r * sld + 4 * c4));
      }
    } else {
      for (int i = lane; i < live * cols; i += 32) {
        const int r = i / cols, c = i - r * cols;
        atomicAdd(out + (size_t)r * ld + c, stage[r * sld + c]);
      }
    }
  }
}

template <int MT>
MZ_DEV void zero(float (&acc)[MT][NTW][4]) {
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int n = 0; n < NTW; ++n)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[mt][n][c] = 0.0f;
}

// H = relu(acc + b1) for the warp's CW hidden units -> Hs; returns the sign bits (bit 4 n + c of mask[mt]: the
// layout of mz_learner_tc.cu, so mz_chain_mask_words sizes both)
template <int MT>
MZ_DEV void hidden_epilogue(const mz_tc_head& h, const float (&acc)[MT][NTW][4], float* Hs, uint32_t (&mask)[MT], int warp,
                            int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int mt = 0; mt < MT; ++mt) mask[mt] = 0u;
#pragma unroll
  for (int n = 0; n < NTW; ++n) {
    const int j = CW * warp + 8 * n + 2 * t;
    const float2 bb = make_float2(__ldg(h.b1 + j), __ldg(h.b1 + j + 1));  // views of a flat buffer: 4-byte aligned
#pragma unroll
    for (int mt = 0; mt < MT; ++mt) {
      const float v0 = fmaxf(acc[mt][n][0] + bb.x, 0.0f), v1 = fmaxf(acc[mt][n][1] + bb.y, 0.0f);
      const float v2 = fmaxf(acc[mt][n][2] + bb.x, 0.0f), v3 = fmaxf(acc[mt][n][3] + bb.y, 0.0f);
      mask[mt] |= (v0 > 0.0f ? 1u : 0u) << (4 * n) | (v1 > 0.0f ? 2u : 0u) << (4 * n) | (v2 > 0.0f ? 4u : 0u) << (4 * n) |
                  (v3 > 0.0f ? 8u : 0u) << (4 * n);
      *reinterpret_cast<float2*>(Hs + (16 * mt + g) * HLD + j) = make_float2(v0, v1);
      *reinterpret_cast<float2*>(Hs + (16 * mt + g + 8) * HLD + j) = make_float2(v2, v3);
    }
  }
}

// H = relu(W1 X + b1) for the warp's CW hidden units, X in Xs (d_in <= SLICE, zero padded to a multiple of 8)
template <int MT>
MZ_DEV void hidden_phase(const mz_tc_head& h, const float* Xs, float* Hs, uint32_t (&mask)[MT], int warp, int lane) {
  float acc[MT][NTW][4];
  zero<MT>(acc);
  const int KS = round_up8(h.d_in) >> 3;
  gemm_wide<MT>(acc, Xs, XLD, h.w1p, KS, NTW * warp, lane, KS);
  hidden_epilogue<MT>(h, acc, Hs, mask, warp, lane);
}

// The same for any d_in <= MAXIN, X read from global memory (rows row0 .. row0 + 16 MT of `rows`): layer 1 runs over
// K slices of up to SLICE features, each staged through Xs by the whole CTA, with the accumulators kept across slices.
// Xs holds the last slice on return.  Every thread of the CTA calls it (barriers inside).
template <int MT>
MZ_DEV void hidden_phase_sliced(const mz_tc_head& h, const float* __restrict__ X, int ldx, int row0, int rows, float* Xs,
                                float* Hs, uint32_t (&mask)[MT], int warp, int lane) {
  float acc[MT][NTW][4];
  zero<MT>(acc);
  const int KS = round_up8(h.d_in) >> 3;
  for (int k0 = 0; k0 < h.d_in; k0 += SLICE) {
    const int w = min(SLICE, h.d_in - k0);
    if (k0) __syncthreads();  // every warp is done with the slice before
    load_rows<16 * MT>(Xs, XLD, X + k0, ldx, row0, rows, w, round_up8(w));
    __syncthreads();
    // k-step k0 / 8 of every n-tile: 128 words per k-step
    gemm_wide<MT>(acc, Xs, XLD, h.w1p + (size_t)k0 * 16, round_up8(w) >> 3, NTW * warp, lane, KS);
  }
  hidden_epilogue<MT>(h, acc, Hs, mask, warp, lane);
}

// Y = H W2^T + b2: warp w < ceil(d_out / 8) owns outputs [8 w, 8 w + 8).  To global memory.
MZ_DEV void output_phase(const mz_tc_head& h, const float* Hs, float* __restrict__ Y, int ldy, int row0, int rows, int warp,
                         int lane) {
  if (8 * warp >= h.d_out) return;
  float acc[2][4];
  gemm_tall<2>(acc, Hs, HLD, h.w2p, warp, lane);
  const int g = lane >> 2, o = 8 * warp + 2 * (lane & 3);
  const float b0 = o < h.d_out ? __ldg(h.b2 + o) : 0.0f, b1 = o + 1 < h.d_out ? __ldg(h.b2 + o + 1) : 0.0f;
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
      const int r = 16 * mt + g + 8 * half;
      if (row0 + r < rows) {
        if (o < h.d_out) Y[(size_t)(row0 + r) * ldy + o] = acc[mt][2 * half] + b0;
        if (o + 1 < h.d_out) Y[(size_t)(row0 + r) * ldy + o + 1] = acc[mt][2 * half + 1] + b1;
      }
    }
  }
}

// gW1[j][k] += sum_r dH[r][j] X[r][k] for columns [0, cols) of the X tile in Xs, to gw1[j * ld + k]: M = the warp's
// hidden units, N = input features in chunks of 64, K = the CTA's 32 rows (transposed fragments of both tiles)
MZ_DEV void gw1_phase(float* gw1, int ld, int cols, const float* Xs, const float* dHs, float* stage, int warp, int lane) {
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
      tile_add<8>(gw1 + (size_t)(CW * warp + 16 * mt) * ld + 64 * chunk, ld, 16, min(64, cols - 64 * chunk), acc, stage, lane);
    }
  }
}

// Backward of one head over the CTA's 32 rows.  In: Xs (input rows; not loaded by the caller when WIDE), dYs (output
// gradient, zero padded to a multiple of 16 columns).  Out: the four parameter gradients and dX (columns
// [0, dx_cols)) accumulated into global memory.  WIDE (heads up to MAXIN inputs, no dX above SLICE): the recomputed
// activation and gW1 each stream X through Xs in slices of SLICE features.
template <bool WIDE>
MZ_DEV void backward_tile(const mz_tc_head& h, const float* __restrict__ X, int ldx, float* Xs, const float* dYs, float* Hs,
                          float* dHs, float* __restrict__ dX, int lddx, int dx_cols, int row0, int rows, float* stage, int warp,
                          int lane) {
  const int g = lane >> 2, t = lane & 3;
  uint32_t mask[2];
  if (WIDE)
    hidden_phase_sliced<2>(h, X, ldx, row0, rows, Xs, Hs, mask, warp, lane);
  else
    hidden_phase<2>(h, Xs, Hs, mask, warp, lane);
  {  // dH = dY W2 for the warp's hidden units, masked by the ReLU -> dHs; gb1 = column sums of dH
    float acc[2][NTW][4];
    zero<2>(acc);
    const int KS = round_up8(h.d_out) >> 3;
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
        *reinterpret_cast<float2*>(dHs + (16 * mt + g) * HLD + j) = make_float2(v0, v1);
        *reinterpret_cast<float2*>(dHs + (16 * mt + g + 8) * HLD + j) = make_float2(v2, v3);
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
        load_rows(Xs, XLD, X + k0, ldx, row0, rows, w, round_up8(w));
        __syncthreads();
      }
      gw1_phase(h.gw1 + k0, h.d_in, w, Xs, dHs, stage, warp, lane);
    }
  }
}

constexpr int STAGE = 8 * 68;  // floats per warp: eight rows of a weight-gradient tile
constexpr size_t FWD_SMEM = (size_t)RT * (XLD + HLD) * 4;
constexpr size_t BWD_SMEM = (size_t)RT * (XLD + 2 * HLD + DYLD) * 4 + (size_t)NW * STAGE * 4;  // 190 KB

// ---- the output heads: one job per blockIdx.y --------------------------------------------------------------------
// WIDE: some job has d_in > SLICE; every job's layer 1 then runs over slices (hidden_phase_sliced)
template <bool WIDE>
__global__ void __launch_bounds__(NTH) heads_fwd_tf32x3_kernel(PlainParams p) {
  extern __shared__ __align__(16) float tf_smem[];
  const mz_tc_job& job = p.jobs[blockIdx.y];
  const int row0 = blockIdx.x * RT;
  if (row0 >= job.rows) return;
  float* Xs = tf_smem;
  float* Hs = Xs + RT * XLD;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t mask[2];
  if (WIDE) {
    hidden_phase_sliced<2>(job.head, job.x, job.ldx, row0, job.rows, Xs, Hs, mask, warp, lane);
  } else {
    load_rows(Xs, XLD, job.x, job.ldx, row0, job.rows, job.head.d_in, round_up8(job.head.d_in));
    __syncthreads();
    hidden_phase<2>(job.head, Xs, Hs, mask, warp, lane);
  }
  __syncthreads();
  output_phase(job.head, Hs, job.y, job.ldy, row0, job.rows, warp, lane);
}

// Shared memory: 32 rows of X (XLD), H and dH (HLD), dY (DYLD) in float32, plus NW staging areas: 190 KB of the 227 KB.
template <bool WIDE>
__global__ void __launch_bounds__(NTH) heads_bwd_tf32x3_kernel(PlainParams p) {
  extern __shared__ __align__(16) float tf_smem[];
  const mz_tc_job& job = p.jobs[blockIdx.y];
  const int row0 = blockIdx.x * RT;
  if (row0 >= job.rows) return;
  float* Xs = tf_smem;
  float* Hs = Xs + RT * XLD;
  float* dHs = Hs + RT * HLD;
  float* dYs = dHs + RT * HLD;
  float* stage = dYs + RT * DYLD;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const mz_tc_head& h = job.head;
  if (!WIDE) load_rows(Xs, XLD, job.x, job.ldx, row0, job.rows, h.d_in, round_up8(h.d_in));
  load_rows(dYs, DYLD, job.dy, job.ldy, row0, job.rows, h.d_out, (h.d_out + 15) & ~15);  // gW2 reads m-tiles of 16
  if ((int)threadIdx.x < h.d_out) {  // gb2[o] = sum_r dY[r][o]
    float part[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll 8
    for (int r = 0; r < RT; ++r)
      if (row0 + r < job.rows) part[r & 3] += job.dy[(size_t)(row0 + r) * job.ldy + threadIdx.x];
    atomicAdd(h.gb2 + threadIdx.x, (part[0] + part[1]) + (part[2] + part[3]));
  }
  __syncthreads();
  backward_tile<WIDE>(h, job.x, job.ldx, Xs, dYs, Hs, dHs, job.dx, job.lddx, job.dx != nullptr ? h.d_in : 0, row0, job.rows,
                      stage + warp * STAGE, warp, lane);
}

// ---- the recurrent chain ---------------------------------------------------------------------------------------
// A CTA owns 16 MT rows for all steps (MT = 1 whenever that still fits one wave, as in mz_learner_tc.cu).
// LayerNorm phases: a warp owns 16 MT / NW rows at once, LPR lanes per row; lane (rr, c8) holds columns c8 + LPR i
// (i < CPL) of its row.
template <int MT>
struct ChainGeo {
  static constexpr int ROWS = 16 * MT;
  static constexpr int LPR = 32 * NW / ROWS;  // lanes per row (MT = 1: 32, MT = 2: 16)
  static constexpr int CPL = 64 / LPR;        // columns per lane
  static constexpr size_t FWD_SMEM = (size_t)ROWS * (XLD + HLD + FLD) * 4;
  static constexpr size_t BWD_SMEM = (size_t)ROWS * (DYLD + HLD + FLD) * 4 + 2 * 64 * 4;
};

// WIDE: first.d_in > SLICE -- step 0 streams x0 through Xs in slices (hidden_phase_sliced)
template <int MT, bool WIDE>
__global__ void __launch_bounds__(NTH) chain_fwd_tf32x3_kernel(mz_tc_chain c) {
  using G = ChainGeo<MT>;
  constexpr int ROWS = G::ROWS, LPR = G::LPR, CPL = G::CPL;
  extern __shared__ __align__(16) float tf_smem[];
  const int row0 = blockIdx.x * ROWS;
  float* Xs = tf_smem;
  float* Hs = Xs + ROWS * XLD;
  float* Fs = Hs + ROWS * HLD;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = c.d, A = c.num_actions, next_pad = round_up8(d + A);
  const int r = (32 / LPR) * warp + lane / LPR, c8 = lane % LPR, row = row0 + r;
  const bool live = row < c.rows;
  const float inv_d = 1.0f / (float)d;
  const int g = lane >> 2, t = lane & 3;
  if (!WIDE) {
    load_rows<ROWS>(Xs, XLD, c.x0, c.ldx0, row0, c.rows, c.first.d_in, round_up8(c.first.d_in));
    __syncthreads();
  }
  for (int step = 0; step < c.steps; ++step) {
    const mz_tc_head& h = step ? c.next : c.first;
    const int act = (live && c.actions != nullptr && step < c.action_steps)
                        ? __ldg(c.actions + (size_t)row * c.action_stride + step) : -1;  // in flight during the head
    uint32_t mask[MT];
    if (WIDE && step == 0)
      hidden_phase_sliced<MT>(h, c.x0, c.ldx0, row0, c.rows, Xs, Hs, mask, warp, lane);
    else
      hidden_phase<MT>(h, Xs, Hs, mask, warp, lane);
    if (step && c.relu_mask != nullptr)  // the backward chain gates dH with these bits instead of recomputing the layer
      reinterpret_cast<uint2*>(c.relu_mask)[((size_t)step * gridDim.x + blockIdx.x) * NTH + threadIdx.x] =
          make_uint2(mask[0], MT > 1 ? mask[MT - 1] : 0u);
    __syncthreads();
    if (8 * warp < d) {  // Y = H W2^T + b2: warp w owns outputs [8 w, 8 w + 8) -> Fs
      float acc[MT][4];
      gemm_tall<MT>(acc, Hs, HLD, h.w2p, warp, lane);
      const int o = 8 * warp + 2 * t;
      const float b0 = o < d ? __ldg(h.b2 + o) : 0.0f, b1 = o + 1 < d ? __ldg(h.b2 + o + 1) : 0.0f;
#pragma unroll
      for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          Fs[(16 * mt + g + 8 * half) * FLD + o] = acc[mt][2 * half] + b0;
          Fs[(16 * mt + g + 8 * half) * FLD + o + 1] = acc[mt][2 * half + 1] + b1;
        }
      }
    }
    __syncthreads();
    // LayerNorm (networks.py:144, eps 1e-5, biased variance) + ReLU, one-hot action appended: the next step's input
    // (gamma / beta from L1 per step: registers held across the contractions would spill)
    float v[CPL], gam[CPL], bet[CPL], sum = 0.0f;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int col = c8 + LPR * i;
      v[i] = col < d ? Fs[r * FLD + col] : 0.0f;
      gam[i] = col < d ? __ldg(c.gamma + col) : 0.0f;
      bet[i] = col < d ? __ldg(c.beta + col) : 0.0f;
      sum += v[i];
    }
#pragma unroll
    for (int m = 1; m < LPR; m <<= 1) sum += __shfl_xor_sync(MZ_FULL, sum, m);
    const float mean = sum * inv_d;
    float q = 0.0f;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const float cen = c8 + LPR * i < d ? v[i] - mean : 0.0f;
      q += cen * cen;
    }
#pragma unroll
    for (int m = 1; m < LPR; m <<= 1) q += __shfl_xor_sync(MZ_FULL, q, m);
    const float rstd = rsqrtf(q * inv_d + 1e-5f);
    const size_t grow = (size_t)step * c.rows + row;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int col = c8 + LPR * i;
      float out = 0.0f;
      if (col < d) {
        out = fmaxf((v[i] - mean) * rstd * gam[i] + bet[i], 0.0f);
        if (live) c.yall[grow * d + col] = v[i];
      } else if (col < d + A) {
        out = (col - d == act) ? 1.0f : 0.0f;
      }
      if (live && col < d + A) c.xs[grow * c.ldxs + col] = out;
      Xs[r * XLD + col] = live ? out : 0.0f;
    }
    for (int col = 64 + c8; col < next_pad; col += LPR) {  // d + A > 64 (A = 18): the rest of the one-hot
      const float out = (col < d + A && col - d == act) ? 1.0f : 0.0f;
      if (live && col < d + A) c.xs[grow * c.ldxs + col] = out;
      Xs[r * XLD + col] = out;
    }
    if (live && c8 == 0) {
      c.mean[grow] = mean;
      c.rstd[grow] = rstd;
    }
    __syncthreads();
  }
}

// The serial part of the chain's backward: per step LayerNorm backward -> dY (kept in dyall for the weight gradients)
// -> dH = dY W2 gated by the forward's ReLU bits -> dX = dH W1 -> next LayerNorm backward.  The parameter gradients of
// the two heads are mz_heads_backward_tf32x3's job, over all K B + B rows in parallel.
template <int CPL>
struct LnIn {
  float up[CPL], hv[CPL], yv[CPL], mean, rstd;
};
template <int CPL, int LPR>
MZ_DEV void ln_load(LnIn<CPL>& v, const mz_tc_chain& c, int step, int row, bool live, int c8) {
  const size_t grow = (size_t)step * c.rows + row;
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int col = c8 + LPR * i;
    const bool in = live && col < c.d;
    v.up[i] = in ? c.dxs[grow * c.ldxs + col] : 0.0f;
    v.hv[i] = in ? c.xs[grow * c.ldxs + col] : 0.0f;
    v.yv[i] = in ? c.yall[grow * c.d + col] : 0.0f;
  }
  v.mean = live ? c.mean[grow] : 0.0f;
  v.rstd = live ? c.rstd[grow] : 0.0f;
}

template <int MT>
__global__ void __launch_bounds__(NTH) chain_bwd_tf32x3_kernel(mz_tc_chain c) {
  using G = ChainGeo<MT>;
  constexpr int ROWS = G::ROWS, LPR = G::LPR, CPL = G::CPL;
  extern __shared__ __align__(16) float tf_smem[];
  const int row0 = blockIdx.x * ROWS;
  float* dYs = tf_smem;
  float* dHs = dYs + ROWS * DYLD;
  float* Fs = dHs + ROWS * HLD;
  float* red = Fs + ROWS * FLD;  // [2][64]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = c.d, out_pad = round_up8(d);
  const int r = (32 / LPR) * warp + lane / LPR, c8 = lane % LPR, row = row0 + r;
  const bool live = row < c.rows;
  const float inv_d = 1.0f / (float)d;
  if (threadIdx.x < 2 * 64) red[threadIdx.x] = 0.0f;
  __syncthreads();
  float gam[CPL], gg[CPL], gb[CPL];
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    gam[i] = c8 + LPR * i < d ? __ldg(c.gamma + c8 + LPR * i) : 0.0f;
    gg[i] = gb[i] = 0.0f;
  }
  LnIn<CPL> cur, nxt;
  ln_load<CPL, LPR>(cur, c, c.steps - 1, row, live, c8);
  for (int step = c.steps - 1; step >= 0; --step) {
    uint2 mbits = make_uint2(0u, 0u);
    if (step) mbits = reinterpret_cast<const uint2*>(c.relu_mask)[((size_t)step * gridDim.x + blockIdx.x) * NTH + threadIdx.x];
    // backward of relu(LayerNorm(y)): gradient = heads' part (+ the dynamics head's dX of the step after), scaled by
    // the hook (learners.py:201) for the states the dynamics produced
    const float scale = step ? c.hook_scale : 1.0f;
    float gi[CPL], xh[CPL], s1 = 0.0f, s2 = 0.0f;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int col = c8 + LPR * i;
      float u = cur.up[i];
      if (step + 1 < c.steps && col < d) u += Fs[r * FLD + col];
      gi[i] = cur.hv[i] > 0.0f ? u * scale : 0.0f;
      xh[i] = (cur.yv[i] - cur.mean) * cur.rstd;
      const float dxh = gi[i] * gam[i];
      s1 += dxh;
      s2 += dxh * xh[i];
    }
#pragma unroll
    for (int m = 1; m < LPR; m <<= 1) {
      s1 += __shfl_xor_sync(MZ_FULL, s1, m);
      s2 += __shfl_xor_sync(MZ_FULL, s2, m);
    }
    const float m1 = s1 * inv_d, m2 = s2 * inv_d;
    const size_t grow = (size_t)step * c.rows + row;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int col = c8 + LPR * i;
      const float dy = (live && col < d) ? cur.rstd * (gi[i] * gam[i] - m1 - xh[i] * m2) : 0.0f;
      if (col < out_pad) dYs[r * DYLD + col] = dy;
      if (live && col < d) c.dyall[grow * d + col] = dy;
      gg[i] += gi[i] * xh[i];
      gb[i] += gi[i];
    }
    if (step == 0) break;  // the representation head's input needs no gradient
    __syncthreads();
    {  // dH = dY W2 for the warp's hidden units, gated by the forward's ReLU bits -> dHs
      const mz_tc_head& h = c.next;
      const int g = lane >> 2, t = lane & 3;
      float acc[MT][NTW][4];
      zero<MT>(acc);
      const int KS = round_up8(h.d_out) >> 3;
      gemm_wide<MT>(acc, dYs, DYLD, h.w2tp, KS, NTW * warp, lane, KS);
#pragma unroll
      for (int n = 0; n < NTW; ++n) {
        const int j = CW * warp + 8 * n + 2 * t;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          const uint32_t m = (mt ? mbits.y : mbits.x) >> (4 * n);
          *reinterpret_cast<float2*>(dHs + (16 * mt + g) * HLD + j) =
              make_float2((m & 1u) ? acc[mt][n][0] : 0.0f, (m & 2u) ? acc[mt][n][1] : 0.0f);
          *reinterpret_cast<float2*>(dHs + (16 * mt + g + 8) * HLD + j) =
              make_float2((m & 4u) ? acc[mt][n][2] : 0.0f, (m & 8u) ? acc[mt][n][3] : 0.0f);
        }
      }
      ln_load<CPL, LPR>(nxt, c, step - 1, row, live, c8);  // in flight during the dX contraction (registers of
      __syncthreads();                                    // the dH one would spill)
      // dX = dH W1, the hidden-state columns only -> Fs
      for (int nt = warp; 8 * nt < d; nt += NW) {
        float a2[MT][4];
        gemm_tall<MT>(a2, dHs, HLD, h.w1tp, nt, lane);
        const int k = 8 * nt + 2 * t;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            Fs[(16 * mt + g + 8 * half) * FLD + k] = a2[mt][2 * half];
            Fs[(16 * mt + g + 8 * half) * FLD + k + 1] = a2[mt][2 * half + 1];
          }
        }
      }
    }
    __syncthreads();
    cur = nxt;
  }
  // LayerNorm weight / bias gradients: the rows of a warp by shuffles, the warps through shared memory
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
#pragma unroll
    for (int m = LPR; m < 32; m <<= 1) {
      gg[i] += __shfl_xor_sync(MZ_FULL, gg[i], m);
      gb[i] += __shfl_xor_sync(MZ_FULL, gb[i], m);
    }
    if (lane < LPR && c8 + LPR * i < d) {
      atomicAdd(&red[c8 + LPR * i], gg[i]);
      atomicAdd(&red[64 + c8 + LPR * i], gb[i]);
    }
  }
  __syncthreads();
  if ((int)threadIdx.x < d) {
    atomicAdd(c.ggamma + threadIdx.x, red[threadIdx.x]);
    atomicAdd(c.gbeta + threadIdx.x, red[64 + threadIdx.x]);
  }
}

bool g_attr = false;
int set_attrs() {
  if (g_attr) return 0;
  cudaError_t e;
  const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
  if ((e = cudaFuncSetAttribute(heads_fwd_tf32x3_kernel<false>, attr, (int)FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(heads_fwd_tf32x3_kernel<true>, attr, (int)FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(heads_bwd_tf32x3_kernel<false>, attr, (int)BWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(heads_bwd_tf32x3_kernel<true>, attr, (int)BWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_fwd_tf32x3_kernel<1, false>, attr, (int)ChainGeo<1>::FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_fwd_tf32x3_kernel<2, false>, attr, (int)ChainGeo<2>::FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_fwd_tf32x3_kernel<1, true>, attr, (int)ChainGeo<1>::FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_fwd_tf32x3_kernel<2, true>, attr, (int)ChainGeo<2>::FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_bwd_tf32x3_kernel<1>, attr, (int)ChainGeo<1>::BWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_bwd_tf32x3_kernel<2>, attr, (int)ChainGeo<2>::BWD_SMEM)) != cudaSuccess)
    return (int)e;
  g_attr = true;
  return 0;
}

// rows per CTA of the chain kernels: 16 while that is at most one wave of CTAs, else 32 (forward and backward of a
// step must agree: the ReLU bits are stored per CTA and thread)
int chain_mt(int rows) { return (rows + 15) / 16 <= 148 ? 1 : 2; }

// MZ_OK, MZ_ERR_UNSUPPORTED for a shape beyond the kernels (d_in > MAXIN, d_out > 64), else MZ_ERR_BAD_ARG.
// (w1tp only feeds dX, which a head wider than SLICE does not have: its image need not exist)
int head_check(const mz_tc_head& h, bool backward) {
  if (h.d_in > MAXIN || h.d_out > 64) return MZ_ERR_UNSUPPORTED;
  if (h.d_in < 1 || h.d_out < 1 || !h.w1p || !h.w2p || !h.b1 || !h.b2) return MZ_ERR_BAD_ARG;
  if (backward && (!h.w2tp || (h.d_in <= SLICE && !h.w1tp) || !h.gw1 || !h.gb1 || !h.gw2 || !h.gb2)) return MZ_ERR_BAD_ARG;
  if (backward && (((uintptr_t)h.gw1 | (uintptr_t)h.gw2) & 15)) return MZ_ERR_BAD_ARG;  // weight gradients leave as red.v4
  return MZ_OK;
}

int chain_check(const mz_tc_chain* c, bool backward) {
  if (!c) return MZ_ERR_BAD_ARG;
  if (c->d > 64 || c->d + c->num_actions > SLICE) return MZ_ERR_UNSUPPORTED;
  if (c->rows < 1 || c->steps < 1 || c->d < 1 || c->num_actions < 0) return MZ_ERR_BAD_ARG;
  if (int rc = head_check(c->first, false)) return rc;
  if (c->first.d_out != c->d) return MZ_ERR_BAD_ARG;
  if (c->steps > 1) {
    if (int rc = head_check(c->next, false)) return rc;
    if (c->next.d_out != c->d || c->next.d_in != c->d + c->num_actions) return MZ_ERR_BAD_ARG;
  }
  if (backward && c->steps > 1 && (!c->next.w2tp || !c->next.w1tp)) return MZ_ERR_BAD_ARG;
  if (!c->x0 || c->ldx0 < c->first.d_in || !c->gamma || !c->beta || !c->xs || c->ldxs < c->d + c->num_actions || !c->yall ||
      !c->mean || !c->rstd)
    return MZ_ERR_BAD_ARG;
  if (c->actions && (c->action_stride < c->action_steps || c->action_steps < 0)) return MZ_ERR_BAD_ARG;
  if (backward && (!c->dxs || !c->ggamma || !c->gbeta || !c->dyall || (c->steps > 1 && !c->relu_mask))) return MZ_ERR_BAD_ARG;
  return MZ_OK;
}

}  // namespace

extern "C" {

int64_t mz_learner_packed_words_tf32x3(int32_t n, int32_t k) {
  if (n < 1 || k < 1) return 0;
  return (int64_t)((n + 7) / 8) * ((k + 7) / 8) * 128;
}

int mz_learner_pack_tf32x3(int32_t njobs, const mz_pack_job* jobs, void* stream) {
  if (njobs < 1 || njobs > MAXPACK || !jobs) return MZ_ERR_BAD_ARG;
  PackParams p;
  int64_t most = 0;
  for (int i = 0; i < njobs; ++i) {
    if (!jobs[i].dst || jobs[i].n < 1 || (jobs[i].src && jobs[i].k < 1)) return MZ_ERR_BAD_ARG;
    p.jobs[i] = jobs[i];
    const int64_t w = jobs[i].src ? mz_learner_packed_words_tf32x3(jobs[i].n, jobs[i].k) : jobs[i].n;
    most = w > most ? w : most;
  }
  int blocks = (int)((most + 2047) / 2048);
  blocks = blocks < 1 ? 1 : (blocks > 148 ? 148 : blocks);
  pack_kernel<<<dim3(blocks, njobs), 256, 0, (cudaStream_t)stream>>>(p);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_heads_forward_tf32x3(int32_t njobs, const mz_tc_job* jobs, void* stream) {
  if (njobs < 1 || njobs > MAXJOBS || !jobs) return MZ_ERR_BAD_ARG;
  PlainParams p;
  int most = 0;
  bool wide = false;
  for (int i = 0; i < njobs; ++i) {
    const mz_tc_job& j = jobs[i];
    if (int rc = head_check(j.head, false)) return rc;
    if (j.rows < 1 || !j.x || !j.y || j.ldx < j.head.d_in || j.ldy < j.head.d_out) return MZ_ERR_BAD_ARG;
    p.jobs[i] = j;
    most = j.rows > most ? j.rows : most;
    wide = wide || j.head.d_in > SLICE;
  }
  if (int rc = set_attrs()) return rc;
  const dim3 grid((most + RT - 1) / RT, njobs);
  if (wide)
    heads_fwd_tf32x3_kernel<true><<<grid, NTH, FWD_SMEM, (cudaStream_t)stream>>>(p);
  else
    heads_fwd_tf32x3_kernel<false><<<grid, NTH, FWD_SMEM, (cudaStream_t)stream>>>(p);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_heads_backward_tf32x3(int32_t njobs, const mz_tc_job* jobs, void* stream) {
  if (njobs < 1 || njobs > MAXJOBS || !jobs) return MZ_ERR_BAD_ARG;
  PlainParams p;
  int most = 0;
  bool wide = false;
  for (int i = 0; i < njobs; ++i) {
    const mz_tc_job& j = jobs[i];
    if (int rc = head_check(j.head, true)) return rc;
    if (j.rows < 1 || !j.x || !j.dy || j.ldx < j.head.d_in || j.ldy < j.head.d_out ||
        (j.dx && (j.lddx < j.head.d_in || j.head.d_in > SLICE)))
      return MZ_ERR_BAD_ARG;
    p.jobs[i] = j;
    most = j.rows > most ? j.rows : most;
    wide = wide || j.head.d_in > SLICE;
  }
  if (int rc = set_attrs()) return rc;
  const dim3 grid((most + RT - 1) / RT, njobs);
  if (wide)
    heads_bwd_tf32x3_kernel<true><<<grid, NTH, BWD_SMEM, (cudaStream_t)stream>>>(p);
  else
    heads_bwd_tf32x3_kernel<false><<<grid, NTH, BWD_SMEM, (cudaStream_t)stream>>>(p);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_chain_forward_tf32x3(const mz_tc_chain* chain, void* stream) {
  if (int rc = chain_check(chain, false)) return rc;
  if (int rc = set_attrs()) return rc;
  const bool wide = chain->first.d_in > SLICE;
  cudaStream_t st = (cudaStream_t)stream;
  if (chain_mt(chain->rows) == 1 && wide)
    chain_fwd_tf32x3_kernel<1, true><<<(chain->rows + 15) / 16, NTH, ChainGeo<1>::FWD_SMEM, st>>>(*chain);
  else if (chain_mt(chain->rows) == 1)
    chain_fwd_tf32x3_kernel<1, false><<<(chain->rows + 15) / 16, NTH, ChainGeo<1>::FWD_SMEM, st>>>(*chain);
  else if (wide)
    chain_fwd_tf32x3_kernel<2, true><<<(chain->rows + 31) / 32, NTH, ChainGeo<2>::FWD_SMEM, st>>>(*chain);
  else
    chain_fwd_tf32x3_kernel<2, false><<<(chain->rows + 31) / 32, NTH, ChainGeo<2>::FWD_SMEM, st>>>(*chain);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_chain_backward_tf32x3(const mz_tc_chain* chain, void* stream) {
  if (int rc = chain_check(chain, true)) return rc;
  if (int rc = set_attrs()) return rc;
  if (chain_mt(chain->rows) == 1)
    chain_bwd_tf32x3_kernel<1><<<(chain->rows + 15) / 16, NTH, ChainGeo<1>::BWD_SMEM, (cudaStream_t)stream>>>(*chain);
  else
    chain_bwd_tf32x3_kernel<2><<<(chain->rows + 31) / 32, NTH, ChainGeo<2>::BWD_SMEM, (cudaStream_t)stream>>>(*chain);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

}  // extern "C"
