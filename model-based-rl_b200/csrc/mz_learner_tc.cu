// The learner's network forward and backward (Learner.update_weights, learners.py:164-230) on the tensor cores:
// bf16 operands, float32 accumulation, float32 master weights and gradients.
//
// The step of the FCNetwork architecture (networks.py:55-174) is 4 GFLOP behind a chain of 2 (K + 1) + 3 dependent
// two-layer heads, 32..3072 rows each: what bounds it is the length of that chain, not tensor throughput.  So the
// kernels here are built to make the chain short rather than the tiles big:
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
#include <math.h>

#include "mz_common.cuh"

namespace {

constexpr int LW = 512;    // hidden width of every head (networks.py:55-119)
constexpr int RT = 32;     // rows per CTA
constexpr int NW = 16;             // warps per CTA: a CTA runs alone on its SM and every phase is a dependent chain
constexpr int NTH = 32 * NW;       // threads per CTA
constexpr int CW = LW / NW;        // hidden units per warp: warp w owns [CW w, CW w + CW)
constexpr int NTW = CW / 8;        // n-tiles per warp
constexpr int XLD = 136;   // bf16 per row of the input tile (<= 128 features; 272 B: ldmatrix rows 16 B apart mod 128)
constexpr int SLICE = 128;  // features per pass through the input tile: a wider head's input is staged in K slices
constexpr int MAXIN = 1024; // widest head input (the representation head on a wide observation; no dX above SLICE)
constexpr int HLD = 520;   // bf16 per row of the activation tiles
constexpr int DYLD = 72;   // bf16 per row of the output-gradient tile (<= 64 outputs)
constexpr int FLD = 68;    // floats per row of the float32 tile (layer-2 output / dX of the dynamics head)
constexpr int MAXJOBS = 3, MAXPACK = 24;
#ifndef MZ_TC_SKIP
#define MZ_TC_SKIP 0  // diagnostics builds: 1 = weight-gradient atomics only for an impossible value, 2 = no weight-gradient phases, 4 = no dX phase
#endif
#if MZ_TC_SKIP & 1
#define MZ_WG_ADD(p, v) do { if ((v) == 12345.678f) atomicAdd((p), (v)); } while (0)
#else
#define MZ_WG_ADD(p, v) atomicAdd((p), (v))
#endif

#ifdef MZ_TC_TRACE  // diagnostics build: clock64 stamps of CTA 0 (warps 0 and NW - 1) per phase of chain_fwd
__device__ long long g_tc_trace[2][2][16][8];  // [kernel][warp 0 / last][step][phase]
#define TC_T(kern, step, ph)                                                                               \
  do {                                                                                                     \
    if (blockIdx.x == 0 && (threadIdx.x == 0 || threadIdx.x == NTH - 32)) g_tc_trace[kern][threadIdx.x != 0][step][ph] = clock64(); \
  } while (0)
#else
#define TC_T(kern, step, ph)
#endif

struct PlainParams {
  mz_tc_job jobs[MAXJOBS];
};
struct PackParams {
  mz_pack_job jobs[MAXPACK];
};

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
MZ_DEV int round_up32(int v) { return (v + 31) & ~31; }

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

// acc[MT][NTW][4] += A (16 MT rows x 32 KQ, row-major bf16 in shared memory) * B (packed; n-tiles nt0 .. nt0 + NTW - 1).
// ldq: k-step pairs per n-tile of the packed image (KQ, or more when Bp points at a K slice of a wider image).
template <int MT>
MZ_DEV void gemm_wide(float (&acc)[MT][NTW][4], const __nv_bfloat16* As, int lda, const uint32_t* __restrict__ Bp, int KQ,
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
template <int MT>
MZ_DEV void gemm_wide(float (&acc)[MT][NTW][4], const __nv_bfloat16* As, int lda, const uint32_t* __restrict__ Bp, int KQ,
                      int nt0, int lane) {
  gemm_wide<MT>(acc, As, lda, Bp, KQ, nt0, lane, KQ);
}

// acc[MT][4] = A (16 MT rows x 512, row-major bf16 in shared memory) * B (packed, KQ = 16; n-tile nt)
template <int MT>
MZ_DEV void gemm_tall(float (&acc)[MT][4], const __nv_bfloat16* As, int lda, const uint32_t* __restrict__ Bp, int nt,
                      int lane) {
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

// rows [row0, row0 + ROWS) x columns [0, d) of a float32 matrix -> bf16 tile, zeros up to column dpad (a multiple of 32)
// and behind `rows`.  A warp moves 32-column segments; all of a thread's loads are in flight before its first store.
template <int ROWS = RT>
MZ_DEV void load_rows(__nv_bfloat16* Ts, int ld, const float* __restrict__ X, int ldx, int row0, int rows, int d, int dpad) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int spr = dpad >> 5, segs = ROWS * spr;  // segments per row (1..4), in all
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
    if (sg < segs) Ts[r * ld + c] = __float2bfloat16_rn(v[i]);
  }
}

MZ_DEV void red4(float* p, const float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// A warp's 16 x 8 NT accumulator tile (C fragments: rows g, g + 8; columns 8 n + 2 t + {0, 1}) added to global memory:
// element (r, c) -> dst[r * ld + c] for r < rows_ok, c < cols.  Eight rows at a time cross the warp's staging area and
// leave as 16-byte vector reductions over whole lines (one red.v4 per lane moves 512 contiguous bytes per warp) where
// the alignment allows: always when the rows are dense in memory (cols == ld: the eight rows are one span that starts
// at a multiple of 8 ld floats), per row when ld and cols are multiples of 4; scalar atomics otherwise.
// dst must be 16-byte aligned.
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

// H = relu(acc + b1) for the warp's CW hidden units -> Hs (bf16); returns the sign bits (bit 4 n + c of mask[mt])
template <int MT>
MZ_DEV void hidden_epilogue(const mz_tc_head& h, const float (&acc)[MT][NTW][4], __nv_bfloat16* Hs, uint32_t (&mask)[MT],
                            int warp, int lane) {
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
      *reinterpret_cast<uint32_t*>(Hs + (16 * mt + g) * HLD + j) = pack2(v0, v1);
      *reinterpret_cast<uint32_t*>(Hs + (16 * mt + g + 8) * HLD + j) = pack2(v2, v3);
    }
  }
}

// H = relu(W1 X + b1) for the warp's CW hidden units, X in Xs (d_in <= SLICE)
template <int MT>
MZ_DEV void hidden_phase(const mz_tc_head& h, const __nv_bfloat16* Xs, __nv_bfloat16* Hs, uint32_t (&mask)[MT], int warp,
                         int lane) {
  float acc[MT][NTW][4];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int n = 0; n < NTW; ++n)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[mt][n][c] = 0.0f;
  gemm_wide(acc, Xs, XLD, h.w1p, round_up32(h.d_in) >> 5, NTW * warp, lane);
  hidden_epilogue<MT>(h, acc, Hs, mask, warp, lane);
}

// The same for any d_in <= MAXIN, X read from global memory (rows row0 .. row0 + 16 MT of `rows`): layer 1 runs over
// K slices of up to SLICE features, each staged through Xs (16 MT x XLD) by the whole CTA, with the accumulators kept
// across slices -- the k-steps in the order of one pass, so the same sums.  Xs holds the last slice on return.  Every
// thread of the CTA calls it (barriers inside).
template <int MT>
MZ_DEV void hidden_phase_sliced(const mz_tc_head& h, const float* __restrict__ X, int ldx, int row0, int rows,
                                __nv_bfloat16* Xs, __nv_bfloat16* Hs, uint32_t (&mask)[MT], int warp, int lane) {
  float acc[MT][NTW][4];
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int n = 0; n < NTW; ++n)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[mt][n][c] = 0.0f;
  const int KQ = round_up32(h.d_in) >> 5;
  for (int k0 = 0; k0 < h.d_in; k0 += SLICE) {
    const int w = min(SLICE, h.d_in - k0);
    if (k0) __syncthreads();  // every warp is done with the slice before
    load_rows<16 * MT>(Xs, XLD, X + k0, ldx, row0, rows, w, round_up32(w));
    __syncthreads();
    // k-step pair k0 / 32 of every n-tile: 128 words per pair
    gemm_wide<MT>(acc, Xs, XLD, h.w1p + (size_t)k0 * 4, round_up32(w) >> 5, NTW * warp, lane, KQ);
  }
  hidden_epilogue<MT>(h, acc, Hs, mask, warp, lane);
}

// Y = H W2^T + b2: warp w < ceil(d_out / 8) owns outputs [8 w, 8 w + 8).  To global memory (Y != nullptr) or to the
// float32 tile Fs.
MZ_DEV void output_phase(const mz_tc_head& h, const __nv_bfloat16* Hs, float* __restrict__ Y, int ldy, int row0, int rows,
                         float* Fs, int warp, int lane) {
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
      const float y0 = acc[mt][2 * half] + b0, y1 = acc[mt][2 * half + 1] + b1;
      if (Y != nullptr) {
        if (row0 + r < rows) {
          if (o < h.d_out) Y[(size_t)(row0 + r) * ldy + o] = y0;
          if (o + 1 < h.d_out) Y[(size_t)(row0 + r) * ldy + o + 1] = y1;
        }
      } else {
        Fs[r * FLD + o] = y0;
        Fs[r * FLD + o + 1] = y1;
      }
    }
  }
}

// gW1[j][k] += sum_r dH[r][j] X[r][k] for columns [0, cols) of the X tiles in Xs, to gw1[j * ld + k]: M = the warp's
// hidden units, N = input features in chunks of 64, K = the CTA's rows.  One slice of a WIDE head's input; narrow heads
// run the same loop inline over all of X (as one function it changes their register allocation).
template <int TILES>
MZ_DEV void gw1_phase(float* gw1, int ld, int cols, const __nv_bfloat16* Xs, const __nv_bfloat16* dHs, float* stage,
                      int warp, int lane) {
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
      tile_add<8>(gw1 + (size_t)(CW * warp + 16 * mt) * ld + 64 * chunk, ld, 16, min(64, cols - 64 * chunk), acc, stage, lane);
    }
  }
}

// Backward of one head over the CTA's TILES tiles of 32 rows.  In: Xs (input rows, bf16), dYs (output gradient, bf16,
// zero padded to a multiple of 32 columns).  Out: the four parameter gradients (vector reductions: one per weight and
// CTA, so two tiles per CTA halve that traffic), and dX (columns [0, dx_cols)) accumulated into global memory.
// WIDE (heads up to MAXIN inputs, no dX above SLICE): Xs is not loaded by the caller; the recomputed activation and gW1
// each stream X (rows of `ldx` floats) through Xs in slices of SLICE features, so the shared-memory plan is that of a
// narrow head (heads_bwd_smem).
template <int TILES, bool WIDE>
MZ_DEV void backward_tiles(const mz_tc_head& h, const float* __restrict__ X, int ldx, __nv_bfloat16* Xs,
                           const __nv_bfloat16* dYs, __nv_bfloat16* Hs, __nv_bfloat16* dHs, float* __restrict__ dX, int lddx,
                           int dx_cols, int row0, int rows, float* stage, int warp, int lane) {
  const int g = lane >> 2, t = lane & 3;
  TC_T(1, 0, 1);
  float s0[NTW], s1[NTW];  // column sums of the gated dH: gb1
#pragma unroll
  for (int n = 0; n < NTW; ++n) s0[n] = s1[n] = 0.0f;
#pragma unroll 1
  for (int tile = 0; tile < TILES; ++tile) {
    const __nv_bfloat16* Xt = Xs + tile * RT * XLD;
    const __nv_bfloat16* dYt = dYs + tile * RT * DYLD;
    __nv_bfloat16* Ht = Hs + tile * RT * HLD;
    __nv_bfloat16* dHt = dHs + tile * RT * HLD;
    uint32_t mask[2];
    if (WIDE)
      hidden_phase_sliced<2>(h, X, ldx, row0 + RT * tile, rows, Xs + tile * RT * XLD, Ht, mask, warp, lane);
    else
      hidden_phase<2>(h, Xt, Ht, mask, warp, lane);
    // dH = dY W2 for the warp's hidden units, masked by the ReLU -> dHs
    float acc[2][NTW][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int n = 0; n < NTW; ++n)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[mt][n][c] = 0.0f;
    gemm_wide<2>(acc, dYt, DYLD, h.w2tp, round_up32(h.d_out) >> 5, NTW * warp, lane);
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
        *reinterpret_cast<uint32_t*>(dHt + (16 * mt + g) * HLD + j) = pack2(v0, v1);
        *reinterpret_cast<uint32_t*>(dHt + (16 * mt + g + 8) * HLD + j) = pack2(v2, v3);
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
  if (dx_cols > 0 && !(MZ_TC_SKIP & 4)) {
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
  if (MZ_TC_SKIP & 2) return;
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
      tile_add<8>(h.gw1 + (size_t)(CW * warp + 16 * mt) * h.d_in + 64 * chunk, h.d_in, 16, min(64, h.d_in - 64 * chunk), acc,
                  stage, lane);
    }
  }
  } else {
    for (int k0 = 0; k0 < h.d_in; k0 += SLICE) {
      const int w = min(SLICE, h.d_in - k0);
      if (h.d_in > SLICE) {  // one slice: still in Xs from the hidden phase
        __syncthreads();
#pragma unroll
        for (int tile = 0; tile < TILES; ++tile)
          load_rows(Xs + tile * RT * XLD, XLD, X + k0, ldx, row0 + RT * tile, rows, w, round_up32(w));
        __syncthreads();
      }
      gw1_phase<TILES>(h.gw1 + k0, h.d_in, w, Xs, dHs, stage, warp, lane);
    }
  }
  TC_T(1, 0, 6);
}

struct Tiles {
  __nv_bfloat16 *Xs, *Hs, *dHs, *dYs;
  float* Fs;
};
constexpr int STAGE = 8 * 68;  // floats per warp: eight rows of a weight-gradient tile
constexpr size_t FWD_SMEM = (size_t)RT * XLD * 2 + (size_t)RT * HLD * 2 + (size_t)RT * FLD * 4;
MZ_DEV Tiles carve(unsigned char* base) {  // the forward kernels' tiles
  Tiles t;
  t.Xs = reinterpret_cast<__nv_bfloat16*>(base);
  t.Hs = t.Xs + RT * XLD;
  t.dHs = nullptr;
  t.dYs = nullptr;
  t.Fs = reinterpret_cast<float*>(t.Hs + RT * HLD);
  return t;
}

// ---- the output heads: one job per blockIdx.y --------------------------------------------------------------------
// WIDE: some job has d_in > SLICE; every job's layer 1 then runs over slices (hidden_phase_sliced)
template <bool WIDE>
__global__ void __launch_bounds__(NTH) heads_fwd_kernel(PlainParams p) {
  extern __shared__ __align__(16) unsigned char tc_smem[];
  const mz_tc_job& job = p.jobs[blockIdx.y];
  const int row0 = blockIdx.x * RT;
  if (row0 >= job.rows) return;
  const Tiles s = carve(tc_smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t mask[2];
  if (WIDE) {
    hidden_phase_sliced<2>(job.head, job.x, job.ldx, row0, job.rows, s.Xs, s.Hs, mask, warp, lane);
  } else {
    load_rows(s.Xs, XLD, job.x, job.ldx, row0, job.rows, job.head.d_in, round_up32(job.head.d_in));
    __syncthreads();
    hidden_phase<2>(job.head, s.Xs, s.Hs, mask, warp, lane);
  }
  __syncthreads();
  output_phase(job.head, s.Hs, job.y, job.ldy, row0, job.rows, nullptr, warp, lane);
}

// Shared memory: TILES x 32 rows of X (XLD), H and dH (HLD), dY (DYLD) in bf16, plus NW staging areas -- 112 KB at
// TILES = 1, 190 KB at TILES = 2 of the 227 KB.  Full-width X tiles of a 1024-feature head (64.5 KB per 32 rows instead
// of 8.5 KB) would not fit at TILES = 2, so WIDE streams X through the same XLD tiles in slices of SLICE features
// (backward_tiles): the same plan, the same heads_bwd_smem, for every width.
template <int TILES, bool WIDE>
__global__ void __launch_bounds__(NTH) heads_bwd_kernel(PlainParams p) {
  extern __shared__ __align__(16) unsigned char tc_smem[];
  const mz_tc_job& job = p.jobs[blockIdx.y];
  constexpr int RTT = RT * TILES;  // rows per CTA
  const int row0 = blockIdx.x * RTT;
  if (row0 >= job.rows) return;
  __nv_bfloat16* Xs = reinterpret_cast<__nv_bfloat16*>(tc_smem);
  __nv_bfloat16* Hs = Xs + RTT * XLD;
  __nv_bfloat16* dHs = Hs + RTT * HLD;
  __nv_bfloat16* dYs = dHs + RTT * HLD;
  float* stage = reinterpret_cast<float*>(dYs + RTT * DYLD);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const mz_tc_head& h = job.head;
  TC_T(1, 0, 0);
#pragma unroll
  for (int tile = 0; tile < TILES; ++tile) {
    if (!WIDE) load_rows(Xs + tile * RT * XLD, XLD, job.x, job.ldx, row0 + RT * tile, job.rows, h.d_in, round_up32(h.d_in));
    load_rows(dYs + tile * RT * DYLD, DYLD, job.dy, job.ldy, row0 + RT * tile, job.rows, h.d_out, round_up32(h.d_out));
  }
  if ((int)threadIdx.x < h.d_out) {  // gb2[o] = sum_r dY[r][o]
    float part[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll 8
    for (int r = 0; r < RTT; ++r)
      if (row0 + r < job.rows) part[r & 3] += job.dy[(size_t)(row0 + r) * job.ldy + threadIdx.x];
    atomicAdd(h.gb2 + threadIdx.x, (part[0] + part[1]) + (part[2] + part[3]));
  }
  __syncthreads();
  backward_tiles<TILES, WIDE>(h, job.x, job.ldx, Xs, dYs, Hs, dHs, job.dx, job.lddx, job.dx != nullptr ? h.d_in : 0, row0,
                               job.rows, stage + warp * STAGE, warp, lane);
}
constexpr size_t heads_bwd_smem(int tiles) {
  return (size_t)tiles * RT * (XLD + 2 * HLD + DYLD) * 2 + (size_t)NW * STAGE * 4;
}

// ---- the recurrent chain ---------------------------------------------------------------------------------------
// A CTA owns 16 MT rows for all steps.  MT = 1 (16 rows, twice the CTAs) whenever that still fits one wave: the phases
// of a step are bound by the issue rate of the warp-level mma on the CTA's SM (~16 cycles per m16n8k16 and scheduler),
// so half the rows per CTA is half the time per step.
// LayerNorm phases: a warp owns 16 MT / NW rows at once, LPR lanes per row; lane (rr, c8) holds columns c8 + LPR i
// (i < CPL) of its row, so the row statistics are log2(LPR) shuffle steps and the rows run side by side.
template <int MT>
struct ChainGeo {
  static constexpr int ROWS = 16 * MT;
  static constexpr int LPR = 32 * NW / ROWS;  // lanes per row (MT = 1: 32, MT = 2: 16)
  static constexpr int CPL = 64 / LPR;        // columns per lane
  static constexpr size_t FWD_SMEM = (size_t)ROWS * XLD * 2 + (size_t)ROWS * HLD * 2 + (size_t)ROWS * FLD * 4;
  static constexpr size_t BWD_SMEM = (size_t)ROWS * DYLD * 2 + (size_t)ROWS * HLD * 2 + (size_t)ROWS * FLD * 4 + 2 * 64 * 4;
};

// WIDE: first.d_in > SLICE -- step 0 streams x0 through Xs in slices (hidden_phase_sliced); the LayerNorm epilogues
// write the next step's input into Xs as for a narrow first head
template <int MT, bool WIDE>
__global__ void __launch_bounds__(NTH) chain_fwd_kernel(mz_tc_chain c) {
  using G = ChainGeo<MT>;
  constexpr int ROWS = G::ROWS, LPR = G::LPR, CPL = G::CPL;
  extern __shared__ __align__(16) unsigned char tc_smem[];
  const int row0 = blockIdx.x * ROWS;
  __nv_bfloat16* Xs = reinterpret_cast<__nv_bfloat16*>(tc_smem);
  __nv_bfloat16* Hs = Xs + ROWS * XLD;
  float* Fs = reinterpret_cast<float*>(Hs + ROWS * HLD);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = c.d, A = c.num_actions, next_pad = round_up32(d + A);
  const int r = (32 / LPR) * warp + lane / LPR, c8 = lane % LPR, row = row0 + r;
  const bool live = row < c.rows;
  const float inv_d = 1.0f / (float)d;
  const int g = lane >> 2, t = lane & 3;
  float gam[CPL], bet[CPL];
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int col = c8 + LPR * i;
    gam[i] = col < d ? __ldg(c.gamma + col) : 0.0f;
    bet[i] = col < d ? __ldg(c.beta + col) : 0.0f;
  }
  if (!WIDE) {
    load_rows<ROWS>(Xs, XLD, c.x0, c.ldx0, row0, c.rows, c.first.d_in, round_up32(c.first.d_in));
    __syncthreads();
  }
  for (int step = 0; step < c.steps; ++step) {
    const mz_tc_head& h = step ? c.next : c.first;
    const int act = (live && c.actions != nullptr && step < c.action_steps)
                        ? __ldg(c.actions + (size_t)row * c.action_stride + step) : -1;  // in flight during the head
    TC_T(0, step, 0);
    uint32_t mask[MT];
    if (WIDE && step == 0)
      hidden_phase_sliced<MT>(h, c.x0, c.ldx0, row0, c.rows, Xs, Hs, mask, warp, lane);
    else
      hidden_phase<MT>(h, Xs, Hs, mask, warp, lane);
    TC_T(0, step, 1);
    if (step && c.relu_mask != nullptr)  // the backward chain gates dH with these bits instead of recomputing the layer
      reinterpret_cast<uint2*>(c.relu_mask)[((size_t)step * gridDim.x + blockIdx.x) * NTH + threadIdx.x] =
          make_uint2(mask[0], MT > 1 ? mask[MT - 1] : 0u);
    __syncthreads();
    TC_T(0, step, 2);
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
    TC_T(0, step, 3);
    __syncthreads();
    TC_T(0, step, 4);
    // LayerNorm (networks.py:144, eps 1e-5, biased variance) + ReLU, one-hot action appended: the next step's input
    float v[CPL], sum = 0.0f;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      v[i] = c8 + LPR * i < d ? Fs[r * FLD + c8 + LPR * i] : 0.0f;
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
      Xs[r * XLD + col] = __float2bfloat16_rn(live ? out : 0.0f);
    }
    for (int col = 64 + c8; col < next_pad; col += LPR) {  // d + A > 64 (A = 18): the rest of the one-hot
      const float out = (col < d + A && col - d == act) ? 1.0f : 0.0f;
      if (live && col < d + A) c.xs[grow * c.ldxs + col] = out;
      Xs[r * XLD + col] = __float2bfloat16_rn(out);
    }
    if (live && c8 == 0) {
      c.mean[grow] = mean;
      c.rstd[grow] = rstd;
    }
    TC_T(0, step, 5);
    __syncthreads();
    TC_T(0, step, 6);
  }
}

// The serial part of the chain's backward: per step LayerNorm backward -> dY (kept in dyall for the weight gradients)
// -> dH = dY W2 gated by the forward's ReLU bits -> dX = dH W1 -> next LayerNorm backward.  The parameter gradients of
// the two heads do not sit on this chain: mz_heads_backward_tc computes them afterwards from (xs, dyall) over all
// K B + B rows in parallel.
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
__global__ void __launch_bounds__(NTH) chain_bwd_kernel(mz_tc_chain c) {
  using G = ChainGeo<MT>;
  constexpr int ROWS = G::ROWS, LPR = G::LPR, CPL = G::CPL;
  extern __shared__ __align__(16) unsigned char tc_smem[];
  const int row0 = blockIdx.x * ROWS;
  __nv_bfloat16* dYs = reinterpret_cast<__nv_bfloat16*>(tc_smem);
  __nv_bfloat16* dHs = dYs + ROWS * DYLD;
  float* Fs = reinterpret_cast<float*>(dHs + ROWS * HLD);
  float* red = Fs + ROWS * FLD;  // [2][64]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = c.d, out_pad = round_up32(d);
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
    if (step) ln_load<CPL, LPR>(nxt, c, step - 1, row, live, c8);  // in flight during this step's contractions
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
      if (col < out_pad) dYs[r * DYLD + col] = __float2bfloat16_rn(dy);
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
#pragma unroll
      for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int n = 0; n < NTW; ++n)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[mt][n][q] = 0.0f;
      gemm_wide<MT>(acc, dYs, DYLD, h.w2tp, round_up32(h.d_out) >> 5, NTW * warp, lane);
#pragma unroll
      for (int n = 0; n < NTW; ++n) {
        const int j = CW * warp + 8 * n + 2 * t;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          const uint32_t m = (mt ? mbits.y : mbits.x) >> (4 * n);
          *reinterpret_cast<uint32_t*>(dHs + (16 * mt + g) * HLD + j) =
              pack2((m & 1u) ? acc[mt][n][0] : 0.0f, (m & 2u) ? acc[mt][n][1] : 0.0f);
          *reinterpret_cast<uint32_t*>(dHs + (16 * mt + g + 8) * HLD + j) =
              pack2((m & 4u) ? acc[mt][n][2] : 0.0f, (m & 8u) ? acc[mt][n][3] : 0.0f);
        }
      }
      __syncthreads();
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

bool g_tc_attr = false;
int tc_attrs() {
  if (g_tc_attr) return 0;
  cudaError_t e;
  const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
  if ((e = cudaFuncSetAttribute(heads_fwd_kernel<false>, attr, (int)FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(heads_fwd_kernel<true>, attr, (int)FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_fwd_kernel<1, false>, attr, (int)ChainGeo<1>::FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_fwd_kernel<2, false>, attr, (int)ChainGeo<2>::FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_fwd_kernel<1, true>, attr, (int)ChainGeo<1>::FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_fwd_kernel<2, true>, attr, (int)ChainGeo<2>::FWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(heads_bwd_kernel<1, false>, attr, (int)heads_bwd_smem(1))) != cudaSuccess ||
      (e = cudaFuncSetAttribute(heads_bwd_kernel<2, false>, attr, (int)heads_bwd_smem(2))) != cudaSuccess ||
      (e = cudaFuncSetAttribute(heads_bwd_kernel<1, true>, attr, (int)heads_bwd_smem(1))) != cudaSuccess ||
      (e = cudaFuncSetAttribute(heads_bwd_kernel<2, true>, attr, (int)heads_bwd_smem(2))) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_bwd_kernel<1>, attr, (int)ChainGeo<1>::BWD_SMEM)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(chain_bwd_kernel<2>, attr, (int)ChainGeo<2>::BWD_SMEM)) != cudaSuccess)
    return (int)e;
  g_tc_attr = true;
  return 0;
}

// rows per CTA of the chain kernels: 16 while that is at most one wave of CTAs, else 32 (forward and backward of a
// step must agree: the ReLU bits are stored per CTA and thread)
int chain_mt(int rows) { return (rows + 15) / 16 <= 148 ? 1 : 2; }

// (w1tp only feeds dX, which a head wider than SLICE does not have: its image need not exist)
bool head_ok(const mz_tc_head& h, bool backward) {
  if (h.d_in < 1 || h.d_in > MAXIN || h.d_out < 1 || h.d_out > 64 || !h.w1p || !h.w2p || !h.b1 || !h.b2) return false;
  if (backward && (!h.w2tp || (h.d_in <= SLICE && !h.w1tp) || !h.gw1 || !h.gb1 || !h.gw2 || !h.gb2)) return false;
  if (backward && (((uintptr_t)h.gw1 | (uintptr_t)h.gw2) & 15)) return false;  // weight gradients leave as red.v4
  return true;
}

bool chain_ok(const mz_tc_chain* c, bool backward) {
  if (!c || c->rows < 1 || c->steps < 1 || c->d < 1 || c->d > 64 || c->num_actions < 0 || c->d + c->num_actions > 128) return false;
  // (the chain's backward reads the packed images only; the heads' gradients are mz_heads_backward_tc's job)
  if (!head_ok(c->first, false) || c->first.d_out != c->d) return false;
  if (c->steps > 1 && (!head_ok(c->next, false) || c->next.d_out != c->d || c->next.d_in != c->d + c->num_actions)) return false;
  if (backward && c->steps > 1 && (!c->next.w2tp || !c->next.w1tp)) return false;
  if (!c->x0 || c->ldx0 < c->first.d_in || !c->gamma || !c->beta || !c->xs || c->ldxs < c->d + c->num_actions || !c->yall ||
      !c->mean || !c->rstd)
    return false;
  if (c->actions && (c->action_stride < c->action_steps || c->action_steps < 0)) return false;
  if (backward && (!c->dxs || !c->ggamma || !c->gbeta || !c->dyall || (c->steps > 1 && !c->relu_mask))) return false;
  return true;
}

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

int64_t mz_learner_packed_words(int32_t n, int32_t k) {
  if (n < 1 || k < 1) return 0;
  return (int64_t)((n + 7) / 8) * ((k + 31) / 32) * 128;
}

int mz_learner_pack(int32_t njobs, const mz_pack_job* jobs, void* stream) {
  if (njobs < 1 || njobs > MAXPACK || !jobs) return MZ_ERR_BAD_ARG;
  PackParams p;
  int64_t most = 0;
  for (int i = 0; i < njobs; ++i) {
    if (!jobs[i].dst || jobs[i].n < 1 || (jobs[i].src && jobs[i].k < 1)) return MZ_ERR_BAD_ARG;
    p.jobs[i] = jobs[i];
    const int64_t w = jobs[i].src ? mz_learner_packed_words(jobs[i].n, jobs[i].k) : (jobs[i].n + 3) / 4;
    most = w > most ? w : most;
  }
  int blocks = (int)((most + 1023) / 1024);
  blocks = blocks < 1 ? 1 : (blocks > 96 ? 96 : blocks);
  pack_kernel<<<dim3(blocks, njobs), 256, 0, (cudaStream_t)stream>>>(p);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_heads_forward_tc(int32_t njobs, const mz_tc_job* jobs, void* stream) {
  if (njobs < 1 || njobs > MAXJOBS || !jobs) return MZ_ERR_BAD_ARG;
  PlainParams p;
  int most = 0;
  bool wide = false;
  for (int i = 0; i < njobs; ++i) {
    const mz_tc_job& j = jobs[i];
    if (!head_ok(j.head, false) || j.rows < 1 || !j.x || !j.y || j.ldx < j.head.d_in || j.ldy < j.head.d_out) return MZ_ERR_BAD_ARG;
    p.jobs[i] = j;
    most = j.rows > most ? j.rows : most;
    wide = wide || j.head.d_in > SLICE;
  }
  if (int rc = tc_attrs()) return rc;
  const dim3 grid((most + RT - 1) / RT, njobs);
  if (wide)
    heads_fwd_kernel<true><<<grid, NTH, FWD_SMEM, (cudaStream_t)stream>>>(p);
  else
    heads_fwd_kernel<false><<<grid, NTH, FWD_SMEM, (cudaStream_t)stream>>>(p);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_heads_backward_tc(int32_t njobs, const mz_tc_job* jobs, void* stream) {
  if (njobs < 1 || njobs > MAXJOBS || !jobs) return MZ_ERR_BAD_ARG;
  PlainParams p;
  int most = 0;
  bool wide = false;
  for (int i = 0; i < njobs; ++i) {
    const mz_tc_job& j = jobs[i];
    if (!head_ok(j.head, true) || j.rows < 1 || !j.x || !j.dy || j.ldx < j.head.d_in || j.ldy < j.head.d_out ||
        (j.dx && (j.lddx < j.head.d_in || j.head.d_in > SLICE)))
      return MZ_ERR_BAD_ARG;
    p.jobs[i] = j;
    most = j.rows > most ? j.rows : most;
    wide = wide || j.head.d_in > SLICE;
  }
  if (int rc = tc_attrs()) return rc;
  // more CTAs than one wave of single-tile CTAs: two tiles per CTA (half the weight-gradient reductions, one wave)
  int ctas = 0;
  for (int i = 0; i < njobs; ++i) ctas += (jobs[i].rows + RT - 1) / RT;
  const dim3 grid2((most + 2 * RT - 1) / (2 * RT), njobs), grid1((most + RT - 1) / RT, njobs);
  cudaStream_t st = (cudaStream_t)stream;
  if (ctas > 148 && wide)
    heads_bwd_kernel<2, true><<<grid2, NTH, heads_bwd_smem(2), st>>>(p);
  else if (ctas > 148)
    heads_bwd_kernel<2, false><<<grid2, NTH, heads_bwd_smem(2), st>>>(p);
  else if (wide)
    heads_bwd_kernel<1, true><<<grid1, NTH, heads_bwd_smem(1), st>>>(p);
  else
    heads_bwd_kernel<1, false><<<grid1, NTH, heads_bwd_smem(1), st>>>(p);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_chain_forward_tc(const mz_tc_chain* chain, void* stream) {
  if (!chain_ok(chain, false)) return MZ_ERR_BAD_ARG;
  if (int rc = tc_attrs()) return rc;
  const bool wide = chain->first.d_in > SLICE;
  cudaStream_t st = (cudaStream_t)stream;
  if (chain_mt(chain->rows) == 1 && wide)
    chain_fwd_kernel<1, true><<<(chain->rows + 15) / 16, NTH, ChainGeo<1>::FWD_SMEM, st>>>(*chain);
  else if (chain_mt(chain->rows) == 1)
    chain_fwd_kernel<1, false><<<(chain->rows + 15) / 16, NTH, ChainGeo<1>::FWD_SMEM, st>>>(*chain);
  else if (wide)
    chain_fwd_kernel<2, true><<<(chain->rows + 31) / 32, NTH, ChainGeo<2>::FWD_SMEM, st>>>(*chain);
  else
    chain_fwd_kernel<2, false><<<(chain->rows + 31) / 32, NTH, ChainGeo<2>::FWD_SMEM, st>>>(*chain);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_chain_backward_tc(const mz_tc_chain* chain, void* stream) {
  if (!chain_ok(chain, true)) return MZ_ERR_BAD_ARG;
  if (int rc = tc_attrs()) return rc;
  if (chain_mt(chain->rows) == 1)
    chain_bwd_kernel<1><<<(chain->rows + 15) / 16, NTH, ChainGeo<1>::BWD_SMEM, (cudaStream_t)stream>>>(*chain);
  else
    chain_bwd_kernel<2><<<(chain->rows + 31) / 32, NTH, ChainGeo<2>::BWD_SMEM, (cudaStream_t)stream>>>(*chain);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

}  // extern "C"
