// The learner's network forward and backward on the tensor cores, everything but the operand format: the tile plan,
// the four kernels of a step and their host side.  mz_learner_tc.cu (bf16 operands) and mz_learner_tf32.cu (3xTF32
// operands, float32 accuracy) each define a format policy F and instantiate these templates with it:
//
//   using T                 the element of the shared-memory tiles (X, H, dH, dY)
//   T cvt(float)            a float stored into a tile;  T2 pair(a, b): two adjacent ones (pair_at)
//   K                       features per packed k unit: tiles are zero padded to multiples of K columns, and the
//                           packed weight images hold 128 words per n-tile and k unit
//   gemm_wide / gemm_tall   the contractions over packed B images: 16 MT rows x k units into the warp's NTW n-tiles,
//                           and 16 MT rows x 512 into one n-tile
//   backward<TILES, WIDE>   the backward of one head over a heads_bwd CTA's TILES x 32 rows, after its X / dY tiles
//   MAX_TILES               the most 32-row tiles per heads_bwd CTA that fit the shared memory
//   GAMMA_IN_REGS           chain_fwd keeps the LayerNorm gamma / beta in registers across the steps (else: read from
//                           L1 in every step's LayerNorm)
//   EARLY_LN_LOAD           chain_bwd loads the next step's LayerNorm inputs at the top of a step (else: after the dH
//                           contraction, while dX computes)
//   pack_kernel, packed_words, PACK_CTA_WORDS, CLEAR_CTA_WORDS, PACK_MAX_CTAS   the weight images and their launch
//
// The policy is the last template argument of a kernel, so its instantiations keep the mangled-name prefixes of the
// per-format kernels they replaced (heads_bwd_kernel<2, false, Bf16> starts as heads_bwd_kernel<2, false> did).
//
// The two register-pressure choices are what keeps each format's chain kernels free of spills.
#pragma once
#include <math.h>

#include "mz_common.cuh"

namespace {

constexpr int LW = 512;    // hidden width of every head (networks.py:55-119)
constexpr int RT = 32;     // rows per tile: the heads' CTAs own TILES of them
constexpr int NW = 16;             // warps per CTA: a CTA runs alone on its SM and every phase is a dependent chain
constexpr int NTH = 32 * NW;       // threads per CTA
constexpr int CW = LW / NW;        // hidden units per warp: warp w owns [CW w, CW w + CW)
constexpr int NTW = CW / 8;        // n-tiles per warp
// Tile row strides in elements: 8 (mod 32) 32-bit words for the float32 tiles, ldmatrix rows 16 B apart (mod 128) for
// the bf16 ones -- both free of bank conflicts for their fragment loads
constexpr int XLD = 136;   // the input tile (<= 128 features)
constexpr int SLICE = 128;  // features per pass through the input tile: a wider head's input is staged in K slices
constexpr int MAXIN = 1024; // widest head input (the representation head on a wide observation; no dX above SLICE)
constexpr int HLD = 520;   // the activation tiles
constexpr int DYLD = 72;   // the output-gradient tile (<= 64 outputs)
constexpr int FLD = 68;    // floats per row of the float32 tile (layer-2 output / dX of the dynamics head)
constexpr int STAGE = 8 * 68;  // floats per warp: eight rows of a weight-gradient tile
constexpr int MAXJOBS = 3, MAXPACK = 24;

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

template <int P>
MZ_DEV int round_up(int v) { return (v + P - 1) & ~(P - 1); }
// the two adjacent tile elements at p, as one store: pair_at<F>(p) = F::pair(a, b)
template <class F>
MZ_DEV typename F::T2& pair_at(typename F::T* p) { return *reinterpret_cast<typename F::T2*>(p); }
// k units of a contraction over d features
template <class F>
MZ_DEV int kunits(int d) { return round_up<F::K>(d) / F::K; }

// rows [row0, row0 + ROWS) x columns [0, d) of a float32 matrix -> tile, zeros up to column dpad (a multiple of K,
// <= 128) and behind `rows`.  A warp moves 32-column segments (with K = 32, dpad ends one); all of a thread's loads are
// in flight before its first store.
template <class F, int ROWS = RT>
MZ_DEV void load_rows(typename F::T* Ts, int ld, const float* __restrict__ X, int ldx, int row0, int rows, int d, int dpad) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int spr = (F::K == 32 ? dpad : dpad + 31) >> 5, segs = ROWS * spr;  // segments per row (1..4), in all
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
    if (sg < segs && (F::K == 32 || c < dpad)) Ts[r * ld + c] = F::cvt(v[i]);
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

template <int MT>
MZ_DEV void zero(float (&acc)[MT][NTW][4]) {
#pragma unroll
  for (int mt = 0; mt < MT; ++mt)
#pragma unroll
    for (int n = 0; n < NTW; ++n)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[mt][n][c] = 0.0f;
}

// H = relu(acc + b1) for the warp's CW hidden units -> Hs; returns the sign bits (bit 4 n + c of mask[mt]: the layout
// mz_chain_mask_words sizes)
template <class F, int MT>
MZ_DEV void hidden_epilogue(const mz_tc_head& h, const float (&acc)[MT][NTW][4], typename F::T* Hs, uint32_t (&mask)[MT],
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
      pair_at<F>(Hs + (16 * mt + g) * HLD + j) = F::pair(v0, v1);
      pair_at<F>(Hs + (16 * mt + g + 8) * HLD + j) = F::pair(v2, v3);
    }
  }
}

// H = relu(W1 X + b1) for the warp's CW hidden units, X in Xs (d_in <= SLICE)
template <class F, int MT>
MZ_DEV void hidden_phase(const mz_tc_head& h, const typename F::T* Xs, typename F::T* Hs, uint32_t (&mask)[MT], int warp,
                         int lane) {
  float acc[MT][NTW][4];
  zero<MT>(acc);
  F::template gemm_wide<MT>(acc, Xs, XLD, h.w1p, kunits<F>(h.d_in), NTW * warp, lane, kunits<F>(h.d_in));
  hidden_epilogue<F, MT>(h, acc, Hs, mask, warp, lane);
}

// The same for any d_in <= MAXIN, X read from global memory (rows row0 .. row0 + 16 MT of `rows`): layer 1 runs over
// K slices of up to SLICE features, each staged through Xs (16 MT x XLD) by the whole CTA, with the accumulators kept
// across slices -- the k-steps in the order of one pass, so the same sums.  Xs holds the last slice on return.  Every
// thread of the CTA calls it (barriers inside).
template <class F, int MT>
MZ_DEV void hidden_phase_sliced(const mz_tc_head& h, const float* __restrict__ X, int ldx, int row0, int rows,
                                typename F::T* Xs, typename F::T* Hs, uint32_t (&mask)[MT], int warp, int lane) {
  float acc[MT][NTW][4];
  zero<MT>(acc);
  const int KU = kunits<F>(h.d_in);
  for (int k0 = 0; k0 < h.d_in; k0 += SLICE) {
    const int w = min(SLICE, h.d_in - k0);
    if (k0) __syncthreads();  // every warp is done with the slice before
    load_rows<F, 16 * MT>(Xs, XLD, X + k0, ldx, row0, rows, w, round_up<F::K>(w));
    __syncthreads();
    // k unit k0 / K of every n-tile: 128 words per unit
    F::template gemm_wide<MT>(acc, Xs, XLD, h.w1p + (size_t)k0 * (128 / F::K), kunits<F>(w), NTW * warp, lane, KU);
  }
  hidden_epilogue<F, MT>(h, acc, Hs, mask, warp, lane);
}

// Y = H W2^T + b2 to global memory: warp w < ceil(d_out / 8) owns outputs [8 w, 8 w + 8)
template <class F>
MZ_DEV void output_phase(const mz_tc_head& h, const typename F::T* Hs, float* __restrict__ Y, int ldy, int row0, int rows,
                         int warp, int lane) {
  if (8 * warp >= h.d_out) return;
  float acc[2][4];
  F::template gemm_tall<2>(acc, Hs, HLD, h.w2p, warp, lane);
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

// ---- shared-memory plans ------------------------------------------------------------------------------------------
template <class F>
constexpr size_t heads_fwd_smem() {
  return (size_t)RT * (XLD + HLD) * sizeof(typename F::T);
}
// TILES x 32 rows of X (XLD), H and dH (HLD), dY (DYLD), plus NW staging areas.  A WIDE head streams its X through the
// same XLD tiles in slices of SLICE features (F::backward), so every width has this plan.
template <class F>
constexpr size_t heads_bwd_smem(int tiles) {
  return (size_t)tiles * RT * (XLD + 2 * HLD + DYLD) * sizeof(typename F::T) + (size_t)NW * STAGE * 4;
}
template <class F>
constexpr size_t chain_fwd_smem(int rows) {
  return (size_t)rows * (XLD + HLD) * sizeof(typename F::T) + (size_t)rows * FLD * 4;
}
template <class F>
constexpr size_t chain_bwd_smem(int rows) {
  return (size_t)rows * (DYLD + HLD) * sizeof(typename F::T) + (size_t)rows * FLD * 4 + 2 * 64 * 4;
}

// ---- the output heads: one job per blockIdx.y --------------------------------------------------------------------
// WIDE: some job has d_in > SLICE; every job's layer 1 then runs over slices (hidden_phase_sliced)
template <bool WIDE, class F>
__global__ void __launch_bounds__(NTH) heads_fwd_kernel(PlainParams p) {
  using T = typename F::T;
  extern __shared__ __align__(16) unsigned char tc_smem[];
  const mz_tc_job& job = p.jobs[blockIdx.y];
  const int row0 = blockIdx.x * RT;
  if (row0 >= job.rows) return;
  T* Xs = reinterpret_cast<T*>(tc_smem);
  T* Hs = Xs + RT * XLD;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint32_t mask[2];
  if (WIDE) {
    hidden_phase_sliced<F, 2>(job.head, job.x, job.ldx, row0, job.rows, Xs, Hs, mask, warp, lane);
  } else {
    load_rows<F>(Xs, XLD, job.x, job.ldx, row0, job.rows, job.head.d_in, round_up<F::K>(job.head.d_in));
    __syncthreads();
    hidden_phase<F, 2>(job.head, Xs, Hs, mask, warp, lane);
  }
  __syncthreads();
  output_phase<F>(job.head, Hs, job.y, job.ldy, row0, job.rows, warp, lane);
}

// The backward of the heads over TILES x 32 rows per CTA: X and dY tiles loaded here, gb2 from dY, the rest in
// F::backward.
template <int TILES, bool WIDE, class F>
__global__ void __launch_bounds__(NTH) heads_bwd_kernel(PlainParams p) {
  using T = typename F::T;
  extern __shared__ __align__(16) unsigned char tc_smem[];
  const mz_tc_job& job = p.jobs[blockIdx.y];
  constexpr int RTT = RT * TILES;  // rows per CTA
  const int row0 = blockIdx.x * RTT;
  if (row0 >= job.rows) return;
  T* Xs = reinterpret_cast<T*>(tc_smem);
  T* Hs = Xs + RTT * XLD;
  T* dHs = Hs + RTT * HLD;
  T* dYs = dHs + RTT * HLD;
  float* stage = reinterpret_cast<float*>(dYs + RTT * DYLD);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const mz_tc_head& h = job.head;
  TC_T(1, 0, 0);
  constexpr int DYPAD = F::K > 16 ? F::K : 16;  // dY feeds k units (dH) and m-tiles of 16 outputs (gW2)
#pragma unroll
  for (int tile = 0; tile < TILES; ++tile) {
    if (!WIDE) load_rows<F>(Xs + tile * RT * XLD, XLD, job.x, job.ldx, row0 + RT * tile, job.rows, h.d_in, round_up<F::K>(h.d_in));
    load_rows<F>(dYs + tile * RT * DYLD, DYLD, job.dy, job.ldy, row0 + RT * tile, job.rows, h.d_out, round_up<DYPAD>(h.d_out));
  }
  if ((int)threadIdx.x < h.d_out) {  // gb2[o] = sum_r dY[r][o]
    float part[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll 8
    for (int r = 0; r < RTT; ++r)
      if (row0 + r < job.rows) part[r & 3] += job.dy[(size_t)(row0 + r) * job.ldy + threadIdx.x];
    atomicAdd(h.gb2 + threadIdx.x, (part[0] + part[1]) + (part[2] + part[3]));
  }
  __syncthreads();
  F::template backward<TILES, WIDE>(h, job.x, job.ldx, Xs, dYs, Hs, dHs, job.dx, job.lddx, job.dx != nullptr ? h.d_in : 0,
                                    row0, job.rows, stage + warp * STAGE, warp, lane);
}

// ---- the recurrent chain ---------------------------------------------------------------------------------------
// A CTA owns 16 MT rows for all steps.  MT = 1 (16 rows, twice the CTAs) whenever that still fits one wave: the phases
// of a step are bound by the issue rate of the warp-level mma on the CTA's SM, so half the rows per CTA is half the
// time per step.
// LayerNorm phases: a warp owns 16 MT / NW rows at once, LPR lanes per row; lane (rr, c8) holds columns c8 + LPR i
// (i < CPL) of its row, so the row statistics are log2(LPR) shuffle steps and the rows run side by side.
template <int MT>
struct ChainGeo {
  static constexpr int ROWS = 16 * MT;
  static constexpr int LPR = 32 * NW / ROWS;  // lanes per row (MT = 1: 32, MT = 2: 16)
  static constexpr int CPL = 64 / LPR;        // columns per lane
};

// WIDE: first.d_in > SLICE -- step 0 streams x0 through Xs in slices (hidden_phase_sliced); the LayerNorm epilogues
// write the next step's input into Xs as for a narrow first head
template <int MT, bool WIDE, class F>
__global__ void __launch_bounds__(NTH) chain_fwd_kernel(mz_tc_chain c) {
  using T = typename F::T;
  using G = ChainGeo<MT>;
  constexpr int ROWS = G::ROWS, LPR = G::LPR, CPL = G::CPL;
  extern __shared__ __align__(16) unsigned char tc_smem[];
  const int row0 = blockIdx.x * ROWS;
  T* Xs = reinterpret_cast<T*>(tc_smem);
  T* Hs = Xs + ROWS * XLD;
  float* Fs = reinterpret_cast<float*>(Hs + ROWS * HLD);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = c.d, A = c.num_actions, next_pad = round_up<F::K>(d + A);
  const int r = (32 / LPR) * warp + lane / LPR, c8 = lane % LPR, row = row0 + r;
  const bool live = row < c.rows;
  const float inv_d = 1.0f / (float)d;
  const int g = lane >> 2, t = lane & 3;
  float gam[CPL], bet[CPL];
  if (F::GAMMA_IN_REGS) {
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int col = c8 + LPR * i;
      gam[i] = col < d ? __ldg(c.gamma + col) : 0.0f;
      bet[i] = col < d ? __ldg(c.beta + col) : 0.0f;
    }
  }
  if (!WIDE) {
    load_rows<F, ROWS>(Xs, XLD, c.x0, c.ldx0, row0, c.rows, c.first.d_in, round_up<F::K>(c.first.d_in));
    __syncthreads();
  }
  for (int step = 0; step < c.steps; ++step) {
    const mz_tc_head& h = step ? c.next : c.first;
    const int act = (live && c.actions != nullptr && step < c.action_steps)
                        ? __ldg(c.actions + (size_t)row * c.action_stride + step) : -1;  // in flight during the head
    TC_T(0, step, 0);
    uint32_t mask[MT];
    if (WIDE && step == 0)
      hidden_phase_sliced<F, MT>(h, c.x0, c.ldx0, row0, c.rows, Xs, Hs, mask, warp, lane);
    else
      hidden_phase<F, MT>(h, Xs, Hs, mask, warp, lane);
    TC_T(0, step, 1);
    if (step && c.relu_mask != nullptr)  // the backward chain gates dH with these bits instead of recomputing the layer
      reinterpret_cast<uint2*>(c.relu_mask)[((size_t)step * gridDim.x + blockIdx.x) * NTH + threadIdx.x] =
          make_uint2(mask[0], MT > 1 ? mask[MT - 1] : 0u);
    __syncthreads();
    TC_T(0, step, 2);
    if (8 * warp < d) {  // Y = H W2^T + b2: warp w owns outputs [8 w, 8 w + 8) -> Fs
      float acc[MT][4];
      F::template gemm_tall<MT>(acc, Hs, HLD, h.w2p, warp, lane);
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
      const int col = c8 + LPR * i;
      v[i] = col < d ? Fs[r * FLD + col] : 0.0f;
      if (!F::GAMMA_IN_REGS) {
        gam[i] = col < d ? __ldg(c.gamma + col) : 0.0f;
        bet[i] = col < d ? __ldg(c.beta + col) : 0.0f;
      }
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
      Xs[r * XLD + col] = F::cvt(live ? out : 0.0f);
    }
    for (int col = 64 + c8; col < next_pad; col += LPR) {  // d + A > 64 (A = 18): the rest of the one-hot
      const float out = (col < d + A && col - d == act) ? 1.0f : 0.0f;
      if (live && col < d + A) c.xs[grow * c.ldxs + col] = out;
      Xs[r * XLD + col] = F::cvt(out);
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
// the two heads do not sit on this chain: the heads' backward computes them afterwards from (xs, dyall) over all
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

template <int MT, class F>
__global__ void __launch_bounds__(NTH) chain_bwd_kernel(mz_tc_chain c) {
  using T = typename F::T;
  using G = ChainGeo<MT>;
  constexpr int ROWS = G::ROWS, LPR = G::LPR, CPL = G::CPL;
  extern __shared__ __align__(16) unsigned char tc_smem[];
  const int row0 = blockIdx.x * ROWS;
  T* dYs = reinterpret_cast<T*>(tc_smem);
  T* dHs = dYs + ROWS * DYLD;
  float* Fs = reinterpret_cast<float*>(dHs + ROWS * HLD);
  float* red = Fs + ROWS * FLD;  // [2][64]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int d = c.d, out_pad = round_up<F::K>(d);
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
    if (F::EARLY_LN_LOAD && step) ln_load<CPL, LPR>(nxt, c, step - 1, row, live, c8);  // in flight during the contractions
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
      if (col < out_pad) dYs[r * DYLD + col] = F::cvt(dy);
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
      const int KU = kunits<F>(h.d_out);
      F::template gemm_wide<MT>(acc, dYs, DYLD, h.w2tp, KU, NTW * warp, lane, KU);
#pragma unroll
      for (int n = 0; n < NTW; ++n) {
        const int j = CW * warp + 8 * n + 2 * t;
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          const uint32_t m = (mt ? mbits.y : mbits.x) >> (4 * n);
          pair_at<F>(dHs + (16 * mt + g) * HLD + j) =
              F::pair((m & 1u) ? acc[mt][n][0] : 0.0f, (m & 2u) ? acc[mt][n][1] : 0.0f);
          pair_at<F>(dHs + (16 * mt + g + 8) * HLD + j) =
              F::pair((m & 4u) ? acc[mt][n][2] : 0.0f, (m & 8u) ? acc[mt][n][3] : 0.0f);
        }
      }
      if (!F::EARLY_LN_LOAD) ln_load<CPL, LPR>(nxt, c, step - 1, row, live, c8);  // in flight during the dX contraction
      __syncthreads();
      // dX = dH W1, the hidden-state columns only -> Fs
      for (int nt = warp; 8 * nt < d; nt += NW) {
        float a2[MT][4];
        F::template gemm_tall<MT>(a2, dHs, HLD, h.w1tp, nt, lane);
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

// ---- host side ---------------------------------------------------------------------------------------------------
template <class Kernel>
cudaError_t smem_attr(Kernel* kernel, size_t bytes) {
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

template <class F>
int set_attrs() {
  static bool done = false;
  if (done) return 0;
  constexpr int TM = F::MAX_TILES;  // (1: the single-tile kernels twice)
  cudaError_t e;
  if ((e = smem_attr(heads_fwd_kernel<false, F>, heads_fwd_smem<F>())) != cudaSuccess ||
      (e = smem_attr(heads_fwd_kernel<true, F>, heads_fwd_smem<F>())) != cudaSuccess ||
      (e = smem_attr(heads_bwd_kernel<1, false, F>, heads_bwd_smem<F>(1))) != cudaSuccess ||
      (e = smem_attr(heads_bwd_kernel<1, true, F>, heads_bwd_smem<F>(1))) != cudaSuccess ||
      (e = smem_attr(heads_bwd_kernel<TM, false, F>, heads_bwd_smem<F>(TM))) != cudaSuccess ||
      (e = smem_attr(heads_bwd_kernel<TM, true, F>, heads_bwd_smem<F>(TM))) != cudaSuccess ||
      (e = smem_attr(chain_fwd_kernel<1, false, F>, chain_fwd_smem<F>(16))) != cudaSuccess ||
      (e = smem_attr(chain_fwd_kernel<2, false, F>, chain_fwd_smem<F>(32))) != cudaSuccess ||
      (e = smem_attr(chain_fwd_kernel<1, true, F>, chain_fwd_smem<F>(16))) != cudaSuccess ||
      (e = smem_attr(chain_fwd_kernel<2, true, F>, chain_fwd_smem<F>(32))) != cudaSuccess ||
      (e = smem_attr(chain_bwd_kernel<1, F>, chain_bwd_smem<F>(16))) != cudaSuccess ||
      (e = smem_attr(chain_bwd_kernel<2, F>, chain_bwd_smem<F>(32))) != cudaSuccess)
    return (int)e;
  done = true;
  return 0;
}

// rows per CTA of the chain kernels: 16 while that is at most one wave of CTAs, else 32 (forward and backward of a
// step must agree: the ReLU bits are stored per CTA and thread)
inline int chain_mt(int rows) { return (rows + 15) / 16 <= 148 ? 1 : 2; }

// MZ_OK, MZ_ERR_UNSUPPORTED for a shape beyond the kernels (d_in > MAXIN, d_out > 64), else MZ_ERR_BAD_ARG.
// (w1tp only feeds dX, which a head wider than SLICE does not have: its image need not exist)
inline int head_check(const mz_tc_head& h, bool backward) {
  if (h.d_in > MAXIN || h.d_out > 64) return MZ_ERR_UNSUPPORTED;
  if (h.d_in < 1 || h.d_out < 1 || !h.w1p || !h.w2p || !h.b1 || !h.b2) return MZ_ERR_BAD_ARG;
  if (backward && (!h.w2tp || (h.d_in <= SLICE && !h.w1tp) || !h.gw1 || !h.gb1 || !h.gw2 || !h.gb2)) return MZ_ERR_BAD_ARG;
  if (backward && (((uintptr_t)h.gw1 | (uintptr_t)h.gw2) & 15)) return MZ_ERR_BAD_ARG;  // weight gradients leave as red.v4
  return MZ_OK;
}

// the same for a chain: MZ_ERR_UNSUPPORTED also for d > 64 or d + num_actions > SLICE
inline int chain_check(const mz_tc_chain* c, bool backward) {
  if (!c) return MZ_ERR_BAD_ARG;
  if (c->d > 64 || c->d + c->num_actions > SLICE) return MZ_ERR_UNSUPPORTED;
  if (c->rows < 1 || c->steps < 1 || c->d < 1 || c->num_actions < 0) return MZ_ERR_BAD_ARG;
  if (int rc = head_check(c->first, false)) return rc;
  if (c->first.d_out != c->d) return MZ_ERR_BAD_ARG;
  if (c->steps > 1) {
    if (int rc = head_check(c->next, false)) return rc;
    if (c->next.d_out != c->d || c->next.d_in != c->d + c->num_actions) return MZ_ERR_BAD_ARG;
  }
  // (the chain's backward reads the packed images only; the heads' gradients are the heads' backward's job)
  if (backward && c->steps > 1 && (!c->next.w2tp || !c->next.w1tp)) return MZ_ERR_BAD_ARG;
  if (!c->x0 || c->ldx0 < c->first.d_in || !c->gamma || !c->beta || !c->xs || c->ldxs < c->d + c->num_actions || !c->yall ||
      !c->mean || !c->rstd)
    return MZ_ERR_BAD_ARG;
  if (c->actions && (c->action_stride < c->action_steps || c->action_steps < 0)) return MZ_ERR_BAD_ARG;
  if (backward && (!c->dxs || !c->ggamma || !c->gbeta || !c->dyall || (c->steps > 1 && !c->relu_mask))) return MZ_ERR_BAD_ARG;
  return MZ_OK;
}

// The weight images (and the gradient buffers to clear) of a step: one launch, one job per blockIdx.y
template <class F>
int pack(int32_t njobs, const mz_pack_job* jobs, void* stream) {
  if (njobs < 1 || njobs > MAXPACK || !jobs) return MZ_ERR_BAD_ARG;
  PackParams p;
  int64_t ctas = 1;
  for (int i = 0; i < njobs; ++i) {
    if (!jobs[i].dst || jobs[i].n < 1 || (jobs[i].src && jobs[i].k < 1)) return MZ_ERR_BAD_ARG;
    p.jobs[i] = jobs[i];
    const int64_t c = jobs[i].src ? (F::packed_words(jobs[i].n, jobs[i].k) + F::PACK_CTA_WORDS - 1) / F::PACK_CTA_WORDS
                                  : ((int64_t)jobs[i].n + F::CLEAR_CTA_WORDS - 1) / F::CLEAR_CTA_WORDS;
    ctas = c > ctas ? c : ctas;
  }
  const int blocks = (int)(ctas < F::PACK_MAX_CTAS ? ctas : F::PACK_MAX_CTAS);
  F::pack_kernel<<<dim3(blocks, njobs), 256, 0, (cudaStream_t)stream>>>(p);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

template <class F>
int heads_forward(int32_t njobs, const mz_tc_job* jobs, void* stream) {
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
  if (int rc = set_attrs<F>()) return rc;
  const dim3 grid((most + RT - 1) / RT, njobs);
  if (wide)
    heads_fwd_kernel<true, F><<<grid, NTH, heads_fwd_smem<F>(), (cudaStream_t)stream>>>(p);
  else
    heads_fwd_kernel<false, F><<<grid, NTH, heads_fwd_smem<F>(), (cudaStream_t)stream>>>(p);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

template <class F, int TILES>
void launch_heads_bwd(const PlainParams& p, int njobs, int most, bool wide, cudaStream_t st) {
  const dim3 grid((most + TILES * RT - 1) / (TILES * RT), njobs);
  if (wide)
    heads_bwd_kernel<TILES, true, F><<<grid, NTH, heads_bwd_smem<F>(TILES), st>>>(p);
  else
    heads_bwd_kernel<TILES, false, F><<<grid, NTH, heads_bwd_smem<F>(TILES), st>>>(p);
}

template <class F>
int heads_backward(int32_t njobs, const mz_tc_job* jobs, void* stream) {
  if (njobs < 1 || njobs > MAXJOBS || !jobs) return MZ_ERR_BAD_ARG;
  PlainParams p;
  int most = 0, ctas = 0;
  bool wide = false;
  for (int i = 0; i < njobs; ++i) {
    const mz_tc_job& j = jobs[i];
    if (int rc = head_check(j.head, true)) return rc;
    if (j.rows < 1 || !j.x || !j.dy || j.ldx < j.head.d_in || j.ldy < j.head.d_out ||
        (j.dx && (j.lddx < j.head.d_in || j.head.d_in > SLICE)))
      return MZ_ERR_BAD_ARG;
    p.jobs[i] = j;
    most = j.rows > most ? j.rows : most;
    ctas += (j.rows + RT - 1) / RT;
    wide = wide || j.head.d_in > SLICE;
  }
  if (int rc = set_attrs<F>()) return rc;
  // more CTAs than one wave of single-tile CTAs: more tiles per CTA where they fit (fewer weight-gradient reductions)
  if (ctas > 148)
    launch_heads_bwd<F, F::MAX_TILES>(p, njobs, most, wide, (cudaStream_t)stream);
  else
    launch_heads_bwd<F, 1>(p, njobs, most, wide, (cudaStream_t)stream);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

template <class F>
int chain_forward(const mz_tc_chain* chain, void* stream) {
  if (int rc = chain_check(chain, false)) return rc;
  if (int rc = set_attrs<F>()) return rc;
  const bool wide = chain->first.d_in > SLICE;
  cudaStream_t st = (cudaStream_t)stream;
  if (chain_mt(chain->rows) == 1 && wide)
    chain_fwd_kernel<1, true, F><<<(chain->rows + 15) / 16, NTH, chain_fwd_smem<F>(16), st>>>(*chain);
  else if (chain_mt(chain->rows) == 1)
    chain_fwd_kernel<1, false, F><<<(chain->rows + 15) / 16, NTH, chain_fwd_smem<F>(16), st>>>(*chain);
  else if (wide)
    chain_fwd_kernel<2, true, F><<<(chain->rows + 31) / 32, NTH, chain_fwd_smem<F>(32), st>>>(*chain);
  else
    chain_fwd_kernel<2, false, F><<<(chain->rows + 31) / 32, NTH, chain_fwd_smem<F>(32), st>>>(*chain);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

template <class F>
int chain_backward(const mz_tc_chain* chain, void* stream) {
  if (int rc = chain_check(chain, true)) return rc;
  if (int rc = set_attrs<F>()) return rc;
  if (chain_mt(chain->rows) == 1)
    chain_bwd_kernel<1, F><<<(chain->rows + 15) / 16, NTH, chain_bwd_smem<F>(16), (cudaStream_t)stream>>>(*chain);
  else
    chain_bwd_kernel<2, F><<<(chain->rows + 31) / 32, NTH, chain_bwd_smem<F>(32), (cudaStream_t)stream>>>(*chain);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

}  // namespace
