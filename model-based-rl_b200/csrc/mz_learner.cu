// The learner's network forward and backward (Learner.update_weights, learners.py:164-230) as hand-written kernels
// for the FCNetwork architecture (networks.py:55-174): every head is Linear(d_in, 512) -> ReLU -> Linear(512, d_out)
// and the hidden state goes through LayerNorm + ReLU, so a training step is made of four kernels:
//
//   mlp2_forward   Y = W2 relu(W1 X + b1) + b2 for a tile of 32 rows per CTA (the 512-wide activation never leaves
//                  shared memory)
//   mlp2_backward  the same tile again: recomputes relu(W1 X + b1), then dH, dX (accumulated into the caller's
//                  buffer: several heads feed the same hidden state) and the four parameter gradients, which go to
//                  global memory as float32 atomics (one per weight and CTA)
//   ln_relu_forward / ln_relu_backward   LayerNorm + ReLU of the hidden state, the one-hot action appended in the
//                  forward (the next head's input row), the reference's 0.5 gradient hook (learners.py:201) as a
//                  scale in the backward
//   adamw_step     the optimiser over the flat parameter buffer (optional global-norm clipping)
//
// A step of the C3 shape (B = 512, K = 5) is 15 + 15 of these launches plus the fused loss (mz_unroll_loss) instead of
// the ~270 library kernels of the torch module; arithmetic is float32 throughout, like the reference's.
// The step is bound by launch latency and dependent small tiles (3 GFLOP in all), not by tensor throughput, so the
// contractions run on the CUDA cores with register tiles: 64 accumulators per thread in the wide layers.
//
// Weight layouts: the flat parameter buffer keeps torch's [out][in] matrices (the state dict is a set of views);
// the forward also reads k-major copies (W1T [d_in][512], W2T [512][d_out]) that mz_learner_transpose refreshes once
// per step, so that every global weight read of every phase is coalesced.
#include <math.h>

#include "mz_common.cuh"

namespace {

constexpr int LW = 512;   // hidden width of every head (networks.py:55-119)
constexpr int LR = 32;    // rows per CTA
constexpr int LT = 256;   // threads per CTA
constexpr int LDH = 36;   // floats per row of the transposed [feature][row] tiles: 32 rows + 4 (bank spread)
constexpr int LMAXIN = 128, LMAXOUT = 64;  // widest input tile (features per slice of X), widest output
constexpr int LMAXD = 1024;                // widest head input: the representation head's slices of LMAXIN features

// X tile -> shared memory, transposed: Xs[k * LDH + r] = X[(row0 + r) * ldx + k], zeros behind the last row
MZ_DEV void load_tile_T(float* Xs, const float* __restrict__ X, int ldx, int row0, int rows, int d) {
  for (int idx = threadIdx.x; idx < LR * d; idx += LT) {
    const int r = idx / d, k = idx - r * d;
    Xs[k * LDH + r] = (row0 + r < rows) ? X[(size_t)(row0 + r) * ldx + k] : 0.0f;
  }
}

// H = relu(W1 X + b1) for the tile: thread t owns hidden units t and t + 256, 32 rows each, and leaves them in
// Hs[j * LDH + r].  Narrow (d_in <= LMAXIN): X is already in Xs.  WIDE: X goes through Xs in slices of LMAXIN
// features, the accumulators kept across slices (the same sums in the same order as one pass); Xs holds the last
// slice on return.
template <bool WIDE>
MZ_DEV void hidden_layer(float* Xs, float* Hs, const float* __restrict__ X, int ldx, int row0, int rows,
                         const float* __restrict__ W1T, const float* __restrict__ b1, int d_in) {
  const int j0 = threadIdx.x, j1 = threadIdx.x + LT;
  float a0[LR], a1[LR];
#pragma unroll
  for (int r = 0; r < LR; ++r) a0[r] = a1[r] = 0.0f;
  for (int k0 = 0; k0 < d_in; k0 += LMAXIN) {
    const int dk = WIDE ? min(LMAXIN, d_in - k0) : d_in;
    if (WIDE) {
      if (k0) __syncthreads();  // every thread is done with the slice before
      load_tile_T(Xs, X + k0, ldx, row0, rows, dk);
      __syncthreads();
    }
    for (int k = 0; k < dk; ++k) {
      const float w0 = __ldg(W1T + (size_t)(k0 + k) * LW + j0), w1 = __ldg(W1T + (size_t)(k0 + k) * LW + j1);
      const float4* xr = reinterpret_cast<const float4*>(Xs + k * LDH);
#pragma unroll
      for (int q = 0; q < LR / 4; ++q) {
        const float4 x = xr[q];
        a0[4 * q + 0] = fmaf(w0, x.x, a0[4 * q + 0]);
        a0[4 * q + 1] = fmaf(w0, x.y, a0[4 * q + 1]);
        a0[4 * q + 2] = fmaf(w0, x.z, a0[4 * q + 2]);
        a0[4 * q + 3] = fmaf(w0, x.w, a0[4 * q + 3]);
        a1[4 * q + 0] = fmaf(w1, x.x, a1[4 * q + 0]);
        a1[4 * q + 1] = fmaf(w1, x.y, a1[4 * q + 1]);
        a1[4 * q + 2] = fmaf(w1, x.z, a1[4 * q + 2]);
        a1[4 * q + 3] = fmaf(w1, x.w, a1[4 * q + 3]);
      }
    }
    if (!WIDE) break;
  }
  const float c0 = __ldg(b1 + j0), c1 = __ldg(b1 + j1);
  float4* h0 = reinterpret_cast<float4*>(Hs + j0 * LDH);
  float4* h1 = reinterpret_cast<float4*>(Hs + j1 * LDH);
#pragma unroll
  for (int q = 0; q < LR / 4; ++q) {
    h0[q] = make_float4(fmaxf(a0[4 * q] + c0, 0.f), fmaxf(a0[4 * q + 1] + c0, 0.f), fmaxf(a0[4 * q + 2] + c0, 0.f),
                        fmaxf(a0[4 * q + 3] + c0, 0.f));
    h1[q] = make_float4(fmaxf(a1[4 * q] + c1, 0.f), fmaxf(a1[4 * q + 1] + c1, 0.f), fmaxf(a1[4 * q + 2] + c1, 0.f),
                        fmaxf(a1[4 * q + 3] + c1, 0.f));
  }
}

template <bool WIDE>  // d_in > LMAXIN
__global__ void __launch_bounds__(LT)
mlp2_forward_kernel(int rows, int d_in, int ldx, const float* __restrict__ X, const float* __restrict__ W1T,
                    const float* __restrict__ b1, const float* __restrict__ W2T, const float* __restrict__ b2, int d_out,
                    float* __restrict__ Y, int ldy) {
  extern __shared__ __align__(16) float lsm[];
  float* Xs = lsm;                  // [LMAXIN][LDH]: a slice of X
  float* Hs = lsm + LMAXIN * LDH;   // [LW][LDH]
  const int row0 = blockIdx.x * LR;
  if (!WIDE) {
    load_tile_T(Xs, X, ldx, row0, rows, d_in);
    __syncthreads();
  }
  hidden_layer<WIDE>(Xs, Hs, X, ldx, row0, rows, W1T, b1, d_in);
  __syncthreads();
  // Y = H W2^T + b2: thread (og, rg) owns outputs og, og + 16, og + 32, og + 48 of rows 2 rg, 2 rg + 1
  const int og = threadIdx.x & 15, rg = threadIdx.x >> 4;
  float acc[2][4];
#pragma unroll
  for (int c = 0; c < 4; ++c) acc[0][c] = acc[1][c] = 0.0f;
  const int nc = (d_out - og + 15) >> 4;  // valid columns of this thread (0..4)
  for (int j = 0; j < LW; ++j) {
    const float2 h = *reinterpret_cast<const float2*>(Hs + j * LDH + 2 * rg);
    const float* wr = W2T + (size_t)j * d_out + og;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      if (c < nc) {
        const float w = __ldg(wr + 16 * c);
        acc[0][c] = fmaf(h.x, w, acc[0][c]);
        acc[1][c] = fmaf(h.y, w, acc[1][c]);
      }
    }
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const int o = og + 16 * c;
    if (c < nc) {
      const float bb = __ldg(b2 + o);
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const int row = row0 + 2 * rg + i;
        if (row < rows) Y[(size_t)row * ldy + o] = acc[i][c] + bb;
      }
    }
  }
}

// Backward of the two-layer head over one tile.  W1T / W2T: the k-major copies (recompute); W1 [512][d_in], W2
// [d_out][512]: torch layout (dH, dX).  dX (nullable, d_in <= LMAXIN): accumulated, columns [0, d_in).  Gradients:
// atomics.  Shared memory: one LMAXIN-feature slice of X, H, dH, dY -- 171 KB; X wider than a slice (the
// representation head) goes through the slice tile twice, for the recomputed H and for gW1.
template <bool WIDE>  // d_in > LMAXIN
__global__ void __launch_bounds__(LT)
mlp2_backward_kernel(int rows, int d_in, int ldx, const float* __restrict__ X, const float* __restrict__ W1T,
                     const float* __restrict__ b1, const float* __restrict__ W1, const float* __restrict__ W2, int d_out,
                     const float* __restrict__ dY, int ldy, float* __restrict__ dX, int lddx, float* __restrict__ gW1,
                     float* __restrict__ gb1, float* __restrict__ gW2, float* __restrict__ gb2) {
  extern __shared__ __align__(16) float lsm[];
  float* Xs = lsm;                              // [LMAXIN][LDH]: a slice of X
  float* Hs = Xs + LMAXIN * LDH;                // [LW][LDH]   relu(W1 X + b1)
  float* dHs = Hs + LW * LDH;                   // [LW][LDH]
  float* dYs = dHs + LW * LDH;                  // [d_out][LDH]
  const int row0 = blockIdx.x * LR;
  if (!WIDE) load_tile_T(Xs, X, ldx, row0, rows, d_in);
  load_tile_T(dYs, dY, ldy, row0, rows, d_out);
  if (!WIDE) __syncthreads();
  hidden_layer<WIDE>(Xs, Hs, X, ldx, row0, rows, W1T, b1, d_in);
  // thread t: hidden units j0, j1.  One pass over the outputs: dH[r][j] = sum_o dY[r][o] W2[o][j] and
  // gW2[o][j] = sum_r dY[r][o] H[r][j]
  {
    const int j0 = threadIdx.x, j1 = threadIdx.x + LT;
    float h0[LR], h1[LR], d0[LR], d1[LR];
    const float4* hp0 = reinterpret_cast<const float4*>(Hs + j0 * LDH);  // written by this thread
    const float4* hp1 = reinterpret_cast<const float4*>(Hs + j1 * LDH);
#pragma unroll
    for (int q = 0; q < LR / 4; ++q) {
      const float4 u = hp0[q], v = hp1[q];
      h0[4 * q] = u.x; h0[4 * q + 1] = u.y; h0[4 * q + 2] = u.z; h0[4 * q + 3] = u.w;
      h1[4 * q] = v.x; h1[4 * q + 1] = v.y; h1[4 * q + 2] = v.z; h1[4 * q + 3] = v.w;
    }
#pragma unroll
    for (int r = 0; r < LR; ++r) d0[r] = d1[r] = 0.0f;
    for (int o = 0; o < d_out; ++o) {
      const float w0 = __ldg(W2 + (size_t)o * LW + j0), w1 = __ldg(W2 + (size_t)o * LW + j1);
      const float4* yr = reinterpret_cast<const float4*>(dYs + o * LDH);
      float s0 = 0.0f, s1 = 0.0f;
#pragma unroll
      for (int q = 0; q < LR / 4; ++q) {
        const float4 y = yr[q];
        d0[4 * q + 0] = fmaf(w0, y.x, d0[4 * q + 0]);
        d0[4 * q + 1] = fmaf(w0, y.y, d0[4 * q + 1]);
        d0[4 * q + 2] = fmaf(w0, y.z, d0[4 * q + 2]);
        d0[4 * q + 3] = fmaf(w0, y.w, d0[4 * q + 3]);
        d1[4 * q + 0] = fmaf(w1, y.x, d1[4 * q + 0]);
        d1[4 * q + 1] = fmaf(w1, y.y, d1[4 * q + 1]);
        d1[4 * q + 2] = fmaf(w1, y.z, d1[4 * q + 2]);
        d1[4 * q + 3] = fmaf(w1, y.w, d1[4 * q + 3]);
        s0 = fmaf(h0[4 * q + 0], y.x, s0);
        s0 = fmaf(h0[4 * q + 1], y.y, s0);
        s0 = fmaf(h0[4 * q + 2], y.z, s0);
        s0 = fmaf(h0[4 * q + 3], y.w, s0);
        s1 = fmaf(h1[4 * q + 0], y.x, s1);
        s1 = fmaf(h1[4 * q + 1], y.y, s1);
        s1 = fmaf(h1[4 * q + 2], y.z, s1);
        s1 = fmaf(h1[4 * q + 3], y.w, s1);
      }
      atomicAdd(gW2 + (size_t)o * LW + j0, s0);
      atomicAdd(gW2 + (size_t)o * LW + j1, s1);
    }
    float sb0 = 0.0f, sb1 = 0.0f;
    float4* dp0 = reinterpret_cast<float4*>(dHs + j0 * LDH);
    float4* dp1 = reinterpret_cast<float4*>(dHs + j1 * LDH);
#pragma unroll
    for (int q = 0; q < LR / 4; ++q) {
      float4 u, v;
      u.x = h0[4 * q] > 0.f ? d0[4 * q] : 0.f;
      u.y = h0[4 * q + 1] > 0.f ? d0[4 * q + 1] : 0.f;
      u.z = h0[4 * q + 2] > 0.f ? d0[4 * q + 2] : 0.f;
      u.w = h0[4 * q + 3] > 0.f ? d0[4 * q + 3] : 0.f;
      v.x = h1[4 * q] > 0.f ? d1[4 * q] : 0.f;
      v.y = h1[4 * q + 1] > 0.f ? d1[4 * q + 1] : 0.f;
      v.z = h1[4 * q + 2] > 0.f ? d1[4 * q + 2] : 0.f;
      v.w = h1[4 * q + 3] > 0.f ? d1[4 * q + 3] : 0.f;
      dp0[q] = u;
      dp1[q] = v;
      sb0 += u.x + u.y + u.z + u.w;
      sb1 += v.x + v.y + v.z + v.w;
    }
    atomicAdd(gb1 + j0, sb0);
    atomicAdd(gb1 + j1, sb1);
  }
  if (threadIdx.x < d_out) {  // gb2[o] = sum_r dY[r][o]
    float s = 0.0f;
    for (int r = 0; r < LR; ++r) s += dYs[threadIdx.x * LDH + r];
    atomicAdd(gb2 + threadIdx.x, s);
  }
  __syncthreads();
  // thread (k, g): input feature k, a group of rows (dX) / of hidden units (gW1)
  const int KP = d_in <= 64 ? 64 : 128, NG = LT / KP;  // 4 or 2 groups
  const int k = threadIdx.x % KP, g = threadIdx.x / KP;
  if (dX != nullptr && k < d_in) {  // dX[r][k] += sum_j dH[r][j] W1[j][k], rows [g * LR / NG, (g + 1) * LR / NG)
    const int nr = LR / NG, r0 = g * nr;
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.0f;
    for (int j = 0; j < LW; ++j) {
      const float wv = __ldg(W1 + (size_t)j * d_in + k);
      const float4* dr = reinterpret_cast<const float4*>(dHs + j * LDH + r0);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (4 * q < nr) {
          const float4 v = dr[q];
          acc[4 * q + 0] = fmaf(wv, v.x, acc[4 * q + 0]);
          acc[4 * q + 1] = fmaf(wv, v.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(wv, v.z, acc[4 * q + 2]);
          acc[4 * q + 3] = fmaf(wv, v.w, acc[4 * q + 3]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const int row = row0 + r0 + i;
      if (i < nr && row < rows) dX[(size_t)row * lddx + k] += acc[i];
    }
  }
  // gW1[j][k] = sum_r dH[r][j] X[r][k], hidden units [g * LW / NG, (g + 1) * LW / NG), per slice of X
  for (int k0 = 0;; k0 += LMAXIN) {  // d_in >= 1: at least one pass
    const int dk = WIDE ? min(LMAXIN, d_in - k0) : d_in;
    if (WIDE) {
      __syncthreads();
      load_tile_T(Xs, X + k0, ldx, row0, rows, dk);
      __syncthreads();
    }
    if (k < dk) {
      float x[LR];
      const float4* xp = reinterpret_cast<const float4*>(Xs + k * LDH);
#pragma unroll
      for (int q = 0; q < LR / 4; ++q) {
        const float4 v = xp[q];
        x[4 * q] = v.x; x[4 * q + 1] = v.y; x[4 * q + 2] = v.z; x[4 * q + 3] = v.w;
      }
      const int nj = LW / NG;
      for (int j = g * nj; j < (g + 1) * nj; ++j) {
        const float4* dr = reinterpret_cast<const float4*>(dHs + j * LDH);
        float s = 0.0f;
#pragma unroll
        for (int q = 0; q < LR / 4; ++q) {
          const float4 v = dr[q];
          s = fmaf(x[4 * q + 0], v.x, s);
          s = fmaf(x[4 * q + 1], v.y, s);
          s = fmaf(x[4 * q + 2], v.z, s);
          s = fmaf(x[4 * q + 3], v.w, s);
        }
        atomicAdd(gW1 + (size_t)j * d_in + k0 + k, s);
      }
    }
    if (!WIDE || k0 + LMAXIN >= d_in) break;
  }
}

// LayerNorm (networks.py:144, eps 1e-5, biased variance) + ReLU of one row per warp, the next head's input row as
// output: X_out[r] = [relu(LN(Y[r])) (d values) | one-hot(actions[r * action_stride]) (A values)]
__global__ void ln_relu_forward_kernel(int rows, int d, const float* __restrict__ Y, const float* __restrict__ gamma,
                                       const float* __restrict__ beta, const int32_t* __restrict__ actions,
                                       int action_stride, int A, float* __restrict__ X_out, int ldx,
                                       float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float v0 = lane < d ? Y[(size_t)r * d + lane] : 0.0f;
  const float v1 = lane + 32 < d ? Y[(size_t)r * d + lane + 32] : 0.0f;
  float s = v0 + v1;
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) s += __shfl_xor_sync(MZ_FULL, s, m);
  const float mean = s / (float)d;
  const float c0 = lane < d ? v0 - mean : 0.0f, c1 = lane + 32 < d ? v1 - mean : 0.0f;
  float q = c0 * c0 + c1 * c1;
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) q += __shfl_xor_sync(MZ_FULL, q, m);
  const float rstd = 1.0f / sqrtf(q / (float)d + 1e-5f);
  float* out = X_out + (size_t)r * ldx;
  if (lane < d) out[lane] = fmaxf(c0 * rstd * gamma[lane] + beta[lane], 0.0f);
  if (lane + 32 < d) out[lane + 32] = fmaxf(c1 * rstd * gamma[lane + 32] + beta[lane + 32], 0.0f);
  const int act = actions != nullptr ? actions[(size_t)r * action_stride] : -1;
  if (lane < A) out[d + lane] = act == lane ? 1.0f : 0.0f;
  if (lane + 32 < A) out[d + lane + 32] = act == lane + 32 ? 1.0f : 0.0f;
  if (lane == 0) {
    mean_out[r] = mean;
    rstd_out[r] = rstd;
  }
}

// dY = d LN / dY applied to scale * dH masked by the ReLU (H > 0), gamma / beta gradients by atomics (one per
// column and CTA).  dH: the first d columns of the hidden state's gradient rows (lddh floats apart).
__global__ void ln_relu_backward_kernel(int rows, int d, const float* __restrict__ dH, int lddh, float scale,
                                        const float* __restrict__ Y, const float* __restrict__ H, int ldh,
                                        const float* __restrict__ mean_in, const float* __restrict__ rstd_in,
                                        const float* __restrict__ gamma, float* __restrict__ dY,
                                        float* __restrict__ ggamma, float* __restrict__ gbeta) {
  __shared__ float s_gg[64], s_gb[64];
  if (threadIdx.x < 64) s_gg[threadIdx.x] = s_gb[threadIdx.x] = 0.0f;
  __syncthreads();
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r < rows) {
    const float mean = mean_in[r], rstd = rstd_in[r];
    float g[2], xh[2], dxh[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int i = lane + 32 * u;
      g[u] = xh[u] = dxh[u] = 0.0f;
      if (i < d) {
        const float gi = H[(size_t)r * ldh + i] > 0.0f ? dH[(size_t)r * lddh + i] * scale : 0.0f;
        g[u] = gi;
        xh[u] = (Y[(size_t)r * d + i] - mean) * rstd;
        dxh[u] = gi * gamma[i];
      }
    }
    float s1 = dxh[0] + dxh[1], s2 = dxh[0] * xh[0] + dxh[1] * xh[1];
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) {
      s1 += __shfl_xor_sync(MZ_FULL, s1, m);
      s2 += __shfl_xor_sync(MZ_FULL, s2, m);
    }
    const float m1 = s1 / (float)d, m2 = s2 / (float)d;
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int i = lane + 32 * u;
      if (i < d) {
        dY[(size_t)r * d + i] = rstd * (dxh[u] - m1 - xh[u] * m2);
        atomicAdd(&s_gg[i], g[u] * xh[u]);
        atomicAdd(&s_gb[i], g[u]);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < d) {
    atomicAdd(ggamma + threadIdx.x, s_gg[threadIdx.x]);
    atomicAdd(gbeta + threadIdx.x, s_gb[threadIdx.x]);
  }
}

// out[c][r] = in[r][c]
__global__ void transpose_kernel(int rows, int cols, const float* __restrict__ in, float* __restrict__ out) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? in[(size_t)r * cols + c] : 0.0f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) out[(size_t)c * rows + r] = tile[threadIdx.x][i];
  }
}

__global__ void sumsq_kernel(long long n, const float* __restrict__ g, float* __restrict__ out) {
  float s = 0.0f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) s += g[i] * g[i];
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) s += __shfl_xor_sync(MZ_FULL, s, m);
  if ((threadIdx.x & 31) == 0) atomicAdd(out, s);
}

// torch.optim.AdamW / Adam (single-tensor formulas, float32): state[0] = step count (float), state[1] = learning rate,
// state[2] = sum of squared gradients (clipping; written by sumsq_kernel), read on the device so that a CUDA graph
// replays the step with fresh values.
__global__ void adam_step_kernel(long long n, float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                 float* __restrict__ v, const float* __restrict__ state, float beta1, float beta2,
                                 float eps, float weight_decay, int decoupled, float grad_scale, float clip_norm) {
  const float step = state[0], lr = state[1];
  float gs = grad_scale;
  if (clip_norm > 0.0f) {  // torch.nn.utils.clip_grad_norm_: g *= min(1, max_norm / (norm + 1e-6))
    const float norm = sqrtf(state[2]) * grad_scale;
    gs *= fminf(1.0f, clip_norm / (norm + 1e-6f));
  }
  const float bc1 = 1.0f - powf(beta1, step), bc2 = 1.0f - powf(beta2, step);
  const float step_size = lr / bc1, bc2_sqrt = sqrtf(bc2);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float w = p[i], gi = g[i] * gs;
    if (decoupled) w *= 1.0f - lr * weight_decay;  // AdamW
    else gi = fmaf(weight_decay, w, gi);            // Adam: L2 term in the gradient
    const float mi = m[i] + (gi - m[i]) * (1.0f - beta1);  // lerp_
    const float vi = v[i] * beta2 + (1.0f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = w - step_size * (mi / denom);
  }
}

__global__ void counter_inc_kernel(float* state) { state[0] += 1.0f; }

bool g_learner_attr = false;
int learner_attrs() {
  if (g_learner_attr) return 0;
  const auto attr = cudaFuncAttributeMaxDynamicSharedMemorySize;
  const int fwd = (int)((LMAXIN + LW) * LDH * sizeof(float)), bwd = (int)((LMAXIN + 2 * LW + LMAXOUT) * LDH * sizeof(float));
  cudaError_t e;
  if ((e = cudaFuncSetAttribute(mlp2_forward_kernel<false>, attr, fwd)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(mlp2_forward_kernel<true>, attr, fwd)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(mlp2_backward_kernel<false>, attr, bwd)) != cudaSuccess ||
      (e = cudaFuncSetAttribute(mlp2_backward_kernel<true>, attr, bwd)) != cudaSuccess)
    return (int)e;
  g_learner_attr = true;
  return 0;
}

}  // namespace

extern "C" {

int mz_mlp2_forward(int32_t rows, int32_t d_in, int32_t ldx, const float* X, const float* W1T, const float* b1,
                    const float* W2T, const float* b2, int32_t d_out, float* Y, int32_t ldy, void* stream) {
  if (rows < 1 || d_in < 1 || d_in > LMAXD || d_out < 1 || d_out > LMAXOUT || ldx < d_in || ldy < d_out || !X || !W1T ||
      !b1 || !W2T || !b2 || !Y)
    return MZ_ERR_BAD_ARG;
  if (int rc = learner_attrs()) return rc;
  const size_t smem = (LMAXIN + LW) * LDH * sizeof(float);
  if (d_in > LMAXIN)
    mlp2_forward_kernel<true><<<(rows + LR - 1) / LR, LT, smem, (cudaStream_t)stream>>>(rows, d_in, ldx, X, W1T, b1, W2T, b2,
                                                                                      d_out, Y, ldy);
  else
    mlp2_forward_kernel<false><<<(rows + LR - 1) / LR, LT, smem, (cudaStream_t)stream>>>(rows, d_in, ldx, X, W1T, b1, W2T, b2,
                                                                                       d_out, Y, ldy);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_mlp2_backward(int32_t rows, int32_t d_in, int32_t ldx, const float* X, const float* W1T, const float* b1,
                     const float* W1, const float* W2, int32_t d_out, const float* dY, int32_t ldy, float* dX,
                     int32_t lddx, float* gW1, float* gb1, float* gW2, float* gb2, void* stream) {
  if (rows < 1 || d_in < 1 || d_in > LMAXD || d_out < 1 || d_out > LMAXOUT || ldx < d_in || ldy < d_out || !X || !W1T ||
      !b1 || !W1 || !W2 || !dY || !gW1 || !gb1 || !gW2 || !gb2 || (dX && (lddx < d_in || d_in > LMAXIN)))
    return MZ_ERR_BAD_ARG;
  if (int rc = learner_attrs()) return rc;
  const size_t smem = (LMAXIN + 2 * LW + LMAXOUT) * LDH * sizeof(float);
  if (d_in > LMAXIN)
    mlp2_backward_kernel<true><<<(rows + LR - 1) / LR, LT, smem, (cudaStream_t)stream>>>(
        rows, d_in, ldx, X, W1T, b1, W1, W2, d_out, dY, ldy, dX, lddx, gW1, gb1, gW2, gb2);
  else
    mlp2_backward_kernel<false><<<(rows + LR - 1) / LR, LT, smem, (cudaStream_t)stream>>>(
        rows, d_in, ldx, X, W1T, b1, W1, W2, d_out, dY, ldy, dX, lddx, gW1, gb1, gW2, gb2);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_ln_relu_forward(int32_t rows, int32_t d, const float* Y, const float* gamma, const float* beta,
                       const int32_t* actions, int32_t action_stride, int32_t num_actions, float* X_out, int32_t ldx,
                       float* mean, float* rstd, void* stream) {
  if (rows < 1 || d < 1 || d > 64 || num_actions < 0 || num_actions > 64 || ldx < d + num_actions || !Y || !gamma || !beta ||
      !X_out || !mean || !rstd)
    return MZ_ERR_BAD_ARG;
  ln_relu_forward_kernel<<<(rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(rows, d, Y, gamma, beta, actions, action_stride,
                                                                          num_actions, X_out, ldx, mean, rstd);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_ln_relu_backward(int32_t rows, int32_t d, const float* dH, int32_t lddh, float scale, const float* Y,
                        const float* H, int32_t ldh, const float* mean, const float* rstd, const float* gamma, float* dY,
                        float* ggamma, float* gbeta, void* stream) {
  if (rows < 1 || d < 1 || d > 64 || lddh < d || ldh < d || !dH || !Y || !H || !mean || !rstd || !gamma || !dY || !ggamma ||
      !gbeta)
    return MZ_ERR_BAD_ARG;
  ln_relu_backward_kernel<<<(rows + 7) / 8, 256, 0, (cudaStream_t)stream>>>(rows, d, dH, lddh, scale, Y, H, ldh, mean, rstd,
                                                                           gamma, dY, ggamma, gbeta);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_learner_transpose(int32_t rows, int32_t cols, const float* in, float* out, void* stream) {
  if (rows < 1 || cols < 1 || !in || !out) return MZ_ERR_BAD_ARG;
  transpose_kernel<<<dim3((cols + 31) / 32, (rows + 31) / 32), dim3(32, 8), 0, (cudaStream_t)stream>>>(rows, cols, in, out);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_adam_step(int64_t n, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float* state,
                 float beta1, float beta2, float eps, float weight_decay, int32_t decoupled, float grad_scale,
                 float clip_norm, void* stream) {
  if (n < 1 || !params || !grads || !exp_avg || !exp_avg_sq || !state) return MZ_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  counter_inc_kernel<<<1, 1, 0, st>>>(state);
  if (clip_norm > 0.0f) {
    cudaMemsetAsync(state + 2, 0, sizeof(float), st);
    sumsq_kernel<<<148, 256, 0, st>>>(n, grads, state + 2);
  }
  adam_step_kernel<<<148 * 2, 256, 0, st>>>(n, params, grads, exp_avg, exp_avg_sq, state, beta1, beta2, eps, weight_decay,
                                            decoupled, grad_scale, clip_norm);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

}  // extern "C"
