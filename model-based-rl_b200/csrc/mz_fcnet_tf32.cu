// FCNetwork inference at float32 accuracy ON THE TENSOR CORES: every product of the eight Linear layers runs as
// three TF32 tensor-core instructions on split operands (x = x_hi + x_lo, w = w_hi + w_lo, see split_tf32;
// x*w ~= x_lo*w_hi + x_hi*w_lo + x_hi*w_hi, float32 accumulation: what is dropped is below 2^-20 of the product,
// the level of the float32 kernels' own summation-order differences).  Same interface, same weights struct and the same
// results within float32 rounding as the CUDA-core kernels of mz_fcnet_f32.cu (tests/test_gpu_fcnet.py: 1e-4
// against the reference's torch module like the float32 kernel, 2e-5 against the float32 kernel itself).
//
// One CTA of sixteen warps evaluates the whole network for 32 rows (two m16 tiles), activations never leave shared
// memory.  First layers (K <= 56 or obs_dim, N = 512): a warp owns 32 output columns of both row tiles and
// streams its weight columns from L2 as 16-byte loads two k steps ahead (MMA column j of tile nt <-> column
// 4 j + nt, so a thread's four B values of a k row are contiguous).  Second layers (K = 512, N <= 64): the K range
// is split over eight warp pairs x two row tiles (MMA k index j <-> k = 8 s + 2 (j mod 4) + j / 4: 8-byte operand
// loads on both sides), partial sums meet in shared memory in a fixed order (deterministic).  The three
// instructions of a product go out term by term over all of a warp's accumulators, never back to back on one.
// Reference: networks.py:26-34, 55-174; config.py:27-33 (JimOhman/model-based-rl).
#include <math.h>

#include "mz_common.cuh"
#include "mz_transforms.cuh"

namespace {

constexpr int R = 32;            // rows per CTA
constexpr int kThr = 512;        // sixteen warps
constexpr int kWarps = kThr / 32;
constexpr int H = MZ_FC_HIDDEN;  // 50
constexpr int W = MZ_FC_WIDTH;   // 512
constexpr int LDH = 60;          // row stride of a [R][56] hidden image: 60 = 28 (mod 32), A-fragment loads hit 32 banks
constexpr int LDA = 520;         // row stride of the first-layer activations: 8 (mod 32), 8-byte fragment loads conflict free
constexpr int LDO = 72;          // row stride of second-layer outputs (<= 64 columns)
constexpr int LDR = 64;          // row stride of a partial-sum slot

MZ_DEV void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, "
      "{%0, %1, %2, %3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

// weight row k of a first layer, this thread's four columns; rows past K - 1 read row K - 1 (their x column is zero)
MZ_DEV float4 load4(const float* __restrict__ wcol, int k, int K) {
  return __ldg(reinterpret_cast<const float4*>(wcol + (size_t)min(k, K - 1) * W));
}

// out[r][n] = relu(b1[n] + sum_{k < K} x[r][k] * w1t[k][n] (+ w1t[K + act[r]][n])), n < 512, r < 32.
// x: shared [R][ldx], columns K .. round_up(K, 8) - 1 are zero.  All sixteen warps call.
MZ_DEV void first_layer(const float* __restrict__ w1t, const float* __restrict__ b1, const float* x, int ldx, int K,
                        const int* act, float* out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int n0 = warp * 32;
  float acc[2][4][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[mt][nt][i] = 0.0f;
  // the epilogue's operands (this warp's 128-byte line of the bias and of each row's one-hot weight row) -> L1
  asm volatile("prefetch.global.L1 [%0];" ::"l"(act ? w1t + (size_t)(K + act[lane]) * W + n0 : b1 + n0));
  if (act && lane == 0) asm volatile("prefetch.global.L1 [%0];" ::"l"(b1 + n0));
  const int ksteps = (K + 7) >> 3;
  const float* wcol = w1t + n0 + g * 4;  // this thread's 4 columns; rows t and t + 4 of a k step
  // weight rows of the next two k steps are in flight while a step computes
  float4 p0a = load4(wcol, t, K), p0b = load4(wcol, t + 4, K);
  float4 p1a = load4(wcol, 8 + t, K), p1b = load4(wcol, 12 + t, K);
  for (int ks = 0; ks < ksteps; ++ks) {
    const int k0 = ks * 8;
    const float4 ca = p0a, cb = p0b;
    p0a = p1a, p0b = p1b;
    p1a = load4(wcol, k0 + 16 + t, K);
    p1b = load4(wcol, k0 + 20 + t, K);
    uint32_t ah[2][4], al[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const float* xr = x + (mt * 16 + g) * ldx + k0 + t;
      split_tf32(xr[0], ah[mt][0], al[mt][0]);
      split_tf32(xr[8 * ldx], ah[mt][1], al[mt][1]);
      split_tf32(xr[4], ah[mt][2], al[mt][2]);
      split_tf32(xr[8 * ldx + 4], ah[mt][3], al[mt][3]);
    }
    const float wa[4] = {ca.x, ca.y, ca.z, ca.w}, wb[4] = {cb.x, cb.y, cb.z, cb.w};
    uint32_t bh[4][2], bl[4][2];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      split_tf32(wa[nt], bh[nt][0], bl[nt][0]);
      split_tf32(wb[nt], bh[nt][1], bl[nt][1]);
    }
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      mma_tf32(acc[0][nt], al[0], bh[nt]);
      mma_tf32(acc[1][nt], al[1], bh[nt]);
    }
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      mma_tf32(acc[0][nt], ah[0], bl[nt]);
      mma_tf32(acc[1][nt], ah[1], bl[nt]);
    }
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      mma_tf32(acc[0][nt], ah[0], bh[nt]);
      mma_tf32(acc[1][nt], ah[1], bh[nt]);
    }
  }
  // thread (g, t) holds rows {g, g + 8} of both tiles x columns n0 + 8 t + {0..7}: c0 / c2 = column nt, c1 / c3 = 4 + nt
  const int c0 = n0 + 8 * t;
  float bias[8];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const float4 b = __ldg(reinterpret_cast<const float4*>(b1 + c0) + q);
    bias[4 * q] = b.x, bias[4 * q + 1] = b.y, bias[4 * q + 2] = b.z, bias[4 * q + 3] = b.w;
  }
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const int row = mt * 16 + hf * 8 + g;
      float v[8];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        v[nt] = acc[mt][nt][2 * hf];
        v[4 + nt] = acc[mt][nt][2 * hf + 1];
      }
      if (act) {  // one-hot action column (attach_action, networks.py:167-174)
        const float4* oh = reinterpret_cast<const float4*>(w1t + (size_t)(K + act[row]) * W + c0);
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const float4 o = __ldg(oh + q);
          v[4 * q] += o.x, v[4 * q + 1] += o.y, v[4 * q + 2] += o.z, v[4 * q + 3] += o.w;
        }
      }
      float4* dst = reinterpret_cast<float4*>(out + row * LDA + c0);
#pragma unroll
      for (int q = 0; q < 2; ++q)
        dst[q] = make_float4(fmaxf(v[4 * q] + bias[4 * q], 0.0f), fmaxf(v[4 * q + 1] + bias[4 * q + 1], 0.0f),
                             fmaxf(v[4 * q + 2] + bias[4 * q + 2], 0.0f), fmaxf(v[4 * q + 3] + bias[4 * q + 3], 0.0f));
    }
}

// Second layers.  Warp (warp & 1, warp >> 1) = (row tile, k slice of 64); NT = compile-time bound of the n tiles.
// A warp's B fragments of k step s: NT 8-byte loads, issued one step ahead (the first ones before the barrier that
// ends the first layers) so that the L2 round trip runs under the previous step's instructions.
template <int NT>
struct W2Frag {
  float2 v[NT > 0 ? NT : 1];
};
template <int NT>
MZ_DEV void w2_prefetch(W2Frag<NT>& f, const float* __restrict__ w2, int N2, int s) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const float* wr = w2 + (warp >> 1) * 64 + 2 * t + 8 * s;
  const int ntiles = (N2 + 7) >> 3;
  // rows past N2 read the last row instead: their output columns are never reduced (no select behind the load, which
  // would wait for it right here)
#pragma unroll
  for (int nt = 0; nt < NT; ++nt)
    if (nt < ntiles) f.v[nt] = __ldg(reinterpret_cast<const float2*>(wr + (size_t)min(nt * 8 + g, N2 - 1) * W));
}
// partial second layer of one warp: rows of tile (warp & 1), k in [64 (warp >> 1), +64), all N2 <= 8 NT outputs
template <int NT>
MZ_DEV void second_partial(W2Frag<NT>& f, const float* __restrict__ w2, const float* in, int N2, float (&acc)[NT > 0 ? NT : 1][4]) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int mt = warp & 1, kw = (warp >> 1) * 64;
  const int ntiles = (N2 + 7) >> 3;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt)
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[nt][i] = 0.0f;
  const float* x0 = in + (mt * 16 + g) * LDA + kw + 2 * t;
#pragma unroll 2
  for (int s = 0; s < 8; ++s) {
    uint32_t bh[NT > 0 ? NT : 1][2], bl[NT > 0 ? NT : 1][2];
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
      if (nt < ntiles) {
        split_tf32(f.v[nt].x, bh[nt][0], bl[nt][0]);
        split_tf32(f.v[nt].y, bh[nt][1], bl[nt][1]);
      }
    if (s + 1 < 8) w2_prefetch<NT>(f, w2, N2, s + 1);
    const float2 xa = *reinterpret_cast<const float2*>(x0 + 8 * s);
    const float2 xb = *reinterpret_cast<const float2*>(x0 + 8 * LDA + 8 * s);
    uint32_t ah[4], al[4];
    split_tf32(xa.x, ah[0], al[0]);
    split_tf32(xb.x, ah[1], al[1]);
    split_tf32(xa.y, ah[2], al[2]);
    split_tf32(xb.y, ah[3], al[3]);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
      if (nt < ntiles) mma_tf32(acc[nt], al, bh[nt]);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
      if (nt < ntiles) mma_tf32(acc[nt], ah, bl[nt]);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt)
      if (nt < ntiles) mma_tf32(acc[nt], ah, bh[nt]);
  }
}
// a warp's partial sums -> slot (warp >> 1) of `red` ([8][R][LDR])
template <int NT>
MZ_DEV void store_partial(const float (&acc)[NT > 0 ? NT : 1][4], int N2, float* red) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int mt = warp & 1, ntiles = (N2 + 7) >> 3;
  float* base = red + ((warp >> 1) * R + mt * 16 + g) * LDR + 2 * t;
#pragma unroll
  for (int nt = 0; nt < NT; ++nt)
    if (nt < ntiles) {
      *reinterpret_cast<float2*>(base + nt * 8) = make_float2(acc[nt][0], acc[nt][1]);
      *reinterpret_cast<float2*>(base + 8 * LDR + nt * 8) = make_float2(acc[nt][2], acc[nt][3]);
    }
}
// out[r][n] = b2[n] + the eight partial sums in slot order
MZ_DEV void reduce_partials(const float* red, const float* __restrict__ b2, int N2, float* out, int ldo) {
  for (int i = threadIdx.x; i < R * N2; i += kThr) {
    const int r = i / N2, n = i - r * N2;
    const float* p = red + r * LDR + n;
    float v = p[0];
#pragma unroll
    for (int q = 1; q < 8; ++q) v += p[q * R * LDR];
    out[r * ldo + n] = v + __ldg(b2 + n);
  }
}

// relu(LayerNorm(x)) over H features (networks.py:149, 164), one warp per row; columns H .. 55 are zeroed (K padding)
MZ_DEV void layernorm_relu(const float* __restrict__ ln_w, const float* __restrict__ ln_b, float* x) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < R; r += kWarps) {
    float* row = x + r * LDH;
    float s = 0.0f;
    for (int i = lane; i < H; i += 32) s += row[i];
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) s += __shfl_xor_sync(MZ_FULL, s, m);
    const float mean = s / (float)H;
    float q = 0.0f;
    for (int i = lane; i < H; i += 32) {
      const float d = row[i] - mean;
      q = fmaf(d, d, q);
    }
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) q += __shfl_xor_sync(MZ_FULL, q, m);
    const float rstd = 1.0f / sqrtf(q / (float)H + 1e-5f);
    for (int i = lane; i < H; i += 32) row[i] = fmaxf((row[i] - mean) * rstd * ln_w[i] + ln_b[i], 0.0f);
    if (lane < 56 - H) row[H + lane] = 0.0f;
  }
}

struct Smem {
  float* a;   // [2][R][LDA] first-layer activations of two heads; afterwards the partial sums [2][8][R][LDR]
  float* h;   // [R][LDH] hidden state
  float* o;   // [2][R][LDO] second-layer outputs
  int* act;   // [R]
  float* x;   // [R][ldx] inputs
};
MZ_DEV Smem carve(float* base) {
  Smem s;
  s.a = base;
  s.h = s.a + 2 * R * LDA;
  s.o = s.h + R * LDH;
  s.act = reinterpret_cast<int*>(s.o + 2 * R * LDO);
  s.x = reinterpret_cast<float*>(s.act + R);
  return s;
}
size_t smem_bytes(int ldx) { return sizeof(float) * (size_t)(2 * R * LDA + R * LDH + 2 * R * LDO + R + R * ldx); }

// second layers of two heads whose first-layer activations sit in a[0] / a[1] -> oa [R][ldoa], ob [R][ldob]
// (NTA / NTB: bounds of the heads' n tiles; NTB = 0: one head)
template <int NTA, int NTB>
MZ_DEV void second_stage(float* a, const float* __restrict__ w2a, const float* __restrict__ b2a, int Na,
                                          float* oa, int ldoa, const float* __restrict__ w2b,
                                          const float* __restrict__ b2b, int Nb, float* ob, int ldob) {
  float* a0 = a;
  float* a1 = a + R * LDA;
  W2Frag<NTA> fa;
  W2Frag<NTB> fb;
  w2_prefetch<NTA>(fa, w2a, Na, 0);
  if (NTB > 0) w2_prefetch<NTB>(fb, w2b, Nb, 0);
  __syncthreads();  // the first layers are complete
  float acc_a[NTA][4], acc_b[NTB > 0 ? NTB : 1][4];
  second_partial<NTA>(fa, w2a, a0, Na, acc_a);
  if (NTB > 0) second_partial<NTB>(fb, w2b, a1, Nb, acc_b);
  __syncthreads();  // every warp is done with the activations: their storage takes the partial sums
  float* red_a = a;
  float* red_b = a + 8 * R * LDR;
  store_partial<NTA>(acc_a, Na, red_a);
  if (NTB > 0) store_partial<NTB>(acc_b, Nb, red_b);
  __syncthreads();
  reduce_partials(red_a, b2a, Na, oa, ldoa);
  if (NTB > 0) reduce_partials(red_b, b2b, Nb, ob, ldob);
  __syncthreads();
}
// two heads that read the same input x [R][ldx] (w1b = nullptr: one head)
MZ_DEV void head_pair(const Smem& s, const float* x, int ldx, int K, const int* act, const float* w1a, const float* b1a,
                      const float* w2a, const float* b2a, int Na, float* oa, int ldoa, const float* w1b,
                      const float* b1b, const float* w2b, const float* b2b, int Nb, float* ob, int ldob) {
  first_layer(w1a, b1a, x, ldx, K, act, s.a);
  if (w1b) first_layer(w1b, b1b, x, ldx, K, act, s.a + R * LDA);
  if (!w1b)
    second_stage<8, 0>(s.a, w2a, b2a, Na, oa, ldoa, w2b, b2b, Nb, ob, ldob);
  else if (Na <= 32 && Nb <= 32)
    second_stage<4, 4>(s.a, w2a, b2a, Na, oa, ldoa, w2b, b2b, Nb, ob, ldob);
  else if (Na <= 32)
    second_stage<4, 8>(s.a, w2a, b2a, Na, oa, ldoa, w2b, b2b, Nb, ob, ldob);
  else
    second_stage<8, 8>(s.a, w2a, b2a, Na, oa, ldoa, w2b, b2b, Nb, ob, ldob);
}

// prediction (networks.py:151-157) from s.h; writes value [B], logits [B][A]
MZ_DEV void prediction(const mz_fc_weights& w, const Smem& s, int row0, int batch, float* value, float* logits) {
  float* o0 = s.o;
  float* o1 = s.o + R * LDO;
  head_pair(s, s.h, LDH, H, nullptr, w.val_w1, w.val_b1, w.val_w2, w.val_b2, w.value_bins, o0, LDO, w.pol_w1, w.pol_b1,
            w.pol_w2, w.pol_b2, w.num_actions, o1, LDO);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < R; r += kWarps) {
    const int b = row0 + r;
    if (b >= batch) continue;
    const float v = w.no_support ? o0[r * LDO]  // networks.py:153: the raw output of a one-unit head
                                 : mz_support_to_scalar_warp(o0 + r * LDO, w.value_bins, w.value_min, w.no_target_transform, lane);
    if (lane == 0) value[b] = v;
    for (int a = lane; a < w.num_actions; a += 32) logits[(size_t)b * w.num_actions + a] = o1[r * LDO + a];
  }
}

__global__ void __launch_bounds__(kThr, 1)
fc_recurrent_tf32x3_kernel(mz_fc_weights w, int batch, const float* __restrict__ hidden_in, long long in_row_stride,
                           const int32_t* __restrict__ in_index, const int32_t* __restrict__ actions,
                           float* __restrict__ hidden_out, long long out_row_stride, long long out_offset,
                           float* __restrict__ value, float* __restrict__ reward, float* __restrict__ logits) {
  extern __shared__ __align__(16) float smem[];
  const Smem s = carve(smem);
  const int row0 = blockIdx.x * R;
  for (int i = threadIdx.x; i < R * 56; i += kThr) {
    const int r = i / 56, k = i - r * 56, b = min(row0 + r, batch - 1);
    const float* src = hidden_in + (size_t)b * in_row_stride + (in_index ? (size_t)in_index[b] * H : 0);
    s.x[r * LDH + k] = k < H ? src[k] : 0.0f;
  }
  if (threadIdx.x < R) s.act[threadIdx.x] = actions[min(row0 + (int)threadIdx.x, batch - 1)];
  __syncthreads();
  // dynamics (networks.py:159-165): reward head -> o[0], transition head -> h
  head_pair(s, s.x, LDH, H, s.act, w.rew_w1, w.rew_b1, w.rew_w2, w.rew_b2, w.reward_bins, s.o, LDO, w.dyn_w1, w.dyn_b1,
            w.dyn_w2, w.dyn_b2, H, s.h, LDH);
  layernorm_relu(w.ln_w, w.ln_b, s.h);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r = warp; r < R; r += kWarps) {
    const int b = row0 + r;
    if (b >= batch) continue;
    const float rv = w.no_support ? s.o[r * LDO]  // networks.py:161
                                  : mz_support_to_scalar_warp(s.o + r * LDO, w.reward_bins, w.reward_min, w.no_target_transform, lane);
    if (lane == 0) reward[b] = rv;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < R * H; i += kThr) {
    const int r = i / H, k = i - r * H, b = row0 + r;
    if (b < batch) hidden_out[(size_t)b * out_row_stride + out_offset + k] = s.h[r * LDH + k];
  }
  prediction(w, s, row0, batch, value, logits);
}

__global__ void __launch_bounds__(kThr, 1)
fc_initial_tf32x3_kernel(mz_fc_weights w, int batch, const float* __restrict__ obs, float* __restrict__ hidden,
                         long long hidden_stride, float* __restrict__ value, float* __restrict__ logits, int ldx) {
  extern __shared__ __align__(16) float smem[];
  const Smem s = carve(smem);
  const int row0 = blockIdx.x * R;
  const int K = w.obs_dim, Kp = (K + 7) & ~7;
  for (int i = threadIdx.x; i < R * Kp; i += kThr) {
    const int r = i / Kp, k = i - r * Kp, b = min(row0 + r, batch - 1);
    s.x[r * ldx + k] = k < K ? obs[(size_t)b * K + k] : 0.0f;
  }
  __syncthreads();
  // representation (networks.py:146-149)
  head_pair(s, s.x, ldx, K, nullptr, w.rep_w1, w.rep_b1, w.rep_w2, w.rep_b2, H, s.h, LDH, nullptr, nullptr, nullptr,
            nullptr, 0, nullptr, 0);
  layernorm_relu(w.ln_w, w.ln_b, s.h);
  __syncthreads();
  for (int i = threadIdx.x; i < R * H; i += kThr) {
    const int r = i / H, k = i - r * H, b = row0 + r;
    if (b < batch) hidden[(size_t)b * hidden_stride + k] = s.h[r * LDH + k];
  }
  prediction(w, s, row0, batch, value, logits);
}

int check_weights(const mz_fc_weights* w, bool need_rep) {
  if (!w) return MZ_ERR_BAD_ARG;
  if (w->num_actions < 1 || w->num_actions > 64 || w->value_bins < 1 || w->value_bins > 64 || w->reward_bins < 1 ||
      w->reward_bins > 64)
    return MZ_ERR_UNSUPPORTED;
  if (w->no_support && (w->value_bins != 1 || w->reward_bins != 1)) return MZ_ERR_BAD_ARG;
  if (!w->dyn_w1 || !w->rew_w1 || !w->val_w1 || !w->pol_w1 || !w->ln_w || !w->ln_b) return MZ_ERR_BAD_ARG;
  if (need_rep && (!w->rep_w1 || !w->rep_w2 || w->obs_dim < 1)) return MZ_ERR_BAD_ARG;
  return MZ_OK;
}

}  // namespace

extern "C" {

int mz_fc_initial_tf32x3(const mz_fc_weights* w, int32_t batch, const float* obs, float* hidden, int64_t hidden_stride,
                         float* value, float* logits, void* stream) {
  int rc = check_weights(w, true);
  if (rc) return rc;
  if (batch < 1 || !obs || !hidden || !value || !logits) return MZ_ERR_BAD_ARG;
  const int ldx = ((w->obs_dim + 7) & ~7) + 4;  // 4 (mod 8): conflict-free A-fragment loads
  const size_t smem = smem_bytes(ldx);
  if (smem > 227 * 1024) return MZ_ERR_UNSUPPORTED;
  cudaError_t e = cudaFuncSetAttribute(fc_initial_tf32x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const int grid = (batch + R - 1) / R;
  fc_initial_tf32x3_kernel<<<grid, kThr, smem, (cudaStream_t)stream>>>(*w, batch, obs, hidden, hidden_stride, value,
                                                                      logits, ldx);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

int mz_fc_recurrent_tf32x3(const mz_fc_weights* w, int32_t batch, const float* hidden_in, int64_t in_row_stride,
                           const int32_t* in_index, const int32_t* actions, float* hidden_out, int64_t out_row_stride,
                           int64_t out_offset, float* value, float* reward, float* logits, void* stream) {
  int rc = check_weights(w, false);
  if (rc) return rc;
  if (batch < 1 || !hidden_in || !actions || !hidden_out || !value || !reward || !logits) return MZ_ERR_BAD_ARG;
  const size_t smem = smem_bytes(LDH);
  cudaError_t e =
      cudaFuncSetAttribute(fc_recurrent_tf32x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  const int grid = (batch + R - 1) / R;
  fc_recurrent_tf32x3_kernel<<<grid, kThr, smem, (cudaStream_t)stream>>>(
      *w, batch, hidden_in, in_row_stride, in_index, actions, hidden_out, out_row_stride, out_offset, value, reward,
      logits);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

}  // extern "C"
