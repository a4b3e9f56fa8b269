// Learner unroll loss (Learner.update_weights, learners.py:182-213) as one fused pass over the logits
// of all K+1 unroll steps: h(x) of the scalar targets (config.py:51-54), two-hot projection
// (config.py:56-68), the three cross-entropies (utils.py:53-56), their importance weighting in
// float64 (learners.py:208-210), the priority errors (learners.py:182-183) and the gradient with
// respect to every logit, including the 1/K scale of learners.py:213.  mz_scalar_unroll_loss is the same pass for
// `--no_support` networks, whose value and reward heads emit one scalar (MSE or Huber, utils.py:61-70).
//
// HBM bound and tiny: every logit is read once and its gradient written once.
#include <math.h>

#include "mz_transforms.cuh"

namespace {

// One warp: cross-entropy of a row of `n` logits against a two-hot target (lo, hi, p_lo, p_hi), and
// the gradient g * (softmax * sum(t) - t) in the operation order of torch's autograd
// (mul / neg / log_softmax backward).  float32 like the reference.
MZ_DEV void warp_max_sum(const float* x, int n, int lane, float& m, float& lse) {
  m = -INFINITY;
  for (int j = lane; j < n; j += 32) m = fmaxf(m, x[j]);
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) m = fmaxf(m, __shfl_xor_sync(MZ_FULL, m, s));
  float den = 0.0f;
  for (int j = lane; j < n; j += 32) den += expf(x[j] - m);
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) den += __shfl_xor_sync(MZ_FULL, den, s);
  lse = logf(den);
}

MZ_DEV float warp_sum(float v) {
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(MZ_FULL, v, s);
  return v;
}

MZ_DEV float ce_two_hot(const float* x, float* dx, int n, float target, int smin, int smax, int no_tt, float g,
                        int lane) {
  if (!no_tt) target = mz_scalar_transform_f(target);
  const MzTwoHot t = mz_two_hot(target, smin, smax);
  float m, lse;
  warp_max_sum(x, n, lane, m, lse);
  float loss = 0.0f, go_sum = 0.0f;
  // target row: p_hi at hi, then p_lo at lo (integer x: lo == hi holds 1.0)
  for (int j = lane; j < n; j += 32) {
    float tj = 0.0f;
    if (j == t.hi) tj = t.p_hi;
    if (j == t.lo) tj = t.p_lo;
    const float logsm = __fsub_rn(__fsub_rn(x[j], m), lse);
    loss += __fmul_rn(-tj, logsm);
    go_sum += -__fmul_rn(tj, g);
  }
  loss = warp_sum(loss);
  go_sum = warp_sum(go_sum);
  if (dx) {
    for (int j = lane; j < n; j += 32) {
      float tj = 0.0f;
      if (j == t.hi) tj = t.p_hi;
      if (j == t.lo) tj = t.p_lo;
      const float logsm = __fsub_rn(__fsub_rn(x[j], m), lse);
      dx[j] = __fsub_rn(-__fmul_rn(tj, g), __fmul_rn(expf(logsm), go_sum));
    }
  }
  return loss;
}

MZ_DEV float ce_dense(const float* x, float* dx, const float* t, int n, float g, int lane) {
  float m, lse;
  warp_max_sum(x, n, lane, m, lse);
  float loss = 0.0f, go_sum = 0.0f;
  for (int j = lane; j < n; j += 32) {
    const float logsm = __fsub_rn(__fsub_rn(x[j], m), lse);
    loss += __fmul_rn(-t[j], logsm);
    go_sum += -__fmul_rn(t[j], g);
  }
  loss = warp_sum(loss);
  go_sum = warp_sum(go_sum);
  if (dx) {
    for (int j = lane; j < n; j += 32) {
      const float logsm = __fsub_rn(__fsub_rn(x[j], m), lse);
      dx[j] = __fsub_rn(-__fmul_rn(t[j], g), __fmul_rn(expf(logsm), go_sum));
    }
  }
  return loss;
}

// grid = batch rows, block = 32 * (K + 1): warp i owns unroll step i of row b.
__global__ void unroll_loss_kernel(mz_loss_cfg c, const float* __restrict__ value_logits,
                                   const float* __restrict__ reward_logits,
                                   const float* __restrict__ policy_logits, const float* __restrict__ t_values,
                                   const float* __restrict__ t_rewards, const float* __restrict__ t_policies,
                                   const double* __restrict__ is_weights, float* __restrict__ d_value,
                                   float* __restrict__ d_reward, float* __restrict__ d_policy,
                                   double* __restrict__ row_losses, float* __restrict__ new_errors) {
  __shared__ float s_loss[3][32];
  const int b = blockIdx.x, i = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int B = c.batch, K = c.num_unroll_steps, A = c.num_actions;
  const int V = c.value_max - c.value_min + 1, R = c.reward_max - c.reward_min + 1;
  const double w = is_weights ? is_weights[b] : 1.0;
  // d(full loss) / d(row loss): hook (1/K) -> mean (/B) -> * is_weights, float64, then the cast to
  // the float32 of the per-row losses (learners.py:208-213)
  const float g = (float)(((1.0 / (double)K) / (double)B) * w);

  const size_t vrow = ((size_t)i * B + b) * V;
  const float tv = t_values[(size_t)b * (K + 1) + i];
  const float lv = ce_two_hot(value_logits + vrow, d_value ? d_value + vrow : nullptr, V, tv, c.value_min,
                              c.value_max, c.no_target_transform, g, lane);
  float lr = 0.0f;
  if (i >= 1) {
    const size_t rrow = ((size_t)(i - 1) * B + b) * R;
    const float tr = t_rewards[(size_t)b * (K + 1) + i];
    lr = ce_two_hot(reward_logits + rrow, d_reward ? d_reward + rrow : nullptr, R, tr, c.reward_min, c.reward_max,
                    c.no_target_transform, g, lane);
  }
  const size_t prow = ((size_t)i * B + b) * A;
  const float lp = ce_dense(policy_logits + prow, d_policy ? d_policy + prow : nullptr,
                            t_policies + ((size_t)b * (K + 1) + i) * A, A, g, lane);
  if (lane == 0) {
    s_loss[0][i] = lr;
    s_loss[1][i] = lv;
    s_loss[2][i] = lp;
  }
  if (i == 0 && new_errors) {
    // learners.py:182-183: inverse_value_transform(value) - target_values[:, 0] (raw target)
    const float v0 = mz_support_to_scalar_warp(value_logits + vrow, V, c.value_min, c.no_target_transform, lane);
    if (lane == 0) new_errors[b] = __fsub_rn(v0, tv);
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    // float32 accumulation over the steps in step order (`loss += ...`, learners.py:199-206)
    float acc = (threadIdx.x == 0) ? 0.0f : s_loss[threadIdx.x][0];
    for (int k = 1; k <= K; ++k) acc = __fadd_rn(acc, s_loss[threadIdx.x][k]);
    row_losses[(size_t)threadIdx.x * B + b] = w * (double)acc;
  }
}

// One scalar head output against its target: MSELoss / SmoothL1Loss(beta = 1) with reduction='none' (utils.py:61-70),
// and the gradient g * dl/dx in the operation order of torch's mse_loss_backward (2 (x - t) g) and
// smooth_l1_loss_backward (-g / g outside [-1, 1], x g inside).  Explicit _rn intrinsics: no FMA contraction.
MZ_DEV float scalar_loss_and_grad(float x, float t, int huber, float g, float* dx) {
  const float d = __fsub_rn(x, t);
  if (!huber) {
    *dx = __fmul_rn(__fmul_rn(2.0f, d), g);
    return __fmul_rn(d, d);
  }
  *dx = d < -1.0f ? -g : (d > 1.0f ? g : __fmul_rn(d, g));
  const float z = fabsf(d);
  return z < 1.0f ? __fmul_rn(__fmul_rn(0.5f, z), z) : __fsub_rn(z, 0.5f);
}

// learners.scalar_unroll_loss for `--no_support` networks: value_logits [K+1][B][1] and reward_logits [K][B][1] are the
// scalar head outputs.  grid = batch rows, block = 32 * (K + 1): warp i owns unroll step i of row b; lane 0 does the
// scalar value / reward terms, the warp the policy cross-entropy.
__global__ void scalar_unroll_loss_kernel(mz_loss_cfg c, int huber, const float* __restrict__ value_out,
                                          const float* __restrict__ reward_out, const float* __restrict__ policy_logits,
                                          const float* __restrict__ t_values, const float* __restrict__ t_rewards,
                                          const float* __restrict__ t_policies, const double* __restrict__ is_weights,
                                          float* __restrict__ d_value, float* __restrict__ d_reward,
                                          float* __restrict__ d_policy, double* __restrict__ row_losses,
                                          float* __restrict__ new_errors) {
  __shared__ float s_loss[3][32];
  const int b = blockIdx.x, i = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int B = c.batch, K = c.num_unroll_steps, A = c.num_actions;
  const double w = is_weights ? is_weights[b] : 1.0;
  const float g = (float)(((1.0 / (double)K) / (double)B) * w);  // as in unroll_loss_kernel

  const size_t prow = ((size_t)i * B + b) * A;
  const float lp = ce_dense(policy_logits + prow, d_policy ? d_policy + prow : nullptr,
                            t_policies + ((size_t)b * (K + 1) + i) * A, A, g, lane);
  if (lane == 0) {
    const size_t vrow = (size_t)i * B + b;
    const float v = value_out[vrow], tv_raw = t_values[(size_t)b * (K + 1) + i];
    const float tv = c.no_target_transform ? tv_raw : mz_scalar_transform_f(tv_raw);
    float dv, dr, lr = 0.0f;
    const float lv = scalar_loss_and_grad(v, tv, huber, g, &dv);
    if (d_value) d_value[vrow] = dv;
    if (i >= 1) {
      const size_t rrow = (size_t)(i - 1) * B + b;
      const float tr_raw = t_rewards[(size_t)b * (K + 1) + i];
      const float tr = c.no_target_transform ? tr_raw : mz_scalar_transform_f(tr_raw);
      lr = scalar_loss_and_grad(reward_out[rrow], tr, huber, g, &dr);
      if (d_reward) d_reward[rrow] = dr;
    }
    // learners.py:182-183: the raw value output minus the raw target, no inverse transform
    if (i == 0 && new_errors) new_errors[b] = __fsub_rn(v, tv_raw);
    s_loss[0][i] = lr;
    s_loss[1][i] = lv;
    s_loss[2][i] = lp;
  }
  __syncthreads();
  if (threadIdx.x < 3) {
    // float32 accumulation over the steps in step order, as in unroll_loss_kernel
    float acc = (threadIdx.x == 0) ? 0.0f : s_loss[threadIdx.x][0];
    for (int k = 1; k <= K; ++k) acc = __fadd_rn(acc, s_loss[threadIdx.x][k]);
    row_losses[(size_t)threadIdx.x * B + b] = w * (double)acc;
  }
}

// (is_weights * loss).mean() for the three losses: fixed-order float64 tree, one CTA per loss.
__global__ void loss_mean_kernel(int B, const double* __restrict__ row_losses, double* __restrict__ losses) {
  __shared__ double s[256];
  const int which = blockIdx.x;
  double acc = 0.0;
  for (int b = threadIdx.x; b < B; b += 256) acc += row_losses[(size_t)which * B + b];
  s[threadIdx.x] = acc;
  __syncthreads();
  for (int k = 128; k > 0; k >>= 1) {
    if (threadIdx.x < k) s[threadIdx.x] += s[threadIdx.x + k];
    __syncthreads();
  }
  if (threadIdx.x == 0) losses[which] = s[0] / (double)B;
}

}  // namespace

extern "C" int mz_unroll_loss(const mz_loss_cfg* c, const float* value_logits, const float* reward_logits,
                              const float* policy_logits, const float* t_values, const float* t_rewards,
                              const float* t_policies, const double* is_weights, float* d_value_logits,
                              float* d_reward_logits, float* d_policy_logits, double* row_losses, double* losses,
                              float* new_errors, void* stream) {
  if (!c || c->batch <= 0 || c->num_unroll_steps < 1 || c->num_unroll_steps > 31 || c->num_actions < 1 ||
      c->value_max < c->value_min || c->reward_max < c->reward_min)
    return -1;
  if (!value_logits || !reward_logits || !policy_logits || !t_values || !t_rewards || !t_policies || !row_losses ||
      !losses)
    return -2;
  cudaStream_t st = (cudaStream_t)stream;
  unroll_loss_kernel<<<c->batch, 32 * (c->num_unroll_steps + 1), 0, st>>>(
      *c, value_logits, reward_logits, policy_logits, t_values, t_rewards, t_policies, is_weights, d_value_logits,
      d_reward_logits, d_policy_logits, row_losses, new_errors);
  MZ_LAUNCH_CHECK();
  loss_mean_kernel<<<3, 256, 0, st>>>(c->batch, row_losses, losses);
  MZ_LAUNCH_CHECK();
  return 0;
}

extern "C" int mz_scalar_unroll_loss(const mz_loss_cfg* c, int32_t scalar_loss, const float* value_out,
                                     const float* reward_out, const float* policy_logits, const float* t_values,
                                     const float* t_rewards, const float* t_policies, const double* is_weights,
                                     float* d_value_out, float* d_reward_out, float* d_policy_logits,
                                     double* row_losses, double* losses, float* new_errors, void* stream) {
  if (!c || c->batch <= 0 || c->num_unroll_steps < 1 || c->num_unroll_steps > 31 || c->num_actions < 1 ||
      (scalar_loss != 0 && scalar_loss != 1))
    return -1;
  if (!value_out || !reward_out || !policy_logits || !t_values || !t_rewards || !t_policies || !row_losses || !losses)
    return -2;
  cudaStream_t st = (cudaStream_t)stream;
  scalar_unroll_loss_kernel<<<c->batch, 32 * (c->num_unroll_steps + 1), 0, st>>>(
      *c, scalar_loss, value_out, reward_out, policy_logits, t_values, t_rewards, t_policies, is_weights, d_value_out,
      d_reward_out, d_policy_logits, row_losses, new_errors);
  MZ_LAUNCH_CHECK();
  loss_mean_kernel<<<3, 256, 0, st>>>(c->batch, row_losses, losses);
  MZ_LAUNCH_CHECK();
  return 0;
}
