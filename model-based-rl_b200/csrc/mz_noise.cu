// Root exploration noise drawn on the device: np.random.dirichlet([alpha] * len(actions)) of
// Node.add_exploration_noise (mcts.py:57-61) for every game of a move, written in the layout mz_tree_set_root /
// mz_fc_search read (row g: one value per LEGAL action of game g, in action order, dense from column 0).
//
// Same distribution as the reference's draw, another random stream (Philox4x32-10 keyed by seed, game, action and
// the move counter): a Gamma(alpha, 1) variate per legal action -- Marsaglia-Tsang for shape alpha + 1, times
// U ** (1 / alpha) when alpha < 1 -- normalised over the row in binary64.  The host-supplied buffer stays the
// bit-exact path (tests replay the reference's draws through it); this kernel removes 8 * G * A bytes of PCIe
// traffic and the host's G * A gamma draws from every self-play move (2.8 ms at 4096 games x 18 actions).
#include <curand_kernel.h>
#include <math.h>

#include "mz_common.cuh"

namespace {

MZ_DEV double gamma_variate(curandStatePhilox4_32_10_t* st, double alpha) {
  const double a = alpha < 1.0 ? alpha + 1.0 : alpha;
  const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
  double out;
  for (;;) {
    double x, v;
    do {
      x = curand_normal_double(st);
      v = 1.0 + c * x;
    } while (v <= 0.0);
    v = v * v * v;
    const double u = curand_uniform_double(st);  // (0, 1]
    if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) {
      out = d * v;
      break;
    }
  }
  if (alpha < 1.0) out *= pow(curand_uniform_double(st), 1.0 / alpha);
  return out;
}

// a warp per game, lane l draws for the legal actions of ranks l and l + 32.  The Philox subsequence is
// g * 32 + rank for A <= 32 and g * 64 + rank above.
__global__ void dirichlet_noise_kernel(int G, int A, double alpha, const int32_t* __restrict__ legal,
                                       unsigned long long seed, unsigned long long move, double* __restrict__ noise) {
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (g >= G) return;
  const int W = (A + 31) >> 5;
  int n = 0;
  for (int w = 0; w < W; ++w) {
    uint32_t mask = legal ? (uint32_t)legal[(size_t)g * W + w] : 0xffffffffu;
    if (A < 32 * (w + 1)) mask &= (1u << (A - 32 * w)) - 1u;
    n += __popc(mask);
  }
  double x[2] = {0.0, 0.0};
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int rank = lane + 32 * h;
    if (h < W && rank < n) {
      curandStatePhilox4_32_10_t st;
      curand_init(seed, (unsigned long long)g * 32 * W + rank, move * 64, &st);
      x[h] = gamma_variate(&st, alpha);
    }
  }
  double sum = W > 1 ? x[0] + x[1] : x[0];
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) sum += shfl_xor_f64<32>(sum, m);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int rank = lane + 32 * h;
    if (h < W && rank < A) noise[(size_t)g * A + rank] = rank < n ? (sum > 0.0 ? x[h] / sum : 1.0 / n) : 0.0;
  }
}

}  // namespace

extern "C" {

int mz_dirichlet_noise(int32_t num_games, int32_t num_actions, double alpha, const int32_t* legal_mask,
                       uint64_t seed, uint64_t move, double* noise, void* stream) {
  if (num_games < 1 || num_actions < 1 || num_actions > MZ_MAX_ACTIONS || !(alpha > 0.0) || !noise)
    return MZ_ERR_BAD_ARG;
  dirichlet_noise_kernel<<<(num_games + 3) / 4, 128, 0, (cudaStream_t)stream>>>(num_games, num_actions, alpha, legal_mask,
                                                                                seed, move, noise);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

}  // extern "C"
