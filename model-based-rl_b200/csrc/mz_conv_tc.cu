// MuZeroNetwork (residual conv tower on 6x6x128 hidden states) on the 5th-generation tensor cores.
//
// One persistent implicit-GEMM kernel serves every dense layer of recurrent_inference
// (networks.py:393-554: MuZeroDynamics conv + 16 ResidualBlocks + reward head, MuZeroPrediction 16
// ResidualBlocks + value / policy heads):
//
//   conv3x3 (pad 1, stride 1) with BatchNorm folded:  D[row, n] = sum_{tap, c} X[row + off(tap), c] *
//       W[n, tap * 128 + c],   off(tap) = (ky - 1) * 8 + (kx - 1)
//   on activations stored channels-last in bf16 with shared zero padding: a game is 49 rows of 128
//   channels -- one zero row of 7, then 6 image rows of 6 pixels + 1 zero -- so every 3x3 neighbour
//   of a pixel that falls outside the image lands on a zero row (of this game or the next one), a tap
//   is a pure row shift of the flat [games * 49][128] matrix, and the A operand of every tap is a
//   TMA tile load at a shifted row coordinate -- no im2col buffer exists anywhere.  36 of 49 rows
//   are real pixels.  Tiles are 128 consecutive rows (they do not align with games).
//   Linear(6*6*128 -> 512) heads: the same kernel with one "tap", K = 49 * 128 (the padding rows
//   are zero, the weights are permuted to the padded channels-last order at pack time).
//
// Tile: 128 rows (two games, or 128 games for the heads) x 128 outputs, K blocks of 64 bf16 (one
// 128-byte swizzle row).  Warp roles: warp 0 = TMA producer, warp 1 = MMA issuer (tcgen05.mma,
// accumulators in TMEM, double buffered so the epilogue of tile i overlaps the MMAs of tile i+1),
// warps 2..5 = epilogue (tcgen05.ld, bias / action plane / residual / ReLU / per-pixel min-max
// scaling, bf16 stores).  CTAs are persistent over tiles.
#include <cuda.h>
#include <cuda_bf16.h>
#include <math.h>

#include "mz_common.cuh"

namespace {

constexpr int BM = 128, BN = 128, BK = 64;
constexpr int GROWS = 49;                        // rows per game: 7 zero | 6 x (6 pixels + 1 zero)
// M tiles per work item (they share every weight-tile load).  Measured at 4096 games: TU = 2 with 4
// stages 60.5 us per convolution vs TU = 1 with 6 stages 63.7 us, but 24.1 vs 21.9 us at 1024 games
// (coarser work items) and no gain once the residual epilogue is on: kept at 1.
constexpr int TU = 1;
constexpr int STAGES = TU == 1 ? 6 : 4;
constexpr int STAGE_BYTES = (TU * BM + BN) * BK * 2;  // 32 KB (48 KB with TU = 2)
constexpr int CONV_THREADS = 192;                // producer, MMA, 4 epilogue warps
constexpr int ACC_COLS = 2 * TU * BN;            // double-buffered accumulators of TU x 128 fp32 columns

enum : int {
  EPI_RELU = 1,        // max(x, 0)
  EPI_RESIDUAL = 2,    // += residual[row] before the ReLU
  EPI_ACTION = 4,      // += action[g] / A * plane_term[pixel][n]   (MuZeroNetwork.attach_action)
  EPI_SCALE = 8,       // also emit (x - min_c) / (max_c - min_c) per pixel (scale_state)
  EPI_F32_OUT = 16,    // heads: fp32 row-major output [M][ldo], no border masking
  EPI_TO_PADDED = 32,  // plain GEMM whose row r = (game, y, x): bf16 rows scattered into the padded layout
};

struct ConvParams {
  int mode_fc;               // 0: conv taps, 1: plain GEMM (heads)
  int num_tiles_m, num_tiles_n, num_kblocks;
  int rows_total;            // conv: games * 64; fc: games
  int flags;
  int num_actions;
  int wp, grows;             // conv: padded row width (W + 1) and rows per game (wp * wp)
  int ncols;                 // output channels per tile = channels per activation row: 64 or 128
  int kb_per_tap;            // conv: K blocks of 64 input channels per tap (1 or 2)
  int out_w;                 // EPI_TO_PADDED: GEMM row r = (game, y, x) of an out_w x out_w image
  const float* bias;         // [N_total]
  const float* plane_term;   // [36][128] (EPI_ACTION)
  const int32_t* actions;    // [games]   (EPI_ACTION)
  const __nv_bfloat16* residual;  // [rows][128] (EPI_RESIDUAL)
  __nv_bfloat16* out;        // conv: [rows][128] bf16
  __nv_bfloat16* out_scaled; // EPI_SCALE: [rows][128] scaled state (flat, input of the prediction tower)
  __nv_bfloat16* pool_out;   // EPI_SCALE, optional: the same rows scattered into the hidden pool,
  const int32_t* pool_row_base;  //   game g's 49 rows starting at row pool_row_base[g]
  float* out_f32;            // EPI_F32_OUT: [M][ldo]
  int ldo;
};

MZ_DEV bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}" : "=r"(pred));
  return pred != 0;
}
MZ_DEV void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
MZ_DEV void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
MZ_DEV void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
MZ_DEV void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
MZ_DEV void tmem_dealloc(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
MZ_DEV void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
MZ_DEV void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
MZ_DEV void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
MZ_DEV void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
MZ_DEV void tmem_ld32(uint32_t addr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]),
        "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]),
        "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]),
        "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(addr)
      : "memory");
}
template <bool ACC>
MZ_DEV void umma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  if (ACC)
    asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, 1, 1;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc) : "memory");
  else
    asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, 1, 0;\ntcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc) : "memory");
}
// K-major operand tile written by TMA with SWIZZLE_128B: rows of 128 bytes, 8-row atoms of 1024 B
MZ_DEV uint64_t make_desc_sw128(uint32_t smem_addr) {
  uint64_t d = (uint64_t)((smem_addr >> 4) & 0x3FFFu);
  d |= (uint64_t)1 << 16;                        // leading byte offset: unused for swizzled K-major
  d |= (uint64_t)(1024 >> 4) << 32;              // stride byte offset: one 8-row atom
  d |= (uint64_t)1 << 46;                        // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                        // SWIZZLE_128B
  return d;
}
// D = f32, A = B = bf16, both K-major, M = 128, N = n
MZ_DEV uint32_t make_idesc_128xN(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}
MZ_DEV uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 p = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&p);
}

__global__ void __launch_bounds__(CONV_THREADS, 1)
conv_gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    ConvParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* acc_full = empty + STAGES;   // [2]
  uint64_t* acc_empty = acc_full + 2;    // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* s_bias = reinterpret_cast<float*>(tmem_ptr + 4);  // [num_tiles_n * 128] (<= 1024 floats)
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_tiles = ((p.num_tiles_m + TU - 1) / TU) * p.num_tiles_n;  // work items
  const int NC = p.ncols;
  for (int i = threadIdx.x; i < p.num_tiles_n * NC; i += CONV_THREADS) s_bias[i] = p.bias[i];

  if (threadIdx.x == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 4);  // one (relaxed) arrival per epilogue warp
    }
    mbar_fence_init();
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr, ACC_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;
  // launched as a programmatic dependent: the set-up above overlapped the previous layer's tail;
  // activations, residuals and row offsets written by earlier kernels are only touched below
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    // ===== TMA producer =====
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int gm = tile / p.num_tiles_n, tn = tile % p.num_tiles_n;
      const int rb0 = gm * TU * BM;
      for (int kb = 0; kb < p.num_kblocks; ++kb, ++it) {
        const int st = it % STAGES;
        mbar_wait(&empty[st], ((it / STAGES) & 1) ^ 1);
        if (elect_one()) {
          uint8_t* sa = smem + st * STAGE_BYTES;
          uint8_t* sb = sa + TU * BM * BK * 2;
          int shift = 0, ka = kb * BK;
          if (!p.mode_fc) {  // k block = (tap, block of 64 input channels)
            const int tap = kb / p.kb_per_tap;
            shift = (tap / 3 - 1) * p.wp + (tap % 3 - 1);
            ka = (kb - tap * p.kb_per_tap) * BK;
          }
          mbar_arrive_expect_tx(&full[st], (uint32_t)((TU * BM + NC) * BK * 2));
#pragma unroll
          for (int h = 0; h < 2 * TU; ++h)  // rows beyond the tensor (odd tail, halo) arrive as zeros
            tma_load_2d(sa + h * 64 * BK * 2, &map_a, ka, rb0 + h * 64 + shift, &full[st]);
          tma_load_2d(sb, &map_b, kb * BK, tn * NC, &full[st]);
          if (NC > 64) tma_load_2d(sb + 64 * BK * 2, &map_b, kb * BK, tn * NC + 64, &full[st]);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer =====
    const uint32_t idesc = make_idesc_128xN(p.ncols);
    int it = 0, t = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++t) {
      const int acc = t & 1;
      mbar_wait(&acc_empty[acc], ((t >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d0 = tmem + acc * TU * BN;
      for (int kb = 0; kb < p.num_kblocks; ++kb, ++it) {
        const int st = it % STAGES;
        mbar_wait(&full[st], (it / STAGES) & 1);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + st * STAGE_BYTES);
        const uint64_t bd = make_desc_sw128(sa + TU * BM * BK * 2);
        if (elect_one()) {
#pragma unroll
          for (int u = 0; u < TU; ++u) {  // both M tiles against the same weight tile
            const uint32_t d = d0 + u * BN;
            const uint64_t ad = make_desc_sw128(sa + u * BM * BK * 2);
            if (kb == 0) umma_ss<false>(d, ad, bd, idesc);
            else umma_ss<true>(d, ad, bd, idesc);
#pragma unroll
            for (int ks = 1; ks < BK / 16; ++ks)  // +32 bytes along K inside the 128-byte swizzle row
              umma_ss<true>(d, ad + (uint64_t)(ks * 2), bd + (uint64_t)(ks * 2), idesc);
          }
          tc_commit(&empty[st]);
          if (kb == p.num_kblocks - 1) tc_commit(&acc_full[acc]);
        }
        __syncwarp();
      }
    }
  } else {
    // ===== epilogue: thread = accumulator row =====
    const int quarter = warp & 3;
    const int r_in_tile = quarter * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(quarter * 32) << 16);
    int t = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++t) {
      const int acc = t & 1;
      const int gm = tile / p.num_tiles_n, tn = tile % p.num_tiles_n;
#pragma unroll 1
      for (int u = 0; u < TU; ++u) {
      const int tm = gm * TU + u;
      // residual rows are requested before waiting for the accumulator: they arrive while the MMAs
      // of this work item are still running (second tile: while the first is being written out)
      uint4 resv[BN / 8];
      if (!(p.flags & EPI_F32_OUT) && (p.flags & EPI_RESIDUAL)) {
        const int Rp = tm * BM + r_in_tile;
        const int gp = Rp / p.grows, posp = Rp - gp * p.grows;
        const bool intp = posp >= p.wp && ((posp - p.wp) % p.wp) < p.wp - 1 && Rp < p.rows_total;
        const uint4* rp = reinterpret_cast<const uint4*>(p.residual + (size_t)Rp * NC);
#pragma unroll
        for (int q = 0; q < BN / 8; ++q) resv[q] = (intp && q * 8 < NC) ? rp[q] : make_uint4(0u, 0u, 0u, 0u);
      }
      if (u == 0) {
        mbar_wait(&acc_full[acc], (t >> 1) & 1);
        tc_fence_after();
      }
      const uint32_t d = lane_addr + (acc * TU + u) * BN;
      if (p.flags & (EPI_F32_OUT | EPI_TO_PADDED)) {
        const int row = tm * BM + r_in_tile;
        const bool ok = row < p.rows_total;
        float* orow = p.out_f32 + (size_t)row * p.ldo + tn * NC;
        __nv_bfloat16* prow = nullptr;
        if ((p.flags & EPI_TO_PADDED) && ok) {  // GEMM row = (game, y, x) -> row of the padded layout
          const int ww = p.out_w * p.out_w, wpo = p.out_w + 1;
          const int gg = row / ww, rem = row - gg * ww, yy = rem / p.out_w, xx = rem - yy * p.out_w;
          prow = p.out + ((size_t)gg * wpo * wpo + wpo + yy * wpo + xx) * NC;
        }
#pragma unroll 1
        for (int c0 = 0; c0 < NC; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(d + c0, v);
          tmem_wait_ld();
          if (ok) {
            float x[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              x[j] = __uint_as_float(v[j]) + s_bias[tn * NC + c0 + j];
              if (p.flags & EPI_RELU) x[j] = fmaxf(x[j], 0.0f);
            }
            if (prow) {
#pragma unroll
              for (int q = 0; q < 4; ++q)
                reinterpret_cast<uint4*>(prow + c0)[q] =
                    make_uint4(pack_bf16(x[q * 8], x[q * 8 + 1]), pack_bf16(x[q * 8 + 2], x[q * 8 + 3]),
                               pack_bf16(x[q * 8 + 4], x[q * 8 + 5]), pack_bf16(x[q * 8 + 6], x[q * 8 + 7]));
            } else {
#pragma unroll
              for (int j = 0; j < 32; j += 4)
                *reinterpret_cast<float4*>(orow + c0 + j) = make_float4(x[j], x[j + 1], x[j + 2], x[j + 3]);
            }
          }
        }
      } else {
        const int R = tm * BM + r_in_tile;  // flat row
        const int g = R / p.grows, pos = R - g * p.grows;
        const int py = (pos - p.wp) / p.wp, px = (pos - p.wp) - py * p.wp;
        const bool interior = pos >= p.wp && px < p.wp - 1;
        const size_t row = (size_t)R;
        const bool in_range = R < p.rows_total;
        float act_scale = 0.0f;
        const float* plane = nullptr;
        if ((p.flags & EPI_ACTION) && interior && in_range) {
          act_scale = (float)p.actions[g] / (float)p.num_actions;
          plane = p.plane_term + (py * (p.wp - 1) + px) * NC;
        }
        uint4* orow = reinterpret_cast<uint4*>(p.out + row * NC);
        const bool add_res = (p.flags & EPI_RESIDUAL) && interior && in_range;
        // x[0..32) = layer output for channels c0..c0+31 of this row (zero on the border)
        auto chunk = [&](int c0, float (&x)[32]) {
          uint32_t v[32];
          tmem_ld32(d + c0, v);
          tmem_wait_ld();
#pragma unroll
          for (int j = 0; j < 32; ++j) x[j] = __uint_as_float(v[j]) + s_bias[c0 + j];
          if (plane) {
#pragma unroll
            for (int j = 0; j < 32; ++j) x[j] = fmaf(act_scale, __ldg(plane + c0 + j), x[j]);
          }
          if (add_res) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const uint4 rv = resv[(c0 >> 3) + q];
              const uint32_t w[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
              for (int h = 0; h < 4; ++h) {
                const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162*>(&w[h]);
                x[q * 8 + 2 * h] += __low2float(b2);
                x[q * 8 + 2 * h + 1] += __high2float(b2);
              }
            }
          }
          if (p.flags & EPI_RELU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) x[j] = fmaxf(x[j], 0.0f);
          }
          if (!interior) {
#pragma unroll
            for (int j = 0; j < 32; ++j) x[j] = 0.0f;  // keep the zero border of the padded layout
          }
        };
        float mn = INFINITY, mx = -INFINITY;
#pragma unroll
        for (int c0 = 0; c0 < BN; c0 += 32) {
          if (c0 >= NC) break;
          float x[32];
          chunk(c0, x);
          if (p.flags & EPI_SCALE) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              mn = fminf(mn, x[j]);
              mx = fmaxf(mx, x[j]);
            }
          }
          if (in_range && p.out) {
#pragma unroll
            for (int q = 0; q < 4; ++q)
              orow[(c0 >> 3) + q] = make_uint4(pack_bf16(x[q * 8], x[q * 8 + 1]), pack_bf16(x[q * 8 + 2], x[q * 8 + 3]),
                                               pack_bf16(x[q * 8 + 4], x[q * 8 + 5]), pack_bf16(x[q * 8 + 6], x[q * 8 + 7]));
          }
        }
        if (p.flags & EPI_SCALE) {
          // MuZeroNetwork.scale_state networks.py:543-547: second pass over the accumulator row.
          // tcgen05.ld is warp-collective: every lane walks the pass, only the stores are predicated
          // (tiles do not align with games, so `in_range` is not warp-uniform)
          uint4* so = reinterpret_cast<uint4*>(p.out_scaled + row * NC);
          uint4* po = (p.pool_out && in_range)
                          ? reinterpret_cast<uint4*>(p.pool_out + ((size_t)p.pool_row_base[g] + pos) * NC)
                          : nullptr;
          const float den = mx - mn;
#pragma unroll
          for (int c0 = 0; c0 < BN; c0 += 32) {
            if (c0 >= NC) break;
            float x[32];
            chunk(c0, x);
#pragma unroll
            for (int j = 0; j < 32; ++j) x[j] = interior ? (x[j] - mn) / den : 0.0f;
            if (in_range) {
#pragma unroll
              for (int q = 0; q < 4; ++q) {
                const uint4 o = make_uint4(pack_bf16(x[q * 8], x[q * 8 + 1]), pack_bf16(x[q * 8 + 2], x[q * 8 + 3]),
                                           pack_bf16(x[q * 8 + 4], x[q * 8 + 5]), pack_bf16(x[q * 8 + 6], x[q * 8 + 7]));
                so[(c0 >> 3) + q] = o;
                if (po) po[(c0 >> 3) + q] = o;
              }
            }
          }
        }
      }
      }  // u
      // relaxed: the hand-back orders TMEM reads (tcgen05.wait::ld + fence), not this warp's global stores
      tc_fence_before();
      __syncwarp();
      if (lane == 0)
        asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&acc_empty[acc])) : "memory");
    }
  }

  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, ACC_COLS);
  }
}


// ================================================================================================
// CTA-pair variant for the 128-channel 3x3 convolutions (63 of the 65 convolutions of one
// recurrent_inference): clusters of two CTAs issue tcgen05.mma.cta_group::2 with M = 256 (128 rows per
// CTA), N = 128, and keep the WHOLE weight matrix resident in shared memory -- each CTA holds the 64
// output channels the pair's B operand assigns to it (18 K blocks x 8 KB = 144 KB), loaded once per
// launch and before griddepcontrol.wait (weights do not depend on the previous layer).  Per K block a
// CTA then only streams its 16 KB activation tile: 16 KB written by TMA + 24 KB read by the tensor core
// (A 16 KB + its half of B 8 KB) = 40 KB against 64 KB for the single-CTA kernel, whose 128 x 128 tile
// with both operands streamed is shared-memory-bandwidth bound (DESIGN.md section 4).
//
// Protocol (CUTLASS' 2-SM scheme): every TMA load of either CTA completes its bytes on the LEADER's
// (cluster rank 0) barrier (.cta_group::2, peer bit of the barrier address cleared); only the leader's
// MMA warp issues MMAs; tcgen05.commit multicasts its arrival to the same barrier offset in both CTAs
// (stage release, accumulator ready); epilogue threads of both CTAs arrive on the leader's
// accumulator-empty barrier (remote arrive for the peer).
// ================================================================================================
constexpr int P_STAGES = 4;
constexpr int P_A_BYTES = BM * BK * 2;                  // 16 KB activation tile per K block
constexpr int P_KBLOCKS = 18;                           // 9 taps x 2 blocks of 64 input channels
constexpr int P_BH_BYTES = 64 * BK * 2;                 // 8 KB: this CTA's 64 output channels of one K block
// Window mode (padded row width <= 7, i.e. the 6 x 6 hidden state): the nine taps of a tile read row
// windows shifted by at most 8 rows, so ONE load of rows [tile - 8, tile + 136) per block of 64 input
// channels serves all of them -- the tap is a row offset in the A descriptor's start address (the
// 128-byte swizzle is a function of the shared-memory address bits, so TMA's placement and the tensor
// core's reads agree at any row offset; setting the descriptor's matrix-base-offset field for the
// shifted start gives wrong results -- measured).  2 x 18 KB written per tile instead of 18 x 16 KB.
constexpr int P_WIN_PAD = 8;                            // rows before / after the tile
constexpr int P_WIN_ROWS = BM + 2 * P_WIN_PAD;          // 144
constexpr int P_WIN_HALF = P_WIN_ROWS * BK * 2;         // 18 KB: one block of 64 channels
constexpr int P_WIN_BYTES = 2 * P_WIN_HALF;             // 36 KB per tile
constexpr int P_WIN_STAGES = 2;
constexpr int P_A_REGION = P_WIN_STAGES * P_WIN_BYTES > P_STAGES * P_A_BYTES ? P_WIN_STAGES * P_WIN_BYTES
                                                                             : P_STAGES * P_A_BYTES;
constexpr int P_ACC = 2;                                // accumulator buffers in TMEM (4 measured: no gain, the tile period is the MMA time at the power-capped clock)
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;          // shared::cluster address -> same offset in the even CTA

MZ_DEV uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
MZ_DEV void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
MZ_DEV void tma_load_2d_pair(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* leader_bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(map), "r"(smem_u32(leader_bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
MZ_DEV void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
               "r"(ncols)
               : "memory");
}
MZ_DEV void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
MZ_DEV void tmem_dealloc_pair(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
MZ_DEV void tc_commit_pair(uint64_t* bar) {  // arrives on `bar`'s offset in both CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3)
               : "memory");
}
template <bool ACC>
MZ_DEV void umma_ss_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  if (ACC)
    asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, 1, 1;\ntcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc) : "memory");
  else
    asm volatile("{\n.reg .pred p;\nsetp.eq.u32 p, 1, 0;\ntcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}"
                 ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc) : "memory");
}
// Accumulator hand-back to the leader's MMA warp.  Relaxed on purpose: what the arrival has to order is
// the epilogue's TMEM reads (complete after tcgen05.wait::ld, ordered by tcgen05.fence::before_thread_sync),
// not its global stores -- a releasing arrive compiles to MEMBAR + ERRBAR (.cta) or MEMBAR.ALL.GPU +
// CCTL.IVALL (.cluster) and made every epilogue warp wait for its output rows to drain (ncu: 18 % of the
// kernel's stall samples).
MZ_DEV void mbar_arrive_leader(uint64_t* bar, uint32_t rank) {
  uint32_t addr = smem_u32(bar);
  if (rank != 0) asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(addr) : "r"(smem_u32(bar)), "r"(0));
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(addr) : "memory");
}
// D = f32, A = B = bf16, both K-major, M = 256 over the CTA pair, N = 128
constexpr uint32_t kIdescPair = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);

__global__ void __launch_bounds__(CONV_THREADS, 1)
conv_pair_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const __grid_constant__ CUtensorMap map_w, ConvParams p, int window) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_b = smem;                                        // [18][64 rows][64 k] bf16, 128-byte swizzle
  uint8_t* s_a = smem + P_KBLOCKS * P_BH_BYTES;               // [P_STAGES][128 rows][64 k]
  uint64_t* full = reinterpret_cast<uint64_t*>(s_a + P_A_REGION);
  uint64_t* empty = full + P_STAGES;
  uint64_t* acc_full = empty + P_STAGES;   // [P_ACC]
  uint64_t* acc_empty = acc_full + P_ACC;  // [P_ACC] (used in the leader only)
  uint64_t* b_full = acc_empty + P_ACC;    // [1] (used in the leader only)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(b_full + 1);
  float* s_bias = reinterpret_cast<float*>(tmem_ptr + 4);  // [128]
  uint8_t* s_stage = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(s_bias + BN) + 15) & ~(uintptr_t)15);  // [4 epilogue warps][32 rows][64 B]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_rank();
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;
  const int num_pairs = (p.num_tiles_m + 1) >> 1;
  constexpr int NC = BN;
  for (int i = threadIdx.x; i < NC; i += CONV_THREADS) s_bias[i] = p.bias[i];

  if (threadIdx.x == 0) {
    for (int i = 0; i < P_STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < P_ACC; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 8);  // one arrival per epilogue warp of both CTAs
    }
    mbar_init(b_full, 1);
    mbar_fence_init();
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    tma_prefetch_desc(&map_w);
  }
  __syncthreads();
  cluster_sync();  // both CTAs' barriers exist before anything is signalled across the pair
  if (warp == 0) {
    tmem_alloc_pair(tmem_ptr, P_ACC * BN);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;

  if (warp == 0) {
    // ===== TMA producer =====
    if (elect_one()) {
      // resident weights: rows [rank * 64, +64) of W[128][1152], one 8 KB box per K block
      if (rank == 0) mbar_arrive_expect_tx(b_full, 2u * P_KBLOCKS * P_BH_BYTES);
      for (int kb = 0; kb < P_KBLOCKS; ++kb)
        tma_load_2d_pair(s_b + kb * P_BH_BYTES, &map_b, kb * BK, (int)rank * 64, b_full);
    }
    __syncwarp();
    pdl_wait();  // activations of the previous layer are only touched below
    pdl_trigger();
    int it = 0;
    for (int pt = cluster_id; pt < num_pairs; pt += num_clusters) {
      const int rb0 = (2 * pt + (int)rank) * BM;
      if (window) {  // one stage = the tile's row window for both blocks of 64 channels
        const int st = it % P_WIN_STAGES;
        mbar_wait(&empty[st], ((it / P_WIN_STAGES) & 1) ^ 1);
        if (elect_one()) {
          uint8_t* sa = s_a + st * P_WIN_BYTES;
          if (rank == 0) mbar_arrive_expect_tx(&full[st], 2u * P_WIN_BYTES);
          tma_load_2d_pair(sa, &map_w, 0, rb0 - P_WIN_PAD, &full[st]);
          tma_load_2d_pair(sa + P_WIN_HALF, &map_w, BK, rb0 - P_WIN_PAD, &full[st]);
        }
        __syncwarp();
        ++it;
        continue;
      }
      for (int kb = 0; kb < P_KBLOCKS; ++kb, ++it) {
        const int st = it % P_STAGES;
        mbar_wait(&empty[st], ((it / P_STAGES) & 1) ^ 1);
        if (elect_one()) {
          uint8_t* sa = s_a + st * P_A_BYTES;
          const int tap = kb >> 1;
          const int shift = (tap / 3 - 1) * p.wp + (tap % 3 - 1);
          const int ka = (kb & 1) * BK;
          if (rank == 0) mbar_arrive_expect_tx(&full[st], 2u * P_A_BYTES);
          tma_load_2d_pair(sa, &map_a, ka, rb0 + shift, &full[st]);
          tma_load_2d_pair(sa + 64 * BK * 2, &map_a, ka, rb0 + 64 + shift, &full[st]);
        }
        __syncwarp();
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (leader CTA only) =====
    pdl_wait();
    pdl_trigger();
    if (rank == 0) {
      mbar_wait(b_full, 0);
      tc_fence_after();
      int it = 0, t = 0;
      for (int pt = cluster_id; pt < num_pairs; pt += num_clusters, ++t) {
        const int acc = t % P_ACC;
        mbar_wait(&acc_empty[acc], ((t / P_ACC) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d = tmem + acc * BN;
        if (window) {
          const int st = it % P_WIN_STAGES;
          mbar_wait(&full[st], (it / P_WIN_STAGES) & 1);
          tc_fence_after();
          const uint32_t win = smem_u32(s_a + st * P_WIN_BYTES);
          if (elect_one()) {
#pragma unroll 1
            for (int kb = 0; kb < P_KBLOCKS; ++kb) {  // same K order as the per-tap pipeline
              const int tap = kb >> 1;
              const int shift = (tap / 3 - 1) * p.wp + (tap % 3 - 1);
              const uint32_t a_addr = win + (kb & 1) * P_WIN_HALF + (uint32_t)((P_WIN_PAD + shift) * (BK * 2));
              const uint64_t ad = make_desc_sw128(a_addr);  // no matrix base offset: measured, bit-identical
              const uint64_t bd = make_desc_sw128(smem_u32(s_b + kb * P_BH_BYTES));
              if (kb == 0) umma_ss_pair<false>(d, ad, bd, kIdescPair);
              else umma_ss_pair<true>(d, ad, bd, kIdescPair);
#pragma unroll
              for (int ks = 1; ks < BK / 16; ++ks)
                umma_ss_pair<true>(d, ad + (uint64_t)(ks * 2), bd + (uint64_t)(ks * 2), kIdescPair);
            }
            tc_commit_pair(&empty[st]);
            tc_commit_pair(&acc_full[acc]);
          }
          __syncwarp();
          ++it;
          continue;
        }
        for (int kb = 0; kb < P_KBLOCKS; ++kb, ++it) {
          const int st = it % P_STAGES;
          mbar_wait(&full[st], (it / P_STAGES) & 1);
          tc_fence_after();
          const uint64_t ad = make_desc_sw128(smem_u32(s_a + st * P_A_BYTES));
          const uint64_t bd = make_desc_sw128(smem_u32(s_b + kb * P_BH_BYTES));
          if (elect_one()) {
            if (kb == 0) umma_ss_pair<false>(d, ad, bd, kIdescPair);
            else umma_ss_pair<true>(d, ad, bd, kIdescPair);
#pragma unroll
            for (int ks = 1; ks < BK / 16; ++ks)
              umma_ss_pair<true>(d, ad + (uint64_t)(ks * 2), bd + (uint64_t)(ks * 2), kIdescPair);
            tc_commit_pair(&empty[st]);
            if (kb == P_KBLOCKS - 1) tc_commit_pair(&acc_full[acc]);
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ===== epilogue: thread = accumulator row of this CTA's half of the pair tile =====
    pdl_wait();
    pdl_trigger();
    const int quarter = warp & 3;
    const int r_in_tile = quarter * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(quarter * 32) << 16);
    // Row-per-thread global accesses cost 32 L1 wavefronts per warp instruction (32 rows x 16 bytes) and made
    // the epilogue, not the MMA issuer, set the tile period of the residual variant (4 k L1 cycles per tile for
    // loads + stores against 4.6 k cycles of MMA).  Rows therefore cross a 2 KB per-warp staging area in shared
    // memory: global side = 8 rows x 64 contiguous bytes per instruction (lane -> row 8 i + lane / 4, 16-byte
    // piece lane % 4), thread side = its own row; pieces are XOR-swizzled so both sides are conflict free.
    const uint32_t stage = smem_u32(s_stage) + (uint32_t)quarter * 2048u;
    const int c_row = lane >> 2, c_piece = lane & 3;  // coalesced side: row within a group of 8, piece
    auto swz = [](int r, int k) { return (uint32_t)(r * 64 + ((k ^ ((r >> 1) & 3)) << 4)); };
    auto sts = [](uint32_t a, uint4 v) {
      asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    };
    auto lds = [](uint32_t a) {
      uint4 v;
      asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
      return v;
    };
    int t = 0;
    for (int pt = cluster_id; pt < num_pairs; pt += num_clusters, ++t) {
      const int acc = t % P_ACC;
      const int tm = 2 * pt + (int)rank;
      const int R = tm * BM + r_in_tile;  // flat row of this thread
      const int g = R / p.grows, pos = R - g * p.grows;
      const int py = (pos - p.wp) / p.wp, px = (pos - p.wp) - py * p.wp;
      const bool interior = pos >= p.wp && px < p.wp - 1;
      const bool in_range = R < p.rows_total;
      const bool add_res = (p.flags & EPI_RESIDUAL) && interior && in_range;
      const int Rw = tm * BM + quarter * 32;  // first row of this warp
      // residual rows of the warp, coalesced: resg[c * 4 + i] = row 8 i + lane / 4, channels 32 c + 8 (lane % 4) ..
      uint4 resg[BN / 8];
      if (p.flags & EPI_RESIDUAL) {  // requested before the accumulator wait
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int Rq = Rw + 8 * i + c_row;
            resg[c * 4 + i] = Rq < p.rows_total
                                  ? *reinterpret_cast<const uint4*>(p.residual + (size_t)Rq * NC + c * 32 + c_piece * 8)
                                  : make_uint4(0u, 0u, 0u, 0u);
          }
        // the residual is the block's input, written two launches ago: usually evicted from L2 by now.
        // Start the next tile's rows towards L2 while this tile is processed.
        const long long Rn = (long long)R + (long long)num_clusters * 2 * BM;
        if (Rn < p.rows_total) {
          const uint8_t* np_ = reinterpret_cast<const uint8_t*>(p.residual + (size_t)Rn * NC);
          asm volatile("prefetch.global.L2 [%0];" ::"l"(np_));
          asm volatile("prefetch.global.L2 [%0];" ::"l"(np_ + 128));
        }
      }
      float act_scale = 0.0f;
      const float* plane = nullptr;
      if ((p.flags & EPI_ACTION) && interior && in_range) {
        act_scale = (float)p.actions[g] / (float)p.num_actions;
        plane = p.plane_term + (py * (p.wp - 1) + px) * NC;
      }
      mbar_wait(&acc_full[acc], (t / P_ACC) & 1);
      tc_fence_after();
      const uint32_t d = lane_addr + acc * BN;
      // x[0..32) = layer output for channels c0..c0+31 of this thread's row (zero on the border)
      auto chunk = [&](int c0, float (&x)[32]) {
        uint4 own[4];
        if (p.flags & EPI_RESIDUAL) {  // the warp's residual rows for these 32 channels -> this thread's row
          const int c = c0 >> 5;
#pragma unroll
          for (int i = 0; i < 4; ++i) sts(stage + swz(8 * i + c_row, c_piece), resg[c * 4 + i]);
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 4; ++k) own[k] = lds(stage + swz(lane, k));
          __syncwarp();
        }
        uint32_t v[32];
        tmem_ld32(d + c0, v);
        tmem_wait_ld();
#pragma unroll
        for (int j = 0; j < 32; ++j) x[j] = __uint_as_float(v[j]) + s_bias[c0 + j];
        if (plane) {
#pragma unroll
          for (int j = 0; j < 32; ++j) x[j] = fmaf(act_scale, __ldg(plane + c0 + j), x[j]);
        }
        if (add_res) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const uint32_t w[4] = {own[q].x, own[q].y, own[q].z, own[q].w};
#pragma unroll
            for (int h = 0; h < 4; ++h) {
              const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162*>(&w[h]);
              x[q * 8 + 2 * h] += __low2float(b2);
              x[q * 8 + 2 * h + 1] += __high2float(b2);
            }
          }
        }
        if (p.flags & EPI_RELU) {
#pragma unroll
          for (int j = 0; j < 32; ++j) x[j] = fmaxf(x[j], 0.0f);
        }
        if (!interior) {
#pragma unroll
          for (int j = 0; j < 32; ++j) x[j] = 0.0f;  // keep the zero border of the padded layout
        }
      };
      // this thread's 32 packed channels -> staging -> 8 rows x 64 contiguous bytes per store instruction
      auto store_rows = [&](__nv_bfloat16* base, int c0, const float (&x)[32], const int32_t* row_base) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          sts(stage + swz(lane, k), make_uint4(pack_bf16(x[k * 8], x[k * 8 + 1]), pack_bf16(x[k * 8 + 2], x[k * 8 + 3]),
                                               pack_bf16(x[k * 8 + 4], x[k * 8 + 5]), pack_bf16(x[k * 8 + 6], x[k * 8 + 7])));
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint4 o = lds(stage + swz(8 * i + c_row, c_piece));
          const int Rq = Rw + 8 * i + c_row;
          if (Rq < p.rows_total) {
            size_t orow_q = (size_t)Rq;
            if (row_base) {  // scatter into the hidden pool: game g's rows start at row_base[g]
              const int gq = Rq / p.grows;
              orow_q = (size_t)row_base[gq] + (size_t)(Rq - gq * p.grows);
            }
            *reinterpret_cast<uint4*>(base + orow_q * NC + c0 + c_piece * 8) = o;
          }
        }
        __syncwarp();
      };
      float mn = INFINITY, mx = -INFINITY;
#pragma unroll
      for (int c0 = 0; c0 < BN; c0 += 32) {
        float x[32];
        chunk(c0, x);
        if (p.flags & EPI_SCALE) {
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            mn = fminf(mn, x[j]);
            mx = fmaxf(mx, x[j]);
          }
        }
        if (p.out) store_rows(p.out, c0, x, nullptr);
      }
      if (p.flags & EPI_SCALE) {  // MuZeroNetwork.scale_state networks.py:543-547 (second pass)
        const float den = mx - mn;
#pragma unroll
        for (int c0 = 0; c0 < BN; c0 += 32) {
          float x[32];
          chunk(c0, x);
#pragma unroll
          for (int j = 0; j < 32; ++j) x[j] = interior ? (x[j] - mn) / den : 0.0f;
          store_rows(p.out_scaled, c0, x, nullptr);
          if (p.pool_out) store_rows(p.pool_out, c0, x, p.pool_row_base);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_leader(&acc_empty[acc], rank);
    }
  }

  // neither CTA may leave while its peer can still signal its barriers or read its shared memory
  tc_fence_before();
  __syncthreads();
  cluster_sync();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc_pair(tmem, P_ACC * BN);
  }
}

// ================================================================================================
// Value / reward support heads wider than 32 bins (the paper's Atari support is 601):
//   out[g] = h^-1( sum_i softmax(logits[g])_i * (support_min + i) ),  logits[g] = hidden[g, 0:512] . W2^T + b2
// (networks.py:438-440, 477-483; config.py:27-33).  One CTA per tile of 128 games, M = 128 rows = games.
//   A: the tile's float32 head hidden rows, rounded to bf16 (round-to-nearest-even) by the epilogue warps
//      while they stage it into shared memory in the 128-byte-swizzle K-major layout: 8 K blocks of 64,
//      128 KB, resident for the whole tile.  This is the only rounding of the hidden layer; fc1's epilogue
//      keeps it float32 in global memory.
//   B: W2 as plain row-major bf16 [bins][512] (rounded once at load_weights), streamed by TMA in chunks of
//      128 outputs x 64 K through a 4-stage mbarrier ring; rows >= bins arrive as zeros (TMA out-of-bounds
//      fill) and their columns get a -inf bias, so they add exp(-inf) = 0 to the softmax.
//   D: float32 in TMEM, two 128-column accumulators: the epilogue of chunk c overlaps the MMAs of c + 1.
// Epilogue = online softmax, one thread per game: running max m, denominator den and numerator num (sum of
// e_i * support_i), rescaled by exp(m_old - m_new) whenever a group of 32 columns raises the max.  The
// reduction order is fixed: columns in increasing order, one group of 32 at a time, each group's max first,
// then its terms added one by one -- no cross-thread reduction, so a given input gives the same bits on
// every run and at every grid size.
// ================================================================================================
constexpr int SH_K = 512;                      // head hidden width
constexpr int SH_KB = SH_K / BK;               // 8 K blocks
constexpr int SH_N = 128;                      // outputs per chunk (one accumulator)
constexpr int SH_STAGES = 4;
constexpr int SH_A_BYTES = BM * SH_K * 2;      // 128 KB
constexpr int SH_A_KB_BYTES = BM * BK * 2;     // 16 KB per K block
constexpr int SH_B_BYTES = SH_N * BK * 2;      // 16 KB per stage
constexpr int SH_MIN_BINS = 33, SH_MAX_BINS = 1024;
constexpr int SH_THREADS = 192;                // TMA producer, MMA issuer, 4 staging / epilogue warps

__global__ void __launch_bounds__(SH_THREADS, 1)
conv_support_head_tc_kernel(const __grid_constant__ CUtensorMap map_w, int G, const float* __restrict__ hidden,
                            int ldh, const float* __restrict__ b2, int bins, int support_min, int no_tt,
                            float* __restrict__ out, int ldo) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* s_a = smem;                                  // [8 K blocks][128 rows][128 B]
  uint8_t* s_b = smem + SH_A_BYTES;                     // [SH_STAGES][128 rows][128 B]
  uint64_t* full = reinterpret_cast<uint64_t*>(s_b + SH_STAGES * SH_B_BYTES);
  uint64_t* empty = full + SH_STAGES;
  uint64_t* acc_full = empty + SH_STAGES;   // [2]
  uint64_t* acc_empty = acc_full + 2;       // [2]
  uint64_t* a_full = acc_empty + 2;         // [1]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(a_full + 1);
  float* s_bias = reinterpret_cast<float*>(tmem_ptr + 4);  // [nchunks * 128], -inf past `bins`
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nchunks = (bins + SH_N - 1) / SH_N;
  // weights only: nothing here depends on the previous kernel
  for (int i = threadIdx.x; i < nchunks * SH_N; i += SH_THREADS) s_bias[i] = i < bins ? b2[i] : -INFINITY;

  if (threadIdx.x == 0) {
    for (int i = 0; i < SH_STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 4);  // one arrival per epilogue warp
    }
    mbar_init(a_full, 4);           // one arrival per staging warp
    mbar_fence_init();
    tma_prefetch_desc(&map_w);
  }
  if (warp == 0) {
    tmem_alloc(tmem_ptr, 2 * SH_N);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_ptr;

  if (warp == 0) {
    // ===== TMA producer: W2 is a weight, its loads may overlap the previous kernel's tail =====
    for (int it = 0; it < nchunks * SH_KB; ++it) {
      const int st = it % SH_STAGES, chunk = it / SH_KB, kb = it - chunk * SH_KB;
      mbar_wait(&empty[st], ((it / SH_STAGES) & 1) ^ 1);
      if (elect_one()) {
        uint8_t* sb = s_b + st * SH_B_BYTES;
        mbar_arrive_expect_tx(&full[st], (uint32_t)SH_B_BYTES);  // out-of-bounds rows count as loaded zeros
        tma_load_2d(sb, &map_w, kb * BK, chunk * SH_N, &full[st]);
        tma_load_2d(sb + 64 * BK * 2, &map_w, kb * BK, chunk * SH_N + 64, &full[st]);
      }
      __syncwarp();
    }
    pdl_wait();
    pdl_trigger();
  } else if (warp == 1) {
    // ===== MMA issuer =====
    pdl_wait();
    pdl_trigger();
    const uint32_t idesc = make_idesc_128xN(SH_N);
    mbar_wait(a_full, 0);
    tc_fence_after();
    int it = 0;
    for (int chunk = 0; chunk < nchunks; ++chunk) {
      const int acc = chunk & 1;
      mbar_wait(&acc_empty[acc], ((chunk >> 1) & 1) ^ 1);
      tc_fence_after();
      const uint32_t d = tmem + acc * SH_N;
      for (int kb = 0; kb < SH_KB; ++kb, ++it) {
        const int st = it % SH_STAGES;
        mbar_wait(&full[st], (it / SH_STAGES) & 1);
        tc_fence_after();
        const uint64_t ad = make_desc_sw128(smem_u32(s_a + kb * SH_A_KB_BYTES));
        const uint64_t bd = make_desc_sw128(smem_u32(s_b + st * SH_B_BYTES));
        if (elect_one()) {
          if (kb == 0) umma_ss<false>(d, ad, bd, idesc);
          else umma_ss<true>(d, ad, bd, idesc);
#pragma unroll
          for (int ks = 1; ks < BK / 16; ++ks)  // +32 bytes along K inside the 128-byte swizzle row
            umma_ss<true>(d, ad + (uint64_t)(ks * 2), bd + (uint64_t)(ks * 2), idesc);
          tc_commit(&empty[st]);
          if (kb == SH_KB - 1) tc_commit(&acc_full[acc]);
        }
        __syncwarp();
      }
    }
  } else {
    // ===== staging of A, then epilogue: thread = accumulator row = game =====
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    const int g0 = blockIdx.x * BM;
    pdl_wait();  // the hidden rows are the previous kernel's output
    pdl_trigger();
    // this warp's 32 rows, one row per step: lane l converts floats [8 q, 8 q + 8) for q = l and l + 32
    // (coalesced 1 KB per row and step) into 16-byte chunk q % 8 of K block q / 8, at its swizzled place
#pragma unroll 4
    for (int i = 0; i < 32; ++i) {
      const int r = quarter * 32 + i, g = g0 + r;
      const float4* src = reinterpret_cast<const float4*>(hidden + (size_t)g * ldh);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int q = lane + 32 * h;
        uint4 v = make_uint4(0u, 0u, 0u, 0u);  // rows past the last game: zeros
        if (g < G) {
          const float4 lo = __ldg(src + 2 * q), hi = __ldg(src + 2 * q + 1);
          v = make_uint4(pack_bf16(lo.x, lo.y), pack_bf16(lo.z, lo.w), pack_bf16(hi.x, hi.y), pack_bf16(hi.z, hi.w));
        }
        const uint32_t dst = smem_u32(s_a + (q >> 3) * SH_A_KB_BYTES + r * 128 + (((q & 7) ^ (r & 7)) << 4));
        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                     : "memory");
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> tensor core reads
    __syncwarp();
    if (lane == 0) mbar_arrive(a_full);

    const uint32_t lane_addr = tmem + ((uint32_t)(quarter * 32) << 16);
    float m = -INFINITY, den = 0.0f, num = 0.0f;
    for (int chunk = 0; chunk < nchunks; ++chunk) {
      const int acc = chunk & 1;
      mbar_wait(&acc_full[acc], (chunk >> 1) & 1);
      tc_fence_after();
#pragma unroll 1
      for (int c0 = 0; c0 < SH_N; c0 += 32) {
        const int col0 = chunk * SH_N + c0;
        if (col0 >= bins) break;  // uniform: whole groups past the support are never read
        uint32_t v[32];
        tmem_ld32(lane_addr + acc * SH_N + c0, v);
        tmem_wait_ld();
        float x[32];
        float gm = -INFINITY;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          x[j] = __uint_as_float(v[j]) + s_bias[col0 + j];
          gm = fmaxf(gm, x[j]);
        }
        const float nm = fmaxf(m, gm);   // finite: every group read holds at least one real bin
        const float sc = expf(m - nm);   // 0 on the first group (m = -inf), 1 when the max holds
        den *= sc;
        num *= sc;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float e = expf(x[j] - nm);
          den += e;
          num = fmaf(e, (float)(support_min + col0 + j), num);
        }
        m = nm;
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0)
        asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&acc_empty[acc])) : "memory");
    }
    const int g = g0 + row;
    if (g < G) {
      float x = num / den;
      if (!no_tt) {  // same h^-1 arithmetic as conv_head_kernel
        const float eps = 0.001f;
        const float sgn = x > 0.0f ? 1.0f : (x < 0.0f ? -1.0f : 0.0f);
        const float t = (sqrtf(1.0f + 4.0f * eps * (fabsf(x) + 1.0f + eps)) - 1.0f) / (2.0f * eps);
        x = sgn * (t * t - 1.0f);
      }
      out[(size_t)g * ldo] = x;
    }
  }

  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem, 2 * SH_N);
  }
}

// ---- heads: relu(fc1) [G][512] -> Linear(512 -> bins) (+ softmax expectation + h^-1) --------------
// One warp per game.  networks.py:438-440, 477-483; config.py:27-33.
__global__ void conv_head_kernel(int G, const float* __restrict__ hidden, int ldh, const float* __restrict__ w2,
                                 const float* __restrict__ b2, int outs, int to_scalar, int support_min,
                                 int no_tt, float* __restrict__ out, int ldo);

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

// [rows][cols] bf16 row-major (cols contiguous), box = 64 rows x 64 cols, 128-byte swizzle
int make_map(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows = 64) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return MZ_ERR_UNSUPPORTED;
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {cols * 2};
  const cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? MZ_OK : 1000 + (int)r;
}

constexpr size_t kConvSmem = 1024 + (size_t)STAGES * STAGE_BYTES + (2 * STAGES + 4) * sizeof(uint64_t) + 16 +
                             1024 * sizeof(float);

int launch_conv(const CUtensorMap& ma, const CUtensorMap& mb, const ConvParams& p, void* stream) {
  static bool attr = false;
  static int sms = 0;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(conv_gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kConvSmem);
    if (e != cudaSuccess) return (int)e;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    attr = true;
  }
  const int tiles = ((p.num_tiles_m + TU - 1) / TU) * p.num_tiles_n;
  const int grid = tiles < sms ? tiles : sms;
  cudaError_t e = mz_launch(conv_gemm_tc_kernel, dim3(grid), dim3(CONV_THREADS), kConvSmem,
                            (cudaStream_t)stream, true, ma, mb, p);
  if (e != cudaSuccess) return (int)e;
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

constexpr size_t kPairSmem = 1024 + (size_t)P_KBLOCKS * P_BH_BYTES + (size_t)P_A_REGION +
                             (2 * P_STAGES + 2 * P_ACC + 1) * sizeof(uint64_t) + 16 + BN * sizeof(float) + 16 + 4 * 2048;
// 128-channel 3x3 convolutions: 0 = single-CTA kernel, 1 = CTA-pair kernel with one activation load per
// tap, 2 = CTA-pair kernel with one row window per tile where the image is narrow enough (wider images
// fall back to 1)
int g_conv_pair = 2;

int launch_conv_pair(const CUtensorMap& ma, const CUtensorMap& mb, const CUtensorMap& mw, const ConvParams& p,
                     int window, void* stream) {
  static bool attr = false;
  static int sms = 0;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(conv_pair_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)kPairSmem);
    if (e != cudaSuccess) return (int)e;
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    attr = true;
  }
  const int pairs = (p.num_tiles_m + 1) / 2;
  const int grid = 2 * (pairs < sms / 2 ? pairs : sms / 2);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(CONV_THREADS);
  cfg.dynamicSmemBytes = kPairSmem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attrs[2];
  attrs[0].id = cudaLaunchAttributeClusterDimension;
  attrs[0].val.clusterDim.x = 2;
  attrs[0].val.clusterDim.y = 1;
  attrs[0].val.clusterDim.z = 1;
  attrs[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attrs[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attrs;
  cfg.numAttrs = g_mz_pdl ? 2 : 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, conv_pair_tc_kernel, ma, mb, mw, p, window);
  if (e != cudaSuccess) return (int)e;
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

__global__ void conv_head_kernel(int G, const float* __restrict__ hidden, int ldh, const float* __restrict__ w2,
                                 const float* __restrict__ b2, int outs, int to_scalar, int support_min,
                                 int no_tt, float* __restrict__ out, int ldo) {
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (g >= G) return;
  const float* h = hidden + (size_t)g * ldh;
  float hv[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) hv[i] = h[lane + 32 * i];
  float mine = 0.0f;  // lane o keeps output o
  for (int o = 0; o < outs; ++o) {
    const float* w = w2 + (size_t)o * 512;
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < 16; ++i) s = fmaf(hv[i], w[lane + 32 * i], s);
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) s += __shfl_xor_sync(MZ_FULL, s, m);
    if (lane == o) mine = s + b2[o];
  }
  if (!to_scalar) {
    if (lane < outs) out[(size_t)g * ldo + lane] = mine;
    return;
  }
  // Config.inverse_transform config.py:27-33: softmax expectation over the support, then h^-1
  float m = lane < outs ? mine : -INFINITY;
#pragma unroll
  for (int k = 16; k > 0; k >>= 1) m = fmaxf(m, __shfl_xor_sync(MZ_FULL, m, k));
  const float e = lane < outs ? expf(mine - m) : 0.0f;
  float den = e, num = e * (float)(support_min + lane);
#pragma unroll
  for (int k = 16; k > 0; k >>= 1) {
    den += __shfl_xor_sync(MZ_FULL, den, k);
    num += __shfl_xor_sync(MZ_FULL, num, k);
  }
  if (lane == 0) {
    float x = num / den;
    if (!no_tt) {
      const float eps = 0.001f;
      const float sgn = x > 0.0f ? 1.0f : (x < 0.0f ? -1.0f : 0.0f);
      const float t = (sqrtf(1.0f + 4.0f * eps * (fabsf(x) + 1.0f + eps)) - 1.0f) / (2.0f * eps);
      x = sgn * (t * t - 1.0f);
    }
    out[(size_t)g * ldo] = x;
  }
}

// out rows [g * 49, g * 49 + 49) = pool slot [g][node[g]] (pool = [G][nodes_per_game][49][128] bf16):
// the gather of search_path[-2].hidden_state (mcts.py:94-96) into the flat layout the GEMM tiles.
// One warp per row (256 B), 16-byte loads.
__global__ void conv_gather_kernel(int G, int nodes_per_game, const int32_t* __restrict__ node,
                                   const uint4* __restrict__ pool, uint4* __restrict__ out) {
  const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (w >= G * GROWS) return;
  const int g = w / GROWS, r = w - g * GROWS;
  const size_t src = ((size_t)g * nodes_per_game + node[g]) * GROWS + r;
  if (lane < 16) out[(size_t)w * 16 + lane] = pool[src * 16 + lane];
}

// Stride-2 3x3 patches of a padded channels-last image as GEMM rows: out[(g, y, x)][tap * C + c] =
// in[g][2y + ky - 1][2x + kx - 1][c].  The zero padding is physically present in the layout, so the
// gather needs no bounds checks.  One thread per 16-byte chunk.
__global__ void conv_im2col_s2_kernel(int games, int w_in, int C, int k_pad, const uint4* __restrict__ in,
                                      uint4* __restrict__ out) {
  const int w_out = w_in / 2, wp = w_in + 1, cpr = C / 8, kchunks = k_pad / 8;
  const long long total = (long long)games * w_out * w_out * kchunks;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int kc = (int)(i % kchunks);
    const long long r = i / kchunks;
    const int x = (int)(r % w_out), y = (int)((r / w_out) % w_out), g = (int)(r / ((long long)w_out * w_out));
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    const int tap = kc / cpr;
    if (tap < 9) {
      const int cc = kc - tap * cpr, ky = tap / 3, kx = tap - 3 * ky;
      const long long src = (long long)g * wp * wp + wp + (long long)(2 * y + ky - 1) * wp + (2 * x + kx - 1);
      if (src >= 0) v = in[src * cpr + cc];  // row -1 of game 0 lies before the buffer: zero padding
    }
    out[i] = v;
  }
}

// AvgPool2d(3, stride 2, padding 1, count_include_pad) between two padded channels-last layouts.
__global__ void conv_avgpool_kernel(int games, int w_in, int C, const uint4* __restrict__ in,
                                    uint4* __restrict__ out) {
  const int w_out = w_in / 2, wp = w_in + 1, wpo = w_out + 1, cpr = C / 8;
  const long long total = (long long)games * w_out * w_out * cpr;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int cc = (int)(i % cpr);
    const long long r = i / cpr;
    const int x = (int)(r % w_out), y = (int)((r / w_out) % w_out), g = (int)(r / ((long long)w_out * w_out));
    float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int ky = tap / 3, kx = tap - 3 * ky;
      const long long src = (long long)g * wp * wp + wp + (long long)(2 * y + ky - 1) * wp + (2 * x + kx - 1);
      const uint4 v = src >= 0 ? in[src * cpr + cc] : make_uint4(0u, 0u, 0u, 0u);
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int h = 0; h < 4; ++h) {
        const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162*>(&w[h]);
        acc[2 * h] += __low2float(b2);
        acc[2 * h + 1] += __high2float(b2);
      }
    }
    const float s = 1.0f / 9.0f;
    const long long dst = (long long)g * wpo * wpo + wpo + (long long)y * wpo + x;
    out[dst * cpr + cc] = make_uint4(pack_bf16(acc[0] * s, acc[1] * s), pack_bf16(acc[2] * s, acc[3] * s),
                                     pack_bf16(acc[4] * s, acc[5] * s), pack_bf16(acc[6] * s, acc[7] * s));
  }
}

}  // namespace

extern "C" {

// Stride-2 convolution, step 1: patches -> GEMM rows.  in: padded channels-last image
// [games * (w_in + 1)^2][C] bf16; out: [games * (w_in / 2)^2][k_pad] bf16 with k = tap * C + c
// (columns >= 9 C are zero).  C % 8 == 0, k_pad % 64 == 0.
int mz_conv_im2col_s2(int32_t games, int32_t w_in, int32_t channels, int32_t k_pad, const void* in, void* out,
                      void* stream) {
  if (games < 1 || w_in < 2 || (w_in & 1) || channels < 8 || (channels % 8) || k_pad < 9 * channels ||
      (k_pad % 64) || !in || !out)
    return MZ_ERR_BAD_ARG;
  conv_im2col_s2_kernel<<<148 * 16, 256, 0, (cudaStream_t)stream>>>(games, w_in, channels, k_pad,
                                                                    (const uint4*)in, (uint4*)out);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

// Stride-2 convolution, step 2 (and any Linear layer whose output is an image): out[(g, y, x)] =
// a[(g, y, x)] . w^T + bias (+ReLU) as bf16 rows of the padded layout of an out_w x out_w image with
// n_out (64 or 128) channels.  a [rows][k] bf16, w [n_out][k] bf16, k % 64 == 0.  The padding rows of
// `out` are not touched (zero them once).
int mz_conv_gemm_to_padded(int32_t games, int32_t out_w, int32_t k, int32_t n_out, const void* a, const void* w,
                           const float* bias, int32_t relu, void* out, void* stream) {
  if (games < 1 || out_w < 1 || k < 64 || (k % 64) || (n_out != 64 && n_out != 128) || !a || !w || !bias || !out)
    return MZ_ERR_BAD_ARG;
  const long long rows = (long long)games * out_w * out_w;
  if (rows > 0x7fffffffLL - 2 * BM) return MZ_ERR_UNSUPPORTED;
  CUtensorMap ma, mb;
  int rc = make_map(&ma, a, (uint64_t)rows, (uint64_t)k);
  if (rc) return rc;
  rc = make_map(&mb, w, (uint64_t)n_out, (uint64_t)k);
  if (rc) return rc;
  ConvParams p = {};
  p.mode_fc = 1;
  p.num_tiles_m = (int)((rows + BM - 1) / BM);
  p.num_tiles_n = 1;
  p.ncols = n_out;
  p.kb_per_tap = 1;
  p.num_kblocks = k / BK;
  p.rows_total = (int)rows;
  p.flags = EPI_TO_PADDED | (relu ? EPI_RELU : 0);
  p.bias = bias;
  p.out = (__nv_bfloat16*)out;
  p.out_w = out_w;
  return launch_conv(ma, mb, p, stream);
}

// AvgPool2d(kernel 3, stride 2, padding 1) (networks.py:406, 409) between padded channels-last layouts:
// in [games * (w_in + 1)^2][C] -> out [games * (w_in / 2 + 1)^2][C] (padding rows of `out` untouched).
int mz_conv_avgpool(int32_t games, int32_t w_in, int32_t channels, const void* in, void* out, void* stream) {
  if (games < 1 || w_in < 2 || (w_in & 1) || channels < 8 || (channels % 8) || !in || !out) return MZ_ERR_BAD_ARG;
  conv_avgpool_kernel<<<148 * 16, 256, 0, (cudaStream_t)stream>>>(games, w_in, channels, (const uint4*)in,
                                                                  (uint4*)out);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

// Gathers hidden-pool slots [g][node[g]] into the flat activation layout: out [games * 49][128] bf16.
int mz_conv_gather(int32_t games, int32_t nodes_per_game, const int32_t* node, const void* pool, void* out,
                   void* stream) {
  if (games < 1 || nodes_per_game < 1 || !node || !pool || !out) return MZ_ERR_BAD_ARG;
  const long long warps = (long long)games * GROWS;
  conv_gather_kernel<<<(unsigned)((warps * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      games, nodes_per_game, node, (const uint4*)pool, (uint4*)out);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

// 3x3 convolution (+ folded BatchNorm, bias, optional action plane / residual / ReLU / state scaling)
// over `games` images of width x width pixels in the flat padded channels-last bf16 layout
// ((width + 1)^2 rows x 128 channels per game: a zero row, then `width` image rows of `width`
// pixels + 1 zero; 49 rows for the 6 x 6 hidden state).
//   x, residual, out, out_scaled   [games * (width + 1)^2][128] bf16
//   w_packed     [128][9 * 128] bf16, k = (ky * 3 + kx) * 128 + c_in
//   bias         [128] f32;  plane_term [36][128] f32 and actions [games] when flags & 4
//   pool_out + pool_row_base: with flags & 8 the scaled rows of game g are also written at rows
//   pool_row_base[g] .. + 49 of pool_out (the hidden pool slot of the new node)
int mz_conv3x3_tc(int32_t games, int32_t width, int32_t channels, const void* x, const void* w_packed,
                  const float* bias, int32_t flags,
                  const float* plane_term, const int32_t* actions, int32_t num_actions,
                  const void* residual, void* out, void* out_scaled, void* pool_out,
                  const int32_t* pool_row_base, void* stream) {
  if (games < 1 || width < 1 || width > 255 || !x || !w_packed || !bias) return MZ_ERR_BAD_ARG;
  if (channels != 64 && channels != 128) return MZ_ERR_UNSUPPORTED;
  if ((flags & EPI_ACTION) && (!plane_term || !actions || num_actions < 1)) return MZ_ERR_BAD_ARG;
  if ((flags & EPI_RESIDUAL) && !residual) return MZ_ERR_BAD_ARG;
  if ((flags & EPI_SCALE) && !out_scaled) return MZ_ERR_BAD_ARG;
  if (!(flags & EPI_SCALE) && !out) return MZ_ERR_BAD_ARG;
  if (pool_out && !pool_row_base) return MZ_ERR_BAD_ARG;
  if (flags & EPI_F32_OUT) return MZ_ERR_BAD_ARG;
  const int wp = width + 1, grows = wp * wp;
  const long long rows = (long long)games * grows;
  if (rows > 0x7fffffffLL - 2 * BM) return MZ_ERR_UNSUPPORTED;
  CUtensorMap ma, mb;
  int rc = make_map(&ma, x, (uint64_t)rows, (uint64_t)channels);
  if (rc) return rc;
  rc = make_map(&mb, w_packed, (uint64_t)channels, 9 * (uint64_t)channels);
  if (rc) return rc;
  ConvParams p = {};
  p.mode_fc = 0;
  p.num_tiles_m = (int)((rows + BM - 1) / BM);
  p.num_tiles_n = 1;
  p.ncols = channels;
  p.kb_per_tap = channels / BK;
  p.num_kblocks = 9 * p.kb_per_tap;
  p.rows_total = (int)rows;
  p.flags = flags;
  p.num_actions = num_actions;
  p.wp = wp;
  p.grows = grows;
  p.bias = bias;
  p.plane_term = plane_term;
  p.actions = actions;
  p.residual = (const __nv_bfloat16*)residual;
  p.out = (__nv_bfloat16*)out;
  p.out_scaled = (__nv_bfloat16*)out_scaled;
  p.pool_out = (__nv_bfloat16*)pool_out;
  p.pool_row_base = pool_row_base;
  if (channels == 128 && g_conv_pair) {
    const int window = (g_conv_pair >= 2 && wp + 1 <= P_WIN_PAD) ? 1 : 0;
    CUtensorMap mw = ma;
    if (window) {
      rc = make_map(&mw, x, (uint64_t)rows, (uint64_t)channels, P_WIN_ROWS);
      if (rc) return rc;
    }
    return launch_conv_pair(ma, mb, mw, p, window, stream);
  }
  return launch_conv(ma, mb, p, stream);
}

int mz_conv_set_pair(int32_t mode) {
  if (mode < 0 || mode > 2) return MZ_ERR_BAD_ARG;
  g_conv_pair = mode;
  return MZ_OK;
}

// Linear(49 * 128 -> n_out) over the padded channels-last state (padding rows are zero), bias + ReLU:
//   x [games][6272] bf16 (the activation buffer itself), w_packed [n_out][6272] bf16 (n_out % 128 == 0),
//   out [games][ldo] f32.   networks.py:436-439, 470-478.
int mz_conv_fc_tc(int32_t games, const void* x, const void* w_packed, const float* bias, int32_t n_out,
                  int32_t relu, float* out, int32_t ldo, void* stream) {
  if (games < 1 || !x || !w_packed || !bias || !out || n_out < 128 || (n_out % 128) || ldo < n_out)
    return MZ_ERR_BAD_ARG;
  CUtensorMap ma, mb;
  constexpr int KFC = GROWS * 128;
  int rc = make_map(&ma, x, (uint64_t)games, KFC);
  if (rc) return rc;
  rc = make_map(&mb, w_packed, (uint64_t)n_out, KFC);
  if (rc) return rc;
  ConvParams p = {};
  p.mode_fc = 1;
  p.num_tiles_m = (games + BM - 1) / BM;
  p.num_tiles_n = n_out / BN;
  p.ncols = BN;
  p.kb_per_tap = 1;
  p.num_kblocks = KFC / BK;
  p.rows_total = games;
  p.flags = EPI_F32_OUT | (relu ? EPI_RELU : 0);
  p.bias = bias;
  p.out_f32 = out;
  p.ldo = ldo;
  return launch_conv(ma, mb, p, stream);
}

// Second layer of a head on CUDA cores: out = hidden[g] . w2^T + b2 (outs <= 32); to_scalar != 0
// applies Config.inverse_transform (softmax expectation over [support_min, support_min + outs) and
// h^-1 unless no_target_transform) and writes one float per game.
int mz_conv_head(int32_t games, const float* hidden, int32_t ldh, const float* w2, const float* b2,
                 int32_t outs, int32_t to_scalar, int32_t support_min, int32_t no_target_transform,
                 float* out, int32_t ldo, void* stream) {
  if (games < 1 || !hidden || !w2 || !b2 || !out || outs < 1 || outs > 32 || ldh < 512) return MZ_ERR_BAD_ARG;
  const int threads = 256, grid = (games * 32 + threads - 1) / threads;
  conv_head_kernel<<<grid, threads, 0, (cudaStream_t)stream>>>(games, hidden, ldh, w2, b2, outs, to_scalar,
                                                               support_min, no_target_transform, out, ldo);
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

// Value / reward head Linear(512 -> bins) on the tensor cores for 33 <= bins <= 1024, followed by
// Config.inverse_transform (config.py:27-33): one float per game at out[g * ldo].  hidden: float32 rows
// of stride ldh (16-byte aligned), w2: bf16 [bins][512] row-major (16-byte aligned), b2: float32 [bins].
int mz_conv_support_head_tc(int32_t games, const float* hidden, int32_t ldh, const void* w2, const float* b2,
                            int32_t bins, int32_t support_min, int32_t no_target_transform, float* out, int32_t ldo,
                            void* stream) {
  if (games < 1 || !hidden || !w2 || !b2 || !out || ldh < SH_K || (ldh % 4) || ldo < 1 ||
      (reinterpret_cast<uintptr_t>(hidden) & 15) || (reinterpret_cast<uintptr_t>(w2) & 15))
    return MZ_ERR_BAD_ARG;
  if (bins < SH_MIN_BINS || bins > SH_MAX_BINS) return MZ_ERR_UNSUPPORTED;
  static bool attr = false;
  const size_t smem = 1024 + (size_t)SH_A_BYTES + (size_t)SH_STAGES * SH_B_BYTES +
                      (2 * SH_STAGES + 5) * sizeof(uint64_t) + 16 + SH_MAX_BINS * sizeof(float);
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(conv_support_head_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  CUtensorMap mw;
  const int rc = make_map(&mw, w2, (uint64_t)bins, SH_K);
  if (rc) return rc;
  cudaError_t e = mz_launch(conv_support_head_tc_kernel, dim3((games + BM - 1) / BM), dim3(SH_THREADS), smem,
                            (cudaStream_t)stream, true, mw, (int)games, hidden, (int)ldh, b2, (int)bins,
                            (int)support_min, (int)no_target_transform, out, (int)ldo);
  if (e != cudaSuccess) return (int)e;
  MZ_LAUNCH_CHECK();
  return MZ_OK;
}

}  // extern "C"
