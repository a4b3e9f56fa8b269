// Shared device helpers for libmzb200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "mzb200.h"

#define MZ_DEV __device__ __forceinline__
#define MZ_FULL 0xffffffffu

#define MZ_LAUNCH_CHECK()                         \
  do {                                            \
    cudaError_t e__ = cudaGetLastError();         \
    if (e__ != cudaSuccess) return (int)e__;      \
  } while (0)

// ---- node record accessors (layout documented in include/mzb200.h) ---------------------------
struct MzNode {
  uint8_t* p;
  int A;
  MZ_DEV double& q() const { return *reinterpret_cast<double*>(p); }
  MZ_DEV int32_t& visit() const { return *reinterpret_cast<int32_t*>(p + 8); }
  MZ_DEV float& reward() const { return *reinterpret_cast<float*>(p + 12); }
  MZ_DEV double& vsum() const { return *reinterpret_cast<double*>(p + 16); }
  MZ_DEV double* prior() const { return reinterpret_cast<double*>(p + MZ_NODE_STATS_BYTES); }
  MZ_DEV int16_t* child() const {
    return reinterpret_cast<int16_t*>(p + MZ_NODE_STATS_BYTES + 8 * A);
  }
};

struct MzGame {
  uint8_t* base;
  int node_bytes;
  int A;
  MZ_DEV double& mn() const { return *reinterpret_cast<double*>(base); }
  MZ_DEV double& mx() const { return *reinterpret_cast<double*>(base + 8); }
  MZ_DEV int32_t& root_to_play() const { return *reinterpret_cast<int32_t*>(base + 16); }
  MZ_DEV MzNode node(int n) const {
    return MzNode{base + MZ_GAME_HEADER_BYTES + (size_t)n * node_bytes, A};
  }
};

// ---- programmatic dependent launch ---------------------------------------------------------------
// A kernel launched with the programmatic-stream-serialization attribute may start while its
// predecessor in the stream is still running; everything it does before pdl_wait() must neither read
// what the predecessor writes nor write what it reads.  pdl_trigger() lets the NEXT kernel start its
// own prologue; it is issued after pdl_wait() so that overlap never spans more than one kernel.
// Both are no-ops for a plain launch.
MZ_DEV void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
MZ_DEV void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

extern int g_mz_pdl;  // 1: the per-simulation kernels are launched as programmatic dependents

template <typename... KArgs, typename... Args>
inline cudaError_t mz_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                             bool dependent, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (dependent && g_mz_pdl) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---- 3xTF32 operands ----------------------------------------------------------------------------
// The split of the float32-accurate tensor-core products x w ~= x_lo w_hi + x_hi w_lo + x_hi w_hi (three TF32 mma,
// float32 accumulation).  x = hi + lo: hi = x cut to TF32's 11 significant bits (one LOP3; `cvt.rna.tf32.f32` compiles to five
// instructions on sm_100a), lo = the exact float32 remainder (|lo| < 2^-10 |x|), of which the tensor core reads the
// top 11 bits (the low 13 mantissa bits of a .tf32 operand register are ignored).  What a product loses -- lo's own
// cut and the x_lo * w_lo term -- is below 2^-20 of it.
MZ_DEV void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}

// ---- 64-bit shuffles ---------------------------------------------------------------------------
template <int W>
MZ_DEV double shfl_f64(double v, int src) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_sync(MZ_FULL, lo, src, W);
  hi = __shfl_sync(MZ_FULL, hi, src, W);
  return __hiloint2double(hi, lo);
}
template <int W>
MZ_DEV double shfl_xor_f64(double v, int m) {
  int lo = __double2loint(v), hi = __double2hiint(v);
  lo = __shfl_xor_sync(MZ_FULL, lo, m, W);
  hi = __shfl_xor_sync(MZ_FULL, hi, m, W);
  return __hiloint2double(hi, lo);
}

// ---- mbarrier + 1-D bulk async copy (TMA unit, no tensor map) -----------------------------------
MZ_DEV uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
MZ_DEV void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
MZ_DEV void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
MZ_DEV void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
MZ_DEV void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
MZ_DEV bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
MZ_DEV void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// global -> shared, `bytes` multiple of 16, both addresses 16-byte aligned; completes on `bar`
MZ_DEV void bulk_copy_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}
