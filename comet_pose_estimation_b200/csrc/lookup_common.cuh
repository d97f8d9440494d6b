// Shared by the fused lookup kernels (corr_lookup.cu, corr_lookup_up2.cu): parameter block, TMA / mbarrier helpers,
// tensor-map encoding of one channel-last pyramid level.
#pragma once
#include "comet_common.cuh"

#include <cuda.h>
#include <cstring>

namespace comet {

struct LookupParams {
  const float* fmaps;
  const float* pyr;
  const float* targets;
  long long t_sb, t_ss, t_sn;
  int t_level_stride;
  const float* coords;
  long long c_sb, c_ss, c_sn;
  float* out;
  long long o_sb, o_ss, o_sn;
  const float* pos;  // TOKENS: (B,N,D_tok)
  const int* ntr;    // TOKENS: (B,) query count of each sequence (rows n >= ntr[b] are written as zeros), or null
  const int* nfr;    // TOKENS: (B,) frame count of each sequence (rows s >= nfr[b] are written as zeros), or null
  const int* fidx;   // TOKENS: (B,S) frame of fmaps / pyr that (item b, position s) reads, or null (b * S + s)
  int BS_src;        // TOKENS with fidx: frames of fmaps / pyr (entries are clamped to [0, BS_src))
  int D_tok;
  int B, S, N, C, L, r;
  int pad_border, bf16;
  int lvlH[COMET_MAX_LEVELS], lvlW[COMET_MAX_LEVELS];
  long long lvlOff[COMET_MAX_LEVELS];
  int channel_last;  // levels >= 1 stored (BS, H_l, W_l, C) instead of (BS, C, H_l, W_l)
  int cl0;           // level 0 (the caller's fmaps) is channel-last too
  float sqrt_c;
  float inv_sqrt_c;
};

namespace tma {
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  // a protocol bug must fail visibly, not hang the device: trap after 10 s of WALL time (not a poll count, so that
  // sanitizers / debuggers / time-slicing cannot fire it on a healthy kernel)
  uint32_t spins = 0;
  uint64_t t0 = 0;
  while (!mbar_try(bar, parity)) {
    if ((++spins & 4095u) == 0) {
      uint64_t now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 10000000000ull) __trap();
    }
  }
}
__device__ __forceinline__ void load_box_4d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
}  // namespace tma

struct TmaMaps { CUtensorMap m[3]; };

// 4-D tensor map over one channel-last level: dims (fastest first) {32 channels, W_l, H_l, BS}, box {32, G, G, 1},
// 128-byte swizzle, zero fill outside the map.
static inline int encode_level_map(CUtensorMap* tm, const float* base, int BS, int Hl, int Wl, int G) {
  TensorMapEncodeFn enc = tensor_map_encoder();
  if (!enc) return fail(COMET_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled is not available");
  const cuuint64_t gdim[4] = {32, (cuuint64_t)Wl, (cuuint64_t)Hl, (cuuint64_t)BS};
  const cuuint64_t gstride[3] = {128, (cuuint64_t)Wl * 128, (cuuint64_t)Hl * Wl * 128};
  const cuuint32_t box[4] = {32, (cuuint32_t)G, (cuuint32_t)G, 1};
  const cuuint32_t estride[4] = {1, 1, 1, 1};
  CUresult cr = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), gdim, gstride, box, estride,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) return fail(COMET_ERR_CUDA, "cuTensorMapEncodeTiled failed with %d", (int)cr);
  return COMET_OK;
}


}  // namespace comet
