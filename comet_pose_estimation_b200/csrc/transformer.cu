// Row-wise pieces of the track-update transformer between the tensor-core GEMMs of gemm_tc.cu
// (EfficientUpdateFormer, comet/models/track_modules/blocks.py:298-348; AttnBlock / CrossAttnBlock,
// comet/models/modules.py:248-344):
//
//   layernorm_planes_kernel   nn.LayerNorm over the last dimension (with or without affine), result written as float32
//                             (the reference's blocks add the attention output to the NORMALISED input, so it is needed
//                             as a residual) and / or as bf16 planes = the A operand of the next GEMM;
//   attention_kernel          softmax(q k^T / sqrt(dh)) v per (batch item, head) of nn.MultiheadAttention for the short
//                             sequences of this model: T = 16 frames (time blocks), 64 virtual tracks x N point tracks
//                             (space blocks).  Arbitrary batch / position strides, so neither the "(b n) t c" nor the
//                             "(b t) n c" rearrangement of the reference is ever materialised; float32 arithmetic on the
//                             CUDA cores (0.2 - 0.8 GFLOP per block: not tensor-core work); output directly as bf16
//                             planes for the out-projection GEMM.
#include "comet_common.cuh"

namespace comet {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// store v as np bf16 planes at index idx of planes p0 + k * plane_stride
__device__ __forceinline__ void store_planes(__nv_bfloat16* p0, long long plane_stride, long long idx, float v, int np) {
  for (int k = 0; k < np; ++k) {
    const __nv_bfloat16 b = __float2bfloat16_rn(v);
    p0[k * plane_stride + idx] = b;
    v -= __bfloat162float(b);
  }
}

// four consecutive values as np bf16 planes: one 8-byte store per plane (idx and plane_stride multiples of 4, base 8-byte aligned)
__device__ __forceinline__ void store_planes4(__nv_bfloat16* p0, long long plane_stride, long long idx, float4 v, int np) {
  for (int k = 0; k < np; ++k) {
    const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
    uint2 pk;
    pk.x = *reinterpret_cast<const uint32_t*>(&a);
    pk.y = *reinterpret_cast<const uint32_t*>(&b);
    *reinterpret_cast<uint2*>(p0 + k * plane_stride + idx) = pk;
    v.x -= __low2float(a); v.y -= __high2float(a); v.z -= __low2float(b); v.w -= __high2float(b);
  }
}

// One warp per row; D <= 32 * KPL (KPL values per lane, compile time).
constexpr int LN_MAX_PER_LANE = 32;
template <int KPL>
__global__ void __launch_bounds__(256) layernorm_planes_kernel(const float* __restrict__ x, long long x_ld,
                                                                const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                float eps, float* __restrict__ out, long long out_ld,
                                                                __nv_bfloat16* __restrict__ planes, long long plane_stride,
                                                                long long p_ld, int np, long long rows, int D) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long r = warp0; r < rows; r += nwarps) {
    const float* xr = x + r * x_ld;
    float v[KPL];
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < KPL; ++k) {
      const int c = lane + 32 * k;
      v[k] = c < D ? __ldg(xr + c) : 0.f;
      s += v[k];
    }
    const float mean = warp_sum(s) / (float)D;
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < KPL; ++k) {
      const int c = lane + 32 * k;
      const float d = c < D ? v[k] - mean : 0.f;
      q += d * d;
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)D + eps);
#pragma unroll
    for (int k = 0; k < KPL; ++k) {
      const int c = lane + 32 * k;
      if (c < D) {
        float y = (v[k] - mean) * rstd;
        if (gamma) y = y * __ldg(gamma + c) + __ldg(beta + c);
        if (out) out[r * out_ld + c] = y;
        if (planes) store_planes(planes, plane_stride, r * p_ld + c, y, np);
      }
    }
  }
}

// The same with 16-byte accesses: a lane owns KG groups of four consecutive columns (column 4 * lane + 128 * g), so a row
// is read with LDG.128, written with STG.128 (float32) and STG.64 (four bf16 of a plane) -- the scalar kernel issues
// 12 + 12 + 36 memory instructions per lane for a 384-wide row with three planes, this one 3 + 3 + 9.
// Needs D % 4 == 0 and 16-byte aligned rows (8-byte for the planes); D <= 128 * KG.
template <int KG>
__global__ void __launch_bounds__(256) layernorm_planes_v4_kernel(const float* __restrict__ x, long long x_ld,
                                                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                   float eps, float* __restrict__ out, long long out_ld,
                                                                   __nv_bfloat16* __restrict__ planes, long long plane_stride,
                                                                   long long p_ld, int np, long long rows, int D) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
  float4 gm[KG], bt[KG];
#pragma unroll
  for (int g = 0; g < KG; ++g) {
    const int c = 4 * lane + 128 * g;
    gm[g] = (gamma && c < D) ? __ldg(reinterpret_cast<const float4*>(gamma + c)) : make_float4(1.f, 1.f, 1.f, 1.f);
    bt[g] = (beta && c < D) ? __ldg(reinterpret_cast<const float4*>(beta + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (long long r = warp0; r < rows; r += nwarps) {
    const float* xr = x + r * x_ld;
    float4 v[KG];
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < KG; ++g) {
      const int c = 4 * lane + 128 * g;
      v[g] = c < D ? __ldg(reinterpret_cast<const float4*>(xr + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
      s += (v[g].x + v[g].y) + (v[g].z + v[g].w);
    }
    const float mean = warp_sum(s) / (float)D;
    float q = 0.f;
#pragma unroll
    for (int g = 0; g < KG; ++g) {
      const int c = 4 * lane + 128 * g;
      if (c < D) {
        const float dx = v[g].x - mean, dy = v[g].y - mean, dz = v[g].z - mean, dw = v[g].w - mean;
        q += (dx * dx + dy * dy) + (dz * dz + dw * dw);
      }
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)D + eps);
#pragma unroll
    for (int g = 0; g < KG; ++g) {
      const int c = 4 * lane + 128 * g;
      if (c < D) {
        float y[4] = {(v[g].x - mean) * rstd, (v[g].y - mean) * rstd, (v[g].z - mean) * rstd, (v[g].w - mean) * rstd};
        if (gamma) {
          y[0] = y[0] * gm[g].x + bt[g].x; y[1] = y[1] * gm[g].y + bt[g].y;
          y[2] = y[2] * gm[g].z + bt[g].z; y[3] = y[3] * gm[g].w + bt[g].w;
        }
        if (out) *reinterpret_cast<float4*>(out + r * out_ld + c) = make_float4(y[0], y[1], y[2], y[3]);
        if (planes) {
          for (int k = 0; k < np; ++k) {
            const __nv_bfloat162 a = __floats2bfloat162_rn(y[0], y[1]), b = __floats2bfloat162_rn(y[2], y[3]);
            uint2 pk;
            pk.x = *reinterpret_cast<const uint32_t*>(&a);
            pk.y = *reinterpret_cast<const uint32_t*>(&b);
            *reinterpret_cast<uint2*>(planes + k * plane_stride + r * p_ld + c) = pk;
            y[0] -= __low2float(a); y[1] -= __high2float(a); y[2] -= __low2float(b); y[3] -= __high2float(b);
          }
        }
      }
    }
  }
}

// q/k/v element (batch b, position i, head h, dim d) at ptr + b * sb + i * si + h * dh + d  (float32).
// One warp per (batch, head, query position); scores of a query live in shared memory (Lk floats per warp).
struct AttnParams {
  const float* q; long long q_sb, q_si;
  const float* k; long long k_sb, k_si;
  const float* v; long long v_sb, v_si;
  __nv_bfloat16* out; long long o_plane_stride, o_sb, o_si;   // planes, element (b, i, h*dh + d) at b*o_sb + i*o_si + ...
  int np;
  int B, H, Lq, Lk, dh;
  float scale;
  int vec_out;   // output planes can be written four values (8 bytes) at a time
  // Variable lengths (comet_attention_varlen_planes_f32), null otherwise: item b's queries / outputs start at row q_off[b]
  // and its keys / values at row k_off[b] (the *_sb strides are then row pitches), with q_len[b] / k_len[b] positions.
  // Lq / Lk hold the largest lengths.  A launch serves only the items whose attn_path() is `path`.
  // `groups` (varlen, nullable): item b's problem count for attn_path() is groups[b] instead of `group`.
  const int* q_off; const int* q_len; const int* k_off; const int* k_len;
  int path, group, mma_opt, mma_align;
  const int* groups;
};

// Kernel family of an attention problem: one definition for the host dispatch of comet_attention_planes_f32 and for the
// per-item choice of the varlen launches, so that an item of a varlen call gets exactly the arithmetic a single call of
// the same shape gets.  `B` is the number of problems of that single call (it sizes the grid of the key-split kernel).
enum { AP_SMALL_MMA, AP_SMALL, AP_ROWS_MMA, AP_ROWS, AP_KSPLIT, AP_TILED, AP_COUNT };
constexpr int ATR_KMAX = 64;
__host__ __device__ __forceinline__ int attn_path(int np, int Lq, int Lk, int dh, long long B, int H, int mma_opt,
                                                  int mma_align) {
  if (np == 1 && Lq <= 16 && Lk <= 32 && (dh == 32 || dh == 48) && (mma_opt & 2) && mma_align) return AP_SMALL_MMA;
  if (Lq <= 32 && Lk <= 32) return AP_SMALL;
  if (np == 1 && Lq >= 64 && (dh == 32 || dh == 48 || dh == 64) && (mma_opt & 1) && mma_align) return AP_ROWS_MMA;
  if (Lk <= ATR_KMAX && Lq >= 64) return AP_ROWS;
  if (Lk > ATR_KMAX && B * H * ((Lq + 63) / 64) <= 148LL * 4) return AP_KSPLIT;
  return AP_TILED;
}

// Rows and lengths of problem b.  Varlen: false when this launch does not serve the item, or the query chunk starting at
// q0 is past its queries (block-uniform: b and q0 are).
struct AttnItem { long long qb, kb, vb, ob; int Lq, Lk; };
template <bool VARLEN>
__device__ __forceinline__ bool attn_item(const AttnParams& p, int b, int q0, AttnItem& it) {
  if (!VARLEN) {
    it.qb = b * p.q_sb; it.kb = b * p.k_sb; it.vb = b * p.v_sb; it.ob = b * p.o_sb; it.Lq = p.Lq; it.Lk = p.Lk;
    return true;
  }
  it.Lq = __ldg(p.q_len + b); it.Lk = __ldg(p.k_len + b);
  if (q0 >= it.Lq || it.Lk < 1) return false;
  const int group = p.groups ? __ldg(p.groups + b) : p.group;
  if (attn_path(p.np, it.Lq, it.Lk, p.dh, group, p.H, p.mma_opt, p.mma_align) != p.path) return false;
  const long long qo = __ldg(p.q_off + b), ko = __ldg(p.k_off + b);
  it.qb = qo * p.q_sb; it.kb = ko * p.k_sb; it.vb = ko * p.v_sb; it.ob = qo * p.o_sb;
  return true;
}
// One CTA per (batch item, head, chunk of ATT_QB queries): the query chunk and one tile of ATT_KT keys / values are staged
// in shared memory (coalesced 128-bit loads, rows padded by 4 floats so that lanes <-> keys read conflict-free
// LDS.128), every warp walks its queries over the tile with an online softmax (running max / sum / output, rescaled per
// tile), so K and V are read from L2 once per CTA instead of once per query (the first version of this kernel did the
// latter and was L2-bound: 215 us per launch on the 64 x 512 space attention, 4.5 of the 8 ms of a coarse forward).
constexpr int ATT_QB = 64, ATT_KT = 64, ATT_WARPS = 8;
template <int DH4, bool VARLEN>   // dh / 4 (dh <= 4 * DH4)
__global__ void __launch_bounds__(ATT_WARPS * 32) attention_kernel(const AttnParams p) {
  constexpr int DH = 4 * DH4, KLD = DH + 4;
  constexpr int QPW = ATT_QB / ATT_WARPS;   // queries per warp
  extern __shared__ __align__(16) float att_smem[];
  float* const Qs = att_smem;                       // [ATT_QB][DH]
  float* const Ks = Qs + ATT_QB * DH;               // [ATT_KT][KLD]
  float* const Vs = Ks + ATT_KT * KLD;              // [ATT_KT][DH]
  float (*Ps)[ATT_KT] = reinterpret_cast<float (*)[ATT_KT]>(Vs + ATT_KT * DH);   // [ATT_QB][ATT_KT]: one row per query of the chunk
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qchunks = (p.Lq + ATT_QB - 1) / ATT_QB;
  const long long nblocks = (long long)p.B * p.H * qchunks;
  for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
    const int qc = (int)(blk % qchunks);
    const int h = (int)((blk / qchunks) % p.H);
    const int b = (int)(blk / ((long long)qchunks * p.H));
    AttnItem it;
    if (!attn_item<VARLEN>(p, b, qc * ATT_QB, it)) continue;
    const int q0 = qc * ATT_QB, nq = min(ATT_QB, it.Lq - q0);
    const float* qp = p.q + it.qb + h * p.dh;
    const float* kp = p.k + it.kb + h * p.dh;
    const float* vp = p.v + it.vb + h * p.dh;
    const int dh4 = p.dh >> 2;
    __syncthreads();                       // previous chunk fully consumed
    for (int e = threadIdx.x; e < nq * DH4; e += blockDim.x) {
      const int r = e / DH4, t = e - r * DH4;
      float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t < dh4) g = __ldg(reinterpret_cast<const float4*>(qp + (long long)(q0 + r) * p.q_si) + t);
      g.x *= p.scale; g.y *= p.scale; g.z *= p.scale; g.w *= p.scale;     // MHA scales q before q k^T
      reinterpret_cast<float4*>(Qs)[r * DH4 + t] = g;
    }
    float m[QPW], l[QPW], acc0[QPW], acc1[QPW];
#pragma unroll
    for (int u = 0; u < QPW; ++u) { m[u] = -INFINITY; l[u] = 0.f; acc0[u] = 0.f; acc1[u] = 0.f; }
    // the QPW queries of a warp (qi = u * ATT_WARPS + warp) are processed TOGETHER per key tile: a K / V value is loaded
    // from shared memory once and used by all of them, and the QPW independent softmax / accumulation chains give the
    // scheduler instruction-level parallelism (one query at a time: 132 us on the 64 x 512 space attention, ncu r02).
    const int nmine = nq > warp ? (nq - warp + ATT_WARPS - 1) / ATT_WARPS : 0;     // warp-uniform

    for (int k0 = 0; k0 < it.Lk; k0 += ATT_KT) {
      const int nk = min(ATT_KT, it.Lk - k0);
      __syncthreads();                     // Q staged / previous tile consumed
      for (int e = threadIdx.x; e < ATT_KT * DH4; e += blockDim.x) {
        const int r = e / DH4, t = e - r * DH4;
        float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
        if (r < nk && t < dh4) {
          kk = __ldg(reinterpret_cast<const float4*>(kp + (long long)(k0 + r) * p.k_si) + t);
          vv = __ldg(reinterpret_cast<const float4*>(vp + (long long)(k0 + r) * p.v_si) + t);
        }
        *reinterpret_cast<float4*>(Ks + r * KLD + 4 * t) = kk;
        *reinterpret_cast<float4*>(Vs + r * DH + 4 * t) = vv;
      }
      __syncthreads();
      if (nmine > 0) {
        // scores of keys lane and lane + 32 for all queries of this warp
        float s0[QPW], s1[QPW];
#pragma unroll
        for (int u = 0; u < QPW; ++u) { s0[u] = 0.f; s1[u] = 0.f; }
        const float4* ka = reinterpret_cast<const float4*>(Ks + lane * KLD);
        const float4* kb = reinterpret_cast<const float4*>(Ks + (lane + 32) * KLD);
#pragma unroll
        for (int t = 0; t < DH4; ++t) {
          const float4 x = ka[t], y = kb[t];
#pragma unroll
          for (int u = 0; u < QPW; ++u) {
            if (u < nmine) {
              const float4 qv = reinterpret_cast<const float4*>(Qs + (u * ATT_WARPS + warp) * DH)[t];   // broadcast
              s0[u] = fmaf(qv.x, x.x, s0[u]); s0[u] = fmaf(qv.y, x.y, s0[u]); s0[u] = fmaf(qv.z, x.z, s0[u]); s0[u] = fmaf(qv.w, x.w, s0[u]);
              s1[u] = fmaf(qv.x, y.x, s1[u]); s1[u] = fmaf(qv.y, y.y, s1[u]); s1[u] = fmaf(qv.z, y.z, s1[u]); s1[u] = fmaf(qv.w, y.w, s1[u]);
            }
          }
        }
        __syncwarp();                      // previous tile's probabilities fully consumed
#pragma unroll
        for (int u = 0; u < QPW; ++u) {
          if (u < nmine) {
            if (lane >= nk) s0[u] = -INFINITY;
            if (lane + 32 >= nk) s1[u] = -INFINITY;
            const float mn = fmaxf(m[u], warp_max(fmaxf(s0[u], s1[u])));
            const float e0 = expf(s0[u] - mn), e1 = expf(s1[u] - mn);      // exp(-inf) = 0 for the padded keys
            const float corr = expf(m[u] - mn);                             // 0 on the first tile (m = -inf)
            l[u] = l[u] * corr + warp_sum(e0 + e1);
            m[u] = mn;
            acc0[u] *= corr; acc1[u] *= corr;
            Ps[warp * QPW + u][lane] = e0;
            Ps[warp * QPW + u][lane + 32] = e1;
          }
        }
        __syncwarp();
        // output dims lane and lane + 32: one V load serves all queries, probabilities are broadcast reads
        const int nk4 = (nk + 3) & ~3;      // padded keys carry probability 0 and zero V rows
        const float* v0 = Vs + (lane < DH ? lane : 0);
        const float* v1 = Vs + (lane + 32 < DH ? lane + 32 : 0);
        constexpr bool two = DH > 32;
#pragma unroll 1
        for (int j = 0; j < nk4; j += 4) {
          const float a0 = v0[j * DH], a1 = v0[(j + 1) * DH], a2 = v0[(j + 2) * DH], a3 = v0[(j + 3) * DH];
          float b0 = 0.f, b1 = 0.f, b2 = 0.f, b3 = 0.f;
          if (two) { b0 = v1[j * DH]; b1 = v1[(j + 1) * DH]; b2 = v1[(j + 2) * DH]; b3 = v1[(j + 3) * DH]; }
#pragma unroll
          for (int u = 0; u < QPW; ++u) {
            if (u < nmine) {
              const float4 pj = *reinterpret_cast<const float4*>(&Ps[warp * QPW + u][j]);
              acc0[u] = fmaf(pj.x, a0, acc0[u]); acc0[u] = fmaf(pj.y, a1, acc0[u]);
              acc0[u] = fmaf(pj.z, a2, acc0[u]); acc0[u] = fmaf(pj.w, a3, acc0[u]);
              if (two) {
                acc1[u] = fmaf(pj.x, b0, acc1[u]); acc1[u] = fmaf(pj.y, b1, acc1[u]);
                acc1[u] = fmaf(pj.z, b2, acc1[u]); acc1[u] = fmaf(pj.w, b3, acc1[u]);
              }
            }
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < QPW; ++u) {
      const int qi = u * ATT_WARPS + warp;
      if (qi >= nq) break;
      const float inv = 1.f / l[u];
      const long long base = it.ob + (long long)(q0 + qi) * p.o_si + h * p.dh;
      if (lane < p.dh) store_planes(p.out, p.o_plane_stride, base + lane, acc0[u] * inv, p.np);
      if (lane + 32 < p.dh) store_planes(p.out, p.o_plane_stride, base + lane + 32, acc1[u] * inv, p.np);
    }
  }
}

// Short sequences (Lq, Lk <= 32: the time attention, T = 16 frames per track): ONE WARP per (batch item, head), lane =
// query.  K and V of the (batch, head) are staged in the warp's shared-memory slice, every lane keeps its query row in
// registers, computes its Lk scores (K rows are broadcast reads), a softmax without any cross-lane traffic, and its
// output row; outputs go back through shared memory so that the plane stores are coalesced.  (The tiled kernel above
// spends a CTA with two block-wide barriers per (batch, head) on 16 x 16 scores: 113 us per launch for 4608 of them.)
constexpr int ATS_WARPS = 4;
template <int DH4, bool VARLEN>
__global__ void __launch_bounds__(ATS_WARPS * 32) attention_small_kernel(const AttnParams p) {
  constexpr int DH = 4 * DH4;
  extern __shared__ __align__(16) float ats_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int OLD = DH + 4;                                       // output row pitch: conflict-free 128-bit stores
  float* Ks = ats_smem + (size_t)warp * (32 * DH + 32 * OLD + 32 * 33);   // [32][DH]
  float* Vs = Ks + 32 * DH;                                         // [32][DH]; the region (32 x OLD) is reused for the output rows
  float* Ss = Vs + 32 * OLD;                                        // [Lk][33]: scores, one column per query lane
  const int dh4 = p.dh >> 2;
  const long long total = (long long)p.B * p.H;
  for (long long w = (long long)blockIdx.x * ATS_WARPS + warp; w < total; w += (long long)gridDim.x * ATS_WARPS) {
    const int h = (int)(w % p.H);
    const int b = (int)(w / p.H);
    AttnItem it;
    if (!attn_item<VARLEN>(p, b, 0, it)) continue;     // (warp-uniform)
    const int Lq = it.Lq, Lk = it.Lk;
    const float* qp = p.q + it.qb + h * p.dh;
    const float* kp = p.k + it.kb + h * p.dh;
    const float* vp = p.v + it.vb + h * p.dh;
    __syncwarp();
    for (int e = lane; e < Lk * DH4; e += 32) {
      const int r = e / DH4, t = e - r * DH4;
      float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
      if (t < dh4) {
        kk = __ldg(reinterpret_cast<const float4*>(kp + (long long)r * p.k_si) + t);
        vv = __ldg(reinterpret_cast<const float4*>(vp + (long long)r * p.v_si) + t);
      }
      reinterpret_cast<float4*>(Ks)[e] = kk;
      reinterpret_cast<float4*>(Vs)[e] = vv;
    }
    float4 q4[DH4];
    // At most 16 queries (the T = 16 time attention): both half-warps take the same queries and split the KEYS -- lanes
    // 0-15 the first half, lanes 16-31 the second -- and merge their running (max, sum, output row) with the online-softmax
    // rescale through 16-lane shuffles; otherwise half of the warp would idle through the whole (batch item, head).
    const bool split = Lq <= 16;
    const int qrow = split ? (lane & 15) : lane;
    const int khalf = (Lk + 1) >> 1;
    const int j0 = split ? (lane >> 4) * khalf : 0, jn = split ? khalf : Lk;
    const bool active = qrow < Lq;
#pragma unroll
    for (int t = 0; t < DH4; ++t) {
      q4[t] = (active && t < dh4) ? __ldg(reinterpret_cast<const float4*>(qp + (long long)qrow * p.q_si) + t)
                                  : make_float4(0.f, 0.f, 0.f, 0.f);
      q4[t].x *= p.scale; q4[t].y *= p.scale; q4[t].z *= p.scale; q4[t].w *= p.scale;   // MHA scales q before q k^T
    }
    __syncwarp();
    float mx = -INFINITY;
    for (int jj = 0; jj < jn; ++jj) {
      const int j = j0 + jj;
      if (j >= Lk) break;                // (odd Lk: the second half is one key shorter)
      const float4* kr = reinterpret_cast<const float4*>(Ks + j * DH);
      float sx = 0.f, sy = 0.f, sz = 0.f, sw = 0.f;      // four independent chains: one serial chain of dh FMAs is latency-bound
#pragma unroll
      for (int t = 0; t < DH4; ++t) {
        const float4 kk = kr[t];
        sx = fmaf(q4[t].x, kk.x, sx); sy = fmaf(q4[t].y, kk.y, sy); sz = fmaf(q4[t].z, kk.z, sz); sw = fmaf(q4[t].w, kk.w, sw);
      }
      const float sc = (sx + sy) + (sz + sw);
      Ss[j * 33 + lane] = sc;
      mx = fmaxf(mx, sc);
    }
    float4 acc[DH4];
#pragma unroll
    for (int t = 0; t < DH4; ++t) acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    float sum = 0.f;
    for (int jj = 0; jj < jn; ++jj) {
      const int j = j0 + jj;
      if (j >= Lk) break;
      const float pj = expf(Ss[j * 33 + lane] - mx);
      sum += pj;
      const float4* vr = reinterpret_cast<const float4*>(Vs + j * DH);
#pragma unroll
      for (int t = 0; t < DH4; ++t) {
        const float4 vv = vr[t];
        acc[t].x = fmaf(pj, vv.x, acc[t].x); acc[t].y = fmaf(pj, vv.y, acc[t].y);
        acc[t].z = fmaf(pj, vv.z, acc[t].z); acc[t].w = fmaf(pj, vv.w, acc[t].w);
      }
    }
    __syncwarp();
    if (split) {
      const float mo = __shfl_xor_sync(0xffffffffu, mx, 16), so = __shfl_xor_sync(0xffffffffu, sum, 16);
      const float m = fmaxf(mx, mo);
      const float e1 = expf(mx - m), e2 = expf(mo - m);      // a half without keys has max -inf and weight 0
      sum = sum * e1 + so * e2;
#pragma unroll
      for (int t = 0; t < DH4; ++t) {
        acc[t].x = acc[t].x * e1 + __shfl_xor_sync(0xffffffffu, acc[t].x, 16) * e2;
        acc[t].y = acc[t].y * e1 + __shfl_xor_sync(0xffffffffu, acc[t].y, 16) * e2;
        acc[t].z = acc[t].z * e1 + __shfl_xor_sync(0xffffffffu, acc[t].z, 16) * e2;
        acc[t].w = acc[t].w * e1 + __shfl_xor_sync(0xffffffffu, acc[t].w, 16) * e2;
      }
    }
    const float inv = 1.f / sum;
    __syncwarp();                          // every lane is done reading V before its rows are overwritten
    float* Os = Vs;                        // [32][OLD]
    if (active && (!split || lane < 16)) {
#pragma unroll
      for (int t = 0; t < DH4; ++t)
        *reinterpret_cast<float4*>(Os + lane * OLD + 4 * t) = make_float4(acc[t].x * inv, acc[t].y * inv, acc[t].z * inv, acc[t].w * inv);
    }
    __syncwarp();
    if (p.vec_out) {
      for (int e = lane; e < Lq * dh4; e += 32) {
        const int i = e / dh4, t = e - i * dh4;
        store_planes4(p.out, p.o_plane_stride, it.ob + (long long)i * p.o_si + h * p.dh + 4 * t,
                      *reinterpret_cast<const float4*>(Os + i * OLD + 4 * t), p.np);
      }
    } else
    for (int e = lane; e < Lq * p.dh; e += 32) {
      const int i = e / p.dh, d = e - i * p.dh;
      store_planes(p.out, p.o_plane_stride, it.ob + (long long)i * p.o_si + h * p.dh + d, Os[i * OLD + d], p.np);
    }
  }
}

// Few keys, many queries (Lk <= 64: points attending to the 64 virtual tracks, the virtual tracks' self attention):
// one CTA per (batch item, head, 128 queries); K and V of the (batch, head) are staged once per CTA, lane = query as in
// attention_small_kernel -- no cross-lane reductions, K / V rows are broadcast reads.  (The tiled kernel needs ~500
// instructions per query here, half of them warp reductions and probability traffic: 85 us per launch for the 512 x 64
// point -> virtual attention; this formulation needs ~250.)
constexpr int ATR_WARPS = 4;
template <int DH4, bool VARLEN>
__global__ void __launch_bounds__(ATR_WARPS * 32) attention_rows_kernel(const AttnParams p) {
  constexpr int DH = 4 * DH4, OLD = DH + 4;
  extern __shared__ __align__(16) float atr_smem[];
  float* Ks = atr_smem;                         // [ATR_KMAX][DH]
  float* Vs = Ks + ATR_KMAX * DH;               // [ATR_KMAX][DH]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* Ss = Vs + ATR_KMAX * DH + (size_t)warp * (ATR_KMAX * 33 + 32 * OLD);   // [Lk][33] scores of this warp's queries
  float* Os = Ss + ATR_KMAX * 33;               // [32][OLD] output rows of this warp
  const int dh4 = p.dh >> 2;
  const int qchunks = (p.Lq + ATR_WARPS * 32 - 1) / (ATR_WARPS * 32);
  const long long nblocks = (long long)p.B * p.H * qchunks;
  for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
    const int qc = (int)(blk % qchunks);
    const int h = (int)((blk / qchunks) % p.H);
    const int b = (int)(blk / ((long long)qchunks * p.H));
    AttnItem it;
    if (!attn_item<VARLEN>(p, b, qc * (ATR_WARPS * 32), it)) continue;
    const float* qp = p.q + it.qb + h * p.dh;
    const float* kp = p.k + it.kb + h * p.dh;
    const float* vp = p.v + it.vb + h * p.dh;
    __syncthreads();                            // previous chunk's K / V fully consumed
    for (int e = threadIdx.x; e < it.Lk * DH4; e += blockDim.x) {
      const int r = e / DH4, t = e - r * DH4;
      float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
      if (t < dh4) {
        kk = __ldg(reinterpret_cast<const float4*>(kp + (long long)r * p.k_si) + t);
        vv = __ldg(reinterpret_cast<const float4*>(vp + (long long)r * p.v_si) + t);
      }
      reinterpret_cast<float4*>(Ks)[e] = kk;
      reinterpret_cast<float4*>(Vs)[e] = vv;
    }
    const int qi = qc * (ATR_WARPS * 32) + warp * 32 + lane;
    const bool active = qi < it.Lq;
    float4 q4[DH4];
#pragma unroll
    for (int t = 0; t < DH4; ++t) {
      q4[t] = (active && t < dh4) ? __ldg(reinterpret_cast<const float4*>(qp + (long long)qi * p.q_si) + t)
                                  : make_float4(0.f, 0.f, 0.f, 0.f);
      q4[t].x *= p.scale; q4[t].y *= p.scale; q4[t].z *= p.scale; q4[t].w *= p.scale;
    }
    __syncthreads();
    float mx = -INFINITY;
    for (int j = 0; j < it.Lk; ++j) {
      const float4* kr = reinterpret_cast<const float4*>(Ks + j * DH);
      float sx = 0.f, sy = 0.f, sz = 0.f, sw = 0.f;      // four independent chains: one serial chain of dh FMAs is latency-bound
#pragma unroll
      for (int t = 0; t < DH4; ++t) {
        const float4 kk = kr[t];
        sx = fmaf(q4[t].x, kk.x, sx); sy = fmaf(q4[t].y, kk.y, sy); sz = fmaf(q4[t].z, kk.z, sz); sw = fmaf(q4[t].w, kk.w, sw);
      }
      const float sc = (sx + sy) + (sz + sw);
      Ss[j * 33 + lane] = sc;
      mx = fmaxf(mx, sc);
    }
    float4 acc[DH4];
#pragma unroll
    for (int t = 0; t < DH4; ++t) acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    float sum = 0.f;
    for (int j = 0; j < it.Lk; ++j) {
      const float pj = expf(Ss[j * 33 + lane] - mx);
      sum += pj;
      const float4* vr = reinterpret_cast<const float4*>(Vs + j * DH);
#pragma unroll
      for (int t = 0; t < DH4; ++t) {
        const float4 vv = vr[t];
        acc[t].x = fmaf(pj, vv.x, acc[t].x); acc[t].y = fmaf(pj, vv.y, acc[t].y);
        acc[t].z = fmaf(pj, vv.z, acc[t].z); acc[t].w = fmaf(pj, vv.w, acc[t].w);
      }
    }
    const float inv = 1.f / sum;
#pragma unroll
    for (int t = 0; t < DH4; ++t)
      *reinterpret_cast<float4*>(Os + lane * OLD + 4 * t) = make_float4(acc[t].x * inv, acc[t].y * inv, acc[t].z * inv, acc[t].w * inv);
    __syncwarp();
    const int q0w = qc * (ATR_WARPS * 32) + warp * 32;
    const int nqw = min(32, it.Lq - q0w);
    if (p.vec_out) {
      for (int e = lane; e < nqw * dh4; e += 32) {
        const int i = e / dh4, t = e - i * dh4;
        store_planes4(p.out, p.o_plane_stride, it.ob + (long long)(q0w + i) * p.o_si + h * p.dh + 4 * t,
                      *reinterpret_cast<const float4*>(Os + i * OLD + 4 * t), p.np);
      }
    } else
    for (int e = lane; e < nqw * p.dh; e += 32) {
      const int i = e / p.dh, d = e - i * p.dh;
      store_planes(p.out, p.o_plane_stride, it.ob + (long long)(q0w + i) * p.o_si + h * p.dh + d, Os[i * OLD + d], p.np);
    }
    __syncwarp();
  }
}

// At least 64 queries in AUTOCAST mode, any number of keys (tiles of 64 with the online-softmax rescale), on the tensor cores: under torch.autocast the reference's
// q / k / v are bf16 and its attention kernel multiplies in bf16 with float32 accumulation, so S = q k^T and O = P v run
// as mma.sync.m16n8k16 (bf16 x bf16 -> float32).  A warp owns 16 queries: S (16 x 64) stays in the accumulator
// registers, the softmax runs on them (a row lives in the four lanes of a quad: two shuffles per reduction), and the
// probabilities are repacked in registers into the A fragments of the second product -- the accumulator layout of two
// neighbouring 8-key tiles IS the A layout of one 16-key step.  K is staged as bf16 rows [key][dh + 8], V transposed
// [dim][64 + 8] (both pitches conflict-free for the 32-bit fragment loads).  The float32 lane-per-query kernel above
// spends ~250 instructions per query and head on this; here a warp issues 48 MMAs per 16 queries.
constexpr int ATM_WARPS = 8;
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}
template <int DH, bool VARLEN>   // head dimension, a multiple of 16
__global__ void __launch_bounds__(ATM_WARPS * 32) attention_rows_mma_kernel(const AttnParams p) {
  constexpr int KLD = DH + 8, VLD = 64 + 8, KS = DH / 16, DT = DH / 8;
  __shared__ __align__(16) __nv_bfloat16 Ks[64 * KLD];    // [key][dh]
  __shared__ __align__(16) __nv_bfloat16 Vt[DH * VLD];    // [dim][key]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int qchunks = (p.Lq + ATM_WARPS * 16 - 1) / (ATM_WARPS * 16);
  const long long nblocks = (long long)p.B * p.H * qchunks;
  for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
    const int qc = (int)(blk % qchunks);
    const int h = (int)((blk / qchunks) % p.H);
    const int b = (int)(blk / ((long long)qchunks * p.H));
    AttnItem it;
    if (!attn_item<VARLEN>(p, b, qc * (ATM_WARPS * 16), it)) continue;
    const int ktiles = (it.Lk + 63) / 64;        // more than 64 keys: tiles of 64 with the online-softmax rescale
    const float* qp = p.q + it.qb + h * DH;
    const float* kp = p.k + it.kb + h * DH;
    const float* vp = p.v + it.vb + h * DH;
    // this warp's 16 queries as A fragments (rows g and g + 8; MHA scales q before the product)
    const int q0 = qc * (ATM_WARPS * 16) + warp * 16;
    const int r0 = q0 + g, r1 = q0 + g + 8;
    uint32_t qa[KS][4];
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      float2 x00 = make_float2(0.f, 0.f), x01 = x00, x10 = x00, x11 = x00;
      if (r0 < it.Lq) {
        x00 = __ldg(reinterpret_cast<const float2*>(qp + (long long)r0 * p.q_si + ks * 16 + 2 * t));
        x01 = __ldg(reinterpret_cast<const float2*>(qp + (long long)r0 * p.q_si + ks * 16 + 2 * t + 8));
      }
      if (r1 < it.Lq) {
        x10 = __ldg(reinterpret_cast<const float2*>(qp + (long long)r1 * p.q_si + ks * 16 + 2 * t));
        x11 = __ldg(reinterpret_cast<const float2*>(qp + (long long)r1 * p.q_si + ks * 16 + 2 * t + 8));
      }
      qa[ks][0] = pack_bf16(x00.x * p.scale, x00.y * p.scale);
      qa[ks][1] = pack_bf16(x10.x * p.scale, x10.y * p.scale);
      qa[ks][2] = pack_bf16(x01.x * p.scale, x01.y * p.scale);
      qa[ks][3] = pack_bf16(x11.x * p.scale, x11.y * p.scale);
    }
    float oacc[DT][4];
#pragma unroll
    for (int dt = 0; dt < DT; ++dt) oacc[dt][0] = oacc[dt][1] = oacc[dt][2] = oacc[dt][3] = 0.f;
    float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;     // running max / sum of rows g and g + 8
#pragma unroll 1
    for (int kt = 0; kt < ktiles; ++kt) {
      const int key0 = kt * 64;
      __syncthreads();                          // the previous tile / block is fully consumed
      for (int e = threadIdx.x; e < 64 * (DH / 4); e += blockDim.x) {
        const int r = e / (DH / 4), c4 = e - r * (DH / 4);
        float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
        if (key0 + r < it.Lk) {
          kk = __ldg(reinterpret_cast<const float4*>(kp + (long long)(key0 + r) * p.k_si) + c4);
          vv = __ldg(reinterpret_cast<const float4*>(vp + (long long)(key0 + r) * p.v_si) + c4);
        }
        *reinterpret_cast<uint2*>(Ks + r * KLD + 4 * c4) = make_uint2(pack_bf16(kk.x, kk.y), pack_bf16(kk.z, kk.w));
        Vt[(4 * c4 + 0) * VLD + r] = __float2bfloat16_rn(vv.x);
        Vt[(4 * c4 + 1) * VLD + r] = __float2bfloat16_rn(vv.y);
        Vt[(4 * c4 + 2) * VLD + r] = __float2bfloat16_rn(vv.z);
        Vt[(4 * c4 + 3) * VLD + r] = __float2bfloat16_rn(vv.w);
      }
      __syncthreads();
      if (q0 >= it.Lq) continue;                 // warp-uniform: this warp only helps with the staging
      // S = q k^T: 8 key tiles of 8
      float sacc[8][4];
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        sacc[nt][0] = sacc[nt][1] = sacc[nt][2] = sacc[nt][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
          const __nv_bfloat16* kr = Ks + (nt * 8 + g) * KLD + ks * 16 + 2 * t;
          mma_bf16_16816(sacc[nt], qa[ks], *reinterpret_cast<const uint32_t*>(kr), *reinterpret_cast<const uint32_t*>(kr + 8));
        }
      }
      // softmax over the keys of rows g (c0, c1) and g + 8 (c2, c3); keys >= Lk are masked (every tile has a valid key)
      float t0 = -INFINITY, t1 = -INFINITY;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const int key = key0 + nt * 8 + 2 * t;
        if (key >= it.Lk) { sacc[nt][0] = -INFINITY; sacc[nt][2] = -INFINITY; }
        if (key + 1 >= it.Lk) { sacc[nt][1] = -INFINITY; sacc[nt][3] = -INFINITY; }
        t0 = fmaxf(t0, fmaxf(sacc[nt][0], sacc[nt][1]));
        t1 = fmaxf(t1, fmaxf(sacc[nt][2], sacc[nt][3]));
      }
      t0 = fmaxf(t0, __shfl_xor_sync(0xffffffffu, t0, 1)); t0 = fmaxf(t0, __shfl_xor_sync(0xffffffffu, t0, 2));
      t1 = fmaxf(t1, __shfl_xor_sync(0xffffffffu, t1, 1)); t1 = fmaxf(t1, __shfl_xor_sync(0xffffffffu, t1, 2));
      const float n0 = fmaxf(m0, t0), n1 = fmaxf(m1, t1);
      const float c0 = __expf(m0 - n0), c1 = __expf(m1 - n1);      // 0 on the first tile (running max -inf)
      m0 = n0; m1 = n1;
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        sacc[nt][0] = __expf(sacc[nt][0] - m0); sacc[nt][1] = __expf(sacc[nt][1] - m0);
        sacc[nt][2] = __expf(sacc[nt][2] - m1); sacc[nt][3] = __expf(sacc[nt][3] - m1);
        s0 += sacc[nt][0] + sacc[nt][1];
        s1 += sacc[nt][2] + sacc[nt][3];
      }
      s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
      s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
      l0 = l0 * c0 + s0; l1 = l1 * c1 + s1;
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) { oacc[dt][0] *= c0; oacc[dt][1] *= c0; oacc[dt][2] *= c1; oacc[dt][3] *= c1; }
      // O += P v: 4 steps of 16 keys, DT tiles of 8 dims
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        uint32_t pa[4];
        pa[0] = pack_bf16(sacc[2 * kk][0], sacc[2 * kk][1]);
        pa[1] = pack_bf16(sacc[2 * kk][2], sacc[2 * kk][3]);
        pa[2] = pack_bf16(sacc[2 * kk + 1][0], sacc[2 * kk + 1][1]);
        pa[3] = pack_bf16(sacc[2 * kk + 1][2], sacc[2 * kk + 1][3]);
#pragma unroll
        for (int dt = 0; dt < DT; ++dt) {
          const __nv_bfloat16* vr = Vt + (dt * 8 + g) * VLD + kk * 16 + 2 * t;
          mma_bf16_16816(oacc[dt], pa, *reinterpret_cast<const uint32_t*>(vr), *reinterpret_cast<const uint32_t*>(vr + 8));
        }
      }
    }
    if (q0 < it.Lq) {
      const float i0 = 1.f / l0, i1 = 1.f / l1;
      __nv_bfloat16* o0 = p.out + it.ob + (long long)r0 * p.o_si + h * DH + 2 * t;
      __nv_bfloat16* o1 = p.out + it.ob + (long long)r1 * p.o_si + h * DH + 2 * t;
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        if (r0 < it.Lq) *reinterpret_cast<uint32_t*>(o0 + dt * 8) = pack_bf16(oacc[dt][0] * i0, oacc[dt][1] * i0);
        if (r1 < it.Lq) *reinterpret_cast<uint32_t*>(o1 + dt * 8) = pack_bf16(oacc[dt][2] * i1, oacc[dt][3] * i1);
      }
    }
  }
}

// Short sequences (at most 16 queries, at most 32 keys: the T = 16 time attention) in AUTOCAST mode: one WARP per (batch
// item, head) as in attention_small_kernel, with the two products on the tensor cores as in attention_rows_mma_kernel --
// 12 + 12 MMAs instead of ~2000 FMA-pipe instructions.  K / V of the (batch, head) sit in the warp's own shared-memory
// slice (bf16; V transposed); no block-wide barrier.
constexpr int ATSM_WARPS = 4;
template <int DH, bool VARLEN>
__global__ void __launch_bounds__(ATSM_WARPS * 32) attention_small_mma_kernel(const AttnParams p) {
  constexpr int KLD = DH + 8, VLD = 32 + 8, KS = DH / 16, DT = DH / 8;
  __shared__ __align__(16) __nv_bfloat16 Ks_all[ATSM_WARPS][32 * KLD];    // [key][dh]
  __shared__ __align__(16) __nv_bfloat16 Vt_all[ATSM_WARPS][DH * VLD];    // [dim][key]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  __nv_bfloat16* Ks = Ks_all[warp];
  __nv_bfloat16* Vt = Vt_all[warp];
  const long long total = (long long)p.B * p.H;
  for (long long w = (long long)blockIdx.x * ATSM_WARPS + warp; w < total; w += (long long)gridDim.x * ATSM_WARPS) {
    const int h = (int)(w % p.H);
    const int b = (int)(w / p.H);
    AttnItem it;
    if (!attn_item<VARLEN>(p, b, 0, it)) continue;     // (warp-uniform)
    const int Lq = it.Lq, Lk = it.Lk;
    const float* qp = p.q + it.qb + h * DH;
    const float* kp = p.k + it.kb + h * DH;
    const float* vp = p.v + it.vb + h * DH;
    __syncwarp();                               // the previous (batch, head) is fully consumed
    for (int e = lane; e < 32 * (DH / 4); e += 32) {
      const int r = e / (DH / 4), c4 = e - r * (DH / 4);
      float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
      if (r < Lk) {
        kk = __ldg(reinterpret_cast<const float4*>(kp + (long long)r * p.k_si) + c4);
        vv = __ldg(reinterpret_cast<const float4*>(vp + (long long)r * p.v_si) + c4);
      }
      *reinterpret_cast<uint2*>(Ks + r * KLD + 4 * c4) = make_uint2(pack_bf16(kk.x, kk.y), pack_bf16(kk.z, kk.w));
      Vt[(4 * c4 + 0) * VLD + r] = __float2bfloat16_rn(vv.x);
      Vt[(4 * c4 + 1) * VLD + r] = __float2bfloat16_rn(vv.y);
      Vt[(4 * c4 + 2) * VLD + r] = __float2bfloat16_rn(vv.z);
      Vt[(4 * c4 + 3) * VLD + r] = __float2bfloat16_rn(vv.w);
    }
    const int r0 = g, r1 = g + 8;
    uint32_t qa[KS][4];
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      float2 x00 = make_float2(0.f, 0.f), x01 = x00, x10 = x00, x11 = x00;
      if (r0 < Lq) {
        x00 = __ldg(reinterpret_cast<const float2*>(qp + (long long)r0 * p.q_si + ks * 16 + 2 * t));
        x01 = __ldg(reinterpret_cast<const float2*>(qp + (long long)r0 * p.q_si + ks * 16 + 2 * t + 8));
      }
      if (r1 < Lq) {
        x10 = __ldg(reinterpret_cast<const float2*>(qp + (long long)r1 * p.q_si + ks * 16 + 2 * t));
        x11 = __ldg(reinterpret_cast<const float2*>(qp + (long long)r1 * p.q_si + ks * 16 + 2 * t + 8));
      }
      qa[ks][0] = pack_bf16(x00.x * p.scale, x00.y * p.scale);
      qa[ks][1] = pack_bf16(x10.x * p.scale, x10.y * p.scale);
      qa[ks][2] = pack_bf16(x01.x * p.scale, x01.y * p.scale);
      qa[ks][3] = pack_bf16(x11.x * p.scale, x11.y * p.scale);
    }
    __syncwarp();
    float sacc[4][4];
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      sacc[nt][0] = sacc[nt][1] = sacc[nt][2] = sacc[nt][3] = 0.f;
#pragma unroll
      for (int ks = 0; ks < KS; ++ks) {
        const __nv_bfloat16* kr = Ks + (nt * 8 + g) * KLD + ks * 16 + 2 * t;
        mma_bf16_16816(sacc[nt], qa[ks], *reinterpret_cast<const uint32_t*>(kr), *reinterpret_cast<const uint32_t*>(kr + 8));
      }
    }
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const int key = nt * 8 + 2 * t;
      if (key >= Lk) { sacc[nt][0] = -INFINITY; sacc[nt][2] = -INFINITY; }
      if (key + 1 >= Lk) { sacc[nt][1] = -INFINITY; sacc[nt][3] = -INFINITY; }
      m0 = fmaxf(m0, fmaxf(sacc[nt][0], sacc[nt][1]));
      m1 = fmaxf(m1, fmaxf(sacc[nt][2], sacc[nt][3]));
    }
    m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1)); m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
    m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      sacc[nt][0] = __expf(sacc[nt][0] - m0); sacc[nt][1] = __expf(sacc[nt][1] - m0);
      sacc[nt][2] = __expf(sacc[nt][2] - m1); sacc[nt][3] = __expf(sacc[nt][3] - m1);
      s0 += sacc[nt][0] + sacc[nt][1];
      s1 += sacc[nt][2] + sacc[nt][3];
    }
    s0 += __shfl_xor_sync(0xffffffffu, s0, 1); s0 += __shfl_xor_sync(0xffffffffu, s0, 2);
    s1 += __shfl_xor_sync(0xffffffffu, s1, 1); s1 += __shfl_xor_sync(0xffffffffu, s1, 2);
    float oacc[DT][4];
#pragma unroll
    for (int dt = 0; dt < DT; ++dt) oacc[dt][0] = oacc[dt][1] = oacc[dt][2] = oacc[dt][3] = 0.f;
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
      uint32_t pa[4];
      pa[0] = pack_bf16(sacc[2 * kk][0], sacc[2 * kk][1]);
      pa[1] = pack_bf16(sacc[2 * kk][2], sacc[2 * kk][3]);
      pa[2] = pack_bf16(sacc[2 * kk + 1][0], sacc[2 * kk + 1][1]);
      pa[3] = pack_bf16(sacc[2 * kk + 1][2], sacc[2 * kk + 1][3]);
#pragma unroll
      for (int dt = 0; dt < DT; ++dt) {
        const __nv_bfloat16* vr = Vt + (dt * 8 + g) * VLD + kk * 16 + 2 * t;
        mma_bf16_16816(oacc[dt], pa, *reinterpret_cast<const uint32_t*>(vr), *reinterpret_cast<const uint32_t*>(vr + 8));
      }
    }
    const float i0 = 1.f / s0, i1 = 1.f / s1;
    __nv_bfloat16* o0 = p.out + it.ob + (long long)r0 * p.o_si + h * DH + 2 * t;
    __nv_bfloat16* o1 = p.out + it.ob + (long long)r1 * p.o_si + h * DH + 2 * t;
#pragma unroll
    for (int dt = 0; dt < DT; ++dt) {
      if (r0 < Lq) *reinterpret_cast<uint32_t*>(o0 + dt * 8) = pack_bf16(oacc[dt][0] * i0, oacc[dt][1] * i0);
      if (r1 < Lq) *reinterpret_cast<uint32_t*>(o1 + dt * 8) = pack_bf16(oacc[dt][2] * i1, oacc[dt][3] * i1);
    }
  }
}

// Few queries, many keys (the 64 virtual tracks attending to all N point tracks): one CTA per (batch item, head,
// 64-query chunk), 8 warps = 2 query groups of 32 (lane = query, as in attention_rows_kernel) x 4 KEY SPLITS.  Every split
// walks its quarter of the keys in 64-key tiles (4 tiles staged at a time) with a per-lane online softmax; the four partial
// results (running max, sum, output row) of a query are merged through shared memory at the end.  (The tiled kernel gives
// this shape 128 CTAs of dependent warp reductions: 108 us per launch at N = 512.)
constexpr int AKS_SPLITS = 4, AKS_KT = 64;
template <int DH4, bool VARLEN>
__global__ void __launch_bounds__(256) attention_ksplit_kernel(const AttnParams p) {
  constexpr int DH = 4 * DH4, MP = DH + 8;       // merge row pitch: DH outputs, max, sum; a multiple of 4 floats (float4 rows)
  extern __shared__ __align__(16) float aks_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int grp = warp & 1, split = warp >> 1;
  float* Ks = aks_smem + (size_t)split * (2 * AKS_KT * DH);       // [AKS_KT][DH] of this split
  float* Vs = Ks + AKS_KT * DH;                                    // [AKS_KT][DH]
  float* Ss = aks_smem + (size_t)AKS_SPLITS * (2 * AKS_KT * DH) + (size_t)warp * (AKS_KT * 33);   // [AKS_KT][33]
  float* Mg = aks_smem;                                            // merge area (reuses the K / V tiles): [split][64][MP]
  const int dh4 = p.dh >> 2;
  const int qchunks = (p.Lq + 63) / 64;
  const long long nblocks = (long long)p.B * p.H * qchunks;
  for (long long blk = blockIdx.x; blk < nblocks; blk += gridDim.x) {
    const int qc = (int)(blk % qchunks);
    const int h = (int)((blk / qchunks) % p.H);
    const int b = (int)(blk / ((long long)qchunks * p.H));
    AttnItem it;
    if (!attn_item<VARLEN>(p, b, qc * 64, it)) continue;
    const int per_split = (((it.Lk + AKS_SPLITS - 1) / AKS_SPLITS) + AKS_KT - 1) / AKS_KT * AKS_KT;   // keys per split, tile multiple
    const float* qp = p.q + it.qb + h * p.dh;
    const float* kp = p.k + it.kb + h * p.dh;
    const float* vp = p.v + it.vb + h * p.dh;
    const int qi = qc * 64 + grp * 32 + lane;
    const bool active = qi < it.Lq;
    float4 q4[DH4];
#pragma unroll
    for (int t = 0; t < DH4; ++t) {
      q4[t] = (active && t < dh4) ? __ldg(reinterpret_cast<const float4*>(qp + (long long)qi * p.q_si) + t)
                                  : make_float4(0.f, 0.f, 0.f, 0.f);
      q4[t].x *= p.scale; q4[t].y *= p.scale; q4[t].z *= p.scale; q4[t].w *= p.scale;
    }
    float4 acc[DH4];
#pragma unroll
    for (int t = 0; t < DH4; ++t) acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
    float mrun = -INFINITY, lrun = 0.f;
    for (int t0 = 0; t0 < per_split; t0 += AKS_KT) {
      __syncthreads();                                 // previous tiles (or the previous block's merge area) consumed
      // stage tile t0 of every split: 4 x [AKS_KT][DH] of K and of V, all 256 threads
      for (int e = threadIdx.x; e < AKS_SPLITS * AKS_KT * DH4; e += blockDim.x) {
        const int sp = e / (AKS_KT * DH4), r = (e / DH4) % AKS_KT, t = e % DH4;
        const int key = sp * per_split + t0 + r;
        float4 kk = make_float4(0.f, 0.f, 0.f, 0.f), vv = kk;
        if (key < it.Lk && key < (sp + 1) * per_split && t < dh4) {
          kk = __ldg(reinterpret_cast<const float4*>(kp + (long long)key * p.k_si) + t);
          vv = __ldg(reinterpret_cast<const float4*>(vp + (long long)key * p.v_si) + t);
        }
        float* dstk = aks_smem + (size_t)sp * (2 * AKS_KT * DH);
        reinterpret_cast<float4*>(dstk)[r * DH4 + t] = kk;
        reinterpret_cast<float4*>(dstk + AKS_KT * DH)[r * DH4 + t] = vv;
      }
      __syncthreads();
      const int nk = max(0, min(AKS_KT, min(it.Lk, (split + 1) * per_split) - (split * per_split + t0)));   // warp-uniform
      if (nk > 0) {
        float mx = mrun;
        for (int j = 0; j < nk; ++j) {
          const float4* kr = reinterpret_cast<const float4*>(Ks + j * DH);
          float sx = 0.f, sy = 0.f, sz = 0.f, sw = 0.f;
#pragma unroll
          for (int t = 0; t < DH4; ++t) {
            const float4 kk = kr[t];
            sx = fmaf(q4[t].x, kk.x, sx); sy = fmaf(q4[t].y, kk.y, sy); sz = fmaf(q4[t].z, kk.z, sz); sw = fmaf(q4[t].w, kk.w, sw);
          }
          const float sc = (sx + sy) + (sz + sw);
          Ss[j * 33 + lane] = sc;
          mx = fmaxf(mx, sc);
        }
        const float corr = expf(mrun - mx);            // 0 on the first tile (mrun = -inf)
        lrun *= corr;
#pragma unroll
        for (int t = 0; t < DH4; ++t) { acc[t].x *= corr; acc[t].y *= corr; acc[t].z *= corr; acc[t].w *= corr; }
        mrun = mx;
        for (int j = 0; j < nk; ++j) {
          const float pj = expf(Ss[j * 33 + lane] - mx);
          lrun += pj;
          const float4* vr = reinterpret_cast<const float4*>(Vs + j * DH);
#pragma unroll
          for (int t = 0; t < DH4; ++t) {
            const float4 vv = vr[t];
            acc[t].x = fmaf(pj, vv.x, acc[t].x); acc[t].y = fmaf(pj, vv.y, acc[t].y);
            acc[t].z = fmaf(pj, vv.z, acc[t].z); acc[t].w = fmaf(pj, vv.w, acc[t].w);
          }
        }
      }
    }
    __syncthreads();                                   // all tiles consumed: the K / V area becomes the merge area
    {
      float* mine = Mg + ((size_t)split * 64 + grp * 32 + lane) * MP;
#pragma unroll
      for (int t = 0; t < DH4; ++t) *reinterpret_cast<float4*>(mine + 4 * t) = acc[t];
      mine[DH] = mrun;
      mine[DH + 1] = lrun;
    }
    __syncthreads();
    if (split == 0) {
      float M = -INFINITY;
#pragma unroll
      for (int sp = 0; sp < AKS_SPLITS; ++sp) M = fmaxf(M, Mg[((size_t)sp * 64 + grp * 32 + lane) * MP + DH]);
      float L = 0.f;
#pragma unroll
      for (int t = 0; t < DH4; ++t) acc[t] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int sp = 0; sp < AKS_SPLITS; ++sp) {
        const float* o = Mg + ((size_t)sp * 64 + grp * 32 + lane) * MP;
        const float w = expf(o[DH] - M);              // 0 for a split that saw no key (m = -inf)
        L = fmaf(o[DH + 1], w, L);
#pragma unroll
        for (int t = 0; t < DH4; ++t) {
          const float4 a = *reinterpret_cast<const float4*>(o + 4 * t);
          acc[t].x = fmaf(a.x, w, acc[t].x); acc[t].y = fmaf(a.y, w, acc[t].y);
          acc[t].z = fmaf(a.z, w, acc[t].z); acc[t].w = fmaf(a.w, w, acc[t].w);
        }
      }
      const float inv = 1.f / L;
      __syncwarp();
      float* Os = Mg + ((size_t)grp * 32) * MP;     // this group's split-0 rows, now free: output staging
#pragma unroll
      for (int t = 0; t < DH4; ++t)
        *reinterpret_cast<float4*>(Os + lane * MP + 4 * t) = make_float4(acc[t].x * inv, acc[t].y * inv, acc[t].z * inv, acc[t].w * inv);
      __syncwarp();
      const int q0w = qc * 64 + grp * 32;
      const int nqw = min(32, it.Lq - q0w);
      if (p.vec_out) {
        for (int e = lane; e < nqw * (p.dh >> 2); e += 32) {
          const int i = e / (p.dh >> 2), t = e - i * (p.dh >> 2);
          store_planes4(p.out, p.o_plane_stride, it.ob + (long long)(q0w + i) * p.o_si + h * p.dh + 4 * t,
                        *reinterpret_cast<const float4*>(Os + i * MP + 4 * t), p.np);
        }
      } else
      for (int e = lane; e < nqw * p.dh; e += 32) {
        const int i = e / p.dh, d = e - i * p.dh;
        store_planes(p.out, p.o_plane_stride, it.ob + (long long)(q0w + i) * p.o_si + h * p.dh + d, Os[i * MP + d], p.np);
      }
    }
  }
}

// y = a + b (elementwise, float32, contiguous) -- the "tokens + init_tokens" before the flow head, written as planes
__global__ void __launch_bounds__(256) add_planes_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                          __nv_bfloat16* __restrict__ planes, long long plane_stride, int np,
                                                          long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    store_planes(planes, plane_stride, i, __ldg(a + i) + __ldg(b + i), np);
}

}  // namespace comet

using namespace comet;

extern "C" int comet_layernorm_planes_f32(const float* x, long long x_ld, const float* gamma, const float* beta, float eps,
                                          float* out, long long out_ld, void* planes, long long plane_stride, long long p_ld,
                                          int np, long long rows, int D, comet_stream_t stream) {
  COMET_REQUIRE(rows >= 0 && D >= 1 && D <= 32 * LN_MAX_PER_LANE, "LayerNorm width %d outside [1, %d]", D, 32 * LN_MAX_PER_LANE);
  COMET_REQUIRE(np == 0 || np == 1 || np == 3, "np must be 0, 1 or 3");
  COMET_REQUIRE((gamma == nullptr) == (beta == nullptr), "gamma and beta must be given together");
  if (rows == 0) return COMET_OK;
  COMET_REQUIRE(x && (out || (planes && np > 0)), "null pointer");
  long long blocks = (rows + 7) / 8;
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  __nv_bfloat16* pl = np > 0 ? reinterpret_cast<__nv_bfloat16*>(planes) : nullptr;
  const bool v4 = (D % 4) == 0 && D <= 512 && (x_ld % 4) == 0 && ((uintptr_t)x % 16) == 0 &&
                  (!out || ((out_ld % 4) == 0 && ((uintptr_t)out % 16) == 0)) &&
                  (!pl || ((p_ld % 4) == 0 && (plane_stride % 4) == 0 && ((uintptr_t)pl % 8) == 0)) &&
                  (!gamma || (((uintptr_t)gamma % 16) == 0 && ((uintptr_t)beta % 16) == 0));
  if (v4) {
#define COMET_LN4_LAUNCH(KG)                                                                                        \
  layernorm_planes_v4_kernel<KG><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, x_ld, gamma, beta, eps, out, out_ld, pl, \
                                                                                     plane_stride, p_ld, np, rows, D)
    if (D <= 128) COMET_LN4_LAUNCH(1);
    else if (D <= 256) COMET_LN4_LAUNCH(2);
    else if (D <= 384) COMET_LN4_LAUNCH(3);
    else COMET_LN4_LAUNCH(4);
#undef COMET_LN4_LAUNCH
    return launch_status("layernorm_planes_v4_kernel");
  }
#define COMET_LN_LAUNCH(KPL)                                                                                        \
  layernorm_planes_kernel<KPL><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(x, x_ld, gamma, beta, eps, out, out_ld, pl, \
                                                                                  plane_stride, p_ld, np, rows, D)
  if (D <= 32) COMET_LN_LAUNCH(1);
  else if (D <= 128) COMET_LN_LAUNCH(4);
  else if (D <= 256) COMET_LN_LAUNCH(8);
  else if (D <= 384) COMET_LN_LAUNCH(12);
  else if (D <= 512) COMET_LN_LAUNCH(16);
  else COMET_LN_LAUNCH(32);
#undef COMET_LN_LAUNCH
  return launch_status("layernorm_planes_kernel");
}

// One launch of kernel family `path` over p.B problems (grid sized from the largest query length p.Lq).
template <bool VARLEN>
static int launch_attention(int path, const AttnParams& p, cudaStream_t stream) {
  const long long B = p.B;
  const int H = p.H, Lq = p.Lq, dh = p.dh;
  if (path == AP_SMALL_MMA) {
    long long nb = (B * H + ATSM_WARPS - 1) / ATSM_WARPS;
    if (nb > 148LL * 16) nb = 148LL * 16;
    if (dh == 32) attention_small_mma_kernel<32, VARLEN><<<(unsigned)nb, ATSM_WARPS * 32, 0, stream>>>(p);
    else attention_small_mma_kernel<48, VARLEN><<<(unsigned)nb, ATSM_WARPS * 32, 0, stream>>>(p);
    return launch_status("attention_small_mma_kernel");
  }
  if (path == AP_SMALL) {
    long long nb = (B * H + ATS_WARPS - 1) / ATS_WARPS;
    if (nb > 148LL * 16) nb = 148LL * 16;
#define COMET_ATS_LAUNCH(D4)                                                                                       \
  do {                                                                                                             \
    const int smem = ATS_WARPS * (32 * 4 * D4 + 32 * (4 * D4 + 4) + 32 * 33) * (int)sizeof(float);                 \
    if (smem > 48 * 1024)                                                                                          \
      COMET_CUDA(cudaFuncSetAttribute(attention_small_kernel<D4, VARLEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
    attention_small_kernel<D4, VARLEN><<<(unsigned)nb, ATS_WARPS * 32, smem, stream>>>(p);                                 \
  } while (0)
    if (dh <= 4) COMET_ATS_LAUNCH(1);
    else if (dh <= 16) COMET_ATS_LAUNCH(4);
    else if (dh <= 32) COMET_ATS_LAUNCH(8);
    else if (dh <= 48) COMET_ATS_LAUNCH(12);
    else COMET_ATS_LAUNCH(16);
#undef COMET_ATS_LAUNCH
    return launch_status("attention_small_kernel");
  }
  if (path == AP_ROWS_MMA) {
    long long nb = B * H * ((Lq + ATM_WARPS * 16 - 1) / (ATM_WARPS * 16));
    if (nb > 148LL * 16) nb = 148LL * 16;
    if (dh == 32) attention_rows_mma_kernel<32, VARLEN><<<(unsigned)nb, ATM_WARPS * 32, 0, stream>>>(p);
    else if (dh == 48) attention_rows_mma_kernel<48, VARLEN><<<(unsigned)nb, ATM_WARPS * 32, 0, stream>>>(p);
    else attention_rows_mma_kernel<64, VARLEN><<<(unsigned)nb, ATM_WARPS * 32, 0, stream>>>(p);
    return launch_status("attention_rows_mma_kernel");
  }
  if (path == AP_ROWS) {
    long long nb = B * H * ((Lq + ATR_WARPS * 32 - 1) / (ATR_WARPS * 32));
    if (nb > 148LL * 16) nb = 148LL * 16;
#define COMET_ATR_LAUNCH(D4)                                                                                       \
  do {                                                                                                             \
    const int smem = (2 * ATR_KMAX * 4 * D4 + ATR_WARPS * (ATR_KMAX * 33 + 32 * (4 * D4 + 4))) * (int)sizeof(float); \
    if (smem > 48 * 1024)                                                                                          \
      COMET_CUDA(cudaFuncSetAttribute(attention_rows_kernel<D4, VARLEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
    attention_rows_kernel<D4, VARLEN><<<(unsigned)nb, ATR_WARPS * 32, smem, stream>>>(p);                                  \
  } while (0)
    if (dh <= 4) COMET_ATR_LAUNCH(1);
    else if (dh <= 16) COMET_ATR_LAUNCH(4);
    else if (dh <= 32) COMET_ATR_LAUNCH(8);
    else if (dh <= 48) COMET_ATR_LAUNCH(12);
    else COMET_ATR_LAUNCH(16);
#undef COMET_ATR_LAUNCH
    return launch_status("attention_rows_kernel");
  }
  if (path == AP_KSPLIT) {
    long long nb = B * H * ((Lq + 63) / 64);
    if (nb > 148LL * 16) nb = 148LL * 16;   // (a single call takes this path only at <= 148 * 4 CTAs)
#define COMET_AKS_LAUNCH(D4)                                                                                       \
  do {                                                                                                             \
    const int smem = (AKS_SPLITS * 2 * AKS_KT * 4 * D4 + 8 * AKS_KT * 33) * (int)sizeof(float);                    \
    if (smem > 48 * 1024)                                                                                          \
      COMET_CUDA(cudaFuncSetAttribute(attention_ksplit_kernel<D4, VARLEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem)); \
    attention_ksplit_kernel<D4, VARLEN><<<(unsigned)nb, 256, smem, stream>>>(p);                                           \
  } while (0)
    if (dh <= 4) COMET_AKS_LAUNCH(1);
    else if (dh <= 16) COMET_AKS_LAUNCH(4);
    else if (dh <= 32) COMET_AKS_LAUNCH(8);
    else if (dh <= 48) COMET_AKS_LAUNCH(12);
    else COMET_AKS_LAUNCH(16);
#undef COMET_AKS_LAUNCH
    return launch_status("attention_ksplit_kernel");
  }
  long long blocks = B * H * ((Lq + ATT_QB - 1) / ATT_QB);
  if (blocks > 148LL * 16) blocks = 148LL * 16;
#define COMET_ATTN_LAUNCH(D4)                                                                                       \
  do {                                                                                                              \
    const int smem = (ATT_QB * 4 * D4 + ATT_KT * (4 * D4 + 4) + ATT_KT * 4 * D4 + ATT_QB * ATT_KT) * (int)sizeof(float); \
    if (smem > 48 * 1024)                                                                                           \
      COMET_CUDA(cudaFuncSetAttribute(attention_kernel<D4, VARLEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));    \
    attention_kernel<D4, VARLEN><<<(unsigned)blocks, ATT_WARPS * 32, smem, stream>>>(p);                                    \
  } while (0)
  if (dh <= 4) COMET_ATTN_LAUNCH(1);
  else if (dh <= 16) COMET_ATTN_LAUNCH(4);
  else if (dh <= 32) COMET_ATTN_LAUNCH(8);
  else if (dh <= 48) COMET_ATTN_LAUNCH(12);
  else COMET_ATTN_LAUNCH(16);
#undef COMET_ATTN_LAUNCH
  return launch_status("attention_kernel");
}

static int mma_alignment(long long q_sb, long long q_si, long long o_sb, long long o_si, const void* out_planes) {
  return (o_sb % 2 == 0 && o_si % 2 == 0 && ((uintptr_t)out_planes % 4) == 0 && q_si % 2 == 0 && q_sb % 2 == 0) ? 1 : 0;
}

extern "C" int comet_attention_planes_f32(const float* q, long long q_sb, long long q_si, const float* k, long long k_sb,
                                          long long k_si, const float* v, long long v_sb, long long v_si, void* out_planes,
                                          long long o_plane_stride, long long o_sb, long long o_si, int np, int B, int H,
                                          int Lq, int Lk, int dh, comet_stream_t stream) {
  COMET_REQUIRE(B >= 0 && H >= 1 && Lq >= 0 && Lk >= 1 && dh >= 4 && dh <= 64 && dh % 4 == 0,
                "bad attention shape (B=%d H=%d Lq=%d Lk=%d dh=%d)", B, H, Lq, Lk, dh);
  COMET_REQUIRE(np == 1 || np == 3, "np must be 1 or 3");
  const long long total = (long long)B * H * Lq;
  if (total == 0) return COMET_OK;
  COMET_REQUIRE(q && k && v && out_planes, "null pointer");
  COMET_REQUIRE(((uintptr_t)q % 16) == 0 && ((uintptr_t)k % 16) == 0 && q_sb % 4 == 0 && q_si % 4 == 0 && k_sb % 4 == 0 &&
                    k_si % 4 == 0, "q / k rows must be 16-byte aligned");
  COMET_REQUIRE(((uintptr_t)v % 16) == 0 && v_sb % 4 == 0 && v_si % 4 == 0, "v rows must be 16-byte aligned");
  AttnParams p{q, q_sb, q_si, k, k_sb, k_si, v, v_sb, v_si, reinterpret_cast<__nv_bfloat16*>(out_planes),
               o_plane_stride, o_sb, o_si, np, B, H, Lq, Lk, dh, 1.0f / sqrtf((float)dh),
               (o_sb % 4 == 0 && o_si % 4 == 0 && o_plane_stride % 4 == 0 && ((uintptr_t)out_planes % 8) == 0) ? 1 : 0};
  const int path = attn_path(np, Lq, Lk, dh, B, H, option(COMET_OPT_ATTN_MMA),
                             mma_alignment(q_sb, q_si, o_sb, o_si, out_planes));
  return launch_attention<false>(path, p, (cudaStream_t)stream);
}

extern "C" int comet_attention_varlen_grouped_planes_f32(const float* q, long long q_ld, long long q_step, const float* k,
                                                         long long k_ld, long long k_step, const float* v, void* out_planes,
                                                         long long o_plane_stride, long long o_ld, int np, int items, int H,
                                                         int dh, const int* q_off, const int* q_len, const int* k_off,
                                                         const int* k_len, int min_lq, int max_lq, int min_lk, int max_lk,
                                                         const int* groups, int min_group, int max_group,
                                                         comet_stream_t stream) {
  COMET_REQUIRE(items >= 0 && H >= 1 && min_lq >= 0 && max_lq >= min_lq && min_lk >= 0 && max_lk >= min_lk &&
                    min_group >= 1 && max_group >= min_group && (groups || min_group == max_group) && dh >= 4 && dh <= 64 &&
                    dh % 4 == 0,
                "bad varlen attention shape (items=%d H=%d Lq in [%d, %d] Lk in [%d, %d] group in [%d, %d] dh=%d)", items, H,
                min_lq, max_lq, min_lk, max_lk, min_group, max_group, dh);
  COMET_REQUIRE(np == 1 || np == 3, "np must be 1 or 3");
  if ((long long)items * max_lq * max_lk == 0) return COMET_OK;
  COMET_REQUIRE(q && k && v && out_planes && q_off && q_len && k_off && k_len, "null pointer");
  COMET_REQUIRE(((uintptr_t)q % 16) == 0 && ((uintptr_t)k % 16) == 0 && ((uintptr_t)v % 16) == 0 && q_ld % 4 == 0 &&
                    k_ld % 4 == 0, "q / k / v rows must be 16-byte aligned");
  AttnParams p{q, q_ld, q_step * q_ld, k, k_ld, k_step * k_ld, v, k_ld, k_step * k_ld,
               reinterpret_cast<__nv_bfloat16*>(out_planes), o_plane_stride, o_ld, q_step * o_ld, np, items, H, max_lq,
               max_lk, dh, 1.0f / sqrtf((float)dh),
               (o_ld % 4 == 0 && (q_step * o_ld) % 4 == 0 && o_plane_stride % 4 == 0 && ((uintptr_t)out_planes % 8) == 0) ? 1 : 0};
  p.q_off = q_off; p.q_len = q_len; p.k_off = k_off; p.k_len = k_len;
  p.group = max_group;
  p.groups = groups;
  p.mma_opt = option(COMET_OPT_ATTN_MMA);
  p.mma_align = mma_alignment(q_ld, q_step * q_ld, o_ld, q_step * o_ld, out_planes);
  // The lengths live on the device: launch every family that some (length pair, group) of the given ranges selects (the
  // path depends on a length only through the thresholds 16 / 32 / 64 and the number of 64-query chunks, so every length
  // up to 65 and then every 64th is enough; on the group only through one upper bound, so both ends are enough).  Items
  // of length 0 select no family; each CTA serves the items of its own family.
  auto next = [](int x, int hi) { return x < 65 ? x + 1 : x < hi ? (x + 64 < hi ? x + 64 : hi) : hi + 1; };
  bool used[AP_COUNT] = {};
  for (int lq = min_lq > 1 ? min_lq : 1; lq <= max_lq; lq = next(lq, max_lq))
    for (int lk = min_lk > 1 ? min_lk : 1; lk <= max_lk; lk = next(lk, max_lk))
      for (int g : {min_group, max_group}) used[attn_path(np, lq, lk, dh, g, H, p.mma_opt, p.mma_align)] = true;
  for (int path = 0; path < AP_COUNT; ++path) {
    if (!used[path]) continue;
    p.path = path;
    const int rc = launch_attention<true>(path, p, (cudaStream_t)stream);
    if (rc != COMET_OK) return rc;
  }
  return COMET_OK;
}

extern "C" int comet_attention_varlen_planes_f32(const float* q, long long q_ld, long long q_step, const float* k,
                                                 long long k_ld, long long k_step, const float* v, void* out_planes,
                                                 long long o_plane_stride, long long o_ld, int np, int items, int H, int dh,
                                                 const int* q_off, const int* q_len, const int* k_off, const int* k_len,
                                                 int min_lq, int max_lq, int min_lk, int max_lk, int group,
                                                 comet_stream_t stream) {
  COMET_REQUIRE(min_lq >= 1 && min_lk >= 1, "bad varlen attention lengths (Lq in [%d, %d], Lk in [%d, %d])", min_lq, max_lq,
                min_lk, max_lk);
  return comet_attention_varlen_grouped_planes_f32(q, q_ld, q_step, k, k_ld, k_step, v, out_planes, o_plane_stride, o_ld, np,
                                                   items, H, dh, q_off, q_len, k_off, k_len, min_lq, max_lq, min_lk, max_lk,
                                                   nullptr, group, group, stream);
}

extern "C" int comet_add_planes_f32(const float* a, const float* b, void* planes, long long plane_stride, int np, long long n,
                                    comet_stream_t stream) {
  COMET_REQUIRE(n >= 0 && (np == 1 || np == 3), "bad arguments");
  if (n == 0) return COMET_OK;
  COMET_REQUIRE(a && b && planes, "null pointer");
  long long blocks = (n + 255) / 256;
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  add_planes_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(a, b, reinterpret_cast<__nv_bfloat16*>(planes), plane_stride, np, n);
  return launch_status("add_planes_kernel");
}
