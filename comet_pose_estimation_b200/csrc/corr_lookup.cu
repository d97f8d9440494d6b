// Fused correlation + multi-level window lookup (+ optional track-token epilogue), SIMT float32.
//
// Replaces CorrBlock.corr + CorrBlock.sample (comet/models/track_modules/blocks.py:376-429),
// EfficientCorrBlock.sample (blocks.py:446-484) and, with TOKENS, the token assembly of
// BaseTrackerPredictor.forward (base_track_predictor.py:165-224).
//
// Formulation.  Every entry of the (2r+1)^2 window of level l is a bilinear blend of the correlation
// volume V_l at four integer taps, and all entries share the same fractional offsets, so the window
// only needs V_l on a (2r+2)^2 integer grid around the query.  One warp owns one (b, s, n) query:
//   1. lanes <- grid positions; each lane accumulates dot(T[b,s,n,:], F_l[b,s,:,y,x]) over channels
//      (target vector broadcast from shared memory, feature reads coalesced along x);
//   2. the grid goes to shared memory, lanes <- window entries, blend, coalesced store.
// The volume is never written to global memory.  This is the general path (any C, H, W, L, r<=7, both
// padding modes, strided views) and the HBM-bound path of the fine tracker (one query per map, GEMV-shaped);
// the dense coarse shapes go through the tcgen05 kernel in corr_tc.cu when available.
#include "lookup_common.cuh"

#include <cuda.h>
#include <cstdlib>
#include <cstring>

namespace comet {

// element strides of level l: channel, row, column
__device__ __forceinline__ void level_strides(const LookupParams& p, int l, long long& sc, int& sy, int& sx) {
  if (p.channel_last && (l > 0 || p.cl0)) { sc = 1; sy = p.lvlW[l] * p.C; sx = p.C; }
  else { sc = (long long)p.lvlH[l] * p.lvlW[l]; sy = p.lvlW[l]; sx = 1; }
}

template <int KPL, bool TOKENS>
__global__ void __launch_bounds__(256) corr_lookup_kernel(const LookupParams p) {
  extern __shared__ float smem[];
  const int warps_per_block = blockDim.x >> 5;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int G = 2 * p.r + 2, Wr = 2 * p.r + 1;
  const int GG = G * G, WW = Wr * Wr;
  float* Ts = smem + (size_t)warp * (p.C + GG);  // target vector of this warp's query
  float* Vs = Ts + p.C;                          // (2r+2)^2 grid of correlations

  const long long q = (long long)blockIdx.x * warps_per_block + warp;
  const long long total = (long long)p.B * p.S * p.N;
  if (q >= total) return;
  const int n = (int)(q % p.N);
  const int s = (int)((q / p.N) % p.S);
  const int b = (int)(q / ((long long)p.N * p.S));
  long long bs = (long long)b * p.S + s;
  if (TOKENS && p.fidx) bs = min(max(__ldg(p.fidx + bs), 0), p.BS_src - 1);   // the frame this (item, position) reads
  if (TOKENS && ((p.ntr && n >= __ldg(p.ntr + b)) || (p.nfr && s >= __ldg(p.nfr + b)))) {   // padded query / frame: zero row
    float* zp = p.out + (((long long)b * p.N + n) * p.S + s) * p.D_tok;
    for (int d = lane; d < p.D_tok; d += 32) zp[d] = 0.f;
    return;
  }

  const float* cp = p.coords + b * p.c_sb + s * p.c_ss + n * p.c_sn;
  const float cx = __ldg(cp), cy = __ldg(cp + 1);
  const float* tp = p.targets + b * p.t_sb + s * p.t_ss + n * p.t_sn;

  float* op;
  const float* pp = nullptr;
  int corr_off = 0;
  if (TOKENS) {
    op = p.out + (((long long)b * p.N + n) * p.S + s) * p.D_tok;
    pp = p.pos + ((long long)b * p.N + n) * p.D_tok;
    corr_off = p.C + 2;
  } else {
    op = p.out + b * p.o_sb + s * p.o_ss + n * p.o_sn;
  }

  for (int l = 0; l < p.L; ++l) {
    const int Hl = p.lvlH[l], Wl = p.lvlW[l];
    const long long HW = (long long)Hl * Wl;
    const float* F = (l == 0 ? p.fmaps : p.pyr + p.lvlOff[l]) + bs * p.C * HW;
    long long sc; int sy, sx;
    level_strides(p, l, sc, sy, sx);

    // stage the target vector (per level only when multiple_track_feats splits channels)
    if (l == 0 || p.t_level_stride != 0) {
      __syncwarp();
      const float* tl = tp + (long long)l * p.t_level_stride;
      for (int c = lane; c < p.C; c += 32) {
        float t = __ldg(tl + c);
        Ts[c] = p.bf16 ? round_bf16(t) : t;
      }
      __syncwarp();
    }

    const float inv = 1.f / (float)(1 << l);
    AxisWindow ax, ay;
    ax.init(cx * inv, Wl, p.r, p.pad_border);
    ay.init(cy * inv, Hl, p.r, p.pad_border);

    // 1. correlations on the integer grid
    long long offs[KPL];
    bool ok[KPL];
    float acc[KPL];
#pragma unroll
    for (int k = 0; k < KPL; ++k) {
      const int idx = lane + 32 * k;
      int gx = 0, gy = 0;
      bool v = idx < GG;
      if (v) {
        const int a = idx / G, bb = idx - a * G;
        const bool vx = ax.tap(bb, gx), vy = ay.tap(a, gy);
        v = vx && vy;
      }
      ok[k] = v;
      offs[k] = v ? (long long)gy * sy + (long long)gx * sx : 0;
      acc[k] = 0.f;
    }
    if (!p.bf16) {
#pragma unroll 4
      for (int c = 0; c < p.C; ++c) {
        const float t = Ts[c];
        const float* Fc = F + (long long)c * sc;
#pragma unroll
        for (int k = 0; k < KPL; ++k)
          if (ok[k]) acc[k] = fmaf(t, __ldg(Fc + offs[k]), acc[k]);
      }
    } else {
#pragma unroll 4
      for (int c = 0; c < p.C; ++c) {
        const float t = Ts[c];
        const float* Fc = F + (long long)c * sc;
#pragma unroll
        for (int k = 0; k < KPL; ++k)
          if (ok[k]) acc[k] = fmaf(t, round_bf16(__ldg(Fc + offs[k])), acc[k]);
      }
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < KPL; ++k) {
      const int idx = lane + 32 * k;
      if (idx < GG) {
        float v = acc[k];
        if (p.bf16) v = round_bf16(v);           // matmul result is stored in bf16 under autocast
        v = __fdiv_rn(v, p.sqrt_c);              // blocks.py:428 divides after the matmul
        if (p.bf16) v = round_bf16(v);
        Vs[idx] = ok[k] ? v : 0.f;
      }
    }
    __syncwarp();

    // 2. blend: out[l*WW + i*Wr + j], i <-> x offset (slow), j <-> y offset (fast)
    for (int o = lane; o < WW; o += 32) {
      const int i = o / Wr, j = o - i * Wr;
      float wx0, wx1, wy0, wy1;
      ax.weights(i, wx0, wx1);
      ay.weights(j, wy0, wy1);
      const float* v = Vs + j * G + i;
      // ATen accumulation order: nw, ne, sw, se
      float val = v[0] * (wx0 * wy0);
      val += v[1] * (wx1 * wy0);
      val += v[G] * (wx0 * wy1);
      val += v[G + 1] * (wx1 * wy1);
      const int d = corr_off + l * WW + o;
      if (TOKENS) val += __ldg(pp + d);
      op[d] = val;
    }
  }

  if (TOKENS) {
    // [ sin/cos(flow * div) (C) | flow (2) | fcorrs | track_feats (C) | zero pad ] + pos_emb
    // get_2d_embedding (utils.py:65-101) with C_emb = latent/2, called at base_track_predictor.py:176-181.
    const float* c0 = p.coords + b * p.c_sb + n * p.c_sn;  // frame 0
    const float fx = cx - __ldg(c0), fy = cy - __ldg(c0 + 1);
    const int Ce = p.C >> 1;
    const float step = 1000.0f / (float)Ce;
    for (int e = lane; e < p.C; e += 32) {
      const int axis = e / Ce, w = e - axis * Ce;
      const float div = (float)(w & ~1) * step;
      const float arg = __fmul_rn(axis ? fy : fx, div);
      const float v = (w & 1) ? cosf(arg) : sinf(arg);
      op[e] = v + __ldg(pp + e);
    }
    if (lane < 2) op[p.C + lane] = (lane ? fy : fx) + __ldg(pp + p.C + lane);
    const int feat_off = corr_off + p.L * WW;
    for (int c = lane; c < p.C; c += 32) op[feat_off + c] = __ldg(tp + c) + __ldg(pp + feat_off + c);
    for (int d = feat_off + p.C + lane; d < p.D_tok; d += 32) op[d] = __ldg(pp + d);
  }
}

// ---- specialisation for the fine tracker: C == 32, compile-time radius R <= 3 (<= 64 grid positions) -----------
// One warp per query, lanes <-> grid positions (2 per lane: rows a and a + G/2 of the same column), so all tap /
// address arithmetic is done once per level and everything else is loads + FMAs (the first version of this kernel
// was issue-bound: 6800 instructions per query, a quarter of them integer index math).
//   level 0  (caller's NCHW map)     : per channel one uniform plane pointer, two scalar gathers per lane;
//   level>=1 (channel-last pyramid)  : the 32 channels of a position are one 128-byte line -> 8 x LDG.128 at
//                                      immediate offsets per position, target vector read as LDS.128 broadcasts.
template <int R, bool TOKENS, bool BF16>
__global__ void __launch_bounds__(256, 2) corr_lookup_c32_kernel(const LookupParams p) {
  constexpr int G = 2 * R + 2, Wr = 2 * R + 1, GG = G * G, WW = Wr * Wr;
  constexpr int ROWS0 = (GG + 31) / 32;  // grid positions per lane (2 for R=3, 1 for R=1)
  __shared__ __align__(16) float Ts_all[8][32];
  __shared__ float Vs_all[8][GG <= 32 ? 32 : 64];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* Ts = Ts_all[warp];
  float* Vs = Vs_all[warp];

  const long long q = (long long)blockIdx.x * 8 + warp;
  const long long total = (long long)p.B * p.S * p.N;
  if (q >= total) return;
  const int n = (int)(q % p.N);
  const int s = (int)((q / p.N) % p.S);
  const int b = (int)(q / ((long long)p.N * p.S));
  long long bs = (long long)b * p.S + s;
  if (TOKENS && p.fidx) bs = min(max(__ldg(p.fidx + bs), 0), p.BS_src - 1);   // the frame this (item, position) reads

  const float* cp = p.coords + b * p.c_sb + s * p.c_ss + n * p.c_sn;
  const float cx = __ldg(cp), cy = __ldg(cp + 1);
  const float* tp = p.targets + b * p.t_sb + s * p.t_ss + n * p.t_sn;
  {
    const float t = __ldg(tp + lane);
    Ts[lane] = BF16 ? round_bf16(t) : t;
  }
  __syncwarp();

  float* op;
  const float* pp = nullptr;
  int corr_off = 0;
  if (TOKENS) {
    op = p.out + (((long long)b * p.N + n) * p.S + s) * p.D_tok;
    pp = p.pos + ((long long)b * p.N + n) * p.D_tok;
    corr_off = 32 + 2;
  } else {
    op = p.out + b * p.o_sb + s * p.o_ss + n * p.o_sn;
  }
  // (a one-warp-per-(query, level) variant was measured slower: the kernel sits at the DRAM transaction limit, so
  //  what pays is memory-level parallelism per warp -- all 64 level-0 gathers of a lane are issued back to back)
#pragma unroll 1
  for (int l = 0; l < p.L; ++l) {
    const int Hl = p.lvlH[l], Wl = p.lvlW[l];
    const int HW = Hl * Wl;
    const float* F = (l == 0 ? p.fmaps : p.pyr + p.lvlOff[l]) + bs * 32 * (long long)HW;
    const float inv = 1.f / (float)(1 << l);
    AxisWindow ax, ay;
    ax.init(cx * inv, Wl, R, p.pad_border);
    ay.init(cy * inv, Hl, R, p.pad_border);

    int pos[ROWS0];
    bool ok[ROWS0];
    float acc[ROWS0];
#pragma unroll
    for (int k = 0; k < ROWS0; ++k) {
      const int idx = lane + 32 * k;
      int gx = 0, gy = 0;
      const bool vx = ax.tap(idx % G, gx), vy = ay.tap(idx / G, gy);
      ok[k] = idx < GG && vx && vy;
      pos[k] = ok[k] ? gy * Wl + gx : 0;
      acc[k] = 0.f;
    }
    if (p.channel_last && (l > 0 || p.cl0)) {
#pragma unroll
      for (int k = 0; k < ROWS0; ++k) {
        const float4* v4 = reinterpret_cast<const float4*>(F) + (long long)pos[k] * 8;
        float4 f[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = __ldg(v4 + i);  // pos = 0 (valid memory) when the tap is masked
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 t = *reinterpret_cast<const float4*>(Ts + 4 * i);
          float4 g = f[i];
          if (BF16) round_bf16x4(g);
          acc[k] = fmaf(t.x, g.x, acc[k]);
          acc[k] = fmaf(t.y, g.y, acc[k]);
          acc[k] = fmaf(t.z, g.z, acc[k]);
          acc[k] = fmaf(t.w, g.w, acc[k]);
        }
      }
    } else {
      float f[ROWS0][32];
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const float* Fc = F + (long long)c * HW;  // warp-uniform plane pointer
#pragma unroll
        for (int k = 0; k < ROWS0; ++k) f[k][c] = __ldg(Fc + pos[k]);
      }
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const float t = Ts[c];
#pragma unroll
        for (int k = 0; k < ROWS0; ++k) acc[k] = fmaf(t, BF16 ? round_bf16(f[k][c]) : f[k][c], acc[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < ROWS0; ++k) {
      const int idx = lane + 32 * k;
      if (idx < GG) {
        float v = acc[k];
        if (BF16) v = round_bf16(v);
        v = __fdiv_rn(v, p.sqrt_c);
        if (BF16) v = round_bf16(v);
        Vs[idx] = ok[k] ? v : 0.f;
      }
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < (WW + 31) / 32; ++k) {
      const int o = lane + 32 * k;
      if (o < WW) {
        const int i = o / Wr, j = o - i * Wr;
        float wx0, wx1, wy0, wy1;
        ax.weights(i, wx0, wx1);
        ay.weights(j, wy0, wy1);
        const float* v = Vs + j * G + i;
        float val = v[0] * (wx0 * wy0);
        val += v[1] * (wx1 * wy0);
        val += v[G] * (wx0 * wy1);
        val += v[G + 1] * (wx1 * wy1);
        const int d = corr_off + l * WW + o;
        if (TOKENS) val += __ldg(pp + d);
        op[d] = val;
      }
    }
    __syncwarp();
  }

  if (TOKENS) {
    const float* c0 = p.coords + b * p.c_sb + n * p.c_sn;  // frame 0
    const float fx = cx - __ldg(c0), fy = cy - __ldg(c0 + 1);
    const int w = lane & 15;                               // C_emb = 16: [pe_x (16) | pe_y (16)]
    const float arg = __fmul_rn(lane >= 16 ? fy : fx, (float)(w & ~1) * (1000.0f / 16.f));
    op[lane] = ((w & 1) ? cosf(arg) : sinf(arg)) + __ldg(pp + lane);
    if (lane < 2) op[32 + lane] = (lane ? fy : fx) + __ldg(pp + 32 + lane);
    const int feat_off = corr_off + p.L * WW;
    op[feat_off + lane] = __ldg(tp + lane) + __ldg(pp + feat_off + lane);
    for (int d = feat_off + 32 + lane; d < p.D_tok; d += 32) op[d] = __ldg(pp + d);
  }
}


// ---- TMA-staged variant of the C == 32 kernel (the fine tracker's hot kernel) -------------------------------------
// The register version above walks the levels one after the other: three dependent DRAM round trips per query, so it
// is latency-bound (62 % of the HBM rate even with every sector fully used).  Here one elected lane per warp issues
// ONE 4-D TMA box load per channel-last level -- box = [32 channels x G x G positions] around the query, out-of-map
// positions zero-filled by the TMA unit (= the reference's zero padding), landing in shared memory with the 128-byte
// swizzle -- so all levels of a query are in flight at once and no address arithmetic or predicate is spent on them.
// A level-0 map in the caller's NCHW layout (CL0 == false) is gathered through registers while the boxes fly.
// Then lanes <-> grid positions read "their" 128-byte line (swizzle makes the 8 lanes of a quarter-warp hit 8 different
// bank groups), dot it with the target vector held in registers, and the blend / token epilogue is the one above.
// Persistent: 8 warps per SM, each owns 3 box buffers (24 KB at r = 3) and loops over queries.

template <int R, bool TOKENS, bool BF16, bool CL0>
__global__ void __launch_bounds__(256, 1) corr_lookup_c32_tma_kernel(const __grid_constant__ TmaMaps maps, const LookupParams p) {
  constexpr int G = 2 * R + 2, Wr = 2 * R + 1, GG = G * G, WW = Wr * Wr;
  constexpr int ROWS0 = (GG + 31) / 32;
  constexpr int BOX = GG * 128;                      // bytes landed per level
  constexpr int BOXP = (BOX + 1023) & ~1023;         // swizzle atoms are 1 KB
  extern __shared__ __align__(1024) uint8_t smem_tma[];
  uint8_t* const smem = smem_tma;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* mybox = smem + warp * 3 * BOXP;
  float* Ts = reinterpret_cast<float*>(smem + 8 * 3 * BOXP) + warp * 32;
  float* Vs = reinterpret_cast<float*>(smem + 8 * 3 * BOXP + 8 * 32 * 4) + warp * 64;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 8 * 3 * BOXP + 8 * 32 * 4 + 8 * 64 * 4) + warp;
  if (lane == 0) {
    tma::mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  uint32_t phase = 0;
  const long long total = (long long)p.B * p.S * p.N;
  const long long nwarps = (long long)gridDim.x * 8;
  const int l_first = CL0 ? 0 : 1;   // first level that arrives by TMA

  // software pipeline over queries: coordinates / target of query i+1 are fetched while query i is processed, so the
  // only global latency a warp waits for is its own TMA boxes
  auto fetch = [&](long long q_, float& cx_, float& cy_, float& fx0_, float& fy0_, float& tl_) {
    cx_ = cy_ = fx0_ = fy0_ = tl_ = 0.f;
    if (q_ < total) {
      const int n_ = (int)(q_ % p.N);
      const int s_ = (int)((q_ / p.N) % p.S);
      const int b_ = (int)(q_ / ((long long)p.N * p.S));
      const float* cp = p.coords + b_ * p.c_sb + s_ * p.c_ss + n_ * p.c_sn;
      cx_ = __ldg(cp); cy_ = __ldg(cp + 1);
      if (TOKENS) {
        const float* c0 = p.coords + b_ * p.c_sb + n_ * p.c_sn;  // frame 0
        fx0_ = __ldg(c0); fy0_ = __ldg(c0 + 1);
      }
      tl_ = __ldg(p.targets + b_ * p.t_sb + s_ * p.t_ss + n_ * p.t_sn + lane);
    }
  };
  float cx, cy, cx0, cy0, tl;
  fetch((long long)blockIdx.x * 8 + warp, cx, cy, cx0, cy0, tl);

  for (long long q = (long long)blockIdx.x * 8 + warp; q < total; q += nwarps) {
    const int n = (int)(q % p.N);
    const int s = (int)((q / p.N) % p.S);
    const int b = (int)(q / ((long long)p.N * p.S));
    int bs = b * p.S + s;
    if (TOKENS && p.fidx) bs = min(max(__ldg(p.fidx + bs), 0), p.BS_src - 1);
    AxisWindow ax[3], ay[3];
#pragma unroll
    for (int l = 0; l < 3; ++l) {
      if (l < p.L) {
        const float inv = 1.f / (float)(1 << l);
        ax[l].init(cx * inv, p.lvlW[l], R, p.pad_border);
        ay[l].init(cy * inv, p.lvlH[l], R, p.pad_border);
      }
    }
    // box origins: zeros -> the unclamped window corner (the TMA unit zero-fills what is off the map);
    //              border -> the clamped corner (every clamped tap then lies inside the box)
    int ox[3], oy[3];
#pragma unroll
    for (int l = 0; l < 3; ++l) {
      if (l < p.L) {
        ox[l] = p.pad_border ? min(max(ax[l].i0, 0), p.lvlW[l] - 1) : min(max(ax[l].i0, -G), p.lvlW[l]);
        oy[l] = p.pad_border ? min(max(ay[l].i0, 0), p.lvlH[l] - 1) : min(max(ay[l].i0, -G), p.lvlH[l]);
      }
    }
    __syncwarp();   // every lane is done with the boxes / Ts / Vs of the previous query
    if (lane == 0) {
      tma::mbar_expect_tx(bar, (uint32_t)((p.L - l_first) * BOX));
#pragma unroll
      for (int l = 0; l < 3; ++l)
        if (l >= l_first && l < p.L) tma::load_box_4d(&maps.m[l], bar, mybox + l * BOXP, 0, ox[l], oy[l], bs);
    }
    Ts[lane] = BF16 ? round_bf16(tl) : tl;
    const float tl_cur = tl, fx = cx - cx0, fy = cy - cy0;
    float cx_n, cy_n, cx0_n, cy0_n, tl_n;
    fetch(q + nwarps, cx_n, cy_n, cx0_n, cy0_n, tl_n);

    float* op;
    const float* pp = nullptr;
    int corr_off = 0;
    constexpr int NB = (WW + 31) / 32;
    float pv[3][NB], pe0 = 0.f, pe1 = 0.f, pe2 = 0.f, pe3 = 0.f;   // position-embedding values of this token row, fetched up front
    if (TOKENS) {
      op = p.out + (((long long)b * p.N + n) * p.S + s) * p.D_tok;
      pp = p.pos + ((long long)b * p.N + n) * p.D_tok;
      corr_off = 32 + 2;
#pragma unroll
      for (int l = 0; l < 3; ++l)
#pragma unroll
        for (int k = 0; k < NB; ++k) pv[l][k] = (l < p.L && lane + 32 * k < WW) ? __ldg(pp + corr_off + l * WW + lane + 32 * k) : 0.f;
      pe0 = __ldg(pp + lane);
      pe1 = lane < 2 ? __ldg(pp + 32 + lane) : 0.f;
      pe2 = __ldg(pp + corr_off + p.L * WW + lane);
      pe3 = (corr_off + p.L * WW + 32 + lane < p.D_tok) ? __ldg(pp + corr_off + p.L * WW + 32 + lane) : 0.f;
    } else {
      op = p.out + b * p.o_sb + s * p.o_ss + n * p.o_sn;
#pragma unroll
      for (int l = 0; l < 3; ++l)
#pragma unroll
        for (int k = 0; k < NB; ++k) pv[l][k] = 0.f;
    }
    __syncwarp();
    float4 t4[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t4[i] = *reinterpret_cast<const float4*>(Ts + 4 * i);

    float acc0[ROWS0];
    bool ok0[ROWS0];
    if (!CL0) {
      // level 0 in the caller's NCHW layout: per channel one warp-uniform plane pointer, gathers in flight with the boxes
      const int Hl = p.lvlH[0], Wl = p.lvlW[0];
      const int HW = Hl * Wl;
      const float* F = p.fmaps + (long long)bs * 32 * HW;
      int pos[ROWS0];
#pragma unroll
      for (int k = 0; k < ROWS0; ++k) {
        const int idx = lane + 32 * k;
        int gx = 0, gy = 0;
        const bool vx = ax[0].tap(idx % G, gx), vy = ay[0].tap(idx / G, gy);
        ok0[k] = idx < GG && vx && vy;
        pos[k] = ok0[k] ? gy * Wl + gx : 0;
        acc0[k] = 0.f;
      }
      float f[ROWS0][32];
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const float* Fc = F + (long long)c * HW;
#pragma unroll
        for (int k = 0; k < ROWS0; ++k) f[k][c] = __ldg(Fc + pos[k]);
      }
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const float t = reinterpret_cast<const float*>(t4)[c];
#pragma unroll
        for (int k = 0; k < ROWS0; ++k) acc0[k] = fmaf(t, BF16 ? round_bf16(f[k][c]) : f[k][c], acc0[k]);
      }
    }

    tma::mbar_wait(bar, phase);
    phase ^= 1;

#pragma unroll
    for (int l = 0; l < 3; ++l) {
      if (l < p.L) {
        float acc[ROWS0];
        bool ok[ROWS0];
        if (l == 0 && !CL0) {
#pragma unroll
          for (int k = 0; k < ROWS0; ++k) { acc[k] = acc0[k]; ok[k] = ok0[k]; }
        } else {
          const uint8_t* box = mybox + l * BOXP;
#pragma unroll
          for (int k = 0; k < ROWS0; ++k) {
            const int idx = lane + 32 * k;
            int gx = 0, gy = 0;
            const bool vx = ax[l].tap(idx % G, gx), vy = ay[l].tap(idx / G, gy);
            ok[k] = idx < GG && vx && vy;
            const int slot = ok[k] ? (gy - oy[l]) * G + (gx - ox[l]) : 0;
            const uint8_t* line = box + slot * 128;
            const int sw = slot & 7;
            float a = 0.f;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              float4 g = *reinterpret_cast<const float4*>(line + ((i ^ sw) << 4));
              if (BF16) round_bf16x4(g);
              a = fmaf(t4[i].x, g.x, a);
              a = fmaf(t4[i].y, g.y, a);
              a = fmaf(t4[i].z, g.z, a);
              a = fmaf(t4[i].w, g.w, a);
            }
            acc[k] = a;
          }
        }
#pragma unroll
        for (int k = 0; k < ROWS0; ++k) {
          const int idx = lane + 32 * k;
          if (idx < GG) {
            float v = acc[k];
            if (BF16) v = round_bf16(v);
            v = __fdiv_rn(v, p.sqrt_c);
            if (BF16) v = round_bf16(v);
            Vs[idx] = ok[k] ? v : 0.f;
          }
        }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < (WW + 31) / 32; ++k) {
          const int o = lane + 32 * k;
          if (o < WW) {
            const int i = o / Wr, j = o - i * Wr;
            float wx0, wx1, wy0, wy1;
            ax[l].weights(i, wx0, wx1);
            ay[l].weights(j, wy0, wy1);
            const float* v = Vs + j * G + i;
            float val = v[0] * (wx0 * wy0);
            val += v[1] * (wx1 * wy0);
            val += v[G] * (wx0 * wy1);
            val += v[G + 1] * (wx1 * wy1);
            const int d = corr_off + l * WW + o;
            op[d] = val + pv[l][k];
          }
        }
        __syncwarp();
      }
    }

    if (TOKENS) {
      const int w = lane & 15;                               // C_emb = 16: [pe_x (16) | pe_y (16)]
      const float arg = __fmul_rn(lane >= 16 ? fy : fx, (float)(w & ~1) * (1000.0f / 16.f));
      op[lane] = ((w & 1) ? cosf(arg) : sinf(arg)) + pe0;
      if (lane < 2) op[32 + lane] = (lane ? fy : fx) + pe1;
      const int feat_off = corr_off + p.L * WW;
      op[feat_off + lane] = tl_cur + pe2;
      if (feat_off + 32 + lane < p.D_tok) op[feat_off + 32 + lane] = pe3;          // zero pad + pos_emb
      for (int d = feat_off + 64 + lane; d < p.D_tok; d += 32) op[d] = __ldg(pp + d);
    }
    cx = cx_n; cy = cy_n; cx0 = cx0_n; cy0 = cy0_n; tl = tl_n;
  }
}

constexpr int tma_smem_bytes(int R) {
  const int G = 2 * R + 2;
  const int boxp = (G * G * 128 + 1023) & ~1023;
  return 8 * 3 * boxp + 8 * 32 * 4 + 8 * 64 * 4 + 8 * 8;
}

template <int R, bool TOKENS>
static int launch_c32_tma(const LookupParams& p, const TmaMaps& maps, int grid, cudaStream_t stream) {
  const int smem = tma_smem_bytes(R);
#define COMET_TMA_LAUNCH(BF, CL)                                                                               \
  do {                                                                                                         \
    COMET_CUDA(cudaFuncSetAttribute(corr_lookup_c32_tma_kernel<R, TOKENS, BF, CL>,                             \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, smem));                       \
    corr_lookup_c32_tma_kernel<R, TOKENS, BF, CL><<<grid, 256, smem, stream>>>(maps, p);                       \
  } while (0)
  if (p.bf16) { if (p.cl0) COMET_TMA_LAUNCH(true, true); else COMET_TMA_LAUNCH(true, false); }
  else { if (p.cl0) COMET_TMA_LAUNCH(false, true); else COMET_TMA_LAUNCH(false, false); }
#undef COMET_TMA_LAUNCH
  return launch_status("corr_lookup_c32_tma_kernel");
}

template <int R, bool TOKENS>
static void launch_c32(const LookupParams& p, unsigned blocks, cudaStream_t stream) {
  if (p.bf16) corr_lookup_c32_kernel<R, TOKENS, true><<<blocks, 256, 0, stream>>>(p);
  else corr_lookup_c32_kernel<R, TOKENS, false><<<blocks, 256, 0, stream>>>(p);
}

template <bool TOKENS>
static int launch_lookup(const LookupParams& p, cudaStream_t stream) {
  const int G = 2 * p.r + 2;
  const int kpl = (G * G + 31) / 32;
  const int warps = 8;
  const size_t smem = (size_t)warps * (p.C + G * G) * sizeof(float);
  const long long total = (long long)p.B * p.S * p.N;
  if (total == 0) return COMET_OK;
  const long long blocks = (total + warps - 1) / warps;
  if (blocks > 0x7fffffffLL) return fail(COMET_ERR_UNSUPPORTED, "too many queries for one launch");
  if (p.C == 32 && p.r >= 1 && p.r <= 3 && p.t_level_stride == 0 && ((uintptr_t)p.pyr % 16) == 0 &&
      (!p.cl0 || ((uintptr_t)p.fmaps % 16) == 0)) {
    if (p.ntr || p.nfr)
      return fail(COMET_ERR_UNSUPPORTED, "per-sequence query / frame counts are served by the generic lookup kernel (C != 32) "
                                         "and, frame counts, by COMET_PYR_UP2_SOURCE");
    const bool use_tma = option(COMET_OPT_TMA_LOOKUP) && device_sm_count_if_sm100() > 0 && tensor_map_encoder() != nullptr;
    if (use_tma && p.cl0 && p.L <= 3 && total < (1LL << 40)) {
      TmaMaps maps;
      memset(&maps, 0, sizeof(maps));
      const int G2 = 2 * p.r + 2;
      for (int l = p.cl0 ? 0 : 1; l < p.L; ++l) {
        const float* base = l == 0 ? p.fmaps : p.pyr + p.lvlOff[l];
        int rc = encode_level_map(&maps.m[l], base, p.fidx ? p.BS_src : p.B * p.S, p.lvlH[l], p.lvlW[l], G2);
        if (rc != COMET_OK) return rc;
      }
      const int sms = device_sm_count_if_sm100();
      const long long want = (total + 7) / 8;
      const int grid = (int)(want < sms ? want : sms);
      if (p.r == 3) return launch_c32_tma<3, TOKENS>(p, maps, grid, stream);
      if (p.r == 2) return launch_c32_tma<2, TOKENS>(p, maps, grid, stream);
      return launch_c32_tma<1, TOKENS>(p, maps, grid, stream);
    }
    if (p.r == 3) launch_c32<3, TOKENS>(p, (unsigned)blocks, stream);
    else if (p.r == 2) launch_c32<2, TOKENS>(p, (unsigned)blocks, stream);
    else launch_c32<1, TOKENS>(p, (unsigned)blocks, stream);
    return launch_status("corr_lookup_c32_kernel");
  }
  if (smem > 200 * 1024) return fail(COMET_ERR_UNSUPPORTED, "C=%d too large for the lookup kernel", p.C);
#define COMET_LAUNCH(K)                                                                                   \
  do {                                                                                                    \
    if (smem > 48 * 1024)                                                                                 \
      COMET_CUDA(cudaFuncSetAttribute(corr_lookup_kernel<K, TOKENS>,                                      \
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));           \
    corr_lookup_kernel<K, TOKENS><<<(unsigned)blocks, warps * 32, smem, stream>>>(p);                     \
  } while (0)
  if (kpl <= 1) COMET_LAUNCH(1);
  else if (kpl <= 2) COMET_LAUNCH(2);
  else if (kpl <= 4) COMET_LAUNCH(4);
  else COMET_LAUNCH(8);
#undef COMET_LAUNCH
  return launch_status("corr_lookup_kernel");
}

static int fill_params(LookupParams& p, const float* fmaps, const float* pyr, const float* targets, long long t_sb,
                       long long t_ss, long long t_sn, int t_level_stride, const float* coords, long long c_sb,
                       long long c_ss, long long c_sn, int B, int S, int N, int C, int H, int W, int L, int r,
                       int pad_mode, int prec_mode, int pyr_layout) {
  COMET_REQUIRE(B >= 0 && S >= 0 && N >= 0, "negative batch dimension");
  COMET_REQUIRE(C >= 1 && H >= 1 && W >= 1, "C, H, W must be positive (got %d, %d, %d)", C, H, W);
  COMET_REQUIRE(L >= 1 && L <= COMET_MAX_LEVELS, "num_levels must be in [1, %d] (got %d)", COMET_MAX_LEVELS, L);
  COMET_REQUIRE(r >= 0 && r <= COMET_MAX_RADIUS, "radius must be in [0, %d] (got %d)", COMET_MAX_RADIUS, r);
  COMET_REQUIRE(pad_mode == COMET_PAD_ZEROS || pad_mode == COMET_PAD_BORDER, "bad pad_mode %d", pad_mode);
  COMET_REQUIRE(prec_mode == COMET_PREC_F32 || prec_mode == COMET_PREC_BF16_AUTOCAST, "bad prec_mode %d", prec_mode);
  COMET_REQUIRE(pyr_layout == COMET_PYR_NCHW || pyr_layout == COMET_PYR_CHANNEL_LAST ||
                    pyr_layout == COMET_PYR_ALL_CHANNEL_LAST || pyr_layout == COMET_PYR_UP2_SOURCE,
                "bad pyr_layout %d", pyr_layout);
  COMET_REQUIRE((H >> (L - 1)) >= 1 && (W >> (L - 1)) >= 1, "map %dx%d too small for %d levels", H, W, L);
  const long long total = (long long)B * S * N;
  COMET_REQUIRE(total == 0 || (fmaps && targets && coords), "null input pointer");
  COMET_REQUIRE(total == 0 || L == 1 || pyr, "pyr is null but num_levels > 1");
  p.fmaps = fmaps; p.pyr = pyr; p.targets = targets;
  p.t_sb = t_sb; p.t_ss = t_ss; p.t_sn = t_sn; p.t_level_stride = t_level_stride;
  p.coords = coords; p.c_sb = c_sb; p.c_ss = c_ss; p.c_sn = c_sn;
  p.B = B; p.S = S; p.N = N; p.C = C; p.L = L; p.r = r;
  p.pad_border = pad_mode == COMET_PAD_BORDER;
  p.bf16 = prec_mode == COMET_PREC_BF16_AUTOCAST;
  Levels lv = make_levels(B * S, C, H, W, L);
  for (int l = 0; l < L; ++l) { p.lvlH[l] = lv.H[l]; p.lvlW[l] = lv.W[l]; p.lvlOff[l] = lv.off[l]; }
  p.sqrt_c = sqrtf((float)C);
  p.inv_sqrt_c = 1.0f / p.sqrt_c;
  p.channel_last = pyr_layout != COMET_PYR_NCHW;
  p.cl0 = pyr_layout == COMET_PYR_ALL_CHANNEL_LAST;
  p.pos = nullptr; p.D_tok = 0;
  return COMET_OK;
}

// corr_lookup_up2.cu: the fine tracker reading the encoder's half-resolution map (COMET_PYR_UP2_SOURCE)
int up2_supported(int C, int H, int W, int L, int r, int pad_mode);
template <bool TOKENS>
int launch_lookup_up2(LookupParams& p, const float* src, const float* p2, cudaStream_t stream);

}  // namespace comet

using namespace comet;

extern "C" int comet_corr_lookup_f32(const float* fmaps, const float* pyr, const float* targets, long long t_sb,
                                     long long t_ss, long long t_sn, int t_level_stride, const float* coords,
                                     long long c_sb, long long c_ss, long long c_sn, float* out, long long o_sb,
                                     long long o_ss, long long o_sn, int B, int S, int N, int C, int H, int W, int L,
                                     int r, int pad_mode, int prec_mode, int pyr_layout, comet_stream_t stream) {
  LookupParams p{};
  int rc = fill_params(p, fmaps, pyr, targets, t_sb, t_ss, t_sn, t_level_stride, coords, c_sb, c_ss, c_sn, B, S, N,
                       C, H, W, L, r, pad_mode, prec_mode, pyr_layout);
  if (rc != COMET_OK) return rc;
  COMET_REQUIRE(t_level_stride == 0 || t_level_stride == C, "t_level_stride must be 0 or C");
  COMET_REQUIRE((long long)B * S * N == 0 || out, "null output pointer");
  p.out = out; p.o_sb = o_sb; p.o_ss = o_ss; p.o_sn = o_sn;
  if (pyr_layout == COMET_PYR_UP2_SOURCE) {
    rc = up2_supported(C, H, W, L, r, pad_mode);
    if (rc != COMET_OK) return rc;
    COMET_REQUIRE(t_level_stride == 0, "multiple_track_feats is not served by COMET_PYR_UP2_SOURCE");
    return launch_lookup_up2<false>(p, fmaps, pyr, (cudaStream_t)stream);
  }
  return launch_lookup<false>(p, (cudaStream_t)stream);
}

static int track_tokens(const float* fmaps, const float* pyr, const float* track_feats, long long t_sb, long long t_ss,
                        long long t_sn, const float* coords, long long c_sb, long long c_ss, long long c_sn,
                        const float* pos_emb, float* tokens, const int* num_tracks, const int* num_frames,
                        const int* frame_index, int BS_src, int B, int S, int N, int C, int H, int W, int L, int r,
                        int pad_mode, int prec_mode, int pyr_layout, int D_tok, comet_stream_t stream) {
  LookupParams p{};
  int rc = fill_params(p, fmaps, pyr, track_feats, t_sb, t_ss, t_sn, 0, coords, c_sb, c_ss, c_sn, B, S, N, C, H, W,
                       L, r, pad_mode, prec_mode, pyr_layout);
  if (rc != COMET_OK) return rc;
  const int need = 2 * C + 2 + L * (2 * r + 1) * (2 * r + 1);
  COMET_REQUIRE(C % 4 == 0, "latent_dim must be a multiple of 4 for the flow embedding (got %d)", C);
  COMET_REQUIRE(D_tok >= need, "D_tok=%d smaller than the %d token channels", D_tok, need);
  COMET_REQUIRE((long long)B * S * N == 0 || (tokens && pos_emb), "null tokens / pos_emb pointer");
  p.out = tokens; p.pos = pos_emb; p.D_tok = D_tok; p.ntr = num_tracks; p.nfr = num_frames;
  if (frame_index) {
    // the pyramid holds BS_src frames: its level offsets follow from that count, not from B * S
    COMET_REQUIRE(BS_src >= 1, "BS_src must be positive with a frame table (got %d)", BS_src);
    Levels lv = make_levels(BS_src, C, H, W, L);
    for (int l = 0; l < L; ++l) p.lvlOff[l] = lv.off[l];
    p.fidx = frame_index; p.BS_src = BS_src;
  }
  if (pyr_layout == COMET_PYR_UP2_SOURCE) {
    COMET_REQUIRE(!num_tracks, "per-sequence query counts are not served by COMET_PYR_UP2_SOURCE");
    COMET_REQUIRE(!frame_index, "frame tables are not served by COMET_PYR_UP2_SOURCE");
    rc = up2_supported(C, H, W, L, r, pad_mode);
    if (rc != COMET_OK) return rc;
    return launch_lookup_up2<true>(p, fmaps, pyr, (cudaStream_t)stream);
  }
  return launch_lookup<true>(p, (cudaStream_t)stream);
}

extern "C" int comet_track_tokens_f32(const float* fmaps, const float* pyr, const float* track_feats, long long t_sb,
                                      long long t_ss, long long t_sn, const float* coords, long long c_sb,
                                      long long c_ss, long long c_sn, const float* pos_emb, float* tokens, int B,
                                      int S, int N, int C, int H, int W, int L, int r, int pad_mode, int prec_mode,
                                      int pyr_layout, int D_tok, comet_stream_t stream) {
  return track_tokens(fmaps, pyr, track_feats, t_sb, t_ss, t_sn, coords, c_sb, c_ss, c_sn, pos_emb, tokens, nullptr, nullptr, nullptr,
                      B * S, B, S, N, C, H, W, L, r, pad_mode, prec_mode, pyr_layout, D_tok, stream);
}

extern "C" int comet_track_tokens_ragged_f32(const float* fmaps, const float* pyr, const float* track_feats, long long t_sb,
                                             long long t_ss, long long t_sn, const float* coords, long long c_sb,
                                             long long c_ss, long long c_sn, const float* pos_emb, float* tokens,
                                             const int* num_tracks, int B, int S, int N, int C, int H, int W, int L, int r,
                                             int pad_mode, int prec_mode, int pyr_layout, int D_tok, comet_stream_t stream) {
  COMET_REQUIRE((long long)B * S * N == 0 || num_tracks, "null num_tracks");
  return track_tokens(fmaps, pyr, track_feats, t_sb, t_ss, t_sn, coords, c_sb, c_ss, c_sn, pos_emb, tokens, num_tracks, nullptr,
                      nullptr, B * S, B, S, N, C, H, W, L, r, pad_mode, prec_mode, pyr_layout, D_tok, stream);
}

extern "C" int comet_track_tokens_varlen_f32(const float* fmaps, const float* pyr, const float* track_feats, long long t_sb,
                                             long long t_ss, long long t_sn, const float* coords, long long c_sb,
                                             long long c_ss, long long c_sn, const float* pos_emb, float* tokens,
                                             const int* num_tracks, const int* num_frames, int B, int S, int N, int C, int H,
                                             int W, int L, int r, int pad_mode, int prec_mode, int pyr_layout, int D_tok,
                                             comet_stream_t stream) {
  return track_tokens(fmaps, pyr, track_feats, t_sb, t_ss, t_sn, coords, c_sb, c_ss, c_sn, pos_emb, tokens, num_tracks,
                      num_frames, nullptr, B * S, B, S, N, C, H, W, L, r, pad_mode, prec_mode, pyr_layout, D_tok, stream);
}

extern "C" int comet_track_tokens_indexed_f32(const float* fmaps, const float* pyr, const float* track_feats, long long t_sb,
                                              long long t_ss, long long t_sn, const float* coords, long long c_sb,
                                              long long c_ss, long long c_sn, const float* pos_emb, float* tokens,
                                              const int* num_tracks, const int* num_frames, const int* frame_index, int BS_src,
                                              int B, int S, int N, int C, int H, int W, int L, int r, int pad_mode,
                                              int prec_mode, int pyr_layout, int D_tok, comet_stream_t stream) {
  return track_tokens(fmaps, pyr, track_feats, t_sb, t_ss, t_sn, coords, c_sb, c_ss, c_sn, pos_emb, tokens, num_tracks,
                      num_frames, frame_index, BS_src, B, S, N, C, H, W, L, r, pad_mode, prec_mode, pyr_layout, D_tok,
                      stream);
}
