// Fused correlation + window lookup (+ track tokens) for the fine tracker, reading the patch encoder's HALF-RESOLUTION
// output instead of the up-sampled feature maps -- COMET_PYR_UP2_SOURCE.
//
// The fine tracker's fmaps are, by construction, ShallowEncoder's last op applied to a (Hs x Ws) map S:
// F.interpolate(S, (2Hs-1, 2Ws-1), mode="bilinear", align_corners=True) (comet/models/track_modules/blocks.py:176-190;
// Hs = Ws = 16 -> 31 x 31).  With that exact 2x-1 ratio the up-sampled map T and its pooled pyramid
// (CorrBlock.__init__, blocks.py:368-374) are fixed linear stencils of S, per axis:
//     level 0   T[2k] = S[k]                      T[2k+1] = (S[k] + S[k+1]) / 2              0 <= i <= 2Hs-2
//     level 1   P1[a] = (T[2a] + T[2a+1]) / 2   = 3/4 S[a] + 1/4 S[a+1]                      0 <= a <= Hs-2
//     level 2   P2[c] = (P1[2c] + P1[2c+1]) / 2 = 3/8 S[2c] + 1/2 S[2c+1] + 1/8 S[2c+2]      0 <= c <= (Hs-1)/2 - 1
// and the correlation is linear in the features, so the correlation volume of levels 0 and 1 on the (2r+2)^2 tap
// grids of a query follows from the correlation with S on ONE 9 x 9 box of S around the query (zero padding is
// applied on the tap grid of each level, exactly where the reference applies it).  Level 2 (7 x 7) would need the whole
// S map per query, so it is pooled once per call (pyramid_up2_kernel below) and read through its own 8 x 8 box.
//
// What this removes (per 16-frame sequence at 512 tracks): the 1.0 GB up-sampled feature tensor is never written nor
// read (the producer's last kernel, the pyramid's 1.0 GB read + 0.23 GB level-1 write), and a query moves 16.7 KB
// (81 + 64 lines of 128 B) instead of 22.6 KB.  The up-sampled tensor is what the reference's CorrBlock receives;
// CorrBlock.from_upsampled() takes S and is used by this package's refine_track only (DESIGN.md section 4).
//
// One warp per (patch, frame) query, persistent, 11 warps per SM (what shared memory holds); per query two 4-D TMA boxes land in shared memory with
// the 128-byte swizzle (off-map positions zero-filled); structure otherwise as corr_lookup_c32_tma_kernel.
#include "lookup_common.cuh"

namespace comet {

constexpr int UP2_R = 3, UP2_G = 8, UP2_WR = 7, UP2_WW = 49, UP2_GG = 64;
constexpr int UP2_SB = 9;                                  // S box edge
constexpr int UP2_BOXS = UP2_SB * UP2_SB * 128;            // 10368 B landed
constexpr int UP2_BOXS_PAD = (UP2_BOXS + 1023) & ~1023;    // 11264
constexpr int UP2_BOX2 = UP2_GG * 128;                     // 8192
constexpr int UP2_WARP_BYTES = UP2_BOXS_PAD + UP2_BOX2;
// Warps per CTA (= per SM): as many as shared memory holds.  The kernel is latency-bound at low occupancy (ncu r02 with
// 8 warps: issue slots 39 % busy, 1.9 fixed-latency stall cycles per issue), so every extra warp in flight pays.
#ifndef COMET_UP2_WARPS
#define COMET_UP2_WARPS 11
#endif
constexpr int UP2_WARPS = COMET_UP2_WARPS;
constexpr int UP2_SMEM = UP2_WARPS * UP2_WARP_BYTES + UP2_WARPS * 32 * 4 + UP2_WARPS * 96 * 4 + UP2_WARPS * 64 * 4 + UP2_WARPS * 8;

struct Up2Maps { CUtensorMap s, p2; };

// per-axis stencil of a level-0 tap i (on the 2Hs-1 grid) / level-1 tap a (on the Hs-1 grid) in S:
//   value = w0 * S[k] + w1 * S[k+1]
__device__ __forceinline__ void up2_stencil0(int i, int& k, float& w0, float& w1) {
  k = i >> 1;
  const bool odd = i & 1;
  w0 = odd ? 0.5f : 1.f;
  w1 = odd ? 0.5f : 0.f;
}

template <bool TOKENS, bool BF16>
__global__ void __launch_bounds__(UP2_WARPS * 32, 1) corr_lookup_c32_up2_kernel(const __grid_constant__ Up2Maps maps, const LookupParams p) {
  constexpr int R = UP2_R, G = UP2_G, Wr = UP2_WR, WW = UP2_WW, GG = UP2_GG;
  extern __shared__ __align__(1024) uint8_t smem_up2[];
  uint8_t* const smem = smem_up2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* boxS = smem + warp * UP2_WARP_BYTES;
  uint8_t* box2 = boxS + UP2_BOXS_PAD;
  constexpr int NW = UP2_WARPS;
  float* Ts = reinterpret_cast<float*>(smem + NW * UP2_WARP_BYTES) + warp * 32;
  float* V16 = reinterpret_cast<float*>(smem + NW * UP2_WARP_BYTES + NW * 32 * 4) + warp * 96;   // 9 x 9 correlations with S
  float* Vs = reinterpret_cast<float*>(smem + NW * UP2_WARP_BYTES + NW * 32 * 4 + NW * 96 * 4) + warp * 64;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + NW * UP2_WARP_BYTES + NW * 32 * 4 + NW * 96 * 4 + NW * 64 * 4) + warp;
  if (lane == 0) {
    tma::mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  uint32_t phase = 0;
  const long long total = (long long)p.B * p.S * p.N;
  const long long nwarps = (long long)gridDim.x * NW;
  // level sizes: lvl 0 = (2Hs-1, 2Ws-1) virtual, lvl 1 = (Hs-1, Ws-1) virtual, lvl 2 stored; source map = lvlH/W[0]/2+1
  const int Hs = p.lvlH[0] / 2 + 1, Ws = p.lvlW[0] / 2 + 1;

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
  fetch((long long)blockIdx.x * NW + warp, cx, cy, cx0, cy0, tl);

  for (long long q = (long long)blockIdx.x * NW + warp; q < total; q += nwarps) {
    const int n = (int)(q % p.N);
    const int s = (int)((q / p.N) % p.S);
    const int b = (int)(q / ((long long)p.N * p.S));
    const int bs = b * p.S + s;
    if (TOKENS && p.nfr && s >= __ldg(p.nfr + b)) {   // padded frame: zero row, no map is read
      float* zp = p.out + (((long long)b * p.N + n) * p.S + s) * p.D_tok;
      for (int d = lane; d < p.D_tok; d += 32) zp[d] = 0.f;
      fetch(q + nwarps, cx, cy, cx0, cy0, tl);
      continue;
    }
    AxisWindow ax[3], ay[3];
#pragma unroll
    for (int l = 0; l < 3; ++l) {
      const float inv = 1.f / (float)(1 << l);
      ax[l].init(cx * inv, p.lvlW[l], R, false);
      ay[l].init(cy * inv, p.lvlH[l], R, false);
    }
    // S box: origin = first level-1 tap (the level-0 taps' S positions lie inside it, see the file header);
    // level-2 box: the unclamped window corner.  Origins are bounded so that a wild query still addresses a box the
    // TMA unit can describe (everything it would read is then off the map, i.e. zero).
    const int oxs = min(max(ax[1].i0, -UP2_SB), Ws), oys = min(max(ay[1].i0, -UP2_SB), Hs);
    const int ox2 = min(max(ax[2].i0, -G), p.lvlW[2]), oy2 = min(max(ay[2].i0, -G), p.lvlH[2]);
    __syncwarp();   // every lane is done with the boxes / Ts / V16 / Vs of the previous query
    if (lane == 0) {
      tma::mbar_expect_tx(bar, (uint32_t)(UP2_BOXS + UP2_BOX2));
      tma::load_box_4d(&maps.s, bar, boxS, 0, oxs, oys, bs);
      tma::load_box_4d(&maps.p2, bar, box2, 0, ox2, oy2, bs);
    }
    // float32 mode: 1/sqrt(C) (blocks.py:428 divides the volume after the matmul) is folded into the target vector --
    // the kernel is issue-bound (~900 instructions per query), a per-tap division costs ~50 of them
    Ts[lane] = BF16 ? round_bf16(tl) : tl * p.inv_sqrt_c;
    const float tl_cur = tl, fx = cx - cx0, fy = cy - cy0;
    float cx_n, cy_n, cx0_n, cy0_n, tl_n;
    fetch(q + nwarps, cx_n, cy_n, cx0_n, cy0_n, tl_n);

    float* op;
    const float* pp = nullptr;
    int corr_off = 0;
    float pv[3][2], pe0 = 0.f, pe1 = 0.f, pe2 = 0.f, pe3 = 0.f;   // position-embedding values of this token row
    if (TOKENS) {
      op = p.out + (((long long)b * p.N + n) * p.S + s) * p.D_tok;
      pp = p.pos + ((long long)b * p.N + n) * p.D_tok;
      corr_off = 32 + 2;
#pragma unroll
      for (int l = 0; l < 3; ++l)
#pragma unroll
        for (int k = 0; k < 2; ++k) pv[l][k] = (lane + 32 * k < WW) ? __ldg(pp + corr_off + l * WW + lane + 32 * k) : 0.f;
      pe0 = __ldg(pp + lane);
      pe1 = lane < 2 ? __ldg(pp + 32 + lane) : 0.f;
      pe2 = __ldg(pp + corr_off + 3 * WW + lane);
      pe3 = (corr_off + 3 * WW + 32 + lane < p.D_tok) ? __ldg(pp + corr_off + 3 * WW + 32 + lane) : 0.f;
    } else {
      op = p.out + b * p.o_sb + s * p.o_ss + n * p.o_sn;
#pragma unroll
      for (int l = 0; l < 3; ++l) { pv[l][0] = 0.f; pv[l][1] = 0.f; }
    }
    __syncwarp();
    float4 t4[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) t4[i] = *reinterpret_cast<const float4*>(Ts + 4 * i);

    tma::mbar_wait(bar, phase);
    phase ^= 1;

    auto dot_line = [&](const uint8_t* box, int slot) {
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
      return a;
    };
    // correlation with S on the 9 x 9 box (81 positions over 3 rounds of lanes), unscaled
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const int idx = lane + 32 * k;
      if (idx < UP2_SB * UP2_SB) V16[idx] = dot_line(boxS, idx);
    }
    __syncwarp();

    auto scale = [&](float v) {          // autocast rounds the matmul result and the scaled volume to bf16
      if (BF16) v = round_bf16(round_bf16(v) * p.inv_sqrt_c);
      return v;
    };
    auto blend_store = [&](int l) {
#pragma unroll
      for (int k = 0; k < 2; ++k) {
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
          op[corr_off + l * WW + o] = val + pv[l][k];
        }
      }
    };
    // local S-box coordinate of absolute S index k along an axis (clamped: a clamped read only ever feeds a masked tap
    // or carries weight 0)
    auto lx = [&](int k) { return min(max(k - oxs, 0), UP2_SB - 1); };
    auto ly = [&](int k) { return min(max(k - oys, 0), UP2_SB - 1); };

    // ---- level 0: taps on the (2Hs-1) grid
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int idx = lane + 32 * k;
      int gx = 0, gy = 0;
      const bool ok = ax[0].tap(idx % G, gx) & ay[0].tap(idx / G, gy);
      float v = 0.f;
      if (ok) {
        int kx, ky;
        float wx0, wx1, wy0, wy1;
        up2_stencil0(gx, kx, wx0, wx1);
        up2_stencil0(gy, ky, wy0, wy1);
        const float* r0 = V16 + ly(ky) * UP2_SB;
        const float* r1 = V16 + ly(ky + 1) * UP2_SB;
        const int x0 = lx(kx), x1 = lx(kx + 1);
        v = wy0 * (wx0 * r0[x0] + wx1 * r0[x1]) + wy1 * (wx0 * r1[x0] + wx1 * r1[x1]);
        v = scale(v);
      }
      Vs[idx] = v;
    }
    __syncwarp();
    blend_store(0);
    __syncwarp();
    // ---- level 1: taps on the (Hs-1) grid, P1[a] = 3/4 S[a] + 1/4 S[a+1] per axis
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int idx = lane + 32 * k;
      int gx = 0, gy = 0;
      const bool ok = ax[1].tap(idx % G, gx) & ay[1].tap(idx / G, gy);
      float v = 0.f;
      if (ok) {
        const float* r0 = V16 + ly(gy) * UP2_SB;
        const float* r1 = V16 + ly(gy + 1) * UP2_SB;
        const int x0 = lx(gx), x1 = lx(gx + 1);
        v = 0.75f * (0.75f * r0[x0] + 0.25f * r0[x1]) + 0.25f * (0.75f * r1[x0] + 0.25f * r1[x1]);
        v = scale(v);
      }
      Vs[idx] = v;
    }
    __syncwarp();
    blend_store(1);
    __syncwarp();
    // ---- level 2: stored map, its own box
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int idx = lane + 32 * k;
      int gx = 0, gy = 0;
      const bool ok = ax[2].tap(idx % G, gx) & ay[2].tap(idx / G, gy);
      const int slot = ok ? (gy - oy2) * G + (gx - ox2) : 0;
      const float a = dot_line(box2, slot);
      Vs[idx] = ok ? scale(a) : 0.f;
    }
    __syncwarp();
    blend_store(2);

    if (TOKENS) {
      const int w = lane & 15;                               // C_emb = 16: [pe_x (16) | pe_y (16)]
      const float arg = __fmul_rn(lane >= 16 ? fy : fx, (float)(w & ~1) * (1000.0f / 16.f));
      float sv, cv;
      sincosf(arg, &sv, &cv);            // one range reduction, no divergence between the sin and the cos lanes
      op[lane] = ((w & 1) ? cv : sv) + pe0;
      if (lane < 2) op[32 + lane] = (lane ? fy : fx) + pe1;
      const int feat_off = corr_off + 3 * WW;
      op[feat_off + lane] = tl_cur + pe2;
      if (feat_off + 32 + lane < p.D_tok) op[feat_off + 32 + lane] = pe3;          // zero pad + pos_emb
      for (int d = feat_off + 64 + lane; d < p.D_tok; d += 32) op[d] = __ldg(pp + d);
    }
    cx = cx_n; cy = cy_n; cx0 = cx0_n; cy0 = cy0_n; tl = tl_n;
  }
}

// ---- level 2 of the pyramid of the up-sampled map, straight from S (channel-last in, channel-last out) -----------
// P2[c][d] = sum_{u,v in 0..2} k[u] k[v] S[2c+u][2d+v],  k = (3/8, 1/2, 1/8).  A map is one contiguous block of
// Hs*Ws*C floats (32 KB for the fine tracker): persistent CTAs stream maps through a ring of shared-memory buffers with
// ONE bulk async copy per map (cp.async.bulk -> mbarrier, PU2_STAGES maps in flight per CTA), threads then produce one
// float4 of one output position each.  HBM: reads Hs*Ws*C*4 bytes, writes H2*W2*C*4 per map.  (The first version
// loaded each map with plain loads and a __syncthreads: 0.257 ms for 32768 maps = 68 % of the HBM rate.)
constexpr int PU2_STAGES = 3;
__global__ void __launch_bounds__(256) pyramid_up2_kernel(const float4* __restrict__ src, float4* __restrict__ p2, int BS,
                                                           int C4, int Hs, int Ws, int H2, int W2) {
  extern __shared__ __align__(128) uint8_t pu2_smem[];
  const int nin = Hs * Ws * C4, nout = H2 * W2 * C4;
  const uint32_t map_bytes = (uint32_t)nin * 16u;
  const uint32_t stage_bytes = (map_bytes + 127u) & ~127u;
  uint64_t* bars = reinterpret_cast<uint64_t*>(pu2_smem + PU2_STAGES * stage_bytes);
  if (threadIdx.x == 0) {
    for (int i = 0; i < PU2_STAGES; ++i) tma::mbar_init(&bars[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const long long first = blockIdx.x, step = gridDim.x;
  auto issue = [&](long long m, int stage) {
    if (threadIdx.x == 0 && m < BS) {
      tma::mbar_expect_tx(&bars[stage], map_bytes);
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(tma::smem_u32(pu2_smem + stage * stage_bytes)), "l"(src + m * nin), "r"(map_bytes),
                     "r"(tma::smem_u32(&bars[stage])) : "memory");
    }
  };
  for (int i = 0; i < PU2_STAGES - 1; ++i) issue(first + i * step, i);
  int stage = 0;
  uint32_t phase = 0;
  const float kw[3] = {0.375f, 0.5f, 0.125f};
  for (long long m = first; m < BS; m += step) {
    // refill the stage that was consumed in the previous iteration (every thread passed the barrier below since)
    issue(m + (PU2_STAGES - 1) * step, (stage + PU2_STAGES - 1) % PU2_STAGES);
    tma::mbar_wait(&bars[stage], phase);
    const float4* smap = reinterpret_cast<const float4*>(pu2_smem + stage * stage_bytes);
    for (int o = threadIdx.x; o < nout; o += blockDim.x) {
      const int c = o % C4, pos = o / C4;
      const int x = pos % W2, y = pos / W2;
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int u = 0; u < 3; ++u) {
        float4 row = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int v = 0; v < 3; ++v) {
          const float4 g = smap[((2 * y + u) * Ws + 2 * x + v) * C4 + c];
          row.x = fmaf(kw[v], g.x, row.x); row.y = fmaf(kw[v], g.y, row.y);
          row.z = fmaf(kw[v], g.z, row.z); row.w = fmaf(kw[v], g.w, row.w);
        }
        acc.x = fmaf(kw[u], row.x, acc.x); acc.y = fmaf(kw[u], row.y, acc.y);
        acc.z = fmaf(kw[u], row.z, acc.z); acc.w = fmaf(kw[u], row.w, acc.w);
      }
      p2[m * nout + o] = acc;
    }
    __syncthreads();          // everybody is done reading this stage before it is refilled
    if (++stage == PU2_STAGES) { stage = 0; phase ^= 1; }
  }
}

static int up2_check(int C, int H, int W, int L, int r, int pad_mode) {
  if (!(C == 32 && L == 3 && r == UP2_R && pad_mode == COMET_PAD_ZEROS && (H & 1) && (W & 1) && H >= 9 && W >= 9))
    return fail(COMET_ERR_UNSUPPORTED,
                "COMET_PYR_UP2_SOURCE serves C=32, 3 levels, radius 3, zero padding, odd map sizes >= 9 (got C=%d L=%d r=%d "
                "pad=%d %dx%d)", C, L, r, pad_mode, H, W);
  if (!(device_sm_count_if_sm100() > 0 && tensor_map_encoder() != nullptr))
    return fail(COMET_ERR_UNSUPPORTED, "COMET_PYR_UP2_SOURCE needs an sm_100 device with TMA descriptors");
  return COMET_OK;
}

// `src` = S (BS, Hs, Ws, 32) channel-last; `p2` = level 2 (BS, H2, W2, 32) channel-last; H, W = level-0 (virtual) size.
template <bool TOKENS>
int launch_lookup_up2(LookupParams& p, const float* src, const float* p2, cudaStream_t stream) {
  const long long total = (long long)p.B * p.S * p.N;
  if (total == 0) return COMET_OK;
  COMET_REQUIRE(((uintptr_t)src % 16) == 0 && ((uintptr_t)p2 % 16) == 0, "source / level-2 maps must be 16-byte aligned");
  const int Hs = p.lvlH[0] / 2 + 1, Ws = p.lvlW[0] / 2 + 1;
  Up2Maps maps;
  memset(&maps, 0, sizeof(maps));
  int rc = encode_level_map(&maps.s, src, p.B * p.S, Hs, Ws, UP2_SB);
  if (rc != COMET_OK) return rc;
  rc = encode_level_map(&maps.p2, p2, p.B * p.S, p.lvlH[2], p.lvlW[2], UP2_G);
  if (rc != COMET_OK) return rc;
  const int sms = device_sm_count_if_sm100();
  const long long want = (total + UP2_WARPS - 1) / UP2_WARPS;
  const int grid = (int)(want < sms ? want : sms);
#define COMET_UP2_LAUNCH(BF)                                                                                       \
  do {                                                                                                             \
    COMET_CUDA(cudaFuncSetAttribute(corr_lookup_c32_up2_kernel<TOKENS, BF>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                    UP2_SMEM));                                                                    \
    corr_lookup_c32_up2_kernel<TOKENS, BF><<<grid, UP2_WARPS * 32, UP2_SMEM, stream>>>(maps, p);                              \
  } while (0)
  if (p.bf16) COMET_UP2_LAUNCH(true); else COMET_UP2_LAUNCH(false);
#undef COMET_UP2_LAUNCH
  return launch_status("corr_lookup_c32_up2_kernel");
}

int up2_supported(int C, int H, int W, int L, int r, int pad_mode) { return up2_check(C, H, W, L, r, pad_mode); }
template int launch_lookup_up2<false>(LookupParams&, const float*, const float*, cudaStream_t);
template int launch_lookup_up2<true>(LookupParams&, const float*, const float*, cudaStream_t);

}  // namespace comet

using namespace comet;

extern "C" int comet_up2_supported(int C, int H, int W, int L, int r, int pad_mode) {
  const int rc = up2_check(C, H, W, L, r, pad_mode);
  return rc == COMET_OK ? 1 : 0;
}

extern "C" long long comet_pyramid_up2_elems(int BS, int C, int Hs, int Ws) {
  if (BS < 0 || C < 1 || Hs < 5 || Ws < 5) return -1;
  return (long long)BS * C * ((Hs - 1) / 2) * ((Ws - 1) / 2);
}

extern "C" int comet_pyramid_up2_f32(const float* src, float* p2, int BS, int C, int Hs, int Ws, comet_stream_t stream) {
  COMET_REQUIRE(BS >= 0 && C >= 4 && C % 4 == 0 && Hs >= 5 && Ws >= 5, "bad shape (BS=%d C=%d %dx%d)", BS, C, Hs, Ws);
  if (BS == 0) return COMET_OK;
  COMET_REQUIRE(src && p2 && ((uintptr_t)src % 16) == 0 && ((uintptr_t)p2 % 16) == 0, "null or misaligned pointer");
  const size_t map_bytes = (size_t)Hs * Ws * C * sizeof(float);
  const size_t smem = PU2_STAGES * ((map_bytes + 127) & ~(size_t)127) + PU2_STAGES * 8;
  COMET_REQUIRE(smem <= 200 * 1024, "source map too large for the shared-memory pyramid (%zu bytes per map)", map_bytes);
  COMET_CUDA(cudaFuncSetAttribute(pyramid_up2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int sms = device_sm_count_if_sm100();
  if (sms <= 0) sms = 148;
  const int per_sm = (int)((220 * 1024) / smem) < 1 ? 1 : (int)((220 * 1024) / smem);
  long long grid = (long long)sms * per_sm;
  if (grid > BS) grid = BS;
  pyramid_up2_kernel<<<(unsigned)grid, 256, smem, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(src), reinterpret_cast<float4*>(p2), BS, C / 4, Hs, Ws, (Hs - 1) / 2, (Ws - 1) / 2);
  return launch_status("pyramid_up2_kernel");
}
