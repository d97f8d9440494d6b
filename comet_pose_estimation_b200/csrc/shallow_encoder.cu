// ShallowEncoder of the fine tracker (comet/models/track_modules/blocks.py:114-196, norm_fn="instance"; ResidualBlock:
// comet/models/modules.py:39-117) as ONE kernel: patch gather (refine_track.py:71-111) -> conv1 3x3/2 -> InstanceNorm ->
// ReLU -> two stride-2 residual blocks -> two bilinear residual up-samplings -> 1x1 conv + skip, for 31x31 patches.
//
// Every operator of the encoder is local to one patch (instance norm reduces over the positions of one patch and one
// channel), so a patch never has to leave the SM between its 3-channel pixels and the 16x16x32 map the fine tracker
// consumes (blocks.Upsampled2x evaluates the encoder's last 16x16 -> 31x31 resize lazily).  One CTA carries two
// patches through all layers in shared memory (87 KB each); HBM sees 11.5 KB in and 32 KB out per patch.  The library
// convolutions + separate norm / resize kernels this replaces wrote and re-read ten intermediate maps per patch.
//
// Arithmetic is float32 FMA (the reference's float32 convolution; no TF32): 2.04 M multiply-adds per patch, so this
// kernel is bound by the FP32 pipe, not by HBM: 8192 patches of a 512-track, 16-frame sequence are 16.7 G multiply-adds
// against 37 T/s (148 SMs x 128 lanes x 1.965 GHz).
//
// Work split inside the CTA (8 warps): a warp task is 16 output positions x 32 output channels; a lane owns a 4 x 4
// block of it (positions pq, pq+4, pq+8, pq+12 x channels 4cq..4cq+3, lane = 8 pq + cq).  Per 4 input channels a lane
// reads 4 weight vectors and 4 input vectors (16-byte shared loads) for 64 FMA -- the first version (lane = channel,
// inputs as warp-wide broadcasts: 17 loads = 36 shared wavefronts per 64 FMA) sat at 25 % of the FMA pipe, bound by
// shared-memory wavefronts (profiles/r02c_shallow_encoder_v1_summary.csv).  Activations are channel-last with 36 floats
// per position (32 + 4 of padding) so that the four positions a half-warp reads fall into different banks.  Weights of
// the current layer sit in shared memory ([tap][ci/4][co%4][co/4][4]), fetched with cp.async while the previous layer's
// instance norm runs.  The 4x4 layers have only 32 positions per CTA: their 288-deep sums are split four ways over the
// input channels and combined in a fixed order (deterministic).
#include "comet_common.cuh"

namespace comet {
namespace senc {

constexpr int C = 32;            // feature channels
constexpr int CS = 36;           // floats per position of a channel-last activation buffer (32 + 4 padding: bank shift)
constexpr int G = 2;             // patches per CTA
constexpr int THREADS = 256;
constexpr int PSZ = 31;          // patch extent

// per-patch shared-memory map (float offsets).  Padded buffers carry the zero border the next convolution reads.
constexpr int IN_W = 33;                       // input 31x31 padded by one on every side, 4 floats per position (RGB0)
constexpr int OFF_IN = 0;                      // [33*33][4]   = 4356
constexpr int OFF_A8P = 0;                     // [10*10][CS]  = 3600   (aliases IN once conv1 is done)
constexpr int OFF_A4P = 3600;                  // [6*6][CS]    = 1296   (aliases IN)
constexpr int XP_W = 17;                       // 16x16 map padded on top / left
constexpr int OFF_XP = 4896;                   // [17*17][CS]  = 10404
constexpr int OFF_B8 = OFF_XP + 10404;         // [8*8][CS]    = 2304   (later: the four partial sums of the 4x4 layers)
constexpr int T1P_W = 9;                       // 8x8 map padded on top / left
constexpr int OFF_T1P = OFF_B8 + 2304;         // [9*9][CS]    = 2916
constexpr int OFF_B4 = OFF_T1P + 2916;         // [4*4][CS]    = 576
constexpr int OFF_T2 = OFF_B4 + 576;           // [4*4][CS]    = 576
constexpr int PATCH_FLOATS = OFF_T2 + 576;     // 21672 floats = 86688 bytes
// CTA-wide regions behind the G patch regions
constexpr int OFF_WB = G * PATCH_FLOATS;       // weights of the current 3x3 32->32 layer (9216)
constexpr int OFF_WS = OFF_WB + 9216;          // conv1 (1152) | layer1.downsample (1024) | layer2.downsample | conv2
constexpr int WS_CONV1 = 0, WS_L1DN = 1152, WS_L2DN = 2176, WS_CONV2 = 3200, WS_FLOATS = 4224;
constexpr int OFF_BIAS = OFF_WS + WS_FLOATS;   // 8 x 32 biases, layer order of the packed blob
constexpr int OFF_RED = OFF_BIAS + 256;        // two reduction scratch arrays [G][4][32]
constexpr int SMEM_FLOATS = OFF_RED + 2 * G * 4 * C;
constexpr int SMEM_BYTES = SMEM_FLOATS * 4;    // 230208
static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
static_assert(OFF_XP % 4 == 0 && OFF_B8 % 4 == 0 && OFF_T1P % 4 == 0 && OFF_B4 % 4 == 0 && PATCH_FLOATS % 4 == 0, "16-byte alignment");

// packed parameter blob (float offsets): per layer the weights [tap][ci/4][co%4][co/4][ci%4], then 32 biases
constexpr int W_CONV1 = 0, B_CONV1 = 1152;
constexpr int W_L1C1 = 1184, B_L1C1 = W_L1C1 + 9216;
constexpr int W_L1C2 = B_L1C1 + 32, B_L1C2 = W_L1C2 + 9216;
constexpr int W_L1DN = B_L1C2 + 32, B_L1DN = W_L1DN + 1024;
constexpr int W_L2C1 = B_L1DN + 32, B_L2C1 = W_L2C1 + 9216;
constexpr int W_L2C2 = B_L2C1 + 32, B_L2C2 = W_L2C2 + 9216;
constexpr int W_L2DN = B_L2C2 + 32, B_L2DN = W_L2DN + 1024;
constexpr int W_CONV2 = B_L2DN + 32, B_CONV2 = W_CONV2 + 1024;
constexpr int PACKED_FLOATS = B_CONV2 + 32;    // 41344
// bias slots in shared memory
enum { L_CONV1 = 0, L_L1C1, L_L1C2, L_L1DN, L_L2C1, L_L2C2, L_L2DN, L_CONV2 };

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
// all threads: copy n floats (multiple of 4) global -> shared
__device__ __forceinline__ void stage(float* dst, const float* __restrict__ src, int n, int tid) {
  for (int i = tid * 4; i < n; i += THREADS * 4) cp_async16(dst + i, src + i);
}

// One warp task: 16 positions x 32 channels of a convolution, a 4 x 4 block per lane.
//   acc[jj][k] += sum over taps and the input-channel groups [cb, cb+NC) of in[position 4jj+pq, tap, ci] * w[tap, ci, 4cq+k]
// Position j of the task sits at (j / OW, j % OW) of an OW-wide output block (OW % 4 == 0: the four positions of one
// jj are neighbours in a row); `in_lane` = (padded) input address of position pq's first tap, WP the padded input
// width, CPP the floats per input position, KW x KW the kernel, CH input-channel groups per tap in the weight layout.
template <int OW, int STRIDE, int WP, int CPP, int KW, int CH, int NC>
__device__ __forceinline__ void conv16(const float* __restrict__ in_lane, const float* __restrict__ w, int cq, int cb,
                                       float (&acc)[4][4]) {
  static_assert(OW % 4 == 0, "a lane's four positions share a row");
  const float4* w4 = reinterpret_cast<const float4*>(w) + cq;
#pragma unroll 1
  for (int tap = 0; tap < KW * KW; ++tap) {
    const int ky = tap / KW, kx = tap - ky * KW;
    const float* pt = in_lane + (ky * WP + kx) * CPP + cb * 4;
    const float4* wt = w4 + (tap * CH + cb) * 32;
#pragma unroll 2
    for (int i = 0; i < NC; ++i) {
      float4 wv[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) wv[k] = wt[i * 32 + k * 8];
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const float4 x = *reinterpret_cast<const float4*>(pt + i * 4 + (((jj * 4) / OW) * STRIDE * WP + ((jj * 4) % OW) * STRIDE) * CPP);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          acc[jj][k] = fmaf(x.x, wv[k].x, acc[jj][k]);
          acc[jj][k] = fmaf(x.y, wv[k].y, acc[jj][k]);
          acc[jj][k] = fmaf(x.z, wv[k].z, acc[jj][k]);
          acc[jj][k] = fmaf(x.w, wv[k].w, acc[jj][k]);
        }
      }
    }
  }
}

// store the block: position 4jj+pq -> out_lane + ((4jj / OW) * OWP + 4jj % OW) * CS, out_lane = out0 + pq * CS + 4 cq
template <int OW, int OWP>
__device__ __forceinline__ void store16(float* out_lane, const float (&acc)[4][4]) {
#pragma unroll
  for (int jj = 0; jj < 4; ++jj)
    *reinterpret_cast<float4*>(out_lane + (((jj * 4) / OW) * OWP + (jj * 4) % OW) * CS) =
        make_float4(acc[jj][0], acc[jj][1], acc[jj][2], acc[jj][3]);
}

__device__ __forceinline__ void fill16(float (&acc)[4][4], const float4 b) {
#pragma unroll
  for (int jj = 0; jj < 4; ++jj) { acc[jj][0] = b.x; acc[jj][1] = b.y; acc[jj][2] = b.z; acc[jj][3] = b.w; }
}

// The same for the layers with >= 128 positions per CTA: 32 positions x 32 channels per warp task, an 8 x 4 block per
// lane (positions pq + 4 jj, channels 4 cq .. 4 cq + 3) with lane = 4 cq + pq: the four quarter-warps of an input load
// then read identical addresses (2 shared wavefronts instead of 4), and a weight vector is reused for 8 positions:
// 12 loads = 32 wavefronts per 128 FMA, against 8 loads = 24 wavefronts per 64 FMA of the 4 x 4 block.
template <int OW, int STRIDE, int WP, int CPP, int KW, int CH, int NC>
__device__ __forceinline__ void conv32(const float* __restrict__ in_lane, const float* __restrict__ w, int cq, int cb,
                                       float (&acc)[8][4]) {
  static_assert(OW % 4 == 0, "a lane's positions of one jj share a row");
  const float4* w4 = reinterpret_cast<const float4*>(w) + cq;
#pragma unroll 1
  for (int tap = 0; tap < KW * KW; ++tap) {
    const int ky = tap / KW, kx = tap - ky * KW;
    const float* pt = in_lane + (ky * WP + kx) * CPP + cb * 4;
    const float4* wt = w4 + (tap * CH + cb) * 32;
#pragma unroll 2
    for (int i = 0; i < NC; ++i) {
      float4 wv[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) wv[k] = wt[i * 32 + k * 8];
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const float4 x = *reinterpret_cast<const float4*>(pt + i * 4 + (((jj * 4) / OW) * STRIDE * WP + ((jj * 4) % OW) * STRIDE) * CPP);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          acc[jj][k] = fmaf(x.x, wv[k].x, acc[jj][k]);
          acc[jj][k] = fmaf(x.y, wv[k].y, acc[jj][k]);
          acc[jj][k] = fmaf(x.z, wv[k].z, acc[jj][k]);
          acc[jj][k] = fmaf(x.w, wv[k].w, acc[jj][k]);
        }
      }
    }
  }
}

// store (ADD = false) or add onto (ADD = true: the second half of a sum split over the input channels) the block:
// position 4jj+pq -> out_lane + ((4jj / OW) * OWP + 4jj % OW) * CS, out_lane = out0 + pq * CS + 4 cq
template <int OW, int OWP, bool ADD>
__device__ __forceinline__ void store32(float* out_lane, const float (&acc)[8][4]) {
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) {
    float4* o = reinterpret_cast<float4*>(out_lane + (((jj * 4) / OW) * OWP + (jj * 4) % OW) * CS);
    float4 v = make_float4(acc[jj][0], acc[jj][1], acc[jj][2], acc[jj][3]);
    if (ADD) {
      const float4 h = *o;
      v = make_float4(h.x + v.x, h.y + v.y, h.z + v.z, h.w + v.w);
    }
    *o = v;
  }
}

__device__ __forceinline__ void fill32(float (&acc)[8][4], const float4 b) {
#pragma unroll
  for (int jj = 0; jj < 8; ++jj) { acc[jj][0] = b.x; acc[jj][1] = b.y; acc[jj][2] = b.z; acc[jj][3] = b.w; }
}

// nn.InstanceNorm2d(affine=False) over the OW x OW interior of a buffer whose rows are OWP positions wide, for both
// patches of the CTA: thread <-> (patch g, position class q = positions q, q+4, .., channel).  Biased variance, two
// passes.  `x0` / `acc0` point at patch 0 (patch g: + g * PATCH_FLOATS).  relu: y = max(y, 0).  With `acc0` the result
// is not written back but folded into the residual sum: acc = max(acc + y, 0)  (modules.py:115-117).
template <int OW, int OWP, int AWP>
__device__ __forceinline__ void inorm(float* x0, float* acc0, bool relu, float eps, float* red, int tid) {
  constexpr int NPOS = OW * OW, XQ = OW / 4;
  const int g = tid >> 7, q = (tid >> 5) & 3, co = tid & 31;
  float* x = x0 + g * PATCH_FLOATS + q * CS + co;     // positions (row, q + 4 xi)
  float* r1 = red + (g * 4) * C + co;
  float* r2 = r1 + G * 4 * C;
  float s = 0.f;
#pragma unroll 4
  for (int row = 0; row < OW; ++row)
#pragma unroll
    for (int xi = 0; xi < XQ; ++xi) s += x[(row * OWP + 4 * xi) * CS];
  r1[q * C] = s;
  __syncthreads();
  const float mean = (((r1[0] + r1[C]) + r1[2 * C]) + r1[3 * C]) * (1.f / (float)NPOS);
  float v = 0.f;
#pragma unroll 4
  for (int row = 0; row < OW; ++row)
#pragma unroll
    for (int xi = 0; xi < XQ; ++xi) {
      const float d = x[(row * OWP + 4 * xi) * CS] - mean;
      v = fmaf(d, d, v);
    }
  r2[q * C] = v;
  __syncthreads();
  const float rstd = rsqrtf((((r2[0] + r2[C]) + r2[2 * C]) + r2[3 * C]) * (1.f / (float)NPOS) + eps);
  float* a = acc0 ? acc0 + g * PATCH_FLOATS + q * CS + co : nullptr;
#pragma unroll 4
  for (int row = 0; row < OW; ++row)
#pragma unroll
    for (int xi = 0; xi < XQ; ++xi) {
      const int o = (row * OWP + 4 * xi) * CS;
      float y = (x[o] - mean) * rstd;
      if (relu) y = fmaxf(y, 0.f);
      if (a) {
        const int oa = (row * AWP + 4 * xi) * CS;
        a[oa] = fmaxf(a[oa] + y, 0.f);
      } else {
        x[o] = y;
      }
    }
  __syncthreads();
}

// x (16x16 interior of the padded XP buffer) += F.interpolate(t, (16, 16), "bilinear", align_corners=True) of the
// IW x IW map `t0` (rows TWP positions wide); ATen's arithmetic: src = dst * (in-1)/(out-1), i0 = (int)src,
// i1 = i0 + (i0 < in-1), w1 = src - i0, w0 = 1 - w1, value = wy0*(wx0*v00 + wx1*v01) + wy1*(wx0*v10 + wx1*v11).
template <int IW, int TWP>
__device__ __forceinline__ void upsample_add(float* xp0, const float* t0, int warp, int pq, int cq) {
  // warp <-> (patch, four output rows); lane <-> (output column pq + 4 i, channels 4 cq .. 4 cq + 3)
  const int g = warp >> 2;
  float* xp = xp0 + g * PATCH_FLOATS + 4 * cq;
  const float* t = t0 + g * PATCH_FLOATS + 4 * cq;
  const float scale = (float)(IW - 1) / 15.f;
#pragma unroll 1
  for (int yo = (warp & 3) * 4; yo < (warp & 3) * 4 + 4; ++yo) {
    const float sy = scale * (float)yo;
    const int y0 = (int)sy, y1 = y0 + (y0 < IW - 1 ? 1 : 0);
    const float wy1 = sy - (float)y0, wy0 = 1.f - wy1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int xo = pq + 4 * i;
      const float sx = scale * (float)xo;
      const int x0 = (int)sx, x1 = x0 + (x0 < IW - 1 ? 1 : 0);
      const float wx1 = sx - (float)x0, wx0 = 1.f - wx1;
      const float4 v00 = *reinterpret_cast<const float4*>(t + (y0 * TWP + x0) * CS), v01 = *reinterpret_cast<const float4*>(t + (y0 * TWP + x1) * CS);
      const float4 v10 = *reinterpret_cast<const float4*>(t + (y1 * TWP + x0) * CS), v11 = *reinterpret_cast<const float4*>(t + (y1 * TWP + x1) * CS);
      float4* o = reinterpret_cast<float4*>(xp + ((yo + 1) * XP_W + xo + 1) * CS);
      float4 r = *o;
      r.x += wy0 * (wx0 * v00.x + wx1 * v01.x) + wy1 * (wx0 * v10.x + wx1 * v11.x);
      r.y += wy0 * (wx0 * v00.y + wx1 * v01.y) + wy1 * (wx0 * v10.y + wx1 * v11.y);
      r.z += wy0 * (wx0 * v00.z + wx1 * v01.z) + wy1 * (wx0 * v10.z + wx1 * v11.z);
      r.w += wy0 * (wx0 * v00.w + wx1 * v01.w) + wy1 * (wx0 * v10.w + wx1 * v11.w);
      *o = r;
    }
  }
}

// zero the border cells of a padded [WP][WP][CPP] buffer of both patches (FULL: all four sides, else top row / left
// column), one 16-byte store per (border cell, 4 floats)
template <int WP, int CPP, bool FULL>
__device__ __forceinline__ void zero_border(float* b0, int tid) {
  constexpr int NB = FULL ? 4 * WP - 4 : 2 * WP - 1, V = CPP / 4;
  for (int i = tid; i < G * NB * V; i += THREADS) {
    const int g = i / (NB * V), r = i - g * (NB * V), b = r / V, v = r - b * V;
    int y, x;
    if (b < WP) { y = 0; x = b; }
    else if (FULL && b < 2 * WP) { y = WP - 1; x = b - WP; }
    else if (FULL) { y = 1 + ((b - 2 * WP) >> 1); x = ((b - 2 * WP) & 1) * (WP - 1); }
    else { y = b - WP + 1; x = 0; }
    *reinterpret_cast<float4*>(b0 + g * PATCH_FLOATS + (y * WP + x) * CPP + 4 * v) = make_float4(0.f, 0.f, 0.f, 0.f);
  }
}

struct Params {
  const float* src;        // images (B,S,3,H,W) or a patch tensor
  const int* topleft;      // (B,S,N,2) (x, y) corners, or null: `src` holds the patches themselves
  const int* seq_of_track; // packed tracks, or null: topleft is (N,S,2) and track n reads the frames of sequence seq_of_track[n]
  const float* packed;
  float* out;              // (P, 16, 16, 32) channel-last
  long long P;             // number of patches
  long long sn, sc, sy, sx;  // element strides of the patch tensor (topleft == null) / of the image (sc, sy, sx)
  int S, N, H, W;
  int nseq;                // packed tracks: number of sequences in `src`
  const int* num_frames;   // packed tracks, nullable: sequence b has num_frames[b] real frames; the patches of the others
                           // are not read and their maps are written as zeros
  const int* frame_index;  // packed tracks, nullable: (nseq, S) image frame that frame s of sequence b reads (else b * S + s)
  long long nframes_src;   // packed tracks with frame_index: frames of `src` (entries are clamped to [0, nframes_src))
  float eps;
  const long long* frame_offset;  // packed frames (PACKED kernels only): frame f starts at element frame_offset[f] of `src`
  const int* frame_hw;            // ... and is frame_hw[2f] x frame_hw[2f+1] pixels (H, W); nframes_src frames in all
};

// Packed tracks with frame counts: patch pi lies in a frame past its sequence's count.
__device__ __forceinline__ bool padded_patch(const Params& p, long long pi) {
  if (!p.num_frames) return false;
  const int s = (int)(pi % p.S);
  const int b = min(max(__ldg(p.seq_of_track + pi / p.S), 0), p.nseq - 1);
  return s >= __ldg(p.num_frames + b);
}

// pixels of patch pair `pair` -> registers: thread <-> cells tid + 256 k of the 2 x 31 x 31 cells, 3 channels each.
// PACKED: `src` is a packed frame buffer (packed tracks only); a patch's frame brings its own offset, size and strides.
template <bool PACKED>
__device__ __forceinline__ void prefetch_pixels(const Params& p, long long pair, int tid, float (&pre)[24]) {
  const float* base[G];
  long long plane[G];      // PACKED: channel stride and row stride of each patch's frame
  int row[G];
#pragma unroll
  for (int g = 0; g < G; ++g) {
    long long pi = pair * G + g;
    if (pi >= p.P) pi = p.P - 1;   // odd patch count: the last pair encodes the last patch twice and stores it once
    if (padded_patch(p, pi)) {
      base[g] = nullptr;           // encodes a zero patch; its output is written as zeros
    } else if (p.topleft) {
      const int s = (int)(pi % p.S);
      const long long bn = pi / p.S;
      const int n = (int)(bn % p.N);
      long long b = bn / p.N;
      const int* tl = p.topleft + ((b * p.S + s) * p.N + n) * 2;
      long long frame = b * p.S + s;
      if (p.seq_of_track) {
        b = min(max(__ldg(p.seq_of_track + n), 0), p.nseq - 1);
        tl = p.topleft + ((long long)n * p.S + s) * 2;
        frame = b * p.S + s;
        if (p.frame_index) frame = min(max((long long)__ldg(p.frame_index + frame), 0LL), p.nframes_src - 1);
      }
      if constexpr (PACKED) {
        frame = min(max(frame, 0LL), p.nframes_src - 1);
        const int fh = __ldg(p.frame_hw + 2 * frame), fw = __ldg(p.frame_hw + 2 * frame + 1);
        // the corner is clamped to the patch's own frame, so no read leaves it; a frame smaller than a patch is not read
        const int x0 = min(max(__ldg(tl), 0), fw - PSZ), y0 = min(max(__ldg(tl + 1), 0), fh - PSZ);
        base[g] = fh < PSZ || fw < PSZ ? nullptr : p.src + __ldg(p.frame_offset + frame) + (long long)y0 * fw + x0;
        plane[g] = (long long)fh * fw;
        row[g] = fw;
        continue;
      }
      const int x0 = min(max(__ldg(tl), 0), p.W - PSZ), y0 = min(max(__ldg(tl + 1), 0), p.H - PSZ);
      base[g] = p.src + frame * 3 * p.sc + (long long)y0 * p.sy + (long long)x0 * p.sx;
    } else {
      base[g] = p.src + pi * p.sn;
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int cell = tid + k * THREADS;
    if (cell < G * PSZ * PSZ) {
      const int g = cell >= PSZ * PSZ ? 1 : 0, r = cell - g * (PSZ * PSZ), y = r / PSZ, x = r - y * PSZ;
      const float* b = g == 0 ? base[0] : base[1];
      if (PACKED && b) {
        const long long pl = g == 0 ? plane[0] : plane[1];
        b += y * (g == 0 ? row[0] : row[1]) + x;
        pre[3 * k] = __ldg(b);
        pre[3 * k + 1] = __ldg(b + pl);
        pre[3 * k + 2] = __ldg(b + 2 * pl);
      } else if (b) {
        b += y * p.sy + x * p.sx;
        pre[3 * k] = __ldg(b);
        pre[3 * k + 1] = __ldg(b + p.sc);
        pre[3 * k + 2] = __ldg(b + 2 * p.sc);
      } else {
        pre[3 * k] = pre[3 * k + 1] = pre[3 * k + 2] = 0.f;
      }
    }
  }
}
__device__ __forceinline__ void store_pixels(float* smem, int tid, const float (&pre)[24]) {
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const int cell = tid + k * THREADS;
    if (cell < G * PSZ * PSZ) {
      const int g = cell >= PSZ * PSZ ? 1 : 0, r = cell - g * (PSZ * PSZ), y = r / PSZ, x = r - y * PSZ;
      *reinterpret_cast<float4*>(smem + g * PATCH_FLOATS + OFF_IN + ((y + 1) * IN_W + x + 1) * 4) =
          make_float4(pre[3 * k], pre[3 * k + 1], pre[3 * k + 2], 0.f);
    }
  }
}

// Persistent: CTA b encodes patch pairs b, b + gridDim.x, ...  The pixels of the next pair are loaded into registers
// while the current pair is in its convolutions and stored once the region they share with the 8x8 / 4x4 maps is free.
// PACKED: patches are read from a packed frame buffer (frames of different sizes); a separate instantiation, so that
// the image and patch-tensor forms keep their code and register allocation.
template <bool PACKED>
__global__ void __launch_bounds__(THREADS, 1) shallow_encoder_kernel(const Params p) {
  extern __shared__ __align__(16) float smem[];
  float* red = smem + OFF_RED;
  float* wb = smem + OFF_WB;
  const float* ws = smem + OFF_WS;
  const float4* bias4 = reinterpret_cast<const float4*>(smem + OFF_BIAS);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int pq = lane >> 3, cq = lane & 7;   // 4 x 4 blocks (conv16, up-sampling)
  const int pw = lane & 3, cw = lane >> 2;   // 8 x 4 blocks (conv32)
  const float* __restrict__ pk = p.packed;
  const long long npairs = (p.P + G - 1) / G;
  long long pair = blockIdx.x;
  if (pair >= npairs) return;

  // ---- once per CTA: small-layer weights and biases (cp.async), borders nobody overwrites, the first pair's pixels ---
  stage(smem + OFF_WS + WS_CONV1, pk + W_CONV1, 1152, tid);
  stage(smem + OFF_WS + WS_L1DN, pk + W_L1DN, 1024, tid);
  stage(smem + OFF_WS + WS_L2DN, pk + W_L2DN, 1024, tid);
  stage(smem + OFF_WS + WS_CONV2, pk + W_CONV2, 1024, tid);
  if (tid < 64) {
    const int l = tid >> 3;
    const int boff = l == 0 ? B_CONV1 : l == 1 ? B_L1C1 : l == 2 ? B_L1C2 : l == 3 ? B_L1DN : l == 4 ? B_L2C1 : l == 5 ? B_L2C2 : l == 6 ? B_L2DN : B_CONV2;
    cp_async16(smem + OFF_BIAS + tid * 4, pk + boff + (tid & 7) * 4);
  }
  stage(wb, pk + W_L1C1, 9216, tid);
  cp_async_commit();
  float pre[24];
  prefetch_pixels<PACKED>(p, pair, tid, pre);
  zero_border<XP_W, CS, false>(smem + OFF_XP, tid);
  zero_border<T1P_W, CS, false>(smem + OFF_T1P, tid);
  zero_border<IN_W, 4, true>(smem + OFF_IN, tid);
  store_pixels(smem, tid, pre);
  cp_async_wait_all();
  __syncthreads();

  float acc[4][4];
  float acw[8][4];
  while (true) {
    const long long next = pair + gridDim.x;
    const bool has_next = next < npairs;

    // ---- phase 1: conv1 (3 -> 32, 3x3, stride 2): 16 tasks (patch, two output rows) ---------------------------------
#pragma unroll 1
    for (int t = warp; t < G * 8; t += 8) {
      const int g = t >> 3, oy = 2 * (t & 7);
      fill32(acw, bias4[L_CONV1 * 8 + cw]);
      conv32<16, 2, IN_W, 4, 3, 1, 1>(smem + g * PATCH_FLOATS + OFF_IN + (2 * oy * IN_W + 2 * pw) * 4, ws + WS_CONV1, cw, 0, acw);
      store32<16, XP_W, false>(smem + g * PATCH_FLOATS + OFF_XP + ((oy + 1) * XP_W + 1 + pw) * CS + 4 * cw, acw);
    }
    __syncthreads();
    if (has_next) prefetch_pixels<PACKED>(p, next, tid, pre);   // in flight until this pair's convolutions are done
    // the input is dead: its space now holds the padded 8x8 / 4x4 maps, whose borders must read as zero
    zero_border<10, CS, true>(smem + OFF_A8P, tid);
    zero_border<6, CS, true>(smem + OFF_A4P, tid);
    cp_async_wait_all();                                                                     // layer1.conv1 weights
    inorm<16, XP_W, 0>(smem + OFF_XP + (XP_W + 1) * CS, nullptr, true, p.eps, red, tid);     // x0 = relu(norm1(conv1))

    // ---- phase 2: layer1.conv1 (3x3 / 2) -> A8, layer1.downsample (1x1 / 2) -> T1: warp <-> (patch, four output rows,
    // half of the input channels); the second halves are added once the first ones are stored
    {
      const int tk = warp >> 1, ks = warp & 1, g = tk >> 1, r0 = (tk & 1) * 4;
      const float* xp = smem + g * PATCH_FLOATS + OFF_XP;
      float* a8 = smem + g * PATCH_FLOATS + OFF_A8P + ((r0 + 1) * 10 + 1 + pw) * CS + 4 * cw;
      float* t1 = smem + g * PATCH_FLOATS + OFF_T1P + ((r0 + 1) * T1P_W + 1 + pw) * CS + 4 * cw;
      fill32(acw, ks ? make_float4(0.f, 0.f, 0.f, 0.f) : bias4[L_L1C1 * 8 + cw]);
      conv32<8, 2, XP_W, CS, 3, 8, 4>(xp + (2 * r0 * XP_W + 2 * pw) * CS, wb, cw, 4 * ks, acw);
      if (!ks) store32<8, 10, false>(a8, acw);
      float acd[8][4];
      fill32(acd, ks ? make_float4(0.f, 0.f, 0.f, 0.f) : bias4[L_L1DN * 8 + cw]);
      conv32<8, 2, XP_W, CS, 1, 8, 4>(xp + ((2 * r0 + 1) * XP_W + 1 + 2 * pw) * CS, ws + WS_L1DN, cw, 4 * ks, acd);
      if (!ks) store32<8, T1P_W, false>(t1, acd);
      __syncthreads();
      if (ks) {
        store32<8, 10, true>(a8, acw);
        store32<8, T1P_W, true>(t1, acd);
      }
    }
    __syncthreads();
    stage(wb, pk + W_L1C2, 9216, tid);
    cp_async_commit();
    inorm<8, 10, 0>(smem + OFF_A8P + (10 + 1) * CS, nullptr, true, p.eps, red, tid);          // relu(norm1(conv1))
    cp_async_wait_all();
    inorm<8, T1P_W, 0>(smem + OFF_T1P + (T1P_W + 1) * CS, nullptr, false, p.eps, red, tid);   // norm3(downsample)

    // ---- phase 3: layer1.conv2 (3x3) -> B8, same split; T1 = relu(T1 + relu(norm2(B8))) ------------------------------
    {
      const int tk = warp >> 1, ks = warp & 1, g = tk >> 1, r0 = (tk & 1) * 4;
      float* b8 = smem + g * PATCH_FLOATS + OFF_B8 + (r0 * 8 + pw) * CS + 4 * cw;
      fill32(acw, ks ? make_float4(0.f, 0.f, 0.f, 0.f) : bias4[L_L1C2 * 8 + cw]);
      conv32<8, 1, 10, CS, 3, 8, 4>(smem + g * PATCH_FLOATS + OFF_A8P + (r0 * 10 + pw) * CS, wb, cw, 4 * ks, acw);
      if (!ks) store32<8, 8, false>(b8, acw);
      __syncthreads();
      if (ks) store32<8, 8, true>(b8, acw);
    }
    __syncthreads();
    stage(wb, pk + W_L2C1, 9216, tid);
    cp_async_commit();
    cp_async_wait_all();
    inorm<8, 8, T1P_W>(smem + OFF_B8, smem + OFF_T1P + (T1P_W + 1) * CS, true, p.eps, red, tid);

    // ---- phase 4: x += up(T1);  layer2.conv1 (3x3 / 2) four-way split over ci -> partial sums;  layer2.downsample -> T2
    {
      const int g = warp >> 2, ks = warp & 3;
      const float* t1 = smem + g * PATCH_FLOATS + OFF_T1P;
      fill16(acc, make_float4(0.f, 0.f, 0.f, 0.f));
      conv16<4, 2, T1P_W, CS, 3, 8, 2>(t1 + 2 * pq * CS, wb, cq, 2 * ks, acc);
      store16<4, 4>(smem + g * PATCH_FLOATS + OFF_B8 + ks * (16 * CS) + pq * CS + 4 * cq, acc);
      if (ks == 0) {
        fill16(acc, bias4[L_L2DN * 8 + cq]);
        conv16<4, 2, T1P_W, CS, 1, 8, 8>(t1 + (T1P_W + 1 + 2 * pq) * CS, ws + WS_L2DN, cq, 0, acc);
        store16<4, 4>(smem + g * PATCH_FLOATS + OFF_T2 + pq * CS + 4 * cq, acc);
      }
      upsample_add<8, T1P_W>(smem + OFF_XP, smem + OFF_T1P + (T1P_W + 1) * CS, warp, pq, cq);
    }
    __syncthreads();
    stage(wb, pk + W_L2C2, 9216, tid);
    cp_async_commit();
    for (int i = tid; i < G * 512; i += THREADS) {
      const int g = i >> 9, r = i & 511, pos = r >> 5, co = r & 31;
      const float* part = smem + g * PATCH_FLOATS + OFF_B8 + pos * CS + co;
      smem[g * PATCH_FLOATS + OFF_A4P + (((pos >> 2) + 1) * 6 + (pos & 3) + 1) * CS + co] =
          smem[OFF_BIAS + L_L2C1 * 32 + co] + (((part[0] + part[16 * CS]) + part[32 * CS]) + part[48 * CS]);
    }
    __syncthreads();
    inorm<4, 6, 0>(smem + OFF_A4P + (6 + 1) * CS, nullptr, true, p.eps, red, tid);
    cp_async_wait_all();
    inorm<4, 4, 0>(smem + OFF_T2, nullptr, false, p.eps, red, tid);

    // ---- phase 5: layer2.conv2 (3x3), same split -> B4; T2 = relu(T2 + relu(norm2(B4))) -----------------------------
    {
      const int g = warp >> 2, ks = warp & 3;
      fill16(acc, make_float4(0.f, 0.f, 0.f, 0.f));
      conv16<4, 1, 6, CS, 3, 8, 2>(smem + g * PATCH_FLOATS + OFF_A4P + pq * CS, wb, cq, 2 * ks, acc);
      store16<4, 4>(smem + g * PATCH_FLOATS + OFF_B8 + ks * (16 * CS) + pq * CS + 4 * cq, acc);
    }
    __syncthreads();
    if (has_next) {
      // the 8x8 / 4x4 maps and the 3x3 weights are dead: next pair's pixels and first 3x3 layer move in
      stage(wb, pk + W_L1C1, 9216, tid);
      cp_async_commit();
      zero_border<IN_W, 4, true>(smem + OFF_IN, tid);
      store_pixels(smem, tid, pre);
    }
    for (int i = tid; i < G * 512; i += THREADS) {
      const int g = i >> 9, r = i & 511, pos = r >> 5, co = r & 31;
      const float* part = smem + g * PATCH_FLOATS + OFF_B8 + pos * CS + co;
      smem[g * PATCH_FLOATS + OFF_B4 + pos * CS + co] =
          smem[OFF_BIAS + L_L2C2 * 32 + co] + (((part[0] + part[16 * CS]) + part[32 * CS]) + part[48 * CS]);
    }
    __syncthreads();
    inorm<4, 4, 4>(smem + OFF_B4, smem + OFF_T2, true, p.eps, red, tid);

    // ---- phase 6: x += up(T2);  out = conv2(x) + x (1x1) -------------------------------------------------------------
    upsample_add<4, 4>(smem + OFF_XP, smem + OFF_T2, warp, pq, cq);
    __syncthreads();
#pragma unroll 1
    for (int t = warp; t < G * 8; t += 8) {
      const int g = t >> 3, oy = 2 * (t & 7);
      const long long pi = pair * G + g;
      if (pi >= p.P) continue;
      const float* row = smem + g * PATCH_FLOATS + OFF_XP + ((oy + 1) * XP_W + 1 + pw) * CS;
      float* o = p.out + (pi * 256 + oy * 16 + pw) * C + 4 * cw;
      if (padded_patch(p, pi)) {
#pragma unroll
        for (int jj = 0; jj < 8; ++jj)
          *reinterpret_cast<float4*>(o + ((jj >> 2) * 16 + (jj & 3) * 4) * C) = make_float4(0.f, 0.f, 0.f, 0.f);
        continue;
      }
      fill32(acw, bias4[L_CONV2 * 8 + cw]);
      conv32<16, 1, XP_W, CS, 1, 8, 8>(row, ws + WS_CONV2, cw, 0, acw);
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const float4 x = *reinterpret_cast<const float4*>(row + ((jj >> 2) * XP_W + (jj & 3) * 4) * CS + 4 * cw);
        *reinterpret_cast<float4*>(o + ((jj >> 2) * 16 + (jj & 3) * 4) * C) =
            make_float4(acw[jj][0] + x.x, acw[jj][1] + x.y, acw[jj][2] + x.z, acw[jj][3] + x.w);
      }
    }
    if (!has_next) break;
    pair = next;
    __syncthreads();   // conv1 of the next pair overwrites the map conv2 has just read
  }
}

// parameter packing: raw state-dict tensors (OIHW weights, biases) -> the blob the kernel reads
struct PackParams {
  const float* t[16];
  float* packed;
};
__global__ void __launch_bounds__(256) shallow_encoder_pack_kernel(const PackParams pp) {
  // layer l: weight t[2l] (32, CI, K, K), bias t[2l+1]; order conv1, layer1.{conv1,conv2,downsample.0},
  // layer2.{conv1,conv2,downsample.0}, conv2
  const int woff[8] = {W_CONV1, W_L1C1, W_L1C2, W_L1DN, W_L2C1, W_L2C2, W_L2DN, W_CONV2};
  const int boff[8] = {B_CONV1, B_L1C1, B_L1C2, B_L1DN, B_L2C1, B_L2C2, B_L2DN, B_CONV2};
  const int ci_n[8] = {3, 32, 32, 32, 32, 32, 32, 32};
  const int kk[8] = {3, 3, 3, 1, 3, 3, 1, 1};
  for (int l = 0; l < 8; ++l) {
    const int CI = ci_n[l], K = kk[l], CH = (CI + 3) / 4, n = K * K * CH * 32 * 4;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
      // [tap][c4][k][cq][e]: output channel 4 cq + k, input channel 4 c4 + e
      const int e = i & 3, cq = (i >> 2) & 7, k = (i >> 5) & 3, r = i >> 7, c4 = r % CH, tap = r / CH;
      const int co = cq * 4 + k, ci = c4 * 4 + e;
      pp.packed[woff[l] + i] = ci < CI ? __ldg(pp.t[2 * l] + ((long long)co * CI + ci) * K * K + tap) : 0.f;
    }
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 32; i += gridDim.x * blockDim.x)
      pp.packed[boff[l] + i] = __ldg(pp.t[2 * l + 1] + i);
  }
}

}  // namespace senc
}  // namespace comet

using namespace comet;

extern "C" long long comet_shallow_encoder_packed_elems(void) { return senc::PACKED_FLOATS; }

extern "C" int comet_shallow_encoder_pack_f32(const float* const* params_host, float* packed, comet_stream_t stream) {
  COMET_REQUIRE(params_host && packed, "null pointer");
  senc::PackParams pp;
  for (int i = 0; i < 16; ++i) {
    COMET_REQUIRE(params_host[i], "parameter %d is null", i);
    pp.t[i] = params_host[i];
  }
  pp.packed = packed;
  senc::shallow_encoder_pack_kernel<<<32, 256, 0, (cudaStream_t)stream>>>(pp);
  return launch_status("shallow_encoder_pack_kernel");
}

template <bool PACKED>
static int launch_shallow_encoder(const senc::Params& p, comet_stream_t stream) {
  static bool configured[64] = {false};
  int dev = 0;
  COMET_CUDA(cudaGetDevice(&dev));
  COMET_REQUIRE(device_sm_count_if_sm100() > 0, "the fused patch encoder needs an sm_100 device");
  if (dev < 64 && !configured[dev]) {
    COMET_CUDA(cudaFuncSetAttribute(senc::shallow_encoder_kernel<PACKED>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    senc::SMEM_BYTES));
    configured[dev] = true;
  }
  const int sms = device_sm_count_if_sm100();
  long long ctas = (p.P + senc::G - 1) / senc::G;
  if (ctas > sms) ctas = sms;    // persistent: one CTA per SM, patch pairs strided over the grid
  senc::shallow_encoder_kernel<PACKED><<<(unsigned)ctas, senc::THREADS, senc::SMEM_BYTES, (cudaStream_t)stream>>>(p);
  return launch_status(PACKED ? "shallow_encoder_kernel<packed>" : "shallow_encoder_kernel");
}

extern "C" int comet_shallow_encoder_f32(const float* patches, long long sn, long long sc, long long sy, long long sx,
                                         const float* packed, float* out, long long P, float eps, comet_stream_t stream) {
  COMET_REQUIRE(P >= 0, "bad shape");
  if (P == 0) return COMET_OK;
  COMET_REQUIRE(patches && packed && out, "null pointer");
  COMET_REQUIRE(((uintptr_t)packed % 16) == 0, "packed parameters must be 16-byte aligned");
  senc::Params p{};
  p.src = patches; p.topleft = nullptr; p.packed = packed; p.out = out; p.P = P;
  p.sn = sn; p.sc = sc; p.sy = sy; p.sx = sx;
  p.S = 1; p.N = 1; p.H = senc::PSZ; p.W = senc::PSZ; p.eps = eps;
  return launch_shallow_encoder<false>(p, stream);
}

extern "C" int comet_shallow_encoder_from_images_f32(const float* images, const int* topleft, const float* packed, float* out,
                                                     int B, int S, int N, int H, int W, float eps, comet_stream_t stream) {
  COMET_REQUIRE(B >= 0 && S >= 0 && N >= 0 && H >= senc::PSZ && W >= senc::PSZ, "bad shape");
  const long long P = (long long)B * S * N;
  if (P == 0) return COMET_OK;
  COMET_REQUIRE(images && topleft && packed && out, "null pointer");
  COMET_REQUIRE(((uintptr_t)packed % 16) == 0, "packed parameters must be 16-byte aligned");
  senc::Params p{};
  p.src = images; p.topleft = topleft; p.packed = packed; p.out = out; p.P = P;
  p.sn = 0; p.sc = (long long)H * W; p.sy = W; p.sx = 1;
  p.S = S; p.N = N; p.H = H; p.W = W; p.eps = eps;
  return launch_shallow_encoder<false>(p, stream);
}

extern "C" int comet_shallow_encoder_from_images_indexed_f32(const float* images, const int* topleft, const int* seq_of_track,
                                                             const int* num_frames, const int* frame_index, int BS_src,
                                                             const float* packed, float* out, int P, int B, int S, int H, int W,
                                                             float eps, comet_stream_t stream) {
  COMET_REQUIRE(P >= 0 && B >= 1 && S >= 0 && H >= senc::PSZ && W >= senc::PSZ, "bad shape");
  COMET_REQUIRE(!frame_index || BS_src >= 1, "BS_src must be positive with a frame table (got %d)", BS_src);
  if ((long long)P * S == 0) return COMET_OK;
  COMET_REQUIRE(images && topleft && seq_of_track && packed && out, "null pointer");
  COMET_REQUIRE(((uintptr_t)packed % 16) == 0, "packed parameters must be 16-byte aligned");
  senc::Params p{};
  p.src = images; p.topleft = topleft; p.seq_of_track = seq_of_track; p.num_frames = num_frames; p.packed = packed; p.out = out;
  p.frame_index = frame_index; p.nframes_src = BS_src;
  p.P = (long long)P * S;
  p.sn = 0; p.sc = (long long)H * W; p.sy = W; p.sx = 1;
  p.S = S; p.N = P; p.H = H; p.W = W; p.nseq = B; p.eps = eps;
  return launch_shallow_encoder<false>(p, stream);
}

extern "C" int comet_shallow_encoder_from_images_packed_f32(const float* frames, const long long* frame_offset,
                                                            const int* frame_hw, long long num_packed_frames,
                                                            const int* topleft, const int* seq_of_track, const int* num_frames,
                                                            const int* frame_index, const float* packed, float* out, int P,
                                                            int B, int S, float eps, comet_stream_t stream) {
  COMET_REQUIRE(P >= 0 && B >= 1 && S >= 0 && num_packed_frames >= 1, "bad shape");
  if ((long long)P * S == 0) return COMET_OK;
  COMET_REQUIRE(frames && frame_offset && frame_hw && topleft && seq_of_track && packed && out, "null pointer");
  COMET_REQUIRE(((uintptr_t)packed % 16) == 0, "packed parameters must be 16-byte aligned");
  senc::Params p{};
  p.src = frames; p.topleft = topleft; p.seq_of_track = seq_of_track; p.num_frames = num_frames; p.packed = packed; p.out = out;
  p.frame_index = frame_index; p.nframes_src = num_packed_frames;
  p.frame_offset = frame_offset; p.frame_hw = frame_hw;
  p.P = (long long)P * S;
  p.sn = 0; p.sc = 0; p.sy = 0; p.sx = 1;
  p.S = S; p.N = P; p.H = senc::PSZ; p.W = senc::PSZ; p.nseq = B; p.eps = eps;
  return launch_shallow_encoder<true>(p, stream);
}

extern "C" int comet_shallow_encoder_from_images_varlen_f32(const float* images, const int* topleft, const int* seq_of_track,
                                                            const int* num_frames, const float* packed, float* out, int P, int B,
                                                            int S, int H, int W, float eps, comet_stream_t stream) {
  return comet_shallow_encoder_from_images_indexed_f32(images, topleft, seq_of_track, num_frames, nullptr, B * S, packed, out, P,
                                                       B, S, H, W, eps, stream);
}

extern "C" int comet_shallow_encoder_from_images_ragged_f32(const float* images, const int* topleft, const int* seq_of_track,
                                                            const float* packed, float* out, int P, int B, int S, int H, int W,
                                                            float eps, comet_stream_t stream) {
  return comet_shallow_encoder_from_images_varlen_f32(images, topleft, seq_of_track, nullptr, packed, out, P, B, S, H, W, eps,
                                                      stream);
}
