/*
 * comet_b200.h -- C ABI of the B200-native COMET tracking hot path.
 *
 * The reference (wulibingbinglin/COMET-Pose-Estimation) is pure Python/PyTorch
 * and has no FFI: its "plugin interface" for this path is the set of Python
 * symbols listed in SURVEY.md section 8(b).  Every entry point below replaces
 * the arithmetic behind one of those symbols; the Python mirror in
 * comet_pose_estimation_b200/ binds them with ctypes (see INTEGRATION.md for
 * the stub a maintainer of the reference would add).
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - tensors are float32, innermost dimension contiguous; where a tensor may
 *     be a permuted view the element strides of its outer dimensions are
 *     passed explicitly (sb, ss, sn = batch, frame, track);
 *   - coordinates are (x, y) pairs in level-0 cell units;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - every function returns COMET_OK (0) or an error code and never throws;
 *     comet_last_error() returns a thread-local description of the last
 *     failure.  Launches are asynchronous on `stream`.
 *   - there is no CPU fallback: without a CUDA device every compute entry
 *     point fails with COMET_ERR_CUDA.
 *
 * Reference citations are file:line into the reference repository.
 */
#ifndef COMET_B200_H
#define COMET_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define COMET_OK 0
#define COMET_ERR_INVALID 1     /* bad argument (the reference would raise AssertionError) */
#define COMET_ERR_CUDA 2        /* CUDA runtime / launch failure */
#define COMET_ERR_UNSUPPORTED 3 /* shape outside what the kernels implement */

#define COMET_PAD_ZEROS 0  /* CorrBlock default, blocks.py:357 */
#define COMET_PAD_BORDER 1 /* EfficientCorrBlock / bilinear_sampler default, utils.py:874 */

#define COMET_PREC_F32 0           /* float32 arithmetic everywhere (parity bar 1e-4) */
#define COMET_PREC_BF16_AUTOCAST 1 /* what torch.autocast(bf16) makes of CorrBlock.corr: bf16 operands,
                                      f32 accumulate, volume rounded to bf16, f32 lookup (bar 2e-2) */

#define COMET_PYR_NCHW 0         /* pyramid levels 1..L-1 stored (BS, C, H_l, W_l), like the reference */
#define COMET_PYR_CHANNEL_LAST 1 /* ... stored (BS, H_l, W_l, C): one contiguous line per position (fine tracker) */
#define COMET_PYR_ALL_CHANNEL_LAST 2 /* as 1, and level 0 (the caller's fmaps) is channel-last (BS, H, W, C) too */
#define COMET_PYR_UP2_SOURCE 3       /* level 0 is NOT stored: `fmaps` is the half-resolution map S (BS, Hs, Ws, C),
                                        channel-last, whose bilinear align_corners up-sampling to (H, W) = (2Hs-1, 2Ws-1)
                                        is the level-0 map (ShallowEncoder's last op, blocks.py:176-190); levels 0 and 1
                                        are evaluated from S inside the lookup, `pyr` holds level L-1 = 2 only
                                        (BS, H/4, W/4, C), written by comet_pyramid_up2_f32.  C=32, L=3, r=3, zeros. */

#define COMET_FMAPS_NCHW 0         /* fmaps (BS, C, H, W) contiguous, as the reference's encoders return them */
#define COMET_FMAPS_CHANNEL_LAST 1 /* fmaps (BS, H, W, C) dense: a torch.channels_last encoder output, used zero-copy */

#define COMET_MAX_LEVELS 8
#define COMET_MAX_RADIUS 7

typedef void* comet_stream_t;

/* ---- library ---------------------------------------------------------- */
int comet_version(void);
const char* comet_last_error(void);
/* 1 if the tcgen05/TMEM/TMA correlation kernels were compiled in, the current device is sm_100 and
 * COMET_OPT_TENSOR_PATH is on. */
int comet_has_tensor_path(void);
/* Library-wide switches for A/B measurements (no environment variable is read on the launch path):
 *   COMET_OPT_TENSOR_PATH  the tcgen05 kernels serve the dense coarse shape; off = general SIMT kernels
 *   COMET_OPT_TMA_LOOKUP   the TMA-staged C=32 lookup serves channel-last small maps; off = register version */
#define COMET_OPT_TENSOR_PATH 0
#define COMET_OPT_TMA_LOOKUP 1
#define COMET_OPT_GEMM_BK32 2   /* float32-grade GEMM: K=32 pipeline stages (64-byte swizzle, 4 in flight) instead of K=64 (2 in
                                   flight).  OFF by default: measured 7.28 vs 6.16 ms per coarse forward (scripts/gemm_ab.py) */
#define COMET_OPT_TC_OVERLAP_MISC 3 /* coarse tokens: the correlation-independent channels as a third launch that runs BESIDE the
                                      tensor kernel (programmatic dependent launch) instead of before it.  OFF by default:
                                      measured 0.155 vs 0.112 ms per iteration (scripts/coarse_ab.py) -- the tensor CTAs leave
                                      room for 4 warps per SM, too few for a bandwidth kernel */
#define COMET_OPT_TC_REDUCE_STORE 4 /* coarse tokens: the windows are added to the token rows by bulk reductions
                                      (cp.reduce.async.bulk add.f32, one per query and level) onto the position embedding the
                                      pre-kernel wrote there; off = per-entry stores by the stager warps.  ON by default */
#define COMET_OPT_GEMM_TMA_STORE 5 /* transformer GEMM: results leave through shared memory and bulk tensor stores (full
                                    128-byte lines) instead of per-lane row stores; on by default */
#define COMET_OPT_GEMM_EW16 6 /* transformer GEMM, one-plane (autocast) mode: sixteen epilogue warps instead of eight */
#define COMET_OPT_GEMM_BN96 7 /* transformer GEMM: 96-column output tiles where they divide N and save a round of CTAs */
#define COMET_OPT_GEMM_PAIR 8 /* transformer GEMM: clusters of two CTAs share every W tile (each loads half and multicasts it);
                                bit mask: 1 float32-grade mode (K >= 1024: the default), 2 autocast mode, 4 any K */
#define COMET_OPT_ATTN_MMA 9 /* autocast mode: attention on the tensor cores (mma.sync bf16); bit mask: 1 = at least 64 queries,
                                 2 = the short time attention (at most 16 queries, 32 keys) */
#define COMET_OPT_COUNT 10
int comet_set_option(int option, int value);
int comet_get_option(int option);
/* Number of kernel launches this library has issued since it was loaded (bench.py's `gpu_launches`). */
long long comet_launch_count(void);

/* ---- feature pyramid: CorrBlock.__init__ / EfficientCorrBlock.__init__,
 *      comet/models/track_modules/blocks.py:352-374 and :433-444 ------------
 * Level 0 is the caller's `fmaps` (BS, C, H, W).  Levels 1..L-1 (2x2 average
 * pooling, stride 2, floor sizes) are written back to back into `pyr`:
 * level l occupies BS*C*H_l*W_l floats starting at comet_pyramid_offset(l). */
long long comet_pyramid_offset(int BS, int C, int H, int W, int level); /* elements; level>=1 */
long long comet_pyramid_elems(int BS, int C, int H, int W, int L);      /* total for levels 1..L-1 */
int comet_pyramid_f32(const float* fmaps, float* pyr, int BS, int C, int H, int W, int L, comet_stream_t stream);
/* Same pooling, levels 1..L-1 written channel-last (COMET_PYR_CHANNEL_LAST) at the same offsets.
 * COMET_FMAPS_NCHW input requires W <= 32, H <= 33 and a pooled tile that fits shared memory (small maps: the fine
 * tracker's patches); COMET_FMAPS_CHANNEL_LAST input requires C % 4 == 0 and 16-byte aligned buffers. */
int comet_pyramid_cl_f32(const float* fmaps, float* pyr, int BS, int C, int H, int W, int L, int fmaps_layout,
                         comet_stream_t stream);

/* Level 2 of the pyramid of the up-sampled map, straight from the half-resolution source (COMET_PYR_UP2_SOURCE):
 * src (BS, Hs, Ws, C) channel-last -> p2 (BS, (Hs-1)/2, (Ws-1)/2, C) channel-last.  Replaces, for this package's own
 * refine_track, the reference's F.interpolate (blocks.py:176-190) + CorrBlock.__init__ pooling (blocks.py:368-374). */
long long comet_pyramid_up2_elems(int BS, int C, int Hs, int Ws);
int comet_pyramid_up2_f32(const float* src, float* p2, int BS, int C, int Hs, int Ws, comet_stream_t stream);
/* 1 if (C, level-0 H x W, L, r, pad_mode) is served by COMET_PYR_UP2_SOURCE on the current device. */
int comet_up2_supported(int C, int H, int W, int L, int r, int pad_mode);

/* ---- correlation volume: CorrBlock.corr, blocks.py:409-429 -------------
 * vol[bs, n, hw] = (sum_c targets[bs, n, c] * fmap[bs, c, hw]) / sqrt(C) for ONE pyramid level.
 * Provided for API completeness (CorrBlock.corrs_pyramid); the product path never materialises it. */
int comet_corr_volume_f32(const float* targets, long long t_sbs, long long t_sn, const float* fmap_level, float* vol,
                          int BS, int N, int C, int HW, int prec_mode, comet_stream_t stream);

/* ---- fused correlation + window lookup: CorrBlock.corr + CorrBlock.sample
 *      (blocks.py:376-429, padding zeros) and EfficientCorrBlock.sample
 *      (blocks.py:446-484, padding border) ---------------------------------
 * out[b,s,n, l*(2r+1)^2 + i*(2r+1) + j] = bilinear(V_l[b,s,n], x/2^l + (i-r), y/2^l + (j-r))
 * (the x offset is the slow index, as in the reference).  The volume V_l is never written to memory.
 * targets: (B,S,N,C) view with element strides t_sb,t_ss,t_sn (C contiguous); t_level_stride = 0, or C for
 * `multiple_track_feats` (targets then hold L*C channels, level l uses channels [l*C,(l+1)*C)).
 * coords: (B,S,N,2) view with strides c_sb,c_ss,c_sn.  out: element strides o_sb,o_ss,o_sn, innermost contiguous. */
int comet_corr_lookup_f32(const float* fmaps, const float* pyr, const float* targets, long long t_sb, long long t_ss,
                          long long t_sn, int t_level_stride, const float* coords, long long c_sb, long long c_ss,
                          long long c_sn, float* out, long long o_sb, long long o_ss, long long o_sn, int B, int S,
                          int N, int C, int H, int W, int L, int r, int pad_mode, int prec_mode, int pyr_layout,
                          comet_stream_t stream);

/* ---- fused track tokens: the token assembly of BaseTrackerPredictor.forward,
 *      comet/models/track_modules/base_track_predictor.py:153-224 ----------
 * tokens[b,n,s,:] = [ sin/cos(flow) (latent) | flow (2) | fcorrs (L*(2r+1)^2) | track_feats (latent) | 0 pad ]
 *                   + pos_emb[b,n,:]
 * with flow = coords[b,s,n] - coords[b,0,n] and fcorrs computed as in comet_corr_lookup_f32 (never stored
 * separately).  pos_emb (B,N,D_tok) comes from comet_sampled_pos_emb_f32 and is iteration-invariant.
 * latent == C.  tokens is (B,N,S,D_tok) contiguous. */
int comet_track_tokens_f32(const float* fmaps, const float* pyr, const float* track_feats, long long t_sb,
                           long long t_ss, long long t_sn, const float* coords, long long c_sb, long long c_ss,
                           long long c_sn, const float* pos_emb, float* tokens, int B, int S, int N, int C, int H,
                           int W, int L, int r, int pad_mode, int prec_mode, int pyr_layout, int D_tok,
                           comet_stream_t stream);
/* The same for a batch of sequences with different track counts: num_tracks (B,) int32 in DEVICE memory, 1 <= num_tracks[b]
 * <= N.  Queries n >= num_tracks[b] are padding: their token rows are written as zeros and nothing else is computed for
 * them; every other row equals comet_track_tokens_f32 on sequence b alone with N = num_tracks[b].  Not served for
 * COMET_PYR_UP2_SOURCE or C == 32 (COMET_ERR_UNSUPPORTED / COMET_ERR_INVALID). */
int comet_track_tokens_ragged_f32(const float* fmaps, const float* pyr, const float* track_feats, long long t_sb,
                                  long long t_ss, long long t_sn, const float* coords, long long c_sb, long long c_ss,
                                  long long c_sn, const float* pos_emb, float* tokens, const int* num_tracks, int B, int S,
                                  int N, int C, int H, int W, int L, int r, int pad_mode, int prec_mode, int pyr_layout,
                                  int D_tok, comet_stream_t stream);
/* The same with per-sequence track counts and / or frame counts (num_tracks, num_frames: (B,) int32 in DEVICE memory, each
 * nullable).  Rows of frames s >= num_frames[b] are written as zeros and read nothing; every other row equals
 * comet_track_tokens_f32 on sequence b alone.  Frame counts are also served for COMET_PYR_UP2_SOURCE (track counts are
 * not); neither is served for the other C == 32 layouts. */
int comet_track_tokens_varlen_f32(const float* fmaps, const float* pyr, const float* track_feats, long long t_sb,
                                  long long t_ss, long long t_sn, const float* coords, long long c_sb, long long c_ss,
                                  long long c_sn, const float* pos_emb, float* tokens, const int* num_tracks,
                                  const int* num_frames, int B, int S, int N, int C, int H, int W, int L, int r, int pad_mode,
                                  int prec_mode, int pyr_layout, int D_tok, comet_stream_t stream);
/* The same for B items that read the BS_src frames of fmaps / pyr (pyramid of all BS_src frames, as comet_pyramid_f32 lays it
 * out for BS = BS_src) in their own order: frame_index (B,S) int32 in device memory gives the frame that item b reads at
 * position s (entries outside [0, BS_src) are clamped).  BS_src need not be a multiple of S, and a table may reference any
 * source frame any number of times, within a row or across rows.  Coordinates, track features, position embedding and tokens stay
 * per (item, position); num_tracks / num_frames keep their meaning.  Every row equals comet_track_tokens_varlen_f32 on
 * fmaps gathered as fmaps.reshape(BS_src, ...)[frame_index].  frame_index NULL is comet_track_tokens_varlen_f32.  The
 * C == 32 layouts serve a frame table without counts; COMET_PYR_UP2_SOURCE serves none. */
int comet_track_tokens_indexed_f32(const float* fmaps, const float* pyr, const float* track_feats, long long t_sb,
                                   long long t_ss, long long t_sn, const float* coords, long long c_sb, long long c_ss,
                                   long long c_sn, const float* pos_emb, float* tokens, const int* num_tracks,
                                   const int* num_frames, const int* frame_index, int BS_src, int B, int S, int N, int C, int H,
                                   int W, int L, int r, int pad_mode, int prec_mode, int pyr_layout, int D_tok,
                                   comet_stream_t stream);

/* sampled_pos_emb = sample_features4d(get_2d_sincos_pos_embed(D,(H,W)), coords[:,0])
 * (base_track_predictor.py:200-208; utils.py:724-755, :942-974): the float64 table is evaluated on the fly at
 * the four integer taps, cast to float32 and blended -- no table is stored.  coords0: (B,N,2) view with strides
 * c_sb, c_sn.  out (B,N,D) contiguous.  D % 4 == 0. */
int comet_sampled_pos_emb_f32(const float* coords0, long long c_sb, long long c_sn, float* out, int B, int N, int D,
                              int H, int W, comet_stream_t stream);

/* ---- samplers: comet/models/utils.py:874-974 --------------------------- */
/* bilinear_sampler, 4-D input (B,C,H,W), coords (B,Ho,Wo,2)=(x,y) in pixels -> out (B,C,Ho,Wo). */
int comet_bilinear_sampler4d_f32(const float* input, const float* coords, float* out, int B, int C, int H, int W,
                                 int Ho, int Wo, int align_corners, int pad_mode, comet_stream_t stream);
/* bilinear_sampler, 5-D input (B,C,T,H,W), coords (B,Do,Ho,Wo,3)=(t,x,y) -> out (B,C,Do,Ho,Wo). */
int comet_bilinear_sampler5d_f32(const float* input, const float* coords, float* out, int B, int C, int T, int H,
                                 int W, int Do, int Ho, int Wo, int align_corners, int pad_mode,
                                 comet_stream_t stream);
/* sample_features4d: input (B,C,H,W) with batch stride in_sb (elements), coords (B,R,2) with strides c_sb,c_sr
 * -> out (B,R,C) contiguous; border padding, align_corners=True. */
int comet_sample_features4d_f32(const float* input, long long in_sb, const float* coords, long long c_sb,
                                long long c_sr, float* out, int B, int C, int H, int W, int R,
                                comet_stream_t stream);

/* Same, input channel-last (B,H,W,C) with batch stride in_sb (0 = one map shared by the whole batch, e.g. the cached
 * sin/cos table): every tap is one contiguous C-float line. */
int comet_sample_features4d_cl_f32(const float* input, long long in_sb, const float* coords, long long c_sb,
                                   long long c_sr, float* out, int B, int C, int H, int W, int R,
                                   comet_stream_t stream);

/* ---- bilinear resize, align_corners=True: the F.interpolate calls of the fine tracker's patch encoder
 *      (ShallowEncoder.forward, comet/models/track_modules/blocks.py:176-190), whose last one produces the fine
 *      tracker's fmaps.  in (N,C,Hi,Wi) -> out (N,C,Ho,Wo), both COMET_FMAPS_NCHW or both COMET_FMAPS_CHANNEL_LAST. */
int comet_upsample_bilinear_ac_f32(const float* in, float* out, long long N, int C, int Hi, int Wi, int Ho, int Wo,
                                   int layout, comet_stream_t stream);

/* The same for bf16 tensors in NCHW layout (float32 arithmetic, result rounded to bf16). */
int comet_upsample_bilinear_ac_bf16(const void* in, void* out, long long N, int C, int Hi, int Wi, int Ho, int Wo,
                                    comet_stream_t stream);

/* nn.InstanceNorm2d(affine=False, eps) (+ ReLU when relu != 0) of the same encoder (blocks.py:128-131,
 * comet/models/modules.py:86-90): per (sample, channel) plane of HW elements, biased variance. */
int comet_instance_norm_f32(const float* in, float* out, long long N, int C, int HW, int layout, int relu, float eps,
                            comet_stream_t stream);

/* The same for bf16 tensors in NCHW layout (the encoders under torch.autocast: statistics in float32 of the bf16 values,
 * result rounded to bf16). */
int comet_instance_norm_bf16(const void* in, void* out, long long N, int C, int HW, int relu, float eps, comet_stream_t stream);

/* Patch gather of refine_track (comet/models/refine_track.py:71-111): images (B,S,C,H,W) contiguous, topleft (B,S,N,2)
 * int32 (x, y) corners already clamped to [0, W-P] x [0, H-P] -> out (B*N*S, P, P, C) channel-last, patches in
 * (b, n, s) order. */
int comet_extract_patches_f32(const float* images, const int* topleft, float* out, int B, int S, int N, int C, int H, int W,
                              int P, comet_stream_t stream);

/* ---- ShallowEncoder, the patch encoder of the fine tracker, as one kernel ---------------------------------------
 * comet/models/track_modules/blocks.py:114-196 (norm_fn="instance", input_dim 3, output_dim 32, 31x31 patches) with
 * ResidualBlock of comet/models/modules.py:39-117: conv1 3x3/2 -> InstanceNorm -> ReLU -> layer1 -> layer2 -> two
 * bilinear residual up-samplings -> conv2 1x1 + skip, every intermediate map in shared memory, float32 FMA.
 * The result is the 16x16 map *before* the encoder's final resize to 31x31 (blocks.py:183-190), channel-last:
 * out (P, 16, 16, 32) -- what COMET_PYR_UP2_SOURCE consumes; comet_upsample_bilinear_ac_f32 gives the 31x31 map.
 *
 * comet_shallow_encoder_pack_f32: params_host is a HOST array of 16 DEVICE pointers in state-dict order
 *   conv1.{weight,bias}, layer1.conv1.{w,b}, layer1.conv2.{w,b}, layer1.downsample.0.{w,b}, layer2.(same six),
 *   conv2.{w,b} (contiguous OIHW float32) -> packed (comet_shallow_encoder_packed_elems() floats, 16-byte aligned).
 * comet_shallow_encoder_f32: patches (P,3,31,31) with element strides (sn, sc, sy, sx) -- any memory format.
 * comet_shallow_encoder_from_images_f32: fuses the patch gather of refine_track.py:71-111 (same arguments as
 *   comet_extract_patches_f32 with C = 3, P = 31): patch (b, n, s) is read straight from images (B,S,3,H,W). */
long long comet_shallow_encoder_packed_elems(void);
int comet_shallow_encoder_pack_f32(const float* const* params_host, float* packed, comet_stream_t stream);
int comet_shallow_encoder_f32(const float* patches, long long sn, long long sc, long long sy, long long sx,
                              const float* packed, float* out, long long P, float eps, comet_stream_t stream);
int comet_shallow_encoder_from_images_f32(const float* images, const int* topleft, const float* packed, float* out,
                                          int B, int S, int N, int H, int W, float eps, comet_stream_t stream);
/* The same for P tracks packed from several sequences of images (B,S,3,H,W): topleft (P,S,2) int32 corners, seq_of_track
 * (P,) int32 the sequence of each track (device memory).  out (P*S, 16, 16, 32) in (track, frame) order; each map is
 * bit-identical to comet_shallow_encoder_from_images_f32 on the same patch. */
int comet_shallow_encoder_from_images_ragged_f32(const float* images, const int* topleft, const int* seq_of_track,
                                                 const float* packed, float* out, int P, int B, int S, int H, int W,
                                                 float eps, comet_stream_t stream);
/* The same for sequences with different frame counts: num_frames (B,) int32 in device memory, or NULL (= the call above).
 * The pixels of frames s >= num_frames[seq_of_track[p]] are never read, and their maps are written as zeros. */
int comet_shallow_encoder_from_images_varlen_f32(const float* images, const int* topleft, const int* seq_of_track,
                                                 const int* num_frames, const float* packed, float* out, int P, int B, int S,
                                                 int H, int W, float eps, comet_stream_t stream);
/* The same where frame s of sequence b reads image frame frame_index[b * S + s] of the BS_src frames of `images`
 * ((BS_src, 3, H, W) viewed flat; frame_index (B,S) int32 in device memory, entries clamped to [0, BS_src)) instead of
 * frame b * S + s.  BS_src need not be a multiple of S, and a table may reference any source frame any number of times.
 * frame_index NULL is the call above. */
int comet_shallow_encoder_from_images_indexed_f32(const float* images, const int* topleft, const int* seq_of_track,
                                                  const int* num_frames, const int* frame_index, int BS_src,
                                                  const float* packed, float* out, int P, int B, int S, int H, int W,
                                                  float eps, comet_stream_t stream);
/* The same reading a packed frame buffer of frames with different sizes: frame f starts at element frame_offset[f] of
 * `frames` (int64) and is frame_hw[2f] x frame_hw[2f+1] pixels (H, W; int32), stored (3, H, W) contiguous; both tables
 * in device memory, num_packed_frames entries.  Frame ids (b * S + s, or frame_index[b * S + s]) index the packed frames
 * and are clamped to [0, num_packed_frames); a table may reference any packed frame any number of times.  Each corner
 * is clamped to its own frame, [0, W_f - 31] x [0, H_f - 31], so no read leaves the frame; a frame smaller than 31x31 is
 * not read.  Each map is bit-identical to
 * comet_shallow_encoder_from_images_indexed_f32 on a buffer holding that frame. */
int comet_shallow_encoder_from_images_packed_f32(const float* frames, const long long* frame_offset, const int* frame_hw,
                                                 long long num_packed_frames, const int* topleft, const int* seq_of_track,
                                                 const int* num_frames, const int* frame_index, const float* packed,
                                                 float* out, int P, int B, int S, float eps, comet_stream_t stream);

/* ---- sin/cos encodings: comet/models/utils.py:37-101, :724-832 ----------- */
/* get_2d_embedding(xy, C, cat_coords): xy (M,2) contiguous -> out (M, 2*C [+2 in front if cat_coords]). */
int comet_embed2d_f32(const float* xy, float* out, long long M, int C, int cat_coords, comet_stream_t stream);
/* get_1d_sincos_pos_embed_from_grid(D, pos): pos (M) float32 -> out (M, D) = [sin | cos], float64 inside. */
int comet_sincos1d_from_grid_f32(const float* pos, float* out, long long M, int D, comet_stream_t stream);
/* get_2d_sincos_pos_embed(D, (H,W)) -> out (D, H, W); channel order [sin_x | cos_x | sin_y | cos_y]. */
int comet_sincos2d_f32(float* out, int D, int H, int W, comet_stream_t stream);

/* ---- tensor-core path (tcgen05 + TMEM + TMA), coarse-tracker shape only --------------------------------------
 * Same results as comet_corr_lookup_f32 / comet_track_tokens_f32 / comet_corr_volume_f32 for
 * C=128, H=W=64, L<=5, r<=4, zero padding; float32 parity through a bf16 hi/lo split (3 MMA passes), or the
 * autocast rounding with one pass.  `split` is the packed bf16 pyramid written by comet_tc_prepare_f32
 * (comet_tc_split_elems(BS) bf16 elements); `pyr` (optional, may be NULL) additionally receives the float32 levels
 * 1..L-1 in the comet_pyramid_f32 layout.
 * `workspace`: comet_tc_workspace_bytes(B*S, N) bytes of 16-byte aligned device scratch, rewritten by every call: the
 * queries of each frame are counting-sorted by floor(y) so that the 128 queries of an MMA tile share a narrow band
 * of map rows, and the per-tile job list (which feature tiles each band needs) lives there too.  Results do not
 * depend on the order (every query writes its own output row). */
int comet_tc_supported(int C, int H, int W, int L, int r, int pad_mode);
long long comet_tc_split_elems(int BS);
long long comet_tc_workspace_bytes(int BS, int N);
int comet_tc_prepare_f32(const float* fmaps, void* split, float* pyr, int BS, int C, int H, int W, int L,
                         comet_stream_t stream);
int comet_tc_corr_lookup_f32(const void* split, const float* targets, long long t_sb, long long t_ss, long long t_sn,
                             const float* coords, long long c_sb, long long c_ss, long long c_sn, float* out,
                             long long o_sb, long long o_ss, long long o_sn, int B, int S, int N, int C, int H, int W,
                             int L, int r, int pad_mode, int prec_mode, void* workspace, comet_stream_t stream);
int comet_tc_track_tokens_f32(const void* split, const float* track_feats, long long t_sb, long long t_ss,
                              long long t_sn, const float* coords, long long c_sb, long long c_ss, long long c_sn,
                              const float* pos_emb, float* tokens, int B, int S, int N, int C, int H, int W, int L,
                              int r, int pad_mode, int prec_mode, int D_tok, void* workspace, comet_stream_t stream);
/* comet_tc_track_tokens_f32 for a batch of sequences with different track counts (num_tracks (B,) int32, device memory;
 * see comet_track_tokens_ragged_f32).  Padded queries are left out of the sort: they occupy no tile slot, and a tile
 * that holds none of them is an empty one-row job.  Real rows are bit-identical to the single-sequence call. */
int comet_tc_track_tokens_ragged_f32(const void* split, const float* track_feats, long long t_sb, long long t_ss,
                                     long long t_sn, const float* coords, long long c_sb, long long c_ss, long long c_sn,
                                     const float* pos_emb, float* tokens, const int* num_tracks, int B, int S, int N, int C,
                                     int H, int W, int L, int r, int pad_mode, int prec_mode, int D_tok, void* workspace,
                                     comet_stream_t stream);
/* The same with per-sequence track counts and / or frame counts (each nullable, device memory).  A padded frame sorts no
 * query, so each of its tiles is an empty one-row job, and the pre-kernel writes its token rows as zeros. */
int comet_tc_track_tokens_varlen_f32(const void* split, const float* track_feats, long long t_sb, long long t_ss,
                                     long long t_sn, const float* coords, long long c_sb, long long c_ss, long long c_sn,
                                     const float* pos_emb, float* tokens, const int* num_tracks, const int* num_frames,
                                     int B, int S, int N, int C, int H, int W, int L, int r, int pad_mode, int prec_mode,
                                     int D_tok, void* workspace, comet_stream_t stream);
/* The same for B items that read the BS_src frames of `split` (comet_tc_prepare_f32 with BS = BS_src) in their own order:
 * frame_index (B,S) int32 in device memory, entries clamped to [0, BS_src); BS_src need not be a multiple of S, and a
 * table may reference any source frame any number of times.  The plan kernel reads each frame's entry once
 * and stores it in that frame's job records, from which the operand producer addresses its tiles.  Everything else stays
 * per (item, position), including `workspace` (comet_tc_workspace_bytes(B*S, N)).  Rows are bit-identical to
 * comet_tc_track_tokens_varlen_f32 on a split prepared from the gathered frames.  frame_index NULL is that call. */
int comet_tc_track_tokens_indexed_f32(const void* split, const float* track_feats, long long t_sb, long long t_ss,
                                      long long t_sn, const float* coords, long long c_sb, long long c_ss, long long c_sn,
                                      const float* pos_emb, float* tokens, const int* num_tracks, const int* num_frames,
                                      const int* frame_index, int BS_src, int B, int S, int N, int C, int H, int W, int L,
                                      int r, int pad_mode, int prec_mode, int D_tok, void* workspace, comet_stream_t stream);
/* vols: HOST array of L device pointers, level l = (B*S, N, H_l*W_l) float32. */
int comet_tc_corr_volume_f32(const void* split, const float* targets, long long t_sb, long long t_ss, long long t_sn,
                             float* const* vols, int B, int S, int N, int C, int H, int W, int L, int prec_mode,
                             void* workspace, comet_stream_t stream);
/* 0 = healthy; non-zero = the pipeline watchdog of the tensor kernel fired (a wait exceeded 10 s of wall time; the
 * kernel trapped and the CUDA context is lost): which wait it was.  Synchronises with the device. */
int comet_tc_status(void);

/* ---- track-update transformer: EfficientUpdateFormer (comet/models/track_modules/blocks.py:205-348) and its
 *      AttnBlock / CrossAttnBlock / Mlp (comet/models/modules.py:119-154, :248-344) --------------------------------------
 * Activations that feed a GEMM are held as "bf16 planes": np bf16 matrices p0 = bf16(x), p1 = bf16(x - p0),
 * p2 = bf16(x - p0 - p1), spaced plane_stride ELEMENTS apart.  np = 1 is torch.autocast(bf16) precision (COMET's shipped
 * mixed_precision), np = 3 is float32-grade (six tensor-core passes over the plane pairs i + j <= 2). */
/* x (rows, cols) float32 with row pitch x_ld -> np planes with row pitch p_ld. */
int comet_split_planes_f32(const float* x, long long x_ld, void* planes, long long plane_stride, long long p_ld,
                           long long rows, int cols, int np, comet_stream_t stream);
/* nn.Linear on tcgen05: Y[M,N] = act(X[M,K] . W[N,K]^T + bias) (+ resid).  X / W as np planes (row pitches x_ld / w_ld
 * elements, multiples of 8); result as float32 `out` (may be NULL) and / or out_np planes (out_np = 0: none);
 * gelu != 0 applies the exact (erf) GELU before the residual is added.  bias, resid may be NULL. */
int comet_linear_tc(const void* x_planes, long long x_plane_stride, long long x_ld, const void* w_planes,
                    long long w_plane_stride, long long w_ld, int np, const float* bias, const float* resid,
                    long long resid_ld, float* out, long long out_ld, void* out_planes, long long out_plane_stride,
                    long long outp_ld, int out_np, int gelu, long long M, int N, int K, comet_stream_t stream);
/* nn.LayerNorm over the last dimension (gamma / beta NULL: elementwise_affine=False), written as float32 `out` (may be
 * NULL) and / or np planes (np = 0: none). */
int comet_layernorm_planes_f32(const float* x, long long x_ld, const float* gamma, const float* beta, float eps, float* out,
                               long long out_ld, void* planes, long long plane_stride, long long p_ld, int np,
                               long long rows, int D, comet_stream_t stream);
/* softmax(q k^T / sqrt(dh)) v of nn.MultiheadAttention per (batch item, head); element (b, i, h, d) of q / k / v at
 * ptr + b*sb + i*si + h*dh + d (float32; any batch / position strides: no rearrange copies); output as np planes with
 * element (b, i, h*dh + d) at b*o_sb + i*o_si + h*dh + d. */
int comet_attention_planes_f32(const float* q, long long q_sb, long long q_si, const float* k, long long k_sb, long long k_si,
                               const float* v, long long v_sb, long long v_si, void* out_planes, long long o_plane_stride,
                               long long o_sb, long long o_si, int np, int B, int H, int Lq, int Lk, int dh,
                               comet_stream_t stream);
/* Many attention problems of different lengths in one call (all sequences of a space block): item i's query position j
 * (and output row) is row q_off[i] + j*q_step of q (row pitch q_ld) / of the output planes (row pitch o_ld), its key /
 * value position j is row k_off[i] + j*k_step of k and v (row pitch k_ld), with q_len[i] / k_len[i] positions.  The four
 * int32 arrays live in DEVICE memory; every length must lie in [min_lq, max_lq] / [min_lk, max_lk].  Item i gets exactly
 * the arithmetic comet_attention_planes_f32 uses for (Lq, Lk, dh, np) with B = group problems of that shape (same kernel
 * family, same key split).  min_lq / min_lk must be at least 1. */
int comet_attention_varlen_planes_f32(const float* q, long long q_ld, long long q_step, const float* k, long long k_ld,
                                      long long k_step, const float* v, void* out_planes, long long o_plane_stride,
                                      long long o_ld, int np, int items, int H, int dh, const int* q_off, const int* q_len,
                                      const int* k_off, const int* k_len, int min_lq, int max_lq, int min_lk, int max_lk,
                                      int group, comet_stream_t stream);
/* The same with lengths that may be 0 (the item is skipped and its output rows are not written) and a per-item problem
 * count: item i's kernel family is the one comet_attention_planes_f32 uses with B = groups[i] (int32, device memory, each
 * in [min_group, max_group]); groups NULL: B = max_group (= min_group) for every item.  The time attention of sequences
 * with different frame counts is one such call: item = track, length = its sequence's frame count, group = that
 * sequence's track count plus the virtual tracks. */
int comet_attention_varlen_grouped_planes_f32(const float* q, long long q_ld, long long q_step, const float* k, long long k_ld,
                                              long long k_step, const float* v, void* out_planes, long long o_plane_stride,
                                              long long o_ld, int np, int items, int H, int dh, const int* q_off,
                                              const int* q_len, const int* k_off, const int* k_len, int min_lq, int max_lq,
                                              int min_lk, int max_lk, const int* groups, int min_group, int max_group,
                                              comet_stream_t stream);
/* planes of a + b (contiguous float32 vectors of n elements): `tokens + init_tokens` before the flow head (blocks.py:344). */
int comet_add_planes_f32(const float* a, const float* b, void* planes, long long plane_stride, int np, long long n,
                         comet_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* COMET_B200_H */
