// Correlation on the 5th-generation tensor cores (tcgen05 + TMEM + TMA) with the multi-level window lookup and the
// track-token assembly as the epilogue -- the dense coarse-tracker shape of COMET (C=128, 64x64 maps, L<=5, r<=4,
// zero padding: CorrBlock.corr + CorrBlock.sample, comet/models/track_modules/blocks.py:376-429, and the token
// assembly of base_track_predictor.py:165-224).  The correlation volume lives only in TMEM.
//
// Arithmetic.  float32 parity (1e-4) on bf16 tensor cores: every operand is split x = hi + lo (two bf16) and the
// product is accumulated in float32 as hi*hi + hi*lo + lo*hi (the dropped lo*lo term is ~2^-18 relative), i.e. one
// K=384 bf16 GEMM.  In COMET_PREC_BF16_AUTOCAST mode only hi*hi is issued and the accumulator is rounded to bf16
// exactly where torch.autocast rounds the reference's volume.
//
// Data layout (HBM).  comet_tc_prepare_f32 (once per tracker call) pools the pyramid in float32 and packs, per frame,
// P=5504 positions  [L0 4096 | L1 1024 | L2 256 | L3 64 | L4 16 | 48 zeros] = 86 tiles of 64 positions.  Each tile is
// stored as the exact 32 KB shared-memory image of its two [128 channels x 64 positions] bf16 operand tiles (hi, lo)
// in the MN-major SWIZZLE_128B UMMA layout: split[bs][tile][hi|lo][channel][64].  One pipeline stage is ONE contiguous
// 32 KB bulk async copy (cp.async.bulk -> mbarrier); a tiled TMA load of the same bytes costs ~10 clk per 128-byte row.
//
// Work decomposition.  Launch 1 (tc_pre_kernel): per frame, the queries are counting-sorted by floor(y), so the 128
// queries of an MMA tile -- and the 32 of an epilogue warp -- share a narrow band of map rows; the per-(tile, level)
// band is reduced and turned into job records (nsplit level-0 row chunks with one row of overlap + npyr jobs for
// levels 1..L-1), and per sorted slot {query, x, y} is written for the epilogue's prefetch; the remaining CTAs of that
// launch write the correlation-independent token channels (flow sin/cos, flow, track_feats, pad) -- and, in reduce
// mode, the position embedding of the window channels -- as a persistent loop over token rows whose next row is
// already on its way into shared memory (cp.async), one bulk store per row.  Launch 2 (corr_tc_kernel): persistent
// CTAs (one per SM) walk the job list; only the tiles of a band are loaded and multiplied (~45 % of the dense GEMM at
// 512 random queries per frame), and an epilogue warp skips the tiles none of its queries touches.
//
// CTA = 10 warps:  warp 0 bulk-copy producer (3-stage ring) | warp 1 TMEM alloc + single-thread tcgen05.mma issue
// (A operand = targets in TMEM, `.ts` form; D 128x64 fp32 in TMEM, 4-stage accumulator ring) | warps 2-5 epilogue:
// tcgen05.ld the accumulator row of "their" query (TMEM lane == sorted query slot), park it in a private shared-memory
// row (the window columns are indexed dynamically), horizontal lerp at the query's x window, vertical lerp with the
// previous row, write the staged window; job metadata (record, sorted slot) arrives by cp.async two jobs ahead |
// warps 6-9 stager: stage the next job's targets into TMEM (hi/lo split, tcgen05.st) and send the staged windows out:
// MODE_REDUCE (token rows): one lane per query adds its 16-byte aligned staged row to the token row with a bulk
// reduction (cp.reduce.async.bulk add.f32 -- the TMA unit and the L2 do the work); MODE_STORE (lookup layout,
// unaligned token rows): coalesced stores + position embedding, entry by entry.
// The two launches are chained with programmatic dependent launch: the tensor kernel's prologue (barrier init, TMEM
// allocation) overlaps the drain of tc_pre_kernel and it waits (griddepcontrol.wait) before touching the plan.
//
// Measured and rejected (profiles/r02_coarse_tc_stalls.md, profiles/r02b_coarse_tc_analysis.md; B200, batch of 4
// sequences, ms per iteration): EIGHT epilogue warps, two per TMEM lane quarter: 0.170 vs 0.118 -- with 14 warps one
// scheduler hosts 4 of them, which caps the kernel at 128 registers per thread and spills the accumulator row; an L2
// prefetch ahead of the operand ring: no change (the level-0 phases pull 6.9 TB/s of first-touch tiles -- HBM, not
// latency); staging the targets of job i+2 early: no change; the token rows as a third grid beside the plan: slower;
// the row initialisation inside the stager warps behind global-memory flags: 0.15-0.39 vs 0.108.
#include "comet_common.cuh"

#include <cuda.h>
#include <cstdlib>

namespace comet {
namespace tc {

constexpr int MAP = 64;        // level-0 map is MAP x MAP
constexpr int KC = 128;        // channels == GEMM K per pass
constexpr int TILE_M = 128;    // queries per CTA tile == TMEM lanes
constexpr int TILE_N = 64;     // positions per accumulator tile
constexpr int NSTAGE = 3;      // B-tile ring
constexpr int NACC = 4;        // accumulator ring (4 x 64 TMEM columns)
constexpr int P_TOTAL = 5504;  // packed positions per (frame, channel)
constexpr int NTILES = 86;     // P_TOTAL / TILE_N tiles of 64 positions per frame
constexpr int MAX_WR = 9;      // 2*4+1
#ifndef COMET_TC_PDL
#define COMET_TC_PDL 1
#endif
#ifndef COMET_TC_EVICT_FIRST
#define COMET_TC_EVICT_FIRST 0  // operand tiles loaded with an L2 evict-first policy (experiment)
#endif
#ifndef COMET_TC_L2PF
#define COMET_TC_L2PF 0        // tiles the producer's L2 prefetch runs ahead of the operand ring (0: off)
#endif
constexpr int THREADS = 320;   // 10 warps: TMA | MMA | 4 epilogue | 4 stager

// tensor-memory map (all 512 columns of the SM are allocated, so the base address is 0)
constexpr uint32_t TM_ACC = 0;      // accumulator ring: NACC x 64 columns
constexpr uint32_t TM_A = 256;      // target tile: 2 buffers x [hi 64 cols | lo 64 cols] (two bf16 per column)

constexpr int B_TILE_BYTES = TILE_N * KC * 2;   // 16 KB per hi / lo
constexpr int STAGE_BYTES = 2 * B_TILE_BYTES;   // hi + lo
constexpr int DUMP_STRIDE = 68;                 // floats per private accumulator row (64 + 4: conflict-free STS.128)
constexpr int DUMP_BYTES = TILE_M * DUMP_STRIDE * 4;
// staged windows: per (buffer, epilogue warp) a [83 entries][33] float array -- entry-major, one column per query lane
// (+1 padding), so that both the epilogue (lanes write the same entry of different queries) and the stager (lanes read
// different entries of one query) are bank-conflict free.  Entries 81 / 82 carry the window rows the job owns.
constexpr int WIN_LD = 33;
constexpr int WIN_JLO = 81, WIN_JHI = 82;
constexpr int WIN_WARP = 2740;                  // 83 * 33 = 2739 floats, rounded to a 16-byte multiple
constexpr int WIN_BYTES = 4 * WIN_WARP * 4;
constexpr int NWIN = 2;                         // window buffers (epilogue -> stager hand-off)
constexpr int ROWOFF_BYTES = 2 * TILE_M * 8;      // per query: element offset of its pos_emb row and of its output row
constexpr int META_JOB = TILE_M + 8;                 // int4 per prefetched job: one slot per query + the record, one copy per warp
constexpr int META_BYTES = 2 * META_JOB * 16;        // epilogue prefetch, two jobs deep
constexpr int SMEM_BYTES = NSTAGE * STAGE_BYTES + DUMP_BYTES + NWIN * WIN_BYTES + ROWOFF_BYTES + META_BYTES + 512;

__host__ __device__ inline int level_offset(int l) { return l == 0 ? 0 : l == 1 ? 4096 : l == 2 ? 5120 : l == 3 ? 5376 : 5440; }
__host__ __device__ inline int num_tiles(int L) { return L == 1 ? 64 : L == 2 ? 80 : L == 3 ? 84 : L == 4 ? 85 : 86; }

struct TileInfo {
  int level, y_first, rows, W, H;
};
__device__ __forceinline__ TileInfo tile_info(int t) {
  TileInfo ti;
  if (t < 64) { ti.level = 0; ti.y_first = t; ti.rows = 1; ti.W = 64; }
  else if (t < 80) { ti.level = 1; ti.y_first = (t - 64) * 2; ti.rows = 2; ti.W = 32; }
  else if (t < 84) { ti.level = 2; ti.y_first = (t - 80) * 4; ti.rows = 4; ti.W = 16; }
  else if (t < 85) { ti.level = 3; ti.y_first = 0; ti.rows = 8; ti.W = 8; }
  else { ti.level = 4; ti.y_first = 0; ti.rows = 4; ti.W = 4; }
  ti.H = ti.W;
  return ti;
}

// One unit of work of the persistent kernel: up to four runs of consecutive tiles (a run never spans two pyramid
// levels) of one (frame, 128 sorted queries) pair.  Written by tc_plan_kernel, read by every warp role.
struct __align__(16) JobRec {
  int bs;
  int mnf;            // query tile (bits 0-15) | number of runs (16-23) | flags (24-31)
  uint32_t t0p, t1p;  // run i: first tile / one past the last tile in byte i (global tile numbering of tile_info, < 256)
  int own_lo, own_hi; // level-0 jobs: the window rows ("tops") whose output this job writes
  int src;            // frame of the packed pyramid the job's tiles are read from (== bs without a frame table)
  int pad1;
  __host__ __device__ int mt() const { return mnf & 0xffff; }
  __host__ __device__ int nseg() const { return (mnf >> 16) & 0xff; }
  __host__ __device__ int flags() const { return (mnf >> 24) & 0xff; }
  __host__ __device__ int t0(int i) const { return (t0p >> (8 * i)) & 0xff; }
  __host__ __device__ int t1(int i) const { return (t1p >> (8 * i)) & 0xff; }
};
constexpr int JF_FIRST0 = 1;  // first level-0 job of its (frame, query tile)
constexpr int JF_LAST0 = 2;   // last level-0 job: also writes the non-correlation token channels
constexpr int BIG = 1 << 28;
constexpr int MAX_SPLIT = 4;  // level-0 row chunks per (frame, query tile)
constexpr int MAX_CHUNK = MAX_SPLIT + 2;
constexpr int PLAN_BINS = 96;      // sort key: floor(y) clamped to [-16, 79]
constexpr int PLAN_MAX_MT = 256;   // query tiles per frame the plan kernel tracks row ranges for (N <= 32768)

struct Params {
  const float* targets; long long t_sb, t_ss, t_sn;
  const float* coords;  long long c_sb, c_ss, c_sn;
  float* out;           long long o_sb, o_ss, o_sn;   // lookup layout (B,S,N,L*Wr*Wr) when !tokens
  const float* pos; int D_tok; int tokens;            // token layout (B,N,S,D_tok) when tokens
  int vec4;                                           // tokens: rows of out / pos are 16-byte aligned (float4 token_misc path)
  int red;                                            // tokens: windows are ADDED to the rows (MODE_REDUCE); tc_pre_kernel writes pos_emb there
  const int* ntr;                                     // tokens: (B,) query count of each sequence (queries n >= ntr[b] are padding), or null
  const int* nfr;                                     // tokens: (B,) frame count of each sequence (frames s >= nfr[b] are padding), or null
  const int* fidx;                                    // tokens: (B,S) packed-pyramid frame of each (item, position), or null (identity)
  int BS_src;                                         // frames of the packed pyramid (fidx entries are clamped to [0, BS_src))
  float* vol[5]; int volume_mode;                      // volume mode: per-level (BS,N,H_l,W_l)
  int B, S, N, L, r, npass, bf16;
  int BS, mtiles, npad, nsplit, npyr, nchunk, njobs;
  const uint8_t* split; // packed pyramid (tile-major, pre-swizzled bf16 hi/lo), written by tc_prepare_kernel
  const int* perm;      // [BS][npad]: query index of sorted slot (or -1), written by tc_plan_kernel
  const int4* slots;    // [BS][npad]: {query index or -1, bits of x, bits of y, 0} of the sorted slot (epilogue prefetch)
  const JobRec* jobs;   // [njobs]
  float inv_sqrt_c;
  int* status;  // device int: set non-zero by the watchdog
#ifdef COMET_TC_TRACE
  int debug;    // COMET_TC_DEBUG bit mask (attribution experiments)
  long long* stamps;  // optional clock64 trace of CTA 0: [3 roles][64][2] + stager [8 jobs][16][2]
#endif
};

// Attribution switches and clock64 stamps exist only in -DCOMET_TC_TRACE builds (scripts/gpu_tc_attr.sh); the
// production kernel has no debug branch in its loops.
#ifdef COMET_TC_TRACE
#define TC_DBG(p, bit) (((p).debug & (bit)) != 0)
#else
#define TC_DBG(p, bit) false
#endif

// ------------------------------------------------------------------ PTX helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One elected lane of a fully converged warp (elect.sync): unlike `lane == 0`, ptxas knows exactly one thread is
// active in the guarded region and emits the uniform-datapath UTCHMMA / UTMALDG without a per-instruction
// ELECT + BRA.U.ANY loop (measured: ~70 clk per tcgen05.mma issue with `lane == 0`).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {   // non-blocking probe
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P1;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P1;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (visible failure) instead of hanging the GPU box.  The bound is WALL TIME
// (10 s of %globaltimer, looked at every 4096 polls), not a poll count, so that compute-sanitizer, a debugger,
// MPS or time-slicing cannot make it fire on a healthy kernel.
__device__ __forceinline__ uint64_t global_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int* status, int code) {
  uint32_t spins = 0;
  uint64_t t0 = 0;
  while (!mbar_try(bar, parity)) {
    if ((++spins & 4095u) == 0) {
      const uint64_t now = global_ns();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 10000000000ull) {
        if (status) atomicExch(status, code);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int x, int y) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"((uint64_t)map), "r"(smem_u32(bar)), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// bulk copy with an L2 eviction-priority hint (createpolicy): the operand stream of the tensor kernel is read once or
// twice within microseconds and should not push the token rows -- which the bulk reductions read-modify-write -- out of L2
__device__ __forceinline__ void bulk_load_hint(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy) : "memory");
}
__device__ __forceinline__ void tcgen05_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[tmem] * B[smem], kind::f16 (bf16 in, f32 accumulate), one CTA.  A: row m in TMEM lane m, two
// bf16 K-elements per 32-bit column (16 K-elements = 8 columns per instruction).
__device__ __forceinline__ void umma_bf16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
        "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 64-bit shared-memory matrix descriptor (SWIZZLE_128B, version 1).  lbo/sbo in bytes.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}
// kind::f16 instruction descriptor: D f32, A/B bf16, A K-major, B MN-major, M=128, N=64.
constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (0u << 15) | (1u << 16) |
                           ((uint32_t)(TILE_N >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_resid(float x) { return x - __bfloat162float(__float2bfloat16_rn(x)); }

// Loads whose ISSUE POINT matters (software prefetch across an mbarrier wait): `__ldg` is an invariant load that the
// compiler may sink to its first use -- i.e. behind the wait it was meant to overlap; a volatile asm statement keeps its
// order relative to the other volatile asm statements (the mbarrier waits and arrives).
__device__ __forceinline__ float ldg_pin(const float* ptr) {
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(ptr));
  return v;
}
__device__ __forceinline__ int ldg_pin(const int* ptr) {
  int v;
  asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(ptr));
  return v;
}
__device__ __forceinline__ int4 ldg_pin(const int4* ptr) {
  int4 v;
  asm volatile("ld.global.nc.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr));
  return v;
}

// Shared-memory accesses by 32-bit address.  The "memory" clobber orders them against the plain C++ accesses of the
// same buffers; volatile keeps the loads of one row together, ahead of the arithmetic that consumes them.
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_f32_if(uint32_t addr, float v, uint32_t pred) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %2, 0;\n\t"
      "@p st.shared.f32 [%0], %1;\n\t}"
      ::"r"(addr), "f"(v), "r"(pred) : "memory");
}

__device__ __forceinline__ JobRec load_job(const Params& p, int job) {
  JobRec r;
  if (job < p.njobs) {
    const int4* s = reinterpret_cast<const int4*>(p.jobs + job);
    int4* d = reinterpret_cast<int4*>(&r);
    d[0] = ldg_pin(s);
    d[1] = ldg_pin(s + 1);
  } else {
    r.bs = 0; r.mnf = 0; r.t0p = 0; r.t1p = 0; r.own_lo = 0; r.own_hi = 0; r.src = 0; r.pad1 = 0;
  }
  return r;
}

__device__ __forceinline__ void stamp(const Params& p, int role, int idx, int which) {
#ifdef COMET_TC_TRACE
  if (p.stamps && blockIdx.x == 0 && idx < (role == 3 ? 128 : 64)) p.stamps[(role * 64 + idx) * 2 + which] = clock64();
#endif
}

// Window geometry of one query along y at pyramid level l -- the ONE definition shared by the plan kernel (row
// ranges, sort) and the epilogue (lookup), so both always agree on which map rows a query touches.
__device__ __forceinline__ void level_y(float cy, int level, int r, int& y0, float& fy) {
  const float inv = 1.f / (float)(1 << level);
  const float py = fminf(fmaxf(cy * inv, -1.0e6f), 1.0e6f);
  const float fl = floorf(py);
  fy = py - fl;
  y0 = (int)fl - r;
}

// ------------------------------------------------------------------ plan: sort queries by y, row ranges, job list
// One CTA per frame.  Queries are counting-sorted by floor(y) so that the 128 queries of a tile (and the 32 of an
// epilogue warp) share a narrow band of map rows; per (tile, level) the band [first, last needed row] is reduced
// and turned into job records: `nsplit` level-0 jobs (row chunks with one row of overlap, so every window entry
// finds both of its rows inside one chunk) and `npyr` jobs for levels 1..L-1.  `full` (volume mode): identity
// order, every tile of every level.
__device__ __forceinline__ void plan_frame(const Params& p, int* __restrict__ perm, JobRec* __restrict__ jobs, int full,
                                           int bs) {
  __shared__ int hist[PLAN_BINS];
  __shared__ int rng[PLAN_MAX_MT][10];
  const int b = bs / p.S, s = bs - b * p.S;
  const int Wr = 2 * p.r + 1;
  int* myperm = perm + (long long)bs * p.npad;
  int4* myslots = const_cast<int4*>(p.slots) + (long long)bs * p.npad;
  const bool track = p.mtiles <= PLAN_MAX_MT;  // else: sorted, but every job covers the full maps
  int Nb = p.ntr ? min(max(__ldg(p.ntr + b), 0), p.N) : p.N;   // padded queries are not sorted: no tile, no job work
  if (p.nfr && s >= __ldg(p.nfr + b)) Nb = 0;                   // padded frame: every tile of it is an empty job
  // the frame table is read here, once per frame, into the job records: the producer warp already loads those, so the
  // operand ring gains no dependent global load
  const int src = p.fidx ? min(max(__ldg(p.fidx + bs), 0), p.BS_src - 1) : bs;

  for (int i = threadIdx.x; i < PLAN_BINS; i += blockDim.x) hist[i] = 0;
  if (track)
    for (int i = threadIdx.x; i < p.mtiles * 10; i += blockDim.x) (&rng[0][0])[i] = (i & 1) ? -BIG : BIG;
  __syncthreads();

  if (full) {
    for (int i = threadIdx.x; i < p.npad; i += blockDim.x) {
      myperm[i] = i < p.N ? i : -1;
      float cx = 0.f, cy = 0.f;
      if (i < p.N && p.coords) {
        const float* cp = p.coords + b * p.c_sb + s * p.c_ss + (long long)i * p.c_sn;
        cx = __ldg(cp); cy = __ldg(cp + 1);
      }
      myslots[i] = make_int4(i < p.N ? i : -1, __float_as_int(cx), __float_as_int(cy), 0);
    }
  } else {
    const float* cbase = p.coords + b * p.c_sb + s * p.c_ss + 1;
    for (int n = threadIdx.x; n < Nb; n += blockDim.x) {
      const float cy = __ldg(cbase + (long long)n * p.c_sn);
      const int key = min(max((int)floorf(fminf(fmaxf(cy, -1.0e6f), 1.0e6f)), -16), PLAN_BINS - 17) + 16;
      atomicAdd(&hist[key], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      int run = 0;
      for (int i = 0; i < PLAN_BINS; ++i) { const int c = hist[i]; hist[i] = run; run += c; }
    }
    __syncthreads();
    for (int n = threadIdx.x; n < Nb; n += blockDim.x) {
      const float cy = __ldg(cbase + (long long)n * p.c_sn);
      const int key = min(max((int)floorf(fminf(fmaxf(cy, -1.0e6f), 1.0e6f)), -16), PLAN_BINS - 17) + 16;
      const int slot = atomicAdd(&hist[key], 1);
      myperm[slot] = n;
      myslots[slot] = make_int4(n, __float_as_int(__ldg(cbase - 1 + (long long)n * p.c_sn)), __float_as_int(cy), 0);
      if (track) {
        const int mt = slot >> 7;
        for (int l = 0; l < p.L; ++l) {
          int y0; float fy;
          level_y(cy, l, p.r, y0, fy);
          const int rl = max(y0, 0), rh = min(y0 + Wr, (MAP >> l) - 1);
          if (rl <= rh) { atomicMin(&rng[mt][2 * l], rl); atomicMax(&rng[mt][2 * l + 1], rh); }
        }
      }
    }
    for (int i = Nb + threadIdx.x; i < p.npad; i += blockDim.x) { myperm[i] = -1; myslots[i] = make_int4(-1, 0, 0, 0); }
  }
  __syncthreads();

  for (int idx = threadIdx.x; idx < p.mtiles * p.nchunk; idx += blockDim.x) {
    const int mt = idx / p.nchunk, c = idx - mt * p.nchunk;
    JobRec jr;
    jr.bs = bs; jr.t0p = 0; jr.t1p = 0;
    jr.own_lo = -BIG; jr.own_hi = BIG; jr.src = src; jr.pad1 = 0;
    int nseg = 0, flags = 0;
    auto rows_of = [&](int l, int& R0, int& R1) {
      if (full || !track) { R0 = 0; R1 = (MAP >> l) - 1; }
      else { R0 = rng[mt][2 * l]; R1 = rng[mt][2 * l + 1]; if (R0 > R1) { R0 = 0; R1 = 0; } }
    };
    if (c < p.nsplit) {
      int R0, R1;
      rows_of(0, R0, R1);
      const int nr = R1 - R0 + 1, rpc = (nr + p.nsplit - 1) / p.nsplit;
      const int a = R0 + c * rpc, bb = min(a + rpc, R1);
      const bool real = (c == 0) || (a < R1);
      nseg = 1;
      if (real) {
        const bool last = bb == R1;
        jr.t0p = a; jr.t1p = bb + 1;
        flags = (c == 0 ? JF_FIRST0 : 0) | (last ? JF_LAST0 : 0);
        jr.own_lo = (c == 0) ? -BIG : a;
        jr.own_hi = last ? BIG : bb - 1;
      } else {
        // band narrower than the split: a one-tile job that owns no window rows (keeps the job sequence static)
        jr.t0p = R1; jr.t1p = R1 + 1;
        jr.own_lo = BIG; jr.own_hi = -BIG;
      }
    } else {
      const int k = c - p.nsplit;
      const int l_lo = (p.npyr == 2 && k == 1) ? 2 : 1;
      const int l_hi = (p.npyr == 2 && k == 0) ? 2 : p.L;   // exclusive
      for (int l = l_lo; l < l_hi; ++l) {
        int R0, R1;
        rows_of(l, R0, R1);
        const int sh = l == 1 ? 1 : l == 2 ? 2 : l == 3 ? 3 : 2;  // log2(map rows per tile): 2, 4, 8, 4
        const int base = l == 1 ? 64 : l == 2 ? 80 : l == 3 ? 84 : 85;
        jr.t0p |= (uint32_t)(base + (R0 >> sh)) << (8 * nseg);
        jr.t1p |= (uint32_t)(base + (R1 >> sh) + 1) << (8 * nseg);
        ++nseg;
      }
    }
    jr.mnf = mt | (nseg << 16) | (flags << 24);
    jobs[((long long)bs * p.mtiles + mt) * p.nchunk + c] = jr;
  }
}

// The token channels that do not depend on the correlation (base_track_predictor.py:170-196, :221):
//   [ sin/cos(flow * div) (C) | flow (2) | .. fcorrs: written by corr_tc_kernel .. | track_feats (C) | zero pad ] + pos_emb
// One warp per (b, n, s) token row, rows in output order (coalesced 128-byte stores).
__device__ __forceinline__ void token_misc_rows(const Params& p, long long warp_id, long long nwarps, int lane) {
  const int WW = (2 * p.r + 1) * (2 * p.r + 1);
  const int Ce = KC >> 1;
  const float step = 1000.0f / (float)Ce;
  const int feat_off = KC + 2 + p.L * WW;
  const int ntail = p.D_tok - feat_off;  // track_feats + pad
  const long long rows = (long long)p.B * p.N * p.S;
  for (long long row = warp_id; row < rows; row += nwarps) {
    const int s = (int)(row % p.S);
    const long long bn = row / p.S;
    const int n = (int)(bn % p.N), b = (int)(bn / p.N);
    if ((p.ntr && n >= __ldg(p.ntr + b)) || (p.nfr && s >= __ldg(p.nfr + b))) {   // padded query / frame: zero row
      for (int c = lane; c < p.D_tok; c += 32) p.out[row * p.D_tok + c] = 0.f;
      continue;
    }
    const float* cp = p.coords + b * p.c_sb + s * p.c_ss + (long long)n * p.c_sn;
    const float* c0 = p.coords + b * p.c_sb + (long long)n * p.c_sn;  // frame 0
    const float flx = __ldg(cp) - __ldg(c0), fly = __ldg(cp + 1) - __ldg(c0 + 1);
    const float* pq = p.pos + bn * p.D_tok;
    const float* tq = p.targets + b * p.t_sb + s * p.t_ss + (long long)n * p.t_sn;
    float* o = p.out + row * p.D_tok;
    float pe[4], tf[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { pe[k] = __ldg(pq + lane + 32 * k); tf[k] = __ldg(tq + lane + 32 * k); }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int e = lane + 32 * k;
      const int axis = e / Ce, w = e - axis * Ce;
      const float arg = __fmul_rn(axis ? fly : flx, (float)(w & ~1) * step);
      float sv, cv;
      sincosf(arg, &sv, &cv);      // one range reduction, no divergence between the sin and the cos lanes
      o[e] = ((w & 1) ? cv : sv) + pe[k];
    }
    if (lane < 2) o[KC + lane] = (lane ? fly : flx) + __ldg(pq + KC + lane);
#pragma unroll
    for (int k = 0; k < 4; ++k) o[feat_off + lane + 32 * k] = tf[k] + __ldg(pq + feat_off + lane + 32 * k);
    for (int c = KC + lane; c < ntail; c += 32) o[feat_off + c] = __ldg(pq + feat_off + c);   // zero pad + pos_emb
  }
}

// The same rows with 16-byte accesses (token rows and position-embedding rows 16-byte aligned, D_tok % 4 == 0), as a
// persistent loop: a warp walks its rows with the NEXT row's position-embedding row and track features already on
// their way into shared memory (reduce mode: two bulk copies per row onto the buffer's mbarrier; store mode: cp.async
// of the groups it needs), so the loop runs at issue rate instead of one memory round trip per row.  A lane owns whole float4 groups of the row; one sincosf serves a (sin, cos) channel pair; the
// row is written with STG.128.  Groups that lie entirely inside the window channels are skipped unless p.red (then
// they receive the position embedding the bulk reductions add to).
// `buf`: this warp's 3 x (D_tok + KC) floats of dynamic shared memory.
__device__ __forceinline__ void token_misc_rows_v4(const Params& p, long long warp_id, long long nwarps, int lane,
                                                   float* buf) {
  const int WW = (2 * p.r + 1) * (2 * p.r + 1);
  const int Ce = KC >> 1;
  const float step = 1000.0f / (float)Ce;
  const int feat_off = KC + 2 + p.L * WW;
  const int nv = p.D_tok >> 2;
  const int f_lo = (KC + 2 + 3) >> 2, f_hi = feat_off >> 2;   // float4 groups [f_lo, f_hi) hold window channels only
  const int rows = p.B * p.N * p.S;               // < 2^31 (checked by the host): 32-bit row arithmetic
  const int bstride = p.D_tok + KC;
  constexpr int T = 6;                             // float4 groups per lane: D_tok <= 768 (checked by the host)
  auto needed = [&](int k) { return k < nv && (p.red || k < f_lo || k >= f_hi); };
  // position-embedding groups this lane needs + its float4 of the track features -> shared memory buffer `which`;
  // the flow of the row (coordinates of this frame minus frame 0) into registers
  // reduce mode copies whole rows: two bulk copies per row (position-embedding row, track features) onto the buffer's
  // mbarrier, issued by one lane -- no per-lane copy instructions and nothing through the L1TEX pipe
  uint64_t* mb = reinterpret_cast<uint64_t*>(buf + 3 * bstride);   // [3], one per buffer
  if (p.red) {
    if (lane == 0) {
      for (int i = 0; i < 3; ++i) mbar_init(&mb[i], 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
  }
  uint32_t mphase = 0;                                              // bit i: parity buffer i's next completion has
  auto issue = [&](int row, int which, float& flx, float& fly) {
    flx = 0.f; fly = 0.f;
    if (row < rows) {
      const int bn = row / p.S, s_ = row - bn * p.S;
      const int b_ = bn / p.N, n_ = bn - b_ * p.N;
      const uint32_t dst = smem_u32(buf + which * bstride);
      const float4* pq = reinterpret_cast<const float4*>(p.pos + (long long)bn * p.D_tok);
      const float4* tq = reinterpret_cast<const float4*>(p.targets + b_ * p.t_sb + s_ * p.t_ss + (long long)n_ * p.t_sn);
      if (p.red) {
        if (lane == 0) {
          mbar_expect_tx(&mb[which], (uint32_t)(p.D_tok + KC) * 4u);
          bulk_load(buf + which * bstride, pq, (uint32_t)p.D_tok * 4u, &mb[which]);
          bulk_load(buf + which * bstride + p.D_tok, tq, (uint32_t)KC * 4u, &mb[which]);
        }
      } else {
#pragma unroll
        for (int t = 0; t < T; ++t) {
          const int k = lane + 32 * t;
          if (needed(k))
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (uint32_t)k * 16u), "l"(pq + k) : "memory");
        }
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                     ::"r"(dst + (uint32_t)(nv + lane) * 16u), "l"(tq + lane) : "memory");
      }
      const float* c0 = p.coords + b_ * p.c_sb + (long long)n_ * p.c_sn;  // frame 0
      const float* cp = c0 + s_ * p.c_ss;
      flx = __ldg(cp) - __ldg(c0);
      fly = __ldg(cp + 1) - __ldg(c0 + 1);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  const int w0 = (int)warp_id, nw = (int)nwarps;
  float flx, fly;
  issue(w0, 0, flx, fly);
  int which = 0;   // three buffers in rotation: being filled | being worked on | being read by its bulk store
  for (int row = w0; row < rows; row += nw, which = which == 2 ? 0 : which + 1) {
    float flx1, fly1;
    issue(row + nw, which == 2 ? 0 : which + 1, flx1, fly1);
    if (p.red) {
      mbar_wait(&mb[which], (mphase >> which) & 1u, p.status, 11);
      mphase ^= 1u << which;
    } else {
      asm volatile("cp.async.wait_group 1;" ::: "memory");
      __syncwarp();                                 // the feature row was copied by all 32 lanes
    }
    float* o = p.out + (long long)row * p.D_tok;
    if (p.ntr || p.nfr) {
      const int bn = row / p.S, b_ = bn / p.N;
      if ((p.ntr && bn - b_ * p.N >= __ldg(p.ntr + b_)) || (p.nfr && row - bn * p.S >= __ldg(p.nfr + b_))) {
        // padded query / frame: zero row (its loads above were in bounds and unused)
        for (int k = lane; k < nv; k += 32) reinterpret_cast<float4*>(o)[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.red) {                                // keep the bulk-group count of the store pipeline in step
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        }
        __syncwarp();
        flx = flx1; fly = fly1;
        continue;
      }
    }
    if (p.red) {
      // Whole row leaves as ONE bulk store: the position-embedding row sits in shared memory; add the few channels that
      // carry something else in place (sin/cos: one group per lane; flow; track features) and hand the row to the TMA.
      float* rowb = buf + which * bstride;
      const float* feat_row = rowb + p.D_tok;
      {
        float4 pk = reinterpret_cast<float4*>(rowb)[lane];
        const int c = 4 * lane, axis = c / Ce, w = c - axis * Ce;
        const float f = axis ? fly : flx;
        float v0, v1, v2, v3;
        sincosf(__fmul_rn(f, (float)w * step), &v0, &v1);
        sincosf(__fmul_rn(f, (float)(w + 2) * step), &v2, &v3);
        pk.x += v0; pk.y += v1; pk.z += v2; pk.w += v3;
        reinterpret_cast<float4*>(rowb)[lane] = pk;
      }
      if (lane < 2) rowb[KC + lane] += lane ? fly : flx;
      {
        const float4 f4 = reinterpret_cast<const float4*>(feat_row)[lane];
        float* d = rowb + feat_off + 4 * lane;
        d[0] += f4.x; d[1] += f4.y; d[2] += f4.z; d[3] += f4.w;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0)
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                     ::"l"(o), "r"(smem_u32(rowb)), "r"(p.D_tok * 4) : "memory");
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      // the buffer the NEXT iteration's issue refills is the one whose store was committed one iteration ago: wait
      // until that store has read its source (this iteration's store may still be pending)
      asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      flx = flx1; fly = fly1;
      continue;
    }
    const float4* pe = reinterpret_cast<const float4*>(buf + which * bstride);
    const float* feat_row = buf + which * bstride + p.D_tok;
#pragma unroll
    for (int t = 0; t < T; ++t) {
      const int k = lane + 32 * t;
      if (!needed(k)) continue;
      const int c = 4 * k;
      const float4 pk = pe[k];
      float v[4];
      if (t == 0 && KC >= 128) {                    // groups 0..31 are the 128 sin/cos channels
        const int axis = c / Ce, w = c - axis * Ce;   // w is a multiple of 4: channels (sin, cos) of w and of w + 2
        const float f = axis ? fly : flx;
        sincosf(__fmul_rn(f, (float)w * step), &v[0], &v[1]);
        sincosf(__fmul_rn(f, (float)(w + 2) * step), &v[2], &v[3]);
      } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int cj = c + j;
          v[j] = (cj >= KC && cj < KC + 2) ? (cj == KC ? flx : fly)
               : (cj >= feat_off && cj < feat_off + KC) ? feat_row[cj - feat_off] : 0.f;
        }
      }
      const float4 r = make_float4(v[0] + pk.x, v[1] + pk.y, v[2] + pk.z, v[3] + pk.w);
      if (p.red || c + 3 < KC + 2 || c >= feat_off) {
        *reinterpret_cast<float4*>(o + c) = r;
      } else {   // a group shared with window channels the tensor kernel stores itself
        const float rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (c + j < KC + 2 || c + j >= feat_off) o[c + j] = rr[j];
      }
    }
    __syncwarp();                                   // buffer `which` is refilled by the next iteration's issue
    flx = flx1; fly = fly1;
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// Launch 1 of 2 per call: CTAs [0, BS) plan one frame each, the rest write the correlation-independent token channels.
__global__ void __launch_bounds__(256) tc_pre_kernel(const Params p, int* __restrict__ perm, JobRec* __restrict__ jobs,
                                                      int full) {
  if ((int)blockIdx.x < p.BS) {
    plan_frame(p, perm, jobs, full, blockIdx.x);
  } else {
    const long long nw = (long long)(gridDim.x - p.BS) * 8;
    extern __shared__ __align__(16) float pre_smem[];   // vec4: 8 warps x 3 x (D_tok + KC) floats
    if (p.vec4) token_misc_rows_v4(p, (long long)(blockIdx.x - p.BS) * 8 + (threadIdx.x >> 5), nw, threadIdx.x & 31,
                                   pre_smem + (threadIdx.x >> 5) * (3 * (p.D_tok + KC) + 8));
    else token_misc_rows(p, (long long)(blockIdx.x - p.BS) * 8 + (threadIdx.x >> 5), nw, threadIdx.x & 31);
  }
  // programmatic dependent launch: once every CTA of this grid got here the tensor kernel may be scheduled, so its
  // prologue overlaps this grid's drain; it waits for this grid's completion (griddepcontrol.wait) before it reads
  // perm / jobs / the token rows.  (Triggering at the START of this kernel instead lets the dependent's 218 KB CTAs occupy
  // every SM that falls idle and starve the remaining CTAs of this grid.)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// The correlation-independent token channels as their own launch, AFTER the tensor kernel in stream order and chained to
// it with programmatic dependent launch: the tensor kernel triggers its dependents as soon as its CTAs are resident, so
// these (128 threads, no shared memory, <= 64 registers: they fit beside the 218 KB tensor CTAs) run in the issue slots
// and HBM bandwidth the tensor kernel leaves idle (29 % / 30 % busy).  They write channels the tensor kernel never
// touches; the wait at the END makes this grid's completion imply the tensor kernel's.  COMET_OPT_TC_OVERLAP_MISC, off by
// default: measured 0.155 vs 0.112 ms per iteration -- beside a tensor CTA (53.7 K registers) only 4 such warps fit on an
// SM, and the 56 MB these rows move then take longer than the tensor kernel itself.
__global__ void __launch_bounds__(128, 1) tc_misc_kernel(const Params p) {
  const long long nw = (long long)gridDim.x * 4;
  token_misc_rows(p, (long long)blockIdx.x * 4 + (threadIdx.x >> 5), nw, threadIdx.x & 31);
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ------------------------------------------------------------------ the kernel
// MODE_STORE: windows (+ position embedding) written with plain stores by the stager warps -- the lookup layout
// (B,S,N,L*Wr*Wr), and token rows whose base / pitch are not 16-byte aligned.  MODE_VOLUME: the raw volume.
// MODE_REDUCE (token rows): tc_pre_kernel has already written the position embedding into the window channels; the
// epilogue stages each query's window as one 16-byte aligned row [a | Wr*Wr entries | zeros] and ONE lane per query
// adds it to the token row with a bulk reduction (cp.reduce.async.bulk .add.f32, executed by the TMA unit and the L2):
// the ~1400 instructions per window unit that the stores cost a stager warp (scalar LDS + FADD + predicated STG per
// entry, the stager's critical path in the pyramid jobs) become ~20.  Entries a job does not own are zero in the staged
// row, so the level-0 row chunks of one query simply add up.
constexpr int MODE_STORE = 0, MODE_VOLUME = 1, MODE_REDUCE = 2;

template <int R, bool BF16, int MODE>
__global__ void __launch_bounds__(THREADS, 1)
corr_tc_kernel(const Params p) {
  constexpr bool VOLUME = MODE == MODE_VOLUME;
  constexpr bool RED = MODE == MODE_REDUCE;
  // dynamic shared memory is the only shared allocation of this kernel, so it starts 1024-byte aligned (SWIZZLE_128B
  // tiles need that); no integer round trip on the pointer, so that accesses stay LDS/STS rather than generic LD/ST
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sB = smem;                                                   // NSTAGE x [hi 16 KB][lo 16 KB]
  float* dump = reinterpret_cast<float*>(sB + NSTAGE * STAGE_BYTES);   // private accumulator rows
  float* win = dump + TILE_M * DUMP_STRIDE;                            // staged window rows
  long long* rowoff = reinterpret_cast<long long*>(win + NWIN * 4 * WIN_WARP);  // [2][TILE_M]
  int4* meta = reinterpret_cast<int4*>(rowoff + 2 * TILE_M);           // [2][TILE_M slots | 4 warps x 2 int4 job record]
  uint64_t* bars = reinterpret_cast<uint64_t*>(meta + META_BYTES / 16);
  uint64_t* full = bars;                  // [NSTAGE]  TMA -> MMA
  uint64_t* empty = full + NSTAGE;        // [NSTAGE]  MMA -> TMA
  uint64_t* acc_full = empty + NSTAGE;    // [NACC]    MMA -> epilogue
  uint64_t* acc_empty = acc_full + NACC;  // [NACC]    epilogue -> MMA
  uint64_t* a_full = acc_empty + NACC;    // [2]       stager -> MMA (target tile in TMEM)
  uint64_t* a_empty = a_full + 2;         // [2]       MMA -> stager
  uint64_t* win_full = a_empty + 2;       // [NWIN*4]  epilogue warp -> stager warp of the same lane quarter
  uint64_t* win_empty = win_full + NWIN * 4;  // [NWIN*4]  stager warp -> epilogue warp
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(win_empty + NWIN * 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < NSTAGE; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < NACC; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 4); }
    for (int i = 0; i < 2; ++i) { mbar_init(&a_full[i], 128); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < NWIN * 4; ++i) { mbar_init(&win_full[i], 1); mbar_init(&win_empty[i], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  // The whole tensor memory of the SM is ours (one CTA per SM), so the allocation starts at lane 0 / column 0 and
  // every TMEM address below is a compile-time constant (keeps the MMA issue loop on the uniform datapath).
  if (*tmem_slot != 0 || (smem_u32(smem) & 1023u) != 0) {
    if (threadIdx.x == 0 && p.status) atomicExch(p.status, 9);
    __trap();
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // tc_misc_kernel may run beside this grid
  asm volatile("griddepcontrol.wait;" ::: "memory");   // plan (+ token rows) of tc_pre_kernel are complete and visible

  if (warp == 0) {
    // ===================== TMA producer =====================
    // Two cursors over the CTA's tile sequence: the load cursor feeds the 3-stage ring; the prefetch cursor runs
    // COMET_TC_L2PF tiles ahead of it and only asks the L2 for the tile (cp.async.bulk.prefetch.L2), so that the ring's
    // bulk copies hit in L2 -- the ring alone (96 KB in flight) covers ~2 tiles of MMA time, less than a DRAM round trip.
    if (elect_one()) {
      struct Cursor {
        JobRec cur, nxt;
        int job, sg, t, te;
      };
      const int G = gridDim.x;
      auto cursor_init = [&](Cursor& c) {
        c.job = blockIdx.x;
        c.cur = load_job(p, c.job);
        c.nxt = load_job(p, c.job + G);
        c.sg = 0; c.t = c.cur.t0(0); c.te = c.cur.t1(0);
      };
      auto cursor_next = [&](Cursor& c) {   // precondition: c.job < p.njobs
        if (++c.t < c.te) return;
        if (++c.sg < c.cur.nseg()) { c.t = c.cur.t0(c.sg); c.te = c.cur.t1(c.sg); return; }
        c.job += G;
        c.cur = c.nxt;
        c.nxt = load_job(p, c.job + G);
        c.sg = 0; c.t = c.cur.t0(0); c.te = c.cur.t1(0);
      };
      const uint32_t nbytes = BF16 ? B_TILE_BYTES : STAGE_BYTES;   // autocast mode issues hi x hi only: fetch the hi half
      uint32_t stage = 0, phase = 0;
      int tcount = 0;
#if COMET_TC_EVICT_FIRST
      uint64_t l2_policy;
      asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(l2_policy));
#endif
      Cursor ld;
      cursor_init(ld);
#if COMET_TC_L2PF > 0
      Cursor pf = ld;
      auto prefetch = [&]() {
        if (pf.job < p.njobs) {
          asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;"
                       ::"l"(p.split + ((long long)pf.cur.src * NTILES + pf.t) * STAGE_BYTES), "r"(nbytes) : "memory");
          cursor_next(pf);
        }
      };
      if (pf.job < p.njobs) cursor_next(pf);   // the very first tile goes straight to shared memory
      for (int i = 0; i < COMET_TC_L2PF; ++i) prefetch();
#endif
      while (ld.job < p.njobs) {
        mbar_wait(&empty[stage], phase ^ 1, p.status, 1);
        stamp(p, 0, tcount++, 0);
        uint8_t* dst = sB + stage * STAGE_BYTES;
        if (TC_DBG(p, 64)) {
          mbar_arrive(&full[stage]);
        } else {
          mbar_expect_tx(&full[stage], nbytes);
#if COMET_TC_EVICT_FIRST
          bulk_load_hint(dst, p.split + ((long long)ld.cur.src * NTILES + ld.t) * STAGE_BYTES, nbytes, &full[stage], l2_policy);
#else
          bulk_load(dst, p.split + ((long long)ld.cur.src * NTILES + ld.t) * STAGE_BYTES, nbytes, &full[stage]);
#endif
        }
#if COMET_TC_L2PF > 0
        prefetch();
#endif
        cursor_next(ld);
        if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0, ji = 0;
    int tcount = 0;
    const int npass = TC_DBG(p, 8) ? 0 : p.npass;
    JobRec nxt = load_job(p, blockIdx.x);
    for (int job = blockIdx.x; job < p.njobs; job += gridDim.x, ++ji) {
      const JobRec jr = nxt;
      nxt = load_job(p, job + gridDim.x);
      const int nseg = jr.nseg();
      const uint32_t abuf = ji & 1;
      mbar_wait(&a_full[abuf], (ji >> 1) & 1, p.status, 2);
      const uint32_t a_hi = TM_A + abuf * 128, a_lo = a_hi + 64;
      for (int sg = 0; sg < nseg; ++sg) {
        for (int t = jr.t0(sg), te = jr.t1(sg); t < te; ++t) {
          const bool job_ends = (sg + 1 == nseg) && (t + 1 == te);
          mbar_wait(&acc_empty[acc], acc_phase ^ 1, p.status, 3);
          mbar_wait(&full[stage], phase, p.status, 4);
          tcgen05_fence_after();
          if (lane == 0) stamp(p, 1, tcount, 0);
          if (elect_one()) {
            const uint32_t b_hi = smem_u32(sB + stage * STAGE_BYTES);
            const uint32_t d = TM_ACC + acc * TILE_N;
            uint32_t accum = 0;
            for (int pass = 0; pass < npass; ++pass) {
              const uint32_t a0 = (pass == 2) ? a_lo : a_hi;
              // B: MN-major SW128, K row = 128 B, 8-row groups 1 KB apart; 16 K rows (2 KB) per step
              const uint64_t bd0 = make_desc(b_hi + ((pass == 1) ? B_TILE_BYTES : 0), B_TILE_BYTES, 1024);
#pragma unroll
              for (int k = 0; k < KC / 16; ++k) {
                umma_bf16_ts(d, a0 + k * 8, bd0 + (uint64_t)(k * (2048 >> 4)), IDESC, accum);
                accum = 1;
              }
            }
            tcgen05_commit(&empty[stage]);    // B stage free once these MMAs retire
            tcgen05_commit(&acc_full[acc]);   // accumulator ready
            if (job_ends) tcgen05_commit(&a_empty[abuf]);  // target tile buffer free
            stamp(p, 1, tcount, 1);
          }
          ++tcount;
          __syncwarp();
          if (++stage == NSTAGE) { stage = 0; phase ^= 1; }
          if (++acc == NACC) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else if (warp < 6) {
    // ===================== epilogue warps (2..5) =====================
    // One lane = one query (TMEM lane).  Per pyramid level the lane precomputes, once, everything that does not
    // depend on the map row: clamped column offsets of its x window, horizontal lerp weights with the zero-padding
    // mask and the 1/sqrt(C) scale folded in, and (level 0) which 16-byte groups of a row it must park.  Per needed
    // tile the work is then: tcgen05.ld -> park the row (predicated STS.128) -> per map row 10 LDS + 18 FMA
    // (horizontal) + 9 x (FMA + STS) (vertical lerp with the previous row, written to the staged window).
    const int wq = warp & 3;                    // TMEM lane quarter this warp may access
    const int q = 32 * wq + lane;               // TMEM lane == sorted query slot in the tile
    float* myrow = dump + q * DUMP_STRIDE;
    const uint32_t myrow_u32 = smem_u32(myrow);
    const uint32_t lane_addr = ((uint32_t)(32 * wq) << 16);
    constexpr int Wr = 2 * R + 1;
    constexpr int RW = ((Wr * Wr + 6) / 4) * 4;   // floats per staged row in RED mode (<= 3 leading + Wr*Wr, 16-byte multiple)
    constexpr int EI = RED ? Wr : Wr * WIN_LD;    // float stride between window columns i in the staged window
    constexpr int EJ = RED ? 1 : WIN_LD;          // ... between window rows j
    uint32_t acc = 0, acc_phase = 0, wu = 0;  // wu: window units handed to the stager so far
    int tcount = 0;
    float* wcol = win + lane;                 // this lane's column of the warp's staged window: entry e at wcol[e * WIN_LD]
    float* wwarp = win;

    // Job metadata is prefetched into shared memory with cp.async, two jobs deep: the sorted slot of this lane (query
    // index + coordinates, written by the plan kernel) and the job record.  Its address follows from the job NUMBER
    // (jobs are laid out [frame][query tile][chunk]), so nothing in the chain is a dependent load, and no register
    // carries prefetched data across a job (the register version spilled them -- and waited for the loads to do so).
    const int G = gridDim.x;
    auto prefetch_job = [&](int job, int buf) {
      if (job < p.njobs) {
        const int fq = job / p.nchunk;            // frame * mtiles + query tile
        const uint32_t dst = smem_u32(meta + buf * META_JOB);
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                     ::"r"(dst + (uint32_t)q * 16u), "l"(p.slots + (long long)fq * TILE_M + q) : "memory");
        if (lane < 2)   // every warp keeps its own copy of the record: no synchronisation between the epilogue warps
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                       ::"r"(dst + (uint32_t)(TILE_M + 2 * wq + lane) * 16u),
                         "l"(reinterpret_cast<const int4*>(p.jobs + job) + lane) : "memory");
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    prefetch_job(blockIdx.x, 0);
    prefetch_job(blockIdx.x + G, 1);
    uint32_t jseq = 0;
    for (int job = blockIdx.x; job < p.njobs; job += G, ++jseq) {
      const int mbuf = jseq & 1;
      asm volatile("cp.async.wait_group 1;" ::: "memory");   // this job's group has landed (the next one may be in flight)
      __syncwarp();                                           // the record was fetched by lanes 0 and 1
      const int4* mb = meta + mbuf * META_JOB;
      JobRec jr;
      {
        const int4 r0 = mb[TILE_M + 2 * wq], r1 = mb[TILE_M + 2 * wq + 1];
        jr.bs = r0.x; jr.mnf = r0.y; jr.t0p = (uint32_t)r0.z; jr.t1p = (uint32_t)r0.w;
        jr.own_lo = r1.x; jr.own_hi = r1.y; jr.src = r1.z; jr.pad1 = 0;
      }
      const int4 slot = mb[q];
      const int n = slot.x;
      const float cx = __int_as_float(slot.y), cy = __int_as_float(slot.z);
      const int bs = jr.bs;
      const bool valid = n >= 0;
      const int nseg = jr.nseg();

      for (int sg = 0; sg < nseg; ++sg) {
        const int tfirst = jr.t0(sg), tend = jr.t1(sg);
        const TileInfo t0i = tile_info(tfirst);
        const int level = t0i.level, Hl = t0i.H, Wl = t0i.W;
        const bool is0 = level == 0;
        // ---- window geometry of this query at this level; row band of the whole warp ----
        int x0, y0;
        float fx, fy;
        level_y(cy, level, R, y0, fy);
        {
          const float inv = 1.f / (float)(1 << level);
          const float px = fminf(fmaxf(cx * inv, -1.0e6f), 1.0e6f);
          const float flx = floorf(px);
          fx = px - flx;
          x0 = (int)flx - R;
        }
        // x window: clamped column offsets; lerp weights with the zero-padding mask (and, in fp32 mode, the scale)
        int xo[Wr + 1];
        uint32_t xo4[Wr + 1];
        float wa[Wr], wb[Wr];
        uint32_t xmask = 0, dmask = 0;
#pragma unroll
        for (int i = 0; i <= Wr; ++i) {
          const int xi = x0 + i;
          if (xi >= 0 && xi < Wl) xmask |= 1u << i;
          xo[i] = min(max(xi, 0), Wl - 1);
          xo4[i] = (uint32_t)xo[i] * 4u;
        }
        // map rows this query touches; a window that misses the map (in x or in y) touches none -- such a lane never
        // reads its parked row (a clamped offset could otherwise hit stale shared memory)
        int rl = max(y0, 0), rh = min(y0 + Wr, Hl - 1);
        if (!valid || rl > rh || xmask == 0) { rl = BIG; rh = -BIG; }
        const int wlo = __reduce_min_sync(0xffffffffu, rl), whi = __reduce_max_sync(0xffffffffu, rh);
#pragma unroll
        for (int i = 0; i < Wr; ++i) {
          const float sc = BF16 ? 1.f : p.inv_sqrt_c;
          wa[i] = ((xmask >> i) & 1) ? (1.f - fx) * sc : 0.f;
          wb[i] = ((xmask >> (i + 1)) & 1) ? fx * sc : 0.f;
        }
        if (is0) {
#pragma unroll
          for (int k = 0; k < 16; ++k)
            if (4 * k + 3 >= x0 && 4 * k <= x0 + Wr) dmask |= 1u << k;
        }
        // window rows ("tops") written while streaming: [ta, tb_]; top = H-1 is finished at the end of the level
        const int ta = is0 ? jr.own_lo : -BIG;
        const int tb_ = is0 ? min(jr.own_hi, Hl - 2) : Hl - 2;
        float hprev[Wr];
#pragma unroll
        for (int i = 0; i < Wr; ++i) hprev[i] = 0.f;
        const float gy = 1.f - fy;
        if (!VOLUME && !TC_DBG(p, 1)) {
          // claim a window buffer and clear it cooperatively (entries whose rows are off the map stay 0)
          const uint32_t wbuf = wu % NWIN;
          if (warp == 2 && lane == 0) stamp(p, 5, 2 * wu, 0);
          mbar_wait(&win_empty[wbuf * 4 + wq], ((wu / NWIN) & 1) ^ 1, p.status, 7);
          if (warp == 2 && lane == 0) stamp(p, 5, 2 * wu, 1);
          wwarp = win + (wbuf * 4 + wq) * WIN_WARP;
          // RED: this lane's row, shifted so that entry 0 lands on the 16-byte phase of its token channel
          wcol = RED ? wwarp + lane * RW + ((KC + 2 + level * Wr * Wr) & 3) : wwarp + lane;
#pragma unroll 1
          for (int k = lane * 4; k < WIN_WARP; k += 128) *reinterpret_cast<float4*>(wwarp + k) = make_float4(0.f, 0.f, 0.f, 0.f);
          __syncwarp();
        }

        for (int t = tfirst; t < tend; ++t) {
          const TileInfo ti = tile_info(t);
          const int ylast = ti.y_first + ti.rows - 1;
          // does any query of this warp touch the rows of this tile?  (warp-uniform)
          const bool wneed = VOLUME || ((ti.y_first <= whi && ylast >= wlo) && !TC_DBG(p, 32));
          mbar_wait(&acc_full[acc], acc_phase, p.status, 5);
          if (warp == 2 && lane == 0) stamp(p, 2, tcount, 0);
          float v[64];
          if (wneed) {
            tcgen05_fence_after();
            tmem_ld32(lane_addr + TM_ACC + acc * TILE_N, v);
            tmem_ld32(lane_addr + TM_ACC + acc * TILE_N + 32, v + 32);
            tmem_ld_wait();
            tcgen05_fence_before();
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[acc]);
          if (warp == 2 && lane == 0) stamp(p, 2, tcount, 1);
          ++tcount;
          if (++acc == NACC) { acc = 0; acc_phase ^= 1; }

          if (VOLUME) {
            if (valid) {
              const int cols = ti.level == 4 ? 16 : 64;
              const int HW = ti.W * ti.W;
              float* dst = p.vol[ti.level] + ((long long)bs * p.N + n) * HW + (t * TILE_N - level_offset(ti.level));
#pragma unroll
              for (int i = 0; i < 64; i += 4) {
                if (i < cols) {
                  float4 o;
                  if (BF16) {
                    o = make_float4(round_bf16(round_bf16(v[i]) * p.inv_sqrt_c), round_bf16(round_bf16(v[i + 1]) * p.inv_sqrt_c),
                                    round_bf16(round_bf16(v[i + 2]) * p.inv_sqrt_c), round_bf16(round_bf16(v[i + 3]) * p.inv_sqrt_c));
                  } else {
                    o = make_float4(v[i] * p.inv_sqrt_c, v[i + 1] * p.inv_sqrt_c, v[i + 2] * p.inv_sqrt_c, v[i + 3] * p.inv_sqrt_c);
                  }
                  *reinterpret_cast<float4*>(dst + i) = o;
                }
              }
            }
            continue;
          }
          if (TC_DBG(p, 1) || !wneed) continue;

          // park the accumulator row in this lane's private smem row (the window columns are indexed dynamically):
          // only queries that touch this tile, and at level 0 only the 16-byte groups under their x window
          if (ti.y_first <= rh && ylast >= rl) {
            if (is0) {
#pragma unroll
              for (int k = 0; k < 16; ++k)
                if ((dmask >> k) & 1)
                  *reinterpret_cast<float4*>(myrow + 4 * k) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
            } else {
#pragma unroll
              for (int k = 0; k < 16; ++k)
                *reinterpret_cast<float4*>(myrow + 4 * k) = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
            }
          }
          // ---- stream the map rows of this tile ----
          // Branch-free per row: all Wr+1 loads of a row are issued before the first use (explicit shared-memory
          // addresses, so no generic-pointer conversion inside the loop), rows come in pairs where the tile has them
          // (two loads batches in flight), and the window entries are written with predicated stores.  A row's values
          // are only ever written for lanes whose window contains it (see the predicate), so rows a lane did not park
          // may be read (stale, never stored).
          const uint32_t wcol_u32 = smem_u32(wcol);
          auto load_row = [&](int rr, float (&vv)[Wr + 1]) {
            const uint32_t base = myrow_u32 + (uint32_t)(rr * Wl) * 4u;
#pragma unroll
            for (int i = 0; i <= Wr; ++i) vv[i] = lds_f32(base + xo4[i]);
          };
          auto finish_row = [&](int y, float (&vv)[Wr + 1]) {
            if (BF16) {
              // blocks.py:428 scales the volume after the matmul; under autocast both steps round to bf16
#pragma unroll
              for (int i = 0; i <= Wr; ++i) vv[i] = round_bf16(round_bf16(vv[i]) * p.inv_sqrt_c);
            }
            float h[Wr];
#pragma unroll
            for (int i = 0; i < Wr; ++i) h[i] = wa[i] * vv[i] + wb[i] * vv[i + 1];
            const int top = y - 1, j = top - y0;
            const uint32_t ok = (j >= 0 && j < Wr && top >= ta && top <= tb_ && rl <= rh) ? 1u : 0u;
            const uint32_t wd = wcol_u32 + (uint32_t)(min(max(j, 0), Wr - 1) * EJ) * 4u;
#pragma unroll
            for (int i = 0; i < Wr; ++i) sts_f32_if(wd + (uint32_t)(i * EI) * 4u, gy * hprev[i] + fy * h[i], ok);
#pragma unroll
            for (int i = 0; i < Wr; ++i) hprev[i] = h[i];
          };
          {
            int rr = 0;
#pragma unroll 1
            for (; rr + 1 < ti.rows; rr += 2) {
              float va[Wr + 1], vb[Wr + 1];
              load_row(rr, va);
              load_row(rr + 1, vb);
              finish_row(ti.y_first + rr, va);
              finish_row(ti.y_first + rr + 1, vb);
            }
            if (rr < ti.rows) {
              float va[Wr + 1];
              load_row(rr, va);
              finish_row(ti.y_first + rr, va);
            }
          }
        }

        if (VOLUME || TC_DBG(p, 1)) continue;
        // ---- end of the level inside this job: finish the window and hand it to the stager warp ----
        {
          const bool last = !is0 || (jr.flags() & JF_LAST0);
          if (last && valid) {
            const int jb = (Hl - 1) - y0;  // top = H-1: its bottom row is off the map (hprev is row H-1: jb in range
                                           // means this query touches row H-1, so its warp streamed up to it)
            if (jb >= 0 && jb < Wr && rl <= rh) {
              float* wdst = wcol + jb * EJ;
#pragma unroll
              for (int i = 0; i < Wr; ++i) wdst[i * EI] = (1.f - fy) * hprev[i];
            }
          }
          // window rows (index j) this job owns: tops in [lo_top, hi_top]
          const int lo_top = is0 ? jr.own_lo : -BIG;
          const int hi_top = is0 ? jr.own_hi : BIG;
          if (RED) {
            // the TMA unit (async proxy) reads these rows: make this lane's generic-proxy writes visible to it
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          } else {
            const int j_lo = valid ? max(0, lo_top - y0) : 1, j_hi = valid ? min(Wr - 1, hi_top - y0) : 0;
            wcol[WIN_JLO * WIN_LD] = __int_as_float(j_lo);
            wcol[WIN_JHI * WIN_LD] = __int_as_float(j_hi);
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(&win_full[(wu % NWIN) * 4 + wq]);  // release.cta: the STS above are visible
          if (warp == 2 && lane == 0) stamp(p, 5, 2 * wu + 1, 0);
          ++wu;
        }
      }
      __syncwarp();                         // every lane has read this job's metadata long ago: refill the buffer
      prefetch_job(job + 2 * G, mbuf);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
  } else {
    // ===================== stager warps (6..9): every global load/store except the TMA =====================
    // per job:  (1) stage the NEXT job's 128 target rows into the free TMEM A buffer (hi/lo split, tcgen05.st);
    //           (2) the last level-0 job of a (frame, query tile) writes the non-correlation part of the tokens;
    //           (3) for every window unit the epilogue warp of the same lane quarter hands over: add the position
    //               embedding and store the window rows this job owns, coalesced, with all loads of 16 queries in
    //               flight before the first store.
    const int wq = warp & 3;
    const int q = 32 * wq + lane;
    const uint32_t lane_addr = ((uint32_t)(32 * wq) << 16);
    constexpr int Wr = 2 * R + 1, WW = Wr * Wr;
    uint32_t wu = 0;

    // stage the 128 target rows of job number `jobno` (hi/lo split) into TMEM A buffer (ji & 1); `nq` = this lane's
    // query.  Frame and query tile follow from the job number (jobs are laid out [frame][query tile][chunk]).
    auto stage_targets = [&](int jobno, int nq, uint32_t ji) {
      const int bs_ = (jobno / p.nchunk) / p.mtiles;
      const int b = bs_ / p.S, s = bs_ - b * p.S;
      const uint32_t abuf = ji & 1;
      mbar_wait(&a_empty[abuf], ((ji >> 1) & 1) ^ 1, p.status, 6);
      tcgen05_fence_after();
      if (!TC_DBG(p, 256)) {
        const bool rv = nq >= 0;
        const float4* src = reinterpret_cast<const float4*>(p.targets + b * p.t_sb + s * p.t_ss +
                                                            (long long)(rv ? nq : 0) * p.t_sn);
        const uint32_t ta_hi = lane_addr + TM_A + abuf * 128, ta_lo = ta_hi + 64;
#pragma unroll 1
        for (int half = 0; half < 2; ++half) {  // 64 channels per step: 16 LDG.128 in flight
          float4 f[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) f[i] = rv ? __ldg(src + half * 16 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int blk = 0; blk < 2; ++blk) {
            uint32_t hi[16], lo[16];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 g = f[blk * 8 + i];
              hi[2 * i] = pack_bf16(g.x, g.y);
              hi[2 * i + 1] = pack_bf16(g.z, g.w);
              lo[2 * i] = pack_bf16(bf16_resid(g.x), bf16_resid(g.y));
              lo[2 * i + 1] = pack_bf16(bf16_resid(g.z), bf16_resid(g.w));
            }
            tmem_st16(ta_hi + half * 32 + blk * 16, hi);
            tmem_st16(ta_lo + half * 32 + blk * 16, lo);
          }
        }
        tmem_st_wait();
      }
      tcgen05_fence_before();
      mbar_arrive(&a_full[abuf]);
    };
    auto slot_query = [&](int jobno) {   // perm is [frame][query tile][128]: addressed by the job number alone
      return jobno < p.njobs ? ldg_pin(p.perm + (long long)(jobno / p.nchunk) * TILE_M + q) : -1;
    };

    // software pipeline: record and query index of job i+2 are in flight while job i is served (no dependent loads)
    const int G = gridDim.x;
    int myn = slot_query(blockIdx.x);
    int myn1 = slot_query(blockIdx.x + G);
    JobRec jr = load_job(p, blockIdx.x);
    JobRec jr1 = load_job(p, blockIdx.x + G);
    if ((int)blockIdx.x < p.njobs) stage_targets(blockIdx.x, myn, 0);
    uint32_t ji = 0;
    constexpr int RW = ((WW + 6) / 4) * 4;   // floats per staged row in RED mode
    const bool do_windows = !(VOLUME || TC_DBG(p, 1));
    for (int job = blockIdx.x; job < p.njobs; job += G, ++ji) {
      const JobRec jr2 = load_job(p, job + 2 * G);
      const int myn2 = slot_query(job + 2 * G);
      if (warp == 6 && lane == 0) stamp(p, 3, ji * 16 + 0, 0);
      if (job + G < p.njobs) stage_targets(job + G, myn1, ji + 1);
      if (warp == 6 && lane == 0) stamp(p, 3, ji * 16 + 0, 1);
      const int bs = jr.bs;
      const int b = bs / p.S, s = bs - b * p.S;
      const int nseg = jr.nseg();
#ifdef COMET_TC_TRACE
      if (warp == 6 && lane == 0 && p.stamps && blockIdx.x == 0 && ji < 8) {   // tiles of this job, for the trace reader
        int nt = 0;
        for (int sg = 0; sg < nseg; ++sg) nt += jr.t1(sg) - jr.t0(sg);
        p.stamps[(3 * 64 + ji * 16 + 15) * 2] = nt;
        p.stamps[(3 * 64 + ji * 16 + 15) * 2 + 1] = nseg;
      }
#endif
      if (RED) {
        // One lane = one query: add its staged row to its token row.  The row starts on the 16-byte boundary at or
        // below the level's first window channel (`a` leading zeros) and ends on one (trailing zeros), so neighbouring
        // channels receive + 0.0f.
        float* orow = p.out + (((long long)b * p.N + (myn >= 0 ? myn : 0)) * p.S + s) * p.D_tok;
        for (int sg = 0; do_windows && sg < nseg; ++sg, ++wu) {
          const int lvl = tile_info(jr.t0(sg)).level;
          const uint32_t wbuf = wu % NWIN;
          mbar_wait(&win_full[wbuf * 4 + wq], (wu / NWIN) & 1, p.status, 8);
          if (warp == 6 && lane == 0) stamp(p, 3, ji * 16 + 1 + 2 * sg, 0);
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          if (myn >= 0 && !TC_DBG(p, 2)) {
            const int ch = KC + 2 + lvl * WW;
            asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f32 [%0], [%1], %2;"
                         ::"l"(orow + (ch & ~3)), "r"(smem_u32(win + (wbuf * 4 + wq) * WIN_WARP + lane * RW)), "r"(RW * 4)
                         : "memory");
          }
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the staged rows have been read
          __syncwarp();
          if (lane == 0) mbar_arrive(&win_empty[wbuf * 4 + wq]);
          if (warp == 6 && lane == 0) stamp(p, 3, ji * 16 + 2 + 2 * sg, 1);
        }
        jr = jr1; jr1 = jr2;
        myn = myn1; myn1 = myn2;
        continue;
      }

      // element offsets of this lane's query rows (pos_emb row, output row), shared with the warp through smem:
      // the store loop below then needs one broadcast LDS.64 per row instead of shuffles + 64-bit index math.
      // Padding slots point at row 0 and own no window rows (j_lo > j_hi), so they are never stored.
      {
        const long long nq = myn >= 0 ? myn : 0;
        __syncwarp();
        rowoff[q] = ((long long)b * p.N + nq) * p.D_tok;
        rowoff[TILE_M + q] = p.tokens ? (((long long)b * p.N + nq) * p.S + s) * p.D_tok
                                      : b * p.o_sb + s * p.o_ss + nq * p.o_sn;
        __syncwarp();
      }
      const int nvalid = min(32, p.N - (jr.mt() * TILE_M + 32 * wq));   // sorted slots: valid first, padding last
      // window units of this job: one per tile run (= one pyramid level)
      for (int sg = 0; do_windows && sg < nseg; ++sg, ++wu) {
        const int lvl = tile_info(jr.t0(sg)).level;
        const uint32_t wbuf = wu % NWIN;
        mbar_wait(&win_full[wbuf * 4 + wq], (wu / NWIN) & 1, p.status, 8);
        if (warp == 6 && lane == 0) stamp(p, 3, ji * 16 + 1 + 2 * sg, 0);
        const float* wbase = win + (wbuf * 4 + wq) * WIN_WARP;   // [entry][WIN_LD] of this lane quarter
        const int lvl_off = (p.tokens ? KC + 2 : 0) + lvl * WW;
        const int jj0 = lane % Wr, jj1 = (lane + 32) % Wr, jj2 = (lane + 64) % Wr;
        const bool ok1 = lane + 32 < WW, ok2 = lane + 64 < WW;
        const bool ok0 = lane < WW;
        const float* pbase = p.pos + lvl_off + min(lane, WW - 1);
        const int d1 = min(lane + 32, WW - 1) - min(lane, WW - 1), d2 = min(lane + 64, WW - 1) - min(lane, WW - 1);
        float* obase = p.out + lvl_off + lane;
#pragma unroll 1
        for (int q16 = 0; q16 < 32; q16 += 16) {
          if (q16 >= nvalid || TC_DBG(p, 2)) break;
          // unconditional loads (clamped addresses) into their own registers: all 48 in flight before the first store
          float val[16][3];
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            if (p.tokens && !TC_DBG(p, 16)) {
              const float* pq = pbase + rowoff[32 * wq + q16 + u];
              val[u][0] = __ldg(pq);
              val[u][1] = __ldg(pq + d1);
              val[u][2] = __ldg(pq + d2);
            } else {
              val[u][0] = 0.f; val[u][1] = 0.f; val[u][2] = 0.f;
            }
          }
          const float* wsrc = wbase + q16;
#pragma unroll
          for (int u = 0; u < 16; ++u) {
            float* dst = obase + rowoff[TILE_M + 32 * wq + q16 + u];
            const int jl = __float_as_int(wsrc[WIN_JLO * WIN_LD + u]), jh = __float_as_int(wsrc[WIN_JHI * WIN_LD + u]);
            if (ok0 && jj0 >= jl && jj0 <= jh) dst[0] = wsrc[lane * WIN_LD + u] + val[u][0];
            if (ok1 && jj1 >= jl && jj1 <= jh) dst[32] = wsrc[(lane + 32) * WIN_LD + u] + val[u][1];
            if (ok2 && jj2 >= jl && jj2 <= jh) dst[64] = wsrc[(lane + 64) * WIN_LD + u] + val[u][2];
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&win_empty[wbuf * 4 + wq]);
        if (warp == 6 && lane == 0) stamp(p, 3, ji * 16 + 2 + 2 * sg, 1);
      }
      jr = jr1; jr1 = jr2;
      myn = myn1; myn1 = myn2;
    }
    if (RED) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");   // every reduction of this thread has completed
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(0u), "r"(512));
  }
}

// ------------------------------------------------------------------ prepare: pooled pyramid + hi/lo split
// One CTA per (frame, channel) plane.  Pools in float32 exactly like the reference chain (pool of pool), writes the
// packed bf16 hi / lo rows and (optionally) the float32 pyramid levels used by the SIMT kernels.
__global__ void __launch_bounds__(256) tc_prepare_kernel(const float* __restrict__ fmaps, __nv_bfloat16* __restrict__ split,
                                                          float* __restrict__ pyr, int BS, int L, long long off1,
                                                          long long off2, long long off3, long long off4) {
  __shared__ float s[P_TOTAL];
  const long long plane = blockIdx.x;  // bs * KC + c
  const float4* src = reinterpret_cast<const float4*>(fmaps + plane * 4096);
  for (int i = threadIdx.x; i < 1024; i += 256) reinterpret_cast<float4*>(s)[i] = __ldg(src + i);
  __syncthreads();
  int in_off = 0, W = 64;
  for (int l = 1; l < 5; ++l) {
    const int Wo = W / 2, out_off = level_offset(l);
    for (int i = threadIdx.x; i < Wo * Wo; i += 256) {
      const int y = i / Wo, x = i - y * Wo;
      const float* a = s + in_off + (2 * y) * W + 2 * x;
      s[out_off + i] = ((a[0] + a[1]) + (a[W] + a[W + 1])) * 0.25f;
    }
    __syncthreads();
    in_off = out_off;
    W = Wo;
  }
  for (int i = 5456 + threadIdx.x; i < P_TOTAL; i += 256) s[i] = 0.f;
  __syncthreads();
  // tile-major, pre-swizzled layout: split[bs][tile 0..85][hi|lo][channel 0..127][64 positions] holds, per (frame,
  // tile), the exact 32 KB shared-memory image of the two [128 x 64] bf16 operand tiles in the MN-major SWIZZLE_128B
  // UMMA layout (16-byte chunk index XOR (channel & 7)).  One pipeline stage is then ONE contiguous 32 KB bulk copy:
  // a tiled TMA load of the same data spends ~10 clk per 128-byte row (2600 clk per stage, measured) and starves the MMA.
  const long long bs = plane / KC;
  const int c = (int)(plane - bs * KC);
  __nv_bfloat162* base = reinterpret_cast<__nv_bfloat162*>(split) + (bs * NTILES) * (long long)(2 * KC * TILE_N / 2);
  for (int i = threadIdx.x; i < P_TOTAL / 2; i += 256) {
    const float a = s[2 * i], b = s[2 * i + 1];
    const __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    const int t = i >> 5, n2 = i & 31;                       // tile, bf16-pair inside the tile row
    const int chunk = n2 >> 2, within = n2 & 3;              // 16-byte chunk of the 128-byte row
    const long long o = (long long)t * (2 * KC * TILE_N / 2) + c * (TILE_N / 2) + ((chunk ^ (c & 7)) << 2) + within;
    base[o] = h;
    base[o + KC * TILE_N / 2] = __floats2bfloat162_rn(a - __low2float(h), b - __high2float(h));
  }
  if (pyr) {
    const long long offs[5] = {0, off1, off2, off3, off4};
    int Wl = 32;
    for (int l = 1; l < L; ++l) {
      float* dst = pyr + offs[l] + plane * Wl * Wl;
      const float* sl = s + level_offset(l);
      for (int i = threadIdx.x; i < Wl * Wl; i += 256) dst[i] = sl[i];
      Wl /= 2;
    }
  }
}

// ------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// SM count of the CURRENT device if it is an sm_100 part (0 otherwise); cached per device ordinal -- a process may
// drive several GPUs, possibly of different kinds.
static int device_is_sm100() {
  static int cached[64];
  static bool known[64] = {false};
  int dev = 0, major = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return 0; }
  if (!known[dev]) {
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    cached[dev] = (major == 10 && sms > 0 && encode_fn() != nullptr) ? sms : 0;
    known[dev] = true;
  }
  return cached[dev];
}

#ifdef COMET_TC_TRACE
static long long* g_stamps = nullptr;
#endif

// One watchdog word per device.  Allocated by comet_tc_prepare_f32 (once per tracker call, never inside the
// per-iteration launches, so nothing is allocated under a CUDA-graph capture of the iteration loop).
static int* g_status[64] = {nullptr};
static int* status_word() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return nullptr; }
  return g_status[dev];
}
static int ensure_status_word(cudaStream_t stream) {
  int dev = 0;
  COMET_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || g_status[dev]) return COMET_OK;
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone)
    return COMET_OK;   // prepare itself is being captured: run without the watchdog word (status == nullptr)
  int* d = nullptr;
  COMET_CUDA(cudaMalloc(&d, sizeof(int)));
  COMET_CUDA(cudaMemsetAsync(d, 0, sizeof(int), stream));
  g_status[dev] = d;
  return COMET_OK;
}

// Work decomposition chosen on the host: `nsplit` level-0 row chunks + `npyr` pyramid jobs per (frame, query tile),
// enough jobs for ~4 per SM (COMET_TC_NSPLIT / COMET_TC_NPYR override, for experiments).
static void choose_split(int BS, int mtiles, int L, int sms, int& nsplit, int& npyr) {
  const long long base = (long long)BS * mtiles;
  npyr = L == 1 ? 0 : (L >= 3 && base * 3 < 4LL * sms) ? 2 : 1;
  long long want = (4LL * sms + base - 1) / (base > 0 ? base : 1) - npyr;
  nsplit = (int)(want < 1 ? 1 : want > MAX_SPLIT ? MAX_SPLIT : want);
#ifdef COMET_TC_TRACE
  static int env_split = -1, env_pyr = -1;
  if (env_split < 0) { const char* e = getenv("COMET_TC_NSPLIT"); env_split = e ? atoi(e) : 0; }
  if (env_pyr < 0) { const char* e = getenv("COMET_TC_NPYR"); env_pyr = e ? atoi(e) : 0; }
  if (env_split >= 1 && env_split <= MAX_SPLIT) nsplit = env_split;
  if (env_pyr >= 1 && env_pyr <= 2 && L > 1) npyr = (env_pyr == 2 && L < 3) ? 1 : env_pyr;
#endif
}

static long long workspace_bytes(int BS, int N) {
  const long long mtiles = (N + TILE_M - 1) / TILE_M;
  return (long long)BS * mtiles * TILE_M * (4 + 16) + (long long)BS * mtiles * MAX_CHUNK * (long long)sizeof(JobRec) + 64;
}

static int launch(Params& p, const void* split, void* workspace, cudaStream_t stream) {
  const int sms = device_is_sm100();
  if (!sms) return fail(COMET_ERR_UNSUPPORTED, "tensor path needs an sm_100 device and cuTensorMapEncodeTiled");
  COMET_REQUIRE(workspace && ((uintptr_t)workspace % 16) == 0, "workspace must be a 16-byte aligned device buffer");
  p.BS = p.B * p.S;
  p.mtiles = (p.N + TILE_M - 1) / TILE_M;
  p.npad = p.mtiles * TILE_M;
  choose_split(p.BS, p.mtiles, p.L, sms, p.nsplit, p.npyr);
  p.nchunk = p.nsplit + p.npyr;
  const long long njobs = (long long)p.BS * p.nchunk * p.mtiles;
  if (njobs == 0) return COMET_OK;
  if (njobs > 0x7fffffffLL) return fail(COMET_ERR_UNSUPPORTED, "too many jobs");
  p.njobs = (int)njobs;
  p.inv_sqrt_c = 1.0f / sqrtf((float)KC);
  p.status = status_word();
#ifdef COMET_TC_TRACE
  {
    static int dbg = -1;
    if (dbg < 0) { const char* e = getenv("COMET_TC_DEBUG"); dbg = e ? atoi(e) : 0; }
    p.debug = dbg;
  }
  p.stamps = g_stamps;
#endif
  // workspace: [jobs: BS*mtiles*MAX_CHUNK records][perm: BS*npad ints][slots: BS*npad int4]
  JobRec* jobs = reinterpret_cast<JobRec*>(workspace);
  int* perm = reinterpret_cast<int*>(jobs + (long long)p.BS * p.mtiles * MAX_CHUNK);
  p.jobs = jobs;
  p.perm = perm;
  p.slots = reinterpret_cast<const int4*>(perm + (long long)p.BS * p.npad);
  p.split = reinterpret_cast<const uint8_t*>(split);

  const int full = (p.volume_mode || TC_DBG(p, 512)) ? 1 : 0;   // 512: unsorted, every tile (A/B experiments)
  // token rows with a 16-byte aligned base and pitch take the bulk-reduction output path
  p.vec4 = (p.tokens && ((uintptr_t)p.out % 16) == 0 && ((uintptr_t)p.pos % 16) == 0 && (p.D_tok % 4) == 0 &&
            p.D_tok <= 768 && (long long)p.B * p.N * p.S < 0x7fffffffLL) ? 1 : 0;
  p.red = (p.vec4 && !p.volume_mode && option(COMET_OPT_TC_REDUCE_STORE) && !option(COMET_OPT_TC_OVERLAP_MISC)) ? 1 : 0;
  // launch 1: plan (one CTA per frame) + the correlation-independent token channels (8 token rows per CTA, capped)
  long long misc = 0;
  const bool overlap_misc = p.tokens && COMET_TC_PDL && option(COMET_OPT_TC_OVERLAP_MISC);
  size_t pre_smem = 0;
  if (p.tokens && !overlap_misc) {
    misc = ((long long)p.B * p.N * p.S + 7) / 8;
    if (p.vec4) {
      // persistent rows loop: 2 CTAs per SM (8 warps x 3 row buffers each)
      pre_smem = (size_t)8 * (3 * (p.D_tok + KC) + 8) * sizeof(float);
      if (misc > 2LL * sms) misc = 2LL * sms;
    }
    if (misc > 64LL * sms) misc = 64LL * sms;
    if (pre_smem > 48 * 1024)
      COMET_CUDA(cudaFuncSetAttribute(tc_pre_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pre_smem));
  }
  tc_pre_kernel<<<(unsigned)(p.BS + misc), 256, pre_smem, stream>>>(p, perm, jobs, full);
  int rc = launch_status("tc_pre_kernel");
  if (rc != COMET_OK) return rc;
  const int grid = (int)(njobs < sms ? njobs : sms);
#define COMET_TC_LAUNCH(RR, BF, VOL)                                                                              \
  do {                                                                                                            \
    COMET_CUDA(cudaFuncSetAttribute(corr_tc_kernel<RR, BF, VOL>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                    SMEM_BYTES));                                                                 \
    cudaLaunchConfig_t cfg__{};                                                                                   \
    cfg__.gridDim = dim3(grid); cfg__.blockDim = dim3(THREADS); cfg__.dynamicSmemBytes = SMEM_BYTES;              \
    cfg__.stream = stream;                                                                                        \
    cudaLaunchAttribute at__[1];                                                                                  \
    at__[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                                              \
    at__[0].val.programmaticStreamSerializationAllowed = COMET_TC_PDL;                                            \
    cfg__.attrs = at__; cfg__.numAttrs = 1;                                                                       \
    COMET_CUDA(cudaLaunchKernelEx(&cfg__, corr_tc_kernel<RR, BF, VOL>, p));                                      \
  } while (0)
#define COMET_TC_LAUNCH_R(RR)                                                                                     \
  do {                                                                                                            \
    if (p.red) {                                                                                                  \
      if (p.bf16) COMET_TC_LAUNCH(RR, true, MODE_REDUCE); else COMET_TC_LAUNCH(RR, false, MODE_REDUCE);           \
    } else {                                                                                                      \
      if (p.bf16) COMET_TC_LAUNCH(RR, true, MODE_STORE); else COMET_TC_LAUNCH(RR, false, MODE_STORE);             \
    }                                                                                                             \
  } while (0)
  if (p.volume_mode) {
    if (p.bf16) COMET_TC_LAUNCH(0, true, MODE_VOLUME); else COMET_TC_LAUNCH(0, false, MODE_VOLUME);
  } else {
    switch (p.r) {
      case 0: COMET_TC_LAUNCH_R(0); break;
      case 1: COMET_TC_LAUNCH_R(1); break;
      case 2: COMET_TC_LAUNCH_R(2); break;
      case 3: COMET_TC_LAUNCH_R(3); break;
      default: COMET_TC_LAUNCH_R(4); break;
    }
  }
#undef COMET_TC_LAUNCH_R
#undef COMET_TC_LAUNCH
  rc = launch_status("corr_tc_kernel");
  if (rc != COMET_OK || !overlap_misc) return rc;
  {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(2 * sms)); cfg.blockDim = dim3(128); cfg.dynamicSmemBytes = 0; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    COMET_CUDA(cudaLaunchKernelEx(&cfg, tc_misc_kernel, p));
  }
  return launch_status("tc_misc_kernel");
}

static int check_shape(int C, int H, int W, int L, int r, int pad_mode) {
  COMET_REQUIRE(C == KC && H == MAP && W == MAP, "tensor path is specialised to C=128, 64x64 maps (got C=%d, %dx%d)", C, H, W);
  COMET_REQUIRE(L >= 1 && L <= 5, "tensor path supports 1..5 levels (got %d)", L);
  COMET_REQUIRE(r >= 0 && r <= 4, "tensor path supports radius <= 4 (got %d)", r);
  COMET_REQUIRE(pad_mode == COMET_PAD_ZEROS, "tensor path implements zero padding only");
  return COMET_OK;
}

}  // namespace tc
}  // namespace comet

using namespace comet;

extern "C" int comet_has_tensor_path(void) { return option(COMET_OPT_TENSOR_PATH) && tc::device_is_sm100() > 0; }

extern "C" int comet_tc_supported(int C, int H, int W, int L, int r, int pad_mode) {
  return C == tc::KC && H == tc::MAP && W == tc::MAP && L >= 1 && L <= 5 && r >= 0 && r <= 4 &&
         pad_mode == COMET_PAD_ZEROS;
}

extern "C" long long comet_tc_split_elems(int BS) { return 2LL * BS * tc::KC * tc::P_TOTAL; }

extern "C" long long comet_tc_workspace_bytes(int BS, int N) {
  if (BS < 0 || N < 0) return -1;
  return tc::workspace_bytes(BS, N);
}

extern "C" int comet_tc_prepare_f32(const float* fmaps, void* split, float* pyr, int BS, int C, int H, int W, int L,
                                    comet_stream_t stream) {
  int rc = tc::check_shape(C, H, W, L, 0, COMET_PAD_ZEROS);
  if (rc != COMET_OK) return rc;
  if (BS == 0) return COMET_OK;
  COMET_REQUIRE(fmaps && split, "null pointer");
  rc = tc::ensure_status_word((cudaStream_t)stream);
  if (rc != COMET_OK) return rc;
  Levels lv = make_levels(BS, C, H, W, 5);
  tc::tc_prepare_kernel<<<BS * tc::KC, 256, 0, (cudaStream_t)stream>>>(
      fmaps, reinterpret_cast<__nv_bfloat16*>(split), pyr, BS, L, lv.off[1], lv.off[2], lv.off[3], lv.off[4]);
  return launch_status("tc_prepare_kernel");
}

static int tc_common(tc::Params& p, const float* targets, long long t_sb, long long t_ss, long long t_sn,
                     const float* coords, long long c_sb, long long c_ss, long long c_sn, int B, int S, int N, int C,
                     int H, int W, int L, int r, int pad_mode, int prec_mode) {
  int rc = tc::check_shape(C, H, W, L, r, pad_mode);
  if (rc != COMET_OK) return rc;
  COMET_REQUIRE(B >= 0 && S >= 0 && N >= 0, "negative batch dimension");
  COMET_REQUIRE(prec_mode == COMET_PREC_F32 || prec_mode == COMET_PREC_BF16_AUTOCAST, "bad prec_mode %d", prec_mode);
  COMET_REQUIRE((t_sn % 4) == 0 && (t_ss % 4) == 0 && (t_sb % 4) == 0 && ((uintptr_t)targets % 16) == 0,
                "targets must be 16-byte aligned rows for the tensor path");
  p.targets = targets; p.t_sb = t_sb; p.t_ss = t_ss; p.t_sn = t_sn;
  p.coords = coords; p.c_sb = c_sb; p.c_ss = c_ss; p.c_sn = c_sn;
  p.B = B; p.S = S; p.N = N; p.L = L; p.r = r;
  p.bf16 = prec_mode == COMET_PREC_BF16_AUTOCAST;
  p.npass = p.bf16 ? 1 : 3;
  return COMET_OK;
}

extern "C" int comet_tc_corr_lookup_f32(const void* split, const float* targets, long long t_sb, long long t_ss,
                                        long long t_sn, const float* coords, long long c_sb, long long c_ss,
                                        long long c_sn, float* out, long long o_sb, long long o_ss, long long o_sn,
                                        int B, int S, int N, int C, int H, int W, int L, int r, int pad_mode,
                                        int prec_mode, void* workspace, comet_stream_t stream) {
  tc::Params p{};
  int rc = tc_common(p, targets, t_sb, t_ss, t_sn, coords, c_sb, c_ss, c_sn, B, S, N, C, H, W, L, r, pad_mode, prec_mode);
  if (rc != COMET_OK) return rc;
  if ((long long)B * S * N == 0) return COMET_OK;
  COMET_REQUIRE(split && targets && coords && out, "null pointer");
  p.out = out; p.o_sb = o_sb; p.o_ss = o_ss; p.o_sn = o_sn;
  return tc::launch(p, split, workspace, (cudaStream_t)stream);
}

static int tc_track_tokens(const void* split, const float* track_feats, long long t_sb, long long t_ss, long long t_sn,
                           const float* coords, long long c_sb, long long c_ss, long long c_sn, const float* pos_emb,
                           float* tokens, const int* num_tracks, const int* num_frames, const int* frame_index, int BS_src,
                           int B, int S, int N, int C, int H, int W, int L, int r,
                           int pad_mode, int prec_mode, int D_tok, void* workspace, comet_stream_t stream) {
  tc::Params p{};
  int rc = tc_common(p, track_feats, t_sb, t_ss, t_sn, coords, c_sb, c_ss, c_sn, B, S, N, C, H, W, L, r, pad_mode,
                     prec_mode);
  if (rc != COMET_OK) return rc;
  const int need = 2 * C + 2 + L * (2 * r + 1) * (2 * r + 1);
  COMET_REQUIRE(D_tok >= need, "D_tok=%d smaller than the %d token channels", D_tok, need);
  COMET_REQUIRE(!frame_index || BS_src >= 1, "BS_src must be positive with a frame table (got %d)", BS_src);
  if ((long long)B * S * N == 0) return COMET_OK;
  COMET_REQUIRE(split && track_feats && coords && pos_emb && tokens, "null pointer");
  p.out = tokens; p.pos = pos_emb; p.D_tok = D_tok; p.tokens = 1; p.ntr = num_tracks; p.nfr = num_frames;
  p.fidx = frame_index; p.BS_src = BS_src;
  return tc::launch(p, split, workspace, (cudaStream_t)stream);
}

extern "C" int comet_tc_track_tokens_f32(const void* split, const float* track_feats, long long t_sb, long long t_ss,
                                         long long t_sn, const float* coords, long long c_sb, long long c_ss,
                                         long long c_sn, const float* pos_emb, float* tokens, int B, int S, int N,
                                         int C, int H, int W, int L, int r, int pad_mode, int prec_mode, int D_tok,
                                         void* workspace, comet_stream_t stream) {
  return tc_track_tokens(split, track_feats, t_sb, t_ss, t_sn, coords, c_sb, c_ss, c_sn, pos_emb, tokens, nullptr, nullptr,
                         nullptr, B * S, B, S, N, C, H, W, L, r, pad_mode, prec_mode, D_tok, workspace, stream);
}

extern "C" int comet_tc_track_tokens_ragged_f32(const void* split, const float* track_feats, long long t_sb, long long t_ss,
                                                long long t_sn, const float* coords, long long c_sb, long long c_ss,
                                                long long c_sn, const float* pos_emb, float* tokens, const int* num_tracks,
                                                int B, int S, int N, int C, int H, int W, int L, int r, int pad_mode,
                                                int prec_mode, int D_tok, void* workspace, comet_stream_t stream) {
  COMET_REQUIRE((long long)B * S * N == 0 || num_tracks, "null num_tracks");
  return tc_track_tokens(split, track_feats, t_sb, t_ss, t_sn, coords, c_sb, c_ss, c_sn, pos_emb, tokens, num_tracks, nullptr,
                         nullptr, B * S, B, S, N, C, H, W, L, r, pad_mode, prec_mode, D_tok, workspace, stream);
}

extern "C" int comet_tc_track_tokens_varlen_f32(const void* split, const float* track_feats, long long t_sb, long long t_ss,
                                                long long t_sn, const float* coords, long long c_sb, long long c_ss,
                                                long long c_sn, const float* pos_emb, float* tokens, const int* num_tracks,
                                                const int* num_frames, int B, int S, int N, int C, int H, int W, int L, int r,
                                                int pad_mode, int prec_mode, int D_tok, void* workspace,
                                                comet_stream_t stream) {
  return tc_track_tokens(split, track_feats, t_sb, t_ss, t_sn, coords, c_sb, c_ss, c_sn, pos_emb, tokens, num_tracks,
                         num_frames, nullptr, B * S, B, S, N, C, H, W, L, r, pad_mode, prec_mode, D_tok, workspace, stream);
}

extern "C" int comet_tc_track_tokens_indexed_f32(const void* split, const float* track_feats, long long t_sb, long long t_ss,
                                                 long long t_sn, const float* coords, long long c_sb, long long c_ss,
                                                 long long c_sn, const float* pos_emb, float* tokens, const int* num_tracks,
                                                 const int* num_frames, const int* frame_index, int BS_src, int B, int S, int N,
                                                 int C, int H, int W, int L, int r, int pad_mode, int prec_mode, int D_tok,
                                                 void* workspace, comet_stream_t stream) {
  return tc_track_tokens(split, track_feats, t_sb, t_ss, t_sn, coords, c_sb, c_ss, c_sn, pos_emb, tokens, num_tracks,
                         num_frames, frame_index, BS_src, B, S, N, C, H, W, L, r, pad_mode, prec_mode, D_tok, workspace,
                         stream);
}

extern "C" int comet_tc_corr_volume_f32(const void* split, const float* targets, long long t_sb, long long t_ss,
                                        long long t_sn, float* const* vols, int B, int S, int N, int C, int H, int W,
                                        int L, int prec_mode, void* workspace, comet_stream_t stream) {
  tc::Params p{};
  int rc = tc_common(p, targets, t_sb, t_ss, t_sn, nullptr, 0, 0, 0, B, S, N, C, H, W, L, 0, COMET_PAD_ZEROS, prec_mode);
  if (rc != COMET_OK) return rc;
  if ((long long)B * S * N == 0) return COMET_OK;
  COMET_REQUIRE(split && targets && vols, "null pointer");
  for (int l = 0; l < L; ++l) {
    COMET_REQUIRE(vols[l], "null volume pointer for level %d", l);
    p.vol[l] = vols[l];
  }
  p.volume_mode = 1;
  return tc::launch(p, split, workspace, (cudaStream_t)stream);
}

#ifdef COMET_TC_TRACE
extern "C" void comet_tc_debug_stamps(long long* dev_buf) { comet::tc::g_stamps = dev_buf; }
#endif

extern "C" int comet_tc_status(void) {
  int* d = tc::status_word();
  int h = 0;
  if (!d || cudaMemcpy(&h, d, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;
  return h;
}
