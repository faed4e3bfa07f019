// Tensor-memory sparse FIR (sm_100a): the throughput kernel for planar float32 slabs.
//
// Same arithmetic, in the same order, as VelvetNoise.convolve
// (src/vndecorrelate/decorrelation.py:393-415): bit-identical to fir_tile_kernel and the reference.
//
// Why tensor memory.  The FIR is a gather with data-dependent offsets: every (output, tap) pair
// moves one word from on-chip memory to a register.  Through shared memory that is 4 B x 30 taps
// per output against 128 B/clk/SM, which caps the kernel near 38 % of the HBM roofline however
// the loads are scheduled (profiles/r01_summary.md).  Blackwell has a second on-chip datapath
// into the register file: tcgen05.ld from tensor memory, measured at >= 390 B/clk/SM
// (tools/microbench/tmem_bw.cu) and independent of the LSU pipe.  tcgen05.ld.32x32b hands lane l
// of a warp N CONSECUTIVE columns of TMEM lane (row) l starting at a run-time column — exactly
// "32 consecutive samples starting at a tap offset" if row l holds the samples that follow the
// first output of lane l.
//
// Layout.  A tile is 128 rows x R = 96 outputs.  TMEM row m (512 columns x 4 B) holds
// x[t0 + 96 m + c], c in [0, 512): a Hankel arrangement.  Compute thread (row m, group g < 3)
// owns outputs 96 m + 32 g + r, r < 32; a tap with offset i <= 416 is one 32-column tcgen05.ld at
// column i + 32 g followed by 16 packed adds (FADD2).  With log-distributed impulses 22 of the 30
// taps of BASELINE config 3 qualify.  The remaining (far) taps read the staged tile from shared
// memory with 16-byte loads.  Shared memory holds the tile as 96-sample blocks at a pitch of 100
// words, so that lanes (rows) hit distinct bank groups with LDS.128 / STS.128: one 384-byte TMA
// row, three tile buffers.
//
// Roles (one CTA of 16 warps per SM; warp w works on TMEM lane quarter w & 3, which is also its
// scheduler).  Warps 0-11 compute (setmaxnreg 144).  Warps 12-15, one per quarter (setmaxnreg 80),
// move data: they refill the quarter's TMEM rows with the next tile (LDS.128 -> tcgen05.st) as soon
// as the quarter's compute warps are past their last tensor-memory tap — i.e. while those warps run
// the trailing all-far segments and stage their outputs — and issue the TMA requests: ONE tensor
// load per tile, two tiles ahead (a 100 x nblk box over x seen as rows of 96 samples: the four
// out-of-bounds columns are zero-filled, which produces the 100-word pitch), and one tensor store per
// quarter and tile (the same trick clips the pad columns).  Hand-overs go through mbarriers; there
// is no CTA-wide barrier inside a run.  The data-movement lanes sleep between mbarrier polls so that
// polling does not take issue slots from the compute warps.
//
// The kernel only runs interior tiles (tile + halo completely inside the signal); the launcher
// reports how many frames it covered and the caller finishes the tail of every channel with the
// general tile kernel.

#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)
#include <stdlib.h>

#include "vnd_common.cuh"
#include "vnd_fir.cuh"
#include "vnd_tmem.cuh"

#ifndef VND_TM_RUN_MAX
#define VND_TM_RUN_MAX 512  // most consecutive tiles of one channel in a CTA run
#endif
#ifndef VND_TM_RUN_MIN
#define VND_TM_RUN_MIN 48   // fewest (a run pays a prologue and a pipeline fill of about two tiles)
#endif

#ifdef VND_TM_TRACE
// Debug builds only: clock64() of a few events per warp and tile of CTA 0 (tools/trace_tmem.py).
__device__ unsigned long long g_tm_trace[16][64][8];
#define VND_TRACE(tile, ev)                                                                    \
  do {                                                                                         \
    if (blockIdx.x == 0 && (threadIdx.x & 31) == 0 && (tile) < 64) g_tm_trace[threadIdx.x >> 5][tile][ev] = clock64(); \
  } while (0)
extern "C" int vnd_debug_tm_trace(unsigned long long* out) {
  return (int)cudaMemcpyFromSymbol(out, g_tm_trace, sizeof(g_tm_trace));
}
#else
#define VND_TRACE(tile, ev) \
  do {                      \
  } while (0)
#endif

namespace vnd {

namespace {

using namespace tm;  // tensor-memory primitives and the tap machinery (vnd_tmem.cuh)
constexpr int kBarBytes = 384;

// Shape of the kernel: kG compute warps per lane quarter, each thread owning kRG consecutive outputs of its row (a row is
// kR = kG * kRG outputs), kNBuf tile buffers in shared memory, kRegsCompute / kRegsHelper registers per compute /
// data-movement thread (setmaxnreg; 32 * (4 kG kRegsCompute + 4 kRegsHelper) must not exceed what the launch allocates).
// Round 2 measured other shapes and schedules of this kernel on a B200, 148 channels x 28.8 M frames (Gsamples/s, all
// bit-exact; profiles/r02_summary.md, DESIGN.md section 4) against 357-380 for this one: 2 warps x 48 outputs 325,
// 2 x 64 with rows of 128 338, 2 x 32 298 (272 with software-pipelined tensor-memory taps), the trailing all-far
// segment paired tap by tap with the first 278, quarters taking the far phase in turns 375 / 268, the all-far segment
// first 219-344, two tensor-memory taps per round trip 300 / 278, a symmetric CTA without data-movement warps 355.
// A tap's tcgen05.ld round trip bounds the tensor-memory phase, and every form of overlap inside a warp made the taps
// slower.  Code removed; last present at commit 915ac5a.
constexpr int kG = 3;                       // compute warps per lane quarter
constexpr int kR = kG * kRG;                // outputs per row
constexpr int kCW = 4 * kG;                 // compute warps (warp w: lane quarter w & 3, group w >> 2)
constexpr int kHelpers = 4;                 // one data-movement warp per quarter
constexpr int kNT = (kCW + kHelpers) * 32;
constexpr int kTile = kRows * kR;
constexpr int kPitch = kR + 4;              // row pitch in shared memory (words); an odd number of 16-byte chunks
constexpr int kUnitsPerBlock = kR / 32;
constexpr int kNBuf = 3;
constexpr int kRegsCompute = 144, kRegsHelper = 80;
constexpr int kLaunchRegs = (65536 / kNT) / 8 * 8;
// mbarrier slots (uint64 each)
constexpr int B_IN_FULL = 0, B_IN_FREE = kNBuf, B_ST_FULL = 2 * kNBuf, B_ST_FREE = 2 * kNBuf + 4, B_TM_FULL = 2 * kNBuf + 8,
              B_TM_FREE = 2 * kNBuf + 12, B_COUNT = 2 * kNBuf + 16;
static_assert(kR % 32 == 0 && ((kPitch / 4) & 1) == 1, "rows are whole 32-column units; the pitch is an odd number of chunks");
static_assert(32 * (kCW * kRegsCompute + kHelpers * kRegsHelper) <= kLaunchRegs * kNT, "register file");
static_assert(kRegsCompute % 8 == 0 && kRegsHelper % 8 == 0, "setmaxnreg takes multiples of 8");
static_assert(B_COUNT * 8 <= 256, "mbarriers");
// Largest tap offset served from TMEM (every group of a row: group g alone could reach kRG (kG - 1 - g) samples
// further, but per-group tap mixes measured slower - 366 instead of 384 Gsamples/s on the same box - because the
// three warps of a quarter hand TMEM back together and the quarter waits for its slowest group).
constexpr int kNearMax = kCols - kR;

struct TmParams {
  // TMA descriptors of x and y seen as (R samples, rows, channels).  The boxes are R + 4 wide: the four
  // out-of-bounds elements per row are zero-filled on load and clipped on store, which gives the
  // padded row pitch in shared memory with ONE request per tile instead of one per row.
  alignas(64) CUtensorMap tmx;
  alignas(64) CUtensorMap tmy;
  FirParams f;
  int nblk;      // R-sample blocks staged per tile (tile + halo)
  int opstride;  // words reserved for the program and for each decoded list
  int stagger_ns;  // start-of-run delay between lane quarters (see stagger())
  int tiles_per_run;
  int runs_per_channel;
  int n_runs;
  int tiles_per_channel;  // interior tiles
};

// Dynamic shared memory: [0,256) mbarriers | [256,260) TMEM base | [260,264) first all-far segment |
//   [384, ...) float in[kNBuf][nblk][pitch] | float stage[128][pitch] | int program[] | int ops[kG][] | int4 segtab[]
// The role functions rebuild their pointers from this symbol so that every access stays in the
// shared address space (LDS/STS, not generic loads).
extern __shared__ __align__(128) unsigned char tm_smem[];

struct Smem {
  uint64_t* bars;
  int* s_near_end;  // first segment without a tap in the TMEM window
  float* in_all;
  float* stage;
  int* sprog;
  int* ops;  // [kG][opstride]: decoded tap operations per thread group
  int4* segtab;  // per segment: taps of the negative and positive list, their leading tensor-memory taps, gain bits
  int bufw;
  int opstride;
  __device__ __forceinline__ explicit Smem(const TmParams& P) {
    bars = reinterpret_cast<uint64_t*>(tm_smem);
    s_near_end = reinterpret_cast<int*>(tm_smem + 260);
    in_all = reinterpret_cast<float*>(tm_smem + kBarBytes);
    bufw = (P.nblk * kPitch + 31) & ~31;  // TMA tensor copies want 128-byte aligned shared-memory addresses
    stage = in_all + kNBuf * bufw;
    sprog = reinterpret_cast<int*>(stage + kRows * kPitch);
    opstride = P.opstride;
    ops = sprog + opstride;
    segtab = reinterpret_cast<int4*>(ops + kG * opstride);  // opstride is a multiple of 4 words: 16-byte aligned
  }
};
constexpr size_t tm_tail_words(int opstride) {  // program + decoded lists + segment tables
  return (size_t)(3 + kG) * opstride;
}

struct RunInfo {
  int c, first_tile, n_tiles, nprog;
};

// Per-run prologue shared by both roles (every thread of the CTA takes part): decode the run, copy
// the unfiltered channel through or load and decode the channel's program.  Returns false for a
// copied run.
__device__ __forceinline__ bool begin_run(const TmParams& P, const Smem& sm, int run, int tid, RunInfo& r) {
  const FirParams& p = P.f;
  r.c = run / P.runs_per_channel;
  r.first_tile = (run % P.runs_per_channel) * P.tiles_per_run;
  r.n_tiles = P.tiles_per_channel - r.first_tile;
  if (r.n_tiles > P.tiles_per_run) r.n_tiles = P.tiles_per_run;
  const int w0 = p.offsets[r.c];
  r.nprog = p.offsets[r.c + 1] - w0;
  if (r.nprog == 0) {  // unfiltered channel: copy through (decorrelation.py:399-400)
    const float* xc = reinterpret_cast<const float*>(p.x) + (long long)r.c * p.x_sc;
    float* yc = p.y + (long long)r.c * p.y_sc;
    const long long t_begin = (long long)r.first_tile * kTile, t_end = t_begin + (long long)r.n_tiles * kTile;
    for (long long t = t_begin + 4 * tid; t < t_end; t += 4 * kNT)
      *reinterpret_cast<float4*>(yc + t) = *reinterpret_cast<const float4*>(xc + t);
    return false;
  }
  __syncthreads();  // the pipeline of the previous run has drained: program, buffers and TMEM are free
  for (int i = tid; i < r.nprog; i += kNT) sm.sprog[i] = p.words[w0 + i];
  __syncthreads();
  const int S = sm.sprog[0];
  const int* taps = sm.sprog + 1 + 3 * S;
  const int ntaps = r.nprog - 1 - 3 * S;
  if (tid == 0) {  // the segment table; segments from near_end on have no tap inside the TMEM window
    const int* tq = taps;
    int ne = 0;
    for (int s = 0; s < S; ++s) {
      const int n_neg = sm.sprog[1 + 3 * s], n = n_neg + sm.sprog[2 + 3 * s];
      for (int k = 0; k < n; ++k)
        if (tq[k] <= kNearMax) ne = s + 1;
      int a = 0, b = 0;  // leading tensor-memory taps of the two lists
      while (a < n_neg && tq[a] <= kNearMax) ++a;
      while (n_neg + b < n && tq[n_neg + b] <= kNearMax) ++b;
      sm.segtab[s] = make_int4(n_neg, n - n_neg, a | (b << 16), p.apply_gain ? sm.sprog[3 + 3 * s] : __float_as_int(1.0f));
      tq += n;
    }
    *sm.s_near_end = ne;
  }
  // decode the taps for the thread groups (group g owns outputs kRG g .. kRG g + kRG - 1 of a row)
  for (int t = tid; t < kG * (ntaps + 2); t += kNT) {
    const int g = t / (ntaps + 2), k = t - g * (ntaps + 2);
    int op = 0;  // two slack words behind each list
    if (k < ntaps) {
      const int i = taps[k];
      if (i <= kNearMax) {
        op = i;
      } else {
        const int o = i + kRG * g, A = o & 3, oal = o - A;
        const int blk = oal / kR, w = oal - blk * kR;
        int kx = (kR - w) >> 2;
        if (kx > 31) kx = 31;
        op = kOpFar | (A << 24) | (kx << 16) | (blk * kPitch + w);
      }
    }
    sm.ops[g * sm.opstride + k] = op;
  }
  __syncthreads();
  return true;
}

// The four lane quarters run the same tile pipeline on four schedulers but share ONE shared-memory
// pipe, which the far taps and the TMEM refill load heavily while the tensor-memory taps do not use
// it at all.  Started together, the quarters stay in phase: the pipe saturates while everybody is in
// the far-tap phase and idles during the tensor-memory phase (ncu: issue slots and the shared-memory
// pipe each ~50 % busy).  Delaying quarter q by q x 3 us (half a tile) at the start of every run interleaves
// the phases; nothing couples the quarters tightly enough to pull them back (the tile ring is three
// deep, TMEM and staging hand-overs are per quarter).
__device__ __forceinline__ void stagger(int q, int ns) {
  for (int k = 0; k < q; ++k) __nanosleep((unsigned)ns);
}

// ---------------------------------------------------------------- data-movement warp of lane quarter q
// One elected lane per warp: quarter 0 issues the tile loads (one TMA request per tile, kNBuf - 1 tiles
// ahead), every quarter stores its own 32 staged rows (one request per tile).
__device__ __noinline__ void helper_main(const TmParams& P, uint32_t tbase, int tid) {
  const Smem sm(P);
  const int nblk = P.nblk, n_runs = P.n_runs, stagger_ns = P.stagger_ns;  // P lives behind a generic pointer here
  const int lane = tid & 31, q = (tid >> 5) & 3;
  const int m = 32 * q + lane;
  const uint32_t bars = smem_u32(sm.bars), in0 = smem_u32(sm.in_all), buf_bytes = (uint32_t)sm.bufw * 4u;
  const uint32_t stage_q = smem_u32(sm.stage + 32 * q * kPitch);
  const uint32_t tx_bytes = (uint32_t)nblk * (kPitch * 4u);  // the whole box counts, zero-filled columns included
  const void* tmx = &P.tmx;
  const void* tmy = &P.tmy;
  const bool loader = q == 0 && lane == 0;
  int fb = 0, lb = 0;          // ring slots of the next fill and of the next load
  unsigned fpar = 0, lpar = 1; // in_full parity of the next fill; in_free parity that releases slot lb
  unsigned tpar = 0;           // parity of the tile counter (TMEM and staging barriers)
  for (int run = blockIdx.x; run < n_runs; run += gridDim.x) {
    RunInfo r;
    if (!begin_run(P, sm, run, tid, r)) continue;
    stagger(q, stagger_ns);
    int load_row = r.first_tile * kRows;  // first row (R samples) of the next tile to load
    int store_row = r.first_tile * kRows + 32 * q;
    int to_load = r.n_tiles;
#define VND_ISSUE_LOAD()                                                                   \
  do {                                                                                     \
    if (loader) {                                                                          \
      mbar_wait_u32(bars + 8u * (B_IN_FREE + lb), lpar); /* every warp is done with the tile that was there */ \
      const uint32_t full = bars + 8u * (B_IN_FULL + lb);                                  \
      mbar_expect_tx_u32(full, tx_bytes);                                                  \
      fence_proxy_async();                                                                 \
      tma_load_3d(in0 + (uint32_t)lb * buf_bytes, tmx, 0, load_row, r.c, full);            \
    }                                                                                      \
    load_row += kRows;                                                                     \
    --to_load;                                                                             \
    if (++lb == kNBuf) {                                                                   \
      lb = 0;                                                                              \
      lpar ^= 1u;                                                                          \
    }                                                                                      \
  } while (0)
    for (int d = 0; d < kNBuf - 1 && to_load > 0; ++d) VND_ISSUE_LOAD();
    for (int ti = 0; ti < r.n_tiles; ++ti) {
      mbar_wait_u32(bars + 8u * (B_IN_FULL + fb), fpar);
      VND_TRACE(ti, 4);
      mbar_wait_u32(bars + 8u * (B_TM_FREE + q), tpar ^ 1u);  // the quarter is past its last TMEM tap of the previous tile
      tmem_fence_after();
      VND_TRACE(ti, 0);
      {  // fill row m: 32 columns per step; a block of R samples is R / 32 steps, then the pitch skips 4 words
        const float4* src = reinterpret_cast<const float4*>(sm.in_all + fb * sm.bufw + m * kPitch);
        uint32_t tcol = tbase;
        int sub = 0;
#pragma unroll 1
        for (int k32 = 0; k32 < kUnits; ++k32) {
          float4 v[8];
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) v[jj] = src[jj];
          tmem_st32(tcol, v);
          tcol += 32;
          src += 8;
          if (++sub == kUnitsPerBlock) {
            sub = 0;
            src += 1;
          }
        }
        tmem_wait_st();
      }
      tmem_fence_before();
      __syncwarp();
      VND_TRACE(ti, 1);
      if (lane == 0) {
        mbar_arrive_u32(bars + 8u * (B_TM_FULL + q));
        mbar_arrive_u32(bars + 8u * (B_IN_FREE + fb));
      }
      if (++fb == kNBuf) {
        fb = 0;
        fpar ^= 1u;
      }
      if (to_load > 0) VND_ISSUE_LOAD();
      if (ti > 0 && lane == 0) {  // the previous tile's 32 rows of this quarter
        mbar_wait_u32(bars + 8u * (B_ST_FULL + q), tpar ^ 1u);
        tma_store_3d(tmy, 0, store_row, r.c, stage_q);
        bulk_commit();
        bulk_wait_read0();
        mbar_arrive_u32(bars + 8u * (B_ST_FREE + q));
      }
      if (ti > 0) store_row += kRows;
      __syncwarp();
      VND_TRACE(ti, 2);
      tpar ^= 1u;
    }
#undef VND_ISSUE_LOAD
    if (lane == 0) {
      mbar_wait_u32(bars + 8u * (B_ST_FULL + q), tpar ^ 1u);
      tma_store_3d(tmy, 0, store_row, r.c, stage_q);
      bulk_commit();
      bulk_wait_read0();
      mbar_arrive_u32(bars + 8u * (B_ST_FREE + q));
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------- compute warp (q, g)
__device__ __noinline__ void compute_main(const TmParams& P, uint32_t tbase, int tid) {
  const Smem sm(P);
  const int n_runs = P.n_runs, stagger_ns = P.stagger_ns;  // P lives behind a generic pointer here
  const int lane = tid & 31, warp = tid >> 5;
  const int q = warp & 3, g = warp >> 2;
  const int m = 32 * q + lane;
  uint64_t* bars = sm.bars;
  const uint32_t tcol0 = tbase + (uint32_t)(kRG * g);  // column of this thread's first output
  const int4* segtab = sm.segtab;
  int b = 0;           // ring slot of the current tile
  unsigned fpar = 0;   // in_full parity of slot b
  unsigned tpar = 0;   // parity of the tile counter (TMEM and staging barriers)
  for (int run = blockIdx.x; run < n_runs; run += gridDim.x) {
    RunInfo r;
    if (!begin_run(P, sm, run, tid, r)) continue;
    stagger(q, stagger_ns);
    const int S = sm.sprog[0];
    const int near_end = *sm.s_near_end;
    for (int ti = 0; ti < r.n_tiles; ++ti) {
      const uint32_t row = smem_u32(sm.in_all + b * sm.bufw + m * kPitch);
      const int* ops = sm.ops + g * sm.opstride;
      VND_TRACE(ti, 0);
      mbar_wait(&bars[B_IN_FULL + b], fpar);
      float yv[kRG];
#pragma unroll
      for (int rr = 0; rr < kRG; ++rr) yv[rr] = 0.0f;
      mbar_wait(&bars[B_TM_FULL + q], tpar);
      tmem_fence_after();
      VND_TRACE(ti, 1);
      run_segments<false>(segtab, 0, near_end, ops, tcol0, row, yv);
      VND_TRACE(ti, 2);
      tmem_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_TM_FREE + q]);  // the helper may fill TMEM for the next tile
      VND_TRACE(ti, 6);
      run_segments<true>(segtab, near_end, S, ops, tcol0, row, yv);
      VND_TRACE(ti, 3);
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars[B_IN_FREE + b]);  // this warp is done with the tile buffer
      mbar_wait(&bars[B_ST_FREE + q], tpar ^ 1u);
      VND_TRACE(ti, 5);  // the previous tile's stores have read the staging rows
      {
        float4* dst = reinterpret_cast<float4*>(sm.stage + m * kPitch + kRG * g);
#pragma unroll
        for (int jj = 0; jj < kRG / 4; ++jj) dst[jj] = make_float4(yv[4 * jj], yv[4 * jj + 1], yv[4 * jj + 2], yv[4 * jj + 3]);
      }
      fence_proxy_async();
      __syncwarp();
      VND_TRACE(ti, 4);
      if (lane == 0) mbar_arrive(&bars[B_ST_FULL + q]);
      tpar ^= 1u;
      if (++b == kNBuf) {
        b = 0;
        fpar ^= 1u;
      }
    }
  }
}

__global__ void __launch_bounds__(kNT, 1) fir_tmem_kernel(const __grid_constant__ TmParams P) {
  const Smem sm(P);
  uint32_t* tm_slot = reinterpret_cast<uint32_t*>(tm_smem + 256);

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  if (tid == 0) {
    for (int b = 0; b < kNBuf; ++b) {
      mbar_init(&sm.bars[B_IN_FULL + b], 1);
      mbar_init(&sm.bars[B_IN_FREE + b], kCW + kHelpers);
    }
    for (int k = 0; k < 4; ++k) {
      mbar_init(&sm.bars[B_ST_FULL + k], kG);
      mbar_init(&sm.bars[B_ST_FREE + k], 1);
      mbar_init(&sm.bars[B_TM_FULL + k], 1);
      mbar_init(&sm.bars[B_TM_FREE + k], kG);
    }
    mbar_fence_init();
  }
  if (warp == 0) tmem_alloc_all(tm_slot);
  tmem_fence_before();
  __syncthreads();
  tmem_fence_after();
  const uint32_t tbase = *tm_slot + ((uint32_t)(32 * (warp & 3)) << 16);
  if (warp >= kCW) {
    set_max_regs_dec<kRegsHelper>();
    helper_main(P, tbase, tid);
  } else {
    set_max_regs_inc<kRegsCompute>();
    compute_main(P, tbase, tid);
  }
  tmem_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc_all(*tm_slot);
}

}  // namespace

// VND_TM_STAGGER_NS overrides the start-of-run delay between lane quarters (tuning).
static const int g_stagger_ns = [] {
  const char* e = getenv("VND_TM_STAGGER_NS");
  return e ? atoi(e) : 2000;
}();

// cuTensorMapEncodeTiled through the runtime (no link against libcuda).
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess || qres != cudaDriverEntryPointSuccess) p = nullptr;
    (void)cudaGetLastError();
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// base[c * stride_c + row * R + k] as a (R, rows, channels) float32 tensor with a (R + 4, box_rows, 1) box
static bool encode_rows(CUtensorMap* tm, const void* base, long long frames, long long stride_c, int channels, int box_rows, int R) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)R, (cuuint64_t)(frames / R), (cuuint64_t)channels};
  const cuuint64_t strides[2] = {(cuuint64_t)R * 4u, (cuuint64_t)stride_c * 4u};
  const cuuint32_t box[3] = {(cuuint32_t)(R + 4), (cuuint32_t)box_rows, 1u};
  const cuuint32_t estr[3] = {1u, 1u, 1u};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Split every channel into equal runs so that the persistent CTAs finish together: pick the number of runs per
// channel that minimises (waves of runs) x (tiles per run + two tiles of prologue).
static void plan_runs(long long tiles, int channels, int sm_count, int* tiles_per_run, int* runs_per_channel) {
  long long best_cost = -1;
  int best_rpc = 1;
  const long long rpc_lo = ceil_div<long long>(tiles, VND_TM_RUN_MAX);
  long long rpc_hi = tiles / VND_TM_RUN_MIN;
  if (rpc_hi < rpc_lo) rpc_hi = rpc_lo;
  for (long long rpc = rpc_lo; rpc <= rpc_hi; ++rpc) {
    const long long tpr = ceil_div<long long>(tiles, rpc);
    const long long real_rpc = ceil_div<long long>(tiles, tpr);
    const long long waves = ceil_div<long long>(real_rpc * channels, sm_count);
    const long long cost = waves * (tpr + 2);
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best_rpc = (int)real_rpc;
    }
  }
  *tiles_per_run = (int)ceil_div<long long>(tiles, best_rpc);
  *runs_per_channel = (int)ceil_div<long long>(tiles, *tiles_per_run);
}

// Runs the interior tiles of every channel and reports the frames covered per channel in
// *frames_done (a multiple of the tile).  VND_EUNSUPPORTED (no error text) when the request does
// not qualify; the caller then uses the other kernels for everything.
int fir_tmem_launch(const FirParams& f, int max_prog_words, cudaStream_t st, long long* frames_done) {
  *frames_done = 0;
  if (!f.bulk_ok || f.x_st != 1 || f.y_st != 1) return VND_EUNSUPPORTED;
  if ((reinterpret_cast<uintptr_t>(f.y) % 16) != 0 || (f.y_sc % 4) != 0) return VND_EUNSUPPORTED;
  int nblk = kRows + (f.halo + 4 + kR - 1) / kR;
  const int fill_blocks = kRows + (kCols + kR - 1) / kR;  // the TMEM fill reads 512 columns of every row
  if (nblk < fill_blocks) nblk = fill_blocks;
  const int opstride = (max_prog_words + 4 + 3) & ~3;  // a multiple of 4 words: the segment tables behind the lists stay 16-byte aligned
  const size_t bufw = ((size_t)nblk * kPitch + 31) & ~(size_t)31;
  const size_t smem = kBarBytes + kNBuf * bufw * 4 + (size_t)kRows * kPitch * 4 + tm_tail_words(opstride) * 4;
  if (smem > (size_t)kMaxDynSmem || nblk > 256) return VND_EUNSUPPORTED;  // a TMA box has at most 256 rows
  if (f.channels > 1 && (f.x_sc % 4 != 0 || f.x_sc < f.frames || f.y_sc < f.frames)) return VND_EUNSUPPORTED;
  const long long span = (long long)nblk * kR;  // samples a tile's bulk loads touch
  if (f.frames < span + 3LL * kTile) return VND_EUNSUPPORTED;  // fewer than four interior tiles
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  TmParams P{};
  P.f = f;
  P.nblk = nblk;
  P.opstride = opstride;
  P.stagger_ns = g_stagger_ns;
  const long long sx = f.channels > 1 ? f.x_sc : f.frames, sy = f.channels > 1 ? f.y_sc : f.frames;
  if (!encode_rows(&P.tmx, f.x, f.frames, sx, f.channels, nblk, kR) || !encode_rows(&P.tmy, f.y, f.frames, sy, f.channels, 32, kR))
    return VND_EUNSUPPORTED;  // no tensor-map encoder in this driver: the other kernels take over
  const long long tiles = (f.frames - span) / kTile + 1;
  if (tiles > 0x3fffffffLL / (f.channels > 0 ? f.channels : 1)) return VND_EUNSUPPORTED;
  P.tiles_per_channel = (int)tiles;
  plan_runs(tiles, f.channels, di.sm_count, &P.tiles_per_run, &P.runs_per_channel);
  P.n_runs = P.runs_per_channel * f.channels;
  VND_CUDA_OK(cudaFuncSetAttribute(fir_tmem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int grid = di.sm_count;
  if (grid > P.n_runs) grid = P.n_runs;
  fir_tmem_kernel<<<(unsigned)grid, kNT, smem, st>>>(P);
  rc = after_launch("fir_tmem_kernel");
  if (rc) return rc;
  *frames_done = tiles * kTile;
  return VND_OK;
}

// Debug / test aid (not part of the ABI in include/vnd_b200.h): the run plan of the kernel for a slab -
// out[0] = tiles per run, out[1] = runs per channel, out[2] = frames per tile; bench.py uses it to place a parity
// window across a run boundary.  Returns VND_EUNSUPPORTED when the slab would not take the tensor-memory kernel.
extern "C" int vnd_debug_fir_plan(long long frames, int channels, int halo, int* out) {
  if (!out) return VND_EUNSUPPORTED;
  halo = (halo + 3) & ~3;
  int nblk = kRows + (halo + 4 + kR - 1) / kR;
  const int fill_blocks = kRows + (kCols + kR - 1) / kR;
  if (nblk < fill_blocks) nblk = fill_blocks;
  const long long span = (long long)nblk * kR;
  if (nblk > 256 || frames < span + 3LL * kTile) return VND_EUNSUPPORTED;
  DeviceInfo di;
  if (device_info(&di)) return VND_ECUDA;
  const long long tiles = (frames - span) / kTile + 1;
  int tpr = 0, rpc = 0;
  plan_runs(tiles, channels, di.sm_count, &tpr, &rpc);
  out[0] = tpr;
  out[1] = rpc;
  out[2] = kTile;
  return VND_OK;
}

}  // namespace vnd
