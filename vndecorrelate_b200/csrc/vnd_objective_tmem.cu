// Batched stereo-image objective for velvet-noise candidates, tensor-memory variant (sm_100a).
//
// Same sums as vn_objective_kernel (vnd_objective.cu; reference: src/vndecorrelate/optimization.py:46-105 over the
// candidates of optimization.py:260-272), with the filtered channel's taps served the way fir_tmem_kernel serves
// them: the tile sits in tensor memory as Hankel rows (row m holds x[t0 + 96 m + c], c < 512), a tap with offset
// <= 512 - 32 (g + 1) is ONE tcgen05.ld of 32 columns for 32 consecutive frames of a lane, and only the far taps
// read the staged tile from shared memory (16-byte loads at a conflict-free pitch).  In vn_objective_kernel every tap
// is a shared-memory word per frame: 31 words per frame-evaluation against 128 B/clk/SM, which is what bounded it
// (profiles/r01e_vn_objective_ncu.txt: shared-memory pipe 63 %, issue 55 %).  Here the pipe carries ~9 words per
// frame-evaluation, and - unlike in the FIR - the TMEM refill is free: a tile is written to tensor memory once and
// then read by every candidate of the CTA's group (hundreds to 1024).
//
// Decomposition.  CTA = (chunk of tiles, clip, candidate group) as in vn_objective_kernel; one CTA per SM (it owns the
// SM's 512 TMEM columns).  A tile is 32 rows x 96 frames = 3072 frames, REPLICATED in the four lane quarters of
// tensor memory, because a warp can only read the quarter (warp index & 3): that way every warp owns whole candidates
// (no cross-warp reduction, no atomics, a fixed summation order per candidate): for each of its candidates a warp
// decodes the 43-word tap program (near / far operations for the three 32-frame groups of a row), runs the FIR for
// the groups one after the other, folds the frames into the polar moments (packed FADD2 / FMUL2 / FFMA2), reduces
// with shuffles and adds the tile's contribution to the candidate's float64 slots in shared memory.
//
// Used whenever tile + halo, the candidates' accumulators and the per-warp scratch fit in shared memory (BASELINE
// config 5 does with room to spare); otherwise vn_objective_kernel runs.  The per-frame arithmetic is that kernel's; the order in which a lane meets the frames
// differs, so float32 partial sums may differ in the last bits (far below the 5e-4 the scores are compared with; the
// max|theta| tracker is exact either way).

#include <stdlib.h>

#include "vnd_objective.cuh"
#include "vnd_tmem.cuh"

namespace vnd {

int obj_combine_launch(const double* chunk_partials, double* partials, int n_clips, int n_chunks, int n_cand, cudaStream_t st);

namespace {

using namespace tm;

constexpr int OT_ROWS = 32;                 // rows of a tile = lanes of a TMEM quarter
constexpr int OT_G = 3;                     // groups of RG consecutive frames per row and lane

// Shape of the kernel: RG frames per lane and group (a row is 3 RG frames, the tile 32 rows), W warps per CTA.
//   <32, 12>  one tcgen05.ld.x32 per tap and group; 163 registers -> 12 warps: 81 k evaluations/s (round 2, first build)
//   <16, 20>  one tcgen05.ld.x16 per tap and group; fits the 96 registers of a 20-warp CTA, the warp count the
//             shared-memory kernel needs to hide the polar moments' latencies
template <int RG_, int W_>
struct OtShape {
  static constexpr int RG = RG_, W = W_;
  static constexpr int R = OT_G * RG_;        // frames per row
  static constexpr int TILE = OT_ROWS * R;
  static constexpr int PITCH = R + 4;         // words between rows in shared memory (an odd number of 16-byte chunks)
  static constexpr int NT = W_ * 32;
  static_assert(((PITCH / 4) & 1) == 1 && R % 4 == 0, "conflict-free 16-byte row accesses");
  __host__ __device__ static constexpr int near_max(int g) { return kCols - RG_ * (g + 1); }
};

// Per-warp scratch (words): the candidate's program | decoded operations per group (+ the slack words tap_list
// prefetches) | segment tables per group (int4, 16-byte aligned).  Sized from the longest program of the family.
__host__ __device__ constexpr int ot_progwords(int mpw) { return (mpw + 3) & ~3; }
__host__ __device__ constexpr int ot_opstride(int mpw) { return (mpw + 4 + 3) & ~3; }
__host__ __device__ constexpr int ot_maxseg(int mpw) { return mpw > 4 ? (mpw - 1) / 3 : 1; }
__host__ __device__ constexpr int ot_warp_words(int mpw) { return ot_progwords(mpw) + OT_G * ot_opstride(mpw) + OT_G * ot_maxseg(mpw) * 4; }

struct OtParams {
  ObjParams o;
  int nblk;  // 96-frame blocks staged per tile (tile + halo, at least what the TMEM rows cover)
  int mpw;   // words of the longest candidate program
};

// Shared memory: [0, 16) TMEM base | float in[nblk][100] | float x1[32][100] | double acc[cand_per_group][OBJ_CHUNK_SLOTS] |
//                int scratch[warps][ot_warp_words]
extern __shared__ __align__(128) unsigned char ot_smem[];

// Decode candidate `prog` (SEGMENTED block: S, (n_neg, n_pos, gain) x S, taps) for the warp: operation words per group
// and, per group and segment, the tap counts with the number of LEADING tensor-memory taps of both lists.
template <class T>
__device__ __forceinline__ void decode_candidate(const int* __restrict__ prog, int nprog, int apply_gain, int* ops, int opstride, int4* segtab,
                                                 int smax, int lane) {
  const int S = prog[0];
  const int ntaps = nprog - 1 - 3 * S;
  const int* taps = prog + 1 + 3 * S;
  for (int k = lane; k < ntaps + 2; k += 32) {  // two slack words behind the lists
    const int i = k < ntaps ? taps[k] : 0;
#pragma unroll
    for (int g = 0; g < OT_G; ++g) {
      int op = 0;
      if (k < ntaps) {
        if (i <= T::near_max(g)) {
          op = i;
        } else {
          const int o = i + T::RG * g, A = o & 3, oal = o - A;
          const int blk = oal / T::R, w = oal - blk * T::R;
          int kx = (T::R - w) >> 2;
          if (kx > 31) kx = 31;
          op = kOpFar | (A << 24) | (kx << 16) | (blk * T::PITCH + w);
        }
      }
      ops[g * opstride + k] = op;
    }
  }
  for (int idx = lane; idx < OT_G * S; idx += 32) {  // one lane per (group, segment)
    const int g = idx / S, s = idx - g * S;
    const int* tq = taps;
    for (int k = 0; k < s; ++k) tq += prog[1 + 3 * k] + prog[2 + 3 * k];
    const int n_neg = prog[1 + 3 * s], n_pos = prog[2 + 3 * s], nmax = T::near_max(g);
    int a = 0, b = 0;
    while (a < n_neg && tq[a] <= nmax) ++a;
    while (b < n_pos && tq[n_neg + b] <= nmax) ++b;
    segtab[g * smax + s] = make_int4(n_neg, n_pos, a | (b << 16), apply_gain ? prog[3 + 3 * s] : __float_as_int(1.0f));
  }
}

template <class T>
__global__ void __launch_bounds__(T::NT, 1) vn_objective_tmem_kernel(const OtParams P) {
  constexpr int OT_RG = T::RG, OT_R = T::R, OT_TILE = T::TILE, OT_PITCH = T::PITCH, OT_NT = T::NT, OT_WARPS = T::W;
  const ObjParams& p = P.o;
  uint32_t* tm_slot = reinterpret_cast<uint32_t*>(ot_smem);
  float* s_in = reinterpret_cast<float*>(ot_smem + 16);
  const int in_words = (P.nblk * OT_PITCH + 3) & ~3;
  float* s_x1 = s_in + in_words;
  double* acc = reinterpret_cast<double*>(s_x1 + OT_ROWS * OT_PITCH);
  int* scratch = reinterpret_cast<int*>(acc + (size_t)p.cand_per_group * OBJ_CHUNK_SLOTS);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int chunk = blockIdx.x, clip = blockIdx.y, group = blockIdx.z;
  const int cand0 = group * p.cand_per_group;
  const int ncand = min(p.cand_per_group, p.n_cand - cand0);
  const float* __restrict__ x0 = p.clips + (long long)clip * p.clip_stride;
  const float* __restrict__ x1 = x0 + p.chan_stride;
  const int opstride = ot_opstride(P.mpw), smax = ot_maxseg(P.mpw);
  int* myprog = scratch + warp * ot_warp_words(P.mpw);
  int* myops = myprog + ot_progwords(P.mpw);
  int4* mysegs = reinterpret_cast<int4*>(myops + OT_G * opstride);

  if (warp == 0) tmem_alloc_all(tm_slot);
  for (int i = tid; i < ncand * OBJ_CHUNK_SLOTS; i += OT_NT) acc[i] = obj_acc_init(i % OBJ_CHUNK_SLOTS);
  tmem_fence_before();
  __syncthreads();
  tmem_fence_after();
  const int q = warp & 3;
  const uint32_t tbase = *tm_slot + ((uint32_t)(32 * q) << 16);
  const uint32_t row = smem_u32(s_in + lane * OT_PITCH);  // the lane's row of the staged tile
  const bool vec_ok = ((reinterpret_cast<uintptr_t>(x0) | reinterpret_cast<uintptr_t>(x1)) & 15) == 0;

  const long long tile_first = (long long)chunk * p.tiles_per_chunk;
  for (int ti = 0; ti < p.tiles_per_chunk; ++ti) {
    const long long t0 = (tile_first + ti) * OT_TILE;
    if (t0 >= p.frames) break;
    const long long remain = p.frames - t0;
    tmem_fence_before();
    __syncthreads();  // every warp is done with the previous tile (shared memory and tensor memory)
    // stage channel 0 (tile + halo) and channel 1 (tile) as 96-frame rows at a pitch of 100 words; zeros past the end
    {
      const int n4 = P.nblk * (OT_R / 4);
      for (int c = tid; c < n4; c += OT_NT) {
        const int blk = c / (OT_R / 4), w = 4 * (c - blk * (OT_R / 4));
        const long long i = (long long)blk * OT_R + w;
        float4 v;
        if (vec_ok && i + 4 <= remain) {
          v = *reinterpret_cast<const float4*>(x0 + t0 + i);
        } else {
          v.x = i < remain ? x0[t0 + i] : 0.0f;
          v.y = i + 1 < remain ? x0[t0 + i + 1] : 0.0f;
          v.z = i + 2 < remain ? x0[t0 + i + 2] : 0.0f;
          v.w = i + 3 < remain ? x0[t0 + i + 3] : 0.0f;
        }
        *reinterpret_cast<float4*>(s_in + blk * OT_PITCH + w) = v;
      }
      for (int c = tid; c < OT_ROWS * (OT_R / 4); c += OT_NT) {
        const int blk = c / (OT_R / 4), w = 4 * (c - blk * (OT_R / 4));
        const long long i = (long long)blk * OT_R + w;
        float4 v;
        if (vec_ok && i + 4 <= remain) {
          v = *reinterpret_cast<const float4*>(x1 + t0 + i);
        } else {
          v.x = i < remain ? x1[t0 + i] : 0.0f;
          v.y = i + 1 < remain ? x1[t0 + i + 1] : 0.0f;
          v.z = i + 2 < remain ? x1[t0 + i + 2] : 0.0f;
          v.w = i + 3 < remain ? x1[t0 + i + 3] : 0.0f;
        }
        *reinterpret_cast<float4*>(s_x1 + blk * OT_PITCH + w) = v;
      }
    }
    __syncthreads();
    tmem_fence_after();
    // the tile into tensor memory, once per quarter: the warps of a quarter share its sixteen 32-column units; row m
    // holds x[t0 + R m + c], i.e. 16-byte chunk c / 4 of the staged rows m, m + 1, ... (R / 4 chunks per staged row)
    for (int u = warp >> 2; u < kUnits; u += (OT_WARPS + 3 - q) / 4) {
      float4 v[8];
#pragma unroll
      for (int jj = 0; jj < 8; ++jj) {
        const int c4 = 8 * u + jj, blk = c4 / (OT_R / 4), w4 = c4 - blk * (OT_R / 4);
        v[jj] = *reinterpret_cast<const float4*>(s_in + (lane + blk) * OT_PITCH + 4 * w4);
      }
      tmem_st32(tbase + (uint32_t)(32 * u), v);
    }
    tmem_wait_st();
    tmem_fence_before();
    __syncthreads();
    tmem_fence_after();

    const bool whole = remain >= OT_TILE;
    for (int ci = warp; ci < ncand; ci += OT_WARPS) {
      const int w0 = p.offsets[cand0 + ci];
      const int nprog = p.offsets[cand0 + ci + 1] - w0;
      __syncwarp();
      for (int i = lane; i < nprog; i += 32) myprog[i] = p.words[w0 + i];
      __syncwarp();
      decode_candidate<T>(myprog, nprog, p.apply_gain, myops, opstride, mysegs, smax, lane);
      __syncwarp();
      const int S = myprog[0];
      LaneAcc2 b{{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, 0.f, 1.f, 0.f, 1.f, -1.f, -1.f};
      LaneAcc a{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 1.f, 0.f, 1.f};
#pragma unroll 1
      for (int g = 0; g < OT_G; ++g) {
        float yv[OT_RG];
#pragma unroll
        for (int r = 0; r < OT_RG; ++r) yv[r] = 0.0f;  // (run_segments assigns; keeps the compiler quiet)
        const int* ops = myops + g * opstride;
        run_segments<false, false>(mysegs + g * smax, 0, S, ops, tbase + (uint32_t)(OT_RG * g), row, yv);
        const float4* r1 = reinterpret_cast<const float4*>(s_x1 + lane * OT_PITCH + OT_RG * g);
        if (whole) {
#pragma unroll
          for (int j = 0; j < OT_RG / 4; ++j) {
            const float4 v = r1[j];
            lane_acc_pair(b, yv[4 * j], yv[4 * j + 1], v.x, v.y);
            lane_acc_pair(b, yv[4 * j + 2], yv[4 * j + 3], v.z, v.w);
          }
        } else {
          const long long n0 = (long long)lane * OT_R + OT_RG * g;  // first frame of this lane's group inside the tile
          const float* r1s = reinterpret_cast<const float*>(r1);
#pragma unroll
          for (int r = 0; r < OT_RG; ++r)
            if (n0 + r < remain) lane_acc_frame(a, yv[r], r1s[r]);
        }
      }
      if (whole) {
        a.sr = b.sr[0] + b.sr[1];
        a.srt = b.srt[0] + b.srt[1];
        a.srt2 = b.srt2[0] + b.srt2[1];
        a.srt3 = b.srt3[0] + b.srt3[1];
        a.slr = b.slr[0] + b.slr[1];
        a.sll = b.sll[0] + b.sll[1];
        a.d_pos = b.d_pos;
        a.s_pos = b.s_pos;
        a.d_neg = b.d_neg;
        a.s_neg = b.s_neg;
      }
      a.sr = warp_sum(a.sr);
      a.srt = warp_sum(a.srt);
      a.srt2 = warp_sum(a.srt2);
      a.srt3 = warp_sum(a.srt3);
      a.slr = warp_sum(a.slr);
      a.sll = warp_sum(a.sll);
      warp_best_ratio(a.d_pos, a.s_pos);
      warp_best_ratio(a.d_neg, a.s_neg);
      if (lane == 0) obj_acc_tile(acc + (size_t)ci * OBJ_CHUNK_SLOTS, a, (int)(remain < OT_TILE ? remain : OT_TILE));
    }
  }
  tmem_fence_before();
  __syncthreads();
  double* out = p.chunk_partials + (((size_t)clip * p.n_chunks + chunk) * p.n_cand + cand0) * OBJ_CHUNK_SLOTS;
  for (int i = tid; i < ncand * OBJ_CHUNK_SLOTS; i += OT_NT) out[i] = acc[i];
  if (warp == 0) tmem_dealloc_all(*tm_slot);
}

// Most chunks a clip's tiles are split into (shared rule with vnd_objective.cu): enough for 16 waves over all clips.
long long ot_max_chunks(long long tiles, int n_clips, int sm_count) {
  long long c = ceil_div<long long>((long long)sm_count * 16, n_clips > 0 ? n_clips : 1);
  if (c > tiles) c = tiles;
  return c < 1 ? 1 : c;
}

}  // namespace

using OtWide = OtShape<32, 12>;
using OtNarrow = OtShape<16, 20>;

// VND_OBJ_TMEM: 1 = 16 frames per lane x 20 warps, 2 = 32 frames per lane x 12 warps (anything else: the caller's
// shared-memory kernel)
static int ot_variant() {
  const char* e = getenv("VND_OBJ_TMEM");
  return e ? atoi(e) : 0;
}

size_t objective_tmem_workspace_bytes(long long frames, int n_clips, int n_cand, int sm_count) {
  const long long tiles = ceil_div<long long>(frames, OtNarrow::TILE);  // the finer tiling of the two shapes
  return (size_t)n_clips * ot_max_chunks(tiles, n_clips, sm_count) * n_cand * OBJ_CHUNK_SLOTS * 8 + 256;
}

// VND_EUNSUPPORTED (no error text) when the program family does not qualify; the caller then runs vn_objective_kernel.
template <class T>
static int ot_launch(const float* clips, long long frames, int n_clips, long long clip_stride, long long chan_stride,
                     const vnd_tap_program* cand, double* partials, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  constexpr int OT_R = T::R, OT_TILE = T::TILE, OT_PITCH = T::PITCH, OT_NT = T::NT, OT_WARPS = T::W;
  const int mpw = cand->max_channel_words > 0 ? cand->max_channel_words : 1;
  int halo = cand->halo > 0 ? cand->halo : 0;
  if (halo > frames) halo = (int)frames;
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  int nblk = (OT_TILE + halo + 3 + OT_R - 1) / OT_R + 1;  // far taps read whole 16-byte chunks: a little slack
  const int fill_blocks = OT_ROWS + (kCols + OT_R - 1) / OT_R;
  if (nblk < fill_blocks) nblk = fill_blocks;
  const size_t in_words = ((size_t)nblk * OT_PITCH + 3) & ~(size_t)3;
  const size_t fixed = 16 + (in_words + (size_t)OT_ROWS * OT_PITCH) * 4 + (size_t)OT_WARPS * ot_warp_words(mpw) * 4;
  const size_t budget = (size_t)kMaxDynSmem;
  if (fixed + OBJ_CHUNK_SLOTS * 8 * 16 > budget) return VND_EUNSUPPORTED;
  int cpg = (int)((budget - fixed) / (OBJ_CHUNK_SLOTS * 8));
  if (cpg > cand->channels) cpg = cand->channels;
  if (cpg > 1024) cpg = 1024;
  const long long tiles = ceil_div<long long>(frames, OT_TILE);
  const long long want = (long long)di.sm_count * 4;
  while ((long long)n_clips * tiles * ceil_div(cand->channels, cpg) < want && cpg > 4 * OT_WARPS) cpg = (cpg + 1) / 2;
  const long long groups = ceil_div(cand->channels, cpg);
  if (n_clips > 65535 || groups > 65535) return VND_EUNSUPPORTED;
  long long n_chunks = 1, best = -1;
  const long long cap = ot_max_chunks(tiles, n_clips, di.sm_count);
  for (long long c = 1; c <= cap; ++c) {  // fewest waves x tiles per chunk (see plan_objective)
    const long long tpc_c = ceil_div<long long>(tiles, c);
    const long long real_c = ceil_div<long long>(tiles, tpc_c);
    const long long waves = ceil_div<long long>((long long)n_clips * real_c * groups, di.sm_count);
    const long long cost = waves * tpc_c * 4096 + real_c;
    if (best < 0 || cost < best) {
      best = cost;
      n_chunks = real_c;
    }
  }
  int tpc = (int)ceil_div<long long>(tiles, n_chunks);
  if (const char* e = getenv("VND_OBJ_TPC")) {  // tuning: force the tiles per chunk (clamped to what the workspace was sized for)
    const int v = atoi(e);
    if (v > 0 && ceil_div<long long>(tiles, v) <= cap) tpc = v;
  }
  n_chunks = ceil_div<long long>(tiles, tpc);
  const size_t need = (size_t)n_clips * n_chunks * cand->channels * OBJ_CHUNK_SLOTS * 8;
  VND_REQUIRE(workspace && workspace_bytes >= need, VND_ENOMEM, "objective workspace too small: need %zu bytes, have %zu", need, workspace_bytes);
  OtParams P{};
  P.o.clips = clips;
  P.o.frames = frames;
  P.o.clip_stride = clip_stride;
  P.o.chan_stride = chan_stride;
  P.o.words = cand->words;
  P.o.offsets = cand->offsets;
  P.o.n_cand = cand->channels;
  P.o.apply_gain = cand->apply_gain;
  P.o.halo = halo;
  P.o.cand_per_group = cpg;
  P.o.tiles_per_chunk = tpc;
  P.o.n_chunks = (int)n_chunks;
  P.o.chunk_partials = reinterpret_cast<double*>(workspace);
  P.nblk = nblk;
  P.mpw = mpw;
  const size_t smem = fixed + (size_t)cpg * OBJ_CHUNK_SLOTS * 8;
  VND_CUDA_OK(cudaFuncSetAttribute(vn_objective_tmem_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  dim3 grid((unsigned)n_chunks, (unsigned)n_clips, (unsigned)groups);
  vn_objective_tmem_kernel<T><<<grid, OT_NT, smem, st>>>(P);
  rc = after_launch("vn_objective_tmem_kernel");
  if (rc) return rc;
  return obj_combine_launch(P.o.chunk_partials, partials, n_clips, (int)n_chunks, cand->channels, st);
}

int vn_objective_tmem_launch(const float* clips, long long frames, int n_clips, long long clip_stride, long long chan_stride,
                             const vnd_tap_program* cand, double* partials, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  switch (ot_variant()) {
    case 1: return ot_launch<OtNarrow>(clips, frames, n_clips, clip_stride, chan_stride, cand, partials, workspace, workspace_bytes, st);
    case 2: return ot_launch<OtWide>(clips, frames, n_clips, clip_stride, chan_stride, cand, partials, workspace, workspace_bytes, st);
    default: return VND_EUNSUPPORTED;
  }
}

}  // namespace vnd
