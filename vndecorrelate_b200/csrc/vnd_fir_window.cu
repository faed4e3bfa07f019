// Register-window sparse FIR (sm_100a): the throughput kernel for planar float32 slabs.
//
// Same arithmetic, in the same order, as VelvetNoise.convolve
// (src/vndecorrelate/decorrelation.py:393-415): bit-identical to fir_tile_kernel and the reference.
//
// Why a second kernel.  ncu on fir_tile_kernel (profiles/) shows the shared-memory data pipe at
// 88 % of peak with DRAM at 22 %: every (output, tap) pair moves one 4-byte word from shared memory
// to a register, 128 B/clk/SM, and every CTA pays its prologue for only 32 outputs per thread.
//
//   * Register window.  A velvet-noise filter with log-distributed impulses has a dense head (the
//     whole first decay segment lies within 32 samples).  A lane owns R CONSECUTIVE outputs and
//     keeps x[n0 .. n0 + R + W) in registers; a tap with offset < W becomes R FADDs on statically
//     indexed registers, selected by a warp-uniform switch — no shared-memory traffic.  Only taps
//     with offset >= W read shared memory (R consecutive words per lane, all R loads in flight).
//   * R is odd, so lanes are R words apart and every warp-wide LDS.32 is bank-conflict free on the
//     densely laid out tile (which is what lets one TMA bulk copy stage it).
//   * "acc -= x" for the negative list is done as adds followed by a negation that rides on the
//     operand modifier of the next instruction: fl(-a - b) == -fl(a + b) exactly in
//     round-to-nearest, so the bits are unchanged.
//   * Persistent CTAs.  A CTA walks a run of consecutive tiles of one channel: the tap program is
//     loaded once per run, the next tile's TMA bulk load (cp.async.bulk + mbarrier) is in flight
//     while the current tile is computed (two tile buffers), and a warp's 32 R contiguous outputs
//     leave through a per-warp staging buffer with one TMA bulk store.

#include "vnd_common.cuh"
#include "vnd_fir.cuh"

// Tuning knobs (overridable at build time for experiments): outputs per lane (odd), window length,
// warps per CTA, minimum CTAs per SM for the register allocator, tiles per run.
#ifndef VND_WIN_R
#define VND_WIN_R 29
#endif
#ifndef VND_WIN_W
#define VND_WIN_W 32
#endif
#ifndef VND_WIN_NW
#define VND_WIN_NW 4
#endif
#ifndef VND_WIN_MINB
#define VND_WIN_MINB 4
#endif
#ifndef VND_WIN_RUN
#define VND_WIN_RUN 32
#endif

namespace vnd {

template <int K, int R, int W>
__device__ __forceinline__ void add_win(float (&acc)[R], const float (&w)[R + W]) {
  if constexpr (K < W) {
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = fadd(acc[r], w[r + K]);
  }
}

#define VND_CASE(K) \
  case (K): add_win<(K), R, W>(acc, w); break;
#define VND_CASE4(K) VND_CASE(K) VND_CASE((K) + 1) VND_CASE((K) + 2) VND_CASE((K) + 3)
#define VND_CASE16(K) VND_CASE4(K) VND_CASE4((K) + 4) VND_CASE4((K) + 8) VND_CASE4((K) + 12)

// All R words of a far tap are loaded before the first add: R independent loads in flight.
// NEG folds the pending negation of the accumulator into the add (free operand modifier).
template <int R, bool NEG>
__device__ __forceinline__ void add_far(const float* __restrict__ q, float (&acc)[R]) {
  float t[R];
#pragma unroll
  for (int r = 0; r < R; ++r) t[r] = q[r];
#pragma unroll
  for (int r = 0; r < R; ++r) acc[r] = NEG ? fadd(-acc[r], t[r]) : fadd(acc[r], t[r]);
}

template <int R, int W>
__device__ __forceinline__ void add_tap(int off, const float* __restrict__ px, float (&acc)[R], const float (&w)[R + W]) {
  if (off < W) {
    switch (off) {
      VND_CASE16(0)
      VND_CASE16(16)
      VND_CASE16(32)
      VND_CASE16(48)
      default: break;
    }
  } else {
    add_far<R, false>(px + off, acc);
  }
}

struct WinParams {
  FirParams f;
  int store_bulk_ok;
  int runs_per_channel;
  int tiles_per_run;
  long long n_runs;
};

// One segment whose taps are all beyond the window.  Returns with acc holding the segment sum
// (sign applied), before the gain.
template <int R>
__device__ __forceinline__ void far_segment(const float* __restrict__ px, const int* __restrict__ tp, int n_neg, int n_pos,
                                            float (&acc)[R]) {
#pragma unroll
  for (int r = 0; r < R; ++r) acc[r] = 0.0f;
  int off = tp[0];  // one word of slack follows the program, so the prefetches below stay in bounds
  for (int k = 0; k < n_neg; ++k) {
    const int nxt = tp[k + 1];
    add_far<R, false>(px + off, acc);
    off = nxt;
  }
  if (n_pos > 0) {
    const int* tq = tp + n_neg;
    int nxt = tq[1];
    if (n_neg > 0) add_far<R, true>(px + off, acc);  // acc = -(sum of the negative taps) + x
    else add_far<R, false>(px + off, acc);
    off = nxt;
    for (int k = 1; k < n_pos; ++k) {
      nxt = tq[k + 1];
      add_far<R, false>(px + off, acc);
      off = nxt;
    }
  } else if (n_neg > 0) {
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = -acc[r];
  }
}

// Shared memory: [0,32) two mbarriers | float tile[2][tile + halo] | float stage[NW][32 R] | int program[]
template <int R, int W, int NW, int MINB>
__global__ void __launch_bounds__(NW * 32, MINB) fir_window_kernel(const WinParams P) {
  static_assert(R % 2 == 1 && W <= 64, "R must be odd (conflict-free lane stride), W at most 64");
  constexpr int NT = NW * 32;
  constexpr int BLK = 32 * R;
  constexpr int TILE = NW * BLK;
  const FirParams& p = P.f;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
  const int span = TILE + p.halo;  // multiple of 4
  float* tiles = reinterpret_cast<float*>(smem_raw + 32);
  float* stage_all = tiles + 2 * span;
  int* sprog = reinterpret_cast<int*>(stage_all + NW * BLK);
  __shared__ int s_win_shared;

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  float* stage = stage_all + warp * BLK;
  bool pending_store = false;
  unsigned use0 = 0, use1 = 0;  // how often each tile buffer has been filled (mbarrier phase)

  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_fence_init();
  }
  __syncthreads();

  const long long tiles_in_channel = ceil_div<long long>(p.frames, TILE);
  for (long long run = blockIdx.x; run < P.n_runs; run += gridDim.x) {
    const int c = (int)(run / P.runs_per_channel);
    const long long first_tile = (run % P.runs_per_channel) * (long long)P.tiles_per_run;
    long long n_tiles = tiles_in_channel - first_tile;
    if (n_tiles > P.tiles_per_run) n_tiles = P.tiles_per_run;
    const int w0 = p.offsets[c];
    const int nprog = p.offsets[c + 1] - w0;
    const float* __restrict__ xc = reinterpret_cast<const float*>(p.x) + (long long)c * p.x_sc;
    float* __restrict__ yc = p.y + (long long)c * p.y_sc;

    if (nprog == 0) {  // unfiltered channel: copy through (decorrelation.py:399-400)
      const long long t_begin = first_tile * TILE;
      long long t_end = t_begin + n_tiles * TILE;
      if (t_end > p.frames) t_end = p.frames;
      for (long long t = t_begin + tid; t < t_end; t += NT) yc[t] = xc[t];
      continue;
    }

    // ---- per-run setup: program, window segment count, first tile load ----
    __syncthreads();  // everyone is done with the previous run's program and tile buffers
    for (int i = tid; i < nprog; i += NT) sprog[i] = p.words[w0 + i];
    if (tid == 0) sprog[nprog] = 0;  // slack word read by the tap prefetch
    __syncthreads();
    const int S = sprog[0];
    const int* seg = sprog + 1;
    if (tid == 0) {
      int sw = 0;
      const int* tq = sprog + 1 + 3 * S;
      for (int s = 0; s < S; ++s) {
        const int n = seg[3 * s] + seg[3 * s + 1];
        for (int k = 0; k < n; ++k)
          if (tq[k] < W) sw = s + 1;
        tq += n;
      }
      s_win_shared = sw;
    }

    // issue the load of tile `ti` of this run into buffer `buf`; the part past the end of the
    // signal is zero-filled by all threads (adding +0 == the reference dropping the tap)
    auto issue = [&](long long ti, int buf) -> bool {
      const long long t0 = (first_tile + ti) * TILE;
      const long long remain = p.frames - t0;
      const int nvalid = (int)(remain < span ? remain : span);
      const int nbulk = nvalid & ~3;
      float* dst = tiles + buf * span;
      if (tid == 0 && nbulk > 0) {
        fence_proxy_async();
        mbar_expect_tx(&bars[buf], (uint32_t)nbulk * 4u);
        bulk_g2s(dst, xc + t0, (uint32_t)nbulk * 4u, &bars[buf]);
      }
      for (int i = nbulk + tid; i < span; i += NT) dst[i] = (i < nvalid) ? xc[t0 + i] : 0.0f;
      return nbulk > 0;
    };

    bool armed0 = false, armed1 = false;
    armed0 = issue(0, 0);
    __syncthreads();  // s_win_shared and the zero fill of tile 0 are visible
    const int s_win = s_win_shared;

    for (long long ti = 0; ti < n_tiles; ++ti) {
      const int buf = (int)(ti & 1);
      if (ti + 1 < n_tiles) {  // prefetch the next tile into the other buffer (free since the last barrier)
        const bool a = issue(ti + 1, buf ^ 1);
        if (buf) armed0 = a;
        else armed1 = a;
      }
      if (buf == 0) {
        if (armed0) {
          mbar_wait(&bars[0], use0 & 1);
          ++use0;
        }
      } else {
        if (armed1) {
          mbar_wait(&bars[1], use1 & 1);
          ++use1;
        }
      }
      const float* sx = tiles + buf * span;
      const long long t0 = (first_tile + ti) * TILE;
      const long long remain = p.frames - t0;
      const int b = warp * BLK;

      if (b < remain) {  // warp-uniform
        const float* px = sx + b + R * lane;
        float yv[R];
        const int* tp = sprog + 1 + 3 * S;

        // Phase 1: the leading segments that own taps inside the register window.  While the window
        // is live the running output is NOT kept in registers: after segment 0 it simply is the
        // scaled accumulator, and in the rare case of further window segments it is parked in the
        // warp's staging buffer.  That keeps the kernel at 128 registers (16 warps per SM).
        if (s_win > 0) {
          float w[R + W];
#pragma unroll
          for (int j = 0; j < R + W; ++j) w[j] = px[j];
          if (s_win > 1 && pending_store) {  // the staging buffer is about to be written
            if (lane == 0) bulk_wait_read0();
            __syncwarp();
            pending_store = false;
          }
          float acc[R];
          for (int s = 0; s < s_win; ++s) {
            const int n_neg = seg[3 * s], n_tot = n_neg + seg[3 * s + 1];
#pragma unroll
            for (int r = 0; r < R; ++r) acc[r] = 0.0f;
            int off = tp[0];
            for (int k = 0; k < n_tot; ++k) {
              const int nxt = tp[k + 1];  // prefetch: keeps the offset load off the dispatch chain
              if (k == n_neg && k > 0) {
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] = -acc[r];  // 0 - a - b == -(0 + a + b) bit for bit
              }
              add_tap<R, W>(off, px, acc, w);
              off = nxt;
            }
            if (n_neg == n_tot && n_neg > 0) {
#pragma unroll
              for (int r = 0; r < R; ++r) acc[r] = -acc[r];
            }
            tp += n_tot;
            if (p.apply_gain) {
              const float gain = __int_as_float(seg[3 * s + 2]);
#pragma unroll
              for (int r = 0; r < R; ++r) acc[r] = fmul(acc[r], gain);
            }
            if (s_win > 1) {
              if (s == 0) {
#pragma unroll
                for (int r = 0; r < R; ++r) stage[R * lane + r] = fadd(0.0f, acc[r]);
              } else {
#pragma unroll
                for (int r = 0; r < R; ++r) stage[R * lane + r] = fadd(stage[R * lane + r], acc[r]);
              }
            }
          }
          if (s_win > 1) {
#pragma unroll
            for (int r = 0; r < R; ++r) yv[r] = stage[R * lane + r];
          } else {
#pragma unroll
            for (int r = 0; r < R; ++r) yv[r] = fadd(0.0f, acc[r]);  // y = 0 + acc: the reference adds into zeros
          }
        } else {
#pragma unroll
          for (int r = 0; r < R; ++r) yv[r] = 0.0f;
        }

        // Phase 2: every remaining tap is beyond the window; the window registers are dead here,
        // which leaves room for R independent loads in flight per tap.
        for (int s = s_win; s < S; ++s) {
          const int n_neg = seg[3 * s], n_pos = seg[3 * s + 1];
          float acc[R];
          far_segment<R>(px, tp, n_neg, n_pos, acc);
          tp += n_neg + n_pos;
          if (p.apply_gain) {
            const float gain = __int_as_float(seg[3 * s + 2]);
#pragma unroll
            for (int r = 0; r < R; ++r) acc[r] = fmul(acc[r], gain);
          }
#pragma unroll
          for (int r = 0; r < R; ++r) yv[r] = fadd(yv[r], acc[r]);
        }

        // transpose through the warp's staging buffer, then one bulk store (or a guarded tail)
        if (pending_store) {
          if (lane == 0) bulk_wait_read0();
          __syncwarp();
          pending_store = false;
        }
#pragma unroll
        for (int r = 0; r < R; ++r) stage[R * lane + r] = yv[r];
        const bool full = (long long)b + BLK <= remain;
        if (full && P.store_bulk_ok) {
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) {
            bulk_s2g(yc + t0 + b, stage, BLK * 4u);
            bulk_commit();
          }
          pending_store = true;
        } else {
          __syncwarp();
#pragma unroll 4
          for (int k = 0; k < R; ++k) {
            const int i = k * 32 + lane;
            if (b + i < remain) yc[t0 + b + i] = stage[i];
          }
          __syncwarp();
        }
      }
      __syncthreads();  // all warps are done with this tile buffer; the prefetched one is zero-filled
    }
  }
  if (pending_store && lane == 0) bulk_wait_read0();  // shared memory must outlive the bulk reads
}

template <int R, int W, int NW, int MINB>
static int launch_window(const FirParams& f, int max_prog_words, int store_bulk_ok, cudaStream_t st) {
  constexpr int BLK = 32 * R;
  constexpr int TILE = NW * BLK;
  if (f.frames < TILE) return VND_EUNSUPPORTED;
  const size_t smem = 32 + (size_t)2 * (TILE + f.halo) * 4 + (size_t)NW * BLK * 4 + (size_t)(max_prog_words + 4) * 4;
  auto k = fir_window_kernel<R, W, NW, MINB>;
  // the kernel's static shared memory (s_win_shared, 128-byte aligned) comes out of the same 227 KB as the dynamic part:
  // without it, halos whose dynamic part fits but whose sum does not made cudaFuncSetAttribute fail instead of declining
  cudaFuncAttributes fa;
  VND_CUDA_OK(cudaFuncGetAttributes(&fa, k));
  if (smem + fa.sharedSizeBytes > (size_t)kMaxDynSmem) return VND_EUNSUPPORTED;
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  WinParams P{};
  P.f = f;
  P.f.tile = TILE;
  P.store_bulk_ok = store_bulk_ok;
  const long long tiles = ceil_div<long long>(f.frames, TILE);
  P.tiles_per_run = (int)(tiles < VND_WIN_RUN ? tiles : VND_WIN_RUN);
  P.runs_per_channel = (int)ceil_div<long long>(tiles, P.tiles_per_run);
  P.n_runs = (long long)P.runs_per_channel * f.channels;
  VND_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  VND_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, NW * 32, smem));
  if (per_sm < 1) return VND_EUNSUPPORTED;
  long long grid = (long long)di.sm_count * per_sm;
  if (grid > P.n_runs) grid = P.n_runs;
  k<<<(unsigned)grid, NW * 32, smem, st>>>(P);
  return after_launch("fir_window_kernel");
}

int fir_window_launch(const FirParams& p, int max_prog_words, cudaStream_t st) {
  if (!p.bulk_ok || p.x_st != 1 || p.y_st != 1) return VND_EUNSUPPORTED;
  const int store_bulk_ok = ((reinterpret_cast<uintptr_t>(p.y) % 16) == 0 && (p.y_sc % 4) == 0) ? 1 : 0;
  return launch_window<VND_WIN_R, VND_WIN_W, VND_WIN_NW, VND_WIN_MINB>(p, max_prog_words, store_bulk_ok, st);
}

}  // namespace vnd
