// Shared between the batched decorrelate (vnd_batch.cu) and the sum-of-squares scans (vnd_post.cu).
#pragma once

#include "vnd_common.cuh"

namespace vnd {

// rms_normalize's DUAL_MONO gain of one float32 channel from its two sums of squares (numpy's dtype chain: the mean
// divides in float64 and stores float32, epsilon is cast to float32); rms_gain_kernel and the batch use it alike.
__device__ __forceinline__ float rms_gain_f32(float sum_x, float sum_y, long long frames) {
  const float mx = __double2float_rn((double)sum_x / (double)frames);
  const float my = __double2float_rn((double)sum_y / (double)frames);
  return __fdiv_rn(__fsqrt_rn(mx), __fsqrt_rn(fadd(my, 1e-10f)));
}

// Column 4 i + j of a batch of n clips packed in (rows, 2) float32 arrays: j = 0, 1 are the two channels of clip i's
// input x, j = 2, 3 those of its FIR / M/S / width result y.  Clip i is rows [offs[i], offs[i + 1]) of both.
// The sums pass ends with the clip's two gains, so that the placement pass only multiplies (its SASS holds no
// multiply-add; a correctly rounded division is built from them).
struct BatchSumCols {
  const float* x;
  const float* y;
  const long long* offs;
  float* sums;         // 4 n floats
  float* gains;        // 2 n floats
  unsigned* arrivals;  // n counters of finished columns, zeroed by the stereo pass that precedes the sums
  __device__ __forceinline__ void column(int col, const float** base, long long* st, long long* n) const {
    const int clip = col >> 2, j = col & 3;
    const long long o = offs[clip];
    *base = (j < 2 ? x : y) + 2 * o + (j & 1);
    *st = 2;
    *n = offs[clip + 1] - o;
  }
  __device__ __forceinline__ void store_clip(int clip, float sx0, float sx1, float sy0, float sy1) const {
    const long long frames = offs[clip + 1] - offs[clip];
    float* s = sums + 4 * (long long)clip;
    s[0] = sx0;
    s[1] = sx1;
    s[2] = sy0;
    s[3] = sy1;
    gains[2 * (long long)clip] = rms_gain_f32(sx0, sy0, frames);
    gains[2 * (long long)clip + 1] = rms_gain_f32(sx1, sy1, frames);
  }
  // one column at a time (the cluster scan): the last of a clip's four columns to finish computes its gains
  __device__ __forceinline__ void store(int col, float v) const {
    const int clip = col >> 2;
    sums[col] = v;
    __threadfence();
    if (atomicAdd(&arrivals[clip], 1u) == 3u) {
      __threadfence();
      const volatile float* s = sums + 4 * (long long)clip;
      store_clip(clip, s[0], s[1], s[2], s[3]);
    }
  }
};

// HaasEffect.decorrelate at one output frame (float64 throughout, SURVEY.md A.6): channel 0 comes from input frame
// (a0, b0) and channel 1 from (a1, b1) - one of them the delayed frame -, each 0 where its frame lies outside the
// signal (v0, v1 false).  A mono signal has a == b.  haas_kernel and haas_batch_kernel both call it, so the batch
// gives every clip the single call's bits.
__device__ __forceinline__ double2 haas_frame(float a0, float b0, bool v0, float a1, float b1, bool v1, int mode_ms, int mono,
                                              int use_width, double width) {
  // the channel pair as the reference stores it after the optional LR->MS, at one frame
  auto chan = [&](float af, float bf, bool v, int c) -> double {
    if (!v) return 0.0;
    const double a = (double)af, b = (double)bf;
    if (mode_ms && !mono) return c == 0 ? dmul(dadd(a, b), 0.5) : dmul(dsub(a, b), 0.5);
    return c == 0 ? a : b;
  };
  double c0 = chan(a0, b0, v0, 0);
  double c1 = chan(a1, b1, v1, 1);
  if (mode_ms) {
    const double l = dadd(c0, c1), r = dsub(c0, c1);
    c0 = l;
    c1 = r;
    if (mono) {
      c0 = dmul(c0, 0.5);
      c1 = dmul(c1, 0.5);
    }
  }
  if (use_width) {
    double M = dmul(dadd(c0, c1), 0.5);
    double S = dmul(dsub(c0, c1), 0.5);
    M = dmul(M, dsub(1.0, width));
    S = dmul(S, width);
    c0 = dadd(M, S);
    c1 = dsub(M, S);
  }
  return make_double2(c0, c1);
}

// CTA b of a batched kernel with `tile` outputs per CTA takes clip i, the last one with V[i] <= b where
// V[i] = floor(offs[i] / tile) + i, and that clip's tile b - V[i].  V[i + 1] - V[i] >= max(1, ceil(frames_i / tile)),
// so floor(rows / tile) + n CTAs - a grid known from host scalars alone - cover every tile of every clip and give an
// empty clip one CTA (its Haas zero fill); the few CTAs past a clip's last tile exit.
__device__ __forceinline__ int batch_clip_of(const long long* offs, int n, int tile, long long b) {
  int lo = 0, hi = n - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (offs[mid] / tile + mid <= b) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}

// vnd_fir.cu: the batched fused stereo pass (vn_stereo_kernel over (clip, tile) pairs); out is (rows + n delay, 2)
// C-order, clip i from row offs[i] + i delay.  VND_EUNSUPPORTED (no error text) when tile + halo does not fit.
// `arrivals` (nullable): n counters the pass zeroes for the sums pass behind it.
int vn_batch_stereo_launch(const float* x, long long rows, const long long* offs, int n_clips, const int* prog_of,
                           const vnd_tap_program* taps, const vnd_epilogue* ep, void* out, int out_dtype, int delay, int delay_ch,
                           unsigned* arrivals, cudaStream_t st);

// vnd_post.cu: the cluster scan of seq_sumsq_cluster_kernel over these columns, and its shape constants
int batch_sumsq_cluster_launch(const BatchSumCols& cols, int n_cols, cudaStream_t st);
int seq_sumsq_cluster_width();  // CTAs per column
int seq_sumsq_scan_round();     // addends per CTA and round
int seq_sumsq_scan_head();      // addends chained by one thread before the scan starts

// vnd_batch.cu
#ifndef VND_BATCH_TILE
#define VND_BATCH_TILE 4096
#endif
// Outputs per CTA of the batched stereo and placement kernels.  Measured on a B200 against 1024 (the single-clip kernel's
// tile): 512 clips of 5-15 s, default VelvetNoise, 12.27 -> 11.58 ms; without normaliser 7.91 -> 7.23 ms - the filter's
// halo (1324 frames at 44.1 kHz) is staged once per tile.
constexpr int kBatchTile = VND_BATCH_TILE;
bool vn_batch_smem(int halo, int prog_words, size_t* smem);
size_t vn_batch_workspace_bytes(long long rows, int n_clips, int rms);
int vn_batch_launch(const float* x, long long rows, const long long* offs, int n_clips, const int* prog_of, const vnd_tap_program* taps,
                    const vnd_epilogue* ep, void* out, int out_dtype, void* workspace, cudaStream_t st);

// Output frames per CTA of haas_batch_kernel (16 per thread).
constexpr int kHaasTile = 4096;
// vnd_haas_batch_dev's launch: one haas_batch_kernel over floor(out_rows / kHaasTile) + n_clips CTAs, none when
// out_rows == 0.  offs (n + 1), out_offs (n) and clips (n, 16-byte aligned) are device arrays.
int haas_batch_launch(const float* x, const long long* offs, int n_clips, const vnd_haas_clip* clips, const long long* out_offs,
                      long long out_rows, double* out, cudaStream_t st);

// ------------------------------------------------------------------------------------------------
// One step of many live signals (vnd_vn_block_step_dev, vnd_haas_block_step_dev, vnd_fir_block_step_dev).  Signal i
// has received received[i] = T0 frames before the step and gets rows [offs[i], offs[i + 1]) of the packed (rows, C)
// blocks, so it has T1 = T0 + those rows after it.  Its history holds its frames [T0 - H, T0) as rows [i H, i H + H) of
// hist_in; the step writes frames [T1 - H, T1) to hist_out (frames before 0 as +0).  Together they are the signal's
// virtual input: a frame before T0 - H, before 0 or from T1 on reads as +0.  The first out_blocks CTAs write the
// outputs, one (signal, output tile) pair each (times a channel group for the convolve step) through batch_clip_of over
// out_offs; the n * hchunks CTAs after them write the history.  The stereo steps are float32 with C = 2; the convolve
// step's rows hold C values of its compute dtype.
// ------------------------------------------------------------------------------------------------
struct BlockStepParams {
  const void* x;                // packed (rows, C) blocks
  const long long* offs;        // n + 1
  const long long* received;    // n
  const long long* emitted;     // n, output frames written before the step (the velvet-noise and convolve steps)
  const long long* out_offs;    // n + 1: signal i writes out rows [out_offs[i], out_offs[i + 1])
  const void* hist_in;          // (n, H, C)
  void* hist_out;               // (n, H, C)
  long long out_blocks;
  int n, H, hchunks;
  int C;                        // values per row (the convolve step)
};

// History frames per CTA of the history pass.
constexpr int kHistTile = 4096;

// Frame f of signal `sig`'s virtual input, (+0, +0) where it has no frame.
__device__ __forceinline__ float2 block_step_frame(const BlockStepParams& b, int sig, long long f, long long T0, long long T1, long long x0) {
  if (f >= T0) return f < T1 ? __ldg(reinterpret_cast<const float2*>(b.x) + x0 + (f - T0)) : make_float2(0.0f, 0.0f);
  if (f < 0 || f < T0 - b.H) return make_float2(0.0f, 0.0f);
  return __ldg(reinterpret_cast<const float2*>(b.hist_in) + (long long)sig * b.H + (f - (T0 - b.H)));
}

// History CTA j: chunk j % hchunks of signal j / hchunks's new history.
__device__ __forceinline__ void block_step_history(const BlockStepParams& b, long long j) {
  const int sig = (int)(j / b.hchunks);
  const int lo = (int)(j % b.hchunks) * kHistTile;
  const int hi = lo + kHistTile < b.H ? lo + kHistTile : b.H;
  const long long T0 = b.received[sig], x0 = b.offs[sig];
  const long long T1 = T0 + (b.offs[sig + 1] - x0);
  float2* __restrict__ h2 = reinterpret_cast<float2*>(b.hist_out) + (long long)sig * b.H;
  for (int i = lo + (int)threadIdx.x; i < hi; i += (int)blockDim.x) h2[i] = block_step_frame(b, sig, T1 - b.H + i, T0, T1, x0);
}

// Grid of a block step: output CTAs (tile outputs each) then history CTAs; false when it exceeds the grid limit.
bool block_step_grid(BlockStepParams* b, long long out_rows, int tile, long long* blocks);

// vnd_fir.cu: the velvet-noise step (vn_block_step_kernel); float32 (out_rows, 2) out.  VND_EUNSUPPORTED (no error
// text) when tile + halo does not fit (the vn_batch_smem rule).
int vn_block_step_launch(BlockStepParams b, long long out_rows, const int* prog_of, const vnd_tap_program* taps, const vnd_epilogue* ep,
                         float* out, cudaStream_t st);
// vnd_batch.cu: the Haas step (haas_block_step_kernel); float64 (out_rows, 2) out, signal i's first row is its output
// frame T0.
int haas_block_step_launch(BlockStepParams b, long long out_rows, const vnd_haas_clip* clips, double* out, cudaStream_t st);
// vnd_fir.cu: the convolve step (fir_block_step_kernel) on (rows, b.C) blocks of `dtype` (VND_F32 or VND_F64); float32
// (out_rows, b.C) out.  Program k of `taps` is channels [k C, (k + 1) C).
int fir_block_step_launch(BlockStepParams b, long long out_rows, int dtype, const int* prog_of, const vnd_tap_program* taps, float* out,
                          cudaStream_t st);

}  // namespace vnd
