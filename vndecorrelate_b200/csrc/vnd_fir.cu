// Sparse velvet-noise FIR kernels (sm_100a) and their launchers.
//
// Reference arithmetic reproduced here (paths relative to the reference root):
//   VelvetNoise.convolve          src/vndecorrelate/decorrelation.py:393-415   (SEGMENTED order)
//   convolve_velvet_noise         src/vndecorrelate/decorrelation.py:630-660   (ASCENDING order)
//   VelvetNoise.decorrelate       src/vndecorrelate/decorrelation.py:417-442   (fused epilogue)
//   encode_signal_to_side_channel src/vndecorrelate/utils/dsp.py:40-63
//   apply_stereo_width            src/vndecorrelate/utils/dsp.py:21-37
//
// Design: one CTA owns `tile` consecutive outputs of one channel (or of one stereo pair).  The
// input tile plus a right halo of `halo` samples (the filter is anti-causal: y[t] needs
// x[t + i]) is staged in shared memory — by one TMA bulk copy (cp.async.bulk, UBLKCP) when the
// channel is contiguous in time — together with the channel's tap program.  Lane l of a warp owns
// outputs base + l + 32 r, r < R: for a warp-uniform tap offset the 32 lanes read 32 consecutive
// words (conflict-free LDS), and each of the R stores is one full 128-byte line.  Samples past the
// end of the signal are staged as +0: adding +0 is bit-identical to the reference dropping the tap.

#include <stdlib.h>

#include "vnd_common.cuh"
#include "vnd_batch.cuh"
#include "vnd_fir.cuh"

namespace vnd {

template <typename T>
struct is_f64 { static constexpr bool value = false; };
template <>
struct is_f64<double> { static constexpr bool value = true; };

// One accumulation step in the reference's arithmetic: acc (-|+)= x with fp32 storage.
template <typename TIn>
__device__ __forceinline__ float step_sub(float acc, TIn x) {
  if constexpr (is_f64<TIn>::value) return __double2float_rn(dsub((double)acc, x));
  else return fsub(acc, x);
}
template <typename TIn>
__device__ __forceinline__ float step_add(float acc, TIn x) {
  if constexpr (is_f64<TIn>::value) return __double2float_rn(dadd((double)acc, x));
  else return fadd(acc, x);
}

// Packed float32 arithmetic (sm_100+: FADD2 / FMUL2, two IEEE round-to-nearest operations per instruction on an aligned
// register pair): the same bits as two scalar operations in half the issue slots.  The tile kernel issues one LDS and
// one add per (output, tap) pair; with packed adds the long-filter configuration (300 taps, shared-memory pipe bound)
// spends 1.5 instead of 2 issue slots per pair.
typedef unsigned long long fir_pair_t;
#define VND_FIR_PACKED(name, op)                                                   \
  __device__ __forceinline__ void name(float& a0, float& a1, float b0, float b1) { \
    fir_pair_t ra, rb;                                                             \
    asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a0), "f"(a1));                   \
    asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b0), "f"(b1));                   \
    asm(op ".rn.f32x2 %0, %0, %1;" : "+l"(ra) : "l"(rb));                         \
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(ra));                  \
  }
VND_FIR_PACKED(fir_add2, "add")
VND_FIR_PACKED(fir_sub2, "sub")
VND_FIR_PACKED(fir_mul2, "mul")

// Runs one channel's tap program for R outputs per lane.  `px` points at the staged sample of
// this lane's first output; consecutive outputs of the lane are `STRIDE` samples apart.
template <typename TIn, int MODE, int R, int STRIDE>
__device__ __forceinline__ void run_program(const TIn* __restrict__ px, const int* __restrict__ sprog, int apply_gain,
                                            float (&yv)[R]) {
#pragma unroll
  for (int r = 0; r < R; ++r) yv[r] = 0.0f;
  if constexpr (MODE == MODE_SEG) {
    const int S = sprog[0];
    const int* seg = sprog + 1;
    const int* tp = sprog + 1 + 3 * S;
    for (int s = 0; s < S; ++s) {
      const int n_neg = seg[3 * s + 0];
      const int n_pos = seg[3 * s + 1];
      const float gain = __int_as_float(seg[3 * s + 2]);
      float acc[R];
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r] = 0.0f;
      if constexpr (!is_f64<TIn>::value && (R % 2 == 0)) {  // float32: packed adds, the loads of a tap issued together
        for (int k = 0; k < n_neg; ++k) {
          const TIn* q = px + tp[k];
          float t[R];
#pragma unroll
          for (int r = 0; r < R; ++r) t[r] = q[r * STRIDE];
#pragma unroll
          for (int r = 0; r < R; r += 2) fir_sub2(acc[r], acc[r + 1], t[r], t[r + 1]);
        }
        tp += n_neg;
        for (int k = 0; k < n_pos; ++k) {
          const TIn* q = px + tp[k];
          float t[R];
#pragma unroll
          for (int r = 0; r < R; ++r) t[r] = q[r * STRIDE];
#pragma unroll
          for (int r = 0; r < R; r += 2) fir_add2(acc[r], acc[r + 1], t[r], t[r + 1]);
        }
        tp += n_pos;
        if (apply_gain) {
#pragma unroll
          for (int r = 0; r < R; r += 2) fir_mul2(acc[r], acc[r + 1], gain, gain);
        }
#pragma unroll
        for (int r = 0; r < R; r += 2) fir_add2(yv[r], yv[r + 1], acc[r], acc[r + 1]);
      } else {
        for (int k = 0; k < n_neg; ++k) {
          const TIn* q = px + tp[k];
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = step_sub<TIn>(acc[r], q[r * STRIDE]);
        }
        tp += n_neg;
        for (int k = 0; k < n_pos; ++k) {
          const TIn* q = px + tp[k];
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = step_add<TIn>(acc[r], q[r * STRIDE]);
        }
        tp += n_pos;
        if (apply_gain) {
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = fmul(acc[r], gain);
        }
#pragma unroll
        for (int r = 0; r < R; ++r) yv[r] = fadd(yv[r], acc[r]);
      }
    }
  } else {
    constexpr bool kF64 = is_f64<TIn>::value || MODE == MODE_ASC64;
    const int K = sprog[0];
    const int* e = sprog + 1;
    for (int k = 0; k < K; ++k) {
      const TIn* q = px + e[3 * k];
      const double coef = __hiloint2double(e[3 * k + 2], e[3 * k + 1]);
      if constexpr (kF64) {
#pragma unroll
        for (int r = 0; r < R; ++r) yv[r] = __double2float_rn(dadd((double)yv[r], dmul((double)q[r * STRIDE], coef)));
      } else {
        const float cf = (float)coef;  // exact: the coefficient was a float32
#pragma unroll
        for (int r = 0; r < R; ++r) yv[r] = fadd(yv[r], fmul((float)q[r * STRIDE], cf));
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Planar / strided multichannel FIR: one channel x one tile per CTA.
// Shared memory: [0,16) mbarrier | TIn tile[tile + halo] (16-byte aligned) | int program[]
// ------------------------------------------------------------------------------------------------
template <typename TIn, int MODE, int NT, int R>
__global__ void __launch_bounds__(NT) fir_tile_kernel(const FirParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem_raw);
  TIn* sx = reinterpret_cast<TIn*>(smem_raw + 16);
  const int span = p.tile + p.halo;
  int* sprog = reinterpret_cast<int*>(smem_raw + 16 + (((size_t)span * sizeof(TIn) + 15) & ~(size_t)15));

  const int tid = threadIdx.x;
  const int c = blockIdx.x / p.tiles_per_channel;
  const long long t0 = (long long)(blockIdx.x % p.tiles_per_channel) * p.tile;
  const long long remain = p.frames - t0;
  const int w0 = p.offsets[c];
  const int nprog = p.offsets[c + 1] - w0;
  const TIn* __restrict__ xc = reinterpret_cast<const TIn*>(p.x) + (long long)c * p.x_sc;
  float* __restrict__ yc = p.y + (long long)c * p.y_sc;

  if (nprog == 0) {  // unfiltered channel: copy through (decorrelation.py:399-400)
    const int n = (int)(remain < p.tile ? remain : p.tile);
    for (int i = tid; i < n; i += NT) yc[(t0 + i) * p.y_st] = (float)xc[(t0 + i) * p.x_st];
    return;
  }

  const int nvalid = (int)(remain < span ? remain : span);
  int nbulk = 0;
  if constexpr (!is_f64<TIn>::value) {
    if (p.bulk_ok) {
      nbulk = nvalid & ~3;
      if (tid == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
      }
      __syncthreads();
      if (tid == 0 && nbulk > 0) {
        mbar_expect_tx(bar, (uint32_t)nbulk * 4u);
        bulk_g2s(sx, xc + t0, (uint32_t)nbulk * 4u, bar);
      }
    }
  }
  for (int i = nbulk + tid; i < span; i += NT) sx[i] = (i < nvalid) ? xc[(t0 + i) * p.x_st] : (TIn)0;
  for (int i = tid; i < nprog; i += NT) sprog[i] = p.words[w0 + i];
  __syncthreads();
  if (nbulk > 0) mbar_wait(bar, 0);

  const int warp = tid >> 5, lane = tid & 31;
  constexpr int kWarps = NT / 32;
  constexpr int kSub = 32 * R;
  const int nsub = p.tile / kSub;
  for (int sb = warp; sb < nsub; sb += kWarps) {
    const int base = sb * kSub;
    if (base >= remain) break;
    float yv[R];
    run_program<TIn, MODE, R, 32>(sx + base + lane, sprog, p.apply_gain, yv);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const long long t = t0 + base + lane + 32 * r;
      if (t < p.frames) yc[t * p.y_st] = yv[r];
    }
  }
}

// Fallback for filters whose halo does not fit in shared memory: gather straight from global
// memory (L2 serves the reuse).  Same arithmetic, one output per thread-iteration.
template <typename TIn, int MODE>
__global__ void __launch_bounds__(256) fir_direct_kernel(const FirParams p) {
  const int c = blockIdx.y;
  const int w0 = p.offsets[c];
  const int nprog = p.offsets[c + 1] - w0;
  const TIn* __restrict__ xc = reinterpret_cast<const TIn*>(p.x) + (long long)c * p.x_sc;
  float* __restrict__ yc = p.y + (long long)c * p.y_sc;
  const int* __restrict__ prog = p.words + w0;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < p.frames; t += (long long)gridDim.x * blockDim.x) {
    if (nprog == 0) {
      yc[t * p.y_st] = (float)xc[t * p.x_st];
      continue;
    }
    float y = 0.0f;
    if constexpr (MODE == MODE_SEG) {
      const int S = prog[0];
      const int* seg = prog + 1;
      const int* tp = prog + 1 + 3 * S;
      for (int s = 0; s < S; ++s) {
        const int n_neg = seg[3 * s], n_pos = seg[3 * s + 1];
        float acc = 0.0f;
        for (int k = 0; k < n_neg; ++k) {
          const long long u = t + tp[k];
          acc = step_sub<TIn>(acc, u < p.frames ? xc[u * p.x_st] : (TIn)0);
        }
        tp += n_neg;
        for (int k = 0; k < n_pos; ++k) {
          const long long u = t + tp[k];
          acc = step_add<TIn>(acc, u < p.frames ? xc[u * p.x_st] : (TIn)0);
        }
        tp += n_pos;
        if (p.apply_gain) acc = fmul(acc, __int_as_float(seg[3 * s + 2]));
        y = fadd(y, acc);
      }
    } else {
      constexpr bool kF64 = is_f64<TIn>::value || MODE == MODE_ASC64;
      const int K = prog[0];
      const int* e = prog + 1;
      for (int k = 0; k < K; ++k) {
        const long long u = t + e[3 * k];
        const TIn xv = u < p.frames ? xc[u * p.x_st] : (TIn)0;
        const double coef = __hiloint2double(e[3 * k + 2], e[3 * k + 1]);
        if constexpr (kF64) y = __double2float_rn(dadd((double)y, dmul((double)xv, coef)));
        else y = fadd(y, fmul((float)xv, (float)coef));
      }
    }
    yc[t * p.y_st] = y;
  }
}

// ------------------------------------------------------------------------------------------------
// Fused stereo decorrelate: FIR on both channels of a frame, then M/S encode, width, gain and the
// Haas placement, one read of x and one write of out per sample.
// Shared memory: float x0[tile + halo] | float x1[tile + halo] | int prog0[] | int prog1[]
// ------------------------------------------------------------------------------------------------
struct StereoParams {
  const float* x;
  long long x_st, x_sc;
  void* out;
  long long o_st, o_sc;
  long long frames;
  const int* words;
  const int* offsets;  // 3 entries
  int tile, halo;
  int apply_gain;
  int ms_encode, use_width;
  float w_mid, w_side;  // float32(1 - width), float32(width)
  const float* gains;   // nullable, 2 floats
  int delay, delay_ch;
};

__device__ __forceinline__ void stereo_epilogue(float x0, float x1, float& y0, float& y1, const StereoParams& p, float g0, float g1) {
  ms_width_epilogue(x0, x1, y0, y1, p.ms_encode, p.use_width, p.w_mid, p.w_side);
  if (p.gains) {
    y0 = fmul(y0, g0);
    y1 = fmul(y1, g1);
  }
}

template <typename TOut, int R>
__global__ void __launch_bounds__(256) vn_stereo_kernel(const StereoParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int NT = 256;
  const int span = p.tile + p.halo;
  const int span_al = (span + 3) & ~3;
  float* s0 = reinterpret_cast<float*>(smem_raw);
  float* s1 = s0 + span_al;
  int* prog0 = reinterpret_cast<int*>(s1 + span_al);
  const int n0 = p.offsets[1] - p.offsets[0];
  const int n1 = p.offsets[2] - p.offsets[1];
  int* prog1 = prog0 + n0;

  const int tid = threadIdx.x;
  const long long t0 = (long long)blockIdx.x * p.tile;
  const long long remain = p.frames - t0;
  const int nvalid = (int)(remain < span ? remain : span);
  const float* __restrict__ x = p.x;
  for (int i = tid; i < span; i += NT) {
    float a = 0.0f, b = 0.0f;
    if (i < nvalid) {
      a = x[(t0 + i) * p.x_st];
      b = x[(t0 + i) * p.x_st + p.x_sc];
    }
    s0[i] = a;
    s1[i] = b;
  }
  for (int i = tid; i < n0 + n1; i += NT) prog0[i] = p.words[p.offsets[0] + i];
  __syncthreads();

  TOut* __restrict__ out = reinterpret_cast<TOut*>(p.out);
  const int sh0 = p.delay_ch == 0 ? p.delay : 0;
  const int sh1 = p.delay_ch == 1 ? p.delay : 0;
  float g0 = 1.0f, g1 = 1.0f;
  if (p.gains) {
    g0 = p.gains[0];
    g1 = p.gains[1];
  }
  const int warp = tid >> 5, lane = tid & 31;
  constexpr int kSub = 32 * R;
  const int nsub = p.tile / kSub;
  for (int sb = warp; sb < nsub; sb += NT / 32) {
    const int base = sb * kSub;
    if (base >= remain) break;
    float y0[R], y1[R];
    if (n0 > 0) run_program<float, MODE_SEG, R, 32>(s0 + base + lane, prog0, p.apply_gain, y0);
    if (n1 > 0) run_program<float, MODE_SEG, R, 32>(s1 + base + lane, prog1, p.apply_gain, y1);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int i = base + lane + 32 * r;
      const long long t = t0 + i;
      if (t < p.frames) {
        const float a = s0[i], b = s1[i];
        float u = n0 > 0 ? y0[r] : a;  // unfiltered channel: copied through
        float v = n1 > 0 ? y1[r] : b;
        stereo_epilogue(a, b, u, v, p, g0, g1);
        out[(t + sh0) * p.o_st] = (TOut)u;
        out[(t + sh1) * p.o_st + p.o_sc] = (TOut)v;
      }
    }
  }
  // Haas zero fill: head of the delayed channel, tail of the other one (decorrelation.py:206-222)
  if (p.delay > 0) {
    if (blockIdx.x == 0) {
      for (int i = tid; i < p.delay; i += NT) out[(long long)i * p.o_st + (long long)p.delay_ch * p.o_sc] = (TOut)0;
    }
    if (blockIdx.x == gridDim.x - 1) {
      for (int i = tid; i < p.delay; i += NT) out[(p.frames + i) * p.o_st + (long long)(1 - p.delay_ch) * p.o_sc] = (TOut)0;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Batched fused stereo decorrelate: vn_stereo_kernel's work over the (clip, tile) pairs of many clips packed in one
// (rows, 2) float32 array (batch_clip_of maps CTAs to pairs).  Each CTA stages its tile plus the halo of both channels
// and the two program blocks of its clip's filter; staged samples past the clip's end are +0, as in the single-clip
// kernel, so no tap reads across a clip boundary.  out is (rows + n delay, 2) C-order with clip i from row
// offs[i] + i delay, and gets the Haas head and tail zero fill of every clip.
// ------------------------------------------------------------------------------------------------
struct BatchStereoParams {
  StereoParams sp;        // x, out (C-order pairs), words, offsets (2 channels per program), tile, halo, epilogue, delay
  const long long* offs;  // n + 1 clip offsets into x
  const int* prog_of;     // program of each clip: channels 2 k, 2 k + 1 of sp.offsets
  unsigned* arrivals;     // nullable: per-clip counters of the sums pass, zeroed here
  int n_clips;
};

template <typename TOut, int R>
__global__ void __launch_bounds__(256) vn_batch_stereo_kernel(const BatchStereoParams bp) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int NT = 256;
  const StereoParams& p = bp.sp;
  const int span = p.tile + p.halo;
  const int span_al = (span + 3) & ~3;
  float* s0 = reinterpret_cast<float*>(smem_raw);
  float* s1 = s0 + span_al;
  int* prog0 = reinterpret_cast<int*>(s1 + span_al);

  const int clip = batch_clip_of(bp.offs, bp.n_clips, p.tile, blockIdx.x);
  const long long c0 = bp.offs[clip];
  const long long L = bp.offs[clip + 1] - c0;
  const long long k = (long long)blockIdx.x - (c0 / p.tile + clip);
  const long long ntiles = L > 0 ? ceil_div<long long>(L, p.tile) : 1;
  if (k < 0 || k >= ntiles) return;
  if (bp.arrivals && k == 0 && threadIdx.x == 0) bp.arrivals[clip] = 0u;
  const int pr = bp.prog_of[clip];
  const int w0 = p.offsets[2 * pr];
  const int n0 = p.offsets[2 * pr + 1] - w0;
  const int n1 = p.offsets[2 * pr + 2] - w0 - n0;
  int* prog1 = prog0 + n0;

  const int tid = threadIdx.x;
  const long long t0 = k * p.tile;
  const long long remain = L - t0;
  const int nvalid = (int)(remain < span ? (remain > 0 ? remain : 0) : span);
  const float2* __restrict__ x2 = reinterpret_cast<const float2*>(p.x) + c0 + t0;
  for (int i = tid; i < span; i += NT) {
    float2 v = make_float2(0.0f, 0.0f);
    if (i < nvalid) v = x2[i];
    s0[i] = v.x;
    s1[i] = v.y;
  }
  for (int i = tid; i < n0 + n1; i += NT) prog0[i] = p.words[w0 + i];
  __syncthreads();

  TOut* __restrict__ out = reinterpret_cast<TOut*>(p.out) + 2 * (c0 + (long long)clip * p.delay);
  const int sh0 = p.delay_ch == 0 ? p.delay : 0;
  const int sh1 = p.delay_ch == 1 ? p.delay : 0;
  const int warp = tid >> 5, lane = tid & 31;
  constexpr int kSub = 32 * R;
  const int nsub = p.tile / kSub;
  for (int sb = warp; sb < nsub; sb += NT / 32) {
    const int base = sb * kSub;
    if (base >= remain) break;
    float y0[R], y1[R];
    if (n0 > 0) run_program<float, MODE_SEG, R, 32>(s0 + base + lane, prog0, p.apply_gain, y0);
    if (n1 > 0) run_program<float, MODE_SEG, R, 32>(s1 + base + lane, prog1, p.apply_gain, y1);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int i = base + lane + 32 * r;
      const long long t = t0 + i;
      if (t < L) {
        const float a = s0[i], b = s1[i];
        float u = n0 > 0 ? y0[r] : a;  // unfiltered channel: copied through
        float v = n1 > 0 ? y1[r] : b;
        stereo_epilogue(a, b, u, v, p, 1.0f, 1.0f);
        out[(t + sh0) * 2] = (TOut)u;
        out[(t + sh1) * 2 + 1] = (TOut)v;
      }
    }
  }
  if (p.delay > 0) {  // Haas zero fill of this clip: head of the delayed channel, tail of the other one
    if (k == 0)
      for (int i = tid; i < p.delay; i += NT) out[(long long)i * 2 + p.delay_ch] = (TOut)0;
    if (k == ntiles - 1)
      for (int i = tid; i < p.delay; i += NT) out[(L + i) * 2 + (1 - p.delay_ch)] = (TOut)0;
  }
}

// ------------------------------------------------------------------------------------------------
// One velvet-noise step of many live signals (vnd_vn_block_step_dev): vn_batch_stereo_kernel's work on each signal's
// ready frames [E0, E0 + count), E0 = emitted[sig].  The CTA stages its tile plus the halo of the signal's virtual
// input (history, then block, then +0: block_step_frame), so every output frame reads exactly the samples the one-shot
// call reads, and +0 where the one-shot call drops a tap past the end.  Same tap loop and epilogue, float32 out.
// ------------------------------------------------------------------------------------------------
template <int R>
__global__ void __launch_bounds__(256) vn_block_step_kernel(const StereoParams p, const BlockStepParams b, const int* prog_of) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int NT = 256;
  constexpr int kSub = 32 * R;
  if (blockIdx.x >= b.out_blocks) {
    block_step_history(b, (long long)blockIdx.x - b.out_blocks);
    return;
  }
  const int span_al = (p.tile + p.halo + 3) & ~3;
  float* s0 = reinterpret_cast<float*>(smem_raw);
  float* s1 = s0 + span_al;
  int* prog0 = reinterpret_cast<int*>(s1 + span_al);

  const int sig = batch_clip_of(b.out_offs, b.n, p.tile, blockIdx.x);
  const long long o0 = b.out_offs[sig];
  const long long cnt = b.out_offs[sig + 1] - o0;
  const long long k = (long long)blockIdx.x - (o0 / p.tile + sig);
  if (k < 0 || k * p.tile >= cnt) return;
  const int nout = (int)(cnt - k * p.tile < p.tile ? cnt - k * p.tile : p.tile);
  const int pr = prog_of[sig];
  const int w0 = p.offsets[2 * pr];
  const int n0 = p.offsets[2 * pr + 1] - w0;
  const int n1 = p.offsets[2 * pr + 2] - w0 - n0;
  int* prog1 = prog0 + n0;

  const int tid = threadIdx.x;
  const long long T0 = b.received[sig], x0 = b.offs[sig];
  const long long T1 = T0 + (b.offs[sig + 1] - x0);
  const long long t0 = b.emitted[sig] + k * p.tile;  // first output frame of the tile
  const int nstage = (nout + kSub - 1) / kSub * kSub + p.halo;  // what the warps below read
  for (int i = tid; i < nstage; i += NT) {
    const float2 v = block_step_frame(b, sig, t0 + i, T0, T1, x0);
    s0[i] = v.x;
    s1[i] = v.y;
  }
  for (int i = tid; i < n0 + n1; i += NT) prog0[i] = p.words[w0 + i];
  __syncthreads();

  float2* __restrict__ out = reinterpret_cast<float2*>(p.out) + o0 + k * p.tile;
  const int warp = tid >> 5, lane = tid & 31;
  for (int base = warp * kSub; base < nout; base += NT / 32 * kSub) {
    float y0[R], y1[R];
    if (n0 > 0) run_program<float, MODE_SEG, R, 32>(s0 + base + lane, prog0, p.apply_gain, y0);
    if (n1 > 0) run_program<float, MODE_SEG, R, 32>(s1 + base + lane, prog1, p.apply_gain, y1);
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int i = base + lane + 32 * r;
      if (i < nout) {
        const float a = s0[i], c = s1[i];
        float u = n0 > 0 ? y0[r] : a;  // unfiltered channel: copied through
        float v = n1 > 0 ? y1[r] : c;
        stereo_epilogue(a, c, u, v, p, 1.0f, 1.0f);
        out[i] = make_float2(u, v);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// One convolve step of many live multichannel signals (vnd_fir_block_step_dev): VelvetNoise.convolve on each signal's
// ready frames [E0, E0 + count) of its C channels, E0 = emitted[sig], in the compute dtype TIn (float or double) of the
// one-shot call.  A CTA owns (signal, group of G = 2^lg consecutive channels, output tile).  It reads the signal's
// virtual input (history, then block, then +0) along the C-order rows, G values per row, and transposes it into one
// shared-memory row per channel; the unchanged run_program tap loop then runs with the channel's program (program k is
// channels [k C, (k + 1) C)); the results go back through shared memory and are stored G values per row.
//
// Bit contract: output frame t is byte-identical to frame t of vnd_sparse_fir_dev on the signal's first T frames, for
// any T it can be computed from (t + halo - 1 < T1, or T = T1 at a final step).  The frames read are the same, and a
// tap the one-shot call drops (its index >= T, or t + index >= T) reads +0 here.  In SEGMENTED order that cannot change
// the bits: a +0 tap leaves a segment's acc unchanged, except that it can turn a -0 acc into +0 (a float64 step can
// round acc to -0); then y + acc is the same either way, because y is never -0: it starts at +0, and a round-to-nearest
// sum that lands on zero is +0.  A segment the one-shot program drops because all its taps are dropped adds +-0 to y,
// which again leaves y unchanged.  That is why taps past the end may be staged as zeros.
//
// kGather = false: the CTA stages its tile plus the halo of G channels (G (tile + halo) values) and its G programs in
// shared memory.  kGather = true, for filters whose halo does not fit: every tap is read from global memory (L1 / L2
// serve the reuse, as in fir_direct_kernel) and the programs with it; only the output transpose is in shared memory.
// ------------------------------------------------------------------------------------------------
struct FirBlockParams {
  float* out;           // (out_rows, C)
  const int* words;
  const int* offsets;   // C entries per program, and one more
  const int* prog_of;   // n
  int apply_gain;
  int halo;             // frames each tile reads past its last output, a multiple of 4
  int span;             // shared-memory row of one channel: tile + halo, odd (staging path)
  int tile;             // output frames per CTA, a multiple of 32 R
  int lg;               // log2 of the channel group G
  int groups;           // ceil(C / G)
};

// Elements of history per CTA of the convolve step's history pass.
constexpr int kFirHistChunk = 16384;

// Value (frame f, channel c) of signal `sig`'s virtual input, +0 where it has no frame.
template <typename TIn>
__device__ __forceinline__ TIn fir_block_value(const BlockStepParams& b, int sig, long long f, int c, long long T0, long long T1, long long x0) {
  if (f >= T0) return f < T1 ? __ldg(reinterpret_cast<const TIn*>(b.x) + (x0 + (f - T0)) * b.C + c) : (TIn)0;
  if (f < 0 || f < T0 - b.H) return (TIn)0;
  return __ldg(reinterpret_cast<const TIn*>(b.hist_in) + ((long long)sig * b.H + (f - (T0 - b.H))) * b.C + c);
}

// History CTA j: elements [lo, hi) of signal j / hchunks's new history, H x C values, chunk j % hchunks.  Value e of it is
// value v = (T1 - H) C + e of the virtual input in C-order, so each source is one contiguous run.
template <typename TIn>
__device__ __forceinline__ void fir_block_history(const BlockStepParams& b, long long j) {
  const int sig = (int)(j / b.hchunks);
  const long long HC = (long long)b.H * b.C;
  const long long lo = (j % b.hchunks) * kFirHistChunk;
  const long long hi = lo + kFirHistChunk < HC ? lo + kFirHistChunk : HC;
  const long long T0 = b.received[sig], x0 = b.offs[sig];
  const long long T1 = T0 + (b.offs[sig + 1] - x0);
  const long long v0 = (T1 - b.H) * b.C, vx = T0 * b.C, vh = (T0 - b.H) * b.C;
  const TIn* __restrict__ xs = reinterpret_cast<const TIn*>(b.x) + x0 * b.C;
  const TIn* __restrict__ hin = reinterpret_cast<const TIn*>(b.hist_in) + sig * HC;
  TIn* __restrict__ hout = reinterpret_cast<TIn*>(b.hist_out) + sig * HC;
  for (long long e = lo + threadIdx.x; e < hi; e += blockDim.x) {
    const long long v = v0 + e;
    hout[e] = v >= vx ? __ldg(xs + (v - vx)) : (v >= 0 ? __ldg(hin + (v - vh)) : (TIn)0);
  }
}

template <typename TIn, bool kGather, int R>
__global__ void __launch_bounds__(256) fir_block_step_kernel(const FirBlockParams p, const BlockStepParams b) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int NT = 256;
  constexpr int kSub = 32 * R;
  if (blockIdx.x >= b.out_blocks) {
    fir_block_history<TIn>(b, (long long)blockIdx.x - b.out_blocks);
    return;
  }
  const int G = 1 << p.lg;
  const long long cta = blockIdx.x / p.groups;
  const int c0 = (int)(blockIdx.x % p.groups) << p.lg;
  const int gc = b.C - c0 < G ? b.C - c0 : G;
  const int sig = batch_clip_of(b.out_offs, b.n, p.tile, cta);
  const long long o0 = b.out_offs[sig];
  const long long cnt = b.out_offs[sig + 1] - o0;
  const long long k = cta - (o0 / p.tile + sig);
  if (k < 0 || k * p.tile >= cnt) return;
  const int nout = (int)(cnt - k * p.tile < p.tile ? cnt - k * p.tile : p.tile);
  const int* offs = p.offsets + (long long)p.prog_of[sig] * b.C + c0;  // the group's gc programs are contiguous
  const int w0 = offs[0];

  // shared memory: [TIn sx[G][span] | float sy[tile][G + 1] | int sprog[]] (staging path), [float sy | ] (gather path)
  TIn* sx = reinterpret_cast<TIn*>(smem_raw);
  float* sy = kGather ? reinterpret_cast<float*>(smem_raw) : reinterpret_cast<float*>(sx + (size_t)G * p.span);
  int* sprog = reinterpret_cast<int*>(sy + (size_t)p.tile * (G + 1));
  const int* prog = kGather ? p.words + w0 : sprog;

  const int tid = threadIdx.x;
  const long long T0 = b.received[sig], x0 = b.offs[sig];
  const long long T1 = T0 + (b.offs[sig + 1] - x0);
  const long long t0 = b.emitted[sig] + k * p.tile;  // first output frame of the tile
  const int nsub = (nout + kSub - 1) / kSub;
  if constexpr (!kGather) {
    const int nstage = nsub * kSub + p.halo;  // what the warps below read
    for (int e = tid; e < (nstage << p.lg); e += NT) {
      const int i = e >> p.lg, g = e & (G - 1);
      if (g < gc) sx[g * p.span + i] = fir_block_value<TIn>(b, sig, t0 + i, c0 + g, T0, T1, x0);
    }
    const int nw = offs[gc] - w0;
    for (int i = tid; i < nw; i += NT) sprog[i] = p.words[w0 + i];
    __syncthreads();
  }

  const int warp = tid >> 5, lane = tid & 31;
  if constexpr (!kGather) {
    for (int u = warp; u < nsub * gc; u += NT / 32) {
      const int g = u % gc, base = (u / gc) * kSub;
      const int pw = offs[g] - w0, pn = offs[g + 1] - offs[g];
      const TIn* px = sx + g * p.span + base + lane;
      float y[R];
      if (pn > 0) {
        run_program<TIn, MODE_SEG, R, 32>(px, prog + pw, p.apply_gain, y);
      } else {  // unfiltered channel: copied through (decorrelation.py:399-400)
#pragma unroll
        for (int r = 0; r < R; ++r) y[r] = (float)px[32 * r];
      }
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const int i = base + lane + 32 * r;
        if (i < nout) sy[i * (G + 1) + g] = y[r];
      }
    }
  } else {
    const int n32 = (nout + 31) >> 5;
    for (int u = warp; u < n32 * gc; u += NT / 32) {
      const int g = u % gc, i = (u / gc) * 32 + lane;
      if (i >= nout) continue;
      const int* pg = prog + (offs[g] - w0);
      const long long t = t0 + i;
      // the channel's virtual input at frame t + d: block from d >= dx, history from d >= dh, +0 elsewhere
      const long long C = b.C, dx = T0 - t, dend = T1 - t, dh = (T0 - b.H > 0 ? T0 - b.H : 0) - t;
      const TIn* xb = reinterpret_cast<const TIn*>(b.x) + (x0 - dx) * C + c0 + g;
      const TIn* hb = reinterpret_cast<const TIn*>(b.hist_in) + ((long long)sig * b.H - (T0 - b.H) + t) * C + c0 + g;
      auto at = [&](int d) -> TIn { return d >= dx ? (d < dend ? __ldg(xb + d * C) : (TIn)0) : (d >= dh ? __ldg(hb + d * C) : (TIn)0); };
      float y = 0.0f;
      if (offs[g + 1] == offs[g]) {
        y = (float)at(0);
      } else {  // fir_direct_kernel's SEGMENTED loop on the virtual input
        const int S = pg[0];
        const int* seg = pg + 1;
        const int* tp = pg + 1 + 3 * S;
        for (int s = 0; s < S; ++s) {
          const int n_neg = seg[3 * s], n_pos = seg[3 * s + 1];
          float acc = 0.0f;
          for (int q = 0; q < n_neg; ++q) acc = step_sub<TIn>(acc, at(tp[q]));
          tp += n_neg;
          for (int q = 0; q < n_pos; ++q) acc = step_add<TIn>(acc, at(tp[q]));
          tp += n_pos;
          if (p.apply_gain) acc = fmul(acc, __int_as_float(seg[3 * s + 2]));
          y = fadd(y, acc);
        }
      }
      sy[i * (G + 1) + g] = y;
    }
  }
  __syncthreads();

  float* __restrict__ out = p.out + (o0 + k * p.tile) * b.C + c0;
  for (int e = tid; e < (nout << p.lg); e += NT) {
    const int i = e >> p.lg, g = e & (G - 1);
    if (g < gc) out[(long long)i * b.C + g] = sy[i * (G + 1) + g];
  }
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
constexpr int kR = 8;
// VND_DISABLE_WINDOW=1 in the environment forces the general tile kernel (A/B runs and tests).
static const bool g_disable_window = [] {
  const char* e = getenv("VND_DISABLE_WINDOW");
  return e && e[0] == '1';
}();

// VND_DISABLE_TMEM=1 skips the tensor-memory kernel (A/B runs and tests).
static const bool g_disable_tmem = [] {
  const char* e = getenv("VND_DISABLE_TMEM");
  return e && e[0] == '1';
}();

template <typename TIn, int MODE, int NT>
static int launch_tile(const FirParams& p, size_t smem, cudaStream_t st) {
  auto k = fir_tile_kernel<TIn, MODE, NT, kR>;
  VND_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long blocks = (long long)p.tiles_per_channel * p.channels;
  VND_REQUIRE(blocks < 0x7fffffffLL, VND_EUNSUPPORTED, "grid too large (%lld CTAs)", blocks);
  k<<<(unsigned)blocks, NT, smem, st>>>(p);
  return after_launch("fir_tile_kernel");
}

template <typename TIn, int MODE>
static int launch_tile_nt(const FirParams& p, size_t smem, int nt, cudaStream_t st) {
  switch (nt) {
    case 256: return launch_tile<TIn, MODE, 256>(p, smem, st);
    case 512: return launch_tile<TIn, MODE, 512>(p, smem, st);
    default: return launch_tile<TIn, MODE, 1024>(p, smem, st);
  }
}

// Long filters (halo beyond 4096 samples, e.g. 300 impulses over 0.3 s @ 96 kHz: BASELINE config 4): tile + halo
// fills the SM's shared memory, so ONE CTA of 32 warps runs per SM.  kLongR outputs per lane and pass; the tile is a whole
// number of passes for all 32 warps (round 1 ran 28 672 outputs = 3.5 passes of R = 8: half of the warps idled
// through the fourth pass), and a larger R spreads the tap-index load and the loop overhead of a tap over more outputs.
// Measured on 64 channels x 57.6 M frames (B200, Gsamples/s, shared-memory pipe busy): round 1 (R = 8, 3.5 passes, scalar
// adds) 25.1 / 81 %; R = 8 25.3 / 81 %; R = 12 26.0 / 84 %; R = 16 (one pass of 16 384 outputs) 27.5 / 89 %.  The other
// values of R were removed; last present at commit 915ac5a.
constexpr int kLongR = 16;
static int plan_long_tile(int halo, int max_prog_words, size_t* smem) {
  const long long budget = (long long)kMaxDynSmem - 16 - 16 - (long long)max_prog_words * 4;
  const long long per_pass = 32LL * 32 * kLongR;
  const long long tile = (budget / 4 - halo) / per_pass * per_pass;
  if (tile <= 0) return 0;
  *smem = 16 + (((size_t)(tile + halo) * 4 + 15) & ~(size_t)15) + (size_t)max_prog_words * 4;
  return (int)tile;
}
static int launch_long_tile(const FirParams& p, size_t smem, cudaStream_t st) {
  auto k = fir_tile_kernel<float, MODE_SEG, 1024, kLongR>;
  VND_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const long long blocks = (long long)p.tiles_per_channel * p.channels;
  VND_REQUIRE(blocks < 0x7fffffffLL, VND_EUNSUPPORTED, "grid too large (%lld CTAs)", blocks);
  k<<<(unsigned)blocks, 1024, smem, st>>>(p);
  return after_launch("fir_tile_kernel");
}

template <typename TIn, int MODE>
static int launch_direct(const FirParams& p, cudaStream_t st) {
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  long long bx = ceil_div<long long>(p.frames, 256);
  const long long cap = (long long)di.sm_count * 16;
  if (bx > cap) bx = cap;
  if (bx < 1) bx = 1;
  VND_REQUIRE(p.channels <= 65535, VND_EUNSUPPORTED, "direct FIR path supports at most 65535 channels");
  dim3 grid((unsigned)bx, (unsigned)p.channels);
  fir_direct_kernel<TIn, MODE><<<grid, 256, 0, st>>>(p);
  return after_launch("fir_direct_kernel");
}

// Picks the tile for a given halo so that tile + halo fits in shared memory; returns 0 when the
// halo itself does not fit (caller falls back to the direct kernel).
static int plan_tile(int halo, int elem, int max_prog_words, long long frames, int* nt, size_t* smem) {
  const long long budget = (long long)kMaxDynSmem - 16 - 16 - (long long)max_prog_words * 4;
  const long long span_max = budget / elem;
  constexpr int unit = 32 * kR;  // outputs per warp pass
  long long tile = 8192;
  if (halo > 4096) tile = ((long long)halo + 2047) / 2048 * 2048;  // keep the re-read of the halo <= 2x
  if (tile + halo > span_max) tile = (span_max - halo) / unit * unit;
  if (tile < unit) return 0;
  // no point in a tile longer than the signal
  const long long need = ceil_div<long long>(frames, unit) * unit;
  if (tile > need) tile = need;
  *smem = 16 + (((size_t)(tile + halo) * elem + 15) & ~(size_t)15) + (size_t)max_prog_words * 4;
  const int ctas_per_sm = (int)((228 * 1024) / (*smem + 1024));
  *nt = ctas_per_sm >= 4 ? 256 : (ctas_per_sm >= 2 ? 512 : 1024);
  // small tiles cannot feed many warps
  while (*nt > 256 && tile / unit < *nt / 32) *nt /= 2;
  return (int)tile;
}

int sparse_fir_launch(const vnd_signal* x, const vnd_signal* y, const vnd_tap_program* taps, int max_prog_words,
                      cudaStream_t st) {
  FirParams p{};
  p.x = x->data;
  p.x_st = x->stride_t;
  p.x_sc = x->stride_c;
  p.y = reinterpret_cast<float*>(y->data);
  p.y_st = y->stride_t;
  p.y_sc = y->stride_c;
  p.frames = x->frames;
  p.channels = taps->channels;
  p.words = taps->words;
  p.offsets = taps->offsets;
  p.apply_gain = taps->apply_gain;
  p.halo = taps->halo > 0 ? taps->halo : 0;
  if (p.frames == 0 || p.channels == 0) return VND_OK;
  const bool f64 = x->dtype == VND_F64;
  const int elem = f64 ? 8 : 4;
  int nt = 256;
  size_t smem = 0;
  // the halo never needs to reach past the end of the signal
  if (p.halo > p.frames) p.halo = (int)p.frames;
  p.halo = (p.halo + 3) & ~3;
  const int mode = taps->order == VND_ORDER_SEGMENTED ? MODE_SEG : (taps->order == VND_ORDER_ASCENDING ? MODE_ASC32 : MODE_ASC64);
  p.bulk_ok = (!f64 && x->stride_t == 1 && (x->stride_c % 4) == 0 && (reinterpret_cast<uintptr_t>(x->data) % 16) == 0) ? 1 : 0;
  if (!f64 && mode == MODE_SEG && !g_disable_tmem) {  // throughput path for long planar float32 slabs
    long long done = 0;
    const int rc = fir_tmem_launch(p, max_prog_words, st, &done);
    if (rc != VND_OK && rc != VND_EUNSUPPORTED) return rc;
    if (rc == VND_OK && done > 0) {  // the tail of every channel goes through the kernels below
      p.x = reinterpret_cast<const float*>(p.x) + done;
      p.y += done;
      p.frames -= done;
      if (p.frames == 0) return VND_OK;
      if (p.halo > p.frames) p.halo = (int)((p.frames + 3) & ~3LL);
      p.bulk_ok = (p.bulk_ok && (reinterpret_cast<uintptr_t>(p.x) % 16) == 0) ? 1 : 0;
    }
  }
  if (!f64 && mode == MODE_SEG && !g_disable_window) {  // planar float32 slabs too short for the above
    const int rc = fir_window_launch(p, max_prog_words, st);
    if (rc != VND_EUNSUPPORTED) return rc;
  }
  if (!f64 && mode == MODE_SEG && p.halo > 4096 && p.frames >= 4LL * p.halo) {  // long filters on long signals
    {  // the interior of every channel through the ring-buffer kernel (vnd_fir_ring.cu), the tail through the tile kernels below
      long long done = 0;
      const int rc = fir_ring_launch(p, max_prog_words, st, &done);
      if (rc != VND_OK && rc != VND_EUNSUPPORTED) return rc;
      if (rc == VND_OK && done > 0) {
        p.x = reinterpret_cast<const float*>(p.x) + done;
        p.y += done;
        p.frames -= done;
        if (p.frames == 0) return VND_OK;
        if (p.halo > p.frames) p.halo = (int)((p.frames + 3) & ~3LL);
        p.bulk_ok = (p.bulk_ok && (reinterpret_cast<uintptr_t>(p.x) % 16) == 0) ? 1 : 0;
      }
    }
  }
  if (!f64 && mode == MODE_SEG && p.halo > 4096 && p.frames >= 4LL * p.halo) {
    const int tile = plan_long_tile(p.halo, max_prog_words, &smem);
    if (tile > 0) {
      p.tile = tile;
      p.tiles_per_channel = (int)ceil_div<long long>(p.frames, p.tile);
      return launch_long_tile(p, smem, st);
    }
  }
  p.tile = plan_tile(p.halo, elem, max_prog_words, p.frames, &nt, &smem);
  if (p.tile == 0) {
    if (f64) {
      if (mode == MODE_SEG) return launch_direct<double, MODE_SEG>(p, st);
      return launch_direct<double, MODE_ASC64>(p, st);
    }
    if (mode == MODE_SEG) return launch_direct<float, MODE_SEG>(p, st);
    if (mode == MODE_ASC32) return launch_direct<float, MODE_ASC32>(p, st);
    return launch_direct<float, MODE_ASC64>(p, st);
  }
  p.tiles_per_channel = (int)ceil_div<long long>(p.frames, p.tile);
  if (f64) {
    if (mode == MODE_SEG) return launch_tile_nt<double, MODE_SEG>(p, smem, nt, st);
    return launch_tile_nt<double, MODE_ASC64>(p, smem, nt, st);
  }
  if (mode == MODE_SEG) return launch_tile_nt<float, MODE_SEG>(p, smem, nt, st);
  if (mode == MODE_ASC32) return launch_tile_nt<float, MODE_ASC32>(p, smem, nt, st);
  return launch_tile_nt<float, MODE_ASC64>(p, smem, nt, st);
}

// Returns VND_EUNSUPPORTED (without setting an error) when the fused kernel cannot hold the halo;
// the caller then composes the unfused kernels.
int vn_stereo_launch(const vnd_signal* x, void* out, int out_dtype, long long o_st, long long o_sc, const vnd_tap_program* taps,
                     int prog_words, const vnd_epilogue* ep, const float* gains, int delay, int delay_ch, cudaStream_t st) {
  StereoParams p{};
  p.x = reinterpret_cast<const float*>(x->data);
  p.x_st = x->stride_t;
  p.x_sc = x->stride_c;
  p.out = out;
  p.o_st = o_st;
  p.o_sc = o_sc;
  p.frames = x->frames;
  p.words = taps->words;
  p.offsets = taps->offsets;
  p.apply_gain = taps->apply_gain;
  p.ms_encode = ep->ms_encode;
  p.use_width = ep->use_width;
  p.w_mid = (float)(1.0 - (double)ep->width);
  p.w_side = (float)ep->width;
  p.gains = gains;
  p.delay = delay;
  p.delay_ch = delay_ch;
  int halo = taps->halo > 0 ? taps->halo : 0;
  if (halo > p.frames) halo = (int)p.frames;
  p.halo = (halo + 3) & ~3;
  constexpr int R = 4;
  constexpr int unit = 32 * R;
  long long tile = 1024;
  const long long need = ceil_div<long long>(p.frames, unit) * unit;
  if (tile > need) tile = need;
  size_t smem = (size_t)2 * (((size_t)tile + p.halo + 3) & ~(size_t)3) * 4 + (size_t)prog_words * 4 + 16;
  if (smem > (size_t)kMaxDynSmem) return VND_EUNSUPPORTED;
  p.tile = (int)tile;
  const unsigned blocks = (unsigned)ceil_div<long long>(p.frames, tile);
  if (out_dtype == VND_F64) {
    auto k = vn_stereo_kernel<double, R>;
    VND_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<blocks, 256, smem, st>>>(p);
  } else {
    auto k = vn_stereo_kernel<float, R>;
    VND_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<blocks, 256, smem, st>>>(p);
  }
  return after_launch("vn_stereo_kernel");
}

bool vn_batch_smem(int halo, int prog_words, size_t* smem) {
  const long long h = ((long long)(halo > 0 ? halo : 0) + 3) & ~3LL;
  const long long bytes = 2 * ((kBatchTile + h + 3) & ~3LL) * 4 + (long long)prog_words * 4 + 16;
  *smem = (size_t)bytes;
  return bytes <= kMaxDynSmem;
}

int vn_batch_stereo_launch(const float* x, long long rows, const long long* offs, int n_clips, const int* prog_of,
                           const vnd_tap_program* taps, const vnd_epilogue* ep, void* out, int out_dtype, int delay, int delay_ch,
                           unsigned* arrivals, cudaStream_t st) {
  if (n_clips == 0) return VND_OK;
  BatchStereoParams bp{};
  StereoParams& p = bp.sp;
  p.x = x;
  p.out = out;
  p.words = taps->words;
  p.offsets = taps->offsets;
  p.apply_gain = taps->apply_gain;
  p.ms_encode = ep->ms_encode;
  p.use_width = ep->use_width;
  p.w_mid = (float)(1.0 - (double)ep->width);
  p.w_side = (float)ep->width;
  p.delay = delay;
  p.delay_ch = delay_ch;
  long long halo = taps->halo > 0 ? taps->halo : 0;
  if (halo > rows) halo = rows;  // no clip is longer than the batch
  p.halo = (int)((halo + 3) & ~3LL);
  p.tile = kBatchTile;
  size_t smem = 0;
  if (!vn_batch_smem(p.halo, 2 * taps->max_channel_words, &smem)) return VND_EUNSUPPORTED;
  bp.offs = offs;
  bp.prog_of = prog_of;
  bp.arrivals = arrivals;
  bp.n_clips = n_clips;
  const long long blocks = rows / kBatchTile + n_clips;
  VND_REQUIRE(blocks < 0x7fffffffLL, VND_EUNSUPPORTED, "grid too large (%lld CTAs)", blocks);
  constexpr int R = 4;
  static_assert(kBatchTile % (32 * R * 8) == 0, "the tile is a whole number of passes of the 8 warps");
  if (out_dtype == VND_F64) {
    auto k = vn_batch_stereo_kernel<double, R>;
    VND_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<(unsigned)blocks, 256, smem, st>>>(bp);
  } else {
    auto k = vn_batch_stereo_kernel<float, R>;
    VND_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k<<<(unsigned)blocks, 256, smem, st>>>(bp);
  }
  return after_launch("vn_batch_stereo_kernel");
}

int vn_block_step_launch(BlockStepParams b, long long out_rows, const int* prog_of, const vnd_tap_program* taps, const vnd_epilogue* ep,
                         float* out, cudaStream_t st) {
  StereoParams p{};
  p.out = out;
  p.words = taps->words;
  p.offsets = taps->offsets;
  p.apply_gain = taps->apply_gain;
  p.ms_encode = ep->ms_encode;
  p.use_width = ep->use_width;
  p.w_mid = (float)(1.0 - (double)ep->width);
  p.w_side = (float)ep->width;
  p.halo = ((taps->halo > 0 ? taps->halo : 0) + 3) & ~3;
  p.tile = kBatchTile;
  size_t smem = 0;
  if (!vn_batch_smem(p.halo, 2 * taps->max_channel_words, &smem)) return VND_EUNSUPPORTED;
  long long blocks = 0;
  VND_REQUIRE(block_step_grid(&b, out_rows, kBatchTile, &blocks), VND_EUNSUPPORTED, "grid too large (%lld CTAs)", blocks);
  constexpr int R = 4;
  auto k = vn_block_step_kernel<R>;
  VND_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<(unsigned)blocks, 256, smem, st>>>(p, b, prog_of);
  return after_launch("vn_block_step_kernel");
}

// Output frames per CTA of the convolve step: one 512-frame block per tile, 4 passes of R = 4 for each channel.
constexpr int kFirBlockTile = 512;
// The staging path takes the widest channel group (up to 32, one 128-byte float32 row segment) whose shared memory leaves
// room for a second CTA on the SM; if even one channel does not fit that, one channel alone up to the 227 KB limit; if
// that does not fit either, the gather path.  One channel alone, although its loads and stores are one value per row, beats
// the gather path 4.7 x on 1024 channels with the 0.3 s, 96 kHz filter in float32 (1.50 against 7.08 ms per kernel, B200).
constexpr long long kFirBlockSmemTarget = 113 * 1024;
// The most shared memory the staging path may take (A/B builds: -DVND_FIR_BLOCK_STAGE_MAX=0 sends every filter to the
// gather path).
#ifndef VND_FIR_BLOCK_STAGE_MAX
#define VND_FIR_BLOCK_STAGE_MAX kMaxDynSmem
#endif

template <typename TIn, bool kGather>
static int launch_fir_block(const FirBlockParams& p, const BlockStepParams& b, size_t smem, long long blocks, cudaStream_t st) {
  auto k = fir_block_step_kernel<TIn, kGather, 4>;
  VND_CUDA_OK(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k<<<(unsigned)blocks, 256, smem, st>>>(p, b);
  return after_launch("fir_block_step_kernel");
}

int fir_block_step_launch(BlockStepParams b, long long out_rows, int dtype, const int* prog_of, const vnd_tap_program* taps, float* out,
                          cudaStream_t st) {
  FirBlockParams p{};
  p.out = out;
  p.words = taps->words;
  p.offsets = taps->offsets;
  p.prog_of = prog_of;
  p.apply_gain = taps->apply_gain;
  p.halo = ((taps->halo > 0 ? taps->halo : 0) + 3) & ~3;
  p.tile = kFirBlockTile;
  p.span = (p.tile + p.halo) | 1;  // odd: the G values of one row land in G different banks
  const int elem = dtype == VND_F64 ? 8 : 4;
  int gmax = 0;
  while ((1 << gmax) < 32 && (1 << gmax) < b.C) ++gmax;
  auto bytes = [&](int lg, bool gather) {
    const long long G = 1LL << lg;
    const long long sy = (long long)p.tile * (G + 1) * 4;
    return gather ? sy : G * p.span * elem + sy + G * taps->max_channel_words * 4LL;
  };
  bool gather = false;
  p.lg = gmax;
  while (p.lg > 0 && bytes(p.lg, false) > kFirBlockSmemTarget) --p.lg;
  if (bytes(p.lg, false) > VND_FIR_BLOCK_STAGE_MAX) {
    gather = true;
    p.lg = gmax;
  }
  const size_t smem = (size_t)bytes(p.lg, gather);
  p.groups = (b.C + (1 << p.lg) - 1) >> p.lg;
  b.out_blocks = (out_rows / p.tile + b.n) * p.groups;
  const long long hist = (long long)b.H * b.C;
  b.hchunks = (int)((hist + kFirHistChunk - 1) / kFirHistChunk);
  const long long blocks = b.out_blocks + (long long)b.n * b.hchunks;
  VND_REQUIRE(blocks < 0x7fffffffLL, VND_EUNSUPPORTED, "grid too large (%lld CTAs)", blocks);
  if (dtype == VND_F64) return gather ? launch_fir_block<double, true>(p, b, smem, blocks, st) : launch_fir_block<double, false>(p, b, smem, blocks, st);
  return gather ? launch_fir_block<float, true>(p, b, smem, blocks, st) : launch_fir_block<float, false>(p, b, smem, blocks, st);
}

}  // namespace vnd
