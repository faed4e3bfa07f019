// Post-FIR kernels: numpy-order sum of squares, RMS gains, gain + Haas placement, the standalone
// Haas delay and the in-place stereo helpers.
//
// Reference arithmetic reproduced here:
//   rms_normalize                src/vndecorrelate/utils/dsp.py:87-109
//   HaasEffect.haas_delay        src/vndecorrelate/decorrelation.py:202-230
//   LR_to_MS / MS_to_LR          src/vndecorrelate/utils/dsp.py:124-167
//   apply_stereo_width           src/vndecorrelate/utils/dsp.py:21-37
//   encode_signal_to_side_channel src/vndecorrelate/utils/dsp.py:40-63

#include <cooperative_groups.h>
#include <stdlib.h>

#include "vnd_common.cuh"
#include "vnd_batch.cuh"

namespace vnd {

// ------------------------------------------------------------------------------------------------
// np.mean(np.square(a), axis=0) on a C-order (n, C) array adds row after row into one accumulator
// per column: a strict left-to-right running sum in the array's dtype.  That order loses low bits
// on long signals, and the reference's gains inherit the loss, so it is reproduced: one CTA per
// column, warps 1.. stage the rounded squares of the next chunk in shared memory while lane 0 of
// warp 0 walks the current chunk with a dependent add chain (4 cycles per sample).
// ------------------------------------------------------------------------------------------------
struct SeqParams {
  const void* a;
  long long a_st, a_sc;
  const void* b;  // optional second signal (columns C .. 2C-1)
  long long b_st, b_sc;
  long long frames;
  int channels;
  void* sums;  // T[ncols]
  // float32 column source of seq_sumsq_cluster_kernel
  __device__ __forceinline__ void column(int col, const float** base, long long* st, long long* n) const {
    if (col < channels) {
      *base = reinterpret_cast<const float*>(a) + (long long)col * a_sc;
      *st = a_st;
    } else {
      *base = reinterpret_cast<const float*>(b) + (long long)(col - channels) * b_sc;
      *st = b_st;
    }
    *n = frames;
  }
  __device__ __forceinline__ void store(int col, float s) const { reinterpret_cast<float*>(sums)[col] = s; }
};

template <typename T>
__device__ __forceinline__ T sq(T v);
template <>
__device__ __forceinline__ float sq<float>(float v) { return fmul(v, v); }
template <>
__device__ __forceinline__ double sq<double>(double v) { return dmul(v, v); }
template <typename T>
__device__ __forceinline__ T add_rn(T a, T b);
template <>
__device__ __forceinline__ float add_rn<float>(float a, float b) { return fadd(a, b); }
template <>
__device__ __forceinline__ double add_rn<double>(double a, double b) { return dadd(a, b); }

template <typename T>
__global__ void __launch_bounds__(256) seq_sumsq_kernel(const SeqParams p) {
  constexpr int CHUNK = 16384 / (int)sizeof(T);  // 2 x 16 KB of static shared memory
  constexpr int NT = 256;
  __shared__ __align__(16) T buf[2][CHUNK];
  const int col = blockIdx.x;
  const T* base;
  long long st;
  if (col < p.channels) {
    base = reinterpret_cast<const T*>(p.a) + (long long)col * p.a_sc;
    st = p.a_st;
  } else {
    base = reinterpret_cast<const T*>(p.b) + (long long)(col - p.channels) * p.b_sc;
    st = p.b_st;
  }
  const int tid = threadIdx.x;
  const long long nchunks = ceil_div<long long>(p.frames, CHUNK);
  auto stage = [&](long long k, int slot, int first, int step) {
    const long long off = k * CHUNK;
    for (int i = first; i < CHUNK; i += step) {
      const long long t = off + i;
      buf[slot][i] = t < p.frames ? sq<T>(base[t * st]) : (T)0;  // +0 padding: s + 0 == s
    }
  };
  if (nchunks > 0) stage(0, 0, tid, NT);
  T s = (T)0;
  for (long long k = 0; k < nchunks; ++k) {
    __syncthreads();
    if (tid < 32) {
      if (tid == 0) {
        const T* q = buf[k & 1];
        const long long left = p.frames - k * CHUNK;
        const int n = (int)(left < CHUNK ? left : CHUNK);
        const int n8 = (n + 7) & ~7;
#pragma unroll 2
        for (int i = 0; i < n8; i += 8) {
          T v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = q[i + j];
#pragma unroll
          for (int j = 0; j < 8; ++j) s = add_rn<T>(s, v[j]);
        }
      }
    } else if (k + 1 < nchunks) {
      stage(k + 1, (int)((k + 1) & 1), tid - 32, NT - 32);
    }
  }
  if (tid == 0) reinterpret_cast<T*>(p.sums)[col] = s;
}

// ------------------------------------------------------------------------------------------------
// The same strict left-to-right float32 running sum, evaluated in parallel and still bit for bit.
//
// While the running sum s stays inside one binade [2^e, 2^(e+1)) its ulp u = 2^(e-23) is fixed, s = n u
// with an integer n in [2^23, 2^24), and adding a >= 0 is integer arithmetic: with a / u = q + f,
//     fl(s + a) / u = n + q + r,   r = [f > 1/2], and for the tie f == 1/2:  r = (n + q) & 1
// (round half to even looks at the parity of the significand, i.e. of n + q).  So every addend is a tiny
// transducer on the parity of n: (increment if n is even, increment if n is odd), both known from a and e
// alone, and transducers compose associatively:  (A then B)[p] = A[p] + B[(p + A[p]) & 1].  A CTA scans
// 8192 addends at once: each thread composes its 8 consecutive elements, a block-wide exclusive scan
// gives every thread the state at its first element, and the thread then walks its elements with the
// real parity.  Subnormal sums and the first normal binade share the grid u = 2^-149 (n = the bit
// pattern of s), so zeros and silence need no special case.
// The assumption "s stays in the binade" is checked, not trusted: the first element whose result reaches
// 2^24 ulps (the rounding grid changes there) is found by the walk, everything before it is committed,
// that one addition is done with the real float32 add, and the scan restarts behind it in the new
// binade - about 30 times per signal, since the sum only grows.  Increments saturate at 2^26 ulps (they
// only matter below 2^24); inf / NaN addends or sums fall back to the scalar chain for the rest.
// ------------------------------------------------------------------------------------------------
#ifndef VND_PS_E
#define VND_PS_E 8
#endif
#ifndef VND_PS_NT
#define VND_PS_NT 1024
#endif
constexpr int PS_NT = VND_PS_NT, PS_E = VND_PS_E, PS_B = PS_NT * PS_E;
constexpr unsigned PS_SAT = 1u << 26, PS_TOP = 1u << 24;
#ifndef VND_PS_HEAD
#define VND_PS_HEAD 4096
#endif
constexpr int PS_HEAD = VND_PS_HEAD;  // addends chained by one thread before the scans start

struct Tr {
  unsigned d0, d1;  // increment of n for an even / odd n
};
__device__ __forceinline__ Tr tr_compose(Tr a, Tr b) {  // a first, then b
  Tr r;
  r.d0 = umin(a.d0 + ((a.d0 & 1u) ? b.d1 : b.d0), PS_SAT);
  r.d1 = umin(a.d1 + ((a.d1 & 1u) ? b.d0 : b.d1), PS_SAT);
  return r;
}
// transducer of the addend a (>= 0) for a running sum with ulp u: t = a / u is formed exactly by two
// multiplications with powers of two, sc1 * sc2 = 1 / u (an underflowing t is far below 1/2 and rounds to an
// increment of 0 either way; an overflowing one saturates, as do inf and NaN: they force the real addition)
__device__ __forceinline__ Tr tr_of(float a, float sc1, float sc2) {
  const float t = fmul(fmul(a, sc1), sc2);
  if (!(t < 67108864.0f)) return Tr{PS_SAT, PS_SAT};  // >= 2^26 ulps, inf, NaN
  const unsigned q = (unsigned)t;              // floor (t >= 0)
  const float f = fsub(t, (float)q);           // exact: t has at most 24 significant bits
  const unsigned up = f > 0.5f ? 1u : 0u, tie = f == 0.5f ? 1u : 0u;
  return Tr{q + (up | (tie & q & 1u)), q + (up | (tie & (q + 1u) & 1u))};  // tie: to the even significand
}

static_assert(PS_NT == 1024, "the scan of the warp totals assumes 32 warps");
__global__ void __launch_bounds__(PS_NT) seq_sumsq_par_kernel(const SeqParams p) {
  __shared__ float stage[PS_HEAD];  // the head's addends
  __shared__ Tr warp_tot[PS_NT / 32];
  __shared__ unsigned sh_cross, sh_n;
  __shared__ float sh_a, sh_s;
  const int col = blockIdx.x;
  const float* base;
  long long st;
  if (col < p.channels) {
    base = reinterpret_cast<const float*>(p.a) + (long long)col * p.a_sc;
    st = p.a_st;
  } else {
    base = reinterpret_cast<const float*>(p.b) + (long long)(col - p.channels) * p.b_sc;
    st = p.b_st;
  }
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long N = p.frames;
  float s = 0.0f;
  long long pos = 0;
  {  // The sum changes binade at about every doubling of the position: the first PS_HEAD addends would cost a
     // round each time.  They are staged by everybody and chained by one thread (4 clocks per addend).
    float* head = stage;
    const int nh = (int)(N < PS_HEAD ? N : PS_HEAD);
    for (int i = tid; i < nh; i += PS_NT) head[i] = sq<float>(base[(long long)i * st]);
    __syncthreads();
    if (tid == 0) {
      float h = 0.0f;
      for (int i = 0; i < nh; ++i) h = fadd(h, head[i]);
      sh_s = h;
    }
    __syncthreads();
    s = sh_s;
    pos = nh;
  }
  while (pos < N) {
    const unsigned sb = __float_as_uint(s);
    const unsigned seb = sb >> 23;
    if (seb >= 255u) {  // inf or NaN so far: the scalar chain finishes the column
      if (tid == 0) {
        for (long long t = pos; t < N; ++t) s = fadd(s, sq<float>(base[t * st]));
        sh_s = s;
      }
      __syncthreads();
      s = sh_s;
      break;
    }
    const int e = seb ? (int)seb - 127 : -126;
    const unsigned n_in = seb ? ((sb & 0x7fffffu) | 0x800000u) : sb;
    const int k = 23 - e, k1 = k / 2;  // 1 / u = 2^k as the product of two representable powers of two (k in [-104, 149])
    const float sc1 = __uint_as_float((unsigned)(127 + k1) << 23), sc2 = __uint_as_float((unsigned)(127 + k - k1) << 23);
    if (tid == 0) sh_cross = PS_B;
    // this thread's PS_E consecutive addends (zeros behind the end: they change nothing)
    float a[PS_E];
    Tr el[PS_E];
    Tr loc{0u, 0u};
    // (staging the round coalesced through shared memory was measured slower than these strided loads: the
    // lines stay in L1 across a thread's PS_E loads)
    const long long t0 = pos + (long long)tid * PS_E;
#pragma unroll
    for (int j = 0; j < PS_E; ++j) a[j] = (t0 + j < N) ? sq<float>(base[(t0 + j) * st]) : 0.0f;
#pragma unroll
    for (int j = 0; j < PS_E; ++j) {
      el[j] = tr_of(a[j], sc1, sc2);
      loc = tr_compose(loc, el[j]);
    }
    // block-wide exclusive scan of the thread transducers (lower threads first)
    Tr inc = loc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      Tr up;
      up.d0 = __shfl_up_sync(0xffffffffu, inc.d0, o);
      up.d1 = __shfl_up_sync(0xffffffffu, inc.d1, o);
      if (lane >= o) inc = tr_compose(up, inc);
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      Tr w = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        Tr up;
        up.d0 = __shfl_up_sync(0xffffffffu, w.d0, o);
        up.d1 = __shfl_up_sync(0xffffffffu, w.d1, o);
        if (lane >= o) w = tr_compose(up, w);
      }
      warp_tot[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    Tr pre{0u, 0u};  // everything before this thread
    {
      Tr lanes_before;
      lanes_before.d0 = __shfl_up_sync(0xffffffffu, inc.d0, 1);
      lanes_before.d1 = __shfl_up_sync(0xffffffffu, inc.d1, 1);
      if (lane == 0) lanes_before = Tr{0u, 0u};
      pre = warp > 0 ? tr_compose(warp_tot[warp - 1], lanes_before) : lanes_before;
    }
    // walk the own elements with the real parity; find the first one that leaves the binade
    unsigned n = n_in + ((n_in & 1u) ? pre.d1 : pre.d0);
    unsigned nv[PS_E];
    int cross = -1;
    if (n < PS_TOP) {
#pragma unroll
      for (int j = 0; j < PS_E; ++j) {
        const unsigned nn = n + ((n & 1u) ? el[j].d1 : el[j].d0);
        if (cross < 0) {
          if (nn >= PS_TOP) cross = j;
          else n = nn;
        }
        nv[j] = n;
      }
      if (cross >= 0) atomicMin(&sh_cross, (unsigned)(tid * PS_E + cross));
    }
    __syncthreads();
    const unsigned c = sh_cross;  // elements committed in this binade; element c (if < PS_B) takes the real addition
    if (c > 0u && (int)((c - 1u) / PS_E) == tid) {  // static indices: a run-time subscript would put nv[] in local memory
      const int idx = (int)((c - 1u) % PS_E);
#pragma unroll
      for (int j = 0; j < PS_E; ++j)
        if (j == idx) sh_n = nv[j];
    }
    if (c < (unsigned)PS_B && (int)(c / PS_E) == tid) {
      const int idx = (int)(c % PS_E);
#pragma unroll
      for (int j = 0; j < PS_E; ++j)
        if (j == idx) sh_a = a[j];
    }
    __syncthreads();
    if (c > 0u) s = __uint_as_float(((unsigned)(e + 126) << 23) + sh_n);
    pos += c;
    if (c < (unsigned)PS_B) {
      s = fadd(s, sh_a);
      pos += 1;
    }
    // no barrier here: the next round rewrites sh_cross only after every thread has read it (the barrier
    // above), and sh_n / sh_a / warp_tot only behind barriers that every thread reaches after its reads
  }
  if (tid == 0) reinterpret_cast<float*>(p.sums)[col] = s;
}

// ------------------------------------------------------------------------------------------------
// The same scan over a thread-block CLUSTER: PS_K CTAs (one SM each) share a column, a round covers
// PS_K x 8192 addends, and the CTAs exchange three words per round through distributed shared memory
// (their composed transducer, their first binade change, the committed sum), each exchange closed by a
// cluster barrier.  Every CTA keeps its own copy of the running sum and position, so the control flow is
// identical everywhere; the head and the inf / NaN tail are computed redundantly (no communication).
// ------------------------------------------------------------------------------------------------
#ifndef VND_PS_K
#define VND_PS_K 8
#endif
constexpr int PS_K = VND_PS_K;
constexpr unsigned PS_BK = (unsigned)PS_K * PS_B;  // addends per round

namespace cg = cooperative_groups;

// The column source is a template parameter so that the batched decorrelate (vnd_batch.cu) runs the same scan over
// columns that live at device-side clip offsets: Cols::column(col, &base, &stride, &frames) and Cols::store(col, sum).
template <class Cols>
__global__ void __cluster_dims__(PS_K, 1, 1) __launch_bounds__(PS_NT) seq_sumsq_cluster_kernel(const Cols p) {
  __shared__ float stage[PS_HEAD];
  __shared__ Tr warp_tot[PS_NT / 32];
  __shared__ Tr cta_tot[PS_K];        // written by every CTA of the cluster (slot = its rank)
  __shared__ unsigned cta_min[PS_K];  // likewise: first binade change each CTA found (PS_BK = none)
  __shared__ unsigned sh_cross, sh_n;
  __shared__ float sh_a, sh_s;
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned rank = cluster.block_rank();
  const int col = blockIdx.x / PS_K;
  const float* base;
  long long st, N;
  p.column(col, &base, &st, &N);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float s = 0.0f;
  long long pos = 0;
  {  // head: chained by one thread of every CTA (same result everywhere)
    const int nh = (int)(N < PS_HEAD ? N : PS_HEAD);
    for (int i = tid; i < nh; i += PS_NT) stage[i] = sq<float>(base[(long long)i * st]);
    __syncthreads();
    if (tid == 0) {
      float h = 0.0f;
      for (int i = 0; i < nh; ++i) h = fadd(h, stage[i]);
      sh_s = h;
    }
    __syncthreads();
    s = sh_s;
    pos = nh;
  }
  while (pos < N) {
    const unsigned sb = __float_as_uint(s);
    const unsigned seb = sb >> 23;
    if (seb >= 255u) {  // inf or NaN so far: the scalar chain finishes the column (in every CTA alike)
      if (tid == 0) {
        for (long long t = pos; t < N; ++t) s = fadd(s, sq<float>(base[t * st]));
        sh_s = s;
      }
      __syncthreads();
      s = sh_s;
      break;
    }
    const int e = seb ? (int)seb - 127 : -126;
    const unsigned n_in = seb ? ((sb & 0x7fffffu) | 0x800000u) : sb;
    const int k = 23 - e, k1 = k / 2;
    const float sc1 = __uint_as_float((unsigned)(127 + k1) << 23), sc2 = __uint_as_float((unsigned)(127 + k - k1) << 23);
    if (tid == 0) sh_cross = PS_BK;
    float a[PS_E];
    Tr el[PS_E];
    Tr loc{0u, 0u};
    const unsigned g0 = (rank * (unsigned)PS_NT + (unsigned)tid) * (unsigned)PS_E;  // index of the thread's first addend in the round
    const long long t0 = pos + (long long)g0;
#pragma unroll
    for (int j = 0; j < PS_E; ++j) a[j] = (t0 + j < N) ? sq<float>(base[(t0 + j) * st]) : 0.0f;
#pragma unroll
    for (int j = 0; j < PS_E; ++j) {
      el[j] = tr_of(a[j], sc1, sc2);
      loc = tr_compose(loc, el[j]);
    }
    Tr inc = loc;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      Tr up;
      up.d0 = __shfl_up_sync(0xffffffffu, inc.d0, o);
      up.d1 = __shfl_up_sync(0xffffffffu, inc.d1, o);
      if (lane >= o) inc = tr_compose(up, inc);
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
      Tr w = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        Tr up;
        up.d0 = __shfl_up_sync(0xffffffffu, w.d0, o);
        up.d1 = __shfl_up_sync(0xffffffffu, w.d1, o);
        if (lane >= o) w = tr_compose(up, w);
      }
      warp_tot[lane] = w;
      const Tr tot = Tr{__shfl_sync(0xffffffffu, w.d0, 31), __shfl_sync(0xffffffffu, w.d1, 31)};
      if (lane < PS_K) *cluster.map_shared_rank(&cta_tot[rank], lane) = tot;  // lane r tells CTA r this CTA's composed transducer
    }
    cluster.sync();  // also the CTA barrier behind the scan of the warp totals
    Tr pre{0u, 0u};
    for (unsigned r = 0; r < rank; ++r) pre = tr_compose(pre, cta_tot[r]);  // the CTAs before this one
    {
      Tr lanes_before;
      lanes_before.d0 = __shfl_up_sync(0xffffffffu, inc.d0, 1);
      lanes_before.d1 = __shfl_up_sync(0xffffffffu, inc.d1, 1);
      if (lane == 0) lanes_before = Tr{0u, 0u};
      if (warp > 0) pre = tr_compose(pre, warp_tot[warp - 1]);
      pre = tr_compose(pre, lanes_before);
    }
    unsigned n = n_in + ((n_in & 1u) ? pre.d1 : pre.d0);
    unsigned nv[PS_E];
    int cross = -1;
    if (n < PS_TOP) {
#pragma unroll
      for (int j = 0; j < PS_E; ++j) {
        const unsigned nn = n + ((n & 1u) ? el[j].d1 : el[j].d0);
        if (cross < 0) {
          if (nn >= PS_TOP) cross = j;
          else n = nn;
        }
        nv[j] = n;
      }
      if (cross >= 0) atomicMin(&sh_cross, g0 + (unsigned)cross);
    }
    __syncthreads();
    if (tid < PS_K) *cluster.map_shared_rank(&cta_min[rank], tid) = sh_cross;
    cluster.sync();
    unsigned c = PS_BK;  // addends committed in this binade; addend c (if < PS_BK) takes the real addition
#pragma unroll
    for (int r = 0; r < PS_K; ++r) c = umin(c, cta_min[r]);
    if (c > 0u && (c - 1u) / (unsigned)PS_E == rank * (unsigned)PS_NT + (unsigned)tid) {
      const int idx = (int)((c - 1u) % PS_E);
      unsigned v = 0u;
#pragma unroll
      for (int j = 0; j < PS_E; ++j)
        if (j == idx) v = nv[j];
      for (int r = 0; r < PS_K; ++r) *cluster.map_shared_rank(&sh_n, r) = v;
    }
    if (c < PS_BK && c / (unsigned)PS_E == rank * (unsigned)PS_NT + (unsigned)tid) {
      const int idx = (int)(c % PS_E);
      float v = 0.0f;
#pragma unroll
      for (int j = 0; j < PS_E; ++j)
        if (j == idx) v = a[j];
      for (int r = 0; r < PS_K; ++r) *cluster.map_shared_rank(&sh_a, r) = v;
    }
    cluster.sync();
    if (c > 0u) s = __uint_as_float(((unsigned)(e + 126) << 23) + sh_n);
    pos += c;
    if (c < PS_BK) {
      s = fadd(s, sh_a);
      pos += 1;
    }
    // the next round's first remote writes (cta_tot) come behind its own barriers; sh_n / sh_a / cta_min are
    // rewritten only behind the next round's cluster barriers, which every thread reaches after these reads
  }
  cluster.sync();  // nobody leaves while a peer may still write into its shared memory
  if (rank == 0 && tid == 0) p.store(col, s);
}

// gains[c] = sqrt(mean_x[c]) / sqrt(mean_y[c] + eps) with numpy's dtype chain: the mean divides in
// float64 (np.mean's true_divide by an intp count) and stores the array dtype; eps is a weak
// Python float, i.e. it is cast to the array dtype.  sums = [x columns..., y columns...].
template <typename T>
__global__ void rms_gain_kernel(const T* __restrict__ sums, T* __restrict__ gains, int channels, long long frames) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= channels) return;
  if constexpr (sizeof(T) == 4) {
    gains[c] = rms_gain_f32(sums[c], sums[channels + c], frames);
  } else {
    const double mx = __ddiv_rn(sums[c], (double)frames);
    const double my = __ddiv_rn(sums[channels + c], (double)frames);
    gains[c] = __ddiv_rn(__dsqrt_rn(mx), __dsqrt_rn(dadd(my, 1e-10)));
  }
}

// out[m, c] = y[m - shift_c, c] * gain[c] (0 outside), shift_c = delay for the delayed channel.
struct PlaceParams {
  const float* y;
  long long y_st, y_sc;
  void* out;
  long long o_st, o_sc;
  long long frames;  // of y
  int channels;
  const float* gains;  // nullable
  int delay, delay_ch;
};

template <typename TOut>
__global__ void __launch_bounds__(256) place_kernel(const PlaceParams p) {
  const long long total = (p.frames + p.delay) * p.channels;
  TOut* __restrict__ out = reinterpret_cast<TOut*>(p.out);
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long m = e / p.channels;
    const int c = (int)(e - m * p.channels);
    const long long n = m - (c == p.delay_ch ? p.delay : 0);
    float v = 0.0f;
    if (n >= 0 && n < p.frames) {
      v = p.y[n * p.y_st + c * p.y_sc];
      if (p.gains) v = fmul(v, p.gains[c]);
    }
    out[m * p.o_st + c * p.o_sc] = (TOut)v;
  }
}

// HaasEffect.decorrelate in closed form (float64 throughout, SURVEY.md A.6).
struct HaasParams {
  const float* x;
  long long x_st, x_sc;
  double* out;
  long long o_st, o_sc;
  long long frames;
  int delay, delay_ch;
  int mode_ms, mono, use_width;
  double width;
};

__global__ void __launch_bounds__(256) haas_kernel(const HaasParams p) {
  const long long total = p.frames + p.delay;
  for (long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x; m < total; m += (long long)gridDim.x * blockDim.x) {
    const long long q0 = m - (p.delay_ch == 0 ? p.delay : 0), q1 = m - (p.delay_ch == 1 ? p.delay : 0);
    const bool v0 = q0 >= 0 && q0 < p.frames, v1 = q1 >= 0 && q1 < p.frames;
    float a0 = 0.0f, b0 = 0.0f, a1 = 0.0f, b1 = 0.0f;
    if (v0) {
      a0 = p.x[q0 * p.x_st];
      b0 = p.x[q0 * p.x_st + p.x_sc];
    }
    if (v1) {
      a1 = p.x[q1 * p.x_st];
      b1 = p.x[q1 * p.x_st + p.x_sc];
    }
    const double2 c = haas_frame(a0, b0, v0, a1, b1, v1, p.mode_ms, p.mono, p.use_width, p.width);
    p.out[m * p.o_st] = c.x;
    p.out[m * p.o_st + p.o_sc] = c.y;
  }
}

// In-place helpers on a (frames, 2) signal.
struct StereoOpParams {
  void* a;
  long long a_st, a_sc;
  const void* dry;
  long long d_st, d_sc;
  long long frames;
  int op;
  double width;
  const void* gains;
};

template <typename T>
__device__ __forceinline__ T t_add(T a, T b) { return a + b; }
template <>
__device__ __forceinline__ float t_add<float>(float a, float b) { return fadd(a, b); }
template <>
__device__ __forceinline__ double t_add<double>(double a, double b) { return dadd(a, b); }
template <typename T>
__device__ __forceinline__ T t_sub(T a, T b);
template <>
__device__ __forceinline__ float t_sub<float>(float a, float b) { return fsub(a, b); }
template <>
__device__ __forceinline__ double t_sub<double>(double a, double b) { return dsub(a, b); }
template <typename T>
__device__ __forceinline__ T t_mul(T a, T b);
template <>
__device__ __forceinline__ float t_mul<float>(float a, float b) { return fmul(a, b); }
template <>
__device__ __forceinline__ double t_mul<double>(double a, double b) { return dmul(a, b); }

template <typename T>
__global__ void __launch_bounds__(256) stereo_op_kernel(const StereoOpParams p) {
  T* a = reinterpret_cast<T*>(p.a);
  const T* dry = reinterpret_cast<const T*>(p.dry);
  const T half = (T)0.5;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < p.frames; t += (long long)gridDim.x * blockDim.x) {
    T u = a[t * p.a_st], v = a[t * p.a_st + p.a_sc];
    switch (p.op) {
      case 0: {  // LR_to_MS
        const T M = t_mul<T>(t_add<T>(u, v), half), S = t_mul<T>(t_sub<T>(u, v), half);
        u = M;
        v = S;
      } break;
      case 1: {  // MS_to_LR
        const T L = t_add<T>(u, v), R = t_sub<T>(u, v);
        u = L;
        v = R;
      } break;
      case 2: {  // apply_stereo_width
        T M = t_mul<T>(t_add<T>(u, v), half), S = t_mul<T>(t_sub<T>(u, v), half);
        M = t_mul<T>(M, (T)(1.0 - p.width));
        S = t_mul<T>(S, (T)p.width);
        u = t_add<T>(M, S);
        v = t_sub<T>(M, S);
      } break;
      case 3: {  // encode_signal_to_side_channel
        const T M = t_add<T>(dry[t * p.d_st], dry[t * p.d_st + p.d_sc]);
        const T S = t_mul<T>(t_sub<T>(u, v), half);
        u = t_mul<T>(t_add<T>(M, S), half);
        v = t_mul<T>(t_sub<T>(M, S), half);
      } break;
      default: {  // 4: scale by per-channel gains
        const T* g = reinterpret_cast<const T*>(p.gains);
        u = t_mul<T>(u, g[0]);
        v = t_mul<T>(v, g[1]);
      } break;
    }
    a[t * p.a_st] = u;
    a[t * p.a_st + p.a_sc] = v;
  }
}

// In-place per-channel scale of a (frames, C) float32 signal.
__global__ void __launch_bounds__(256) scale_kernel(float* y, long long y_st, long long y_sc, long long frames, int channels,
                                                    const float* __restrict__ gains) {
  const long long total = frames * channels;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
    const long long t = e / channels;
    const int c = (int)(e - t * channels);
    float* q = y + t * y_st + c * y_sc;
    *q = fmul(*q, gains[c]);
  }
}


// (rows, cols) row-major -> (cols, rows) row-major through a padded shared-memory tile, so that both
// the loads and the stores are coalesced.  Used to turn wide frame-interleaved slabs into planar
// ones (and back) around the planar FIR kernel.
__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ src, float* __restrict__ dst, long long rows,
                                                        long long cols, long long ld_src, long long ld_dst) {
  __shared__ float tile[32][33];
  const long long tiles_c = ceil_div<long long>(cols, 32);
  const long long tr = blockIdx.x / tiles_c, tc = blockIdx.x % tiles_c;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int j = ty; j < 32; j += 8) {
    const long long r = tr * 32 + j, c = tc * 32 + tx;
    if (r < rows && c < cols) tile[j][tx] = src[r * ld_src + c];
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const long long c = tc * 32 + j, r = tr * 32 + tx;
    if (r < rows && c < cols) dst[c * ld_dst + r] = tile[tx][j];
  }
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
static unsigned grid_for(long long n, int per_block = 256) {
  DeviceInfo di;
  if (device_info(&di)) di.sm_count = 148;
  long long b = ceil_div<long long>(n, per_block);
  const long long cap = (long long)di.sm_count * 8;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (unsigned)b;
}

int seq_sumsq_launch(const vnd_signal* a, const vnd_signal* b, void* sums, cudaStream_t st) {
  SeqParams p{};
  p.a = a->data;
  p.a_st = a->stride_t;
  p.a_sc = a->stride_c;
  p.frames = a->frames;
  p.channels = a->channels;
  p.sums = sums;
  int cols = a->channels;
  if (b) {
    p.b = b->data;
    p.b_st = b->stride_t;
    p.b_sc = b->stride_c;
    cols *= 2;
  }
  if (cols == 0) return VND_OK;
  static const bool serial_only = [] {
    const char* e = getenv("VND_SEQSUM_SERIAL");  // testing: the scalar chain for every length
    return e && e[0] == '1';
  }();
  DeviceInfo di;
  {
    const int rc = device_info(&di);
    if (rc) return rc;
  }
  const int sm_count = di.sm_count;
  static const bool cluster_ok = [] {
    const char* e = getenv("VND_SEQSUM_CLUSTER");  // testing: 0 keeps the single-CTA scan
    return !(e && e[0] == '0');
  }();
  if (a->dtype == VND_F64) seq_sumsq_kernel<double><<<cols, 256, 0, st>>>(p);
  else if (serial_only || a->frames < 4096) seq_sumsq_kernel<float><<<cols, 256, 0, st>>>(p);
  else if (cluster_ok && a->frames >= (long long)PS_HEAD + 2 * PS_B && cols * PS_K <= 2 * sm_count)  // few columns: latency matters, SMs are idle
    seq_sumsq_cluster_kernel<SeqParams><<<cols * PS_K, PS_NT, 0, st>>>(p);
  else seq_sumsq_par_kernel<<<cols, PS_NT, 0, st>>>(p);
  return after_launch("seq_sumsq_kernel");
}

// the cluster scan over the 4 columns of every clip of a batch (vnd_batch.cu picks it for few long columns)
int batch_sumsq_cluster_launch(const BatchSumCols& cols, int n_cols, cudaStream_t st) {
  if (n_cols == 0) return VND_OK;
  seq_sumsq_cluster_kernel<BatchSumCols><<<n_cols * PS_K, PS_NT, 0, st>>>(cols);
  return after_launch("seq_sumsq_cluster_kernel");
}
int seq_sumsq_cluster_width() { return PS_K; }
int seq_sumsq_scan_round() { return PS_B; }
int seq_sumsq_scan_head() { return PS_HEAD; }

int pairwise_sumsq_launch(const void* col, int dtype, long long n, void* leaf, void* out, cudaStream_t st);

// numpy reduces np.mean(np.square(a), axis=0) with its inner loop on the axis of the SMALLEST stride: a C-order (frames,
// channels) array is summed frame by frame (a sequential running sum per column), a Fortran-ordered / planar one column by
// column with the pairwise algorithm.  The two give different float32 sums (6e-5 relative on a 250 k-frame file), so the
// order follows the layout of each signal, as it does in the reference.
static bool sums_pairwise(const vnd_signal* s) {
  if (s->channels <= 0 || s->frames <= 1) return false;
  const long long st = s->stride_t < 0 ? -s->stride_t : s->stride_t, sc = s->stride_c < 0 ? -s->stride_c : s->stride_c;
  return s->channels > 1 ? (st == 1 && sc >= s->frames) : false;
}
size_t colsumsq_workspace_bytes(long long frames) { return ((size_t)(frames / 64) + 8) * 8; }

// sums[0 .. Ca) for a's columns, then b's; `leaf` (colsumsq_workspace_bytes) is only touched for planar signals
int colsumsq_launch(const vnd_signal* a, const vnd_signal* b, void* sums, void* leaf, size_t leaf_bytes, cudaStream_t st) {
  const bool pa = sums_pairwise(a), pb = b && sums_pairwise(b);
  if (!pa && !pb) return seq_sumsq_launch(a, b, sums, st);
  const size_t es = a->dtype == VND_F64 ? 8 : 4;
  VND_REQUIRE(leaf != nullptr && leaf_bytes >= colsumsq_workspace_bytes(a->frames), VND_ENOMEM, "workspace too small for a planar signal's pairwise sums");
  int rc;
  const vnd_signal* sig[2] = {a, b};
  const bool pw[2] = {pa, pb};
  char* out = reinterpret_cast<char*>(sums);
  for (int k = 0; k < 2; ++k) {
    if (!sig[k]) continue;
    if (!pw[k]) {
      if ((rc = seq_sumsq_launch(sig[k], nullptr, out, st))) return rc;
    } else {
      for (int c = 0; c < sig[k]->channels; ++c) {
        const char* col = reinterpret_cast<const char*>(sig[k]->data) + (long long)c * sig[k]->stride_c * (long long)es;
        VND_REQUIRE(sig[k]->stride_t == 1 && sig[k]->stride_c > 0, VND_EUNSUPPORTED, "planar signals with negative strides are not supported");
        if ((rc = pairwise_sumsq_launch(col, a->dtype, sig[k]->frames, leaf, out + (size_t)c * es, st))) return rc;
      }
    }
    out += (size_t)sig[k]->channels * es;
  }
  return VND_OK;
}

int rms_gain_launch(const void* sums, void* gains, int channels, long long frames, int dtype, cudaStream_t st) {
  if (channels == 0) return VND_OK;
  const unsigned blocks = (unsigned)ceil_div(channels, 128);
  if (dtype == VND_F64) rms_gain_kernel<double><<<blocks, 128, 0, st>>>((const double*)sums, (double*)gains, channels, frames);
  else rms_gain_kernel<float><<<blocks, 128, 0, st>>>((const float*)sums, (float*)gains, channels, frames);
  return after_launch("rms_gain_kernel");
}

int place_launch(const float* y, long long y_st, long long y_sc, long long frames, int channels, const vnd_signal* out,
                 const float* gains, int delay, int delay_ch, cudaStream_t st) {
  PlaceParams p{};
  p.y = y;
  p.y_st = y_st;
  p.y_sc = y_sc;
  p.out = out->data;
  p.o_st = out->stride_t;
  p.o_sc = out->stride_c;
  p.frames = frames;
  p.channels = channels;
  p.gains = gains;
  p.delay = delay;
  p.delay_ch = delay_ch;
  const long long total = (frames + delay) * channels;
  if (total == 0) return VND_OK;
  if (out->dtype == VND_F64) place_kernel<double><<<grid_for(total), 256, 0, st>>>(p);
  else place_kernel<float><<<grid_for(total), 256, 0, st>>>(p);
  return after_launch("place_kernel");
}

int scale_launch(float* y, long long y_st, long long y_sc, long long frames, int channels, const float* gains, cudaStream_t st) {
  if (frames * channels == 0) return VND_OK;
  scale_kernel<<<grid_for(frames * channels), 256, 0, st>>>(y, y_st, y_sc, frames, channels, gains);
  return after_launch("scale_kernel");
}

int haas_launch(const vnd_signal* x, const vnd_signal* out, int delay, int delay_ch, int mode_ms, int mono, int use_width,
                double width, cudaStream_t st) {
  HaasParams p{};
  p.x = reinterpret_cast<const float*>(x->data);
  p.x_st = x->stride_t;
  p.x_sc = x->stride_c;
  p.out = reinterpret_cast<double*>(out->data);
  p.o_st = out->stride_t;
  p.o_sc = out->stride_c;
  p.frames = x->frames;
  p.delay = delay;
  p.delay_ch = delay_ch;
  p.mode_ms = mode_ms;
  p.mono = mono;
  p.use_width = use_width;
  p.width = width;
  if (p.frames + delay == 0) return VND_OK;
  haas_kernel<<<grid_for(p.frames + delay), 256, 0, st>>>(p);
  return after_launch("haas_kernel");
}

// src is (rows, cols) with row pitch ld_src, dst becomes (cols, rows) with row pitch ld_dst (elements)
int transpose_launch_ld(const float* src, float* dst, long long rows, long long cols, long long ld_src, long long ld_dst, cudaStream_t st) {
  if (rows * cols == 0) return VND_OK;
  const long long blocks = ceil_div<long long>(rows, 32) * ceil_div<long long>(cols, 32);
  VND_REQUIRE(blocks < 0x7fffffffLL, VND_EUNSUPPORTED, "transpose grid too large");
  transpose_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, dst, rows, cols, ld_src, ld_dst);
  return after_launch("transpose_kernel");
}

int transpose_launch(const float* src, float* dst, long long rows, long long cols, cudaStream_t st) {
  return transpose_launch_ld(src, dst, rows, cols, cols, rows, st);
}

int stereo_op_launch(const vnd_signal* a, const vnd_signal* dry, int op, double width, const void* gains, cudaStream_t st) {
  StereoOpParams p{};
  p.a = a->data;
  p.a_st = a->stride_t;
  p.a_sc = a->stride_c;
  if (dry) {
    p.dry = dry->data;
    p.d_st = dry->stride_t;
    p.d_sc = dry->stride_c;
  }
  p.frames = a->frames;
  p.op = op;
  p.width = width;
  p.gains = gains;
  if (p.frames == 0) return VND_OK;
  if (a->dtype == VND_F64) stereo_op_kernel<double><<<grid_for(p.frames), 256, 0, st>>>(p);
  else stereo_op_kernel<float><<<grid_for(p.frames), 256, 0, st>>>(p);
  return after_launch("stereo_op_kernel");
}

}  // namespace vnd
