// Batched stereo-image objective kernels (sm_100a).
//
// Reference arithmetic evaluated here (paths relative to the reference root):
//   symmetry_aware_objective   src/vndecorrelate/optimization.py:46-105
//   polar_coordinates          src/vndecorrelate/utils/dsp.py:374-422  (mode 'MS', semicircular)
//   moment helpers             src/vndecorrelate/optimization.py:11-43
//   candidates                 src/vndecorrelate/optimization.py:260-272 (velvet noise, channel 0
//                              filtered, channel 1 copied, LR, no normaliser) and :183-203 (Haas)
//
// The kernels produce per (clip, candidate) the sums the objective is made of; the host applies the
// reference's scalar dtype chain (SURVEY.md A.5).  Two facts shape the velvet-noise kernel:
//   * folded theta == atan(d / s) with d = L - R, s = L + R, so no atan2 + fold is needed for the
//     amplitude-weighted sums, whose weights make an absolute error of 1e-7 rad irrelevant;
//   * max|theta| IS ulp-sensitive (the penalty term multiplies it by ~1.6e3), but rounding is
//     monotone, so max|theta| is attained at the frame with the largest |d|/|s| among frames with
//     s >= 0 and among frames with s < 0.  The kernel tracks those two frames exactly (track_ratio: the cross
//     products are compared in float64, where they are exact) and the host evaluates a correctly rounded float32
//     arctan2 for just those.
//
// Decomposition: CTA = (chunk of tiles, clip, candidate group).  A tile of both channels (+ the
// filter halo for channel 0) is staged in shared memory once and reused by every candidate of the
// group; each WARP owns whole candidates (no block-level reduction, no __syncthreads in the
// candidate loop), reduces with warp shuffles and accumulates float64 partials in shared memory.

#include <stdlib.h>
#include <string.h>

#include <vector>

#include "vnd_batch.cuh"

namespace vnd {

// The parameter block, the polar moments of a frame (src/vndecorrelate/utils/dsp.py:374-422,
// src/vndecorrelate/optimization.py:11-43) in scalar and packed form, the exact max|theta| ratio tracker and the warp
// reductions.
constexpr int OBJ_SLOTS = 12;  // doubles per (clip, candidate) partial, see vnd_b200.h
// doubles per candidate in a CTA's accumulators and per chunk partial: the 12 slots, then the low parts of the
// double-double sums of slots 0-5
constexpr int OBJ_CHUNK_SLOTS = 18;
#ifndef VND_OBJ_NT
#define VND_OBJ_NT 640  // 20 warps: measured best of 512 / 640 / 768 / 896 / 1024 threads (16 frames per lane)
#endif
constexpr int OBJ_NT = VND_OBJ_NT;
#ifndef VND_OBJ_R
#define VND_OBJ_R 16
#endif
constexpr int OBJ_R = VND_OBJ_R;  // frames per lane and pass (even: the taps are applied with packed adds)
constexpr int OBJ_TILE = 4096;

struct ObjParams {
  const float* clips;
  long long frames, clip_stride, chan_stride;
  const int* words;
  const int* offsets;
  int n_cand;
  int apply_gain;
  int halo;
  int cand_per_group;
  int tiles_per_chunk;
  int n_chunks;
  double* chunk_partials;  // [clip][chunk][cand][OBJ_CHUNK_SLOTS]
};

// One CTA of the run-list objective (vnd_vn_objective_runs_dev): a chunk of one clip's tiles on one group of one run's
// candidates.  Built on the host, read by the CTA from the front of the workspace.
struct ObjRunItem {
  long long base;    // packed column of the clip's frame 0
  long long frames;  // the clip's length
  long long part;    // first chunk-partial row (OBJ_CHUNK_SLOTS doubles) of the item
  int tile_first, n_tiles, cand0, ncand;
};

// atan(t) for t in [0, 1]: t * P(t^2), |error| <= 1e-7 (degree-8 minimax fit, float32 Horner).
__device__ __forceinline__ float atan01(float t) {
  const float z = t * t;
  float p = 0.00245671847107214f;
  p = fmaf(p, z, -0.01440133168500584f);
  p = fmaf(p, z, 0.03978117728736144f);
  p = fmaf(p, z, -0.07234853052703884f);
  p = fmaf(p, z, 0.10498943808759016f);
  p = fmaf(p, z, -0.14161228535203682f);
  p = fmaf(p, z, 0.19985906672823953f);
  p = fmaf(p, z, -0.3333259702410447f);
  p = fmaf(p, z, 0.9999998863844667f);
  return p * t;
}

// Packed fp32 arithmetic (sm_100+): two IEEE round-to-nearest operations per instruction on an aligned
// register pair (FADD2 / FMUL2 / FFMA2 in SASS): same bits as two scalar operations, half the issue slots.
typedef unsigned long long obj_pair_t;
#define VND_OBJ_PACKED(name, op)                                                   \
  __device__ __forceinline__ void name(float& a0, float& a1, float b0, float b1) { \
    obj_pair_t ra, rb;                                                             \
    asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a0), "f"(a1));                   \
    asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b0), "f"(b1));                   \
    asm(op ".rn.f32x2 %0, %0, %1;" : "+l"(ra) : "l"(rb));                         \
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(ra));                  \
  }
VND_OBJ_PACKED(obj_add2, "add")
VND_OBJ_PACKED(obj_sub2, "sub")
VND_OBJ_PACKED(obj_mul2, "mul")
// (a0, a1) = (a0, a1) * (b0, b1) + (c0, c1), one rounding each (FFMA2)
__device__ __forceinline__ void obj_fma2(float& a0, float& a1, float b0, float b1, float c0, float c1) {
  obj_pair_t ra, rb, rc;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b0), "f"(b1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c0), "f"(c1));
  asm("fma.rn.f32x2 %0, %0, %1, %2;" : "+l"(ra) : "l"(rb), "l"(rc));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(ra));
}

// Ratio tracker: record (ad, as) when ad / as > bd / bs, i.e. when ad * bs > bd * as, decided EXACTLY: the product of
// two float32 values is exact in float64 and cannot underflow there.  The float32 pre-test only filters frames that
// are certainly below the record: rounding is monotone, so exact(ad * bs) > exact(bd * as) implies
// fl(ad * bs) >= fl(bd * as) >= fl(fl(bd * as) * 0.99999f), and underflowed (zero) products pass the test too.
// Records are rare (a logarithmic number per lane), so the float64 compare is almost never executed.
__device__ __forceinline__ void track_ratio(float ad, float as, float& bd, float& bs) {
  if (ad * bs >= (bd * as) * 0.99999f) {
    if ((double)ad * (double)bs > (double)bd * (double)as) {  // ties keep the earlier frame
      bd = ad;
      bs = as;
    }
  }
}

struct LaneAcc {
  float sr, srt, srt2, srt3, slr, sll;
  float d_pos, s_pos, d_neg, s_neg;  // |d|, |s| of the frame with the largest |d|/|s| per sign of s
};

__device__ __forceinline__ void lane_acc_frame(LaneAcc& a, float l, float r_) {
  const float d = fsub(l, r_), s = fadd(l, r_);  // utils/dsp.py:399-401
  const float ad = fabsf(d), as = fabsf(s);
  const float mx = fmaxf(ad, as), mn = fminf(ad, as);
  const float t = mx > 0.0f ? __fdividef(mn, mx) : 0.0f;
  float th = atan01(t);
  if (ad > as) th = 1.57079632679489662f - th;
  th = __int_as_float(__float_as_int(th) | ((__float_as_int(d) ^ __float_as_int(s)) & 0x80000000));
  const float rad = __fsqrt_rn(fadd(fmul(l, l), fmul(r_, r_)));  // utils/dsp.py:413
  const float rt = rad * th;
  a.sr += rad;
  a.srt += rt;
  a.srt2 = fmaf(rt, th, a.srt2);
  a.srt3 = fmaf(rt * th, th, a.srt3);
  a.slr = fmaf(l, r_, a.slr);
  a.sll = fmaf(l, l, a.sll);
  if (s >= 0.0f) track_ratio(ad, as, a.d_pos, a.s_pos);
  else track_ratio(ad, as, a.d_neg, a.s_neg);
}

// Two frames at once with packed arithmetic - the inner loop of vn_objective_kernel and vn_stereo_objective_kernel.
// The amplitude-weighted sums run in two interleaved chains per lane (even / odd frames, slot [0] / [1]), added
// together before the warp reduction; the ratio trackers stay scalar and see the frames in order.
//
// Instruction diet (ncu, round 2: ~93 of the ~116 instructions a frame-evaluation costs are these moments, not the
// taps): the radius uses sqrt.approx (2 ulp; it only enters amplitude-weighted sums, whose weights make 1e-7 relative
// irrelevant; it flushes subnormal squares, whose frames take the rare path below), min/max uses rcp.approx on a
// denominator clamped to FLT_MIN instead of div.approx's denormal scaling (frames below 1e-38 carry no weight), and the
// exact max|theta| tracker is entered through ONE test per pair on a
// key that is monotone in |d|/|s| (key = t or 2 - t with t = min/max): a frame can only beat the record if its key is
// within the key's rounding error (< 1e-6) of the record's.
struct LaneAcc2 {
  float sr[2], srt[2], srt2[2], srt3[2], slr[2], sll[2];
  float d_pos, s_pos, d_neg, s_neg;
  float k_pos, k_neg;  // key of the recorded frame minus the safety margin; -1 before the first record
};
constexpr float kKeyMargin = 2e-6f;

__device__ __forceinline__ float obj_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float obj_sqrt(float x) {  // flushes a subnormal x to 0
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float obj_sqrt_keep(float x) {  // a subnormal x keeps its root (a few more instructions)
  float y;
  asm("sqrt.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float obj_theta(float t, float p, bool steep, float d, float s) {
  float th = p * t;
  if (steep) th = 1.57079632679489662f - th;
  return __int_as_float(__float_as_int(th) | ((__float_as_int(d) ^ __float_as_int(s)) & 0x80000000));
}

// exact record update for one frame (the rare path behind the key test)
__device__ __forceinline__ void track_exact(LaneAcc2& a, float ad, float as, float key, bool pos) {
  if (pos) {
    if ((double)ad * (double)a.s_pos > (double)a.d_pos * (double)as) {  // ties keep the earlier frame
      a.d_pos = ad;
      a.s_pos = as;
      a.k_pos = key - kKeyMargin;
    }
  } else {
    if ((double)ad * (double)a.s_neg > (double)a.d_neg * (double)as) {
      a.d_neg = ad;
      a.s_neg = as;
      a.k_neg = key - kKeyMargin;
    }
  }
}

// the r-weighted terms of a radius into chain c of the sums, as lane_acc_pair adds them
__device__ __forceinline__ void obj_add_radius(LaneAcc2& a, int c, float rad, float th) {
  const float rt = rad * th;
  a.sr[c] += rad;
  a.srt[c] += rt;
  a.srt2[c] = fmaf(rt, th, a.srt2[c]);
  a.srt3[c] = fmaf(rt * th, th, a.srt3[c]);
}

__device__ __forceinline__ void lane_acc_pair(LaneAcc2& a, float l0, float l1, float r0, float r1) {
  constexpr float kTiny = 1.17549435e-38f;  // FLT_MIN
  float d0 = l0, d1 = l1, s0 = l0, s1 = l1;
  obj_sub2(d0, d1, r0, r1);  // utils/dsp.py:399-401
  obj_add2(s0, s1, r0, r1);
  const float ad0 = fabsf(d0), as0 = fabsf(s0), ad1 = fabsf(d1), as1 = fabsf(s1);
  const float mx0 = fmaxf(ad0, as0), mn0 = fminf(ad0, as0), mx1 = fmaxf(ad1, as1), mn1 = fminf(ad1, as1);
  const float t0 = mn0 * obj_rcp(fmaxf(mx0, kTiny)), t1 = mn1 * obj_rcp(fmaxf(mx1, kTiny));
  const bool steep0 = ad0 > as0, steep1 = ad1 > as1;
  float z0 = t0, z1 = t1;
  obj_mul2(z0, z1, t0, t1);
  float p0 = 0.00245671847107214f, p1 = p0;  // atan01's polynomial on both frames
  obj_fma2(p0, p1, z0, z1, -0.01440133168500584f, -0.01440133168500584f);
  obj_fma2(p0, p1, z0, z1, 0.03978117728736144f, 0.03978117728736144f);
  obj_fma2(p0, p1, z0, z1, -0.07234853052703884f, -0.07234853052703884f);
  obj_fma2(p0, p1, z0, z1, 0.10498943808759016f, 0.10498943808759016f);
  obj_fma2(p0, p1, z0, z1, -0.14161228535203682f, -0.14161228535203682f);
  obj_fma2(p0, p1, z0, z1, 0.19985906672823953f, 0.19985906672823953f);
  obj_fma2(p0, p1, z0, z1, -0.3333259702410447f, -0.3333259702410447f);
  obj_fma2(p0, p1, z0, z1, 0.9999998863844667f, 0.9999998863844667f);
  const float th0 = obj_theta(t0, p0, steep0, d0, s0), th1 = obj_theta(t1, p1, steep1, d1, s1);
  float q0 = l0, q1 = l1, w0 = r0, w1 = r1;  // utils/dsp.py:413: sqrt(l*l + r*r), products rounded separately
  obj_mul2(q0, q1, l0, l1);
  obj_mul2(w0, w1, r0, r1);
  obj_add2(q0, q1, w0, w1);
  const float rad0 = obj_sqrt(q0), rad1 = obj_sqrt(q1);
  float rt0 = rad0, rt1 = rad1;
  obj_mul2(rt0, rt1, th0, th1);
  obj_add2(a.sr[0], a.sr[1], rad0, rad1);
  obj_add2(a.srt[0], a.srt[1], rt0, rt1);
  float u0 = rt0, u1 = rt1;
  obj_fma2(u0, u1, th0, th1, a.srt2[0], a.srt2[1]);
  a.srt2[0] = u0;
  a.srt2[1] = u1;
  obj_mul2(rt0, rt1, th0, th1);
  obj_fma2(rt0, rt1, th0, th1, a.srt3[0], a.srt3[1]);
  a.srt3[0] = rt0;
  a.srt3[1] = rt1;
  float v0 = l0, v1 = l1;
  obj_fma2(v0, v1, r0, r1, a.slr[0], a.slr[1]);
  a.slr[0] = v0;
  a.slr[1] = v1;
  v0 = l0;
  v1 = l1;
  obj_fma2(v0, v1, l0, l1, a.sll[0], a.sll[1]);
  a.sll[0] = v0;
  a.sll[1] = v1;
  // max|theta| candidates: one test per pair.  Frames whose root came out 0 always take the rare path: their key is
  // meaningless when max(|d|, |s|) < FLT_MIN (then l*l + r*r is 0), and a subnormal l*l + r*r (|l|, |r| below ~1e-19)
  // was flushed by sqrt.approx.ftz: its radius is taken again there with subnormals kept and added to the sums right
  // behind the 0 that stood for it, which gives the bits the kept radius would have given in place.
  const float k0 = steep0 ? 2.0f - t0 : t0, k1 = steep1 ? 2.0f - t1 : t1;
  const bool pos0 = s0 >= 0.0f, pos1 = s1 >= 0.0f;
  const bool hit0 = k0 >= (pos0 ? a.k_pos : a.k_neg) || rad0 == 0.0f, hit1 = k1 >= (pos1 ? a.k_pos : a.k_neg) || rad1 == 0.0f;
  if (hit0 || hit1) {
    if (rad0 == 0.0f) obj_add_radius(a, 0, obj_sqrt_keep(q0), th0);
    if (rad1 == 0.0f) obj_add_radius(a, 1, obj_sqrt_keep(q1), th1);
    if (hit0) track_exact(a, ad0, as0, k0, pos0);
    if (k1 >= (pos1 ? a.k_pos : a.k_neg) || rad1 == 0.0f) track_exact(a, ad1, as1, k1, pos1);  // against the record frame 0 may just have set
  }
}

// (hi, lo) += v with hi + lo exact (TwoSum, then renormalised so that |lo| <= ulp(hi) / 2).  Every operation is exact
// while the addends are float32 values (or such sums) spanning fewer than about 70 binades, so the pair holds the exact
// sum and hi + lo rounds it once, whatever the order of the additions (DESIGN.md section 6).
__device__ __forceinline__ void dd_add(double& hi, double& lo, double v) {
  const double s = hi + v, vb = s - hi;
  const double e = (hi - (s - vb)) + (v - vb);
  const double t = lo + e;
  hi = s + t;
  const double tb = hi - s;
  lo = (s - (hi - tb)) + (t - tb);
}

// A candidate's accumulators (OBJ_CHUNK_SLOTS doubles) as a CTA starts: sums zero, ratio trackers at 0 / 1.
__device__ __forceinline__ double obj_acc_init(int slot) { return (slot == 7 || slot == 9) ? 1.0 : 0.0; }

// One tile's warp-reduced lane sums into a candidate's accumulators q (lane 0 of the warp).
__device__ __forceinline__ void obj_acc_tile(double* q, const LaneAcc& a, int nvalid) {
  dd_add(q[0], q[12], (double)a.sr);
  dd_add(q[1], q[13], (double)a.srt);
  dd_add(q[2], q[14], (double)a.srt2);
  dd_add(q[3], q[15], (double)a.srt3);
  dd_add(q[4], q[16], (double)a.slr);
  dd_add(q[5], q[17], (double)a.sll);
  if ((double)a.d_pos * q[7] > q[6] * (double)a.s_pos) { q[6] = a.d_pos; q[7] = a.s_pos; }
  if ((double)a.d_neg * q[9] > q[8] * (double)a.s_neg) { q[8] = a.d_neg; q[9] = a.s_neg; }
  q[10] += (double)nvalid;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// best ratio across the warp: every lane ends with the same (d, s)
__device__ __forceinline__ void warp_best_ratio(float& d, float& s) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float od = __shfl_xor_sync(0xffffffffu, d, o);
    const float os = __shfl_xor_sync(0xffffffffu, s, o);
    const double lhs = (double)od * (double)s, rhs = (double)d * (double)os;  // exact products
    if (lhs > rhs || (lhs == rhs && od > d)) { d = od; s = os; }
  }
}

template <int R>
__device__ __forceinline__ void run_candidate(const float* __restrict__ px, const int* __restrict__ prog, int apply_gain, float (&yv)[R]) {
#pragma unroll
  for (int r = 0; r < R; ++r) yv[r] = 0.0f;
  const int S = prog[0];
  const int* seg = prog + 1;
  const int* tp = prog + 1 + 3 * S;
  for (int s = 0; s < S; ++s) {
    const int n_neg = seg[3 * s], n_pos = seg[3 * s + 1];
    const float gain = __int_as_float(seg[3 * s + 2]);
    float acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = 0.0f;
    for (int k = 0; k < n_neg; ++k) {
      const float* q = px + tp[k];
#pragma unroll
      for (int r = 0; r < R; r += 2) obj_sub2(acc[r], acc[r + 1], q[32 * r], q[32 * r + 32]);
    }
    tp += n_neg;
    for (int k = 0; k < n_pos; ++k) {
      const float* q = px + tp[k];
#pragma unroll
      for (int r = 0; r < R; r += 2) obj_add2(acc[r], acc[r + 1], q[32 * r], q[32 * r + 32]);
    }
    tp += n_pos;
    if (apply_gain) {
#pragma unroll
      for (int r = 0; r < R; r += 2) obj_mul2(acc[r], acc[r + 1], gain, gain);
    }
#pragma unroll
    for (int r = 0; r < R; r += 2) obj_add2(yv[r], yv[r + 1], acc[r], acc[r + 1]);
  }
}

// Whole tiles: a lane owns OBJ_R / 4 groups of FOUR CONSECUTIVE frames (frames base + 128 j + 4 lane + e),
// and the filtered channel is staged four times, copy c shifted by c samples, so that every tap finds a
// copy in which its operands are 16-byte aligned: one LDS.128 per group and tap instead of four LDS.32
// (same shared-memory wavefronts, a quarter of the load instructions).  `dec` holds the program's taps
// decoded once per candidate as word offsets (offset & 3) * span4 + (offset & ~3) into the copies.
// One segment at a time: two decay segments interleaved per warp, as in fir_ring_kernel, need 128 registers (16 warps)
// and measured 129 k against 156 k evaluations/s on 16 clips x 1024 strengths x 30 s (B200): the warps they cost matter
// more to the polar moments.  Code removed; last present at commit 915ac5a.
template <int R, bool SUB>
__device__ __forceinline__ void obj_tap_v4(const float* __restrict__ px, int off, float (&acc)[R]) {
  const float4* q = reinterpret_cast<const float4*>(px + off);
#pragma unroll
  for (int j = 0; j < R / 4; ++j) {
    const float4 v = q[32 * j];
    if constexpr (SUB) {
      obj_sub2(acc[4 * j], acc[4 * j + 1], v.x, v.y);
      obj_sub2(acc[4 * j + 2], acc[4 * j + 3], v.z, v.w);
    } else {
      obj_add2(acc[4 * j], acc[4 * j + 1], v.x, v.y);
      obj_add2(acc[4 * j + 2], acc[4 * j + 3], v.z, v.w);
    }
  }
}
template <int R>
__device__ __forceinline__ void run_candidate_v4(const float* __restrict__ px, const int* __restrict__ prog, const int* __restrict__ dec,
                                                 int apply_gain, float (&yv)[R]) {
#pragma unroll
  for (int r = 0; r < R; ++r) yv[r] = 0.0f;
  const int S = prog[0];
  const int* seg = prog + 1;
  const int* tp = dec;
  for (int s = 0; s < S; ++s) {
    const int n_neg = seg[3 * s], n_pos = seg[3 * s + 1];
    const float gain = __int_as_float(seg[3 * s + 2]);
    float acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = 0.0f;
    int nxt = tp[0];  // offsets are read one tap ahead (a word of slack follows the decoded list)
    for (int k = 0; k < n_neg; ++k) {
      const int off = nxt;
      nxt = tp[k + 1];
      obj_tap_v4<R, true>(px, off, acc);
    }
    tp += n_neg;
    for (int k = 0; k < n_pos; ++k) {
      const int off = nxt;
      nxt = tp[k + 1];
      obj_tap_v4<R, false>(px, off, acc);
    }
    tp += n_pos;
    if (apply_gain) {
#pragma unroll
      for (int r = 0; r < R; r += 2) obj_mul2(acc[r], acc[r + 1], gain, gain);
    }
#pragma unroll
    for (int r = 0; r < R; r += 2) obj_add2(yv[r], yv[r + 1], acc[r], acc[r + 1]);
  }
}

// Shared memory: float x0[4][span4] (copy c = channel 0 shifted by c samples) | float x1[TILE] |
//                double acc[cand_per_group][OBJ_CHUNK_SLOTS] | int prog[warps][max_prog_words] | int dec[warps][max_prog_words]
#ifndef VND_OBJ_MINB
#define VND_OBJ_MINB 1  // CTAs per SM the register and shared-memory budgets are planned for (measured: 16 frames per lane in one CTA beats 8 in two)
#endif
// Work-item sources of vn_objective_kernel.  A CTA scores the tiles [tile_first, tile_first + n_tiles) of one clip (the
// loop stops at the clip's end) on the candidates [cand0, cand0 + ncand) of the program, and writes ncand x OBJ_CHUNK_SLOTS
// chunk partials to out.  Tiles are counted from frame 0 of the clip and staging reads nothing past the clip's last
// frame, so a (clip, candidate) pair gives the same bits whichever source hands it out.  Each field is asked for
// where the kernel needs it.
//
// grid (chunk, clip, group) over n_clips equal-length planar clips sharing one candidate list
struct ObjGridSrc {
  ObjParams p;
  __device__ __forceinline__ int cand0() const { return blockIdx.z * p.cand_per_group; }
  __device__ __forceinline__ int ncand(int cand0) const { return min(p.cand_per_group, p.n_cand - cand0); }
  __device__ __forceinline__ const float* x0() const { return p.clips + (long long)blockIdx.y * p.clip_stride; }
  __device__ __forceinline__ long long frames() const { return p.frames; }
  __device__ __forceinline__ long long tile_first() const { return (long long)blockIdx.x * p.tiles_per_chunk; }
  __device__ __forceinline__ int n_tiles() const { return p.tiles_per_chunk; }
  __device__ __forceinline__ double* out(int cand0) const {
    return p.chunk_partials + (((size_t)blockIdx.y * p.n_chunks + blockIdx.x) * p.n_cand + cand0) * OBJ_CHUNK_SLOTS;
  }
};

// CTA blockIdx.x runs work item items[blockIdx.x] (built on the host by plan_runs) over ragged clips packed
// channel-planar: element (t, c) of a clip is p.clips[c * chan_stride + base + t]
struct ObjRunSrc {
  ObjParams p;
  const ObjRunItem* items;
  __device__ __forceinline__ int cand0() const { return items[blockIdx.x].cand0; }
  __device__ __forceinline__ int ncand(int) const { return items[blockIdx.x].ncand; }
  __device__ __forceinline__ const float* x0() const { return p.clips + items[blockIdx.x].base; }
  __device__ __forceinline__ long long frames() const { return items[blockIdx.x].frames; }
  __device__ __forceinline__ long long tile_first() const { return items[blockIdx.x].tile_first; }
  __device__ __forceinline__ int n_tiles() const { return items[blockIdx.x].n_tiles; }
  __device__ __forceinline__ double* out(int) const { return p.chunk_partials + (size_t)items[blockIdx.x].part * OBJ_CHUNK_SLOTS; }
};

template <typename Src>
__global__ void __launch_bounds__(OBJ_NT, VND_OBJ_MINB) vn_objective_kernel(const Src src, int max_prog_words) {
  const ObjParams& p = src.p;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int span = OBJ_TILE + p.halo;
  const int span4 = (span + 7) & ~3;  // words per shifted copy (a multiple of 4, room for the shift)
  float* s0 = reinterpret_cast<float*>(smem_raw);
  float* s1 = s0 + 4 * span4;
  double* acc = reinterpret_cast<double*>(s1 + OBJ_TILE);
  int* progs = reinterpret_cast<int*>(acc + (size_t)p.cand_per_group * OBJ_CHUNK_SLOTS);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int kWarps = OBJ_NT / 32;
  const int cand0 = src.cand0();
  const int ncand = src.ncand(cand0);
  const float* __restrict__ x0 = src.x0();
  const float* __restrict__ x1 = x0 + p.chan_stride;
  int* myprog = progs + warp * max_prog_words;
  int* mydec = progs + (kWarps + warp) * max_prog_words;

  for (int i = tid; i < ncand * OBJ_CHUNK_SLOTS; i += OBJ_NT) acc[i] = obj_acc_init(i % OBJ_CHUNK_SLOTS);

  const long long tile_first = src.tile_first();
  for (int ti = 0; ti < src.n_tiles(); ++ti) {
    const long long t0 = (tile_first + ti) * OBJ_TILE;
    if (t0 >= src.frames()) break;
    const long long remain = src.frames() - t0;
    __syncthreads();  // previous tile fully consumed (also orders the acc init)
    for (int i = tid; i < span + 3; i += OBJ_NT) {  // copy c holds x0[t0 + c + j] at j
      const float v = i < remain ? x0[t0 + i] : 0.0f;
      if (i < span) s0[i] = v;
      if (i >= 1 && i - 1 < span) s0[span4 + i - 1] = v;
      if (i >= 2 && i - 2 < span) s0[2 * span4 + i - 2] = v;
      if (i >= 3) s0[3 * span4 + i - 3] = v;
    }
    for (int i = tid; i < OBJ_TILE; i += OBJ_NT) s1[i] = i < remain ? x1[t0 + i] : 0.0f;
    __syncthreads();
    const int nvalid = (int)(remain < OBJ_TILE ? remain : OBJ_TILE);

    for (int ci = warp; ci < ncand; ci += kWarps) {
      const int w0 = p.offsets[cand0 + ci];
      const int nprog = p.offsets[cand0 + ci + 1] - w0;
      __syncwarp();
      for (int i = lane; i < nprog; i += 32) myprog[i] = p.words[w0 + i];
      __syncwarp();
      {  // taps as word offsets into the shifted copies
        const int ntap0 = 1 + 3 * myprog[0];
        for (int i = ntap0 + lane; i < nprog; i += 32) {
          const int off = myprog[i];
          mydec[i - ntap0] = (off & 3) * span4 + (off & ~3);
        }
      }
      __syncwarp();
      LaneAcc a{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 1.f, 0.f, 1.f};
      if (nvalid == OBJ_TILE) {  // whole tile: no bounds checks, frames in packed pairs
        LaneAcc2 b{{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, 0.f, 1.f, 0.f, 1.f, -1.f, -1.f};
        for (int base = 0; base < OBJ_TILE; base += 32 * OBJ_R) {
          float yv[OBJ_R];
          run_candidate_v4<OBJ_R>(s0 + base + 4 * lane, myprog, mydec, p.apply_gain, yv);
          const float4* r1 = reinterpret_cast<const float4*>(s1 + base + 4 * lane);
#pragma unroll
          for (int j = 0; j < OBJ_R / 4; ++j) {
            const float4 v = r1[32 * j];
            lane_acc_pair(b, yv[4 * j], yv[4 * j + 1], v.x, v.y);
            lane_acc_pair(b, yv[4 * j + 2], yv[4 * j + 3], v.z, v.w);
          }
        }
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
      } else {
        for (int base = 0; base < nvalid; base += 32 * OBJ_R) {
          float yv[OBJ_R];
          run_candidate<OBJ_R>(s0 + base + lane, myprog, p.apply_gain, yv);
#pragma unroll
          for (int r = 0; r < OBJ_R; ++r) {
            const int i = base + lane + 32 * r;
            if (i < nvalid) lane_acc_frame(a, yv[r], s1[i]);
          }
        }
      }
      a.sr = warp_sum(a.sr);
      a.srt = warp_sum(a.srt);
      a.srt2 = warp_sum(a.srt2);
      a.srt3 = warp_sum(a.srt3);
      a.slr = warp_sum(a.slr);
      a.sll = warp_sum(a.sll);
      warp_best_ratio(a.d_pos, a.s_pos);
      warp_best_ratio(a.d_neg, a.s_neg);
      if (lane == 0) obj_acc_tile(acc + (size_t)ci * OBJ_CHUNK_SLOTS, a, nvalid);
    }
  }
  __syncthreads();
  double* out = src.out(cand0);
  for (int i = tid; i < ncand * OBJ_CHUNK_SLOTS; i += OBJ_NT) out[i] = acc[i];
}

// Fixed-order combine of the chunk partials (OBJ_CHUNK_SLOTS doubles each): the double-double sums added chunk by
// chunk, high then low part, and rounded once to double at the end; ratio trackers by exact cross multiplication
// (earlier chunk wins ties, like np.max keeps the value either way).  Chunk ch of the row is q[ch * stride]; the row
// written to o has OBJ_SLOTS doubles.
__device__ __forceinline__ void obj_combine_row(const double* __restrict__ q, size_t stride, int n_chunks, double* __restrict__ o) {
  double r[OBJ_CHUNK_SLOTS];
  for (int k = 0; k < OBJ_CHUNK_SLOTS; ++k) r[k] = obj_acc_init(k);
  for (int ch = 0; ch < n_chunks; ++ch, q += stride) {
    for (int k = 0; k < 6; ++k) {
      dd_add(r[k], r[12 + k], q[k]);
      dd_add(r[k], r[12 + k], q[12 + k]);
    }
    if (q[6] * r[7] > r[6] * q[7]) { r[6] = q[6]; r[7] = q[7]; }
    if (q[8] * r[9] > r[8] * q[9]) { r[8] = q[8]; r[9] = q[9]; }
    r[10] += q[10];
  }
  for (int k = 0; k < 6; ++k) o[k] = r[k] + r[12 + k];
  for (int k = 6; k < OBJ_SLOTS; ++k) o[k] = r[k];
}

__global__ void obj_combine_kernel(const double* __restrict__ chunk_partials, double* __restrict__ partials, int n_clips,
                                   int n_chunks, int n_cand) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)n_clips * n_cand) return;
  const int clip = (int)(idx / n_cand), cand = (int)(idx % n_cand);
  obj_combine_row(chunk_partials + ((size_t)clip * n_chunks * n_cand + cand) * OBJ_CHUNK_SLOTS, (size_t)n_cand * OBJ_CHUNK_SLOTS, n_chunks,
                  partials + (size_t)idx * OBJ_SLOTS);
}

// The combine of the run-list objective: CTA r combines run r's rows.  Its chunk partials are [chunk][candidate] from
// row `part`, chunks in tile order.
struct ObjRunCombine {
  long long part, out;
  int n_chunks, count;
};

__global__ void obj_combine_runs_kernel(const double* __restrict__ chunk_partials, double* __restrict__ partials,
                                        const ObjRunCombine* __restrict__ runs) {
  const ObjRunCombine r = runs[blockIdx.x];
  for (int j = threadIdx.x; j < r.count; j += blockDim.x)
    obj_combine_row(chunk_partials + (size_t)(r.part + j) * OBJ_CHUNK_SLOTS, (size_t)r.count * OBJ_CHUNK_SLOTS, r.n_chunks,
                    partials + (size_t)(r.out + j) * OBJ_SLOTS);
}

int obj_combine_launch(const double* chunk_partials, double* partials, int n_clips, int n_chunks, int n_cand, cudaStream_t st) {
  const long long pairs = (long long)n_clips * n_cand;
  obj_combine_kernel<<<(unsigned)ceil_div<long long>(pairs, 128), 128, 0, st>>>(chunk_partials, partials, n_clips, n_chunks, n_cand);
  return after_launch("obj_combine_kernel");
}

// ------------------------------------------------------------------------------------------------
// Velvet-noise stereo candidates (vnd_vn_stereo_objective_dev): VelvetNoise with two outputs and no normaliser, any
// filtered channels, LR or MS, any width.  The score of such a candidate is today's two-step one: decorrelate (the
// fused vn_stereo_kernel: FIR of both channels, unfiltered ones copied, then ms_width_epilogue) and the objective of
// its float32 output with the one-tap identity program.  This kernel computes each candidate's output in registers and
// feeds the moments exactly as vn_objective_kernel sees the materialised output: the left value through the identity
// program's two adds (0 + (0 + y0), which turns -0 into +0), the right value as it is, whole tiles with lane l owning
// the four consecutive frames 128 j + 4 l + e and lane_acc_pair, the last partial tile with frames base + lane + 32 r
// and lane_acc_frame, and the chunks of the one-candidate plan (plan_objective for the identity program) combined by
// obj_combine_kernel.  The per-tile float32 lane sums and the double-double chunk sums therefore see the same values in
// the same order.
//
// The output is computed in the conflict-free layout (lane owns frames base + lane + 32 r, plain LDS per tap, as
// vn_stereo_kernel reads) and passed through a per-warp scratch row into the four-consecutive-frames layout.
// Shared memory: float x0[span] | float x1[span] | float scratch[warps][2][32 OBJ_R] | double acc[cand_per_group][OBJ_CHUNK_SLOTS]
//                | int prog[warps][2 max_prog_words]
// ------------------------------------------------------------------------------------------------
#ifndef VND_OBJ_STEREO_NT
#define VND_OBJ_STEREO_NT 512  // 16 warps: 128 registers a thread (the two channels' taps and outputs of a pass)
#endif
struct VnStereoObjParams {
  const float* x;  // channel 0; channel 1 at x + chan_stride
  long long frames, chan_stride;
  const int* words;
  const int* offsets;  // candidate j: channels 2 j and 2 j + 1
  const vnd_vn_stereo_cand* cands;
  int n_cand, apply_gain, halo, cand_per_group, tiles_per_chunk;
  double* chunk_partials;  // [chunk][cand][OBJ_CHUNK_SLOTS]
};

// One pass of one candidate: its output (l, r) at frames i0 + 32 rr of the staged tile.  With kGain the output is scaled
// by candidate c's rms_normalize gains g[2 c], g[2 c + 1] as place_kernel scales the stored output.  They are read here,
// per pass, through a pointer without __restrict__: loads the compiler may hoist out of the pass loop hold two more
// registers across it, and those spill.
template <bool kGain>
__device__ __forceinline__ void stereo_candidate_pass(const float* __restrict__ s0, const float* __restrict__ s1, int i0, const int* __restrict__ prog,
                                                      int n0, int n1, const vnd_vn_stereo_cand& cd, int apply_gain, const float* g,
                                                      int c, float (&l)[OBJ_R], float (&r)[OBJ_R]) {
  if (n0 > 0) run_candidate<OBJ_R>(s0 + i0, prog, apply_gain, l);
  if (n1 > 0) run_candidate<OBJ_R>(s1 + i0, prog + n0, apply_gain, r);
  float g0 = 1.0f, g1 = 1.0f;
  if constexpr (kGain) {
    g0 = g[2 * c];
    g1 = g[2 * c + 1];
  }
#pragma unroll
  for (int k = 0; k < OBJ_R; ++k) {
    const float a = s0[i0 + 32 * k], b = s1[i0 + 32 * k];
    float u = n0 > 0 ? l[k] : a;  // unfiltered channel: copied through
    float v = n1 > 0 ? r[k] : b;
    ms_width_epilogue(a, b, u, v, cd.ms_encode, cd.use_width, cd.w_mid, cd.w_side);
    if constexpr (kGain) {
      u = fmul(u, g0);
      v = fmul(v, g1);
    }
    l[k] = fadd(0.0f, fadd(0.0f, u));  // the identity program's segment sum and running output
    r[k] = v;
  }
}

// kGain: candidate j's output is scaled by its rms_normalize gains gains[2 j], gains[2 j + 1].  The gains come as a
// parameter of their own behind the others, so that the kernel without them reads its parameters at the same offsets.
template <bool kGain>
__global__ void __launch_bounds__(VND_OBJ_STEREO_NT, 1) vn_stereo_objective_kernel(const VnStereoObjParams p, int max_prog_words,
                                                                                   const float* gains) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int kWarps = VND_OBJ_STEREO_NT / 32;
  constexpr int kPass = 32 * OBJ_R;
  const int span = OBJ_TILE + p.halo;
  const int span_al = (span + 3) & ~3;
  float* s0 = reinterpret_cast<float*>(smem_raw);
  float* s1 = s0 + span_al;
  float* scratch = s1 + span_al;
  double* acc = reinterpret_cast<double*>(scratch + kWarps * 2 * kPass);
  int* progs = reinterpret_cast<int*>(acc + (size_t)p.cand_per_group * OBJ_CHUNK_SLOTS);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cand0 = blockIdx.y * p.cand_per_group;
  const int ncand = min(p.cand_per_group, p.n_cand - cand0);
  const float* __restrict__ x0 = p.x;
  const float* __restrict__ x1 = p.x + p.chan_stride;
  float* my0 = scratch + warp * 2 * kPass;
  float* my1 = my0 + kPass;
  int* myprog = progs + warp * 2 * max_prog_words;

  for (int i = tid; i < ncand * OBJ_CHUNK_SLOTS; i += VND_OBJ_STEREO_NT) acc[i] = obj_acc_init(i % OBJ_CHUNK_SLOTS);

  for (int ti = 0; ti < p.tiles_per_chunk; ++ti) {
    const long long t0 = ((long long)blockIdx.x * p.tiles_per_chunk + ti) * OBJ_TILE;
    if (t0 >= p.frames) break;
    const long long remain = p.frames - t0;
    __syncthreads();  // previous tile fully consumed (also orders the acc init)
    for (int i = tid; i < span; i += VND_OBJ_STEREO_NT) {
      s0[i] = i < remain ? x0[t0 + i] : 0.0f;
      s1[i] = i < remain ? x1[t0 + i] : 0.0f;
    }
    __syncthreads();
    const int nvalid = (int)(remain < OBJ_TILE ? remain : OBJ_TILE);

    for (int ci = warp; ci < ncand; ci += kWarps) {
      const int c = cand0 + ci;
      const int w0 = p.offsets[2 * c];
      const int n0 = p.offsets[2 * c + 1] - w0;
      const int n1 = p.offsets[2 * c + 2] - w0 - n0;
      __syncwarp();
      for (int i = lane; i < n0 + n1; i += 32) myprog[i] = p.words[w0 + i];
      __syncwarp();
      const vnd_vn_stereo_cand cd = p.cands[c];
      LaneAcc a{0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 1.f, 0.f, 1.f};
      if (nvalid == OBJ_TILE) {  // whole tile: lane owns frames base + 128 j + 4 lane + e, in packed pairs
        LaneAcc2 b{{0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, {0.f, 0.f}, 0.f, 1.f, 0.f, 1.f, -1.f, -1.f};
        for (int base = 0; base < OBJ_TILE; base += kPass) {
          float l[OBJ_R], r[OBJ_R];
          stereo_candidate_pass<kGain>(s0, s1, base + lane, myprog, n0, n1, cd, p.apply_gain, gains, c, l, r);
          __syncwarp();  // the previous pass has read the scratch row
#pragma unroll
          for (int k = 0; k < OBJ_R; ++k) {
            my0[lane + 32 * k] = l[k];
            my1[lane + 32 * k] = r[k];
          }
          __syncwarp();
          const float4* q0 = reinterpret_cast<const float4*>(my0 + 4 * lane);
          const float4* q1 = reinterpret_cast<const float4*>(my1 + 4 * lane);
#pragma unroll
          for (int j = 0; j < OBJ_R / 4; ++j) {
            const float4 u = q0[32 * j], v = q1[32 * j];
            lane_acc_pair(b, u.x, u.y, v.x, v.y);
            lane_acc_pair(b, u.z, u.w, v.z, v.w);
          }
        }
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
      } else {
        for (int base = 0; base < nvalid; base += kPass) {
          float l[OBJ_R], r[OBJ_R];
          stereo_candidate_pass<kGain>(s0, s1, base + lane, myprog, n0, n1, cd, p.apply_gain, gains, c, l, r);
#pragma unroll
          for (int k = 0; k < OBJ_R; ++k) {
            const int i = base + lane + 32 * k;
            if (i < nvalid) lane_acc_frame(a, l[k], r[k]);
          }
        }
      }
      a.sr = warp_sum(a.sr);
      a.srt = warp_sum(a.srt);
      a.srt2 = warp_sum(a.srt2);
      a.srt3 = warp_sum(a.srt3);
      a.slr = warp_sum(a.slr);
      a.sll = warp_sum(a.sll);
      warp_best_ratio(a.d_pos, a.s_pos);
      warp_best_ratio(a.d_neg, a.s_neg);
      if (lane == 0) obj_acc_tile(acc + (size_t)ci * OBJ_CHUNK_SLOTS, a, nvalid);
    }
  }
  __syncthreads();
  double* out = p.chunk_partials + ((size_t)blockIdx.x * p.n_cand + cand0) * OBJ_CHUNK_SLOTS;
  for (int i = tid; i < ncand * OBJ_CHUNK_SLOTS; i += VND_OBJ_STEREO_NT) out[i] = acc[i];
}

// ------------------------------------------------------------------------------------------------
// rms_normalize gains of velvet-noise stereo candidates (vnd_vn_stereo_rms_objective_dev).  decorrelate with the default
// normaliser scales channel c of its output y by sqrt(mean(x_c^2)) / sqrt(mean(y_c^2) + eps), where each sum of squares
// is numpy's strict left-to-right float32 running sum over the whole signal (SURVEY.md H1): a dependent chain of one
// rounded add per frame that no reordering may shorten.  This kernel runs those chains for G candidates per CTA at the
// cost of one: producer warps build each candidate's un-normalised output y with stereo_candidate_pass's arithmetic
// (run_candidate, ms_width_epilogue; the identity-program adds belong to the objective, not to y) and write the rounded
// squares of a sub-tile as rows [frame][2 G + 2] of a double-buffered array; one consumer warp walks the rows in frame
// order, lane 2 j + c adding candidate j's channel c and lanes 2 G, 2 G + 1 the two channels of x.  Rows have a pitch of
// 33 words, so the producers' writes (lane = frame) and the consumer's row reads (lane = column) are both conflict-free.
// The sums and gains are those of rms_gain_kernel after seq_sumsq_kernel on decorrelate's C-order (frames, 2) output.
// Shared memory: float x0[span] | float x1[span] | float sq[2][RMS_SUB][RMS_PITCH] | int prog[G][2 max_prog_words]
// ------------------------------------------------------------------------------------------------
constexpr int RMS_NT = 512;                 // 15 producer warps and the consumer warp
constexpr int RMS_PROD = RMS_NT / 32 - 1;
constexpr int RMS_MAX_G = 15;               // 2 G + 2 chains in the consumer warp
constexpr int RMS_SUB = 256;                // frames per squares buffer
constexpr int RMS_XTILE = 2048;             // frames per staged input tile (a multiple of RMS_SUB)
constexpr int RMS_PITCH = 33;
constexpr int RMS_R = 2;                    // frames per lane and unit: a unit is one candidate on 64 frames
constexpr int RMS_UNITS = RMS_SUB / (32 * RMS_R);  // units per candidate and sub-tile

struct VnRmsSumsParams {
  const float* x;  // channel 0; channel 1 at x + chan_stride
  long long frames, chan_stride;
  const int* words;
  const int* offsets;  // candidate j: channels 2 j and 2 j + 1
  const vnd_vn_stereo_cand* cands;
  int n_cand, apply_gain, halo, group;
  float* gains;  // 2 n_cand
};

__global__ void __launch_bounds__(RMS_NT, 1) vn_rms_sums_kernel(const VnRmsSumsParams p, int max_prog_words) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int span = RMS_XTILE + p.halo;
  const int span_al = (span + 3) & ~3;
  float* s0 = reinterpret_cast<float*>(smem_raw);
  float* s1 = s0 + span_al;
  float* sq = s1 + span_al;
  int* progs = reinterpret_cast<int*>(sq + 2 * RMS_SUB * RMS_PITCH);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int cand0 = blockIdx.x * p.group;
  const int ng = min(p.group, p.n_cand - cand0);
  const float* __restrict__ x0 = p.x;
  const float* __restrict__ x1 = p.x + p.chan_stride;
  for (int j = 0; j < ng; ++j) {
    const int w0 = p.offsets[2 * (cand0 + j)], n = p.offsets[2 * (cand0 + j) + 2] - w0;
    for (int i = tid; i < n; i += RMS_NT) progs[j * 2 * max_prog_words + i] = p.words[w0 + i];
  }
  __syncthreads();

  const long long nsub = ceil_div<long long>(p.frames, RMS_SUB);
  float chain = 0.0f;  // consumer lane 2 j + c: candidate j, channel c; lanes 2 ng, 2 ng + 1: x
  for (long long k = 0; k <= nsub; ++k) {
    if (warp < RMS_PROD) {
      if (k < nsub) {
        const int base = (int)(k % (RMS_XTILE / RMS_SUB)) * RMS_SUB;
        if (base == 0) {  // the previous __syncthreads ended every read of the old tile
          const long long t0 = k * RMS_SUB, remain = p.frames - t0;
          for (int i = tid; i < span; i += RMS_PROD * 32) {
            s0[i] = i < remain ? x0[t0 + i] : 0.0f;
            s1[i] = i < remain ? x1[t0 + i] : 0.0f;
          }
          asm volatile("bar.sync 1, %0;" ::"r"(RMS_PROD * 32) : "memory");
        }
        float* buf = sq + (k & 1) * (RMS_SUB * RMS_PITCH);
        for (int i = tid; i < RMS_SUB; i += RMS_PROD * 32) {
          const float a = s0[base + i], b = s1[base + i];
          buf[i * RMS_PITCH + 2 * ng] = fmul(a, a);
          buf[i * RMS_PITCH + 2 * ng + 1] = fmul(b, b);
        }
        for (int u = warp; u < ng * RMS_UNITS; u += RMS_PROD) {
          const int j = u / RMS_UNITS, c = cand0 + j;
          const int f0 = (u % RMS_UNITS) * 32 * RMS_R + lane;  // frames f0 + 32 k of the sub-tile
          const int n0 = p.offsets[2 * c + 1] - p.offsets[2 * c];
          const int n1 = p.offsets[2 * c + 2] - p.offsets[2 * c + 1];
          const int* prog = progs + j * 2 * max_prog_words;
          const vnd_vn_stereo_cand cd = p.cands[c];
          float l[RMS_R], r[RMS_R];
          if (n0 > 0) run_candidate<RMS_R>(s0 + base + f0, prog, p.apply_gain, l);
          if (n1 > 0) run_candidate<RMS_R>(s1 + base + f0, prog + n0, p.apply_gain, r);
#pragma unroll
          for (int q = 0; q < RMS_R; ++q) {
            const float a = s0[base + f0 + 32 * q], b = s1[base + f0 + 32 * q];
            float y0 = n0 > 0 ? l[q] : a;  // unfiltered channel: copied through
            float y1 = n1 > 0 ? r[q] : b;
            ms_width_epilogue(a, b, y0, y1, cd.ms_encode, cd.use_width, cd.w_mid, cd.w_side);
            float* row = buf + (f0 + 32 * q) * RMS_PITCH + 2 * j;
            row[0] = fmul(y0, y0);
            row[1] = fmul(y1, y1);
          }
        }
      }
    } else if (k > 0 && lane < 2 * ng + 2) {  // the consumer: sub-tile k - 1, rows past the last frame skipped
      const float* q = sq + ((k - 1) & 1) * (RMS_SUB * RMS_PITCH) + lane;
      const long long left = p.frames - (k - 1) * RMS_SUB;
      const int n = (int)(left < RMS_SUB ? left : RMS_SUB);
      int i = 0;
#pragma unroll 2
      for (; i + 8 <= n; i += 8) {
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = q[(i + e) * RMS_PITCH];
#pragma unroll
        for (int e = 0; e < 8; ++e) chain = fadd(chain, v[e]);
      }
      for (; i < n; ++i) chain = fadd(chain, q[i * RMS_PITCH]);
    }
    __syncthreads();
  }
  if (warp == RMS_PROD) {
    const float sx = __shfl_sync(0xffffffffu, chain, 2 * ng + (lane & 1));
    if (lane < 2 * ng) p.gains[2 * (long long)cand0 + lane] = rms_gain_f32(sx, chain, p.frames);
  }
}

// ------------------------------------------------------------------------------------------------
// Haas candidates: float64 throughout (optimization.py:183-203 builds LR-mode HaasEffects whose
// output is float64).  One CTA per (clip, candidate); 8 doubles per pair:
//   [sum r, sum r*th, sum r*th^2, sum r*th^3, max|th|, sum L*R, sum L*L, frames]
// ------------------------------------------------------------------------------------------------
constexpr int HAAS_SLOTS = 8;

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// The float64 pipe is what bounds this kernel (one atan2, one sqrt and the moments per frame and delay; the clip itself
// stays in L2 across its delays), so both functions are written out lean instead of calling the library versions with
// their special-case paths: ~45 instead of ~100 float64 instructions per frame.
//
// Folded angle (utils/dsp.py:399-412): atan2(d, s) brought into [-pi/2, pi/2] by adding or subtracting pi is atan(d / s)
// with the sign of d * s (sign of d alone for s == 0, 0 for d == s == 0).  |d| / |s| is reduced to |t| <= tan(pi/16) with
// one of the base angles 0, pi/8, pi/4 (after swapping so that the ratio is <= 1): atan(a / b) = base + atan((a - c b) /
// (b + c a)), c = tan(base); ten Taylor terms then leave < 1e-16.  The base is picked from float32 copies of a and b (any
// choice near a threshold is fine).  Explicit fma() throughout: nothing here is pinned to numpy's rounding (scores are
// compared at 1e-9), unlike the float32 paths of this library.
__device__ __forceinline__ double rcp_lean(double x) {  // x > 0, normal
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  r = fma(r, fma(-x, r, 1.0), r);
  r = fma(r, fma(-x, r, 1.0), r);
  return r;
}
__device__ __forceinline__ double sqrt_lean(double x) {  // x >= 0
  double r;
  asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  const double hx = 0.5 * x;
  r = fma(r, fma(-hx * r, r, 0.5), r);
  r = fma(r, fma(-hx * r, r, 0.5), r);
  return x > 0.0 ? x * r : 0.0;
}
__device__ __forceinline__ double abs_bits(double x) { return __hiloint2double(__double2hiint(x) & 0x7fffffff, __double2loint(x)); }
// d, s: the float64 difference and sum of the two channels; df, sf: float32 copies of them, only used to pick the
// reduction (which operand is larger, which base angle): any choice near a threshold is fine.
__device__ __forceinline__ double folded_angle(double d, double s, float df, float sf) {
  const double kC1 = 0.41421356237309503;  // tan(pi/8)
  const float fa = fabsf(df), fb = fabsf(sf);
  const bool inv = fa > fb;  // atan(a / b) = pi/2 - atan(b / a)
  const double ad = abs_bits(d), as = abs_bits(s);
  const double a = inv ? as : ad, b = inv ? ad : as;
  const float af = inv ? fb : fa, bf = inv ? fa : fb;
  const bool k1 = af > 0.19891237f * bf, k2 = af > 0.66817864f * bf;  // tan(pi/16), tan(3 pi/16)
  const double c = k2 ? 1.0 : (k1 ? kC1 : 0.0);
  const double base = k2 ? 0.7853981633974483 : (k1 ? 0.39269908169872414 : 0.0);
  const double num = fma(-c, b, a), den = fma(c, a, b);
  const double t = den > 0.0 ? num * rcp_lean(den) : 0.0;
  const double z = t * t;
  double p = -1.0 / 19.0;
  p = fma(p, z, 1.0 / 17.0);
  p = fma(p, z, -1.0 / 15.0);
  p = fma(p, z, 1.0 / 13.0);
  p = fma(p, z, -1.0 / 11.0);
  p = fma(p, z, 1.0 / 9.0);
  p = fma(p, z, -1.0 / 7.0);
  p = fma(p, z, 1.0 / 5.0);
  p = fma(p, z, -1.0 / 3.0);
  double th = base + fma(t * z, p, t);
  if (inv) th = 1.5707963267948966 - th;
  // sign of d * s (s == +-0 counts as positive: atan2(d, +-0) = sign(d) * pi/2)
  const int neg = (__double2hiint(d) ^ (s < 0.0 ? 0x80000000 : 0)) & 0x80000000;
  return __hiloint2double(__double2hiint(th) ^ neg, __double2loint(th));
}

struct HaasAcc {
  double v0 = 0, v1 = 0, v2 = 0, v3 = 0, v5 = 0, v6 = 0;
  long long vmax = 0;  // bits of max |theta| (non-negative doubles order like integers)
  __device__ __forceinline__ void add(double l, double r, float lf, float rf) {
    const double th = folded_angle(l - r, l + r, lf - rf, lf + rf);
    const double rad = sqrt_lean(fma(l, l, r * r));
    const double rt = rad * th, t2 = th * th;
    v0 += rad;
    v1 += rt;
    v2 = fma(rad, t2, v2);
    v3 = fma(rt, t2, v3);
    const long long ab = __double_as_longlong(th) & 0x7fffffffffffffffLL;
    vmax = ab > vmax ? ab : vmax;
    v5 = fma(l, r, v5);
    v6 = fma(l, l, v6);
  }
};

// Work-item sources of haas_objective_kernel: each CTA asks its source for one (clip, delay) item - the clip's two
// planar channels, its frame count, the delay and where its 8 partials go.  The body of the kernel is shared, so an
// item gives the same bits whichever source hands it out.
template <typename TIn>
struct HaasItem {
  const TIn* x0;  // channel 0 (the delayed one)
  const TIn* x1;  // channel 1
  long long frames;
  int d;
  double* out;  // HAAS_SLOTS doubles
};

// grid (cand, clip) over n_clips equal-length planar clips: element (clip, c, t) = clips[clip * clip_stride + c * chan_stride + t]
template <typename TIn>
struct HaasGridSrc {
  using T = TIn;
  const TIn* clips;
  long long frames, clip_stride, chan_stride;
  const int* delays;
  int n_cand;
  double* partials;  // (n_clips, n_cand, HAAS_SLOTS)
  __device__ __forceinline__ HaasItem<TIn> item() const {
    const int cand = blockIdx.x, clip = blockIdx.y;
    const TIn* x0 = clips + (long long)clip * clip_stride;
    return {x0, x0 + chan_stride, frames, delays[cand], partials + ((size_t)clip * n_cand + cand) * HAAS_SLOTS};
  }
};

// pair p = blockIdx.x of a flat (clip, delay) list over ragged clips packed channel-planar: element (t, c) of clip i is
// x[c * chan_stride + offs[i] + t]
struct HaasPairSrc {
  using T = float;
  const float* x;
  long long chan_stride;
  const long long* offs;
  const int* pair_clip;
  const int* pair_delay;
  double* partials;  // (n_pairs, HAAS_SLOTS)
  __device__ __forceinline__ HaasItem<float> item() const {
    const int p = blockIdx.x;
    const int clip = pair_clip[p];
    const long long o = offs[clip];
    return {x + o, x + chan_stride + o, offs[clip + 1] - o, pair_delay[p], partials + (size_t)p * HAAS_SLOTS};
  }
};

// candidate c = blockIdx.x: HaasEffect.decorrelate with the settings record cands[c] (any delayed channel, LR or MS, any
// width, mono or stereo) on one float32 channel-planar clip, element (t, ch) = x[ch * chan_stride + t].  Today's score
// of such a candidate is the objective of its float64 output z (frames + delay frames) as a delay-0 item, so frame m of
// z is built with haas_frame, as haas_kernel builds it, and fed with the striding of the delay-0 stretch.
struct HaasEffectSrc {
  using T = float;
  const float* x;
  long long frames, chan_stride;
  const vnd_haas_clip* cands;  // 16-byte aligned
  double* partials;            // (n_cand, HAAS_SLOTS)
};

template <typename Src>
struct haas_effect_src { static constexpr bool value = false; };
template <>
struct haas_effect_src<HaasEffectSrc> { static constexpr bool value = true; };

template <typename Src>
__global__ void __launch_bounds__(256) haas_objective_kernel(const Src src) {
  using TIn = typename Src::T;
  HaasAcc acc;
  long long total;
  double* out;
  if constexpr (haas_effect_src<Src>::value) {
    const int4* rec = reinterpret_cast<const int4*>(src.cands + blockIdx.x);
    const int4 w0 = __ldg(rec), w1 = __ldg(rec + 1);
    const int delay = w0.x, dch = w0.y, mode_ms = w0.z, mono = w0.w, use_width = w1.x;
    const double width = __hiloint2double(w1.w, w1.z);
    const long long L = src.frames;
    const float* __restrict__ x0 = src.x;
    const float* __restrict__ x1 = src.x + src.chan_stride;
    const int sh0 = dch == 0 ? delay : 0, sh1 = dch == 1 ? delay : 0;
    total = L + delay;
    out = src.partials + (size_t)blockIdx.x * HAAS_SLOTS;
    for (long long m = threadIdx.x; m < total; m += blockDim.x) {
      const long long q0 = m - sh0, q1 = m - sh1;
      const bool v0 = q0 >= 0 && q0 < L, v1 = q1 >= 0 && q1 < L;
      float a0 = 0.0f, b0 = 0.0f, a1 = 0.0f, b1 = 0.0f;
      if (v0) {
        a0 = x0[q0];
        b0 = x1[q0];
      }
      if (v1) {
        a1 = x0[q1];
        b1 = x1[q1];
      }
      const double2 z = haas_frame(a0, b0, v0, a1, b1, v1, mode_ms, mono, use_width, width);
      acc.add(z.x, z.y, (float)z.x, (float)z.y);
    }
  } else {
    const HaasItem<TIn> it = src.item();
    const long long frames = it.frames;
    const int d = it.d;
    const TIn* __restrict__ x0 = it.x0;
    const TIn* __restrict__ x1 = it.x1;
    total = frames + d;
    out = it.out;
    // Three stretches (decorrelation.py:220-222: channel 0 delayed by d, both padded to frames + d): only channel 1 for
    // m < d, both channels for d <= m < frames, only the delayed channel 0 behind the end of channel 1.
    const long long head = d < frames ? d : frames;
    for (long long m = threadIdx.x; m < head; m += blockDim.x) {
      const TIn r = x1[m];
      acc.add(0.0, (double)r, 0.0f, (float)r);
    }
    if (d < frames) {
      const TIn* __restrict__ p0 = x0 + threadIdx.x;      // x0[m - d]
      const TIn* __restrict__ p1 = x1 + d + threadIdx.x;  // x1[m]
      const long long n = frames - d;
      for (long long k = threadIdx.x; k < n; k += blockDim.x, p0 += blockDim.x, p1 += blockDim.x) {
        const TIn l = *p0, r = *p1;
        acc.add((double)l, (double)r, (float)l, (float)r);
      }
    }  // (d >= frames: the frames between the two channels are silence and add nothing to any sum)
    const long long tail0 = frames > d ? frames : d;
    for (long long m = tail0 + threadIdx.x; m < total; m += blockDim.x) {
      const TIn l = x0[m - d];
      acc.add((double)l, 0.0, (float)l, 0.0f);
    }
  }
  double v[7] = {acc.v0, acc.v1, acc.v2, acc.v3, __longlong_as_double(acc.vmax), acc.v5, acc.v6};
  __shared__ double red[8][7];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    if (k == 4) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v[4] = fmax(v[4], __shfl_xor_sync(0xffffffffu, v[4], o));
    } else {
      v[k] = warp_sum_d(v[k]);
    }
  }
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < 7; ++k) red[warp][k] = v[k];
  }
  __syncthreads();
  if (threadIdx.x < 7) {
    const int k = threadIdx.x;
    double r = red[0][k];
    for (int w = 1; w < 8; ++w) r = (k == 4) ? fmax(r, red[w][k]) : r + red[w][k];
    out[k] = r;
  }
  if (threadIdx.x == 7) out[7] = (double)total;
}

// ------------------------------------------------------------------------------------------------
// launch planning
// ------------------------------------------------------------------------------------------------
static size_t align_up_sz(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct ObjPlan {
  int cand_per_group, n_groups, tiles_per_chunk, n_chunks;
  size_t smem;
};

// Most chunks a clip's tiles are split into: enough for 16 waves of CTAs over all clips, never more than the tiles.
static long long max_chunks(long long tiles, int n_clips, int sm_count) {
  long long c = ceil_div<long long>((long long)sm_count * 16, n_clips > 0 ? n_clips : 1);
  if (c > tiles) c = tiles;
  return c < 1 ? 1 : c;
}

// Shared memory of vn_objective_kernel for a launch halo: the bytes that do not depend on the group size, and the most
// candidates a group can hold.  VND_EUNSUPPORTED when not even 16 fit.
static int obj_group_budget(int halo, int max_prog_words, size_t* fixed_out, int* cpg_out) {
  const size_t span4 = (size_t)((OBJ_TILE + halo + 7) & ~3);
  const size_t fixed = (4 * span4 + OBJ_TILE) * 4 + (size_t)(OBJ_NT / 32) * 2 * max_prog_words * 4 + 64;
  // VND_OBJ_MINB CTAs share the SM's 228 KB (1 KB of each is reserved by the system); a single CTA may take it all
  size_t budget = (size_t)(233472 / VND_OBJ_MINB - 1024);
  if (budget > (size_t)kMaxDynSmem) budget = (size_t)kMaxDynSmem;
  if (fixed + OBJ_CHUNK_SLOTS * 8 * 16 > budget) budget = (size_t)kMaxDynSmem;  // long filters: one CTA per SM
  if (fixed + OBJ_CHUNK_SLOTS * 8 * 16 > budget) return VND_EUNSUPPORTED;
  *fixed_out = fixed;
  *cpg_out = (int)((budget - fixed) / (OBJ_CHUNK_SLOTS * 8));
  return VND_OK;
}

static int plan_objective(long long frames, int n_clips, int n_cand, int halo, int max_prog_words, ObjPlan* pl) {
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  size_t fixed;
  int cpg;
  if ((rc = obj_group_budget(halo, max_prog_words, &fixed, &cpg))) return rc;
  if (cpg > n_cand) cpg = n_cand;
  if (cpg > 1024) cpg = 1024;
  const long long tiles = ceil_div<long long>(frames, OBJ_TILE);
  // One CTA per SM at a time: the launch takes ceil(CTAs / SMs) waves of (tiles per chunk) tile passes over the
  // candidates of a group.  First make the groups small enough for ~4 waves, then pick the split of the tiles into
  // chunks that minimises waves x tiles per chunk, i.e. that leaves the smallest idle tail in the last wave (64 clips
  // x 10 chunks = 640 CTAs on 148 SMs ran 5 waves for 4.3 waves of work; 37 chunks of 10 tiles run 16 full waves).
  const long long want = (long long)di.sm_count * 4;
  while ((long long)n_clips * tiles * ceil_div(n_cand, cpg) < want && cpg > 16) cpg = (cpg + 1) / 2;
  const long long groups = ceil_div(n_cand, cpg);
  long long n_chunks = 1, best = -1;
  const long long cap = max_chunks(tiles, n_clips, di.sm_count);  // what objective_workspace_bytes sizes the partial blocks for
  for (long long c = 1; c <= cap; ++c) {
    const long long tpc_c = ceil_div<long long>(tiles, c);
    const long long real_c = ceil_div<long long>(tiles, tpc_c);
    const long long waves = ceil_div<long long>((long long)n_clips * real_c * groups, di.sm_count);
    const long long cost = waves * tpc_c * 4096 + real_c;  // ties: fewer chunks (fewer partial blocks to combine)
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
  pl->cand_per_group = cpg;
  pl->n_groups = ceil_div(n_cand, cpg);
  pl->tiles_per_chunk = tpc;
  pl->n_chunks = (int)n_chunks;
  pl->smem = fixed + (size_t)cpg * OBJ_CHUNK_SLOTS * 8;
  return VND_OK;
}

int objective_workspace_bytes(long long frames, int n_clips, int n_cand, size_t* bytes) {
  // upper bound independent of the program: one partial block per (clip, tile, candidate) is never
  // exceeded because n_chunks <= tiles; cap chunks at what plan_objective can ask for.
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  const long long tiles = ceil_div<long long>(frames, OBJ_TILE);
  const long long chunks = max_chunks(tiles, n_clips, di.sm_count);
  *bytes = (size_t)n_clips * chunks * n_cand * OBJ_CHUNK_SLOTS * 8 + 256;
  return VND_OK;
}

int vn_objective_launch(const float* clips, long long frames, int n_clips, long long clip_stride, long long chan_stride,
                        const vnd_tap_program* cand, double* partials, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (n_clips == 0 || cand->channels == 0) return VND_OK;
  // the reference takes max(|theta|) of the frames: an empty signal is a ValueError there (optimization.py:41-43)
  VND_REQUIRE(frames > 0, VND_EINVAL, "objective of an empty signal (zero-size array to reduction operation maximum which has no identity)");
  int halo = cand->halo > 0 ? cand->halo : 0;
  if (halo > frames) halo = (int)frames;
  halo = (halo + 3) & ~3;
  const int mpw = cand->max_channel_words > 0 ? cand->max_channel_words : 1;
  ObjPlan pl;
  int rc = plan_objective(frames, n_clips, cand->channels, halo, mpw, &pl);
  if (rc == VND_EUNSUPPORTED) set_error("objective kernel: filter halo %d does not fit in shared memory", halo);
  if (rc) return rc;
  const size_t need = (size_t)n_clips * pl.n_chunks * cand->channels * OBJ_CHUNK_SLOTS * 8;
  VND_REQUIRE(workspace && workspace_bytes >= need, VND_ENOMEM, "objective workspace too small: need %zu bytes, have %zu", need,
              workspace_bytes);
  VND_REQUIRE(n_clips <= 65535 && pl.n_groups <= 65535, VND_EUNSUPPORTED, "too many clips/candidate groups for one launch");
  ObjParams p{};
  p.clips = clips;
  p.frames = frames;
  p.clip_stride = clip_stride;
  p.chan_stride = chan_stride;
  p.words = cand->words;
  p.offsets = cand->offsets;
  p.n_cand = cand->channels;
  p.apply_gain = cand->apply_gain;
  p.halo = halo;
  p.cand_per_group = pl.cand_per_group;
  p.tiles_per_chunk = pl.tiles_per_chunk;
  p.n_chunks = pl.n_chunks;
  p.chunk_partials = reinterpret_cast<double*>(workspace);
  VND_CUDA_OK(cudaFuncSetAttribute(vn_objective_kernel<ObjGridSrc>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  dim3 grid((unsigned)pl.n_chunks, (unsigned)n_clips, (unsigned)pl.n_groups);
  vn_objective_kernel<ObjGridSrc><<<grid, OBJ_NT, pl.smem, st>>>(ObjGridSrc{p}, mpw);
  rc = after_launch("vn_objective_kernel");
  if (rc) return rc;
  return obj_combine_launch(p.chunk_partials, partials, n_clips, pl.n_chunks, cand->channels, st);
}

// ------------------------------------------------------------------------------------------------
// run-list objective over ragged clips (vnd_vn_objective_runs_dev)
// ------------------------------------------------------------------------------------------------
static long long run_tiles(const long long* offs, int clip) { return ceil_div<long long>(offs[clip + 1] - offs[clip], OBJ_TILE); }

// Chunk-partial rows (and so work items) the plan below can ask for at most: each run is cut into at most
// max_chunks(longest clip, runs) chunks, and no more than its tiles.
static long long runs_partial_rows_bound(const long long* offs, const int* run_clip, const int* run_count, int n_runs, int sm_count) {
  long long tmax = 0, active = 0, rows = 0;
  for (int r = 0; r < n_runs; ++r)
    if (run_count[r] > 0) {
      const long long t = run_tiles(offs, run_clip[r]);
      tmax = t > tmax ? t : tmax;
      ++active;
    }
  if (active == 0) return 0;
  const long long cap = max_chunks(tmax, (int)(active < 0x7fffffff ? active : 0x7fffffff), sm_count);
  for (int r = 0; r < n_runs; ++r)
    if (run_count[r] > 0) {
      const long long t = run_tiles(offs, run_clip[r]);
      rows += (t < cap ? t : cap) * run_count[r];
    }
  return rows;
}

static size_t runs_table_bytes(long long items, long long runs) {
  return align_up_sz((size_t)items * sizeof(ObjRunItem) + (size_t)runs * sizeof(ObjRunCombine), 256);
}

int objective_runs_workspace_bytes(const long long* offs, const int* run_clip, const int* run_count, int n_runs, size_t* bytes) {
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  const long long rows = runs_partial_rows_bound(offs, run_clip, run_count, n_runs, di.sm_count);
  *bytes = runs_table_bytes(rows, n_runs) + (size_t)rows * OBJ_CHUNK_SLOTS * 8 + 256;
  return VND_OK;
}

// plan_objective for a run list: the same group size and the same choice of chunks, with the tiles of each run's clip
// in place of the common clip length.  Groups are as large as shared memory allows, halved while the launch would not
// fill about four waves; then the tiles per chunk (one value for every run, chunks counted from frame 0 of each clip)
// that minimise waves x tiles per chunk, ties to fewer chunks of the longest clip.  With equal clips and equal runs
// this is plan_objective's choice and CTA order.
struct ObjRunPlan {
  int cand_per_group = 0;
  size_t smem = 0;
  std::vector<ObjRunItem> items;
  std::vector<ObjRunCombine> comb;
  long long partial_rows = 0;
};

static int plan_runs(const long long* offs, const int* run_clip, const int* run_cand, const int* run_count, const int* run_out, int n_runs,
                     int halo, int max_prog_words, ObjRunPlan* pl) {
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  size_t fixed;
  int cpg;
  if ((rc = obj_group_budget(halo, max_prog_words, &fixed, &cpg))) return rc;
  int max_count = 0, active = 0;
  long long tmax = 0;
  for (int r = 0; r < n_runs; ++r)
    if (run_count[r] > 0) {
      max_count = run_count[r] > max_count ? run_count[r] : max_count;
      const long long t = run_tiles(offs, run_clip[r]);
      tmax = t > tmax ? t : tmax;
      ++active;
    }
  if (active == 0) return VND_OK;
  if (cpg > max_count) cpg = max_count;
  if (cpg > 1024) cpg = 1024;
  const long long want = (long long)di.sm_count * 4;
  auto tile_groups = [&](int g) {
    long long w = 0;
    for (int r = 0; r < n_runs; ++r)
      if (run_count[r] > 0) w += run_tiles(offs, run_clip[r]) * ceil_div(run_count[r], g);
    return w;
  };
  while (tile_groups(cpg) < want && cpg > 16) cpg = (cpg + 1) / 2;
  const long long cap = max_chunks(tmax, active, di.sm_count);
  long long n_chunks = 1, best = -1;
  for (long long c = 1; c <= cap; ++c) {
    const long long tpc_c = ceil_div<long long>(tmax, c);
    long long ctas = 0;
    for (int r = 0; r < n_runs; ++r)
      if (run_count[r] > 0) ctas += ceil_div<long long>(run_tiles(offs, run_clip[r]), tpc_c) * ceil_div(run_count[r], cpg);
    const long long real_c = ceil_div<long long>(tmax, tpc_c);
    const long long cost = ceil_div<long long>(ctas, di.sm_count) * tpc_c * 4096 + real_c;
    if (best < 0 || cost < best) {
      best = cost;
      n_chunks = real_c;
    }
  }
  const long long tpc = ceil_div<long long>(tmax, n_chunks);
  // partial rows: run r owns [chunk][candidate] from part_r; CTAs ordered (group, run, chunk) like plan_objective's grid
  std::vector<long long> part(n_runs, 0);
  int max_groups = 0;
  long long rows = 0;
  for (int r = 0; r < n_runs; ++r) {
    if (run_count[r] <= 0) continue;
    const long long chunks = ceil_div<long long>(run_tiles(offs, run_clip[r]), tpc);
    part[r] = rows;
    rows += chunks * run_count[r];
    pl->comb.push_back({part[r], run_out[r], (int)chunks, run_count[r]});
    const int g = ceil_div(run_count[r], cpg);
    max_groups = g > max_groups ? g : max_groups;
  }
  for (int g = 0; g < max_groups; ++g)
    for (int r = 0; r < n_runs; ++r) {
      if (run_count[r] <= 0 || g * cpg >= run_count[r]) continue;
      const int clip = run_clip[r];
      const long long tiles = run_tiles(offs, clip);
      const int ncand = run_count[r] - g * cpg < cpg ? run_count[r] - g * cpg : cpg;
      for (long long k = 0; k * tpc < tiles; ++k) {
        const long long nt = tiles - k * tpc < tpc ? tiles - k * tpc : tpc;
        pl->items.push_back({offs[clip], offs[clip + 1] - offs[clip], part[r] + k * run_count[r] + (long long)g * cpg, (int)(k * tpc), (int)nt,
                             run_cand[r] + g * cpg, ncand});
      }
    }
  pl->cand_per_group = cpg;
  pl->smem = fixed + (size_t)cpg * OBJ_CHUNK_SLOTS * 8;
  pl->partial_rows = rows;
  return VND_OK;
}

int vn_objective_runs_launch(const float* x, long long chan_stride, const long long* offs, const int* run_clip, const int* run_cand,
                             const int* run_count, const int* run_out, int n_runs, const vnd_tap_program* cand, double* partials,
                             void* workspace, size_t workspace_bytes, cudaStream_t st) {
  long long max_frames = 0;
  for (int r = 0; r < n_runs; ++r)
    if (run_count[r] > 0) {
      const long long f = offs[run_clip[r] + 1] - offs[run_clip[r]];
      max_frames = f > max_frames ? f : max_frames;
    }
  if (max_frames == 0) return VND_OK;
  int halo = cand->halo > 0 ? cand->halo : 0;  // the program's halo, clamped to the longest clip as for one clip
  if (halo > max_frames) halo = (int)max_frames;
  halo = (halo + 3) & ~3;
  const int mpw = cand->max_channel_words > 0 ? cand->max_channel_words : 1;
  ObjRunPlan pl;
  int rc = plan_runs(offs, run_clip, run_cand, run_count, run_out, n_runs, halo, mpw, &pl);
  if (rc == VND_EUNSUPPORTED) set_error("objective kernel: filter halo %d does not fit in shared memory", halo);
  if (rc) return rc;
  VND_REQUIRE(pl.items.size() <= 0x7fffffffu, VND_EUNSUPPORTED, "too many work items for one launch");
  const size_t table = runs_table_bytes((long long)pl.items.size(), (long long)pl.comb.size());
  const size_t need = table + (size_t)pl.partial_rows * OBJ_CHUNK_SLOTS * 8;
  VND_REQUIRE(workspace && workspace_bytes >= need, VND_ENOMEM, "objective workspace too small: need %zu bytes, have %zu", need, workspace_bytes);
  // the tables, one copy: work items, then the combine table
  std::vector<unsigned char> host(table);
  const size_t item_bytes = pl.items.size() * sizeof(ObjRunItem);
  memcpy(host.data(), pl.items.data(), item_bytes);
  memcpy(host.data() + item_bytes, pl.comb.data(), pl.comb.size() * sizeof(ObjRunCombine));
  unsigned char* ws = reinterpret_cast<unsigned char*>(workspace);
  VND_CUDA_OK(cudaMemcpyAsync(ws, host.data(), item_bytes + pl.comb.size() * sizeof(ObjRunCombine), cudaMemcpyHostToDevice, st));
  ObjRunSrc src{};
  src.p.clips = x;
  src.p.chan_stride = chan_stride;
  src.p.words = cand->words;
  src.p.offsets = cand->offsets;
  src.p.n_cand = cand->channels;
  src.p.apply_gain = cand->apply_gain;
  src.p.halo = halo;
  src.p.cand_per_group = pl.cand_per_group;
  src.p.chunk_partials = reinterpret_cast<double*>(ws + table);
  src.items = reinterpret_cast<const ObjRunItem*>(ws);
  VND_CUDA_OK(cudaFuncSetAttribute(vn_objective_kernel<ObjRunSrc>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pl.smem));
  vn_objective_kernel<ObjRunSrc><<<(unsigned)pl.items.size(), OBJ_NT, pl.smem, st>>>(src, mpw);
  if ((rc = after_launch("vn_objective_kernel"))) return rc;
  obj_combine_runs_kernel<<<(unsigned)pl.comb.size(), 128, 0, st>>>(src.p.chunk_partials, partials,
                                                                    reinterpret_cast<const ObjRunCombine*>(ws + item_bytes));
  return after_launch("obj_combine_runs_kernel");
}

int haas_objective_launch(const void* clips, int clip_dtype, long long frames, int n_clips, long long clip_stride, long long chan_stride,
                          const int* delays, int n_cand, double* partials, cudaStream_t st) {
  if (n_clips == 0 || n_cand == 0) return VND_OK;
  VND_REQUIRE(n_clips <= 65535, VND_EUNSUPPORTED, "too many clips for one launch");
  dim3 grid((unsigned)n_cand, (unsigned)n_clips);
  if (clip_dtype == VND_F64)
    haas_objective_kernel<<<grid, 256, 0, st>>>(HaasGridSrc<double>{(const double*)clips, frames, clip_stride, chan_stride, delays, n_cand, partials});
  else
    haas_objective_kernel<<<grid, 256, 0, st>>>(HaasGridSrc<float>{(const float*)clips, frames, clip_stride, chan_stride, delays, n_cand, partials});
  return after_launch("haas_objective_kernel");
}

int haas_objective_pairs_launch(const float* x, long long chan_stride, const long long* offs, const int* pair_clip, const int* pair_delay,
                                int n_pairs, double* partials, cudaStream_t st) {
  if (n_pairs == 0) return VND_OK;
  haas_objective_kernel<<<(unsigned)n_pairs, 256, 0, st>>>(HaasPairSrc{x, chan_stride, offs, pair_clip, pair_delay, partials});
  return after_launch("haas_objective_kernel");
}

int haas_effect_objective_launch(const float* x, long long frames, long long chan_stride, const vnd_haas_clip* cands, int n_cand, double* partials,
                                 cudaStream_t st) {
  if (n_cand == 0) return VND_OK;
  haas_objective_kernel<<<(unsigned)n_cand, 256, 0, st>>>(HaasEffectSrc{x, frames, chan_stride, cands, partials});
  return after_launch("haas_objective_kernel");
}

// ------------------------------------------------------------------------------------------------
// velvet-noise stereo candidates (vnd_vn_stereo_objective_dev)
// ------------------------------------------------------------------------------------------------
// The chunks of today's score of one candidate: vn_objective_launch on its output with the one-tap identity program
// (halo 1, padded to 4; 5 program words), one clip, one candidate.
static int stereo_chunk_plan(long long frames, ObjPlan* pl) { return plan_objective(frames, 1, 1, 4, 5, pl); }

int vn_stereo_objective_workspace_bytes(long long frames, int n_cand, size_t* bytes) {
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  const long long chunks = max_chunks(ceil_div<long long>(frames, OBJ_TILE), 1, di.sm_count);  // plan_objective's cap for one clip
  *bytes = (size_t)chunks * n_cand * OBJ_CHUNK_SLOTS * 8 + 256;
  return VND_OK;
}

// One call's launch of vn_stereo_objective_kernel: its parameters, grid and shared memory.
struct StereoObjLaunch {
  VnStereoObjParams p;
  int mpw, n_chunks, groups;
  size_t smem;
};

// Plans a call without launching anything: VND_EUNSUPPORTED (no error text, the caller scores candidate by candidate)
// when tile + halo does not fit the kernel's shared memory.
static int plan_stereo_objective(const float* x, long long frames, long long chan_stride, const vnd_tap_program* taps, const vnd_vn_stereo_cand* cands,
                                 int n_cand, void* workspace, size_t workspace_bytes, StereoObjLaunch* out) {
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  ObjPlan chunks;
  if ((rc = stereo_chunk_plan(frames, &chunks))) return rc;
  int halo = taps->halo > 0 ? taps->halo : 0;
  if (halo > frames) halo = (int)frames;
  halo = (halo + 3) & ~3;
  const int mpw = taps->max_channel_words > 0 ? taps->max_channel_words : 1;
  constexpr int kWarps = VND_OBJ_STEREO_NT / 32;
  const size_t fixed = (size_t)2 * ((OBJ_TILE + halo + 3) & ~3) * 4 + (size_t)kWarps * 2 * 32 * OBJ_R * 4 + (size_t)kWarps * 2 * mpw * 4 + 64;
  if (fixed + (size_t)OBJ_CHUNK_SLOTS * 8 > (size_t)kMaxDynSmem) return VND_EUNSUPPORTED;
  int cpg = (int)((kMaxDynSmem - fixed) / (OBJ_CHUNK_SLOTS * 8));
  if (cpg > n_cand) cpg = n_cand;
  if (cpg > 1024) cpg = 1024;
  // groups small enough for about four CTAs per SM, never fewer candidates than warps
  while ((long long)chunks.n_chunks * ceil_div(n_cand, cpg) < (long long)di.sm_count * 4 && cpg > kWarps) cpg = (cpg + 1) / 2;
  const int groups = ceil_div(n_cand, cpg);
  VND_REQUIRE(groups <= 65535, VND_EUNSUPPORTED, "too many candidate groups for one launch");
  const size_t need = (size_t)chunks.n_chunks * n_cand * OBJ_CHUNK_SLOTS * 8;
  VND_REQUIRE(workspace && workspace_bytes >= need, VND_ENOMEM, "objective workspace too small: need %zu bytes, have %zu", need, workspace_bytes);
  VnStereoObjParams p{};
  p.x = x;
  p.frames = frames;
  p.chan_stride = chan_stride;
  p.words = taps->words;
  p.offsets = taps->offsets;
  p.cands = cands;
  p.n_cand = n_cand;
  p.apply_gain = taps->apply_gain;
  p.halo = halo;
  p.cand_per_group = cpg;
  p.tiles_per_chunk = chunks.tiles_per_chunk;
  p.chunk_partials = reinterpret_cast<double*>(workspace);
  *out = {p, mpw, chunks.n_chunks, groups, fixed + (size_t)cpg * OBJ_CHUNK_SLOTS * 8};
  return VND_OK;
}

template <bool kGain>
static int stereo_objective_run(const StereoObjLaunch& l, const float* gains, double* partials, cudaStream_t st) {
  VND_CUDA_OK(cudaFuncSetAttribute(vn_stereo_objective_kernel<kGain>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)l.smem));
  vn_stereo_objective_kernel<kGain><<<dim3((unsigned)l.n_chunks, (unsigned)l.groups), VND_OBJ_STEREO_NT, l.smem, st>>>(l.p, l.mpw, gains);
  const int rc = after_launch("vn_stereo_objective_kernel");
  if (rc) return rc;
  return obj_combine_launch(l.p.chunk_partials, partials, 1, l.n_chunks, l.p.n_cand, st);
}

int vn_stereo_objective_launch(const float* x, long long frames, long long chan_stride, const vnd_tap_program* taps, const vnd_vn_stereo_cand* cands,
                               int n_cand, double* partials, void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (n_cand == 0) return VND_OK;
  StereoObjLaunch l;
  const int rc = plan_stereo_objective(x, frames, chan_stride, taps, cands, n_cand, workspace, workspace_bytes, &l);
  if (rc) return rc;
  return stereo_objective_run<false>(l, nullptr, partials, st);
}

// Shared memory of vn_rms_sums_kernel for a launch halo (a multiple of 4) and program block size.
static size_t rms_sums_smem(int halo, int mpw) {
  return (size_t)2 * ((RMS_XTILE + halo + 3) & ~3) * 4 + (size_t)2 * RMS_SUB * RMS_PITCH * 4 + (size_t)RMS_MAX_G * 2 * mpw * 4;
}

// vn_rms_sums_kernel -> vn_stereo_objective_kernel<true> -> obj_combine_kernel on one stream.  Everything that can refuse
// the call is decided before the first launch.
int vn_stereo_rms_objective_launch(const float* x, long long frames, long long chan_stride, const vnd_tap_program* taps,
                                   const vnd_vn_stereo_cand* cands, int n_cand, float* gains, double* partials, void* workspace,
                                   size_t workspace_bytes, cudaStream_t st) {
  if (n_cand == 0) return VND_OK;
  StereoObjLaunch l;
  int rc = plan_stereo_objective(x, frames, chan_stride, taps, cands, n_cand, workspace, workspace_bytes, &l);
  if (rc == VND_EUNSUPPORTED || (!rc && rms_sums_smem(l.p.halo, l.mpw) > (size_t)kMaxDynSmem)) {
    set_error("rms objective kernels: filter halo %d does not fit in shared memory", taps->halo);
    return VND_EUNSUPPORTED;
  }
  if (rc) return rc;
  const size_t smem = rms_sums_smem(l.p.halo, l.mpw);
  DeviceInfo di;
  if ((rc = device_info(&di))) return rc;
  // the fewest candidates per CTA that keep the launch within one wave: the producers, not the chain, bound a full group
  int group = ceil_div(n_cand, di.sm_count);
  if (group > RMS_MAX_G) group = RMS_MAX_G;
  const VnRmsSumsParams sp{x, frames, chan_stride, taps->words, taps->offsets, cands, n_cand, taps->apply_gain, l.p.halo, group, gains};
  VND_CUDA_OK(cudaFuncSetAttribute(vn_rms_sums_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  vn_rms_sums_kernel<<<(unsigned)ceil_div(n_cand, group), RMS_NT, smem, st>>>(sp, l.mpw);
  if ((rc = after_launch("vn_rms_sums_kernel"))) return rc;
  return stereo_objective_run<true>(l, gains, partials, st);
}

}  // namespace vnd
