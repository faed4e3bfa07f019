// Pieces shared by the batched objective kernels (vnd_objective.cu: every tap through shared memory;
// vnd_objective_tmem.cu: taps inside the tensor-memory window through tcgen05.ld): the parameter block, the polar
// moments of a frame (src/vndecorrelate/utils/dsp.py:374-422, src/vndecorrelate/optimization.py:11-43) in scalar and
// packed form, the exact max|theta| ratio tracker and the warp reductions.
#pragma once

#include "vnd_common.cuh"

namespace vnd {

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

// Two frames at once with packed arithmetic - the inner loop of both objective kernels.  The amplitude-weighted sums
// run in two interleaved chains per lane (even / odd frames, slot [0] / [1]), added together before the warp
// reduction; the ratio trackers stay scalar and see the frames in order.
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

}  // namespace vnd
