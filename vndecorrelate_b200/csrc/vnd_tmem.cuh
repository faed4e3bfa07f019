// Tensor-memory gather primitives of the sparse-FIR kernel (vnd_fir_tmem.cu): tcgen05 allocation / load / store
// wrappers, packed fp32 arithmetic, and the tap machinery that applies one decay segment after the other to a thread's
// kRG consecutive outputs in the reference's order (src/vndecorrelate/decorrelation.py:402-414) - taps inside the TMEM
// window as one tcgen05.ld each, the others as 16-byte shared-memory loads from the staged tile.
#pragma once

#include "vnd_common.cuh"

#ifndef VND_TM_POLL_NS
#define VND_TM_POLL_NS 200  // sleep of a data-movement lane between two polls of an mbarrier
#endif
#define VND_STR2(x) #x
#define VND_STR(x) VND_STR2(x)

namespace vnd {
namespace tm {

constexpr int kRows = 128;             // TMEM lanes = rows of a tile
constexpr int kCols = 512;             // TMEM columns
constexpr int kUnits = kCols / 32;     // 32-column units of a TMEM row
constexpr int kRG = 32;                // consecutive outputs per compute thread: a tensor-memory tap is one x32 tcgen05.ld

// ---- tensor-memory primitives -------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc_all(uint32_t* slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(slot)) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_all(uint32_t addr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void tmem_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

#define VND_O4(v, i) "=f"(v[i]), "=f"(v[i + 1]), "=f"(v[i + 2]), "=f"(v[i + 3])
#define VND_O16(v, i) VND_O4(v, i), VND_O4(v, i + 4), VND_O4(v, i + 8), VND_O4(v, i + 12)
#define VND_IO4(v, i) "+f"(v[i]), "+f"(v[i + 1]), "+f"(v[i + 2]), "+f"(v[i + 3])
#define VND_IO16(v, i) VND_IO4(v, i), VND_IO4(v, i + 4), VND_IO4(v, i + 8), VND_IO4(v, i + 12)
#define VND_I4(v, i) "f"(v[i].x), "f"(v[i].y), "f"(v[i].z), "f"(v[i].w)

// 32 consecutive columns of this thread's TMEM lane, starting at column (taddr & 0xffff).
__device__ __forceinline__ void tmem_ld32(float (&v)[kRG], uint32_t taddr) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : VND_O16(v, 0), VND_O16(v, 16)
      : "r"(taddr));
}
// The loaded registers are only defined after the wait; naming them as in/out operands keeps the
// compiler from moving their consumers above it.
__device__ __forceinline__ void tmem_wait_ld(float (&v)[kRG]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;" : VND_IO16(v, 0), VND_IO16(v, 16)::"memory");
}
// 32 consecutive columns written from eight float4.
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const float4 (&v)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%32], {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31};" ::VND_I4(v, 0),
      VND_I4(v, 1), VND_I4(v, 2), VND_I4(v, 3), VND_I4(v, 4), VND_I4(v, 5), VND_I4(v, 6), VND_I4(v, 7), "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_u32(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx_u32(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// The data-movement lanes wait for whole tiles: they sleep between polls instead of spinning, so the
// polling does not take issue slots from the compute warps of the same scheduler.
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "nanosleep.u32 " VND_STR(VND_TM_POLL_NS) ";\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// One poll of an mbarrier phase (no blocking, no sleep).
__device__ __forceinline__ bool mbar_try_u32(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void* tmap, int c0, int c1, int c2, uint32_t bar) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(dst),
               "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const void* tmap, int c0, int c1, int c2, uint32_t src) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(tmap), "r"(c0), "r"(c1), "r"(c2),
               "r"(src)
               : "memory");
}
template <int N>
__device__ __forceinline__ void set_max_regs_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void set_max_regs_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// ---- packed fp32 arithmetic (sm_100+): FADD2 / FMUL2 do two IEEE round-to-nearest operations per
// instruction on an aligned register pair.  Same bits as two scalar operations, half the issue slots.
// The accumulators stay scalar float variables and are packed around each instruction; ptxas then
// keeps every pair in one aligned register pair and the packing costs nothing.  (Loop-carried
// 64-bit accumulators made it write half of the results over the loaded operand and copy them back.)
typedef unsigned long long pair_t;
#define VND_PACKED_OP(name, op)                                                     \
  __device__ __forceinline__ void name(float& a0, float& a1, float b0, float b1) { \
    pair_t ra, rb;                                                                  \
    asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a0), "f"(a1));                    \
    asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b0), "f"(b1));                    \
    asm(op ".rn.f32x2 %0, %0, %1;" : "+l"(ra) : "l"(rb));                          \
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(ra));                   \
  }
VND_PACKED_OP(add2, "add")
VND_PACKED_OP(sub2, "sub")
VND_PACKED_OP(mul2, "mul")

// A tap served from tensor memory: the thread's kRG columns starting at the tap's column (tmem_ld32), then kRG / 2
// packed adds (or subtracts).
template <bool SUB>
__device__ __forceinline__ void near_add(const float (&t)[kRG], float (&acc)[kRG]) {
#pragma unroll
  for (int j = 0; j < kRG / 2; ++j) {
    if constexpr (SUB) sub2(acc[2 * j], acc[2 * j + 1], t[2 * j], t[2 * j + 1]);
    else add2(acc[2 * j], acc[2 * j + 1], t[2 * j], t[2 * j + 1]);
  }
}

// A tap served from shared memory.  `row` is the shared-memory address of the staged block of this thread's row.  The
// operation word (build_ops) carries the word offset of the aligned 16-byte chunk that holds the
// thread's first operand, the operand's position A inside it and kx, the number of chunks before the
// run crosses into the next block, where the pitch inserts a 4-word gap (kx >= chunks of the tap: no crossing).
// The kRG operands lie in kRG / 4 (A == 0) or kRG / 4 + 1 chunks.
// The chunks are read with explicit 16-byte loads: left to the compiler, the partly used first and last
// chunk become 4- and 8-byte loads, which cost as many shared-memory wavefronts each as the full chunk
// (lanes are a pitch apart: a 4-way conflict for LDS.32, 2-way for LDS.64) and up to twice together.
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
template <int A, bool SUB>
__device__ __forceinline__ void far_tap_a(uint32_t row, int op, float (&acc)[kRG]) {
  constexpr int NC = kRG / 4 + ((A == 0) ? 0 : 1);
  const uint32_t p = row + 4u * (uint32_t)(op & 0xffff);  // `row`: shared-memory address of the thread's row
  const int kx = (op >> 16) & 31;
  float4 c[NC];
  if (kx >= NC) {
#pragma unroll
    for (int k = 0; k < NC; ++k) c[k] = lds128(p + 16u * k);
  } else {
#pragma unroll
    for (int k = 0; k < NC; ++k) c[k] = lds128(p + 16u * k + (k < kx ? 0u : 16u));
  }
  float t[NC * 4];
#pragma unroll
  for (int k = 0; k < NC; ++k) {
    t[4 * k] = c[k].x;
    t[4 * k + 1] = c[k].y;
    t[4 * k + 2] = c[k].z;
    t[4 * k + 3] = c[k].w;
  }
  if constexpr (A % 2 == 0) {  // operands arrive as aligned register pairs
#pragma unroll
    for (int j = 0; j < kRG / 2; ++j) {
      if constexpr (SUB) sub2(acc[2 * j], acc[2 * j + 1], t[2 * j + A], t[2 * j + 1 + A]);
      else add2(acc[2 * j], acc[2 * j + 1], t[2 * j + A], t[2 * j + 1 + A]);
    }
  } else {  // odd shift: the pairs of the loaded data straddle the accumulator pairs -> scalar adds
#pragma unroll
    for (int r = 0; r < kRG; ++r) acc[r] = SUB ? fsub(acc[r], t[r + A]) : fadd(acc[r], t[r + A]);
  }
}

// Tap operations, decoded once per run for each thread group (begin_run):
//   near tap: the tap offset i itself (>= 0): the TMEM column is tcol0 + i
//   far tap:  kOpFar | A << 24 | kx << 16 | word offset of the first chunk relative to the thread's row
constexpr int kOpFar = (int)0x80000000u;

template <bool SUB>
__device__ __forceinline__ void far_tap(uint32_t row, int op, float (&acc)[kRG]) {
  switch ((op >> 24) & 3) {
    case 0: far_tap_a<0, SUB>(row, op, acc); break;
    case 1: far_tap_a<1, SUB>(row, op, acc); break;
    case 2: far_tap_a<2, SUB>(row, op, acc); break;
    default: far_tap_a<3, SUB>(row, op, acc); break;
  }
}

// One tap: from tensor memory (op >= 0) or from shared memory.
template <bool SUB, bool ALLFAR>
__device__ __forceinline__ void one_tap(int op, uint32_t tcol0, uint32_t row, float (&acc)[kRG]) {
  if (!ALLFAR && op >= 0) {
    float t[kRG];
    tmem_ld32(t, tcol0 + (uint32_t)op);
    tmem_wait_ld(t);
    near_add<SUB>(t, acc);
  } else {
    far_tap<SUB>(row, op, acc);
  }
}

// One list of taps applied to acc: the negative impulses of a segment (SUB) or the positive ones.
// ALLFAR: no tap of the list lies inside the TMEM window (no tensor-memory code at all).
// `nn` = number of LEADING taps of the list that are tensor-memory taps (impulses come in ascending
// order, so that is normally all of them): they run in a loop without the per-tap near/far decision.
// The loops are unrolled by two with the operation words in alternating registers, so that each word
// is loaded a whole tap before it is needed and never copied (a single loop-carried register made
// ptxas copy the loaded word at once and stall on the shared-memory latency at every tap).
template <bool SUB, bool ALLFAR>
__device__ __forceinline__ void tap_list(const int* __restrict__ ops, int n, int nn, uint32_t tcol0, uint32_t row, float (&acc)[kRG]) {
  if (n <= 0) return;
  int k = 0;
  int op_a = ops[0];
  if constexpr (!ALLFAR) {
    for (; k < nn; k += 2) {  // near prefix
      const int op_b = ops[k + 1];  // two words of slack follow the lists, so the prefetches stay in bounds
      {
        float t[kRG];
        tmem_ld32(t, tcol0 + (uint32_t)op_a);
        tmem_wait_ld(t);
        near_add<SUB>(t, acc);
      }
      op_a = ops[k + 2];
      if (k + 1 >= nn) {
        op_a = op_b;
        ++k;
        break;
      }
      {
        float t[kRG];
        tmem_ld32(t, tcol0 + (uint32_t)op_b);
        tmem_wait_ld(t);
        near_add<SUB>(t, acc);
      }
    }
    if (k >= n) return;
  }
  for (;; k += 2) {  // the rest: far taps (and any near tap behind a far one)
    const int op_b = ops[k + 1];
    one_tap<SUB, ALLFAR>(op_a, tcol0, row, acc);
    if (k + 1 >= n) break;
    op_a = ops[k + 2];
    one_tap<SUB, ALLFAR>(op_b, tcol0, row, acc);
    if (k + 2 >= n) break;
  }
}

// Segments [s0, s1) of the program added into the running output, in the reference's order
// (decorrelation.py:402-414): acc = 0; acc -= x[n + i] over the negative list; acc += x[n + i] over
// the positive list; acc *= gain; y += acc.
template <bool ALLFAR>
__device__ __forceinline__ void run_segments(const int4* __restrict__ segtab, int s0, int s1, const int*& ops, uint32_t tcol0, uint32_t row,
                                             float (&yv)[kRG]) {
  for (int s = s0; s < s1; ++s) {
    const int4 d = segtab[s];  // x = negative taps, y = positive taps, z = leading tensor-memory taps of both lists, w = gain bits
    const int n_neg = d.x, n_pos = d.y;
    float acc[kRG];
#pragma unroll
    for (int r = 0; r < kRG; ++r) acc[r] = 0.0f;
    const int nn = ALLFAR ? 0 : d.z;  // leading tensor-memory taps: neg list in the low half, pos list in the high half
    tap_list<true, ALLFAR>(ops, n_neg, nn & 0xffff, tcol0, row, acc);
    tap_list<false, ALLFAR>(ops + n_neg, n_pos, nn >> 16, tcol0, row, acc);
    ops += n_neg + n_pos;
    {  // 1.0f when the program carries no gains (x * 1 == x bit for bit)
      const float gain = __int_as_float(d.w);
#pragma unroll
      for (int j = 0; j < kRG / 2; ++j) mul2(acc[2 * j], acc[2 * j + 1], gain, gain);
    }
    if (s == 0) {  // the reference adds into zeros (a -0 partial sum becomes +0)
#pragma unroll
      for (int j = 0; j < kRG / 2; ++j) {
        yv[2 * j] = acc[2 * j];
        yv[2 * j + 1] = acc[2 * j + 1];
        add2(yv[2 * j], yv[2 * j + 1], 0.0f, 0.0f);
      }
    } else {
#pragma unroll
      for (int j = 0; j < kRG / 2; ++j) add2(yv[2 * j], yv[2 * j + 1], acc[2 * j], acc[2 * j + 1]);
    }
  }
}

}  // namespace tm
}  // namespace vnd
