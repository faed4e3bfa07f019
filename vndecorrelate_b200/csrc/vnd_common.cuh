// Shared helpers for the sm_100a kernels behind include/vnd_b200.h.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/vnd_b200.h"

namespace vnd {

// ---- status plumbing -------------------------------------------------------------------------
void set_error(const char* fmt, ...);
extern std::atomic<long long> g_launches;

#define VND_CUDA_OK(expr)                                                                  \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      ::vnd::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return VND_ECUDA;                                                                    \
    }                                                                                      \
  } while (0)

#define VND_REQUIRE(cond, code, ...)   \
  do {                                 \
    if (!(cond)) {                     \
      ::vnd::set_error(__VA_ARGS__);   \
      return (code);                   \
    }                                  \
  } while (0)

inline int after_launch(const char* what) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaPeekAtLastError();
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    set_error("launch of %s failed: %s", what, cudaGetErrorString(e));
    return VND_ECUDA;
  }
  return VND_OK;
}

// ---- arithmetic that must not be contracted ----------------------------------------------------
// The reference rounds after every numpy ufunc; these wrappers make that explicit (the library is
// also compiled with -fmad=false, the intrinsics are the belt to that pair of braces).
__device__ __forceinline__ float fadd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float fsub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float fmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }

// VelvetNoise.decorrelate after the FIR, at one frame: the optional M/S side-channel encode of the filtered pair (y0, y1)
// against the input pair (x0, x1) (utils/dsp.py:59-63), then the optional width (utils/dsp.py:34-37 with LR_to_MS /
// MS_to_LR, utils/dsp.py:140-166), w_mid = float32(1 - width), w_side = float32(width).  The fused decorrelate kernels
// (vnd_fir.cu) and the stereo objective (vnd_objective.cu) both call it, so a scored candidate sees decorrelate's bits.
__device__ __forceinline__ void ms_width_epilogue(float x0, float x1, float& y0, float& y1, int ms_encode, int use_width, float w_mid,
                                                  float w_side) {
  if (ms_encode) {
    const float M = fadd(x0, x1);
    const float S = fmul(fsub(y0, y1), 0.5f);
    y0 = fmul(fadd(M, S), 0.5f);
    y1 = fmul(fsub(M, S), 0.5f);
  }
  if (use_width) {
    float M = fmul(fadd(y0, y1), 0.5f);
    float S = fmul(fsub(y0, y1), 0.5f);
    M = fmul(M, w_mid);
    S = fmul(S, w_side);
    y0 = fadd(M, S);
    y1 = fsub(M, S);
  }
}

// ---- shared-memory / TMA bulk-copy primitives (sm_90+ PTX, UBLKCP in SASS) -------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
// 1-D bulk copy global -> shared; dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// 1-D bulk copy shared -> global (bulk async-group completion).
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

template <typename T>
__host__ __device__ __forceinline__ T ceil_div(T a, T b) { return (a + b - 1) / b; }

constexpr int kMaxDynSmem = 227 * 1024;  // usable shared memory per CTA on sm_100a

// device properties cached per device
struct DeviceInfo {
  int sm_count = 0;
  int max_smem_optin = 0;
};
int device_info(DeviceInfo* out);

}  // namespace vnd
