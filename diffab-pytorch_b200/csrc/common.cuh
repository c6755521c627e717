// Shared helpers for libdiffab_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/diffab_b200.h"

namespace dab {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);   // bookkeeping behind dab_launch_count()

inline int check_launch(const char* what) {
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(err));
    return DAB_ELAUNCH;
  }
  return DAB_OK;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline bool aligned32(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 31u) == 0; }   // 256-bit stores

// Opt a kernel in to `bytes` of dynamic shared memory once per (kernel, device): the attribute is per device, and the
// library may be called from several host threads (an atomic bit mask per call site; a repeated set is harmless).
#define DAB_ENSURE_SMEM(kernel, bytes)                                                                    \
  do {                                                                                                    \
    static std::atomic<unsigned long long> dab_done_mask{0};                                              \
    int dab_dev = 0;                                                                                      \
    cudaGetDevice(&dab_dev);                                                                              \
    const unsigned long long dab_bit = 1ull << (dab_dev & 63);                                            \
    if (!(dab_done_mask.load(std::memory_order_acquire) & dab_bit)) {                                     \
      cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes));           \
      dab_done_mask.fetch_or(dab_bit, std::memory_order_release);                                        \
    }                                                                                                     \
  } while (0)

#define DAB_REQUIRE(cond, code, ...)  \
  do {                                \
    if (!(cond)) {                    \
      ::dab::set_error(__VA_ARGS__);  \
      return (code);                  \
    }                                 \
  } while (0)

// `generate` argument of the diffusion and loss entry points: DAB_GEN_SEQUENCE | DAB_GEN_STRUCTURE, at least one bit
inline int check_generate(int generate, const char* what) {
  DAB_REQUIRE(generate >= 1 && generate <= (DAB_GEN_SEQUENCE | DAB_GEN_STRUCTURE), DAB_EINVAL,
              "%s: generate must be 1 (sequence), 2 (structure) or 3 (both), got %d", what, generate);
  return DAB_OK;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- 3x3 rotation helpers (row-major float[9]) ---------------------------------------------
// Rodrigues, exactly the reference's expression (so3.py:219-237): I + S sin(n)/n + S@S (1-cos n)/n^2
// with n = |v|; no epsilon guard (n = 0 gives NaN as in the reference).
__device__ __forceinline__ void so3_exp(float x, float y, float z, float* R) {
  float n = sqrtf(x * x + y * y + z * z);
  float a = sinf(n) / n;
  float b = (1.0f - cosf(n)) / (n * n);
  // S = [[0,-z,y],[z,0,-x],[-y,x,0]];  S@S = v v^T - n^2 I written out as the matmul would
  float s00 = -z * z - y * y, s01 = y * x, s02 = z * x;
  float s10 = x * y, s11 = -z * z - x * x, s12 = z * y;
  float s20 = x * z, s21 = y * z, s22 = -y * y - x * x;
  R[0] = 1.0f + s00 * b; R[1] = -z * a + s01 * b; R[2] = y * a + s02 * b;
  R[3] = z * a + s10 * b; R[4] = 1.0f + s11 * b; R[5] = -x * a + s12 * b;
  R[6] = -y * a + s20 * b; R[7] = x * a + s21 * b; R[8] = 1.0f + s22 * b;
}

// log map as a rotation vector (so3.py:146-182): theta/(2 sin theta) * vee(R - R^T)
__device__ __forceinline__ void so3_log(const float* R, float& x, float& y, float& z) {
  float c = (R[0] + R[4] + R[8] - 1.0f) * 0.5f;
  float th = acosf(c);
  float k = th / (2.0f * sinf(th));
  x = k * (R[7] - R[5]);
  y = k * (R[2] - R[6]);
  z = k * (R[3] - R[1]);
}

// C = A @ B (row-major 3x3)
__device__ __forceinline__ void mat3_mul(const float* A, const float* B, float* C) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) C[i * 3 + j] = A[i * 3] * B[j] + A[i * 3 + 1] * B[3 + j] + A[i * 3 + 2] * B[6 + j];
}

}  // namespace dab
