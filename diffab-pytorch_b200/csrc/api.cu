// C-ABI bookkeeping: version, thread-local error string, dtype conversion.
#include <cuda_bf16.h>
#include <stdarg.h>

#include <atomic>

#include "common.cuh"

namespace dab {

static thread_local char g_error[512] = "";
static std::atomic<long long> g_launches{0};

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_error, sizeof(g_error), fmt, ap);
  va_end(ap);
}

// fp32 -> bf16 (RNE), 8 elements per thread, 128-bit loads and stores, grid-stride.
__global__ void __launch_bounds__(256) cast_bf16_kernel(const float4* __restrict__ in, uint4* __restrict__ out,
                                                        int64_t n8, const float* __restrict__ in_tail,
                                                        __nv_bfloat16* __restrict__ out_tail, int tail) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    float4 a = __ldg(in + 2 * i), b = __ldg(in + 2 * i + 1);
    __nv_bfloat162 p0 = __floats2bfloat162_rn(a.x, a.y), p1 = __floats2bfloat162_rn(a.z, a.w);
    __nv_bfloat162 p2 = __floats2bfloat162_rn(b.x, b.y), p3 = __floats2bfloat162_rn(b.z, b.w);
    uint4 o;
    o.x = *reinterpret_cast<uint32_t*>(&p0); o.y = *reinterpret_cast<uint32_t*>(&p1);
    o.z = *reinterpret_cast<uint32_t*>(&p2); o.w = *reinterpret_cast<uint32_t*>(&p3);
    out[i] = o;
  }
  if (blockIdx.x == 0 && threadIdx.x < tail) out_tail[threadIdx.x] = __float2bfloat16_rn(in_tail[threadIdx.x]);
}

}  // namespace dab

extern "C" {

int dab_version(void) { return 102; /* 0.1.2: dab_reverse_step_weighted (per-residue amino-acid weights) */ }

const char* dab_last_error(void) { return dab::g_error; }

long long dab_launch_count(void) { return dab::g_launches.load(); }

int dab_cast_f32_to_bf16(const float* in, void* out, int64_t n, void* stream) {
  DAB_REQUIRE(n >= 0, DAB_EINVAL, "dab_cast_f32_to_bf16: negative n");
  if (n == 0) return DAB_OK;
  DAB_REQUIRE(in && out && dab::aligned16(in) && dab::aligned16(out), DAB_EINVAL,
              "dab_cast_f32_to_bf16: null or misaligned pointer");
  int64_t n8 = n / 8;
  int tail = (int)(n - n8 * 8);
  int64_t blocks = (n8 + 255) / 256;
  if (blocks < 1) blocks = 1;
  if (blocks > 148 * 16) blocks = 148 * 16;
  dab::cast_bf16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(in), reinterpret_cast<uint4*>(out), n8, in + n8 * 8,
      reinterpret_cast<__nv_bfloat16*>(out) + n8 * 8, tail);
  dab::count_launch();
  return dab::check_launch("dab_cast_f32_to_bf16");
}

}  // extern "C"
