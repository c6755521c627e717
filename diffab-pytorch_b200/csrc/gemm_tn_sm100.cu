// Weight-gradient GEMM of the tensor-core path on tcgen05 (sm_100a):
//
//   C[M, N] (fp32, row-major, ldc) = A[K, M]^T * B[K, N]        A, B: bf16, row-major (M / N contiguous), K = rows
//
// i.e. both operands are read "MN-major" straight from the activations as they lie in HBM (dy, concat features, dproj, x:
// one row per residue) - the transposes that a K-major GEMM would need are never materialised.  These are the autograd
// gradients of the nn.Linear weights of diffab_pytorch.py:391-408,464:  dWout = dy^T cat,  dWcat = dproj^T x.
//
// The contraction runs over all B*L residues, so the grid is (N tiles, M tiles, K splits): a CTA accumulates its K range
// into one 128 x BN TMEM tile and adds it to C with vector red.global (C is zeroed by the launcher).
//   warp 0: TMA producer (64-row K chunks; every 64-wide column atom of A / B is one 128B-swizzled box, ring of 3)
//   warp 1: tcgen05.mma issuer (whole warp walks the loop, one elected lane issues; M = 128, N = BN, K = 16 per MMA)
//   warps 0-3: epilogue, thread = TMEM lane = row m of the tile
// Also here: the column sum of an fp32 matrix (the bias gradient d b_out = sum over residues of dy).
#include <cuda_bf16.h>

#include "common.cuh"
#include "sm100_prims.cuh"

namespace dab {
namespace sm100 {

constexpr int kTnBM = 128;     // tile rows  (columns of A)
constexpr int kTnKC = 64;      // residues per K chunk
constexpr int kTnStages = 3;

template <int BN>
struct TnSmem {
  static constexpr int kAtom = kTnKC * 128;                  // 8,192: [64 k rows][64 columns] bf16, 128B swizzle
  static constexpr int kABytes = (kTnBM / 64) * kAtom;       // 16,384
  static constexpr int kBBytes = (BN / 64) * kAtom;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kBars = kTnStages * kStageBytes;
  static constexpr int kTotal = kBars + 128 + 1024 /* alignment slack */;
};

template <int BN>
__global__ void __launch_bounds__(128) gemm_tn_bf16_kernel(const __grid_constant__ CUtensorMap map_a,
                                                           const __grid_constant__ CUtensorMap map_b,
                                                           float* __restrict__ C, int64_t ldc, int M, int chunks_per_split,
                                                           int n_chunks) {
  static_assert(BN == 64 || BN == 128, "BN");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  using S = TnSmem<BN>;
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + S::kBars);
  uint64_t* empty = full + kTnStages;
  uint64_t* done = empty + kTnStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BN, m0 = blockIdx.y * kTnBM;
  const int c_lo = blockIdx.z * chunks_per_split;
  const int c_hi = min(n_chunks, c_lo + chunks_per_split);
  const int nk = c_hi - c_lo;
  constexpr uint32_t kTmemCols = BN;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kTnStages; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(done, 1);
    fence_barrier_init();
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(tmem_slot, kTmemCols);
  tcgen05_fence_before_sync();
  __syncthreads();
  tcgen05_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  if (nk <= 0) {            // (cannot happen with the launcher's split; keeps the barrier protocol trivially safe)
    tcgen05_fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_free(tmem_base, kTmemCols);
    return;
  }

  if (warp == 0) {
    for (int kc = 0; kc < nk; ++kc) {
      const int s = kc % kTnStages;
      if (kc >= kTnStages) mbar_wait(&empty[s], ((kc / kTnStages) - 1) & 1);
      if (elect_one()) {
        uint8_t* a = smem + s * S::kStageBytes;
        const int krow = (c_lo + kc) * kTnKC;
        mbar_arrive_expect_tx(&full[s], S::kStageBytes);
        for (int at = 0; at < kTnBM / 64; ++at) tma_load_2d(a + at * S::kAtom, &map_a, &full[s], m0 + at * 64, krow);
        for (int at = 0; at < BN / 64; ++at)
          tma_load_2d(a + S::kABytes + at * S::kAtom, &map_b, &full[s], n0 + at * 64, krow);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    constexpr uint32_t idesc = make_idesc_bf16(kTnBM, BN, 1, 1);      // both operands MN-major
    // MN-major, 128B swizzle: 64-wide column atoms S::kAtom apart (LBO), 8-row K groups 1024 B apart (SBO); a K step of
    // 16 rows is +2048 B
    const uint64_t d0 = make_smem_desc(smem_u32(smem), S::kAtom, 1024, kSwizzle128B);
    for (int kc = 0; kc < nk; ++kc) {
      const int s = kc % kTnStages;
      mbar_wait(&full[s], (kc / kTnStages) & 1);
      tcgen05_fence_after_sync();
      if (elect_one()) {
        const uint64_t da = d0 + (uint32_t)((s * S::kStageBytes) >> 4);
        const uint64_t db = da + (uint32_t)(S::kABytes >> 4);
#pragma unroll
        for (int k = 0; k < kTnKC / 16; ++k)
          umma_bf16(tmem_base, da + (uint32_t)((k * 2048) >> 4), db + (uint32_t)((k * 2048) >> 4), idesc, (kc | k) != 0);
        umma_commit(&empty[s]);
        if (kc == nk - 1) umma_commit(done);
      }
      __syncwarp();
    }
  }
  __syncwarp();
  mbar_wait(done, 0);
  tcgen05_fence_after_sync();

  // epilogue: thread (warp, lane) owns tile row 32 * warp + lane; its partial sums go to C with 16-byte reductions
  const int row = m0 + warp * 32 + lane;
  float* crow = C + (int64_t)row * ldc + n0;
#pragma unroll
  for (int c0 = 0; c0 < BN; c0 += 16) {
    float v[16];
    tmem_ld_x16(tmem_base + ((uint32_t)(warp * 32) << 16) + c0, v);
    tmem_wait_ld();
    if (row < M) {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(crow + c0 + 4 * q), "f"(v[4 * q]),
                     "f"(v[4 * q + 1]), "f"(v[4 * q + 2]), "f"(v[4 * q + 3])
                     : "memory");
    }
  }
  tcgen05_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_free(tmem_base, kTmemCols);
}

template <int BN>
static int launch_gemm_tn(const void* A, int64_t lda, const void* Bm, int64_t ldb, float* C, int64_t ldc, int M, int N, int K,
                          cudaStream_t stream, bool accumulate = false) {
  CUtensorMap ma, mb;
  uint64_t dims_a[2] = {(uint64_t)M, (uint64_t)K}, str_a[1] = {(uint64_t)lda * 2};
  uint64_t dims_b[2] = {(uint64_t)N, (uint64_t)K}, str_b[1] = {(uint64_t)ldb * 2};
  uint32_t box[2] = {64, kTnKC};
  if (int rc = make_tensor_map_bf16(&ma, A, 2, dims_a, str_a, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  if (int rc = make_tensor_map_bf16(&mb, Bm, 2, dims_b, str_b, box, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  DAB_ENSURE_SMEM(gemm_tn_bf16_kernel<BN>, TnSmem<BN>::kTotal);
  const int tiles = ((M + kTnBM - 1) / kTnBM) * (N / BN);
  const int n_chunks = K / kTnKC;
  // K splits for about one wave of CTAs (every split adds a 128 x BN tile of red.global traffic onto the small output:
  // more splits shorten the K loops but the L2 atomic units become the bottleneck), at least four chunks per CTA
  int splits = (148 + tiles - 1) / tiles;
  if (splits > n_chunks / 4) splits = n_chunks / 4 > 0 ? n_chunks / 4 : 1;
  const int per = (n_chunks + splits - 1) / splits;
  splits = (n_chunks + per - 1) / per;
  // only the M x N block: with ldc > N the columns N..ldc-1 of each row belong to the caller (C may be a column block)
  if (!accumulate &&
      cudaMemset2DAsync(C, (size_t)ldc * sizeof(float), 0, (size_t)N * sizeof(float), (size_t)M, stream) != cudaSuccess)
    return check_launch("gemm_tn memset");
  dim3 grid(N / BN, (M + kTnBM - 1) / kTnBM, splits);
  gemm_tn_bf16_kernel<BN><<<grid, 128, TnSmem<BN>::kTotal, stream>>>(ma, mb, C, ldc, M, per, n_chunks);
  count_launch();
  return check_launch("gemm_tn_bf16");
}

// out[c] = sum_r x[r, c]  (cols <= 1024, multiple of 4): blocks own row ranges, one red.global per column and block;
// optionally x is first multiplied by the ReLU mask (y > 0) of a bf16 activation, and optionally the (masked) x is also
// written rounded to bf16 (the operand of the gradient GEMMs) in the same pass.  TIn = float or __nv_bfloat16.
template <typename TIn>
__global__ void __launch_bounds__(256) colsum_kernel(const TIn* __restrict__ x, int64_t rows, int cols, float* __restrict__ out,
                                                     __nv_bfloat16* __restrict__ x_bf16, const __nv_bfloat16* __restrict__ y_mask) {
  __shared__ float4 part[256];
  const int c4 = cols / 4;                       // float4 columns
  const int lanes = c4 < 256 ? c4 : 256;         // threads that own a float4 column each (cols <= 1024)
  const int groups = 256 / lanes;                // row groups inside the block
  const int tc = threadIdx.x % lanes, tg = threadIdx.x / lanes;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (tg < groups) {
    for (int64_t r = (int64_t)blockIdx.x * groups + tg; r < rows; r += (int64_t)gridDim.x * groups) {
      float4 v;
      if (sizeof(TIn) == 4) {
        v = __ldg(reinterpret_cast<const float4*>(x + r * cols) + tc);
      } else {
        const uint2 u = __ldg(reinterpret_cast<const uint2*>(x + r * cols) + tc);
        v = make_float4(__uint_as_float(u.x << 16), __uint_as_float(u.x & 0xFFFF0000u), __uint_as_float(u.y << 16),
                        __uint_as_float(u.y & 0xFFFF0000u));
      }
      if (y_mask) {                              // bf16 > 0: sign clear and not zero
        const uint2 m = __ldg(reinterpret_cast<const uint2*>(y_mask + r * cols) + tc);
        if (!((m.x & 0xFFFFu) - 1u < 0x7FFFu)) v.x = 0.f;
        if (!((m.x >> 16) - 1u < 0x7FFFu)) v.y = 0.f;
        if (!((m.y & 0xFFFFu) - 1u < 0x7FFFu)) v.z = 0.f;
        if (!((m.y >> 16) - 1u < 0x7FFFu)) v.w = 0.f;
      }
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
      if (x_bf16) {
        __nv_bfloat162 p0 = __floats2bfloat162_rn(v.x, v.y), p1 = __floats2bfloat162_rn(v.z, v.w);
        reinterpret_cast<uint2*>(x_bf16 + r * cols)[tc] =
            make_uint2(*reinterpret_cast<uint32_t*>(&p0), *reinterpret_cast<uint32_t*>(&p1));
      }
    }
  }
  part[threadIdx.x] = acc;
  __syncthreads();
  if (tg == 0) {                                  // one reduction per column quad and block (few blocks: little contention)
    for (int k = 1; k < groups; ++k) {
      const float4 o = part[k * lanes + tc];
      acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
    }
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(out + 4 * tc), "f"(acc.x), "f"(acc.y), "f"(acc.z),
                 "f"(acc.w)
                 : "memory");
  }
}

}  // namespace sm100
}  // namespace dab

using namespace dab;
using namespace dab::sm100;

extern "C" {

/* C[M,N] (fp32, overwritten) = A[K,M]^T B[K,N]: bf16 operands with the contraction index as their ROW index (activations
 * as they lie in memory, one row per residue); K % 64 == 0, N % 64 == 0, lda % 8 == 0 and ldb % 8 == 0 (TMA row pitch:
 * a multiple of 16 bytes), ldc % 4 == 0, lda >= M, ldb >= N, ldc >= N, any M > 0 otherwise.  Only the M x N block of C
 * is written: columns N..ldc-1 are left alone, so C may be a column block of a wider matrix.
 * Split over K across CTAs, partial tiles added with red.global (summation order not fixed: last-bit differences
 * between runs).  Autograd weight gradients of the nn.Linear layers, diffab_pytorch.py:391-408,464. */
int dab_gemm_bf16_tn(const void* A, int64_t lda, const void* Bm, int64_t ldb, float* C, int64_t ldc, int M, int N, int K,
                     void* stream) {
  DAB_REQUIRE(A && Bm && C, DAB_EINVAL, "dab_gemm_bf16_tn: null pointer");
  DAB_REQUIRE(M > 0 && N > 0 && K > 0 && K % kTnKC == 0 && N % 64 == 0 && lda % 8 == 0 && ldb % 8 == 0 && ldc % 4 == 0 &&
                  lda >= M && ldb >= N && ldc >= N,
              DAB_EUNSUPPORTED, "dab_gemm_bf16_tn: K %% 64, N %% 64, lda/ldb %% 8, ldc %% 4 required (M=%d N=%d K=%d)", M, N, K);
  DAB_REQUIRE(aligned16(A) && aligned16(Bm) && aligned16(C), DAB_EINVAL, "dab_gemm_bf16_tn: misaligned pointer");
  if (N % 128 == 0) return launch_gemm_tn<128>(A, lda, Bm, ldb, C, ldc, M, N, K, (cudaStream_t)stream);
  return launch_gemm_tn<64>(A, lda, Bm, ldb, C, ldc, M, N, K, (cudaStream_t)stream);
}

/* C[M,N] += A[K,M]^T B[K,N]: dab_gemm_bf16_tn without the fill of C - the caller zeroes (or pre-loads) C, e.g. on a side
 * stream long before the operands exist, so that no fill sits between the producer of the operands and this GEMM. */
int dab_gemm_bf16_tn_acc(const void* A, int64_t lda, const void* Bm, int64_t ldb, float* C, int64_t ldc, int M, int N, int K,
                         void* stream) {
  DAB_REQUIRE(A && Bm && C, DAB_EINVAL, "dab_gemm_bf16_tn_acc: null pointer");
  DAB_REQUIRE(M > 0 && N > 0 && K > 0 && K % kTnKC == 0 && N % 64 == 0 && lda % 8 == 0 && ldb % 8 == 0 && ldc % 4 == 0 &&
                  lda >= M && ldb >= N && ldc >= N,
              DAB_EUNSUPPORTED, "dab_gemm_bf16_tn_acc: K %% 64, N %% 64, lda/ldb %% 8, ldc %% 4 required (M=%d N=%d K=%d)", M, N, K);
  DAB_REQUIRE(aligned16(A) && aligned16(Bm) && aligned16(C), DAB_EINVAL, "dab_gemm_bf16_tn_acc: misaligned pointer");
  if (N % 128 == 0) return launch_gemm_tn<128>(A, lda, Bm, ldb, C, ldc, M, N, K, (cudaStream_t)stream, true);
  return launch_gemm_tn<64>(A, lda, Bm, ldb, C, ldc, M, N, K, (cudaStream_t)stream, true);
}

/* out[cols] (fp32, overwritten) = column sums of x[rows, cols] (fp32, contiguous): bias gradients (sum over residues).
 * x_bf16 (optional, may be NULL): x rounded to bf16, written in the same pass (the operand of the gradient GEMMs). */
int dab_colsum_f32(const float* x, int64_t rows, int cols, float* out, void* x_bf16, void* stream) {
  DAB_REQUIRE(x && out && rows >= 0 && cols > 0 && cols % 4 == 0 && cols <= 1024 && aligned16(x) && aligned16(out), DAB_EINVAL,
              "dab_colsum_f32: bad argument (cols %% 4 == 0, <= 1024; 16-byte aligned pointers)");
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemsetAsync(out, 0, (size_t)cols * sizeof(float), s) != cudaSuccess) return check_launch("dab_colsum_f32 memset");
  if (rows == 0) return DAB_OK;
  // small inputs are latency-bound: one row per thread (more blocks, one red.global per column and block); large ones
  // walk the rows with 148 x 4 blocks
  const int c4 = cols / 4, groups = 256 / (c4 < 256 ? c4 : 256);
  int64_t blocks = (rows + groups - 1) / groups;
  if (blocks > 148 * 4) blocks = 148 * 4;
  colsum_kernel<float><<<(unsigned)blocks, 256, 0, s>>>(x, rows, cols, out, reinterpret_cast<__nv_bfloat16*>(x_bf16), nullptr);
  count_launch();
  return check_launch("dab_colsum_f32");
}

/* Bias gradient of an nn.Linear behind a ReLU, with the operand of its gradient GEMMs: g' = g * (y > 0) (y_bf16 = the ReLU
 * output, NULL: no mask), db[cols] (fp32, overwritten) = column sums of g', g_out_bf16 (optional) = g' rounded to bf16.
 * g: fp32 (g_is_bf16 = 0) or bf16, [rows, cols] contiguous; cols % 4 == 0, <= 1024. */
int dab_bias_grad(const void* g, int g_is_bf16, const void* y_bf16, int64_t rows, int cols, float* db, void* g_out_bf16,
                  void* stream) {
  DAB_REQUIRE(g && db && rows >= 0 && cols > 0 && cols % 4 == 0 && cols <= 1024 && aligned16(g) && aligned16(db) &&
                  aligned16(y_bf16) && aligned16(g_out_bf16) && (!g_is_bf16 || cols % 8 == 0),
              DAB_EINVAL, "dab_bias_grad: bad argument (cols %% 4 == 0 (8 for bf16), <= 1024; 16-byte aligned pointers)");
  cudaStream_t s = (cudaStream_t)stream;
  if (cudaMemsetAsync(db, 0, (size_t)cols * sizeof(float), s) != cudaSuccess) return check_launch("dab_bias_grad memset");
  if (rows == 0) return DAB_OK;
  int64_t blocks = (rows + 31) / 32;
  if (blocks > 148) blocks = 148;
  const __nv_bfloat16* y = reinterpret_cast<const __nv_bfloat16*>(y_bf16);
  __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(g_out_bf16);
  if (g_is_bf16)
    colsum_kernel<__nv_bfloat16><<<(unsigned)blocks, 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(g), rows, cols, db, o, y);
  else
    colsum_kernel<float><<<(unsigned)blocks, 256, 0, s>>>(reinterpret_cast<const float*>(g), rows, cols, db, o, y);
  count_launch();
  return check_launch("dab_bias_grad");
}

}  // extern "C"
