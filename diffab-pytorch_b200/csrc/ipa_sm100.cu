// sm_100a fast path of one InvariantPointAttentionLayer (train.py configuration: L=128, D=128, C=64, H=8, ds=32,
// Pq=Pv=8).  Replaces diffab_pytorch.py:389-465 of the reference.
//
// Three launches per layer (dab_ipa_fwd_sm100_train / _stages):
//   1. ipa_proj_kernel (ipa_proj_sm100.cuh): x -> bf16 -> the six projections on tcgen05 -> frame transform (x R + t,
//      centred on the patch centroid), logit scales folded into q, split-bf16 (hi + lo) point coordinates,
//      -0.5 c |k|^2 as extra K columns -> packed operands Qp, Kp, Vp (TMA stores)
//   2. ipa_core_kernel (this file): one persistent CTA per SM with two tile contexts (tile = patch x 16 query rows);
//      TMA-staged tiles, tcgen05.mma with TMEM accumulators; j (keys) sits on the 128 TMEM lanes:
//        S^T_h = K_h Q_h^T          (M=128 j, N=16 i, K=32+3*32)   scalar + expanded point-distance logits
//        + precomputed pair bias (dab_ipa_pair_bias_multi), fp32 softmax over j (warp butterflies, one exchange per row pair)
//        [pair_2p ; pair_2p+1]^T = [e[2p] | e[2p+1]]^T [P_2p ; P_2p+1]^T   (M=128, N=16, K=128 j)  same e tiles, MN-major
//        [O_2m ; O_2m+1]^T = [V_2m | V_2m+1]^T [P_2m ; P_2m+1]^T          (M=128, N=32, K=128 j)  fp16 operands
//      epilogue: normalise, inverse frame, norms -> concat features (bf16)
//   3. gemm_bf16_kernel (gemm_sm100.cuh): y = concat Wout^T + b
// Logits never leave the SM; the pair tensor is read from HBM exactly once per layer.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <stdlib.h>

#include <mutex>

#include "common.cuh"
#include "gemm_sm100.cuh"
#include "ipa_proj_sm100.cuh"
#include "ipa_sm100_layout.cuh"
#include "sm100_prims.cuh"

namespace dab {

// ------------------------------------------------------------------------------------------------
EncodeTiledFn get_encode_tiled() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

int make_tensor_map_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                         const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swizzle) {
  EncodeTiledFn enc = get_encode_tiled();
  DAB_REQUIRE(enc != nullptr, DAB_ELAUNCH, "cuTensorMapEncodeTiled not available (no CUDA driver?)");
  cuuint64_t gdim[5];
  cuuint64_t gstr[5];
  cuuint32_t bdim[5], estr[5];
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bdim[i] = box[i]; estr[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bdim,
                   estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  DAB_REQUIRE(r == CUDA_SUCCESS, DAB_EINVAL, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
  return DAB_OK;
}

namespace sm100 {

#ifdef DAB_DEBUG_HOOKS
static long long* g_core_dbg = nullptr;   // optional timeline buffer (dab_debug_set_timeline; debug build only)
#else
static constexpr long long* g_core_dbg = nullptr;
#endif

// ---- weight packing (once per weight update) -----------------------------------------------------------
// One 32 x 32 tile of a weight matrix per block: fp32 rows in (coalesced), bf16 rows out twice - as they are
// (Wcat [1344][128], Wout [128][1024]) and transposed through shared memory (Wcat^T [128][1344], Wout^T [1024][128],
// the operands of the backward's data-gradient GEMMs).  Block 0 also copies the small fp32 tensors.
__global__ void __launch_bounds__(256) pack_weights_kernel(DabIpaWeights w, uint8_t* packed) {
  __shared__ float tile[32][33];
  const PackedOffsets o = packed_offsets();
  constexpr int kCatTiles = (NPROJ / 32) * (D / 32);      // 42 x 4
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 8 rows per pass
  const float* src;
  __nv_bfloat16 *dst, *dst_t;
  int r0, c0, ld_src, ld_dst, ld_t, row_off = 0;
  int t = blockIdx.x;
  if (t < kCatTiles) {
    const int tr = t / (D / 32), tcn = t % (D / 32);
    r0 = tr * 32; c0 = tcn * 32;
    // source matrix of the row block: q/k/v scalars (256 rows each), q/k/v points (192 rows each); 32 divides both
    const float* srcs[6] = {w.w_q_scalar, w.w_k_scalar, w.w_v_scalar, w.w_q_point, w.w_k_point, w.w_v_point};
    const int seg = r0 < 3 * NS ? r0 / NS : 3 + (r0 - 3 * NS) / NPT;
    row_off = seg < 3 ? seg * NS : 3 * NS + (seg - 3) * NPT;
    src = srcs[seg]; ld_src = D;
    dst = reinterpret_cast<__nv_bfloat16*>(packed + o.wcat); ld_dst = D;
    dst_t = reinterpret_cast<__nv_bfloat16*>(packed + o.wcat_t); ld_t = NPROJ;
  } else {
    t -= kCatTiles;
    const int tr = t / (NCAT / 32), tcn = t % (NCAT / 32);
    r0 = tr * 32; c0 = tcn * 32;
    src = w.w_out; ld_src = NCAT;
    dst = reinterpret_cast<__nv_bfloat16*>(packed + o.wout); ld_dst = NCAT;
    dst_t = reinterpret_cast<__nv_bfloat16*>(packed + o.wout_t); ld_t = D;
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int r = ty + 8 * k;
    const float v = __ldg(src + (size_t)(r0 - row_off + r) * ld_src + c0 + tx);
    tile[r][tx] = v;
    dst[(size_t)(r0 + r) * ld_dst + c0 + tx] = __float2bfloat16_rn(v);
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int c = ty + 8 * k;                              // column of the source tile = row of the transposed copy
    dst_t[(size_t)(c0 + c) * ld_t + r0 + tx] = __float2bfloat16_rn(tile[tx][c]);
  }
  if (blockIdx.x == 0) {
    // raw fp32 pair-bias weights (H x C), used when a layer call arrives without a precomputed bias plane
    float* wpb = reinterpret_cast<float*>(packed + o.wpb);
    for (int i = threadIdx.x; i < H * C; i += 256) wpb[i] = w.w_pair_bias[i];
    float* bout = reinterpret_cast<float*>(packed + o.bout);
    float* gam = reinterpret_cast<float*>(packed + o.gamma);
    for (int i = threadIdx.x; i < D; i += 256) bout[i] = w.b_out[i];
    for (int i = threadIdx.x; i < H; i += 256) gam[i] = w.gamma[i];
  }
}
constexpr int kPackBlocks = (NPROJ / 32) * (D / 32) + (D / 32) * (NCAT / 32);   // 168 + 128

// ---- attention core ---------------------------------------------------------------------------------
// One persistent CTA per SM holds TWO tile contexts (tile = (patch, 16 query rows); local tile k of a CTA runs in
// context k & 1).  A context is a complete tile pipeline - its own softmax / epilogue warps, MMA issuer, probability
// buffers and 256 TMEM columns - but the operand rings are SHARED and dedicated (nothing aliases them):
//   * K ring (3 x 24 KB): K of the patch head by head, tiles in local order;
//   * e/V ring (4 x 16 KB): per tile its 16 pair rows, then the 8 value tiles of its patch.
// Ring order = tile order, so the two contexts run in anti-phase: while one context streams its pair rows (softmax,
// pair aggregation), the other runs its O^T MMAs, its epilogue and the S^T MMAs of its next tile from operands that
// were loaded in the background.  The pair-tensor stream therefore never pauses (two independent CTAs per SM, which
// the kernel used to be, each stopped streaming for more than half of a tile: every operand shared one shared-memory
// region and was loaded only when the stage needing it began).
struct CoreSmem {
  static constexpr int kSlot = L * C * 2;            // 16,384: one pair row [128 j x 64 c] or one value tile [128 j x 64]
  static constexpr int kSlots = 4;
  static constexpr int kRing = 0;
  static constexpr int kKBuf = 3 * L * 64;           // 24,576: one head of K = three [128 x 64 B] blocks
  static constexpr int kKBufs = 3;
  static constexpr int kKRing = kRing + kSlots * kSlot;          // 98,304
  static constexpr int kCtx0 = kKRing + kKBufs * kKBuf;          // 147,456
  // ---- per context ----
  // probabilities per head, B operand of the O^T MMA: [kb(2)][h][16 rows][128 B], fp16.  Its first 24 KB hold Q until
  // the S^T MMAs have completed.  The epilogue works in the 16 KB behind them (tail of P_h + the P_i slots, all idle by
  // then): 12 KB of global-frame points and a 512-byte staging tile per warp - so the next tile's Q may arrive as soon
  // as the O^T MMAs are done, while the epilogue is still running.
  static constexpr int kPh = 0;
  static constexpr int kPhBytes = H * 2 * IB * 128;  // 32,768
  static constexpr int kQBuf = H * 3 * IB * 64;      // 24,576
  // probabilities of a row pair, B operand of the pair MMA, two slots: [slot][kb(2)][16 rows = 8 g + h][128 B], bf16.
  static constexpr int kPi = kPh + kPhBytes;
  static constexpr int kPiSlot = 2 * 2048;
  static constexpr int kCtxBytes = kPi + 2 * kPiSlot;            // 40,960
  static constexpr int kMisc = kCtx0 + 2 * kCtxBytes;            // 229,376
  static constexpr int kRedMax = kMisc;              // [ctx][2 groups][2 parity][4 warps][16] f32
  static constexpr int kBars = kRedMax + 2 * 1024;
  static constexpr int kNumBars = 48;
  static constexpr int kTmemSlot = kBars + kNumBars * 8;
  static constexpr int kTotal = kTmemSlot + 16;
};
static_assert(CoreSmem::kQBuf <= CoreSmem::kPhBytes, "Q must fit the idle P_h region");
static_assert(CoreSmem::kTotal <= 227 * 1024, "one CTA per SM");

// shared rings
// K_TURN / R_TURN hand the shared rings from one context's issuer to the other's: completion k = the issuer of local
// tile k has observed every K (every pair-row / value) entry of that tile, so the next tile's issuer may start waiting on
// the ring's full barriers (whose parities would otherwise alias with the entries of the tile before).
enum Bar { K_FULL = 0, K_EMPTY = 3, R_FULL = 6, R_EMPTY = 10, K_TURN = 14, R_TURN = 15, CTX_BARS = 16, N_BARS = 16 + 2 * 13 };
// per context (index CTX_BARS + 13 * ctx + ...)
enum CtxBar { Q_FULL = 0, S_DONE = 1, PAIR = 2 /* [slot] */, O_DONE = 4, P_READY = 5 /* [group][slot], 128 arrivals */,
              EPI_TMEM = 9 /* 256 arrivals: epilogue has read every accumulator */,
              EPI_DONE = 10 /* 256: the P_h region is free for the next Q */,
              EPI_SFREE = 11 /* 256: the O^T accumulators (columns of S^T) have been read */, N_CTX_BARS = 13 };
static_assert(N_BARS <= CoreSmem::kNumBars, "barrier storage");

// TMEM columns (per context: + 256 * ctx)
constexpr uint32_t kColS = 0, kColPair = 128 /* 16 rows x 8 */, kTmemCols = 512;

// Reduce 8 per-lane values across the warp with 9 shuffles; lane ends up with the result for head
// hsel = 4*bit4 + 2*bit3 + bit2 of its lane id (every group of 4 lanes holds the same head).
template <bool IS_MAX>
__device__ __forceinline__ float warp_reduce8(const float (&v)[8], int lane) {
  auto op = [](float a, float b) { return IS_MAX ? fmaxf(a, b) : a + b; };
  const bool u1 = lane & 16, u2 = lane & 8, u3 = lane & 4;
  float a[4], bq[2];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float send = u1 ? v[k] : v[k + 4], keep = u1 ? v[k + 4] : v[k];
    a[k] = op(keep, __shfl_xor_sync(0xffffffffu, send, 16));
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    float send = u2 ? a[k] : a[k + 2], keep = u2 ? a[k + 2] : a[k];
    bq[k] = op(keep, __shfl_xor_sync(0xffffffffu, send, 8));
  }
  float send = u3 ? bq[0] : bq[1], keep = u3 ? bq[1] : bq[0];
  float c = op(keep, __shfl_xor_sync(0xffffffffu, send, 4));
  c = op(c, __shfl_xor_sync(0xffffffffu, c, 2));
  c = op(c, __shfl_xor_sync(0xffffffffu, c, 1));
  return c;
}

// Maximum of 16 per-lane values across the warp with 16 shuffles; lane ends up with the result for value
// index 8*bit4 + 4*bit3 + 2*bit2 + bit1 of its lane id (lane pairs hold the same value).
__device__ __forceinline__ float warp_reduce16_max(const float (&v)[16], int lane) {
  const bool u1 = lane & 16, u2 = lane & 8, u3 = lane & 4, u4 = lane & 2;
  float a[8], b4[4], c2[2];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    float send = u1 ? v[k] : v[k + 8], keep = u1 ? v[k + 8] : v[k];
    a[k] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 16));
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    float send = u2 ? a[k] : a[k + 4], keep = u2 ? a[k + 4] : a[k];
    b4[k] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 8));
  }
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    float send = u3 ? b4[k] : b4[k + 2], keep = u3 ? b4[k + 2] : b4[k];
    c2[k] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 4));
  }
  float send = u4 ? c2[0] : c2[1], keep = u4 ? c2[1] : c2[0];
  float d = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, 2));
  return fmaxf(d, __shfl_xor_sync(0xffffffffu, d, 1));
}

__device__ __forceinline__ void tmem_ld_x4(uint32_t taddr, float (&v)[4]) {
  uint32_t r[4];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = __uint_as_float(r[i]);
}

// Warp roles (640 threads).  Context c = 0, 1: warps 8c .. 8c+7 are its two softmax/epilogue groups of 128 threads
// (thread t of a group owns key j = t = TMEM lane t; group g handles query rows i = g, g+2, ...); warp 16 + c lane 0
// issues the context's tcgen05.mma; warp 18 lane 0 issues the K / Q loads of both contexts, warp 19 lane 0 the pair-row
// and value loads.  The roles meet only at mbarriers.
// `bias` is the layer's precomputed pair bias, fp16 [B*L rows i][128 j][8 h], already scaled by
// scale_total * log2(e) (dab_ipa_pair_bias_multi): e is constant over the six layers and the T steps, so the
// e . Wpb contraction is hoisted out of the sampling loop entirely.
// `live` (optional): ascending ids of the query tiles to compute (query tile = global row / 16), their count in
// live_count[0]; the rows of the other tiles are left as they are.  n_tiles is then the upper bound of the kernel tiles.
constexpr int kCoreThreads = 640;
// KB2: key-block mode for patches of 256 residues (see `decode` below); false: the L = 128 kernel.  LIVE: `live` is given
// (a template argument so that the full-grid kernels stay exactly as they were)
template <bool KB2, bool LIVE>
__global__ void __launch_bounds__(kCoreThreads, 1)
ipa_core_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_e,
                const uint4* __restrict__ bias, const float* __restrict__ tc, const float* __restrict__ R,
                __nv_bfloat16* __restrict__ cat, float* __restrict__ stats, uint4* __restrict__ pu,
                int n_tiles, long long* __restrict__ dbg, int64_t out_stride, const int* __restrict__ live,
                const int* __restrict__ live_count) {
  extern __shared__ __align__(1024) uint8_t smem[];
  // optional per-tile timeline: slot k of tile c at dbg[c * 64 + k]
  long long* dbg_cta = nullptr;
#define DAB_STAMP(k) do { if (dbg_cta && (threadIdx.x & 255) == 0) dbg_cta[(k)] = clock64(); } while (0)
#define DAB_STAMP_ISSUER(k) do { if (dbg_cta) dbg_cta[(k)] = clock64(); } while (0)
  // wait on a barrier, adding the cycles spent to `acc` when the timeline is on
#define DAB_TIMED_WAIT(bar, par, acc) do { if (dbg) { long long t0_ = clock64(); mbar_wait((bar), (par)); (acc) += clock64() - t0_; } else mbar_wait((bar), (par)); } while (0)
  using S = CoreSmem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kBars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::kTmemSlot);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0) asm volatile("trap;");
  // with a live-tile list: each live query tile is one kernel tile (two in key-block mode, one per key block); a CTA
  // left without tiles falls straight through to the teardown
  if (LIVE) n_tiles = min(n_tiles, (KB2 ? 2 : 1) * __ldg(live_count));
  // local tiles of this CTA: k = 0, 1, ... -> global tile blockIdx.x + k * gridDim.x, context k & 1
  const int n_local = (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  // Tiles are walked from the LAST patch down: the projection kernel has just written the packed operands in ascending
  // patch order, so the highest patches are the ones still resident in L2 (and the to_out GEMM, which starts with patch
  // 0, finds the concat features this kernel wrote last).  The pair rows are streamed with an evict-first policy so that
  // they do not push those operands out of L2.
  auto tile_of = [&](int k) {
    const int x = n_tiles - 1 - ((int)blockIdx.x + k * (int)gridDim.x);
    if (!LIVE) return x;
    if (!KB2) return __ldg(live + x);
    const int q = __ldg(live + (x >> 1));          // query tile -> (query block, key block x & 1), same row group
    return ((((q >> 3) << 1) | (x & 1)) << 3) | (q & 7);
  };
  // A tile = 16 query rows against one block of 128 keys.  Plain mode (KB2 = false): tile >> 3 = patch, keys = the patch.
  // Key-block mode (KB2, patches of 256 residues = two blocks): tile >> 3 = (query block, key block) pair; the pair
  // tensor / bias rows are 256 pairs long and the key block starts at pair 128 kb of the row; the (normalised) result and
  // its softmax statistics go to slice kb of the outputs (out_stride rows apart) and are merged afterwards.
  struct TileIdx { int64_t q0, kv0, o0; int lrow, joff; };
  auto decode = [&](int tile) {
    TileIdx ti;
    const int v = tile >> 3, it = tile & 7;
    if (KB2) {
      const int qblk = v >> 1, kb = v & 1;
      ti.q0 = (int64_t)qblk * L + it * IB;
      ti.kv0 = (int64_t)((qblk & ~1) + kb) * L;
      ti.o0 = (int64_t)kb * out_stride + ti.q0;
      ti.lrow = 2 * L; ti.joff = kb * L;
    } else {
      ti.q0 = (int64_t)v * L + it * IB; ti.kv0 = (int64_t)v * L; ti.o0 = ti.q0; ti.lrow = L; ti.joff = 0;
    }
    return ti;
  };
  // Ring bookkeeping.  e/V entry at ring position x of a tile (pair row r: x = r; value tile h: x = 16 + h): slot x % 4,
  // completion x / 4 of the tile - 24 entries on 4 slots are 6 completions per slot and tile, an even number, so the
  // parity of an entry depends only on its position inside the tile.  Rows 2p, 2p+1 and value tiles 2m, 2m+1 always sit
  // in adjacent slots (the MMA descriptors address the pair with one leading-dimension stride).
  auto pos_e = [](int r) { return r; };
  auto pos_v = [](int h) { return IB + h; };
  // K ring (3 slots): slots 0 and 1 complete three times per tile, slot 2 twice - the parity carries the local tile index
  auto k_use = [](int k, int h) { return k * (h % 3 == 2 ? 2 : 3) + h / 3; };

  if (tid == 0) {
    for (int i = 0; i < CTX_BARS; ++i) mbar_init(&bars[i], 1u);   // rings and turn barriers
    for (int c = 0; c < 2; ++c)
      for (int i = 0; i < N_CTX_BARS; ++i)
        mbar_init(&bars[CTX_BARS + N_CTX_BARS * c + i], (i >= P_READY && i < P_READY + 4) ? 128u : (i >= EPI_TMEM ? 256u : 1u));
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(tmem_slot, kTmemCols);
  tcgen05_fence_before_sync();
  __syncthreads();
  tcgen05_fence_after_sync();
  const uint32_t tmem_cta = *tmem_slot;

  if (warp == 18) {
    // ======================================= TMA producer: K ring and Q =======================================
    if (lane == 0) {
      tma_prefetch_desc(&map_q); tma_prefetch_desc(&map_k);
      for (int k = 0; k < n_local; ++k) {
        const int c = k & 1, n = k >> 1, tile = tile_of(k);
        const TileIdx ti = decode(tile);
        const int64_t row0 = ti.q0;
        const int kvrow = (int)ti.kv0;
        uint64_t* cb = bars + CTX_BARS + N_CTX_BARS * c;
        uint8_t* cs = smem + S::kCtx0 + c * S::kCtxBytes;
        auto load_k = [&](int h) {
          const int s = h % S::kKBufs;
          if (k > 0 || h >= S::kKBufs) mbar_wait(&bars[K_EMPTY + s], (k_use(k, h) - 1) & 1);
          uint8_t* kb = smem + S::kKRing + s * S::kKBuf;
          mbar_arrive_expect_tx(&bars[K_FULL + s], S::kKBuf);
          for (int blk = 0; blk < 3; ++blk)
            tma_load_2d(kb + blk * (L * 64), &map_k, &bars[K_FULL + s], (h * 3 + blk) * 32, kvrow);
        };
        // the first two heads of K go out as soon as the ring has room (i.e. while the context is still busy with its
        // previous tile); Q goes into the context's P_h region, free once the O^T MMAs of that tile have completed
        load_k(0);
        load_k(1);
        load_k(2);
        if (n > 0) mbar_wait(&cb[O_DONE], (n - 1) & 1);
        mbar_arrive_expect_tx(&cb[Q_FULL], S::kQBuf);
        for (int blk = 0; blk < H * 3; ++blk)    // [blk][16 rows][64 B], 64B swizzle
          tma_load_2d(cs + S::kPh + blk * (IB * 64), &map_q, &cb[Q_FULL], blk * 32, (int)row0);
        for (int h = S::kKBufs; h < H; ++h) load_k(h);
      }
    }
  } else if (warp == 19) {
    // ======================================= TMA producer: pair rows and value tiles =======================================
    // The ring is only four tiles deep, far less than the HBM latency-bandwidth product, so pair rows are pulled
    // HBM -> L2 kL2Ahead rows ahead (across the tile boundary) with TMA prefetches and the ring is fed from L2.
    if (lane == 0) {
      tma_prefetch_desc(&map_v); tma_prefetch_desc(&map_e);
      const uint64_t pol = policy_evict_first();
#ifndef DAB_L2_AHEAD
#define DAB_L2_AHEAD 8
#endif
      constexpr int kL2Ahead = DAB_L2_AHEAD;   // <= IB
      // pair index of (query row r of tile k, first key of the tile's key block)
      auto pair0_of = [&](int k, int r) { const TileIdx ti = decode(tile_of(k)); return (int)((ti.q0 + r) * ti.lrow + ti.joff); };
      if (n_local > 0)
        for (int r = 0; r < kL2Ahead; ++r) tma_prefetch_l2_2d_hint(&map_e, 0, pair0_of(0, r), pol);
      for (int k = 0; k < n_local; ++k) {
        const int kvrow = (int)decode(tile_of(k)).kv0;
        const bool has_next = k + 1 < n_local;
        for (int x = 0; x < IB + H; ++x) {
          const int s = x % S::kSlots;
          if (k > 0 || x >= S::kSlots) mbar_wait(&bars[R_EMPTY + s], ((x / S::kSlots) + 1) & 1);
          mbar_arrive_expect_tx(&bars[R_FULL + s], S::kSlot);
          if (x < IB) {
            tma_load_2d_hint(smem + S::kRing + s * S::kSlot, &map_e, &bars[R_FULL + s], 0, pair0_of(k, x), pol);
            const int a = x + kL2Ahead;
            if (a < IB) tma_prefetch_l2_2d_hint(&map_e, 0, pair0_of(k, a), pol);
            else if (has_next) tma_prefetch_l2_2d_hint(&map_e, 0, pair0_of(k + 1, a - IB), pol);
          } else {
            tma_load_2d(smem + S::kRing + s * S::kSlot, &map_v, &bars[R_FULL + s], (x - IB) * V_W, kvrow);
          }
        }
      }
    }
  } else if (warp >= 16) {
    // ======================================= MMA issuer of context c =======================================
    // The whole warp runs the control flow (warp-uniform values stay in uniform registers: a single divergent lane
    // spent ~20 instructions per MMA moving descriptors into them) and one elected lane issues.
    const int c = __shfl_sync(0xffffffffu, warp, 0) - 16;
    {
      constexpr uint32_t kIdescS = make_idesc_bf16(128, 16, 0, 0);     // S^T
      constexpr uint32_t kIdescPair = make_idesc_bf16(128, 16, 1, 0);  // A = two e tiles, MN-major
      constexpr uint32_t kIdescO = make_idesc_f16(128, 32, 1, 0);      // A = two V tiles, MN-major, fp16 operands
      uint64_t* cb = bars + CTX_BARS + N_CTX_BARS * c;
      const uint32_t cs = smem_base + S::kCtx0 + c * S::kCtxBytes;
      const uint32_t tmem = tmem_cta + 256u * c;
      // descriptors advance by adding (bytes >> 4) to their low word (addresses stay below 256 KB: no carry out of the field)
      const uint64_t dK0 = make_smem_desc(smem_base + S::kKRing, 16, 512, kSwizzle64B);
      const uint64_t dQ0 = make_smem_desc(cs + S::kPh, 16, 512, kSwizzle64B);
      const uint64_t dR0 = make_smem_desc(smem_base + S::kRing, S::kSlot, 1024, kSwizzle128B);
      const uint64_t dPi0 = make_smem_desc(cs + S::kPi, 16, 1024, kSwizzle128B);
      const uint64_t dPh0 = make_smem_desc(cs + S::kPh, 16, 1024, kSwizzle128B);
      for (int k = c, n = 0; k < n_local; k += 2, ++n) {
        dbg_cta = (dbg && lane == 0) ? dbg + (size_t)tile_of(k) * 64 : nullptr;
        long long w_q = 0, w_sfree = 0, w_kturn = 0, w_k = 0, w_epit = 0, w_rturn = 0, w_e = 0, w_p = 0, w_v = 0;
        DAB_STAMP_ISSUER(16);
        // ---- stage 1: S^T_h = K_h Q_h^T for the 8 heads
        DAB_TIMED_WAIT(&cb[Q_FULL], n & 1, w_q);
        if (n > 0) {                                   // the previous tile's epilogue has read the O^T accumulators
          DAB_TIMED_WAIT(&cb[EPI_SFREE], (n - 1) & 1, w_sfree);      // (same columns as S^T; the pair accumulators are waited for below)
        }
        if (k > 0) DAB_TIMED_WAIT(&bars[K_TURN], (k - 1) & 1, w_kturn);
        tcgen05_fence_after_sync();
        DAB_STAMP_ISSUER(1);
        for (int h = 0; h < H; ++h) {
          const int s = h % S::kKBufs;
          DAB_TIMED_WAIT(&bars[K_FULL + s], k_use(k, h) & 1, w_k);
          tcgen05_fence_after_sync();
          DAB_STAMP_ISSUER(48 + h);
          if (elect_one()) {
            const uint64_t ka = dK0 + (uint32_t)((s * S::kKBuf) >> 4);
            const uint64_t qa = dQ0 + (uint32_t)((h * 3 * (IB * 64)) >> 4);
#pragma unroll
            for (int m = 0; m < 4; ++m) {
              // (A block, B block): scalar.scalar, hi.hi (+ norm columns), hi.lo, lo.hi
              const int ablk = (m == 0) ? 0 : (m == 3 ? 2 : 1), bblk = (m == 0) ? 0 : (m == 2 ? 2 : 1);
#pragma unroll
              for (int kk = 0; kk < 2; ++kk)
                umma_bf16(tmem + kColS + h * 16, ka + (uint32_t)((ablk * (L * 64) + kk * 32) >> 4),
                          qa + (uint32_t)((bblk * (IB * 64) + kk * 32) >> 4), kIdescS, (m | kk) != 0);
            }
            umma_commit(&bars[K_EMPTY + s]);
          }
          __syncwarp();
        }
        if (elect_one()) {
          umma_commit(&cb[S_DONE]);
          mbar_arrive(&bars[K_TURN]);
        }
        __syncwarp();
        DAB_STAMP_ISSUER(2);
        // ---- stage 2: pair aggregation of TWO rows per MMA chain (rows 2p and 2p+1, one from each softmax group):
        //      [pair_2p ; pair_2p+1]^T = [e[2p] | e[2p+1]]^T [P_2p ; P_2p+1]^T  (M = 128: 64 channels of each row,
        //      N = 16: 8 heads of each row, K = 128 j).  The two off-diagonal blocks (row 2p channels x row 2p+1
        //      probabilities and vice versa) are computed and ignored: a small tcgen05.mma costs the same
        //      whatever its shape, so halving the instruction count is what matters.
        if (n > 0) DAB_TIMED_WAIT(&cb[EPI_TMEM], (n - 1) & 1, w_epit);    // previous tile's pair accumulators drained
        if (k > 0) DAB_TIMED_WAIT(&bars[R_TURN], (k - 1) & 1, w_rturn);
        DAB_STAMP_ISSUER(17);
        for (int p = 0; p < IB / 2; ++p) {
          const int x = pos_e(2 * p), st = x % S::kSlots;     // rows 2p, 2p+1 sit in consecutive ring slots
          const int slot = p & 1;
          DAB_TIMED_WAIT(&bars[R_FULL + st], (x / S::kSlots) & 1, w_e);
          DAB_TIMED_WAIT(&bars[R_FULL + st + 1], (x / S::kSlots) & 1, w_e);
          if (p == 4) DAB_STAMP_ISSUER(41);
          DAB_TIMED_WAIT(&cb[P_READY + slot], (p >> 1) & 1, w_p);          // group 0, row 2p
          DAB_TIMED_WAIT(&cb[P_READY + 2 + slot], (p >> 1) & 1, w_p);      // group 1, row 2p + 1
          tcgen05_fence_after_sync();
          if (p == 4) DAB_STAMP_ISSUER(42);
          if (elect_one()) {
            // A: two e tiles [j][c] read MN-major: M = 128 = two 64-wide atoms one ring slot apart (LBO);
            //    K = j: 16 rows = 2048 B per step, 8-row groups 1024 B apart (SBO)
            const uint64_t ea = dR0 + (uint32_t)((st * S::kSlot) >> 4);
            const uint64_t pa = dPi0 + (uint32_t)((slot * S::kPiSlot) >> 4);
#pragma unroll
            for (int kk = 0; kk < L / 16; ++kk)
              umma_bf16(tmem + kColPair + p * 16, ea + (uint32_t)((kk * 2048) >> 4),
                        pa + (uint32_t)(((kk >> 2) * 2048 + (kk & 3) * 32) >> 4), kIdescPair, kk != 0);
            umma_commit(&cb[PAIR + slot]);
            umma_commit(&bars[R_EMPTY + st]);
            umma_commit(&bars[R_EMPTY + st + 1]);
          }
          __syncwarp();
          if (p == 4) DAB_STAMP_ISSUER(43);
        }
        DAB_STAMP_ISSUER(3);
        // ---- stage 3: O^T of TWO heads per MMA chain: [O_2m ; O_2m+1]^T = [V_2m | V_2m+1]^T [P_2m ; P_2m+1]^T
        //      (M = 128: 64 value columns of each head, N = 32: 16 rows of each head, K = 128 j)
        for (int m = 0; m < H / 2; ++m) {
          const int x = pos_v(2 * m), st = x % S::kSlots;
          DAB_TIMED_WAIT(&bars[R_FULL + st], (x / S::kSlots) & 1, w_v);
          DAB_TIMED_WAIT(&bars[R_FULL + st + 1], (x / S::kSlots) & 1, w_v);
          tcgen05_fence_after_sync();
          DAB_STAMP_ISSUER(56 + m);
          if (elect_one()) {
            const uint64_t va = dR0 + (uint32_t)((st * S::kSlot) >> 4);
            const uint64_t pa = dPh0 + (uint32_t)(((2 * m) * (IB * 128)) >> 4);
#pragma unroll
            for (int kk = 0; kk < L / 16; ++kk)
              umma_bf16(tmem + kColS + m * 32, va + (uint32_t)((kk * 2048) >> 4),
                        pa + (uint32_t)(((kk >> 2) * (H * IB * 128) + (kk & 3) * 32) >> 4), kIdescO, kk != 0);
            umma_commit(&bars[R_EMPTY + st]);
            umma_commit(&bars[R_EMPTY + st + 1]);
          }
          __syncwarp();
        }
        if (elect_one()) {
          umma_commit(&cb[O_DONE]);
          mbar_arrive(&bars[R_TURN]);
        }
        __syncwarp();
        DAB_STAMP_ISSUER(7);
        if (dbg_cta) {
          dbg_cta[18] = w_q; dbg_cta[19] = w_sfree; dbg_cta[20] = w_kturn; dbg_cta[21] = w_k; dbg_cta[22] = w_epit;
          dbg_cta[23] = w_rturn; dbg_cta[25] = w_e; dbg_cta[26] = w_p; dbg_cta[27] = w_v;
        }
      }
    }
  } else {
    // ======================================= softmax / epilogue groups of context c =======================================
    const int c = warp >> 3, cw = warp & 7;              // context, warp inside the context
    const int g = cw >> 2, gw = cw & 3, gt = tid & 127, ct = tid & 255;
    uint64_t* cb = bars + CTX_BARS + N_CTX_BARS * c;
    uint8_t* cs = smem + S::kCtx0 + c * S::kCtxBytes;
    const uint32_t tmem = tmem_cta + 256u * c;
    const uint32_t tmem_lane = tmem + ((uint32_t)(gw * 32) << 16);
    // value index this lane ends up with after warp_reduce16: 8*bit4 + 4*bit3 + 2*bit2 + bit1
    const int vsel = ((lane >> 4) & 1) * 8 + ((lane >> 3) & 1) * 4 + ((lane >> 2) & 1) * 2 + ((lane >> 1) & 1);
    float* red_max = reinterpret_cast<float*>(smem + S::kRedMax) + c * 256 + g * 128;    // [parity][4 warps][16]
    float* red_ctx = reinterpret_cast<float*>(smem + S::kRedMax) + c * 256;
    float* inv_o = red_ctx;                                    // [16][8] f32: 1 / sum_j p (epilogue only: the maxima buffer of group 0 / 1 is idle then)
    auto bar_group = [&] { asm volatile("bar.sync %0, 128;" ::"r"(1 + 2 * c + g) : "memory"); };
    auto bar_all_compute = [&] { asm volatile("bar.sync %0, 256;" ::"r"(5 + c) : "memory"); };
    (void)ct;

   for (int k = c, tn = 0; k < n_local; k += 2, ++tn) {
    const int tile = tile_of(k);
    const TileIdx ti = decode(tile);
    const int64_t row0 = ti.q0;          // first query row (global residue index): frames, centred translations
    const int64_t orow0 = KB2 ? ti.o0 : row0;       // first row of the outputs (concat features, statistics)
    constexpr int64_t LR = KB2 ? 2 * L : L;         // pairs per row of the pair tensor / the bias planes
    dbg_cta = dbg ? dbg + (size_t)tile * 64 : nullptr;
    long long w_pair = 0;
    DAB_STAMP(0);
    // pair bias of this thread's key for the group's rows, one quarter (two rows) ahead in registers
    const uint4* bias_t = bias + (row0 + g) * LR + (KB2 ? ti.joff : 0) + gt;      // local row n (i = 2n + g)  ->  + n * 2 * LR
    uint4 b_cur[2] = {__ldg(bias_t), __ldg(bias_t + 2 * LR)};
    uint4 b_nxt[2] = {__ldg(bias_t + 4 * LR), __ldg(bias_t + 6 * LR)};
    mbar_wait(&cb[S_DONE], tn & 1);
    tcgen05_fence_after_sync();
    DAB_STAMP(6);
    // Four quarters of the 16 query rows; this group owns rows 4q + g and 4q + 2 + g of each quarter and
    // treats them together: one butterfly and one group barrier give the 2 x 8 row maxima.
    for (int q = 0; q < IB / 4; ++q) {
      const uint4 b_use[2] = {b_cur[0], b_cur[1]};
      b_cur[0] = b_nxt[0]; b_cur[1] = b_nxt[1];
      if (q + 2 < IB / 4) {
        b_nxt[0] = __ldg(bias_t + (size_t)(2 * q + 4) * 2 * LR);
        b_nxt[1] = __ldg(bias_t + (size_t)(2 * q + 5) * 2 * LR);
      }
      float sreg[H][4];
#pragma unroll
      for (int h = 0; h < H; ++h) tmem_ld_x4(tmem_lane + kColS + h * 16 + 4 * q, sreg[h]);
      tmem_wait_ld();
      if (q == IB / 4 - 1) tcgen05_fence_before_sync();
      if (q == 2) DAB_STAMP(33);
      float lg[16];
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const __half2* hb = reinterpret_cast<const __half2*>(&b_use[r]);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          float2 f = __half22float2(hb[kk]);
          lg[r * 8 + 2 * kk] = f.x; lg[r * 8 + 2 * kk + 1] = f.y;
        }
#pragma unroll
        for (int h = 0; h < H; ++h) {
          const float sv = g == 0 ? (r == 0 ? sreg[h][0] : sreg[h][2]) : (r == 0 ? sreg[h][1] : sreg[h][3]);
          lg[r * 8 + h] += sv;
        }
      }
      // ---- row maxima over j (the 128 lanes), in log2 units
      float wm = warp_reduce16_max(lg, lane);
      float* rm = red_max + (q & 1) * 64;
      if ((lane & 1) == 0) rm[gw * 16 + vsel] = wm;
      bar_group();
      if (q == 2) DAB_STAMP(34);
      float mx[16];
      {
        const float4* r4 = reinterpret_cast<const float4*>(rm);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          float4 a = r4[kk], bb = r4[4 + kk], cc = r4[8 + kk], dd = r4[12 + kk];
          mx[4 * kk] = fmaxf(fmaxf(a.x, bb.x), fmaxf(cc.x, dd.x));
          mx[4 * kk + 1] = fmaxf(fmaxf(a.y, bb.y), fmaxf(cc.y, dd.y));
          mx[4 * kk + 2] = fmaxf(fmaxf(a.z, bb.z), fmaxf(cc.z, dd.z));
          mx[4 * kk + 3] = fmaxf(fmaxf(a.w, bb.w), fmaxf(cc.w, dd.w));
        }
      }
      if (stats && gt < 16) {   // row maxima (log2 units) of the group's two rows, kept for the backward
        float v = mx[0];
#pragma unroll
        for (int kk = 1; kk < 16; ++kk) v = (kk == gt) ? mx[kk] : v;
        stats[(orow0 + 2 * (2 * q + (gt >> 3)) + g) * 16 + (gt & 7)] = v;
      }
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int n = 2 * q + r, i = 2 * n + g;
        float p[8];
#pragma unroll
        for (int h = 0; h < H; ++h) p[h] = ex2(lg[r * 8 + h] - mx[r * 8 + h]);
        if (pu)   // training: keep the un-normalised probabilities (bf16, [i][j][h]) for the backward
          pu[(row0 + i) * L + gt] = make_uint4(pack_bf162(p[0], p[1]), pack_bf162(p[2], p[3]), pack_bf162(p[4], p[5]),
                                               pack_bf162(p[6], p[7]));
        // the pair MMA that last read this P_i slot (row n-2 of this group) must have completed
        if (n >= 2) DAB_TIMED_WAIT(&cb[PAIR + (n & 1)], ((n >> 1) - 1) & 1, w_pair);
        // ---- probabilities -> shared memory in the two operand layouts (K-major, 128B swizzle); neighbouring
        //      lanes trade heads so that every store is a packed pair (j, j+1).  Un-normalised: the row sums come
        //      out of the O^T MMA itself (ones column of the V operand) and are applied in the epilogue.
        {
          const int je = gt & ~1;                                   // even key of the pair
          const uint32_t kb = je >> 6, chunk = (je & 63) >> 3, e2 = (je & 7) * 2;
          uint8_t* pi = cs + S::kPi + (n & 1) * S::kPiSlot + kb * 2048 + g * 1024;   // [kb][row = 8 g + h][128 B]
          uint8_t* ph = cs + S::kPh + kb * (H * IB * 128);                            // [kb][h][16 i][128 B]
          const bool odd = lane & 1;
#pragma unroll
          for (int hh = 0; hh < 4; ++hh) {
            float send = odd ? p[2 * hh] : p[2 * hh + 1];
            float recv = __shfl_xor_sync(0xffffffffu, send, 1);
            const int h = 2 * hh + (odd ? 1 : 0);
            float lo = odd ? recv : p[2 * hh], hi = odd ? p[2 * hh + 1] : recv;   // (p_j, p_{j+1}) of head h
            *reinterpret_cast<uint32_t*>(pi + swz128_offset(h, chunk) + e2) = pack_bf162(lo, hi);
            *reinterpret_cast<uint32_t*>(ph + h * (IB * 128) + swz128_offset(i, chunk) + e2) = pack_h2(lo, hi);
          }
        }
        fence_proxy_async_smem();
        tcgen05_fence_before_sync();
        mbar_arrive(&cb[P_READY + g * 2 + (n & 1)]);
        if (g == 0) DAB_STAMP(8 + n);
      }
    }
    DAB_STAMP(24);
    if (dbg_cta && (tid & 255) == 0) dbg_cta[28] = w_pair;

    // ---- epilogue.  O^T of head pair m sits in columns 32 m .. 32 m + 31 (M = 128): TMEM lane d (warps 0, 1)
    //      = value column d of head 2m with the 16 rows in columns 0..15; lane 64 + d (warps 2, 3) = head 2m + 1
    //      with its rows in columns 16..31.  d < 32 scalar values, 32..55 point coordinates, d = 56 the row sum of
    //      the probabilities (ones column of V).  Group g takes head pairs 2g, 2g + 1.
    // frame of the (residue, head) task this thread finishes with: fetched now, used after the O^T MMAs
    float Rm[9], tfr[3];
    {
      const int64_t row = row0 + (gt >> 3);
#pragma unroll
      for (int cc = 0; cc < 9; ++cc) Rm[cc] = __ldg(R + row * 9 + cc);
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) tfr[cc] = __ldg(tc + row * 3 + cc);
    }
    // 512 B per warp behind the global-frame points
    uint8_t* stage_e = cs + S::kPh + S::kQBuf + 12288 + cw * 512;
    mbar_wait(&cb[O_DONE], tn & 1);
    tcgen05_fence_after_sync();
    DAB_STAMP(4);
    const int hsel = gw >> 1;                    // which head of the pair this warp's lanes hold
    const uint32_t ocol = kColS + (uint32_t)hsel * 16;
    if (gw & 1) {                // d = 32 + lane: lane 24 holds the normalisers
#pragma unroll
      for (int mm = 0; mm < 2; ++mm) {
        const int m = 2 * g + mm, h = 2 * m + hsel;
        float o[16];
        tmem_ld_x16(tmem_lane + ocol + m * 32, o);
        tmem_wait_ld();
        if (lane == 24) {
#pragma unroll
          for (int i = 0; i < IB; ++i) inv_o[i * H + h] = __fdividef(1.0f, o[i]);
        }
      }
    }
    bar_all_compute();
    if (stats && g == 0) stats[(orow0 + (gt >> 3)) * 16 + 8 + (gt & 7)] = inv_o[gt];
    // [16 i][8 h][24] global-frame points, behind the Q area of the P_h region
    float* s_og = reinterpret_cast<float*>(cs + S::kPh + S::kQBuf);
#pragma unroll
    for (int mm = 0; mm < 2; ++mm) {
      const int m = 2 * g + mm, h = 2 * m + hsel;
      float o[16];
      tmem_ld_x16(tmem_lane + ocol + m * 32, o);
      tmem_wait_ld();
      if ((gw & 1) == 0) {       // scalar values: d = lane
        __nv_bfloat16* st16 = reinterpret_cast<__nv_bfloat16*>(stage_e);
#pragma unroll
        for (int r = 0; r < 2; ++r) {   // two halves of 8 rows: [8 i][64 B] -> 32 chunks of 16 B, one per lane
#pragma unroll
          for (int i = 0; i < 8; ++i) st16[i * 32 + lane] = __float2bfloat16_rn(o[8 * r + i] * inv_o[(8 * r + i) * H + h]);
          __syncwarp();
          const int i = 8 * r + (lane >> 2), part = lane & 3;
          *reinterpret_cast<uint4*>(cat + (orow0 + i) * NCAT + h * DS + part * 8) = reinterpret_cast<const uint4*>(stage_e)[lane];
          __syncwarp();
        }
      } else if (lane < 3 * P) { // point coordinates: d - 32 = lane
#pragma unroll
        for (int i = 0; i < IB; ++i) s_og[(i * H + h) * 24 + lane] = o[i] * inv_o[i * H + h];
      }
    }
    tcgen05_fence_before_sync();
    mbar_arrive(&cb[EPI_SFREE]);    // O^T read: the next tile's S^T MMAs may overwrite these columns
    bar_all_compute();
    // inverse frame + norms (diffab_pytorch.py:327-336,453-457): ol[c'] = sum_k (og[k] - t[k]) R[c'][k];
    // thread (i, h) handles the 8 points of one head -> 48 + 16 contiguous bytes
    if (g == 0) {
      const int i = gt >> 3, h = gt & 7;
      const int64_t row = row0 + i;
      const float* gp = s_og + (i * H + h) * 24;
      const float tx = tfr[0], ty = tfr[1], tz = tfr[2];
      float out[24], nrm[8];
#pragma unroll
      for (int p = 0; p < P; ++p) {
        float gx = gp[3 * p] - tx, gy = gp[3 * p + 1] - ty, gz = gp[3 * p + 2] - tz;
        float lx = gx * Rm[0] + gy * Rm[1] + gz * Rm[2];
        float ly = gx * Rm[3] + gy * Rm[4] + gz * Rm[5];
        float lz = gx * Rm[6] + gy * Rm[7] + gz * Rm[8];
        out[3 * p] = lx; out[3 * p + 1] = ly; out[3 * p + 2] = lz;
        nrm[p] = sqrtf(lx * lx + ly * ly + lz * lz);
      }
      const int64_t orow = orow0 + i;
      uint4* dpt = reinterpret_cast<uint4*>(cat + orow * NCAT + NS + H * C + h * 24);
#pragma unroll
      for (int q = 0; q < 3; ++q)
        dpt[q] = make_uint4(pack_bf162(out[8 * q], out[8 * q + 1]), pack_bf162(out[8 * q + 2], out[8 * q + 3]),
                            pack_bf162(out[8 * q + 4], out[8 * q + 5]), pack_bf162(out[8 * q + 6], out[8 * q + 7]));
      *reinterpret_cast<uint4*>(cat + orow * NCAT + NS + H * C + NPT + h * 8) =
          make_uint4(pack_bf162(nrm[0], nrm[1]), pack_bf162(nrm[2], nrm[3]), pack_bf162(nrm[4], nrm[5]),
                     pack_bf162(nrm[6], nrm[7]));
    }
    // pair aggregation: accumulator n (16 columns) holds rows 2n (lanes 0-63 = channel c, columns 0-7 = heads) and
    // 2n + 1 (lanes 64-127, columns 8-15).  The last pair MMA is older than the O^T MMAs, so O_DONE covers it.
    // Group g drains the accumulators n = g, g + 2, ...; warp gw holds channels 32 (gw & 1) .. + 31 of row 2n + hsel.
    for (int n = g; n < IB / 2; n += 2) {
      const int i = 2 * n + hsel;
      float v[8];
      tmem_ld_x8(tmem_lane + kColPair + n * 16 + hsel * 8, v);
      tmem_wait_ld();
      {
        const float4 a0 = *reinterpret_cast<const float4*>(inv_o + i * H), a1 = *reinterpret_cast<const float4*>(inv_o + i * H + 4);
        const float na[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
        __nv_bfloat16* st16 = reinterpret_cast<__nv_bfloat16*>(stage_e);
#pragma unroll
        for (int h = 0; h < H; ++h) st16[h * 32 + lane] = __float2bfloat16_rn(v[h] * na[h]);
      }
      __syncwarp();
      {   // [8 h][64 B] -> 32 chunks of 16 B, one per lane
        const int h = lane >> 2, part = lane & 3;
        *reinterpret_cast<uint4*>(cat + (orow0 + i) * NCAT + NS + h * C + (gw & 1) * 32 + part * 8) =
            reinterpret_cast<const uint4*>(stage_e)[lane];
      }
      __syncwarp();
    }
    tcgen05_fence_before_sync();
    mbar_arrive(&cb[EPI_TMEM]);     // every accumulator of this tile has been read: the next tile's MMAs may start
    DAB_STAMP(5);
    bar_all_compute();              // inv_o / the staging tiles are read until here; the next tile's softmax rewrites them
   }
  }
  tcgen05_fence_before_sync();
  __syncthreads();
#undef DAB_STAMP
#undef DAB_STAMP_ISSUER
#undef DAB_TIMED_WAIT
  if (warp == 0) tmem_free(tmem_cta, kTmemCols);
}

// Pair bias of up to six layers in ONE pass over the pair tensor, on the tensor cores:
//   plane_l[pair][h] = scale_total * log2(e) * sum_c e[pair, c] Wpb_l[h, c]      (fp16, [layer][B*L*L][8])
// Persistent CTAs stream [128 pairs x 64 c] tiles by TMA (ring of four); one tcgen05.mma chain per tile
// (M = 128 pairs, N = 16 * n_layers: the scaled weights as bf16 hi rows then bf16 lo rows, K = 64) into one of two
// TMEM accumulators; thread = pair adds hi + lo and stores 16 bytes per layer (coalesced).
struct BiasSmem {
  static constexpr int kStage = 128 * C * 2;         // 16,384
  static constexpr int kStages = 4;
  static constexpr int kW = kStages * kStage;        // up to [96 rows][128 B] bf16, 128B-swizzled
  static constexpr int kBars = kW + 96 * 128;
  static constexpr int kTmemSlot = kBars + 16 * 8;
  static constexpr int kTotal = kTmemSlot + 16;
};
__global__ void __launch_bounds__(192, 2)
ipa_pair_bias_mma_kernel(const __grid_constant__ CUtensorMap map_e, const float* __restrict__ wpb /* [nl][8][64] */,
                         int nl, uint4* __restrict__ planes, int64_t n_pairs, int n_tiles) {
  extern __shared__ __align__(1024) uint8_t smem[];
  using S = BiasSmem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kBars);   // full[4], empty[4], acc_full[2], acc_empty[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::kTmemSlot);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0) asm volatile("trap;");
  const int N = 16 * nl;
  if (tid == 0) {
    for (int i = 0; i < 8; ++i) mbar_init(&bars[i], 1);
    mbar_init(&bars[8], 1); mbar_init(&bars[9], 1);
    mbar_init(&bars[10], 128); mbar_init(&bars[11], 128);
    fence_barrier_init();
  }
  {  // weights: row r < 8 nl = hi of (layer r / 8, head r % 8), rows 8 nl .. 16 nl = lo
    const float sc = rsqrtf(3.0f) * kLog2e;
    for (int i = tid; i < 8 * nl * (C / 2); i += blockDim.x) {
      const int r = i / (C / 2), c2 = (i % (C / 2)) * 2;
      const float a = wpb[r * C + c2] * sc, bq = wpb[r * C + c2 + 1] * sc;
      const float ah = __bfloat162float(__float2bfloat16_rn(a)), bh = __bfloat162float(__float2bfloat16_rn(bq));
      *reinterpret_cast<uint32_t*>(smem + S::kW + swz128_offset(r, c2 >> 3) + (c2 & 7) * 2) = pack_bf162(ah, bh);
      *reinterpret_cast<uint32_t*>(smem + S::kW + swz128_offset(8 * nl + r, c2 >> 3) + (c2 & 7) * 2) =
          pack_bf162(a - ah, bq - bh);
    }
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (warp == 0) tmem_alloc(tmem_slot, 256);
  tcgen05_fence_before_sync();
  __syncthreads();
  tcgen05_fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  const int n_mine = (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  if (warp == 4) {
    if (lane == 0) {
      tma_prefetch_desc(&map_e);
      for (int k = 0; k < n_mine; ++k) {
        const int s = k % S::kStages;
        if (k >= S::kStages) mbar_wait(&bars[4 + s], ((k / S::kStages) - 1) & 1);
        mbar_arrive_expect_tx(&bars[s], S::kStage);
        tma_load_2d(smem + s * S::kStage, &map_e, &bars[s], 0, (int)(((int64_t)blockIdx.x + (int64_t)k * gridDim.x) * 128));
      }
    }
  } else if (warp == 5) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(128, N, 0, 0);
      for (int k = 0; k < n_mine; ++k) {
        const int s = k % S::kStages, acc = k & 1;
        mbar_wait(&bars[s], (k / S::kStages) & 1);
        if (k >= 2) mbar_wait(&bars[10 + acc], ((k >> 1) - 1) & 1);
        tcgen05_fence_after_sync();
#pragma unroll
        for (int kk = 0; kk < C / 16; ++kk) {
          uint64_t da = make_smem_desc(smem_base + s * S::kStage + kk * 32, 16, 1024, kSwizzle128B);
          uint64_t db = make_smem_desc(smem_base + S::kW + kk * 32, 16, 1024, kSwizzle128B);
          umma_bf16(tmem + acc * 128, da, db, idesc, kk != 0);
        }
        umma_commit(&bars[4 + s]);
        umma_commit(&bars[8 + acc]);
      }
    }
  } else {
    const uint32_t tmem_lane = tmem + ((uint32_t)(warp * 32) << 16);
    for (int k = 0; k < n_mine; ++k) {
      const int acc = k & 1;
      const int64_t pair = ((int64_t)blockIdx.x + (int64_t)k * gridDim.x) * 128 + tid;
      mbar_wait(&bars[8 + acc], (k >> 1) & 1);
      tcgen05_fence_after_sync();
      for (int l0 = 0; l0 < nl; l0 += 2) {   // two layers per pass: 16 hi + 16 lo columns
        float hi[16], lo[16];
        tmem_ld_x16(tmem_lane + acc * 128 + l0 * 8, hi);
        tmem_ld_x16(tmem_lane + acc * 128 + 8 * nl + l0 * 8, lo);
        tmem_wait_ld();
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          if (l0 + q < nl && pair < n_pairs)
            planes[(int64_t)(l0 + q) * n_pairs + pair] =
                make_uint4(pack_h2(hi[8 * q] + lo[8 * q], hi[8 * q + 1] + lo[8 * q + 1]),
                           pack_h2(hi[8 * q + 2] + lo[8 * q + 2], hi[8 * q + 3] + lo[8 * q + 3]),
                           pack_h2(hi[8 * q + 4] + lo[8 * q + 4], hi[8 * q + 5] + lo[8 * q + 5]),
                           pack_h2(hi[8 * q + 6] + lo[8 * q + 6], hi[8 * q + 7] + lo[8 * q + 7]));
        }
      }
      tcgen05_fence_before_sync();
      mbar_arrive(&bars[10 + acc]);
    }
  }
  tcgen05_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_free(tmem, 256);
}

// ---- patches of 256 residues: common centroid of the two blocks, merge of the two key blocks ----------------------------
// cen[2 b], cen[2 b + 1] = mean translation of patch b (256 residues)
__global__ void __launch_bounds__(256) centroid256_kernel(const float* __restrict__ t, float* __restrict__ cen) {
  __shared__ float part[8][3];
  const int b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* tp = t + ((int64_t)b * 2 * L + tid) * 3;
  float cx = tp[0], cy = tp[1], cz = tp[2];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    cx += __shfl_xor_sync(0xffffffffu, cx, o); cy += __shfl_xor_sync(0xffffffffu, cy, o); cz += __shfl_xor_sync(0xffffffffu, cz, o);
  }
  if (lane == 0) { part[warp][0] = cx; part[warp][1] = cy; part[warp][2] = cz; }
  __syncthreads();
  if (tid < 3) {
    float v = 0.f;
    for (int w = 0; w < 8; ++w) v += part[w][tid];
    v *= 1.0f / (2 * L);
    cen[(int64_t)b * 6 + tid] = v;
    cen[(int64_t)b * 6 + 3 + tid] = v;
  }
}

// One thread per (query row, head): the two key blocks' features are convex-combined with the weights
//   w_k = S_k 2^(m_k - m) / sum_k' S_k' 2^(m_k' - m),   m_k = row maximum (log2 units), S_k = sum_j p of block k
// - exact for the scalar, pair and (affine inverse-frame) point features; the point norms are recomputed from the merged points.
__global__ void __launch_bounds__(256) merge_kb2_kernel(const __nv_bfloat16* __restrict__ cat2, const float* __restrict__ stats2,
                                                        int64_t rows, __nv_bfloat16* __restrict__ cat) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * H) return;
  const int64_t row = idx >> 3;
  const int h = (int)(idx & 7);
  const float m0 = stats2[row * 16 + h], m1 = stats2[(rows + row) * 16 + h];
  const float s0 = 1.0f / stats2[row * 16 + 8 + h], s1 = 1.0f / stats2[(rows + row) * 16 + 8 + h];
  const float m = fmaxf(m0, m1);
  const float a0 = s0 * ex2(m0 - m), a1 = s1 * ex2(m1 - m);
  const float w0 = a0 / (a0 + a1), w1 = a1 / (a0 + a1);
  const __nv_bfloat16* c0 = cat2 + row * NCAT;
  const __nv_bfloat16* c1 = cat2 + (rows + row) * NCAT;
  __nv_bfloat16* out = cat + row * NCAT;
  auto mix8 = [&](int off, float* keep) {      // eight consecutive features
    const uint4 u0 = *reinterpret_cast<const uint4*>(c0 + off), u1 = *reinterpret_cast<const uint4*>(c1 + off);
    const __nv_bfloat162* p0 = reinterpret_cast<const __nv_bfloat162*>(&u0);
    const __nv_bfloat162* p1 = reinterpret_cast<const __nv_bfloat162*>(&u1);
    float v[8];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f0 = __bfloat1622float2(p0[e]), f1 = __bfloat1622float2(p1[e]);
      v[2 * e] = w0 * f0.x + w1 * f1.x; v[2 * e + 1] = w0 * f0.y + w1 * f1.y;
    }
    if (keep) {
#pragma unroll
      for (int e = 0; e < 8; ++e) keep[e] = v[e];
    }
    *reinterpret_cast<uint4*>(out + off) = make_uint4(pack_bf162(v[0], v[1]), pack_bf162(v[2], v[3]), pack_bf162(v[4], v[5]),
                                                      pack_bf162(v[6], v[7]));
  };
#pragma unroll
  for (int q = 0; q < DS / 8; ++q) mix8(h * DS + 8 * q, nullptr);                 // scalar values
#pragma unroll
  for (int q = 0; q < C / 8; ++q) mix8(NS + h * C + 8 * q, nullptr);             // pair aggregation
  float pt[24];
#pragma unroll
  for (int q = 0; q < 3; ++q) mix8(NS + H * C + h * 24 + 8 * q, pt + 8 * q);     // local-frame points
  float nrm[8];
#pragma unroll
  for (int p = 0; p < P; ++p) nrm[p] = sqrtf(pt[3 * p] * pt[3 * p] + pt[3 * p + 1] * pt[3 * p + 1] + pt[3 * p + 2] * pt[3 * p + 2]);
  *reinterpret_cast<uint4*>(out + NS + H * C + NPT + h * 8) =
      make_uint4(pack_bf162(nrm[0], nrm[1]), pack_bf162(nrm[2], nrm[3]), pack_bf162(nrm[4], nrm[5]), pack_bf162(nrm[6], nrm[7]));
}

static int launch_pair_bias(const void* e_bf16, const float* wpb, int nl, void* planes, int64_t n_pairs, cudaStream_t s) {
  CUtensorMap me;
  uint64_t de[2] = {(uint64_t)C, (uint64_t)n_pairs}, se[1] = {(uint64_t)C * 2};
  uint32_t be[2] = {C, 128};
  if (int rc = make_tensor_map_bf16(&me, e_bf16, 2, de, se, be, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  DAB_ENSURE_SMEM(ipa_pair_bias_mma_kernel, BiasSmem::kTotal);
  const int n_tiles = (int)((n_pairs + 127) / 128);
  const int grid = n_tiles < 296 ? n_tiles : 296;
  ipa_pair_bias_mma_kernel<<<grid, 192, BiasSmem::kTotal, s>>>(me, wpb, nl, reinterpret_cast<uint4*>(planes), n_pairs,
                                                               n_tiles);
  count_launch();
  return DAB_OK;
}

struct CoreArgs {
  CUtensorMap mq, mk, mv, me;
  const uint4* bias;
  const float *tc, *R;
  __nv_bfloat16* cat;
  float* stats;
  uint4* pu;
  int n_tiles;
  int64_t out_stride;
  const int *live, *live_count;
};
// (a function template: DAB_ENSURE_SMEM keeps one flag per instantiation, i.e. per kernel)
template <bool KB2, bool LIVE>
static int launch_core_kernel(const CoreArgs& a, int grid, cudaStream_t s) {
  DAB_ENSURE_SMEM((ipa_core_kernel<KB2, LIVE>), CoreSmem::kTotal);
  ipa_core_kernel<KB2, LIVE><<<grid, kCoreThreads, CoreSmem::kTotal, s>>>(a.mq, a.mk, a.mv, a.me, a.bias, a.tc, a.R, a.cat, a.stats,
                                                                          a.pu, a.n_tiles, g_core_dbg, a.out_stride, a.live,
                                                                          a.live_count);
  return DAB_OK;
}

}  // namespace sm100
}  // namespace dab

using namespace dab;
using namespace dab::sm100;

extern "C" {

size_t dab_ipa_packed_bytes(const DabIpaDims* d) { return shape_ok_fwd(d) ? packed_offsets().total : 0; }

int dab_ipa_pack_weights(const DabIpaDims* d, const DabIpaWeights* w, void* packed, void* stream) {
  DAB_REQUIRE(shape_ok_fwd(d), DAB_EUNSUPPORTED,
              "dab_ipa_pack_weights: the sm_100a fast path needs L=128 (or 256), D=128, C=64, H=8, ds=32, Pq=Pv=8");
  DAB_REQUIRE(w && packed && w->w_q_scalar && w->w_k_scalar && w->w_v_scalar && w->w_q_point && w->w_k_point &&
                  w->w_v_point && w->w_pair_bias && w->gamma && w->w_out && w->b_out,
              DAB_EINVAL, "dab_ipa_pack_weights: null pointer");
  DAB_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 1023) == 0, DAB_EINVAL, "dab_ipa_pack_weights: packed buffer must be 1024-byte aligned");
  pack_weights_kernel<<<kPackBlocks, 256, 0, (cudaStream_t)stream>>>(*w, reinterpret_cast<uint8_t*>(packed));
  count_launch();
  return check_launch("dab_ipa_pack_weights");
}

size_t dab_ipa_sm100_workspace_bytes(const DabIpaDims* d) {
  if (!shape_ok_fwd(d)) return 0;
  return d->L == 2 * L ? carve_ws2(d->B, nullptr).bytes : carve_ws(d->B, nullptr).bytes;
}

/* Byte offsets of the workspace sections: Qp, Kp, Vp, tc, cat, bias, stats, pu (tests read them: `stats` = row maxima in
 * log2 units [8 heads] | 1 / sum_j p [8 heads] per query row, `pu` = un-normalised probabilities 2^(l - max), bf16 [i][j][h],
 * both written by the training forward). */
int dab_ipa_sm100_workspace_layout(const DabIpaDims* d, size_t* offsets /* 8 */) {
  DAB_REQUIRE(shape_ok(d) && offsets, DAB_EINVAL, "dab_ipa_sm100_workspace_layout: bad argument");
  Ws w = carve_ws(d->B, nullptr);
  offsets[0] = reinterpret_cast<size_t>(w.Qp); offsets[1] = reinterpret_cast<size_t>(w.Kp);
  offsets[2] = reinterpret_cast<size_t>(w.Vp); offsets[3] = reinterpret_cast<size_t>(w.tc);
  offsets[4] = reinterpret_cast<size_t>(w.cat); offsets[5] = reinterpret_cast<size_t>(w.bias);
  offsets[6] = reinterpret_cast<size_t>(w.stats);
  offsets[7] = reinterpret_cast<size_t>(w.pu);
  return DAB_OK;
}

/* Pair-bias planes of n_layers <= 6 layers in one pass over the pair tensor: w_pair_bias[n_layers][8][64] fp32
 * (contiguous), planes_f16[n_layers][B*L*L][8] fp16 (contiguous). */
int dab_ipa_pair_bias_multi(const DabIpaDims* d, const void* e_bf16, const float* w_pair_bias, int n_layers,
                            void* planes_f16, void* stream) {
  DAB_REQUIRE(shape_ok_fwd(d), DAB_EUNSUPPORTED,
              "dab_ipa_pair_bias_multi: the sm_100a fast path needs L=128 (or 256), D=128, C=64, H=8, ds=32, Pq=Pv=8");
  DAB_REQUIRE(n_layers >= 1 && n_layers <= 6, DAB_EUNSUPPORTED, "dab_ipa_pair_bias_multi: 1 <= n_layers <= 6");
  if (d->B == 0) return DAB_OK;
  DAB_REQUIRE(e_bf16 && w_pair_bias && planes_f16 && (reinterpret_cast<uintptr_t>(e_bf16) & 127) == 0 &&
                  aligned16(planes_f16),
              DAB_EINVAL, "dab_ipa_pair_bias_multi: null or misaligned pointer");
  const int64_t n_pairs = (int64_t)d->B * d->L * d->L;
  if (int rc = launch_pair_bias(e_bf16, w_pair_bias, n_layers, planes_f16, n_pairs, (cudaStream_t)stream)) return rc;
  return check_launch("dab_ipa_pair_bias_multi");
}

// Projection launch of a layer (weights `pk`), packed operands into `ws`.  With `pk_prev` the kernel first computes the
// PREVIOUS layer's to_out, y = cat Wout^T + b (cat = ws.cat, weights pk_prev), straight into its A tile: x is not read.
// With `w2` (patches of 256 residues, B = 2 x patches) the patch centroids are computed first and the projections are
// centred on them.
// the epsilon network's front MLP as the input of layer 0 (mode 2 of the projection kernel): y = relu(c[row] + t1[seq[row]]) W2^T + b2
struct FrontIn { const float* c; const float* t1; const int64_t* seq; const void* w2_bf16; const float* b2; };
static int launch_proj(int B, const uint8_t* pk, const float* x, const __nv_bfloat16* x16, const float* R, const float* t,
                       const Ws& ws, const Ws2* w2, const uint8_t* pk_prev, cudaStream_t s, const FrontIn* front = nullptr) {
  if (w2) { centroid256_kernel<<<B / 2, 256, 0, s>>>(t, w2->cen); count_launch(); }
  const PackedOffsets po = packed_offsets();
  const int M = B * L;
  CUtensorMap mw64, mw48;
  uint64_t dw[2] = {(uint64_t)D, (uint64_t)NPROJ}, sw[1] = {(uint64_t)D * 2};
  uint32_t b64[2] = {64, 64}, b48[2] = {64, 48};
  if (int rc = make_tensor_map_bf16(&mw64, pk + po.wcat, 2, dw, sw, b64, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  if (int rc = make_tensor_map_bf16(&mw48, pk + po.wcat, 2, dw, sw, b48, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  DAB_ENSURE_SMEM(ipa_proj_kernel, ProjSmem::kTotal);
  CUtensorMap msq, msk, msv;   // TMA-store views of the packed operands: 64-byte segments of 32 rows
  {
    uint64_t dqk[2] = {(uint64_t)H * QK_W, (uint64_t)M}, sqk[1] = {(uint64_t)H * QK_W * 2};
    uint64_t dv[2] = {(uint64_t)H * V_W, (uint64_t)M}, sv[1] = {(uint64_t)H * V_W * 2};
    uint32_t bs[2] = {32, 32};     // one warp's rows
    if (int rc = make_tensor_map_bf16(&msq, ws.Qp, 2, dqk, sqk, bs, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
    if (int rc = make_tensor_map_bf16(&msk, ws.Kp, 2, dqk, sqk, bs, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
    if (int rc = make_tensor_map_bf16(&msv, ws.Vp, 2, dv, sv, bs, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
  }
  CUtensorMap mcat = mw64, mwout = mw64;     // (placeholders when the to_out phase is off)
  const float* b_out = nullptr;
  int n_split = B >= 128 ? 1 : (B >= 64 ? 2 : 4);   // small batches: several CTAs per patch
  if (pk_prev) {
    uint64_t dc[2] = {(uint64_t)NCAT, (uint64_t)M}, dwo[2] = {(uint64_t)NCAT, (uint64_t)D}, sc[1] = {(uint64_t)NCAT * 2};
    uint32_t bc[2] = {64, 128};
    if (int rc = make_tensor_map_bf16(&mcat, ws.cat, 2, dc, sc, bc, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    if (int rc = make_tensor_map_bf16(&mwout, pk_prev + po.wout, 2, dwo, sc, bc, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    b_out = reinterpret_cast<const float*>(pk_prev + po.bout);
    n_split = 1;                             // the to_out phase produces the whole A tile of the patch
  } else if (front) {
    uint64_t dw2[2] = {(uint64_t)D, (uint64_t)D}, sw2[1] = {(uint64_t)D * 2};
    uint32_t bw2[2] = {64, 128};
    if (int rc = make_tensor_map_bf16(&mwout, front->w2_bf16, 2, dw2, sw2, bw2, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    b_out = front->b2;
    n_split = 1;
  }
  ipa_proj_kernel<<<dim3(n_split, B), 288, ProjSmem::kTotal, s>>>(
      mw64, mw48, msq, msk, msv, x, R, t, reinterpret_cast<const float*>(pk + po.gamma), ws.Qp, ws.Kp, ws.Vp, ws.tc,
      g_core_dbg ? g_core_dbg + (1 << 20) : nullptr, x16, mcat, mwout, b_out, pk_prev ? 1 : (front ? 2 : 0),
      w2 ? w2->cen : nullptr,
      front ? reinterpret_cast<const float4*>(front->c) : nullptr, front ? reinterpret_cast<const float4*>(front->t1) : nullptr,
      front ? front->seq : nullptr);
  count_launch();
  return DAB_OK;
}

// Workspace views of a forward call.  A patch of 256 residues = two blocks of 128: everything row-wise (projections,
// to_out) runs on nblk = 2 B blocks, the attention core once per (query block, key block) pair, and the two key blocks'
// results are merged by their softmax statistics (w2).
struct FwdWs {
  bool two;
  int nblk;   // 0: empty batch, nothing to launch
  Ws ws;
  Ws2 w2;
};

// Prologue shared by the forward entry points (`fn`: the one the caller called, for the messages): the shape, the
// pointers (`args_ok` / `args_aligned`: the caller's own operands), the workspace size, and the workspace views.
static int fwd_prologue(const char* fn, const DabIpaDims* d, bool train, bool args_ok, bool args_aligned, const void* packed,
                        void* workspace, size_t workspace_bytes, FwdWs& f) {
  DAB_REQUIRE(train ? shape_ok(d) : shape_ok_fwd(d), DAB_EUNSUPPORTED,
              "%s: the sm_100a fast path needs the train.py configuration (D=128, C=64, H=8, ds=32, Pq=Pv=8) and L=128 "
              "(inference: 128 or 256)", fn);
  f = {};
  f.two = d->L == 2 * L;
  if (d->B == 0) return DAB_OK;
  DAB_REQUIRE(args_ok && packed && workspace, DAB_EINVAL, "%s: null pointer", fn);
  DAB_REQUIRE(args_aligned && (reinterpret_cast<uintptr_t>(workspace) & 1023) == 0 &&
                  (reinterpret_cast<uintptr_t>(packed) & 1023) == 0,
              DAB_EINVAL, "%s: misaligned pointer (workspace / packed weights 1024 B, e 128 B, other arrays 16 B)", fn);
  f.nblk = f.two ? 2 * d->B : d->B;
  f.ws = carve_ws(f.nblk, workspace);
  size_t need = f.ws.bytes;
  if (f.two) { f.w2 = carve_ws2(d->B, workspace); need = f.w2.bytes; }
  DAB_REQUIRE(workspace_bytes >= need, DAB_EWORKSPACE, "%s: workspace %zu < %zu", fn, workspace_bytes, need);
  return DAB_OK;
}

// Attention-core launch of a layer (stage 2) on the packed operands in the workspace; `live` / `live_count` (device
// memory, optional): only these query tiles (see ipa_core_kernel).
static int launch_core(const FwdWs& f, int Lp, const uint8_t* pk, const void* e_bf16, const void* bias_f16, const float* R,
                       bool save_for_bwd, const int* live, const int* live_count, cudaStream_t s) {
  const bool two = f.two;
  const int B = f.nblk, M = B * L;
  const Ws& ws = f.ws;
  const Ws2& w2 = f.w2;
  const PackedOffsets po = packed_offsets();
  const uint4* bias = reinterpret_cast<const uint4*>(bias_f16);
  if (bias == nullptr) {   // one-off call without a precomputed bias: build this layer's plane now
    uint4* plane = two ? w2.bias2 : ws.bias;
    if (int rc = launch_pair_bias(e_bf16, reinterpret_cast<const float*>(pk + po.wpb), 1, plane, (int64_t)M * Lp, s)) return rc;
    bias = plane;
  }
  CUtensorMap mq, mk, mv, me;
  uint64_t dqk[2] = {(uint64_t)H * QK_W, (uint64_t)M}, sqk[1] = {(uint64_t)H * QK_W * 2};
  uint32_t bq[2] = {32, IB}, bk[2] = {32, L};
  if (int rc = make_tensor_map_bf16(&mq, ws.Qp, 2, dqk, sqk, bq, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
  if (int rc = make_tensor_map_bf16(&mk, ws.Kp, 2, dqk, sqk, bk, CU_TENSOR_MAP_SWIZZLE_64B)) return rc;
  uint64_t dv[2] = {(uint64_t)H * V_W, (uint64_t)M}, sv[1] = {(uint64_t)H * V_W * 2};
  uint32_t bv[2] = {V_W, L};
  if (int rc = make_tensor_map_bf16(&mv, ws.Vp, 2, dv, sv, bv, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  uint64_t de[2] = {(uint64_t)C, (uint64_t)M * Lp}, se[1] = {(uint64_t)C * 2};
  uint32_t be[2] = {C, L};
  if (int rc = make_tensor_map_bf16(&me, e_bf16, 2, de, se, be, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  const int n_tiles = (two ? 2 * B : B) * (L / IB);      // 256: one tile set per (query block, key block) pair
  int n_sm = 148;
  {
    int dev_id = 0;
    cudaGetDevice(&dev_id);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev_id);
  }
  const int grid = n_tiles < n_sm ? n_tiles : n_sm;     // persistent: one CTA per SM, two tile contexts each
  const CoreArgs a = {mq, mk, mv, me, bias, ws.tc, R, two ? w2.cat2 : ws.cat, two ? w2.stats2 : (save_for_bwd ? ws.stats : nullptr),
                      two || !save_for_bwd ? nullptr : ws.pu, n_tiles, two ? (int64_t)M : 0, live, live_count};
  if (int rc = two ? (live ? launch_core_kernel<true, true>(a, grid, s) : launch_core_kernel<true, false>(a, grid, s))
                   : (live ? launch_core_kernel<false, true>(a, grid, s) : launch_core_kernel<false, false>(a, grid, s)))
    return rc;
  count_launch();
  if (two) {   // (all rows: those of tiles left out are merged from stale inputs and never read)
    merge_kb2_kernel<<<(unsigned)(((int64_t)M * H + 255) / 256), 256, 0, s>>>(w2.cat2, w2.stats2, (int64_t)M, ws.cat);
    count_launch();
  }
  return DAB_OK;
}

// x / y: fp32, or (x_bf16 / y_bf16 non-null) bf16 - the residue stream handed from layer to layer already rounded
static int fwd_sm100_impl(const char* fn, const DabIpaDims* d, const void* packed, const float* x, const void* e_bf16,
                          const void* bias_f16, const float* R, const float* t, float* y, void* workspace,
                          size_t workspace_bytes, bool save_for_bwd, void* stream, const void* x_bf16, void* y_bf16,
                          int phases) {
  FwdWs f;
  if (int rc = fwd_prologue(fn, d, save_for_bwd, (x || x_bf16) && e_bf16 && R && t && (y || y_bf16),
                            (reinterpret_cast<uintptr_t>(e_bf16) & 127) == 0 && aligned16(x) && aligned16(y) &&
                                aligned16(x_bf16) && aligned16(y_bf16),
                            packed, workspace, workspace_bytes, f))
    return rc;
  if (f.nblk == 0) return DAB_OK;
  const bool two = f.two;
  const int Lp = d->L, B = f.nblk, M = B * L;
  const Ws& ws = f.ws;
  const Ws2& w2 = f.w2;
  const PackedOffsets po = packed_offsets();
  const uint8_t* pk = reinterpret_cast<const uint8_t*>(packed);
  cudaStream_t s = (cudaStream_t)stream;
  if (phases & 1) {
    if (int rc = launch_proj(B, pk, x, reinterpret_cast<const __nv_bfloat16*>(x_bf16), R, t, ws, two ? &w2 : nullptr,
                             nullptr, s))
      return rc;
  }
  if (phases & 2) {
    if (int rc = launch_core(f, Lp, pk, e_bf16, bias_f16, R, save_for_bwd, nullptr, nullptr, s)) return rc;
  }
  if (phases & 4) {
    // y = cat Wout^T + b: one 128-wide N tile per CTA when the batch fills the GPU, four 32-wide ones otherwise
    const float* bo = reinterpret_cast<const float*>(pk + po.bout);
    if (int rc = (M / kGemmBM >= 148) ? launch_gemm_bf16<128>(ws.cat, NCAT, pk + po.wout, NCAT, y, D, bo, M, D, NCAT, s, y_bf16)
                                      : launch_gemm_bf16<32>(ws.cat, NCAT, pk + po.wout, NCAT, y, D, bo, M, D, NCAT, s, y_bf16))
      return rc;
  }
  return check_launch(fn);
}

/* Byte offsets inside the packed weights: offs[0..6] = Wcat bf16 [1344][128] (rows: to_q_scalar, to_k_scalar, to_v_scalar,
 * to_q_point, to_k_point, to_v_point), Wout bf16 [128][1024], to_pair_bias fp32 [8][64], b_out fp32 [128], gamma fp32 [8],
 * Wcat^T bf16 [128][1344], Wout^T bf16 [1024][128] - so that a caller's own GEMMs can reuse the bf16 copies. */
int dab_ipa_packed_layout(const DabIpaDims* d, size_t* offs) {
  DAB_REQUIRE(d && offs, DAB_EINVAL, "dab_ipa_packed_layout: null pointer");
  DAB_REQUIRE(shape_ok_fwd(d), DAB_EUNSUPPORTED, "dab_ipa_packed_layout: the sm_100a fast path needs the train.py configuration");
  const PackedOffsets po = packed_offsets();
  offs[0] = po.wcat; offs[1] = po.wout; offs[2] = po.wpb; offs[3] = po.bout; offs[4] = po.gamma; offs[5] = po.wcat_t;
  offs[6] = po.wout_t;
  return DAB_OK;
}

/* Training forward: same launches; the workspace additionally keeps what dab_ipa_bwd_sm100_main needs (packed operands,
 * concat features, un-normalised probabilities and the softmax statistics) and must be handed to it untouched. */
int dab_ipa_fwd_sm100_train(const DabIpaDims* d, const void* packed, const float* x, const void* e_bf16,
                            const void* bias_f16, const float* R, const float* t, float* y, void* saved,
                            size_t saved_bytes, void* stream) {
  return fwd_sm100_impl("dab_ipa_fwd_sm100_train", d, packed, x, e_bf16, bias_f16, R, t, y, saved, saved_bytes, true, stream,
                        nullptr, nullptr, 7);
}

/* The inference forward, whole (stages = 7) or launch by launch: `stages` = bit0 projections + frame transform, bit1
 * attention core, bit2 to_out.  The workspace must hold the products of the earlier stages (a previous call with the lower
 * bits).  Lets a caller bracket one stage with its own events (bench.py's roofline of the attention core) or interleave its
 * own work between the stages.  The residue stream is fp32 or bf16 on either side: exactly one of x / x_bf16 and one of
 * y / y_bf16 is given.  Between the layers of a stack the stream is consumed as bf16 anyway (the projections' A operand),
 * so handing it over already rounded changes no bit of the result and halves its HBM traffic. */
int dab_ipa_fwd_sm100_stages(const DabIpaDims* d, const void* packed, const float* x, const void* x_bf16, const void* e_bf16,
                             const void* bias_f16, const float* R, const float* t, float* y, void* y_bf16, void* workspace,
                             size_t workspace_bytes, int stages, void* stream) {
  DAB_REQUIRE((x == nullptr) != (x_bf16 == nullptr) && (y == nullptr) != (y_bf16 == nullptr), DAB_EINVAL,
              "dab_ipa_fwd_sm100_stages: give exactly one of x / x_bf16 and one of y / y_bf16");
  DAB_REQUIRE(stages > 0 && stages <= 7, DAB_EINVAL, "dab_ipa_fwd_sm100_stages: stages must be a non-empty subset of bits 0..2");
  return fwd_sm100_impl("dab_ipa_fwd_sm100_stages", d, packed, x, e_bf16, bias_f16, R, t, y, workspace, workspace_bytes, false,
                        stream, x_bf16, y_bf16, stages);
}

/* The attention core (stages(.., 2)) on a list of query tiles only: live_tiles = ascending ids of 16-row tiles (global
 * row / 16 of the B*L rows), live_count[0] = their number; both in device memory, read by the kernel (no host sync, so the
 * list may change between replays of a captured graph).  The concat features of the other rows are left as they were. */
int dab_ipa_core_sm100_live(const DabIpaDims* d, const void* packed, const void* e_bf16, const void* bias_f16, const float* R,
                            const float* t, void* workspace, size_t workspace_bytes, const int* live_tiles,
                            const int* live_count, void* stream) {
  FwdWs f;
  if (int rc = fwd_prologue("dab_ipa_core_sm100_live", d, false, e_bf16 && R && t && live_tiles && live_count,
                            (reinterpret_cast<uintptr_t>(e_bf16) & 127) == 0, packed, workspace, workspace_bytes, f))
    return rc;
  if (f.nblk == 0) return DAB_OK;
  if (int rc = launch_core(f, d->L, reinterpret_cast<const uint8_t*>(packed), e_bf16, bias_f16, R, false, live_tiles,
                           live_count, (cudaStream_t)stream))
    return rc;
  return check_launch("dab_ipa_core_sm100_live");
}

/* Between two layers of a stack (inference): the previous layer's to_out (y = cat Wout^T + b, `packed_prev`; `cat` = the
 * concat features its attention core left in `workspace`) fused with this layer's projections (`packed`): y is rounded to
 * bf16 exactly as dab_ipa_fwd_sm100_stages would hand it over (y_bf16), but goes straight into the projection kernel's
 * operand tile and never exists in HBM; the packed Q / K / V of this layer replace those of the previous one in `workspace`.
 * Sequence for a stack: stages(1) of layer 0, then per layer stages(2) followed by dab_ipa_mid_sm100 (or stages(4) after
 * the last layer).  Bit-identical to the unfused sequence. */
int dab_ipa_mid_sm100(const DabIpaDims* d, const void* packed_prev, const void* packed, const float* R, const float* t,
                      void* workspace, size_t workspace_bytes, void* stream) {
  FwdWs f;
  if (int rc = fwd_prologue("dab_ipa_mid_sm100", d, false, packed_prev && R && t,
                            (reinterpret_cast<uintptr_t>(packed_prev) & 1023) == 0, packed, workspace, workspace_bytes, f))
    return rc;
  if (f.nblk == 0) return DAB_OK;
  if (int rc = launch_proj(f.nblk, reinterpret_cast<const uint8_t*>(packed), nullptr, nullptr, R, t, f.ws,
                           f.two ? &f.w2 : nullptr, reinterpret_cast<const uint8_t*>(packed_prev), (cudaStream_t)stream))
    return rc;
  return check_launch("dab_ipa_mid_sm100");
}

/* The projections of the FIRST layer of the epsilon network's stack with the front MLP (Denoiser.to_res_emb during sampling,
 * diffab_pytorch.py:572-574) fused in: the layer input y = relu(c[row] + t1[seq[row]]) W2^T + b2 (first layer regrouped into
 * the per-run constant c[B*L,128] and the 25-row table t1[25,128], as dab_front_fwd_sm100 computes it; w2_bf16 [128][128],
 * b2 [128]) is formed in the projection kernel's operand tile and never exists in HBM.  Replaces dab_front_fwd_sm100 +
 * stages(1); the same bits. */
int dab_ipa_front_proj_sm100(const DabIpaDims* d, const void* packed, const float* c, const float* t1, const int64_t* seq,
                             const void* w2_bf16, const float* b2, const float* R, const float* t, void* workspace,
                             size_t workspace_bytes, void* stream) {
  FwdWs f;
  if (int rc = fwd_prologue("dab_ipa_front_proj_sm100", d, false, c && t1 && seq && w2_bf16 && b2 && R && t,
                            aligned16(c) && aligned16(t1) && aligned16(w2_bf16), packed, workspace, workspace_bytes, f))
    return rc;
  if (f.nblk == 0) return DAB_OK;
  const FrontIn fr = {c, t1, seq, w2_bf16, b2};
  if (int rc = launch_proj(f.nblk, reinterpret_cast<const uint8_t*>(packed), nullptr, nullptr, R, t, f.ws,
                           f.two ? &f.w2 : nullptr, nullptr, (cudaStream_t)stream, &fr))
    return rc;
  return check_launch("dab_ipa_front_proj_sm100");
}

/* nn.Linear (+ ReLU) on the tcgen05 GEMM: C = act(A[M,K] W[N,K]^T + bias), bf16 operands, fp32 accumulation; the result as
 * fp32 (C_f32) or rounded to bf16 (C_bf16) - exactly one of the two.  M % 128 == 0, N % 64 == 0, K % 64 == 0.
 * Forward of the MLPs of diffab_pytorch.py:57-183,572-599 in mixed-precision training, and (W transposed) their data
 * gradients and those of the IPA layer's nn.Linear layers (dcat = dy Wout, dx = dproj Wcat). */
int dab_linear_bf16(const void* A, const void* W, const float* bias, int relu, int M, int N, int K, float* C_f32, void* C_bf16,
                    void* stream) {
  DAB_REQUIRE(A && W && ((C_f32 == nullptr) != (C_bf16 == nullptr)), DAB_EINVAL,
              "dab_linear_bf16: null pointer (exactly one of C_f32 / C_bf16 must be given)");
  cudaStream_t s = (cudaStream_t)stream;
  // narrow N tiles and a deep ring when 64-wide tiles would leave most SMs idle (e.g. dx = dproj Wcat: N = 128, K = 1344);
  // wide tiles when there are more than two waves of them (e.g. dcat = dy Wout: N = 1024, K = 128)
  if (M > 0 && N % 64 == 0 && (M / kGemmBM) * (N / 64) < 148)
    return launch_gemm_bf16<32>(A, K, W, K, C_f32, N, bias, M, N, K, s, C_bf16, relu);
  if (N % 128 == 0 && (M / kGemmBM) * (N / 128) >= 2 * 148)
    return launch_gemm_bf16<128>(A, K, W, K, C_f32, N, bias, M, N, K, s, C_bf16, relu);
  return launch_gemm_bf16<64>(A, K, W, K, C_f32, N, bias, M, N, K, s, C_bf16, relu);
}

#ifdef DAB_DEBUG_HOOKS
/* Profiling hook (debug build only): per-tile clock64 timeline of the attention core (64 slots per tile), NULL to disable. */
int dab_debug_set_timeline(long long* buf) {
  g_core_dbg = buf;
  return DAB_OK;
}
#endif

}  // extern "C"
