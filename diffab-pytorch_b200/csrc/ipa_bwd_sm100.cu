// sm_100a backward of one InvariantPointAttentionLayer (train.py configuration), i.e. the autograd backward of
// diffab_pytorch.py:389-465 of the reference, from the upstream gradient of the concat features (dcat = dy Wout)
// down to the gradient of the six projections (dproj), of the pair tensor (de), of to_pair_bias and of gamma.
// The four plain GEMMs around it (dcat = dy Wout, dWout = dy^T cat, dx = dproj Wcat, dWcat = dproj^T x) are
// library GEMMs issued by the caller.
//
// With P = softmax_j(l), l_ij,h = a qs_i.ks_j + st b_ij,h - c_h/2 |q~_i - k~_j|^2 (q~, k~: global-frame points):
//   dP_ij,h = dos_i,h . vs_j,h + dog_i,h . v~_j,h + dopair_i,h . e_ij          (gradient of the three aggregations)
//   dl_ij,h = P_ij,h (dP_ij,h - Delta_i,h),   Delta_i,h = sum_j P dP = <dO_i,h, O_i,h>  (from the saved outputs)
//   de_ij   = sum_h P_ij,h dopair_i,h + dl_ij,h st Wpb_h                         dWpb_h = st sum_ij dl_ij,h e_ij
//   dq_i,h  = sum_j dl_ij,h [a ks_j | c_h k~_j]  - c_h q~_i sum_j dl_ij,h        (query side: this kernel)
//   dk_j,h  = sum_i dl_ij,h [a qs_i | c_h q~_i]  - c_h k~_j sum_i dl_ij,h        (key side: second kernel)
//   dv_j,h  = sum_i P_ij,h [dos_i,h | dog_i,h]
//   dgamma_h = (1/gamma_h) sum_ij dl_ij,h lp_ij,h,  lp = l - ls - lb, each sum obtained from quantities at hand:
//              sum dl l from the logits in registers, sum dl ls = <qs, dqs>, sum dl lb = <st Wpb, sum dl e>.
//
// Launch sequence (dab_ipa_bwd_sm100_main: 1 and 2, dab_ipa_bwd_sm100_finish: 3):
//   1. ipa_bwd_core_kernel  : per CTA = (patch, 16 query rows), thread = key j = TMEM lane (as the forward core):
//        prologue: dcat, cat rows of the tile -> dO (fp16 with a per-row power-of-two scale, in shared memory; bf16 copy to
//                  HBM for the key side), dopair (bf16, shared memory), Delta   (a separate launch until round 2)
//        dPv^T_h = V_h dO_h^T              (value part of dP)             M=128 j, N=16 i, K=64        fp16
//        per query row i, on the TMA-staged pair row e[i] (read from HBM once; P comes from the forward's saved Pu):
//          dPp_i = e[i] dopair_i^T         (pair part of dP)              M=128 j, N=16(8 h), K=64 c
//          de_i  = [P_i | dl_i] [dopair_i ; st Wpb]                       M=128 j, N=64 c, K=16        -> HBM (bf16)
//          Z    += e[i]^T dl_i             (to_pair_bias gradient)        M=64 c,  N=8 h,  K=128 j
//      P and dl also go to HBM as bf16 [b][h][i][j] for the key side.
//   2. ipa_bwd_keyside_kernel: per (patch, head): dV_h = P_h^T dO_h, dK_h = dl_h^T Q_h[:, :64], dQ_h = dl_h K_h[:, :64]
//      and, in its epilogue: scales, the -c q~ sum dl corrections, global -> local frame -> dproj rows (bf16)
//   3. bwd_reduce_kernel / bwd_finalize_kernel: reduce the per-CTA partials into dWpb and dgamma
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math.h>

#include "common.cuh"
#include "ipa_sm100_layout.cuh"
#include "sm100_prims.cuh"

namespace dab {
namespace sm100 {

constexpr float kLn2 = 0.6931471805599453f;
#ifdef DAB_DEBUG_HOOKS
static long long* g_bwd_dbg = nullptr;   // optional per-CTA clock64 timeline (dab_debug_set_bwd_timeline; debug build only)
static int g_bwd_keep_qkv = 0;           // debug hook: also write the raw dQ / dK / dV accumulators
#else
static constexpr long long* g_bwd_dbg = nullptr;
static constexpr int g_bwd_keep_qkv = 0;
#endif

// ---- backward workspace ---------------------------------------------------------------------------------
struct BwdWs {
  __nv_bfloat16* dObf;      // [rows][8][64] bf16: [dos 32 | dog 24 | 0 x 8], unscaled (key side; the query side keeps its
                            // scaled fp16 copy, dopair, Delta and the row scales in shared memory)
  __nv_bfloat16 *Pn, *dL;   // [B][8][128 i][128 j] bf16
  float *dQ, *dK, *dV;      // [rows][8][64] fp32: raw key-side accumulators, written only for tests (contiguous)
  float *p_wpb, *p_g1, *p_g2;   // partials: [B*8][512], [B*8][8], [B][8]
  float* r_part;                // [32][528] second-level partials
  size_t bytes;
};
inline BwdWs carve_bwd(int B, void* base) {
  auto al = [](size_t n) { return (n + 1023) / 1024 * 1024; };
  const size_t rows = (size_t)B * L;
  uint8_t* p = reinterpret_cast<uint8_t*>(base);
  BwdWs w;
  w.dObf = reinterpret_cast<__nv_bfloat16*>(p); p += al(rows * H * 64 * 2);
  w.Pn = reinterpret_cast<__nv_bfloat16*>(p); p += al((size_t)B * H * L * L * 2);
  w.dL = reinterpret_cast<__nv_bfloat16*>(p); p += al((size_t)B * H * L * L * 2);
  w.dQ = reinterpret_cast<float*>(p); p += al(rows * H * 64 * 4);
  w.dK = reinterpret_cast<float*>(p); p += al(rows * H * 64 * 4);
  w.dV = reinterpret_cast<float*>(p); p += al(rows * H * 64 * 4);
  w.p_wpb = reinterpret_cast<float*>(p); p += al((size_t)B * 8 * 512 * 4);
  w.p_g1 = reinterpret_cast<float*>(p); p += al((size_t)B * 8 * 8 * 4);
  w.p_g2 = reinterpret_cast<float*>(p); p += al((size_t)B * 8 * 4);
  w.r_part = reinterpret_cast<float*>(p); p += al(32 * 528 * 4);
  w.bytes = (size_t)(p - reinterpret_cast<uint8_t*>(base));
  return w;
}

// ---- 1 + 2. query-side core (with the preparation of its own rows) -------------------------------------------------
// Prologue (what a separate "prep" launch did before: 22 us at B = 32 on the critical path): everything the tile needs
// from dcat is a function of ITS OWN 16 query rows, so the eight compute warps (warp = head) turn the rows' dcat / cat
// (cat row layout, diffab_pytorch.py:456-462: [scalar (h d) 256 | pair (h c) 512 | local points (h p c) 192 | norms (h p) 64])
// into dO (fp16 with a per-row power-of-two scale, straight into the swizzled MMA operand tile; unscaled bf16 copy to HBM
// for the key side), dopair (bf16, the sixteen operand tiles stay resident) and Delta = <dO, O> - while the V tiles and
// the first pair rows are already on their way.
// The forward saved the un-normalised probabilities Pu[b][i][j][8 h] (bf16) and 1 / sum_j p, so the logits are not
// recomputed: no Q / K operands here (dQ moved to the key-side kernel, where dl_h is a resident tile anyway).
struct BwdSmem {
  // region X: stage 1 = ring of four V heads; stage 2 = ring of four pair rows
  static constexpr int kVBuf = L * V_W * 2;          // 16,384
  static constexpr int kVBufs = 4;
  static constexpr int kEStage = L * C * 2;          // 16,384
  static constexpr int kEStages = 4;
  static constexpr int kXBytes = kEStages * kEStage;   // 65,536
  // region P: stage 1 = dO rows of this CTA ([h][16 i][128 B] fp16); stage 2 = four [P | dl] operand buffers
  static constexpr int kDoOff = kXBytes;             // 16,384
  static constexpr int kPcat = kXBytes;              // 4 x { [128 j][16 B] P | [128 j][16 B] dl } bf16
  static constexpr int kDop = kPcat + 16384;         // the CTA's sixteen [8 h][128 B] bf16 dopair rows ...
  static constexpr int kWpb = kDop + IB * 1024;      // ... directly followed by [8 h][128 B] bf16: st * Wpb
  static constexpr int kInv = kWpb + 1024;           // [16 i][8] f32: 1 / sum_j p
  static constexpr int kDelta = kInv + 512;          // [16 i][8] f32
  static constexpr int kRs = kDelta + 512;           // [16] f32
  static constexpr int kRed = kRs + 64;              // [8 warps][8] f32
  static constexpr int kMax = kRed + 256;            // [16 i][8 h] f32: largest |dO| entry per (row, head)  (prologue)
  static constexpr int kFrame = kMax + 512;          // [16 i][12] f32: R (9) | centred t (3) of the CTA's rows
  static constexpr int kScr = kFrame + 768;          // [8 h][16 i] f32: pair part of Delta (prologue)
  static constexpr int kBars = kScr + 512;           // 48 mbarriers
  static constexpr int kTmemSlot = kBars + 384;
  static constexpr int kTotal = kTmemSlot + 16;
};
static_assert(BwdSmem::kVBufs * BwdSmem::kVBuf <= BwdSmem::kXBytes, "V ring must fit region X");
static_assert(BwdSmem::kTotal <= 113 * 1024, "two CTAs per SM");

enum BBar { BV_FULL = 0, BV_EMPTY = 4, BQ_FULL = 8, BS_DONE = 9, BE_FULL = 10, BE_EMPTY = 14,
            DPP_DONE = 18 /* 3 */, DPP_FREE = 21 /* 3, 128 arrivals */, PCAT_READY = 24 /* [g][slot], 128 arrivals */,
            PCAT_FREE = 28, DE_DONE = 32 /* [g] */, DE_FREE = 34 /* 128 arrivals */, B_N_BARS = 35 };

// TMEM columns (256 per CTA): value part of dP for the 16 rows, ring of three pair parts, de, to_pair_bias gradient
constexpr uint32_t kBColDPV = 0, kBColDPP = 128 /* 3 x 16 */, kBColDE = 176 /* 64 */, kBColWPB = 240 /* 16 */;

__device__ __forceinline__ uint4 pack8_bf16(const float (&v)[8]) {
  return make_uint4(pack_bf162(v[0], v[1]), pack_bf162(v[2], v[3]), pack_bf162(v[4], v[5]), pack_bf162(v[6], v[7]));
}
__device__ __forceinline__ float lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__global__ void __launch_bounds__(320, 2)
ipa_bwd_core_kernel(const __grid_constant__ CUtensorMap map_v, const __grid_constant__ CUtensorMap map_e,
                    const float* __restrict__ dcat, const __nv_bfloat16* __restrict__ cat, const float* __restrict__ R,
                    const float* __restrict__ tc, __nv_bfloat16* __restrict__ dObf,
                    const uint4* __restrict__ Pu, const float* __restrict__ stats,
                    const float* __restrict__ wpb, __nv_bfloat16* __restrict__ de,
                    __nv_bfloat16* __restrict__ Pn, __nv_bfloat16* __restrict__ dL, float* __restrict__ p_wpb,
                    float* __restrict__ p_g1, long long* __restrict__ dbg) {
  extern __shared__ __align__(1024) uint8_t smem[];
  long long* dbg_cta = dbg ? dbg + (size_t)(blockIdx.y * gridDim.x + blockIdx.x) * 64 : nullptr;
#define BWD_STAMP(k) do { if (dbg_cta && threadIdx.x == 0) dbg_cta[(k)] = clock64(); } while (0)
#define BWD_STAMP_ISSUER(k) do { if (dbg_cta && (threadIdx.x & 31) == 0) dbg_cta[(k)] = clock64(); } while (0)
#define BWD_TIMED_WAIT(bar, par, acc) do { if (dbg_cta) { long long t0_ = clock64(); mbar_wait((bar), (par)); (acc) += clock64() - t0_; } else mbar_wait((bar), (par)); } while (0)
  BWD_STAMP(0);
  using S = BwdSmem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kBars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::kTmemSlot);
  float* s_inv = reinterpret_cast<float*>(smem + S::kInv);
  float* s_delta = reinterpret_cast<float*>(smem + S::kDelta);
  float* s_rs = reinterpret_cast<float*>(smem + S::kRs);
  float* s_red = reinterpret_cast<float*>(smem + S::kRed);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.y, i0 = blockIdx.x * IB;
  const int cta = blockIdx.y * gridDim.x + blockIdx.x;
  const int64_t row0 = (int64_t)b * L + i0;
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0) asm volatile("trap;");

  auto load_v = [&](int h) {
    const int s = h % S::kVBufs;
    mbar_arrive_expect_tx(&bars[BV_FULL + s], S::kVBuf);
    tma_load_2d(smem + s * S::kVBuf, &map_v, &bars[BV_FULL + s], h * V_W, b * L);
  };
  if (warp == 9 && lane == 0) {
    // the producer lane initialises the barriers and starts the stage-1 loads before the CTA-wide synchronisation
    for (int i = 0; i < B_N_BARS; ++i) {
      const bool many = (i >= DPP_FREE && i < DPP_FREE + 3) || (i >= PCAT_READY && i < PCAT_READY + 4) || i == DE_FREE;
      mbar_init(&bars[i], i == BQ_FULL ? 256u : (many ? 128u : 1u));   // BQ_FULL: the compute threads publish dO / dopair
    }
    fence_barrier_init();
    tma_prefetch_desc(&map_v); tma_prefetch_desc(&map_e);
    for (int h = 0; h < S::kVBufs; ++h) load_v(h);
    // every pair row of the tile starts its way HBM -> L2 now: the stream runs during the prologue (prefetching only the
    // first 4 / 8 rows here, or the tile's dcat / cat rows first, changed nothing)
    for (int r = 0; r < IB; ++r) tma_prefetch_l2_2d(&map_e, 0, (int)((row0 + r) * L));
  }
  // per-row constants of this CTA and the st * Wpb operand tile ([8 h][64 c] bf16, 128B-swizzled rows)
  if (tid < 128) s_inv[tid] = stats[(row0 + (tid >> 3)) * 16 + 8 + (tid & 7)];
  if (tid < IB * 12) {           // frames of the CTA's rows for the prologue
    const int i = tid / 12, k = tid % 12;
    reinterpret_cast<float*>(smem + S::kFrame)[tid] = k < 9 ? R[(row0 + i) * 9 + k] : tc[(row0 + i) * 3 + (k - 9)];
  }
  if (tid < 256) {
    const float st = rsqrtf(3.0f);
    const int hh = tid >> 5, c2 = (tid & 31) * 2;   // two consecutive channels
    *reinterpret_cast<uint32_t*>(smem + S::kWpb + swz128_offset(hh, c2 >> 3) + (c2 & 7) * 2) =
        pack_bf162(st * wpb[hh * C + c2], st * wpb[hh * C + c2 + 1]);
  }
  fence_proxy_async_smem();
  __syncwarp();
  if (warp == 0) tmem_alloc(tmem_slot, 256);
  tcgen05_fence_before_sync();
  __syncthreads();
  tcgen05_fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  BWD_STAMP(1);

  // Issue order of the rows: group 0 works on rows {0,1} of a block of four while group 1 works on rows {2,3}, so
  // the rows become ready in the order 0,2,1,3.  ord() swaps the two low bits and is its own inverse: ord(row) is
  // the row's position in the issue order.
  auto ord = [](int k) { return (k & ~3) + ((k & 1) << 1) + ((k >> 1) & 1); };

  if (warp == 9) {
    // ======================================= TMA producer =======================================
    if (lane == 0) {
      for (int h = S::kVBufs; h < H; ++h) {
        mbar_wait(&bars[BV_EMPTY + h % S::kVBufs], ((h / S::kVBufs) - 1) & 1);
        load_v(h);
      }
      // ---- stage 2: pair rows + their dopair tiles (region X / P are free once every dPv MMA has completed)
      mbar_wait(&bars[BS_DONE], 0);
      for (int k2 = 0; k2 < IB; ++k2) {     // in issue order: the slots of a row pair are released together (Z MMAs below)
        const int r = ord(k2), s = r % S::kEStages;
        if (r >= S::kEStages) mbar_wait(&bars[BE_EMPTY + s], ((r / S::kEStages) - 1) & 1);
        mbar_arrive_expect_tx(&bars[BE_FULL + s], S::kEStage);
        tma_load_2d(smem + s * S::kEStage, &map_e, &bars[BE_FULL + s], 0, (int)((row0 + r) * L));
      }
    }
  } else if (warp == 8) {
    // ======================================= MMA issuer =======================================
    // the whole warp walks the control flow (warp-uniform descriptors stay in uniform registers), one elected lane issues
    {
      constexpr uint32_t kIdescDPV = make_idesc_f16(128, 16, 0, 0);
      constexpr uint32_t kIdescDPP = make_idesc_bf16(128, 16, 0, 0);
      constexpr uint32_t kIdescDE = make_idesc_bf16(128, 64, 0, 1);    // B = [dopair_i ; st Wpb], MN-major
      constexpr uint32_t kIdescZ = make_idesc_bf16(128, 16, 1, 1);     // A = two e tiles MN-major, B = two dl chunks MN-major
      // ---- stage 1: dPv^T_h = V_h dO_h^T
      mbar_wait(&bars[BQ_FULL], 0);
      for (int h = 0; h < H; ++h) {
        const int s = h % S::kVBufs;
        mbar_wait(&bars[BV_FULL + s], (h / S::kVBufs) & 1);
        tcgen05_fence_after_sync();
        if (elect_one()) {
          const uint32_t va = smem_base + s * S::kVBuf;
          const uint32_t oa = smem_base + S::kDoOff + h * 2048;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            uint64_t da = make_smem_desc(va + k * 32, 16, 1024, kSwizzle128B);
            uint64_t db = make_smem_desc(oa + k * 32, 16, 1024, kSwizzle128B);
            umma_bf16(tmem + kBColDPV + h * 16, da, db, kIdescDPV, k != 0);
          }
          umma_commit(&bars[BV_EMPTY + s]);
        }
        __syncwarp();
      }
      if (elect_one()) umma_commit(&bars[BS_DONE]);
      __syncwarp();
      BWD_STAMP_ISSUER(2);
      // ---- stage 2
      auto issue_dpp = [&](int pos) {   // pair part of dP for the row at issue position pos
        const int r = ord(pos), s = r % S::kEStages, ds = pos % 3;
        mbar_wait(&bars[BE_FULL + s], (r / S::kEStages) & 1);
        if (pos >= 3) mbar_wait(&bars[DPP_FREE + ds], ((pos / 3) - 1) & 1);
        tcgen05_fence_after_sync();
        if (elect_one()) {
          const uint32_t ea = smem_base + s * S::kEStage, da0 = smem_base + S::kDop + r * 1024;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            // N = 16: rows 8..15 of B are whatever follows the dopair tile (the next row's tile or the Wpb tile) and
            // land in accumulator columns 8..15, which nobody reads
            uint64_t da = make_smem_desc(ea + k * 32, 16, 1024, kSwizzle128B);
            uint64_t db = make_smem_desc(da0 + k * 32, 16, 1024, kSwizzle128B);
            umma_bf16(tmem + kBColDPP + ds * 16, da, db, kIdescDPP, k != 0);
          }
          umma_commit(&bars[DPP_DONE + ds]);
        }
        __syncwarp();
      };
      for (int k = 0; k < 3; ++k) issue_dpp(k);
      for (int k = 0; k < IB; ++k) {
        const int r = ord(k);
        const int g = (r >> 1) & 1, n = 2 * (r >> 2) + (r & 1), slot = n & 1;
        const int s = r % S::kEStages;
        mbar_wait(&bars[PCAT_READY + g * 2 + slot], (n >> 1) & 1);
        if (k >= 1) mbar_wait(&bars[DE_FREE], (k - 1) & 1);     // previous de drained out of the accumulator
        tcgen05_fence_after_sync();
        if (elect_one()) {
        const uint32_t pc = smem_base + S::kPcat + (g * 2 + slot) * 4096;
        const uint32_t dop = smem_base + S::kDop + r * 1024;
        {
          // A: [128 j][16] K-major, no swizzle: core matrices of 8 rows x 16 B; K chunks 2048 B apart (LBO),
          //    8-row groups 128 B apart (SBO).  B: [16 k][64 c] MN-major 128B-swizzled, two 8-row atoms:
          //    dopair_i, then st Wpb (SBO = distance between the two tiles).
          uint64_t da = make_smem_desc(pc, 2048, 128, kSwizzleNone);
          uint64_t db = make_smem_desc(dop, 1024, (smem_base + S::kWpb) - dop, kSwizzle128B);
          umma_bf16(tmem + kBColDE, da, db, kIdescDE, false);
        }
        umma_commit(&bars[DE_DONE + g]);
        if (k & 1) {
          // Z of the row PAIR at issue positions (k - 1, k) = rows (r - 2, r) = (group 0, group 1), same buffer slot:
          // [Z_a ; Z_b] = [e_a | e_b]^T [dl_a | dl_b]  (M = 128: 64 channels of each row, N = 16: 8 heads of each row,
          // K = 128 j) - a small tcgen05.mma costs ~60-80 issue cycles whatever its shape and this kernel's row loop is
          // bound by them (13 per row before, 9 now); the off-diagonal blocks are computed and ignored.
          // A: two e tiles read MN-major, two ring slots apart (LBO); B: two dl chunks [128 j][8 h] MN-major, no
          //    swizzle: 8-row (K) groups 128 B apart (LBO), the second group's buffer 8192 B behind the first (SBO).
          const uint32_t ea = smem_base + (s - 2) * S::kEStage;
          const uint32_t pc0 = smem_base + S::kPcat + slot * 4096;      // group 0's [P | dl] buffer of this slot
#pragma unroll
          for (int kk = 0; kk < L / 16; ++kk) {
            uint64_t da = make_smem_desc(ea + kk * 2048, 2 * S::kEStage, 1024, kSwizzle128B);
            uint64_t db = make_smem_desc(pc0 + 2048 + kk * 256, 128, 8192, kSwizzleNone);
            umma_bf16(tmem + kBColWPB, da, db, kIdescZ, (k > 1) || (kk != 0));
          }
          umma_commit(&bars[BE_EMPTY + s - 2]);
          umma_commit(&bars[BE_EMPTY + s]);
          umma_commit(&bars[PCAT_FREE + slot]);
          umma_commit(&bars[PCAT_FREE + 2 + slot]);
        }
        }
        __syncwarp();
        if (k + 3 < IB) issue_dpp(k + 3);
        BWD_STAMP_ISSUER(32 + k);
      }
      BWD_STAMP_ISSUER(3);
    }
  } else {
    // ======================================= softmax-gradient groups =======================================
    const int g = warp >> 2, gw = warp & 3, gt = tid & 127;
    const uint32_t tmem_lane = tmem + ((uint32_t)(gw * 32) << 16);
    auto bar_all_compute = [] { asm volatile("bar.sync 3, 256;" ::: "memory"); };
    float accg[H];
#pragma unroll
    for (int h = 0; h < H; ++h) accg[h] = 0.f;

    const uint4* pu_t = Pu + (row0 + 2 * g) * L + gt;     // row 4q + 2g + rr  ->  + (4q + rr) * L
    uint4 u_nxt[2] = {__ldg(pu_t), __ldg(pu_t + L)};

    // ---- prologue: dO / dopair / Delta of the CTA's 16 rows from dcat and cat.  Thread = (head ph, row pi), twice: warps
    //      0-3 take the scalar + point parts of their (row, head), warps 4-7 its pair part - every thread walks its own
    //      contiguous segments of the two rows with 16-byte loads (no shuffles, no per-warp serial work; the version with
    //      warp = head and lanes = columns spent 5k instructions per warp and was issue-bound at 45k cycles).
    {
      const int ph = (tid & 127) >> 4, pi = tid & 15;
      const float* dc = dcat + (row0 + pi) * NCAT;
      const __nv_bfloat16* ct = cat + (row0 + pi) * NCAT;
      float* s_max = reinterpret_cast<float*>(smem + S::kMax);            // [16 i][8 h]
      float* s_dp = reinterpret_cast<float*>(smem + S::kScr);             // [8 h][16 i]: pair part of Delta
      const float* fr = reinterpret_cast<const float*>(smem + S::kFrame) + pi * 12;
      auto bf_lo = [](uint32_t u) { return __uint_as_float(u << 16); };
      auto bf_hi = [](uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); };
      float dos[32], dog[24], acc = 0.f;
      BWD_STAMP(16);
      if (warp >= 4) {
        // pair part: the dopair operand tile of row pi ([8 h][128 B] bf16, 128B-swizzled) and its share of Delta
        uint8_t* tile = smem + S::kDop + pi * 1024 + ph * 128;
        const float* dp = dc + NS + ph * C;
        const __nv_bfloat16* op = ct + NS + ph * C;
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          const int c = (c8 + pi) & 7;     // the 8 lanes of a quarter-warp (rows pi .. pi+7, same head) hit 8 different banks
          const float4 a = __ldg(reinterpret_cast<const float4*>(dp + c * 8));
          const float4 b2 = __ldg(reinterpret_cast<const float4*>(dp + c * 8 + 4));
          const uint4 o = __ldg(reinterpret_cast<const uint4*>(op + c * 8));
          acc += a.x * bf_lo(o.x) + a.y * bf_hi(o.x) + a.z * bf_lo(o.y) + a.w * bf_hi(o.y) + b2.x * bf_lo(o.z) +
                 b2.y * bf_hi(o.z) + b2.z * bf_lo(o.w) + b2.w * bf_hi(o.w);
          *reinterpret_cast<uint4*>(tile + ((c ^ ph) << 4)) =
              make_uint4(pack_bf162(a.x, a.y), pack_bf162(a.z, a.w), pack_bf162(b2.x, b2.y), pack_bf162(b2.z, b2.w));
        }
        s_dp[tid & 127] = acc;
      } else {
        // point part: ol = (og - t) R^T, nrm = |ol| (diffab_pytorch.py:327-336,453-457) -> d_ol += dnrm ol / nrm; dog = d_ol R
        float dl[24], ol[24], dn[8];
#pragma unroll
        for (int c = 0; c < 6; ++c) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(dc + NS + H * C + ph * (P * 3) + c * 4));
          dl[4 * c] = a.x; dl[4 * c + 1] = a.y; dl[4 * c + 2] = a.z; dl[4 * c + 3] = a.w;
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const uint4 o = __ldg(reinterpret_cast<const uint4*>(ct + NS + H * C + ph * (P * 3) + c * 8));
          ol[8 * c] = bf_lo(o.x); ol[8 * c + 1] = bf_hi(o.x); ol[8 * c + 2] = bf_lo(o.y); ol[8 * c + 3] = bf_hi(o.y);
          ol[8 * c + 4] = bf_lo(o.z); ol[8 * c + 5] = bf_hi(o.z); ol[8 * c + 6] = bf_lo(o.w); ol[8 * c + 7] = bf_hi(o.w);
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(dc + NS + H * C + NPT + ph * P + c * 4));
          dn[4 * c] = a.x; dn[4 * c + 1] = a.y; dn[4 * c + 2] = a.z; dn[4 * c + 3] = a.w;
        }
        float mx = 0.f;
#pragma unroll
        for (int p = 0; p < P; ++p) {
          const float x0 = ol[3 * p], x1 = ol[3 * p + 1], x2 = ol[3 * p + 2];
          float d0 = dl[3 * p], d1 = dl[3 * p + 1], d2 = dl[3 * p + 2];
          const float nrm = sqrtf(x0 * x0 + x1 * x1 + x2 * x2);
          if (nrm > 0.f) { d0 += dn[p] * x0 / nrm; d1 += dn[p] * x1 / nrm; d2 += dn[p] * x2 / nrm; }
#pragma unroll
          for (int k = 0; k < 3; ++k) {
            dog[3 * p + k] = d0 * fr[k] + d1 * fr[3 + k] + d2 * fr[6 + k];
            mx = fmaxf(mx, fabsf(dog[3 * p + k]));
          }
          // <dog, og> with og = ol R + t:  (d_ol R).(ol R) = d_ol . ol  (R orthogonal)
          acc += d0 * x0 + d1 * x1 + d2 * x2 + dog[3 * p] * fr[9] + dog[3 * p + 1] * fr[10] + dog[3 * p + 2] * fr[11];
        }
        // scalar part
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float4 a = __ldg(reinterpret_cast<const float4*>(dc + ph * DS + c * 8));
          const float4 b2 = __ldg(reinterpret_cast<const float4*>(dc + ph * DS + c * 8 + 4));
          const uint4 o = __ldg(reinterpret_cast<const uint4*>(ct + ph * DS + c * 8));
          dos[8 * c] = a.x; dos[8 * c + 1] = a.y; dos[8 * c + 2] = a.z; dos[8 * c + 3] = a.w;
          dos[8 * c + 4] = b2.x; dos[8 * c + 5] = b2.y; dos[8 * c + 6] = b2.z; dos[8 * c + 7] = b2.w;
          acc += a.x * bf_lo(o.x) + a.y * bf_hi(o.x) + a.z * bf_lo(o.y) + a.w * bf_hi(o.y) + b2.x * bf_lo(o.z) +
                 b2.y * bf_hi(o.z) + b2.z * bf_lo(o.w) + b2.w * bf_hi(o.w);
        }
#pragma unroll
        for (int k = 0; k < 32; ++k) mx = fmaxf(mx, fabsf(dos[k]));
        s_max[pi * 8 + ph] = mx;
      }
      BWD_STAMP(18);
      bar_all_compute();
      if (warp < 4) {
        s_delta[pi * 8 + ph] = acc + s_dp[tid];
        // power-of-two scale that puts the largest entry of the row in [2^11, 2^12): fp16 keeps >= 11 bits for
        // everything within 2^-25 of it, whatever the magnitude of the upstream gradient
        const float4 m0 = *reinterpret_cast<const float4*>(s_max + pi * 8), m1 = *reinterpret_cast<const float4*>(s_max + pi * 8 + 4);
        const float m = fmaxf(fmaxf(fmaxf(m0.x, m0.y), fmaxf(m0.z, m0.w)), fmaxf(fmaxf(m1.x, m1.y), fmaxf(m1.z, m1.w)));
        float sc = 1.0f;
        if (m > 0.f && m < 3.0e38f) {
          int ex;
          frexpf(m, &ex);
          sc = ldexpf(1.0f, max(-100, min(100, 12 - ex)));
        }
        if (ph == 0) s_rs[pi] = 1.0f / sc;
        // dO row of (head, row): [dos 32 | dog 24 | 0 x 8] -> fp16 scaled into the B operand tile of dPv ([16 i][128 B],
        // 128B-swizzled), bf16 unscaled to HBM for the key side
        uint8_t* ot = smem + S::kDoOff + ph * 2048 + pi * 128;
        uint4* ob = reinterpret_cast<uint4*>(dObf + ((row0 + pi) * H + ph) * 64);
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          float v[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) v[k] = c < 4 ? dos[8 * c + k] : (c < 7 ? dog[8 * (c - 4) + k] : 0.f);
          *reinterpret_cast<uint4*>(ot + ((c ^ (pi & 7)) << 4)) =
              make_uint4(pack_h2(v[0] * sc, v[1] * sc), pack_h2(v[2] * sc, v[3] * sc), pack_h2(v[4] * sc, v[5] * sc),
                         pack_h2(v[6] * sc, v[7] * sc));
          ob[c] = make_uint4(pack_bf162(v[0], v[1]), pack_bf162(v[2], v[3]), pack_bf162(v[4], v[5]), pack_bf162(v[6], v[7]));
        }
      }
      BWD_STAMP(20);
      fence_proxy_async_smem();
      mbar_arrive(&bars[BQ_FULL]);
      bar_all_compute();        // s_delta / s_rs of every row are visible to every compute thread
    }
    mbar_wait(&bars[BS_DONE], 0);
    tcgen05_fence_after_sync();
    BWD_STAMP(4);
    long long w_dpp = 0, w_pcat = 0, w_de = 0;
    for (int q = 0; q < IB / 4; ++q) {
      const uint4 u_use[2] = {u_nxt[0], u_nxt[1]};
      if (q + 1 < IB / 4) {
        u_nxt[0] = __ldg(pu_t + (size_t)(4 * (q + 1)) * L);
        u_nxt[1] = __ldg(pu_t + (size_t)(4 * (q + 1) + 1) * L);
      }
      float dpv[H][2];
#pragma unroll
      for (int h = 0; h < H; ++h) tmem_ld_x2(tmem_lane + kBColDPV + h * 16 + 4 * q + 2 * g, dpv[h]);
      tmem_wait_ld();
#pragma unroll
      for (int rr = 0; rr < 2; ++rr) {
        const int i = 4 * q + 2 * g + rr, n = 2 * q + rr, pos = ord(i);
        float lm[H], p[H], dl[H];
        {
          const __nv_bfloat162* ub = reinterpret_cast<const __nv_bfloat162*>(&u_use[rr]);
          const float4 v0 = *reinterpret_cast<const float4*>(s_inv + i * 8), v1 = *reinterpret_cast<const float4*>(s_inv + i * 8 + 4);
          const float inv[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const float2 f = __bfloat1622float2(ub[k]);
            p[2 * k] = f.x; p[2 * k + 1] = f.y;
          }
#pragma unroll
          for (int h = 0; h < H; ++h) {
            lm[h] = p[h] > 0.f ? lg2(p[h]) : 0.f;      // log2 of the un-normalised probability (<= 0)
            p[h] *= inv[h];
          }
        }
        // pair part of dP for this row
        BWD_TIMED_WAIT(&bars[DPP_DONE + pos % 3], (pos / 3) & 1, w_dpp);
        tcgen05_fence_after_sync();
        float dpp[8];
        tmem_ld_x8(tmem_lane + kBColDPP + (pos % 3) * 16, dpp);
        tmem_wait_ld();
        tcgen05_fence_before_sync();
        mbar_arrive(&bars[DPP_FREE + pos % 3]);
        {
          const float rs = s_rs[i];
          const float4 d0 = *reinterpret_cast<const float4*>(s_delta + i * 8), d1 = *reinterpret_cast<const float4*>(s_delta + i * 8 + 4);
          const float dlt[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
          for (int h = 0; h < H; ++h) {
            const float dP = fmaf(dpv[h][rr], rs, dpp[h]);
            dl[h] = p[h] * (dP - dlt[h]);
            accg[h] = fmaf(dl[h], lm[h], accg[h]);
          }
        }
        if (n >= 2) BWD_TIMED_WAIT(&bars[PCAT_FREE + g * 2 + (n & 1)], ((n >> 1) - 1) & 1, w_pcat);
        // ---- [P | dl] of this key: A operand of the de MMA, and (dl half) B operand of the Z MMA
        {
          uint8_t* pc = smem + S::kPcat + (g * 2 + (n & 1)) * 4096;
          *reinterpret_cast<uint4*>(pc + gt * 16) = pack8_bf16(p);
          *reinterpret_cast<uint4*>(pc + 2048 + gt * 16) = pack8_bf16(dl);
        }
        fence_proxy_async_smem();
        tcgen05_fence_before_sync();
        mbar_arrive(&bars[PCAT_READY + g * 2 + (n & 1)]);
        // ---- P and dl as [h][i][j] rows for the key side; neighbouring lanes trade heads so that every store is a
        //      packed pair (j, j+1).  Runs while the issuer turns the operands above into de_i.
        {
          const int je = gt & ~1;
          const bool odd = lane & 1;
#pragma unroll
          for (int hh = 0; hh < 4; ++hh) {
            const int h = 2 * hh + (odd ? 1 : 0);
            const float ps = odd ? p[2 * hh] : p[2 * hh + 1];
            const float pr = __shfl_xor_sync(0xffffffffu, ps, 1);
            const float ds = odd ? dl[2 * hh] : dl[2 * hh + 1];
            const float dr = __shfl_xor_sync(0xffffffffu, ds, 1);
            const uint32_t pv = odd ? pack_bf162(pr, p[2 * hh + 1]) : pack_bf162(p[2 * hh], pr);
            const uint32_t dv = odd ? pack_bf162(dr, dl[2 * hh + 1]) : pack_bf162(dl[2 * hh], dr);
            const size_t go = (((size_t)b * H + h) * L + (i0 + i)) * L + je;
            *reinterpret_cast<uint32_t*>(Pn + go) = pv;
            *reinterpret_cast<uint32_t*>(dL + go) = dv;
          }
        }
        // ---- de_i: TMEM -> bf16 -> 128 contiguous bytes per key; then hand the accumulator back
        {
          BWD_TIMED_WAIT(&bars[DE_DONE + g], n & 1, w_de);
          tcgen05_fence_after_sync();
          uint4* dst = reinterpret_cast<uint4*>(de + ((row0 + i) * L + gt) * C);
#pragma unroll
          for (int half = 0; half < 2; ++half) {
            float v[32];
            tmem_ld_x32(tmem_lane + kBColDE + half * 32, v);
            tmem_wait_ld();
            if (half == 1) {
              tcgen05_fence_before_sync();
              mbar_arrive(&bars[DE_FREE]);
            }
            // 256-bit stores: every request is one whole 32-byte sector of the key's 128-byte line (16-byte stores at a
            // 128-byte lane stride are half-sector writes, twice as many requests)
#pragma unroll
            for (int qq = 0; qq < 2; ++qq)
              st_global_v8(dst + half * 4 + qq * 2,
                           pack_bf162(v[16 * qq], v[16 * qq + 1]), pack_bf162(v[16 * qq + 2], v[16 * qq + 3]),
                           pack_bf162(v[16 * qq + 4], v[16 * qq + 5]), pack_bf162(v[16 * qq + 6], v[16 * qq + 7]),
                           pack_bf162(v[16 * qq + 8], v[16 * qq + 9]), pack_bf162(v[16 * qq + 10], v[16 * qq + 11]),
                           pack_bf162(v[16 * qq + 12], v[16 * qq + 13]), pack_bf162(v[16 * qq + 14], v[16 * qq + 15]));
          }
        }
        BWD_STAMP(8 + n);
      }
    }
    BWD_STAMP(5);
    if (dbg_cta && tid == 0) { dbg_cta[21] = w_dpp; dbg_cta[22] = w_pcat; dbg_cta[23] = w_de; }

    // ---- sum_ij dl (l - m) per head (natural-log units) for dgamma
#pragma unroll
    for (int h = 0; h < H; ++h) accg[h] = warp_sum(accg[h]);
    if (lane == 0) {
#pragma unroll
      for (int h = 0; h < H; ++h) s_red[warp * 8 + h] = accg[h];
    }
    bar_all_compute();
    if (tid < 8) {
      float s = 0.f;
      for (int w = 0; w < 8; ++w) s += s_red[w * 8 + tid];
      p_g1[(size_t)cta * 8 + tid] = s * kLn2;
    }
    // ---- to_pair_bias partial: TMEM lane = channel c of the pair's first row (lanes 0-63, columns 0-7) / second row
    //      (lanes 64-127, columns 8-15); the two halves meet in shared memory (the [P | dl] buffers are idle by now)
    if (g == 1) {
      mbar_wait(&bars[PCAT_FREE + 3], 1);   // 4th completion of [g=1][slot=1]: commit behind the Z MMAs of the last row pair
      tcgen05_fence_after_sync();
      float z[8];
      tmem_ld_x8(tmem_lane + kBColWPB + (gt >> 6) * 8, z);
      tmem_wait_ld();
      float* s_z = reinterpret_cast<float*>(smem + S::kPcat);      // [64 c][8 h]
      if (gt >= 64) {
#pragma unroll
        for (int h = 0; h < H; ++h) s_z[(gt - 64) * 8 + h] = z[h];
      }
      asm volatile("bar.sync 2, 128;" ::: "memory");
      if (gt < 64) {
#pragma unroll
        for (int h = 0; h < H; ++h) p_wpb[(size_t)cta * 512 + h * C + gt] = z[h] + s_z[gt * 8 + h];
      }
    }
    BWD_STAMP(6);
  }
  tcgen05_fence_before_sync();
  __syncthreads();
  BWD_STAMP(7);
#undef BWD_STAMP
#undef BWD_STAMP_ISSUER
#undef BWD_TIMED_WAIT
  if (warp == 0) tmem_free(tmem, 256);
}

// ---- 3. key side (and dQ) --------------------------------------------------------------------------------------
// Per (patch, head): the [128 i][128 j] tiles of P and dl are resident, so all three contractions over them run here:
//   dV_h = P_h^T dO_h           (M = j, N = 64, K = i)      A = P tile read MN-major
//   dK_h = dl_h^T Q_h[:, :64]   (M = j, N = 64, K = i)      A = dl tile read MN-major
//   dQ_h = dl_h K_h[:, :64]     (M = i, N = 64, K = j)      A = the same dl tile read K-major
struct KsSmem {
  static constexpr int kPn = 0;          // two [128 i][64 j] boxes, 128B-swizzled
  static constexpr int kDl = 32768;
  static constexpr int kDo = 65536;      // [128 i][64 d]
  static constexpr int kQ = 81920;       // [128 i][64: scalar | point hi | 1 1 1]
  static constexpr int kK = 98304;       // [128 j][64: scalar | point hi | norm terms | 1]
  static constexpr int kBars = 114688;
  static constexpr int kTmemSlot = kBars + 64;
  static constexpr int kTotal = kTmemSlot + 16;
};
static_assert(KsSmem::kTotal <= 113 * 1024, "two CTAs per SM");

__global__ void __launch_bounds__(160, 2)
ipa_bwd_keyside_kernel(const __grid_constant__ CUtensorMap map_pn, const __grid_constant__ CUtensorMap map_dl,
                       const __grid_constant__ CUtensorMap map_do, const __grid_constant__ CUtensorMap map_q64,
                       const __grid_constant__ CUtensorMap map_k64, const __nv_bfloat16* __restrict__ Qp,
                       const __nv_bfloat16* __restrict__ Kp, const float* __restrict__ R, const float* __restrict__ gamma,
                       __nv_bfloat16* __restrict__ dproj, float* __restrict__ p_g2, float* __restrict__ dbg_qkv) {
  extern __shared__ __align__(1024) uint8_t smem[];
  using S = KsSmem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kBars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::kTmemSlot);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.x / H, h = blockIdx.x % H;
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0) asm volatile("trap;");
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    mbar_init(&bars[2], 1);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(tmem_slot, 256);
  tcgen05_fence_before_sync();
  __syncthreads();
  tcgen05_fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  if (warp == 4) {
    // whole warp walks the control flow, one elected lane issues the loads and the MMAs
    if (elect_one()) {
      const int prow = (b * H + h) * L;
      mbar_arrive_expect_tx(&bars[0], 32768 + 16384);
      tma_load_2d(smem + S::kPn, &map_pn, &bars[0], 0, prow);
      tma_load_2d(smem + S::kPn + 16384, &map_pn, &bars[0], 64, prow);
      tma_load_2d(smem + S::kDo, &map_do, &bars[0], h * 64, b * L);
      mbar_arrive_expect_tx(&bars[1], 32768 + 32768);
      tma_load_2d(smem + S::kDl, &map_dl, &bars[1], 0, prow);
      tma_load_2d(smem + S::kDl + 16384, &map_dl, &bars[1], 64, prow);
      tma_load_2d(smem + S::kQ, &map_q64, &bars[1], h * QK_W, b * L);
      tma_load_2d(smem + S::kK, &map_k64, &bars[1], h * QK_W, b * L);
    }
    __syncwarp();
    constexpr uint32_t idesc_t = make_idesc_bf16(128, 64, 1, 1);
    constexpr uint32_t idesc_q = make_idesc_bf16(128, 64, 0, 1);
    mbar_wait(&bars[0], 0);
    tcgen05_fence_after_sync();
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < L / 16; ++k) {
        // A: [i][j] tile read MN-major (M = j): two 64-wide atoms 16 KB apart (LBO), 8-row (K = i) groups 1 KB apart
        uint64_t da = make_smem_desc(smem_base + S::kPn + k * 2048, 16384, 1024, kSwizzle128B);
        uint64_t db = make_smem_desc(smem_base + S::kDo + k * 2048, 1024, 1024, kSwizzle128B);
        umma_bf16(tmem, da, db, idesc_t, k != 0);
      }
    }
    __syncwarp();
    mbar_wait(&bars[1], 0);
    tcgen05_fence_after_sync();
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < L / 16; ++k) {
        uint64_t da = make_smem_desc(smem_base + S::kDl + k * 2048, 16384, 1024, kSwizzle128B);
        uint64_t db = make_smem_desc(smem_base + S::kQ + k * 2048, 1024, 1024, kSwizzle128B);
        umma_bf16(tmem + 64, da, db, idesc_t, k != 0);
      }
#pragma unroll
      for (int k = 0; k < L / 16; ++k) {
        // A: the dl tile read K-major (M = i rows of 128 B; K = j: box k / 4, 32 B per step inside the row)
        uint64_t da = make_smem_desc(smem_base + S::kDl + (k >> 2) * 16384 + (k & 3) * 32, 16, 1024, kSwizzle128B);
        uint64_t db = make_smem_desc(smem_base + S::kK + k * 2048, 1024, 1024, kSwizzle128B);
        umma_bf16(tmem + 128, da, db, idesc_q, k != 0);
      }
      umma_commit(&bars[2]);
    }
    __syncwarp();
  } else {
    // ---- epilogue: thread = residue (key row j for dV / dK, query row i for dQ), head h.  Scales, the
    //      -c q~ sum dl corrections, global -> local frame, and the result goes straight into the dproj row
    //      (bf16; row layout = rows of Wcat: [q_s 256 | k_s 256 | v_s 256 | q_p 192 | k_p 192 | v_p 192]).
    float* s_g2 = reinterpret_cast<float*>(smem + S::kBars + 32);
    const int64_t row = (int64_t)b * L + tid;
    float Rm[9];
#pragma unroll
    for (int c = 0; c < 9; ++c) Rm[c] = __ldg(R + row * 9 + c);
    const float ss = rsqrtf((float)DS), sp = rsqrtf(4.5f * P), st = rsqrtf(3.0f);
    const float c1 = st * sp * __ldg(gamma + h);
    __nv_bfloat16* out = dproj + row * NPROJ;
    mbar_wait(&bars[2], 0);
    tcgen05_fence_after_sync();
    const uint32_t tmem_lane = tmem + ((uint32_t)(warp * 32) << 16);
    float U[64];
    auto load64 = [&](int m) {
      float a[32], c[32];
      tmem_ld_x32(tmem_lane + m * 64, a);
      tmem_ld_x32(tmem_lane + m * 64 + 32, c);
      tmem_wait_ld();
#pragma unroll
      for (int i = 0; i < 32; ++i) { U[i] = a[i]; U[32 + i] = c[i]; }
      if (dbg_qkv) {   // test hook: raw accumulators [matrix][row][head][64]
        float* d = dbg_qkv + (((size_t)(2 - m) * (gridDim.x / H) * L + row) * H + h) * 64;   // slots dQ, dK, dV
#pragma unroll
        for (int i = 0; i < 64; ++i) d[i] = U[i];
      }
    };
    auto store_scalars = [&](int seg, float scale) {
      uint4* dst = reinterpret_cast<uint4*>(out + seg * NS + h * DS);      // 64 B, 32-byte aligned: two 256-bit stores
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        uint32_t w[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) w[e] = pack_bf162(U[16 * q + 2 * e] * scale, U[16 * q + 2 * e + 1] * scale);
        st_global_v8(dst + 2 * q, w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7]);
      }
    };
    // global-frame gradient gp[24] -> local frame (p_glob = p_loc R + t  =>  dp_loc = dp_glob R^T)
    auto store_points = [&](int seg, const float (&gp)[24]) {
      float loc[24];
#pragma unroll
      for (int p = 0; p < P; ++p) {
        const float x = gp[3 * p], y = gp[3 * p + 1], z = gp[3 * p + 2];
        loc[3 * p] = x * Rm[0] + y * Rm[1] + z * Rm[2];
        loc[3 * p + 1] = x * Rm[3] + y * Rm[4] + z * Rm[5];
        loc[3 * p + 2] = x * Rm[6] + y * Rm[7] + z * Rm[8];
      }
      // 48 B at a 16-byte aligned offset (48 h): one 256-bit store on the 32-byte aligned part, one 16-byte store
      uint4* dst = reinterpret_cast<uint4*>(out + 3 * NS + seg * NPT + h * 24);
      uint32_t w[12];
#pragma unroll
      for (int e = 0; e < 12; ++e) w[e] = pack_bf162(loc[2 * e], loc[2 * e + 1]);
      if (h & 1) {
        dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
        st_global_v8(dst + 1, w[4], w[5], w[6], w[7], w[8], w[9], w[10], w[11]);
      } else {
        st_global_v8(dst, w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7]);
        dst[2] = make_uint4(w[8], w[9], w[10], w[11]);
      }
    };
    auto load_points = [&](const __nv_bfloat16* src, float (&pt)[24]) {   // hi + lo of the packed row
      const uint4* r = reinterpret_cast<const uint4*>(src + row * (H * QK_W) + h * QK_W);
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const uint4 hi = __ldg(r + 4 + q), lo = __ldg(r + 8 + q);
        const __nv_bfloat162* hp = reinterpret_cast<const __nv_bfloat162*>(&hi);
        const __nv_bfloat162* lp = reinterpret_cast<const __nv_bfloat162*>(&lo);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 a = __bfloat1622float2(hp[e]), c = __bfloat1622float2(lp[e]);
          pt[8 * q + 2 * e] = a.x + c.x;
          pt[8 * q + 2 * e + 1] = a.y + c.y;
        }
      }
    };
    float gp[24], pt[24];
    // ---- values: dV = sum_i P [dos | dog]
    load64(0);
    store_scalars(2, 1.0f);
#pragma unroll
    for (int c = 0; c < 24; ++c) gp[c] = U[32 + c];
    store_points(2, gp);
    // ---- key side: W = sum_i dl [st ss log2e qs | c_h log2e q~hi | 1 1 1 | 0]
    load64(1);
    store_scalars(1, kLn2);
    load_points(Kp, pt);                       // = k~
    {
      const float rj = U[56];
#pragma unroll
      for (int c = 0; c < 24; ++c) gp[c] = U[32 + c] * kLn2 - c1 * pt[c] * rj;
    }
    store_points(1, gp);
    // ---- query side: U = sum_j dl [ks | k~hi | norm columns | 1]
    load64(2);
    float g2 = 0.f;
    {
      const uint4* qr = reinterpret_cast<const uint4*>(Qp + row * (H * QK_W) + h * QK_W);   // Qp_s = st ss log2e qs
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint4 v = __ldg(qr + q);
        const __nv_bfloat162* vp = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 a = __bfloat1622float2(vp[e]);
          g2 = fmaf(a.x, U[8 * q + 2 * e], g2);
          g2 = fmaf(a.y, U[8 * q + 2 * e + 1], g2);
        }
      }
      g2 *= kLn2;
    }
    store_scalars(0, st * ss);
    load_points(Qp, pt);                       // = c_h log2e q~
    {
      const float si = U[59];
#pragma unroll
      for (int c = 0; c < 24; ++c) gp[c] = c1 * U[32 + c] - pt[c] * kLn2 * si;
    }
    store_points(0, gp);
    // ---- sum_i <qs, dqs> of this (patch, head) for dgamma
    g2 = warp_sum(g2);
    if (lane == 0) s_g2[warp] = g2;
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (tid == 0) p_g2[blockIdx.x] = s_g2[0] + s_g2[1] + s_g2[2] + s_g2[3];
  }
  tcgen05_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_free(tmem, 256);
}

// ---- 5. finalize -------------------------------------------------------------------------------------------
// Deterministic two-level reduction of the per-CTA partials.  Level 1: block k sums a slice of the core CTAs
// (and of the assemble blocks) into r_part[k][512 + 16].
constexpr int kRedBlocks = 32;
__global__ void __launch_bounds__(512) bwd_reduce_kernel(const float* __restrict__ p_wpb, int n_cta,
                                                         const float* __restrict__ p_g1, const float* __restrict__ p_g2,
                                                         int n_blk, float* __restrict__ r_part) {
  const int t = threadIdx.x, k = blockIdx.x;
  const int c0 = (int)((int64_t)n_cta * k / kRedBlocks), c1 = (int)((int64_t)n_cta * (k + 1) / kRedBlocks);
  float z0 = 0.f, z1 = 0.f, z2 = 0.f, z3 = 0.f;
  int c = c0;
  for (; c + 3 < c1; c += 4) {
    z0 += p_wpb[(size_t)c * 512 + t]; z1 += p_wpb[(size_t)(c + 1) * 512 + t];
    z2 += p_wpb[(size_t)(c + 2) * 512 + t]; z3 += p_wpb[(size_t)(c + 3) * 512 + t];
  }
  for (; c < c1; ++c) z0 += p_wpb[(size_t)c * 512 + t];
  r_part[(size_t)k * 528 + t] = (z0 + z1) + (z2 + z3);
  if (t < 8) {
    float g1 = 0.f;
    for (int q = c0; q < c1; ++q) g1 += p_g1[(size_t)q * 8 + t];
    r_part[(size_t)k * 528 + 512 + t] = g1;
  } else if (t < 16) {
    const int b0 = (int)((int64_t)n_blk * k / kRedBlocks), b1 = (int)((int64_t)n_blk * (k + 1) / kRedBlocks);
    float g2 = 0.f;
    for (int q = b0; q < b1; ++q) g2 += p_g2[(size_t)q * 8 + (t - 8)];
    r_part[(size_t)k * 528 + 512 + t] = g2;
  }
}
// Level 2: one block.  dWpb = st Z; dgamma = (sum dl l - sum dl ls - sum dl lb) / gamma.
__global__ void __launch_bounds__(512) bwd_finalize_kernel(const float* __restrict__ r_part, const float* __restrict__ wpb,
                                                           const float* __restrict__ gamma, float* __restrict__ d_wpb,
                                                           float* __restrict__ d_gamma) {
  __shared__ float s_g3[512];
  const int t = threadIdx.x;   // = h * 64 + c
  const float st = rsqrtf(3.0f);
  float z = 0.f;
  for (int k = 0; k < kRedBlocks; ++k) z += r_part[(size_t)k * 528 + t];
  d_wpb[t] += st * z;
  s_g3[t] = st * wpb[t] * z;
  __syncthreads();
  if (t < 8) {
    float g3 = 0.f;
    for (int c = 0; c < C; ++c) g3 += s_g3[t * C + c];
    float g1 = 0.f, g2 = 0.f;
    for (int k = 0; k < kRedBlocks; ++k) { g1 += r_part[(size_t)k * 528 + 512 + t]; g2 += r_part[(size_t)k * 528 + 520 + t]; }
    const float gm = gamma[t];
    // lp = gamma * (dlp/dgamma)  =>  dgamma = sum dl lp / gamma (0 when gamma == 0: the point term is then absent)
    if (gm != 0.f) d_gamma[t] += (g1 - g2 - g3) / gm;
  }
}

}  // namespace sm100
}  // namespace dab

using namespace dab;
using namespace dab::sm100;

extern "C" {

size_t dab_ipa_bwd_sm100_workspace_bytes(const DabIpaDims* d) { return shape_ok(d) ? carve_bwd(d->B, nullptr).bytes : 0; }

static int bwd_sm100_impl(const DabIpaDims* d, const void* packed, const void* e_bf16, const float* R, const float* dcat,
                          void* saved, size_t saved_bytes, void* dproj_bf16, void* de_bf16, float* d_w_pair_bias, float* d_gamma,
                          void* workspace, size_t workspace_bytes, void* stream, bool finish) {
  const char* fn = finish ? "dab_ipa_bwd_sm100_finish" : "dab_ipa_bwd_sm100_main";
  DAB_REQUIRE(shape_ok(d), DAB_EUNSUPPORTED, "%s: the sm_100a fast path needs L=128, D=128, C=64, H=8, ds=32, Pq=Pv=8", fn);
  if (d->B == 0) return DAB_OK;
  DAB_REQUIRE(packed && e_bf16 && R && dcat && saved && dproj_bf16 && de_bf16 && d_w_pair_bias && d_gamma && workspace,
              DAB_EINVAL, "%s: null pointer", fn);
  DAB_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0 && (reinterpret_cast<uintptr_t>(saved) & 1023) == 0 &&
                  (reinterpret_cast<uintptr_t>(e_bf16) & 127) == 0 && (reinterpret_cast<uintptr_t>(de_bf16) & 127) == 0 &&
                  aligned16(dcat) && aligned32(dproj_bf16),
              DAB_EINVAL, "%s: misaligned pointer (workspaces 1024 B, e/de 128 B, dcat 16 B, dproj 32 B)", fn);
  const int B = d->B, M = B * L;
  Ws ws = carve_ws(B, saved);
  BwdWs bw = carve_bwd(B, workspace);
  DAB_REQUIRE(saved_bytes >= ws.bytes, DAB_EWORKSPACE, "%s: saved workspace %zu < %zu", fn, saved_bytes, ws.bytes);
  DAB_REQUIRE(workspace_bytes >= bw.bytes, DAB_EWORKSPACE, "%s: workspace %zu < %zu", fn, workspace_bytes, bw.bytes);
  const PackedOffsets po = packed_offsets();
  const uint8_t* pk = reinterpret_cast<const uint8_t*>(packed);
  const float* wpb = reinterpret_cast<const float*>(pk + po.wpb);
  const float* gamma = reinterpret_cast<const float*>(pk + po.gamma);
  cudaStream_t s = (cudaStream_t)stream;

  if (finish) {   // only the final reductions: d_w_pair_bias / d_gamma from the partial sums of an earlier main pass
    bwd_reduce_kernel<<<kRedBlocks, 512, 0, s>>>(bw.p_wpb, B * 8, bw.p_g1, bw.p_g2, B, bw.r_part);
    count_launch();
    bwd_finalize_kernel<<<1, 512, 0, s>>>(bw.r_part, wpb, gamma, d_w_pair_bias, d_gamma);
    count_launch();
    return check_launch(fn);
  }
  CUtensorMap mv, me;
  {
    uint64_t dv[2] = {(uint64_t)H * V_W, (uint64_t)M}, sv[1] = {(uint64_t)H * V_W * 2};
    uint32_t bv[2] = {V_W, L};
    if (int rc = make_tensor_map_bf16(&mv, ws.Vp, 2, dv, sv, bv, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    uint64_t de_[2] = {(uint64_t)C, (uint64_t)M * L}, se[1] = {(uint64_t)C * 2};
    uint32_t be[2] = {C, L};
    if (int rc = make_tensor_map_bf16(&me, e_bf16, 2, de_, se, be, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  }
  DAB_ENSURE_SMEM(ipa_bwd_core_kernel, BwdSmem::kTotal);
  DAB_ENSURE_SMEM(ipa_bwd_keyside_kernel, KsSmem::kTotal);
  ipa_bwd_core_kernel<<<dim3(L / IB, B), 320, BwdSmem::kTotal, s>>>(
      mv, me, dcat, ws.cat, R, ws.tc, bw.dObf, ws.pu, ws.stats, wpb, reinterpret_cast<__nv_bfloat16*>(de_bf16), bw.Pn,
      bw.dL, bw.p_wpb, bw.p_g1, g_bwd_dbg);
  count_launch();

  CUtensorMap mpn, mdl, mdob, mq64, mk64;
  {
    uint64_t dp[2] = {(uint64_t)L, (uint64_t)B * H * L}, sp_[1] = {(uint64_t)L * 2};
    uint32_t bp[2] = {64, L};
    if (int rc = make_tensor_map_bf16(&mpn, bw.Pn, 2, dp, sp_, bp, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    if (int rc = make_tensor_map_bf16(&mdl, bw.dL, 2, dp, sp_, bp, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    uint64_t dv[2] = {(uint64_t)H * 64, (uint64_t)M}, sv[1] = {(uint64_t)H * 64 * 2};
    uint32_t bv[2] = {64, L};
    if (int rc = make_tensor_map_bf16(&mdob, bw.dObf, 2, dv, sv, bv, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    uint64_t dqk[2] = {(uint64_t)H * QK_W, (uint64_t)M}, sqk[1] = {(uint64_t)H * QK_W * 2};
    if (int rc = make_tensor_map_bf16(&mq64, ws.Qp, 2, dqk, sqk, bv, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
    if (int rc = make_tensor_map_bf16(&mk64, ws.Kp, 2, dqk, sqk, bv, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  }
  ipa_bwd_keyside_kernel<<<B * H, 160, KsSmem::kTotal, s>>>(mpn, mdl, mdob, mq64, mk64, ws.Qp, ws.Kp, R, gamma,
                                                            reinterpret_cast<__nv_bfloat16*>(dproj_bf16), bw.p_g2,
                                                            g_bwd_keep_qkv ? bw.dQ : nullptr);
  count_launch();
  return check_launch(fn);
}

/* The backward in two calls, so that a caller can overlap what depends only on dproj (dx, dWcat) with the final
 * reductions: `_main` = everything up to dproj / de and the per-CTA partial sums, `_finish` = d_w_pair_bias / d_gamma from
 * those partial sums (same arguments; it reads only packed, d_w_pair_bias, d_gamma and the workspace).  May run on
 * different streams if the caller orders _finish after _main. */
int dab_ipa_bwd_sm100_main(const DabIpaDims* d, const void* packed, const void* e_bf16, const float* R, const float* dcat,
                           void* saved, size_t saved_bytes, void* dproj_bf16, void* de_bf16, float* d_w_pair_bias,
                           float* d_gamma, void* workspace, size_t workspace_bytes, void* stream) {
  return bwd_sm100_impl(d, packed, e_bf16, R, dcat, saved, saved_bytes, dproj_bf16, de_bf16, d_w_pair_bias, d_gamma, workspace,
                        workspace_bytes, stream, false);
}
int dab_ipa_bwd_sm100_finish(const DabIpaDims* d, const void* packed, const void* e_bf16, const float* R, const float* dcat,
                             void* saved, size_t saved_bytes, void* dproj_bf16, void* de_bf16, float* d_w_pair_bias,
                             float* d_gamma, void* workspace, size_t workspace_bytes, void* stream) {
  return bwd_sm100_impl(d, packed, e_bf16, R, dcat, saved, saved_bytes, dproj_bf16, de_bf16, d_w_pair_bias, d_gamma, workspace,
                        workspace_bytes, stream, true);
}

#ifdef DAB_DEBUG_HOOKS
/* Test hook: keep the raw key-side accumulators (dQ, dK, dV of dab_debug_bwd_sm100_buffers) on later calls. */
int dab_debug_bwd_keep_qkv(int on) {
  g_bwd_keep_qkv = on;
  return DAB_OK;
}

/* Profiling hook: per-CTA clock64 timeline of the backward core (64 slots per CTA), NULL to disable. */
int dab_debug_set_bwd_timeline(long long* buf) {
  g_bwd_dbg = buf;
  return DAB_OK;
}

/* Test hook: the intermediate buffers of the last dab_ipa_bwd_sm100_main call on `workspace` (device pointers). */
int dab_debug_bwd_sm100_buffers(const DabIpaDims* d, void* workspace, void** out /* 10 pointers */) {
  DAB_REQUIRE(shape_ok(d) && workspace && out, DAB_EINVAL, "dab_debug_bwd_sm100_buffers: bad argument");
  BwdWs bw = carve_bwd(d->B, workspace);
  out[0] = nullptr; out[1] = bw.dObf; out[2] = nullptr; out[3] = nullptr; out[4] = nullptr;   // 0, 2-4: no longer in HBM
  out[5] = bw.Pn; out[6] = bw.dL; out[7] = bw.dQ; out[8] = bw.dK; out[9] = bw.dV;
  return DAB_OK;
}

#endif

}  // extern "C"
