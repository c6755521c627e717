// Fused tail of the epsilon network on sm_100a (SURVEY §8f N1): the three denoising heads of Denoiser.forward
// (diffab_pytorch.py:584-599 of the reference) for D = 128 in ONE kernel:
//
//   h = [x | beta, sin beta, cos beta]                                      (x = output of the IPA module)
//   eps    = W3c relu(W2c relu(W1c h + b1c) + b2c) + b3c        -> (.., 3)   coordinate_denoising
//   rotvec = W3o relu(W2o relu(W1o h + b1o) + b2o) + b3o        -> (.., 3)   orientation_denoising
//   post   = softmax(W3s relu(W2s relu(W1s h + b1s) + b2s) + b3s) -> (.., 21) sequence_denoising
//
// In PyTorch this is nine GEMMs whose fp32 activations ((B L) x 384 floats, 50 MB at B = 256) make several HBM
// round trips per reverse step; here a CTA owns 128 residues (one patch, so beta is a CTA constant and the three
// time columns of the first layers collapse into a per-CTA bias), keeps every activation in TMEM / shared memory
// and reads 64 KB of x and writes 13.8 KB of results:
//   layer 1: [128 x 128] x W1^T [128 x 384]  -> TMEM columns 0..383          (tcgen05.mma, bf16 operands, fp32 acc.)
//   per head: + bias, relu -> bf16 -> smem -> [128 x 128] x W2_k^T -> TMEM (same columns) -> + bias, relu -> bf16
//             -> smem -> [128 x 128] x W3_k^T (padded to 32 outputs) -> TMEM columns 384 + 32 k -> epilogue
#include <cuda_bf16.h>
#include <math.h>

#include "common.cuh"
#include "gemm_sm100.cuh"
#include "sm100_prims.cuh"

namespace dab {
namespace sm100 {

constexpr int HD = 128;          // d_residue_emb
constexpr int HN3 = 32;          // padded width of the last layers
struct HeadsPacked {             // byte offsets inside the packed blob
  // bf16 [864][128]: rows 0..383 first layers (head k at 128 k), 384..767 second layers, 768..863 last layers (32 per head)
  static constexpr size_t kW = 0;
  static constexpr size_t kWt1 = (size_t)864 * HD * 2;        // fp32 [384][3]: time columns of the first layers
  static constexpr size_t kB1 = kWt1 + 384 * 3 * 4;           // fp32 [384]
  static constexpr size_t kB2 = kB1 + 384 * 4;                // fp32 [384]
  static constexpr size_t kB3 = kB2 + 384 * 4;                // fp32 [96]
  static constexpr size_t kTotal = kB3 + 96 * 4;
};

struct HeadsSmem {
  static constexpr int kA = 0;                 // x, then the layer-1 activations of the current head: [2 kb][128][128 B]
  static constexpr int kA2 = 32768;            // layer-2 activations of the current head
  static constexpr int kW = 65536;             // ring of two [2 kb][128 rows][128 B] weight tiles
  static constexpr int kW3 = kW + 2 * 32768;   // three [2 kb][32 rows][128 B] last-layer tiles
  static constexpr int kPb = kW3 + 3 * 8192;   // fp32 [8 slots][384]: b1 + Wt1 . (beta, sin beta, cos beta) per block
  static constexpr int kTile = kPb + 8 * 384 * 4;   // int [8]: the tile of each 16-row slot (live-tile mode)
  static constexpr int kBars = kTile + 8 * 4;
  static constexpr int kTmemSlot = kBars + 32 * 8;
  static constexpr int kTotal = kTmemSlot + 16;
};
enum HBar { HW_FULL = 0 /* 2 */, HW_EMPTY = 2 /* 2 */, HW3_FULL = 4, HL1_DONE = 5, HA1_READY = 6 /* 256 arrivals */,
            HL2_DONE = 7, HA2_READY = 8 /* 256 arrivals */, HL3_DONE = 9,
            // fused to_out of the last IPA layer (y = cat Wout^T + b straight into the A tile): ring of three 32 KB stages
            // [128 rows of cat | 128 rows of Wout] x 64 K columns in kA2 and the (still idle) weight ring
            HG_FULL = 10 /* 3 */, HG_EMPTY = 13 /* 3 */, HG_DONE = 16, HX_READY = 17 /* 256 arrivals */, H_N_BARS = 18 };

__device__ __forceinline__ uint32_t hpk(float a, float b) {
  __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&p);
}

__global__ void pack_heads_kernel(DabHeadWeights w, uint8_t* packed) {
  __nv_bfloat16* wb = reinterpret_cast<__nv_bfloat16*>(packed + HeadsPacked::kW);
  float* wt1 = reinterpret_cast<float*>(packed + HeadsPacked::kWt1);
  float* b1 = reinterpret_cast<float*>(packed + HeadsPacked::kB1);
  float* b2 = reinterpret_cast<float*>(packed + HeadsPacked::kB2);
  float* b3 = reinterpret_cast<float*>(packed + HeadsPacked::kB3);
  const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
  const float* w1[3] = {w.c_w1, w.o_w1, w.s_w1};
  const float* w2[3] = {w.c_w2, w.o_w2, w.s_w2};
  const float* w3[3] = {w.c_w3, w.o_w3, w.s_w3};
  const float* bb1[3] = {w.c_b1, w.o_b1, w.s_b1};
  const float* bb2[3] = {w.c_b2, w.o_b2, w.s_b2};
  const float* bb3[3] = {w.c_b3, w.o_b3, w.s_b3};
  const int n3[3] = {3, 3, DAB_VOCAB};
  for (int k = 0; k < 3; ++k) {
    for (int i = tid; i < HD * HD; i += nth) {
      const int r = i / HD, c = i % HD;
      wb[(size_t)(k * HD + r) * HD + c] = __float2bfloat16_rn(w1[k][r * (HD + 3) + c]);      // (128, 131) row-major
      wb[(size_t)(384 + k * HD + r) * HD + c] = __float2bfloat16_rn(w2[k][i]);
    }
    for (int i = tid; i < HN3 * HD; i += nth) {
      const int r = i / HD;
      wb[(size_t)(768 + k * HN3) * HD + i] = __float2bfloat16_rn(r < n3[k] ? w3[k][i] : 0.f);
    }
    for (int i = tid; i < HD; i += nth) {
      for (int c = 0; c < 3; ++c) wt1[(k * HD + i) * 3 + c] = w1[k][i * (HD + 3) + HD + c];
      b1[k * HD + i] = bb1[k][i];
      b2[k * HD + i] = bb2[k][i];
    }
    for (int i = tid; i < HN3; i += nth) b3[k * HN3 + i] = i < n3[k] ? bb3[k][i] : 0.f;
  }
}

// grid = patches (128 residues each); 288 threads: warps 0-7 = epilogue (thread = residue row x column half),
// warp 8 lane 0 = TMA producer + tcgen05.mma issuer.
// Live-tile mode (fuse_out only; `tiles` = ascending ids of 16-row tiles, global row / 16, `tile_count` = their number):
// CTA b takes tiles 8 b .. 8 b + 7 of the list - still 128 MMA rows, the cat rows arrive as eight 16-row boxes (map_cat
// has a 16-row box then) - and writes only their rows; a short last group repeats its last tile in the unused slots and
// masks their writes, CTAs past the end of the list exit.  Every MMA row depends on its own A row only: the same bits.
__global__ void __launch_bounds__(288, 1)
denoiser_heads_kernel(const __grid_constant__ CUtensorMap map_w128, const __grid_constant__ CUtensorMap map_w32,
                      const float* __restrict__ x, const float* __restrict__ beta, const uint8_t* __restrict__ packed,
                      float* __restrict__ eps, float* __restrict__ rotvec, float* __restrict__ post,
                      const __grid_constant__ CUtensorMap map_cat, const __grid_constant__ CUtensorMap map_wout,
                      const float* __restrict__ b_out, int fuse_out, const int* __restrict__ tiles,
                      const int* __restrict__ tile_count) {
  extern __shared__ __align__(1024) uint8_t smem[];
  using S = HeadsSmem;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::kBars);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + S::kTmemSlot);
  float* s_pb = reinterpret_cast<float*>(smem + S::kPb);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int b = blockIdx.x;
  const int n_live = tiles ? __ldg(tile_count) - 8 * b : 8;    // slots of this CTA that hold a tile of the list
  if (n_live <= 0) return;
  int* s_tile = reinterpret_cast<int*>(smem + S::kTile);
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0) asm volatile("trap;");
  const float* b2 = reinterpret_cast<const float*>(packed + HeadsPacked::kB2);
  const float* b3 = reinterpret_cast<const float*>(packed + HeadsPacked::kB3);

  if (tid == 0) {
    for (int i = 0; i < H_N_BARS; ++i) mbar_init(&bars[i], (i == HA1_READY || i == HA2_READY || i == HX_READY) ? 256u : 1u);
    fence_barrier_init();
  }
  __syncwarp();
  if (warp == 0) tmem_alloc(tmem_slot, 512);
  if (warp < 8) {
    // x tile: fp32 global (coalesced float4) -> bf16, K-major 128B-swizzled A operand (16 rows per warp)
    if (!fuse_out) {
      const float* xb = x + (int64_t)b * 128 * HD;
      const uint32_t kb = lane >> 4, chunk = (lane & 15) >> 1, half = (lane & 1) * 8;
#pragma unroll
      for (int rr = 0; rr < 16; ++rr) {   // all 16 loads of the warp in flight before the first conversion
        const int r = warp * 16 + rr;
        const float4 v = __ldg(reinterpret_cast<const float4*>(xb + r * HD) + lane);
        *reinterpret_cast<uint2*>(smem + S::kA + kb * 16384 + swz128_offset(r, chunk) + half) =
            make_uint2(hpk(v.x, v.y), hpk(v.z, v.w));
      }
    }
    if (tiles && tid < 8) s_tile[tid] = __ldg(tiles + 8 * b + min(tid, n_live - 1));
    fence_proxy_async_smem();
  }
  tcgen05_fence_before_sync();
  __syncthreads();
  tcgen05_fence_after_sync();
  const uint32_t tmem = *tmem_slot;

  if (warp == 8) {
    if (lane == 0) {
      tma_prefetch_desc(&map_w128);
      tma_prefetch_desc(&map_w32);
      if (fuse_out) {
        // ---- to_out of the last IPA layer: acc[128 residues x 128] = cat[128 x 1024] Wout^T, 16 K chunks of 64
        tma_prefetch_desc(&map_cat); tma_prefetch_desc(&map_wout);
        constexpr uint32_t idesc_g = make_idesc_bf16(128, 128, 0, 0);
        const int g_off[3] = {S::kA2, S::kW, S::kW + 32768};
        auto load_g = [&](int kc) {
          const int st = kc % 3;
          mbar_arrive_expect_tx(&bars[HG_FULL + st], 32768);
          if (tiles) {
            for (int sl = 0; sl < 8; ++sl)     // 2 KB boxes: the 128B swizzle repeats every 8 rows, the layout is unchanged
              tma_load_2d(smem + g_off[st] + sl * 2048, &map_cat, &bars[HG_FULL + st], kc * 64, s_tile[sl] * 16);
          } else {
            tma_load_2d(smem + g_off[st], &map_cat, &bars[HG_FULL + st], kc * 64, b * 128);
          }
          tma_load_2d(smem + g_off[st] + 16384, &map_wout, &bars[HG_FULL + st], kc * 64, 0);
        };
        for (int kc = 0; kc < 3; ++kc) load_g(kc);
        constexpr int kChunks = 1024 / 64;
        for (int kc = 0; kc < kChunks; ++kc) {
          const int st = kc % 3;
          mbar_wait(&bars[HG_FULL + st], (kc / 3) & 1);
          tcgen05_fence_after_sync();
          const uint64_t da = make_smem_desc(smem_base + g_off[st], 16, 1024, kSwizzle128B);
          const uint64_t db = make_smem_desc(smem_base + g_off[st] + 16384, 16, 1024, kSwizzle128B);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_bf16(tmem, da + (uint32_t)((kk * 32) >> 4), db + (uint32_t)((kk * 32) >> 4), idesc_g, (kc | kk) != 0);
          umma_commit(&bars[HG_EMPTY + st]);
          if (kc == kChunks - 1) umma_commit(&bars[HG_DONE]);
          if (kc + 3 < kChunks) {
            mbar_wait(&bars[HG_EMPTY + st], (kc / 3) & 1);
            load_g(kc + 3);
          }
        }
        // the heads' weight ring shares the to_out ring's memory: every to_out MMA must have completed
        mbar_wait(&bars[HG_DONE], 0);
      }
      // weight tiles through the ring of two: t = 0..2 first layers, 3..5 second layers (rows 128 t of the blob)
      auto load_w = [&](int tt) {
        const int s = tt & 1;
        uint8_t* dst = smem + S::kW + s * 32768;
        mbar_arrive_expect_tx(&bars[HW_FULL + s], 32768);
        tma_load_2d(dst, &map_w128, &bars[HW_FULL + s], 0, tt * 128);
        tma_load_2d(dst + 16384, &map_w128, &bars[HW_FULL + s], 64, tt * 128);
      };
      load_w(0);
      load_w(1);
      mbar_arrive_expect_tx(&bars[HW3_FULL], 3 * 8192);
      for (int k = 0; k < 3; ++k) {
        tma_load_2d(smem + S::kW3 + k * 8192, &map_w32, &bars[HW3_FULL], 0, 768 + k * HN3);
        tma_load_2d(smem + S::kW3 + k * 8192 + 4096, &map_w32, &bars[HW3_FULL], 64, 768 + k * HN3);
      }
      constexpr uint32_t idesc128 = make_idesc_bf16(128, 128, 0, 0);
      constexpr uint32_t idesc32 = make_idesc_bf16(128, HN3, 0, 0);
      auto mma_tile = [&](uint32_t a_addr, uint32_t w_addr, int n_rows, uint32_t idesc, uint32_t dcol) {
#pragma unroll
        for (int k = 0; k < HD / 16; ++k) {
          uint64_t da = make_smem_desc(a_addr + (k >> 2) * 16384 + (k & 3) * 32, 16, 1024, kSwizzle128B);
          uint64_t db = make_smem_desc(w_addr + (k >> 2) * (n_rows * 128) + (k & 3) * 32, 16, 1024, kSwizzle128B);
          umma_bf16(tmem + dcol, da, db, idesc, k != 0);
        }
      };
      if (fuse_out) {                // the epilogue warps have written y (bf16) into the A tile and left the accumulator
        mbar_wait(&bars[HX_READY], 0);
        tcgen05_fence_after_sync();
      }
      // ---- layer 1 of the three heads
      for (int tt = 0; tt < 3; ++tt) {
        const int s = tt & 1;
        mbar_wait(&bars[HW_FULL + s], (tt >> 1) & 1);
        tcgen05_fence_after_sync();
        mma_tile(smem_base + S::kA, smem_base + S::kW + s * 32768, 128, idesc128, tt * 128);
        umma_commit(&bars[HW_EMPTY + s]);
        if (tt == 2) umma_commit(&bars[HL1_DONE]);
        // refill the slot with tile tt + 2 once these MMAs have read it
        mbar_wait(&bars[HW_EMPTY + s], (tt >> 1) & 1);
        load_w(tt + 2);
      }
      mbar_wait(&bars[HW3_FULL], 0);
      // ---- layers 2 and 3, head by head
      for (int k = 0; k < 3; ++k) {
        const int tt = 3 + k, s = tt & 1;
        mbar_wait(&bars[HA1_READY], k & 1);
        mbar_wait(&bars[HW_FULL + s], (tt >> 1) & 1);
        tcgen05_fence_after_sync();
        mma_tile(smem_base + S::kA, smem_base + S::kW + s * 32768, 128, idesc128, k * 128);
        umma_commit(&bars[HL2_DONE]);
        if (tt + 2 < 6) {
          umma_commit(&bars[HW_EMPTY + s]);
          mbar_wait(&bars[HW_EMPTY + s], (tt >> 1) & 1);
          load_w(tt + 2);
        }
        mbar_wait(&bars[HA2_READY], k & 1);
        tcgen05_fence_after_sync();
        mma_tile(smem_base + S::kA2, smem_base + S::kW3 + k * 8192, HN3, idesc32, 384 + k * HN3);
        umma_commit(&bars[HL3_DONE]);
      }
    }
  } else {
    const int row = tid & 127, chalf = tid >> 7;           // column half = K block of the next layer's A operand
    const uint32_t tmem_lane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int slot = row >> 4;
    const int64_t grow = tiles ? (int64_t)s_tile[slot] * 16 + (row & 15) : (int64_t)b * 128 + row;
    const bool write = slot < n_live;
    const float* pb = s_pb + (tiles ? slot * 384 : 0);
    // bias + relu on 64 accumulator columns -> bf16 -> row `row` of K block `chalf` of an A operand
    auto relu_to_smem = [&](uint32_t col0, const float* bias, bool bias_in_smem, uint8_t* dst) {
#pragma unroll
      for (int part = 0; part < 2; ++part) {
        float v[32];
        tmem_ld_x32(tmem_lane + col0 + part * 32, v);
        tmem_wait_ld();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float o[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int c = part * 32 + q * 8 + e;
            const float bv = bias_in_smem ? bias[c] : __ldg(bias + c);
            o[e] = fmaxf(v[q * 8 + e] + bv, 0.f);
          }
          *reinterpret_cast<uint4*>(dst + chalf * 16384 + swz128_offset(row, part * 4 + q)) =
              make_uint4(hpk(o[0], o[1]), hpk(o[2], o[3]), hpk(o[4], o[5]), hpk(o[6], o[7]));
        }
      }
    };
    {
      // per-block bias of the first layers: the three time columns of [x | beta, sin beta, cos beta]; one vector per
      // 16-row slot in live-tile mode (the slots may come from different blocks)
      const float* wt1 = reinterpret_cast<const float*>(packed + HeadsPacked::kWt1);
      const float* b1 = reinterpret_cast<const float*>(packed + HeadsPacked::kB1);
      for (int sl = 0; sl < (tiles ? 8 : 1); ++sl) {
        const float bt = __ldg(beta + (tiles ? s_tile[sl] >> 3 : b)), sb = sinf(bt), cb = cosf(bt);
        for (int i = tid; i < 384; i += 256)
          s_pb[sl * 384 + i] = __ldg(b1 + i) + __ldg(wt1 + i * 3) * bt + __ldg(wt1 + i * 3 + 1) * sb + __ldg(wt1 + i * 3 + 2) * cb;
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");    // the epilogue warps read each other's entries
    }
    if (fuse_out) {
      // y = acc + b_out of the last IPA layer, rounded to bf16 exactly as the heads would round its fp32 output, goes
      // straight into the A tile: this thread converts its row of K block `chalf`
      mbar_wait(&bars[HG_DONE], 0);
      tcgen05_fence_after_sync();
#pragma unroll
      for (int part = 0; part < 2; ++part) {
        float v[32];
        tmem_ld_x32(tmem_lane + chalf * 64 + part * 32, v);
        tmem_wait_ld();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float* b8 = b_out + chalf * 64 + part * 32 + q * 8;
          *reinterpret_cast<uint4*>(smem + S::kA + chalf * 16384 + swz128_offset(row, part * 4 + q)) =
              make_uint4(hpk(v[q * 8] + __ldg(b8), v[q * 8 + 1] + __ldg(b8 + 1)), hpk(v[q * 8 + 2] + __ldg(b8 + 2), v[q * 8 + 3] + __ldg(b8 + 3)),
                         hpk(v[q * 8 + 4] + __ldg(b8 + 4), v[q * 8 + 5] + __ldg(b8 + 5)), hpk(v[q * 8 + 6] + __ldg(b8 + 6), v[q * 8 + 7] + __ldg(b8 + 7)));
        }
      }
      fence_proxy_async_smem();
      tcgen05_fence_before_sync();
      mbar_arrive(&bars[HX_READY]);
    }
    mbar_wait(&bars[HL1_DONE], 0);
    tcgen05_fence_after_sync();
    for (int k = 0; k < 3; ++k) {
      // layer-1 activations of head k (its A1 buffer is free: the previous head's second layer has completed)
      relu_to_smem(k * 128 + chalf * 64, pb + k * 128 + chalf * 64, true, smem + S::kA);
      fence_proxy_async_smem();
      tcgen05_fence_before_sync();
      mbar_arrive(&bars[HA1_READY]);
      mbar_wait(&bars[HL2_DONE], k & 1);
      tcgen05_fence_after_sync();
      relu_to_smem(k * 128 + chalf * 64, b2 + k * 128 + chalf * 64, false, smem + S::kA2);
      fence_proxy_async_smem();
      tcgen05_fence_before_sync();
      mbar_arrive(&bars[HA2_READY]);
      mbar_wait(&bars[HL3_DONE], k & 1);
      tcgen05_fence_after_sync();
      if (chalf == 0) {
        float v[32];
        tmem_ld_x32(tmem_lane + 384 + k * HN3, v);
        tmem_wait_ld();
        if (write && k < 2) {
          float* dst = (k == 0 ? eps : rotvec) + grow * 3;
#pragma unroll
          for (int c = 0; c < 3; ++c) dst[c] = v[c] + __ldg(b3 + k * HN3 + c);
        } else if (write) {                        // nn.Softmax(dim=-1) over the 21 classes (:599)
          float mx = -INFINITY;
#pragma unroll
          for (int c = 0; c < DAB_VOCAB; ++c) { v[c] += __ldg(b3 + 2 * HN3 + c); mx = fmaxf(mx, v[c]); }
          float sum = 0.f;
#pragma unroll
          for (int c = 0; c < DAB_VOCAB; ++c) { v[c] = __expf(v[c] - mx); sum += v[c]; }
          const float inv = 1.0f / sum;
          float* dst = post + grow * DAB_VOCAB;
#pragma unroll
          for (int c = 0; c < DAB_VOCAB; ++c) dst[c] = v[c] * inv;
        }
      }
    }
  }
  tcgen05_fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_free(tmem, 512);
}

// Front of the epsilon network during sampling (diffab_pytorch.py:572-574): layer 1 of to_res_emb acts on
// [res_ctx | emb(s_t)]; its res_ctx half (+ bias) is the per-run constant c and its embedding half the 25-row table
// t1, so the layer is a = relu(c[row] + t1[s_t[row]]), written as bf16 (the A operand of the second layer's GEMM).
__global__ void __launch_bounds__(256) front_act_kernel(const float4* __restrict__ c, const float4* __restrict__ t1,
                                                        const int64_t* __restrict__ s, int64_t n_rows,
                                                        uint2* __restrict__ a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // one float4 of one row
  if (i >= n_rows * (HD / 4)) return;
  const int64_t row = i / (HD / 4);
  const int q = (int)(i % (HD / 4));
  const float4 cv = __ldg(c + i), tv = __ldg(t1 + (int64_t)__ldg(s + row) * (HD / 4) + q);
  a[i] = make_uint2(hpk(fmaxf(cv.x + tv.x, 0.f), fmaxf(cv.y + tv.y, 0.f)),
                    hpk(fmaxf(cv.z + tv.z, 0.f), fmaxf(cv.w + tv.w, 0.f)));
}

}  // namespace sm100
}  // namespace dab

using namespace dab;
using namespace dab::sm100;

extern "C" {

size_t dab_heads_packed_bytes(void) { return HeadsPacked::kTotal; }

int dab_heads_pack_weights(const DabHeadWeights* w, void* packed, void* stream) {
  DAB_REQUIRE(w && packed, DAB_EINVAL, "dab_heads_pack_weights: null pointer");
  const float* const* p = reinterpret_cast<const float* const*>(w);
  for (int i = 0; i < 18; ++i) DAB_REQUIRE(p[i] != nullptr, DAB_EINVAL, "dab_heads_pack_weights: null weight pointer %d", i);
  DAB_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 1023) == 0, DAB_EINVAL, "dab_heads_pack_weights: packed buffer must be 1024-byte aligned");
  pack_heads_kernel<<<148, 256, 0, (cudaStream_t)stream>>>(*w, reinterpret_cast<uint8_t*>(packed));
  count_launch();
  return check_launch("dab_heads_pack_weights");
}

int dab_heads_fwd_sm100(const void* packed, const float* x, const float* beta, int n_patches, int L_, float* eps,
                        float* rotvec, float* post, void* stream) {
  DAB_REQUIRE(L_ == 128, DAB_EUNSUPPORTED, "dab_heads_fwd_sm100: the fused heads kernel needs L = 128 (one patch per CTA)");
  DAB_REQUIRE(n_patches >= 0, DAB_EINVAL, "dab_heads_fwd_sm100: negative batch");
  if (n_patches == 0) return DAB_OK;
  DAB_REQUIRE(packed && x && beta && eps && rotvec && post, DAB_EINVAL, "dab_heads_fwd_sm100: null pointer");
  DAB_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 1023) == 0 && aligned16(x), DAB_EINVAL,
              "dab_heads_fwd_sm100: misaligned pointer (packed 1024 B, x 16 B)");
  CUtensorMap m128, m32;
  uint64_t dims[2] = {(uint64_t)HD, 864}, strides[1] = {(uint64_t)HD * 2};
  uint32_t b128[2] = {64, 128}, b32[2] = {64, HN3};
  const uint8_t* pk = reinterpret_cast<const uint8_t*>(packed);
  if (int rc = make_tensor_map_bf16(&m128, pk + HeadsPacked::kW, 2, dims, strides, b128, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  if (int rc = make_tensor_map_bf16(&m32, pk + HeadsPacked::kW, 2, dims, strides, b32, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  DAB_ENSURE_SMEM(denoiser_heads_kernel, HeadsSmem::kTotal);
  denoiser_heads_kernel<<<n_patches, 288, HeadsSmem::kTotal, (cudaStream_t)stream>>>(m128, m32, x, beta, pk, eps, rotvec, post,
                                                                                      m128, m128, nullptr, 0, nullptr, nullptr);
  count_launch();
  return check_launch("dab_heads_fwd_sm100");
}

/* The same heads with the LAST IPA layer's to_out (diffab_pytorch.py:464: y = cat Wout^T + b) fused in front: cat_bf16
 * [n_patches*128, 1024] = the concat features the layer's attention core left in its workspace, wout_bf16 [128][1024] and
 * b_out [128] from the layer's packed weights (dab_ipa_packed_layout).  The stack's output never exists in HBM; the same bits
 * as dab_ipa_fwd_sm100_stages(.., 4) followed by dab_heads_fwd_sm100.  With tiles / n_tiles (device memory: ascending ids
 * of 16-row tiles, global row / 16, and their number) only the rows of those tiles are computed and written. */
int dab_out_heads_fwd_sm100(const void* packed, const void* cat_bf16, const void* wout_bf16, const float* b_out, const float* beta,
                            int n_patches, int L_, float* eps, float* rotvec, float* post, const int* tiles,
                            const int* n_tiles, void* stream) {
  DAB_REQUIRE(L_ == 128, DAB_EUNSUPPORTED, "dab_out_heads_fwd_sm100: the fused heads kernel needs L = 128 (one block per CTA)");
  DAB_REQUIRE(n_patches >= 0, DAB_EINVAL, "dab_out_heads_fwd_sm100: negative batch");
  if (n_patches == 0) return DAB_OK;
  DAB_REQUIRE(packed && cat_bf16 && wout_bf16 && b_out && beta && eps && rotvec && post && (tiles == nullptr) == (n_tiles == nullptr),
              DAB_EINVAL, "dab_out_heads_fwd_sm100: null pointer (tiles and n_tiles: both or neither)");
  DAB_REQUIRE((reinterpret_cast<uintptr_t>(packed) & 1023) == 0 && aligned16(cat_bf16) && aligned16(wout_bf16), DAB_EINVAL,
              "dab_out_heads_fwd_sm100: misaligned pointer (packed 1024 B, cat / Wout 16 B)");
  CUtensorMap m128, m32, mcat, mwout;
  uint64_t dims[2] = {(uint64_t)HD, 864}, strides[1] = {(uint64_t)HD * 2};
  uint32_t b128[2] = {64, 128}, b32[2] = {64, HN3};
  const uint8_t* pk = reinterpret_cast<const uint8_t*>(packed);
  if (int rc = make_tensor_map_bf16(&m128, pk + HeadsPacked::kW, 2, dims, strides, b128, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  if (int rc = make_tensor_map_bf16(&m32, pk + HeadsPacked::kW, 2, dims, strides, b32, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  uint64_t dc[2] = {1024, (uint64_t)n_patches * 128}, dwo[2] = {1024, (uint64_t)HD}, sc[1] = {1024 * 2};
  uint32_t b16[2] = {64, 16};        // live tiles: one box per 16-row tile
  if (int rc = make_tensor_map_bf16(&mcat, cat_bf16, 2, dc, sc, tiles ? b16 : b128, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  if (int rc = make_tensor_map_bf16(&mwout, wout_bf16, 2, dwo, sc, b128, CU_TENSOR_MAP_SWIZZLE_128B)) return rc;
  DAB_ENSURE_SMEM(denoiser_heads_kernel, HeadsSmem::kTotal);
  denoiser_heads_kernel<<<n_patches, 288, HeadsSmem::kTotal, (cudaStream_t)stream>>>(m128, m32, nullptr, beta, pk, eps, rotvec, post,
                                                                                      mcat, mwout, b_out, 1, tiles, n_tiles);
  count_launch();
  return check_launch("dab_out_heads_fwd_sm100");
}

/* x0[n_rows,128] = relu(c[row] + t1[seq[row]]) . w2^T + b2  (to_res_emb during sampling; n_rows % 128 == 0).
 * w2_bf16: to_res_emb.2.weight as bf16 [128][128]; a_scratch: n_rows * 128 bf16.  Exactly one of x0 (fp32) and x0_bf16
 * (rounded to bf16: the form the first IPA layer's projections consume) is given. */
int dab_front_fwd_sm100(const float* c, const float* t1, const int64_t* seq, int64_t n_rows, const void* w2_bf16,
                        const float* b2, void* a_scratch, float* x0, void* x0_bf16, void* stream) {
  DAB_REQUIRE(n_rows >= 0 && n_rows % 128 == 0, DAB_EUNSUPPORTED, "dab_front_fwd_sm100: n_rows must be a multiple of 128");
  if (n_rows == 0) return DAB_OK;
  DAB_REQUIRE(c && t1 && seq && w2_bf16 && b2 && a_scratch && ((x0 == nullptr) != (x0_bf16 == nullptr)), DAB_EINVAL,
              "dab_front_fwd_sm100: null pointer (exactly one of x0 / x0_bf16 must be given)");
  DAB_REQUIRE(aligned16(c) && aligned16(t1) && aligned16(w2_bf16) && aligned16(a_scratch) && aligned16(x0) && aligned16(x0_bf16),
              DAB_EINVAL, "dab_front_fwd_sm100: pointers must be 16-byte aligned");
  const int64_t n4 = n_rows * (HD / 4);
  front_act_kernel<<<(unsigned)((n4 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(c), reinterpret_cast<const float4*>(t1), seq, n_rows,
      reinterpret_cast<uint2*>(a_scratch));
  count_launch();
  if (int rc = launch_gemm_bf16<128>(a_scratch, HD, w2_bf16, HD, x0, HD, b2, (int)n_rows, HD, HD, (cudaStream_t)stream, x0_bf16))
    return rc;
  return check_launch("dab_front_fwd_sm100");
}

}  // extern "C"
