// The three masked training losses of DiffAb in one pass each way (SURVEY §8f N2; reference diffab_pytorch.py:610-625,
// 856-880):
//   seq  = sum_r m_r sum_k [ xlogy(t_rk, t_rk) - t_rk log p_rk ] / sum_r m_r        (nn.KLDivLoss(reduction="none") on log p)
//   pos  = sum_r m_r sum_c (e_rc - e*_rc)^2 / sum_r m_r                             (nn.MSELoss(reduction="none"))
//   rot  = sum_r m_r || P_r^T T_r - I ||_F^2 / sum_r m_r                            (OrientationLoss)
// with m = generation_mask & residue_mask.  In PyTorch this is ~40 small kernels forward and as many backward on
// (B, L, ...) tensors; here one thread per residue, block-reduced, and the last block to finish divides by the count.
// The backward kernel writes the gradients with respect to the three epsilon-network outputs directly.
#include <math.h>

#include "common.cuh"

namespace dab {

constexpr int LOSS_V = 21;

__device__ __forceinline__ void loss_rot_discrepancy(const float* P, const float* T, float* D) {
#pragma unroll
  for (int j = 0; j < 3; ++j)
#pragma unroll
    for (int k = 0; k < 3; ++k)
      D[j * 3 + k] = P[j] * T[k] + P[3 + j] * T[3 + k] + P[6 + j] * T[6 + k] - (j == k ? 1.f : 0.f);   // (P^T T - I)_jk
}

// acc: [0..2] masked sums, [3] mask count, [4] (as unsigned) finished-block ticket; zeroed by the caller
__global__ void __launch_bounds__(128) losses_fwd_kernel(const float* __restrict__ post_pred, const float* __restrict__ post_tgt,
                                                         const float* __restrict__ eps_pred, const float* __restrict__ eps_tgt,
                                                         const float* __restrict__ O_pred, const float* __restrict__ O_true,
                                                         const uint8_t* __restrict__ mask, int64_t n, int generate,
                                                         float* __restrict__ acc, float* __restrict__ out) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (r < n && mask[r]) {
    if (generate & DAB_GEN_SEQUENCE) {
      float s = 0.f;
      for (int k = 0; k < LOSS_V; ++k) {
        const float t = post_tgt[r * LOSS_V + k], p = post_pred[r * LOSS_V + k];
        s += (t > 0.f ? t * logf(t) : 0.f) - t * logf(p);          // xlogy(t, t) - t * log p
      }
      v[0] = s;
    }
    if (generate & DAB_GEN_STRUCTURE) {
      float q = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float d = eps_pred[r * 3 + c] - eps_tgt[r * 3 + c];
        q = fmaf(d, d, q);
      }
      v[1] = q;
      float P[9], T[9], D[9];
#pragma unroll
      for (int c = 0; c < 9; ++c) { P[c] = O_pred[r * 9 + c]; T[c] = O_true[r * 9 + c]; }
      loss_rot_discrepancy(P, T, D);
      float w = 0.f;
#pragma unroll
      for (int c = 0; c < 9; ++c) w = fmaf(D[c], D[c], w);
      v[2] = w;
    }
    v[3] = 1.f;     // the count is the same in every mode
  }
  __shared__ float s_red[4][4];
  __shared__ bool s_last;
#pragma unroll
  for (int c = 0; c < 4; ++c) v[c] = warp_sum(v[c]);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0)
    for (int c = 0; c < 4; ++c) s_red[warp][c] = v[c];
  __syncthreads();
  if (threadIdx.x < 4) {
    const float t = s_red[0][threadIdx.x] + s_red[1][threadIdx.x] + s_red[2][threadIdx.x] + s_red[3][threadIdx.x];
    if (t != 0.f) atomicAdd(acc + threadIdx.x, t);
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = atomicAdd(reinterpret_cast<unsigned*>(acc + 4), 1u) == gridDim.x - 1;
  __syncthreads();
  if (s_last && threadIdx.x < 4) {
    __threadfence();
    const float cnt = atomicAdd(acc + 3, 0.f);
    out[threadIdx.x] = threadIdx.x < 3 ? atomicAdd(acc + threadIdx.x, 0.f) / cnt : cnt;     // 0 / 0 = nan, as the reference
  }
}

// g[3]: upstream gradients of the three losses; cnt = out[3] of the forward pass
__global__ void __launch_bounds__(128) losses_bwd_kernel(const float* __restrict__ post_pred, const float* __restrict__ post_tgt,
                                                         const float* __restrict__ eps_pred, const float* __restrict__ eps_tgt,
                                                         const float* __restrict__ O_pred, const float* __restrict__ O_true,
                                                         const uint8_t* __restrict__ mask, int64_t n, int generate,
                                                         const float* __restrict__ g, const float* __restrict__ fwd_out,
                                                         float* __restrict__ d_post, float* __restrict__ d_eps,
                                                         float* __restrict__ d_O) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  const bool m = mask[r];
  const bool ms = m && (generate & DAB_GEN_SEQUENCE), mx = m && (generate & DAB_GEN_STRUCTURE);   // launch-uniform bits
  const float inv = m ? 1.f / fwd_out[3] : 0.f;
  const float gs = g[0] * inv, gp = g[1] * inv, gr = g[2] * inv;
  for (int k = 0; k < LOSS_V; ++k)
    d_post[r * LOSS_V + k] = ms ? -gs * post_tgt[r * LOSS_V + k] / post_pred[r * LOSS_V + k] : 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) d_eps[r * 3 + c] = mx ? 2.f * gp * (eps_pred[r * 3 + c] - eps_tgt[r * 3 + c]) : 0.f;
  float P[9], T[9], D[9];
#pragma unroll
  for (int c = 0; c < 9; ++c) { P[c] = O_pred[r * 9 + c]; T[c] = O_true[r * 9 + c]; }
  loss_rot_discrepancy(P, T, D);
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j)       // d/dP_ij sum D^2 = 2 sum_k D_jk T_ik
      d_O[r * 9 + i * 3 + j] = mx ? 2.f * gr * (D[j * 3] * T[i * 3] + D[j * 3 + 1] * T[i * 3 + 1] + D[j * 3 + 2] * T[i * 3 + 2]) : 0.f;
}

// Adam on one flat fp32 parameter vector (torch.optim.Adam with capturable=True, diffab_pytorch.py:925-931 of the
// reference's configure_optimizers): step count on the device (already incremented by the caller), L2 weight decay added
// to the gradient, bias-corrected first / second moments.  HBM-bound: 16 B read + 12 B written per element, float4 per thread.
__global__ void __launch_bounds__(256) adam_flat_kernel(float4* __restrict__ p, const float4* __restrict__ g, float4* __restrict__ m,
                                                        float4* __restrict__ v, const float* __restrict__ step, float lr, float b1,
                                                        float b2, float eps, float wd, int64_t n4) {
  const float t = __ldg(step);
  const float bc1 = 1.0f - powf(b1, t), bc2 = 1.0f - powf(b2, t);
  const float step_size = lr / bc1, inv_sqrt_bc2 = rsqrtf(bc2);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 pp = p[i], gg = g[i], mm = m[i], vv = v[i];
    float* pa = &pp.x; float* ga = &gg.x; float* ma = &mm.x; float* va = &vv.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gk = ga[k] + wd * pa[k];
      ma[k] = b1 * ma[k] + (1.0f - b1) * gk;
      va[k] = b2 * va[k] + (1.0f - b2) * gk * gk;
      pa[k] -= step_size * ma[k] / (sqrtf(va[k]) * inv_sqrt_bc2 + eps);
    }
    p[i] = pp; m[i] = mm; v[i] = vv;
  }
}

}  // namespace dab

using namespace dab;

extern "C" {

/* One Adam step on a flat parameter vector: p, m, v updated in place from the gradient g (n fp32 elements each, n % 4 == 0,
 * 16-byte aligned); `step` = device scalar (float) holding the step count INCLUDING this step (the caller increments it:
 * the call is graph-capturable and has no host state).  torch.optim.Adam semantics (L2 weight decay, bias corrections). */
int dab_adam_flat(float* p, const float* g, float* m, float* v, const float* step, float lr, float beta1, float beta2,
                  float eps, float weight_decay, int64_t n, void* stream) {
  DAB_REQUIRE(p && g && m && v && step, DAB_EINVAL, "dab_adam_flat: null pointer");
  DAB_REQUIRE(n >= 0 && n % 4 == 0 && aligned16(p) && aligned16(g) && aligned16(m) && aligned16(v), DAB_EINVAL,
              "dab_adam_flat: n %% 4 == 0 and 16-byte aligned vectors required");
  if (n == 0) return DAB_OK;
  const int64_t n4 = n / 4;
  int64_t blocks = (n4 + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  adam_flat_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<float4*>(p), reinterpret_cast<const float4*>(g), reinterpret_cast<float4*>(m),
      reinterpret_cast<float4*>(v), step, lr, beta1, beta2, eps, weight_decay, n4);
  count_launch();
  return check_launch("dab_adam_flat");
}

/* out[0..2] = (sequence KL, translation MSE, orientation) losses of DiffAb._shared_step (diffab_pytorch.py:856-880), each the
 * masked sum over the n = B*L residues divided by out[3] = the number of masked residues.  post_*[n,21], eps_*[n,3],
 * O_*[n,3,3] fp32; mask[n] uint8 = generation_mask & residue_mask; acc = 8 zeroed floats of scratch.  `generate` (DAB_GEN_*
 * bits): a term of a modality that is not generated is exactly 0; the count is the same in every mode. */
int dab_losses_fwd(const float* post_pred, const float* post_tgt, const float* eps_pred, const float* eps_tgt, const float* O_pred,
                   const float* O_true, const uint8_t* mask, int64_t n, int generate, float* acc, float* out, void* stream) {
  DAB_REQUIRE(n > 0, DAB_EINVAL, "dab_losses_fwd: n must be positive");
  if (int rc = check_generate(generate, "dab_losses_fwd")) return rc;
  DAB_REQUIRE(post_pred && post_tgt && eps_pred && eps_tgt && O_pred && O_true && mask && acc && out, DAB_EINVAL,
              "dab_losses_fwd: null pointer");
  losses_fwd_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(post_pred, post_tgt, eps_pred, eps_tgt, O_pred,
                                                                                  O_true, mask, n, generate, acc, out);
  count_launch();
  return check_launch("dab_losses_fwd");
}

/* Gradients of g[0]*seq + g[1]*pos + g[2]*rot with respect to the predicted posterior, epsilon and orientation
 * (d_post[n,21], d_eps[n,3], d_O[n,3,3]); fwd_out = the `out` of dab_losses_fwd (for the count). */
int dab_losses_bwd(const float* post_pred, const float* post_tgt, const float* eps_pred, const float* eps_tgt, const float* O_pred,
                   const float* O_true, const uint8_t* mask, int64_t n, int generate, const float* g, const float* fwd_out,
                   float* d_post, float* d_eps, float* d_O, void* stream) {
  DAB_REQUIRE(n > 0, DAB_EINVAL, "dab_losses_bwd: n must be positive");
  if (int rc = check_generate(generate, "dab_losses_bwd")) return rc;
  DAB_REQUIRE(post_pred && post_tgt && eps_pred && eps_tgt && O_pred && O_true && mask && g && fwd_out && d_post && d_eps && d_O,
              DAB_EINVAL, "dab_losses_bwd: null pointer");
  losses_bwd_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(post_pred, post_tgt, eps_pred, eps_tgt, O_pred,
                                                                                  O_true, mask, n, generate, g, fwd_out, d_post, d_eps,
                                                                                  d_O);
  count_launch();
  return check_launch("dab_losses_bwd");
}

}  // extern "C"
