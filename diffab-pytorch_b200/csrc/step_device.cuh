// Device-side pieces of the diffusion kernels (diffusion_kernels.cu): the schedule view, the categorical draw and the
// per-residue reverse update.
#pragma once
#include "common.cuh"

namespace dab {

struct Sched {
  int T;
  const float *alpha, *alpha_bar, *alpha_bar_sqrt, *one_minus_alpha_bar_sqrt, *beta;
};

// argmax_k p_k / q_k with first-index tie-break == torch.multinomial(p, 1) given its Exp(1) draw q
template <typename F>
__device__ __forceinline__ int argmax_ratio(F prob, const float* __restrict__ q) {
  int best = 0;
  float best_key = -1.0f;
#pragma unroll
  for (int k = 0; k < DAB_VOCAB; ++k) {
    float key = __fdiv_rn(prob(k), q[k]);   // q may live in shared memory: plain (generic) load
    if (key > best_key) { best_key = key; best = k; }
  }
  return best;
}

// The draw of argmax_ratio under per-type weights w (DiffAb.sample's aa_bias, w = exp(b - max b)): only types with
// w_k > 0 are eligible, key_k = fl(fl(p_k * w_k) / q_k), first eligible index wins ties.  If every eligible key is 0 (the
// posterior mass on the allowed types underflowed) the draw is redone from the weights alone, key_k = w_k / q_k with
// the same q, so a forbidden type is never drawn.  No eligible type: returns `fallback` (the residue keeps its type).
__device__ __forceinline__ int64_t argmax_ratio_weighted(const float* __restrict__ p, const float* __restrict__ w,
                                                         const float* __restrict__ q, int64_t fallback) {
  int best = -1;
  float best_key = -1.0f;
#pragma unroll
  for (int k = 0; k < DAB_VOCAB; ++k) {
    float wk = __ldg(w + k);
    if (wk > 0.f) {
      float key = __fdiv_rn(__fmul_rn(__ldg(p + k), wk), q[k]);
      if (key > best_key) { best_key = key; best = k; }
    }
  }
  if (best < 0) return fallback;
  if (best_key == 0.f) {
    best_key = -1.0f;
#pragma unroll
    for (int k = 0; k < DAB_VOCAB; ++k) {
      float wk = __ldg(w + k);
      if (wk > 0.f) {
        float key = __fdiv_rn(wk, q[k]);
        if (key > best_key) { best_key = key; best = k; }
      }
    }
  }
  return best;
}

// Reverse step of residue r (patch b, timestep tt = t[b]); composition fixed by oracle/sampler.py (the reference has none).
// `rv` = the residue's IGSO(3) rotation-vector draw (global or shared memory).  seq_t / x_t / O_t may alias the outputs.
// `generate`: DAB_GEN_* bits.  `seq_weight` [B*L, 21] (may be NULL, uniform over the launch): the sequence is drawn by
// argmax_ratio_weighted; its rows are read only where the sequence is generated, like seq_post.
__device__ __forceinline__ void reverse_update_residue(
    const Sched& sc, int64_t r, int tt, const int64_t* seq_t, const float* x_t, const float* O_t,
    const float* __restrict__ eps_theta, const float* __restrict__ v_theta, const float* __restrict__ seq_post,
    const uint8_t* __restrict__ mask, const float* __restrict__ seq_exp, const float* __restrict__ z, const float* rv,
    const float* __restrict__ seq_weight, int generate, int64_t* seq_out, float* x_out, float* O_out, float* O0_out) {
  if (tt < 0 || tt > sc.T) asm volatile("trap;");   // out-of-range timestep: the reference raises IndexError
  bool gen = mask[r] != 0;
  // a modality the run does not generate keeps its old value (`generate` is uniform over the launch)
  bool gen_seq = gen && (generate & DAB_GEN_SEQUENCE), gen_str = gen && (generate & DAB_GEN_STRUCTURE);
  bool noisy = tt > 1;

  // sequence
  int64_t s_old = seq_t[r];
  if (gen_seq) {
    const float* p = seq_post + r * DAB_VOCAB;
    if (seq_weight)
      seq_out[r] = argmax_ratio_weighted(p, seq_weight + r * DAB_VOCAB, seq_exp + r * DAB_VOCAB, s_old);
    else
      seq_out[r] = argmax_ratio([&](int k) { return __ldg(p + k); }, seq_exp + r * DAB_VOCAB);
  } else {
    seq_out[r] = s_old;
  }
  // The network outputs are read only where they are used: sampling computes them for the tiles of generated residues
  // only (DiffAb.sample_from_context), the rows of the other tiles are undefined.
  // positions: (x_t - beta/sqrt(1-abar) eps_theta) * (1/sqrt(alpha)) + sqrt(beta) z
  if (gen_str) {
    float beta = __ldg(sc.beta + tt);
    float c_eps = __fdiv_rn(beta, __ldg(sc.one_minus_alpha_bar_sqrt + tt));
    float inv_sa = __fdiv_rn(1.0f, __fsqrt_rn(__ldg(sc.alpha + tt)));
    float sig = noisy ? __fsqrt_rn(beta) : 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c)
      x_out[r * 3 + c] = __fadd_rn(__fmul_rn(__fsub_rn(x_t[r * 3 + c], __fmul_rn(c_eps, __ldg(eps_theta + r * 3 + c))), inv_sa),
                                   __fmul_rn(sig, __ldg(z + r * 3 + c)));
  } else {
#pragma unroll
    for (int c = 0; c < 3; ++c) x_out[r * 3 + c] = x_t[r * 3 + c];
  }
  // orientations: O0 = O_t @ exp(v_theta)  (Denoiser tail, diffab_pytorch.py:594-596); O' = O0 @ exp(rotvec)
  float Rt[9];
#pragma unroll
  for (int c = 0; c < 9; ++c) Rt[c] = O_t[r * 9 + c];
  if (gen_str || O0_out) {
    float Re[9], R0[9];
    so3_exp(__ldg(v_theta + r * 3), __ldg(v_theta + r * 3 + 1), __ldg(v_theta + r * 3 + 2), Re);
    mat3_mul(Rt, Re, R0);
    if (O0_out) {
#pragma unroll
      for (int c = 0; c < 9; ++c) O0_out[r * 9 + c] = R0[c];
    }
    if (gen_str) {
      if (noisy) {
        float Rn[9];
        so3_exp(rv[0], rv[1], rv[2], Rn);
        mat3_mul(R0, Rn, Rt);
      } else {
#pragma unroll
        for (int c = 0; c < 9; ++c) Rt[c] = R0[c];
      }
    }
  }
#pragma unroll
  for (int c = 0; c < 9; ++c) O_out[r * 9 + c] = Rt[c];
}

}  // namespace dab
