// Forward noising and reverse step of the three diffusers, fused per residue (sm_100a).
//
// Replaces /root/reference/diffab_pytorch/diffusion.py:38-294 and DiffAb._add_noise
// (diffab_pytorch.py:778-806).  HBM-bound, ~0.3 KB per residue: one thread per residue; every
// residue's frames/coordinates/sequence move through HBM exactly once per call.  Integer outputs
// are bit-exact against the reference given the same injected noise: the probability expressions
// use explicit round-to-nearest intrinsics so nvcc cannot contract them into FMAs.
#include "common.cuh"
#include "step_device.cuh"

namespace dab {

__device__ __forceinline__ float kUniform() { return __fdiv_rn(1.0f, 21.0f); }  // fl32(1/21), diffusion.py:71

// p_k = fl(fl(w_keep * onehot_k) + fl(w_noise * u));  diffusion.py:38-41,74-79 (mask off -> one-hot)
__device__ __forceinline__ float mix_prob(bool hot, float w_keep, float w_noise, bool generated) {
  float oh = hot ? 1.0f : 0.0f;
  if (!generated) return oh;
  return __fadd_rn(__fmul_rn(w_keep, oh), __fmul_rn(w_noise, kUniform()));
}

// One thread per residue, 128 residues per block.  Every per-residue record (21 exponential draws, 21 posterior
// probabilities, 9 + 9 rotation entries, 3 + 3 + 3 coordinates) is a short odd-strided row, so a thread-per-row
// global access pattern wastes most of each sector; the block's records are contiguous, so they go through shared
// memory with fully coalesced global traffic (odd row strides: conflict-free shared-memory access).
__global__ void __launch_bounds__(128) forward_noise_kernel(
    Sched sc, const int64_t* __restrict__ seq0, const float* __restrict__ x0, const float* __restrict__ O0,
    const uint8_t* __restrict__ mask, const int64_t* __restrict__ t, int B, int L,
    const float* __restrict__ seq_exp, const float* __restrict__ eps, const float* __restrict__ rotvec, int generate,
    int64_t* __restrict__ seq_t, float* __restrict__ posterior, float* __restrict__ x_t, float* __restrict__ O_t) {
  __shared__ float s_v[128 * DAB_VOCAB];   // exponential draws in, posterior out
  __shared__ float s_o[128 * 9];           // O_0 in, O_t out
  __shared__ float s_x[128 * 3], s_e[128 * 3], s_r[128 * 3];
  const int64_t n = (int64_t)B * L;
  const int64_t r0 = (int64_t)blockIdx.x * 128;
  const int nv = (int)min((int64_t)128, n - r0);
  const int tid = threadIdx.x;
  for (int i = tid; i < nv * DAB_VOCAB; i += 128) s_v[i] = __ldg(seq_exp + r0 * DAB_VOCAB + i);
  for (int i = tid; i < nv * 9; i += 128) s_o[i] = __ldg(O0 + r0 * 9 + i);
  for (int i = tid; i < nv * 3; i += 128) {
    s_x[i] = __ldg(x0 + r0 * 3 + i);
    s_e[i] = __ldg(eps + r0 * 3 + i);
    s_r[i] = __ldg(rotvec + r0 * 3 + i);
  }
  __syncthreads();
  const int64_t r = r0 + tid;
  if (tid < nv) {
    int b = (int)(r / L);
    int tt = (int)t[b];
  if (tt < 0 || tt > sc.T) asm volatile("trap;");   // out-of-range timestep: the reference raises IndexError
    bool gen = mask[r] != 0;
    bool gen_seq = gen && (generate & DAB_GEN_SEQUENCE), gen_str = gen && (generate & DAB_GEN_STRUCTURE);
    int s0 = (int)seq0[r];

    // ---- sequence: s_t ~ Multinomial(abar_t onehot + (1-abar_t)/21)   diffusion.py:105-158
    float ab = __ldg(sc.alpha_bar + tt);
    float one_m_ab = __fsub_rn(1.0f, ab);
    int st = argmax_ratio([&](int k) { return mix_prob(k == s0, ab, one_m_ab, gen_seq); }, s_v + tid * DAB_VOCAB);
    seq_t[r] = st;
    // ---- posterior q(s_{t-1} | s_t, s_0) ∝ p_single(s_t, t) * p_from_t0(s_0, t-1)   diffusion.py:168-192
    float beta = __ldg(sc.beta + tt);
    float one_m_beta = __fsub_rn(1.0f, beta);
    int tm1 = tt - 1;
    if (tm1 < 0) tm1 += sc.T + 1;  // python negative index wrap (reference is never called with t = 0)
    float abm = __ldg(sc.alpha_bar + tm1);
    float one_m_abm = __fsub_rn(1.0f, abm);
    float p[DAB_VOCAB];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < DAB_VOCAB; ++k) {
      p[k] = __fmul_rn(mix_prob(k == st, one_m_beta, beta, gen_seq), mix_prob(k == s0, abm, one_m_abm, gen_seq));
      sum = __fadd_rn(sum, p[k]);
    }
#pragma unroll
    for (int k = 0; k < DAB_VOCAB; ++k) s_v[tid * DAB_VOCAB + k] = __fdiv_rn(p[k], sum);   // own row: draws consumed

    // ---- positions: x_t = sqrt(abar) x_0 + sqrt(1-abar) eps   diffusion.py:219-231
    float a = __ldg(sc.alpha_bar_sqrt + tt), s = __ldg(sc.one_minus_alpha_bar_sqrt + tt);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float v0 = s_x[tid * 3 + c];
      float v = __fadd_rn(__fmul_rn(a, v0), __fmul_rn(s, s_e[tid * 3 + c]));
      s_x[tid * 3 + c] = gen_str ? v : v0;
    }
    // ---- orientations: O_t = scale_rot(O_0, sqrt(abar)) @ exp(rotvec)   diffusion.py:280-292
    if (gen_str) {
      float R0[9], Rm[9], Rn[9], Ro[9];
#pragma unroll
      for (int c = 0; c < 9; ++c) R0[c] = s_o[tid * 9 + c];
      float lx, ly, lz;
      so3_log(R0, lx, ly, lz);
      so3_exp(a * lx, a * ly, a * lz, Rm);
      so3_exp(s_r[tid * 3], s_r[tid * 3 + 1], s_r[tid * 3 + 2], Rn);
      mat3_mul(Rm, Rn, Ro);
#pragma unroll
      for (int c = 0; c < 9; ++c) s_o[tid * 9 + c] = Ro[c];
    }
  }
  __syncthreads();
  for (int i = tid; i < nv * DAB_VOCAB; i += 128) posterior[r0 * DAB_VOCAB + i] = s_v[i];
  for (int i = tid; i < nv * 9; i += 128) O_t[r0 * 9 + i] = s_o[i];
  for (int i = tid; i < nv * 3; i += 128) x_t[r0 * 3 + i] = s_x[i];
}

__global__ void __launch_bounds__(128) seq_probs_kernel(Sched sc, int kind, const int64_t* __restrict__ seq,
                                                        const int64_t* __restrict__ seq0,
                                                        const uint8_t* __restrict__ mask,
                                                        const int64_t* __restrict__ t, int B, int L,
                                                        float* __restrict__ out) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= (int64_t)B * L) return;
  int b = (int)(r / L);
  int tt = (int)t[b];
  if (tt < 0 || tt > sc.T) asm volatile("trap;");   // out-of-range timestep: the reference raises IndexError
  bool gen = mask[r] != 0;
  int s = (int)seq[r];
  if (kind == 0) {  // forward_prob_single_step
    float beta = __ldg(sc.beta + tt);
    for (int k = 0; k < DAB_VOCAB; ++k) out[r * DAB_VOCAB + k] = mix_prob(k == s, __fsub_rn(1.0f, beta), beta, gen);
  } else if (kind == 1) {  // forward_prob_from_t0
    float ab = __ldg(sc.alpha_bar + tt);
    for (int k = 0; k < DAB_VOCAB; ++k) out[r * DAB_VOCAB + k] = mix_prob(k == s, ab, __fsub_rn(1.0f, ab), gen);
  } else {  // posterior_single_step
    int s0 = (int)seq0[r];
    float beta = __ldg(sc.beta + tt);
    int tm1 = tt - 1;
    if (tm1 < 0) tm1 += sc.T + 1;
    float abm = __ldg(sc.alpha_bar + tm1);
    float p[DAB_VOCAB];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < DAB_VOCAB; ++k) {
      p[k] = __fmul_rn(mix_prob(k == s, __fsub_rn(1.0f, beta), beta, gen),
                       mix_prob(k == s0, abm, __fsub_rn(1.0f, abm), gen));
      sum = __fadd_rn(sum, p[k]);
    }
#pragma unroll
    for (int k = 0; k < DAB_VOCAB; ++k) out[r * DAB_VOCAB + k] = __fdiv_rn(p[k], sum);
  }
}

// Reverse step (stand-alone form; the sampling loop runs it fused with the IGSO(3) draw, so3_kernels.cu).
__global__ void __launch_bounds__(128) reverse_step_kernel(
    Sched sc, const int64_t* seq_t, const float* x_t, const float* O_t,  // may alias the outputs (in-place)
    const float* __restrict__ eps_theta, const float* __restrict__ v_theta, const float* __restrict__ seq_post,
    const uint8_t* __restrict__ mask, const int64_t* __restrict__ t, int B, int L,
    const float* __restrict__ seq_exp, const float* __restrict__ z, const float* __restrict__ rotvec,
    const float* __restrict__ seq_weight, int generate, int64_t* seq_out, float* x_out, float* O_out, float* O0_out) {
  int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= (int64_t)B * L) return;
  reverse_update_residue(sc, r, (int)t[r / L], seq_t, x_t, O_t, eps_theta, v_theta, seq_post, mask, seq_exp, z, rotvec + r * 3,
                         seq_weight, generate, seq_out, x_out, O_out, O0_out);
}

static int check_sched(const DabSchedule* s, Sched& out, const char* name) {
  DAB_REQUIRE(s && s->alpha && s->alpha_bar && s->alpha_bar_sqrt && s->one_minus_alpha_bar_sqrt && s->beta && s->T > 0,
              DAB_EINVAL, "%s: incomplete schedule", name);
  out = Sched{s->T, s->alpha, s->alpha_bar, s->alpha_bar_sqrt, s->one_minus_alpha_bar_sqrt, s->beta};
  return DAB_OK;
}

// dab_reverse_step and dab_reverse_step_weighted (seq_weight may be NULL: the unweighted draw)
static int reverse_step_launch(const char* name, const DabSchedule* sched, const int64_t* seq_t, const float* x_t,
                               const float* O_t, const float* eps_theta, const float* v_theta, const float* seq_post,
                               const uint8_t* mask, const int64_t* t, int B, int L, const float* seq_exp,
                               const float* z, const float* rotvec, const float* seq_weight, int generate,
                               int64_t* seq_out, float* x_out, float* O_out, float* O0_out, void* stream) {
  Sched sc;
  if (int rc = check_sched(sched, sc, name)) return rc;
  if (int rc = check_generate(generate, name)) return rc;
  DAB_REQUIRE(B >= 0 && L >= 0, DAB_EINVAL, "%s: negative size", name);
  if ((int64_t)B * L == 0) return DAB_OK;
  DAB_REQUIRE(seq_t && x_t && O_t && eps_theta && v_theta && seq_post && mask && t && seq_exp && z && rotvec &&
                  seq_out && x_out && O_out,
              DAB_EINVAL, "%s: null pointer", name);
  int64_t n = (int64_t)B * L;
  reverse_step_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      sc, seq_t, x_t, O_t, eps_theta, v_theta, seq_post, mask, t, B, L, seq_exp, z, rotvec, seq_weight, generate,
      seq_out, x_out, O_out, O0_out);
  count_launch();
  return check_launch(name);
}

}  // namespace dab

using namespace dab;

extern "C" {

int dab_forward_noise(const DabSchedule* sched, const int64_t* seq0, const float* x0, const float* O0,
                      const uint8_t* mask, const int64_t* t, int B, int L, const float* seq_exp, const float* eps,
                      const float* rotvec, int generate, int64_t* seq_t, float* posterior, float* x_t, float* O_t,
                      void* stream) {
  Sched sc;
  if (int rc = check_sched(sched, sc, "dab_forward_noise")) return rc;
  if (int rc = check_generate(generate, "dab_forward_noise")) return rc;
  DAB_REQUIRE(B >= 0 && L >= 0, DAB_EINVAL, "dab_forward_noise: negative size");
  if ((int64_t)B * L == 0) return DAB_OK;
  DAB_REQUIRE(seq0 && x0 && O0 && mask && t && seq_exp && eps && rotvec && seq_t && posterior && x_t && O_t,
              DAB_EINVAL, "dab_forward_noise: null pointer");
  int64_t n = (int64_t)B * L;
  forward_noise_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(
      sc, seq0, x0, O0, mask, t, B, L, seq_exp, eps, rotvec, generate, seq_t, posterior, x_t, O_t);
  count_launch();
  return check_launch("dab_forward_noise");
}

int dab_seq_probs(const DabSchedule* sched, int kind, const int64_t* seq, const int64_t* seq0, const uint8_t* mask,
                  const int64_t* t, int B, int L, float* out, void* stream) {
  Sched sc;
  if (int rc = check_sched(sched, sc, "dab_seq_probs")) return rc;
  DAB_REQUIRE(kind >= 0 && kind <= 2, DAB_EINVAL, "dab_seq_probs: kind must be 0, 1 or 2");
  DAB_REQUIRE(B >= 0 && L >= 0, DAB_EINVAL, "dab_seq_probs: negative size");
  if ((int64_t)B * L == 0) return DAB_OK;
  DAB_REQUIRE(seq && mask && t && out && (kind != 2 || seq0), DAB_EINVAL, "dab_seq_probs: null pointer");
  int64_t n = (int64_t)B * L;
  seq_probs_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(sc, kind, seq, seq0, mask, t, B, L, out);
  count_launch();
  return check_launch("dab_seq_probs");
}

int dab_reverse_step(const DabSchedule* sched, const int64_t* seq_t, const float* x_t, const float* O_t,
                     const float* eps_theta, const float* v_theta, const float* seq_post, const uint8_t* mask,
                     const int64_t* t, int B, int L, const float* seq_exp, const float* z, const float* rotvec,
                     int generate, int64_t* seq_out, float* x_out, float* O_out, float* O0_out, void* stream) {
  return reverse_step_launch("dab_reverse_step", sched, seq_t, x_t, O_t, eps_theta, v_theta, seq_post, mask, t, B, L,
                             seq_exp, z, rotvec, nullptr, generate, seq_out, x_out, O_out, O0_out, stream);
}

int dab_reverse_step_weighted(const DabSchedule* sched, const int64_t* seq_t, const float* x_t, const float* O_t,
                              const float* eps_theta, const float* v_theta, const float* seq_post, const uint8_t* mask,
                              const int64_t* t, int B, int L, const float* seq_exp, const float* z, const float* rotvec,
                              const float* seq_weight, int generate, int64_t* seq_out, float* x_out, float* O_out,
                              float* O0_out, void* stream) {
  return reverse_step_launch("dab_reverse_step_weighted", sched, seq_t, x_t, O_t, eps_theta, v_theta, seq_post, mask, t,
                             B, L, seq_exp, z, rotvec, seq_weight, generate, seq_out, x_out, O_out, O0_out, stream);
}

}  // extern "C"
