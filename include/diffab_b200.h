/* diffab_b200.h - flat C ABI of libdiffab_b200.so (sm_100a only).
 *
 * The reference (dohlee/diffab-pytorch) is pure Python/PyTorch and has no FFI layer; its boundary
 * for the denoising hot path is the Python class `DiffAb` and the free functions of `so3.py` /
 * `diffusion.py`.  Each entry point below replaces the arithmetic of the reference function(s)
 * cited next to it (paths relative to the reference root).  The Python mirror in
 * `diffab-pytorch_b200/` binds these with ctypes; INTEGRATION.md shows the stub a maintainer of the
 * reference would add.
 *
 * Conventions
 *  - Every pointer is a DEVICE pointer owned by the caller; the library never allocates, frees or
 *    retains memory.  Tensors are contiguous in the layouts given; float pointers must be 16-byte
 *    aligned (bf16 pair tensors handed to the TMA path: 128-byte aligned; bf16 outputs written with 256-bit stores -
 *    dproj_bf16 of the backward, the pair tensor of dab_pair_embed_fwd_sm100, xh_bf16 of the pair-MLP forward: 32-byte).
 *  - Every call is asynchronous on `stream` (a cudaStream_t passed as void*), does no host
 *    synchronisation and no allocation, and is CUDA-graph capturable.
 *  - Return value: 0 on success, negative DAB_E* code otherwise; dab_last_error() gives a
 *    thread-local message.  Nothing aborts or throws across the ABI.  There is no CPU fallback.
 *  - RNG never lives inside the library: noise tensors are inputs, drawn by the caller in the
 *    reference's call order (SURVEY 3.1 draws #2-#7), which is what makes integer outputs
 *    bit-exact against the reference.
 */
#ifndef DIFFAB_B200_H
#define DIFFAB_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DAB_OK 0
#define DAB_EINVAL (-1)      /* bad argument (null pointer, negative size, misalignment) */
#define DAB_EUNSUPPORTED (-2) /* shape outside what the kernels support */
#define DAB_ELAUNCH (-3)     /* CUDA launch / runtime error */
#define DAB_EWORKSPACE (-4)  /* workspace too small */

#define DAB_VOCAB 21 /* diffusion.py:47 (hard-coded there) */

int dab_version(void);
const char* dab_last_error(void);
/* Number of kernels this library has launched in this process (bench.py's "gpu_launches" claim). */
long long dab_launch_count(void);

/* ------------------------------------------------------------------ SO(3) maps, so3.py:142-259 */
/* vector_to_rotation_matrix (so3.py:207-237): v[n,3] -> R[n,3,3], Rodrigues, no epsilon guard. */
int dab_so3_exp(const float* v, float* R, int64_t n, void* stream);
/* rotation_matrix_to_vector (so3.py:173-182): R[n,3,3] -> v[n,3]. */
int dab_so3_log(const float* R, float* v, int64_t n, void* stream);
/* log_rotmat (so3.py:146-162): R[n,3,3] -> skew S[n,3,3]. */
int dab_so3_log_skew(const float* R, float* S, int64_t n, void* stream);
/* exp_skew_symmetric_mat (so3.py:219-237): S[n,3,3] -> R[n,3,3]. */
int dab_so3_exp_skew(const float* S, float* R, int64_t n, void* stream);
/* scale_rot (so3.py:240-259): out = exp(k * log R); rotation i uses k[i / group]. */
int dab_so3_scale_rot(const float* R, const float* k, int64_t n, int64_t group, float* out, void* stream);

/* ------------------------------------------------------------------ IGSO(3), so3.py:37-126 */
/* SO3._precompute_histogram/_angular_pdf (so3.py:52-72): out[n_sigma, n_bins], unnormalised. */
int dab_igso3_table(const float* sigma, int n_sigma, int n_bins, int n_terms, float* out, void* stream);
/* SO3.sample_isotropic_gaussian (so3.py:98-126) with its four draws injected:
 *   axis_noise[B,L,3] randn, exp_noise[B,n_bins] Exp(1) (the draw inside torch.multinomial),
 *   jitter[B,L] U[0,1), gauss[B,L] randn.  sigma_idx[B] int64 indexes hist rows / sigmas.
 *   rotvec[B,L,3] out; bins[B,L] int64 out (may be NULL; then the histogram top-L selection is
 *   skipped for rows whose sigma >= threshold, whose result does not depend on it). */
int dab_igso3_sample(const float* hist, const float* sigmas, int n_sigma, int n_bins,
                     const int64_t* sigma_idx, int B, int L, const float* axis_noise,
                     const float* exp_noise, const float* jitter, const float* gauss,
                     float sigma_threshold, float* rotvec, int64_t* bins, void* stream);

/* ------------------------------------------------------------------ diffusion.py */
/* Schedule tables of cosine_variance_schedule (diffusion.py:11-35), each [T+1] floats on device. */
typedef struct DabSchedule {
  int T;
  const float* alpha;
  const float* alpha_bar;
  const float* alpha_bar_sqrt;
  const float* one_minus_alpha_bar_sqrt;
  const float* beta;
} DabSchedule;

/* DiffAb._add_noise (diffab_pytorch.py:778-806) = SequenceDiffuser.diffuse_from_t0 +
 * posterior_single_step (diffusion.py:137-192), CoordinateDiffuser.diffuse_from_t0 (:199-236),
 * OrientationDiffuser.diffuse_from_t0 (:262-294; `rotvec` is dab_igso3_sample's output).
 * mask[B,L] uint8 (bool); t[B] int64; seq_exp[B*L,21] Exp(1); eps[B,L,3] randn.
 * Outputs: seq_t[B,L] int64, posterior[B,L,21], x_t[B,L,3], O_t[B,L,3,3]. */
int dab_forward_noise(const DabSchedule* sched, const int64_t* seq0, const float* x0, const float* O0,
                      const uint8_t* mask, const int64_t* t, int B, int L, const float* seq_exp,
                      const float* eps, const float* rotvec, int64_t* seq_t, float* posterior,
                      float* x_t, float* O_t, void* stream);

/* SequenceDiffuser.forward_prob_single_step / forward_prob_from_t0 / posterior_single_step
 * (diffusion.py:49-79,105-135,168-192).  kind: 0 single step, 1 from t0, 2 posterior
 * (seq = s_t, seq0 = s_0).  out[B,L,21]. */
int dab_seq_probs(const DabSchedule* sched, int kind, const int64_t* seq, const int64_t* seq0,
                  const uint8_t* mask, const int64_t* t, int B, int L, float* out, void* stream);

/* Reverse step (NOT in the reference: DiffAb.sample is a stub, diffab_pytorch.py:770-776; the
 * composition is fixed by oracle/sampler.py).  Fuses the tail of Denoiser.forward
 * (diffab_pytorch.py:594-596: O0 = O_t @ exp(v_theta)) with the three updates:
 *   s' = argmax(seq_post / seq_exp); x' = (x - beta/sqrt(1-abar) eps_theta)/sqrt(alpha) + sqrt(beta) z;
 *   O' = O0 @ exp(rotvec) (no noise at t = 1); each under where(mask, new, old).
 * O0_out may be NULL.  In-place (seq_out == seq_t etc.) is allowed. */
int dab_reverse_step(const DabSchedule* sched, const int64_t* seq_t, const float* x_t, const float* O_t,
                     const float* eps_theta, const float* v_theta, const float* seq_post,
                     const uint8_t* mask, const int64_t* t, int B, int L, const float* seq_exp,
                     const float* z, const float* rotvec, int64_t* seq_out, float* x_out, float* O_out,
                     float* O0_out, void* stream);

/* ------------------------------------------------------------------ invariant point attention */
/* One InvariantPointAttentionLayer (diffab_pytorch.py:339-465, use_pair_bias=True).
 * Weights are the layer's own state-dict tensors, nn.Linear layout (out, in) row-major. */
typedef struct DabIpaDims {
  int B, L, D, C, H, ds, Pq, Pv;
} DabIpaDims;

typedef struct DabIpaWeights {
  const float* w_q_scalar; /* (H*ds, D)    to_q_scalar.weight */
  const float* w_k_scalar; /* (H*ds, D) */
  const float* w_v_scalar; /* (H*ds, D) */
  const float* w_q_point;  /* (H*Pq*3, D) */
  const float* w_k_point;  /* (H*Pq*3, D) */
  const float* w_v_point;  /* (H*Pv*3, D) */
  const float* w_pair_bias; /* (H, C) */
  const float* gamma;      /* (H)  used raw, no softplus (diffab_pytorch.py:373,429) */
  const float* w_out;      /* (D, H*ds + H*C + H*Pv*3 + H*Pv) */
  const float* b_out;      /* (D) */
} DabIpaWeights;

typedef struct DabIpaGrads { /* same shapes as DabIpaWeights; accumulated INTO (caller zeroes) */
  float* w_q_scalar; float* w_k_scalar; float* w_v_scalar;
  float* w_q_point; float* w_k_point; float* w_v_point;
  float* w_pair_bias; float* gamma; float* w_out; float* b_out;
} DabIpaGrads;

/* Shape-generic fp32 path (the "<= 1e-4" path of north_star; any L, D, C, H, ds, Pq, Pv that fit
 * shared memory).  x[B,L,D], e[B,L,L,C], R[B,L,3,3], t[B,L,3] -> y[B,L,D].
 * Workspace (floats): dab_ipa_f32_workspace_bytes().  If save_for_bwd != 0 the workspace keeps what
 * dab_ipa_bwd_f32 needs (projections, concat features) and must be handed to it untouched. */
size_t dab_ipa_f32_workspace_bytes(const DabIpaDims* d, int for_backward);
int dab_ipa_fwd_f32(const DabIpaDims* d, const DabIpaWeights* w, const float* x, const float* e,
                    const float* R, const float* t, float* y, void* workspace, size_t workspace_bytes,
                    int save_for_bwd, void* stream);
/* Backward of the layer wrt x, e and all ten parameters (R and t are treated as constants: in the
 * reference they are the noised frames, which carry no gradient, diffab_pytorch.py:824-854).
 * dx[B,L,D] and de[B,L,L,C] are overwritten; parameter grads are accumulated into `g`. */
int dab_ipa_bwd_f32(const DabIpaDims* d, const DabIpaWeights* w, const float* x, const float* e,
                    const float* R, const float* t, const float* dy, float* dx, float* de,
                    const DabIpaGrads* g, void* workspace, size_t workspace_bytes, void* stream);

/* sm_100a fast path for the train.py configuration (L=128, D=128, C=64, H=8, ds=32, Pq=Pv=8):
 * bf16 pair tensor streamed by TMA, tcgen05 tensor-core contractions with TMEM accumulators,
 * split-bf16 point-distance logits, fp32 softmax.  `packed` is produced once per layer by
 * dab_ipa_pack_weights (weights are constant during sampling).  x[B,L,D] fp32 in, y[B,L,D] fp32
 * out, e_bf16[B,L,L,C] bf16.
 * The inference entry points (dab_ipa_fwd_sm100, _io, _stages, dab_ipa_mid_sm100, dab_ipa_pair_bias*, the packing and
 * workspace functions) also take L = 256 - the reference's preprocessed patches have 128..256 residues
 * (preprocess_pdb.py:48-58; shorter ones are padded by the caller with -inf in the padded keys' bias columns): a patch is
 * then two blocks of 128 residues - block-wise projections centred on the patch centroid, the attention core once per
 * (query block, key block) pair, the two key blocks' results merged by their softmax statistics (exact for the scalar,
 * pair and local-frame point features; point norms recomputed).  The training pair (_train / dab_ipa_bwd_sm100) is L = 128. */
size_t dab_ipa_packed_bytes(const DabIpaDims* d);
int dab_ipa_pack_weights(const DabIpaDims* d, const DabIpaWeights* w, void* packed, void* stream);
/* offs[0..6]: byte offsets of Wcat bf16 [1344][128] (rows in the order to_q_scalar, to_k_scalar, to_v_scalar, to_q_point,
 * to_k_point, to_v_point), Wout bf16 [128][1024], to_pair_bias fp32, b_out fp32, gamma fp32, Wcat^T bf16, Wout^T bf16 inside
 * `packed` - the caller's own backward GEMMs reuse the bf16 copies instead of casting the weights again. */
int dab_ipa_packed_layout(const DabIpaDims* d, size_t* offs);
size_t dab_ipa_sm100_workspace_bytes(const DabIpaDims* d);
/* Pair bias of one layer, hoisted out of the sampling loop: bias_f16[B*L*L*8] (fp16, [b][i][j][h]) =
 * scale_total * log2(e) * e . w_pair_bias^T (to_pair_bias, diffab_pytorch.py:423,439).  The pair tensor is
 * constant over the T reverse steps, so this is computed once per sampling run per layer. */
int dab_ipa_pair_bias(const DabIpaDims* d, const void* e_bf16, const float* w_pair_bias, void* bias_f16, void* stream);
/* Same for n_layers <= 6 layers in ONE pass over the pair tensor (the six layers of the epsilon network share it):
 * w_pair_bias[n_layers][8][64] fp32 contiguous, planes_f16[n_layers][B*L*L][8] fp16 contiguous. */
int dab_ipa_pair_bias_multi(const DabIpaDims* d, const void* e_bf16, const float* w_pair_bias, int n_layers,
                            void* planes_f16, void* stream);
/* bias_f16: the layer's plane from dab_ipa_pair_bias, or NULL (then it is rebuilt inside the call). */
int dab_ipa_fwd_sm100(const DabIpaDims* d, const void* packed, const float* x, const void* e_bf16,
                      const void* bias_f16, const float* R, const float* t, float* y, void* workspace,
                      size_t workspace_bytes, void* stream);
/* dab_ipa_fwd_sm100 with the residue stream in bf16 on either side (exactly one of x / x_bf16 and one of y / y_bf16 non-NULL):
 * used between the layers of InvariantPointAttentionModule (diffab_pytorch.py:494-498), where the next layer's projections
 * consume x as bf16 anyway - same bits, half the traffic. */
int dab_ipa_fwd_sm100_io(const DabIpaDims* d, const void* packed, const float* x, const void* x_bf16, const void* e_bf16,
                         const void* bias_f16, const float* R, const float* t, float* y, void* y_bf16, void* workspace,
                         size_t workspace_bytes, void* stream);
/* The same layer launch by launch: `stages` = bit0 projections + frame transform, bit1 attention core, bit2 to_out; the
 * workspace must hold the products of the lower stages (an earlier call).  For callers that bracket one stage with their
 * own events (bench.py's roofline of the attention core) - there is no process-global measurement state in the library. */
int dab_ipa_fwd_sm100_stages(const DabIpaDims* d, const void* packed, const float* x, const void* x_bf16, const void* e_bf16,
                             const void* bias_f16, const float* R, const float* t, float* y, void* y_bf16, void* workspace,
                             size_t workspace_bytes, int stages, void* stream);
/* Between two layers of a stack (inference): the previous layer's to_out (`packed_prev`; input = the concat features its
 * attention core left in `workspace`) fused into this layer's projection kernel (`packed`): y is rounded to bf16 as
 * dab_ipa_fwd_sm100_io would hand it over but never exists in HBM.  Stack = stages(1) of layer 0, then per layer stages(2)
 * + dab_ipa_mid_sm100 (stages(4) after the last layer); bit-identical to the unfused sequence
 * (InvariantPointAttentionModule.forward, diffab_pytorch.py:494-498). */
int dab_ipa_mid_sm100(const DabIpaDims* d, const void* packed_prev, const void* packed, const float* R, const float* t,
                      void* workspace, size_t workspace_bytes, void* stream);
/* Projections of the FIRST layer of the stack with the epsilon network's front MLP (Denoiser.to_res_emb during sampling,
 * diffab_pytorch.py:572-574) fused in: the layer input relu(c[row] + t1[seq[row]]) W2^T + b2 - c[B*L,128] / t1[25,128] the
 * regrouped first layer as in dab_front_fwd_sm100, w2_bf16 [128][128], b2 [128] - is formed in the projection kernel's operand
 * tile and never exists in HBM.  Replaces dab_front_fwd_sm100 followed by dab_ipa_fwd_sm100_stages(.., 1); the same bits. */
int dab_ipa_front_proj_sm100(const DabIpaDims* d, const void* packed, const float* c, const float* t1, const int64_t* seq,
                             const void* w2_bf16, const float* b2, const float* R, const float* t, void* workspace,
                             size_t workspace_bytes, void* stream);
/* Training pair of the sm_100a path (bf16 pair tensor, fp32 x / y).  The forward is dab_ipa_fwd_sm100 (the pair
 * bias is rebuilt inside the call when bias_f16 is NULL); `saved` (dab_ipa_sm100_workspace_bytes) additionally keeps
 * the packed operands, the concat features, the un-normalised probabilities and the softmax statistics, and must
 * reach the backward untouched. */
int dab_ipa_fwd_sm100_train(const DabIpaDims* d, const void* packed, const float* x, const void* e_bf16,
                            const void* bias_f16 /* plane of this layer or NULL */, const float* R, const float* t,
                            float* y, void* saved, size_t saved_bytes, void* stream);
/* Backward of the attention part of the layer (autograd of diffab_pytorch.py:389-462) on tcgen05:
 *   in : dcat[B*L,1024] fp32 = dy . to_out.weight (gradient of the concat features; a plain GEMM of the caller),
 *        e_bf16, R, `saved` from dab_ipa_fwd_sm100_train, `packed` weights;
 *   out: dproj_bf16[B*L,1344] bf16 = gradient of the six projections in the row order of
 *        [to_q_scalar; to_k_scalar; to_v_scalar; to_q_point; to_k_point; to_v_point] (so dx = dproj . Wcat and
 *        dWcat = dproj^T . x are plain GEMMs of the caller), de_bf16[B,L,L,C] bf16 (overwritten),
 *        d_w_pair_bias[8,64] and d_gamma[8] (accumulated into).
 * R and t are treated as constants, as in dab_ipa_bwd_f32. */
int dab_ipa_sm100_workspace_layout(const DabIpaDims* d, size_t* offsets /* 8: Qp, Kp, Vp, tc, cat, bias, stats, pu */);
size_t dab_ipa_bwd_sm100_workspace_bytes(const DabIpaDims* d);
int dab_ipa_bwd_sm100(const DabIpaDims* d, const void* packed, const void* e_bf16, const float* R, const float* dcat,
                      void* saved, size_t saved_bytes, void* dproj_bf16, void* de_bf16, float* d_w_pair_bias, float* d_gamma,
                      void* workspace, size_t workspace_bytes, void* stream);
/* The same backward in two calls (same arguments): `_main` = everything up to dproj / de and the per-CTA partial sums,
 * `_finish` = d_w_pair_bias / d_gamma from those sums - lets the caller overlap the final reductions with the GEMMs that
 * depend only on dproj (dx, dWcat). */
int dab_ipa_bwd_sm100_main(const DabIpaDims* d, const void* packed, const void* e_bf16, const float* R, const float* dcat,
                           void* saved, size_t saved_bytes, void* dproj_bf16, void* de_bf16, float* d_w_pair_bias,
                           float* d_gamma, void* workspace, size_t workspace_bytes, void* stream);
int dab_ipa_bwd_sm100_finish(const DabIpaDims* d, const void* packed, const void* e_bf16, const float* R, const float* dcat,
                             void* saved, size_t saved_bytes, void* dproj_bf16, void* de_bf16, float* d_w_pair_bias,
                             float* d_gamma, void* workspace, size_t workspace_bytes, void* stream);
#ifdef DAB_DEBUG_HOOKS /* debug build only (make debug -> libdiffab_b200_dbg.so): process-global profiling / inspection hooks */
int dab_debug_set_bwd_timeline(long long* device_buf /* 64 slots per CTA of the backward core, or NULL */);
int dab_debug_bwd_keep_qkv(int on);
int dab_debug_bwd_sm100_buffers(const DabIpaDims* d, void* workspace, void** out /* 10 device pointers */);
#endif
/* ------------------------------------------------------------------ epsilon-network tail (SURVEY 8f N1)
 * The three denoising heads of Denoiser.forward (diffab_pytorch.py:584-599) for d_residue_emb = 128, L = 128, fused
 * into one tcgen05 kernel: [x | beta, sin beta, cos beta] -> MLP(131 -> 128 -> 128 -> {3, 3, 21}) x 3, softmax on
 * the sequence head.  Weights are the state-dict tensors of coordinate_denoising / orientation_denoising /
 * sequence_denoising (layers .0, .2, .4), nn.Linear layout (out, in) row-major. */
typedef struct DabHeadWeights {
  const float *c_w1, *c_b1, *c_w2, *c_b2, *c_w3, *c_b3; /* coordinate_denoising:  (128,131) (128) (128,128) (128) (3,128) (3) */
  const float *o_w1, *o_b1, *o_w2, *o_b2, *o_w3, *o_b3; /* orientation_denoising: same shapes */
  const float *s_w1, *s_b1, *s_w2, *s_b2, *s_w3, *s_b3; /* sequence_denoising:    last layer (21,128) (21) */
} DabHeadWeights;
size_t dab_heads_packed_bytes(void);
int dab_heads_pack_weights(const DabHeadWeights* w, void* packed, void* stream);
/* x[n_patches*L,128] fp32, beta[n_patches] fp32 -> eps[.,3], rotvec[.,3], seq_posterior[.,21] fp32. */
int dab_heads_fwd_sm100(const void* packed, const float* x, const float* beta, int n_patches, int L, float* eps,
                        float* rotvec, float* seq_posterior, void* stream);
/* The same heads with the LAST IPA layer's to_out (diffab_pytorch.py:464: y = cat Wout^T + b) fused in front: cat_bf16
 * [n_patches*128, 1024] = the concat features the layer's attention core left in its workspace (dab_ipa_sm100_workspace_layout),
 * wout_bf16 [128][1024] and b_out [128] from the layer's packed weights (dab_ipa_packed_layout).  The stack's output never
 * exists in HBM; the same bits as dab_ipa_fwd_sm100_stages(.., 4) followed by dab_heads_fwd_sm100. */
int dab_out_heads_fwd_sm100(const void* packed, const void* cat_bf16, const void* wout_bf16, const float* b_out, const float* beta,
                            int n_patches, int L, float* eps, float* rotvec, float* post, void* stream);

/* Front of the epsilon network during sampling (diffab_pytorch.py:572-574, to_res_emb on [res_ctx | emb(s_t)]):
 * x0[n_rows,128] = relu(c[row] + t1[seq[row]]) . w2^T + b2, where c = res_ctx . W1[:, :128]^T + b1 (per-run constant,
 * fp32 [n_rows,128]) and t1 = emb . W1[:, 128:]^T (fp32 [25,128]) are computed once per run by the caller;
 * w2_bf16 = to_res_emb.2.weight in bf16 [128][128]; a_scratch holds n_rows*128 bf16.  Exactly one of x0 (fp32) and
 * x0_bf16 (the same values rounded to bf16, the form dab_ipa_fwd_sm100_io takes) is non-NULL. */
int dab_front_fwd_sm100(const float* c, const float* t1, const int64_t* seq, int64_t n_rows, const void* w2_bf16,
                        const float* b2, void* a_scratch, float* x0, void* x0_bf16, void* stream);

/* ------------------------------------------------------------------ pair context encoder (SURVEY 8f N3)
 * PairEmbedding.forward (diffab_pytorch.py:186-312) fused into one tcgen05 kernel that writes the pair tensor in bf16
 * (inference / sampling; L = 128 or 256 residues, 15 atoms, d_pair_emb = 64, max_dist_to_consider = 32).  Distances are
 * computed from xyz inside the kernel.  Weights: the module's state-dict tensors, nn.Linear layout (out, in). */
typedef struct DabPairEmbedWeights {
  const float* type_emb;      /* aa_pair_type_embedding.weight (441, 64) */
  const float* relpos_emb;    /* relpos_embedding.weight       (65, 64)  */
  const float* pair2distcoef; /* pair2distcoef.weight          (441, 225) */
  const float *d_w1, *d_b1, *d_w2, *d_b2;               /* distance_embedding.{0,2}: (64,225) (64) (64,64) (64) */
  const float *m_w1, *m_b1, *m_w2, *m_b2, *m_w3, *m_b3; /* mlp.{0,2,4}: (64,210) (64) (64,64) (64) (64,64) (64) */
} DabPairEmbedWeights;
size_t dab_pair_embed_packed_bytes(void);
int dab_pair_embed_pack_weights(const DabPairEmbedWeights* w, void* packed, void* stream);
/* seq_masked[B,L] int64 (sequence with non-context residues already replaced by UNK, :271-273), xyz[B,L,A,3],
 * pairwise_dihedrals[B,L,L,2], residue_idx / chain_idx [B,L] int64, atom_mask[B,L,A] uint8 -> e_bf16[B,L,L,64]. */
int dab_pair_embed_fwd_sm100(const void* packed, const int64_t* seq_masked, const float* xyz, const float* pairwise_dihedrals,
                             const int64_t* residue_idx, const int64_t* chain_idx, const uint8_t* atom_mask, int B, int L,
                             int A, void* e_bf16, void* stream);

/* Distance radial-basis features of PairEmbedding for training (diffab_pytorch.py:287-294): one pass forward
 * (rbf_bf16[B,L,L,232], columns 225..231 zero), one pass backward (d_coef[441,225] accumulated into). */
size_t dab_rbf_workspace_bytes(int B, int L);
int dab_rbf_fwd(const float* distmat, const int64_t* seq_masked, const uint8_t* atom_mask, const float* coef, int B, int L,
                int squared, void* rbf_bf16, void* workspace, size_t workspace_bytes, void* stream);
int dab_rbf_bwd(const void* grad_bf16, const float* distmat, const int64_t* seq_masked, const uint8_t* atom_mask,
                const float* coef, int B, int L, int squared, float* d_coef, void* workspace, size_t workspace_bytes,
                void* stream);

/* Per-pair glue of PairEmbedding's first mlp layer for training (diffab_pytorch.py:262-285,303-311; csrc/pair_train_kernels.cu).
 * dab_pair_base_fwd: base_bf16[B,L,L,64] = t_type[s_i*21+s_j] + chain_i*chain_j * t_rel[clamp(r_i-r_j)+max_dist] and the angular
 * encoding of the pairwise dihedrals xh_bf16[B,L,L,32] (columns 18..31 zero); t_type_bf16[441,64], t_rel_bf16[2*max_dist+1,64].
 * dab_pair_table_grad: class sums of the per-pair gradient g1_bf16[B,L,L,64], accumulated into s_type[441,64] and
 * s_rel[2*max_dist+1,64] (the latter weighted by chain_i*chain_j).
 * dab_pair_zero_masked: x_bf16[B,L,L,64] rows with res_mask[b,i] == 0 or res_mask[b,j] == 0 set to zero in place. */
int dab_pair_base_fwd(const int64_t* seq_masked, const int64_t* residue_idx, const int64_t* chain_idx,
                      const float* pairwise_dihedrals, const void* t_type_bf16, const void* t_rel_bf16, int B, int L,
                      int max_dist, void* base_bf16, void* xh_bf16, void* stream);
size_t dab_pair_table_grad_workspace_bytes(int B, int L, int max_dist);
int dab_pair_table_grad(const void* g1_bf16, const int64_t* seq_masked, const int64_t* residue_idx, const int64_t* chain_idx,
                        int B, int L, int max_dist, float* s_type, float* s_rel, void* workspace, size_t workspace_bytes,
                        void* stream);
int dab_pair_zero_masked(void* x_bf16, const uint8_t* res_mask, int B, int L, void* stream);
/* dab_pair_table_grad on the tensor cores (csrc/pair_table_grad_sm100.cu; L = 128, max_dist <= 63): the class sums as GEMMs of
 * one-hot matrices (residue type of the key: constant per patch; relative position: one entry per key moves per query row)
 * against the g1 tile, read once.  s_type[441,64] and s_rel[2*max_dist+1,64] are ACCUMULATED into with red.global (fp32; the
 * caller zeroes them; summation order not fixed). */
int dab_pair_table_grad_sm100(const void* g1_bf16, const int64_t* seq_masked, const int64_t* residue_idx,
                              const int64_t* chain_idx, int B, int L, int max_dist, float* s_type, float* s_rel, void* stream);
/* out_bf16[n] = sum of n_src (1..8) bf16 tensors, fp32 accumulation, one pass: the pair-tensor gradients of the IPA layers
 * (autograd would add them pairwise, five passes and five bf16 roundings for six layers).  out may be one of the sources. */
int dab_sum_bf16(const void* const* src, int n_src, int64_t n, void* out_bf16, void* stream);
/* ReLU backward of a 64-channel bf16 layer fused with its bias gradient: g_out = g_in where y > 0 else 0 (may alias g_in),
 * colsum[64] += column sums of g_out. */
int dab_relu_bwd_colsum(const void* g_in_bf16, const void* y_bf16, int64_t n, void* g_out_bf16, float* colsum, void* stream);
/* PairEmbedding's MLPs behind the first distance layer, training forward, in ONE kernel (csrc/pair_mlp_fwd_sm100.cu;
 * diffab_pytorch.py:214-223,262-285,303-311): fd = relu(a1 Wd2^T + bd2), h1 = relu(T_type[s_i*21+s_j] + c_i c_j T_rel[clamp(r_i-r_j)]
 * + fd W1d^T + xh W1h^T), h2 = relu(h1 W2^T + b2) m_i m_j, out = (h2 W3^T + b3) m_i m_j; every activation the backward pass needs
 * is written once.  a1_bf16 [B,L,L,64] = relu(Wd1 rbf + bd1); w5_bf16 [5][64 out][64 in] = Wd2, W1[:, 128:192], W1[:, 192:] zero-
 * padded to 64 columns, W2, W3; bias3 [3][64] fp32 = bd2, b2, b3; t_type_bf16 [441,64] = E_type W1[:, :64]^T + b1;
 * t_rel_bf16 [65,64] = E_rel W1[:, 64:128]^T.  Outputs (bf16): fd, h1, h2, out [B,L,L,64] and the angular features
 * xh [B,L,L,32] (columns 18..31 zero).  L = 128 and max_dist = 32 only (DAB_EUNSUPPORTED otherwise). */
int dab_pair_mlp_fwd_train_sm100(const void* a1_bf16, const float* pairwise_dihedrals, const int64_t* seq_masked,
                                 const int64_t* residue_idx, const int64_t* chain_idx, const uint8_t* res_mask,
                                 const void* t_type_bf16, const void* t_rel_bf16, const void* w5_bf16, const float* bias3, int B,
                                 int L, int max_dist, void* fd_bf16, void* h1_bf16, void* h2_bf16, void* out_bf16,
                                 void* xh_bf16, void* stream);
/* One 64-channel layer y = a W^T + b of PairEmbedding's two MLPs (diffab_pytorch.py:214-223,303-311) backward in ONE pass over
 * the B*L*L pairs (csrc/pair_mlp_bwd_sm100.cu): dW[64][64] += g^T a, db[64] += column sums of g over the valid pairs,
 * g_prev = (g W) * (a > 0) - the gradient w.r.t. the pre-activation of the layer before, whose ReLU output a is - and
 * db_prev[64] += column sums of g_prev.  g_bf16, a_bf16, g_prev_bf16: [B*L*L, 64] bf16;
 * W_bf16: [64 out][64 in]; res_mask (optional, [B, L]): pairs with a masked residue are left out of db (their rows of a
 * must be zero: dab_pair_zero_masked).  g_prev_bf16 and db_prev may be null.  dW, db, db_prev are fp32 and ACCUMULATED
 * into with red.global (the caller zeroes them; summation order not fixed). */
int dab_pair_mlp_bwd_layer_sm100(const void* g_bf16, const void* a_bf16, const void* W_bf16, const uint8_t* res_mask, int B,
                                 int L, void* g_prev_bf16, float* dW, float* db, float* db_prev, void* stream);

/* The three masked training losses in one pass each way (DiffAb._shared_step, diffab_pytorch.py:856-880 with KLDivLoss / MSELoss /
 * OrientationLoss :610-625, reduction "none", then masked mean; csrc/loss_kernels.cu).  n = B*L residues; post_*[n,21],
 * eps_*[n,3], O_*[n,3,3] fp32, mask[n] uint8 = generation_mask & residue_mask.  Forward: acc = 8 zeroed floats of scratch,
 * out[0..2] = sequence / translation / orientation loss, out[3] = number of masked residues.  Backward: g[3] = upstream
 * gradients of the three losses, fwd_out = the forward's out; writes d_post[n,21], d_eps[n,3], d_O[n,3,3]. */
int dab_losses_fwd(const float* post_pred, const float* post_tgt, const float* eps_pred, const float* eps_tgt, const float* O_pred,
                   const float* O_true, const uint8_t* mask, int64_t n, float* acc, float* out, void* stream);
int dab_losses_bwd(const float* post_pred, const float* post_tgt, const float* eps_pred, const float* eps_tgt, const float* O_pred,
                   const float* O_true, const uint8_t* mask, int64_t n, const float* g, const float* fwd_out, float* d_post,
                   float* d_eps, float* d_O, void* stream);
/* One Adam step (torch.optim.Adam semantics, the reference's configure_optimizers diffab_pytorch.py:925-931) on a FLAT fp32
 * parameter vector: p, m, v [n] updated in place from the gradient g [n] (n % 4 == 0, 16-byte aligned); `step` = device
 * scalar (float) with the step count including this step, incremented by the caller - no host state, graph-capturable. */
int dab_adam_flat(float* p, const float* g, float* m, float* v, const float* step, float lr, float beta1, float beta2,
                  float eps, float weight_decay, int64_t n, void* stream);

/* The tcgen05 GEMM C[M,N] = A[M,K] B[N,K]^T + bias (bf16 in, fp32 out; M % 128 == 0, N % 64 == 0, K % 64 == 0): nn.Linear
 * (diffab_pytorch.py:464) as a stand-alone entry point. */
int dab_gemm_bf16(const void* A, const void* Bm, float* C, const float* bias, int M, int N, int K, void* stream);
/* C[M,N] (fp32, overwritten) = A[K,M]^T B[K,N]: bf16 operands whose ROW index is the contraction index (activations as
 * they lie in memory, one row per residue), read MN-major by tcgen05 - no transposed copies.  Split over K, partial tiles
 * added with red.global (summation order not fixed).  K % 64 == 0, N % 64 == 0, lda % 8 == 0, ldb % 8 == 0, ldc % 4 == 0,
 * lda >= M, ldb >= N, ldc >= N, any M > 0; only the M x N block of C is written (C may be a column block).  The autograd weight
 * gradients of the nn.Linear layers of diffab_pytorch.py:391-408,464 (dWout = dy^T cat, dWcat = dproj^T x). */
int dab_gemm_bf16_tn(const void* A, int64_t lda, const void* Bm, int64_t ldb, float* C, int64_t ldc, int M, int N, int K,
                     void* stream);
/* C += A^T B: the same GEMM without the fill of C (the caller zeroes C beforehand, off the critical path). */
int dab_gemm_bf16_tn_acc(const void* A, int64_t lda, const void* Bm, int64_t ldb, float* C, int64_t ldc, int M, int N, int K,
                         void* stream);
/* out[cols] (fp32, overwritten) = column sums of x[rows, cols]: bias gradients (d b_out = sum over residues of dy);
 * x_bf16 (may be NULL) receives x rounded to bf16 in the same pass (the operand of the gradient GEMMs). */
int dab_colsum_f32(const float* x, int64_t rows, int cols, float* out, void* x_bf16, void* stream);
/* Mixed-precision nn.Linear layers of the dense glue (ResidueEmbedding.mlp, Denoiser.to_res_emb, the heads:
 * diffab_pytorch.py:57-183,572-599) on the library's tcgen05 GEMM.
 * dab_linear_bf16: C = act(A[M,K] W[N,K]^T + bias), bf16 operands, fp32 accumulation; act = ReLU when relu != 0; the result as
 *   fp32 (C_f32) or rounded to bf16 (C_bf16), exactly one of the two non-NULL.  M % 128 == 0, N % 64 == 0, K % 64 == 0.
 *   Forward y = x W^T + b, and with W transposed the data gradient dx = g W.
 * dab_bias_grad: g' = g * (y > 0) (y_bf16 = the layer's ReLU output, NULL: no mask), db[cols] (fp32, overwritten) = column
 *   sums of g', g_out_bf16 (optional) = g' rounded to bf16 (the operand of dx = g' W and dW = g'^T x, dab_gemm_bf16_tn).
 *   g: fp32 (g_is_bf16 = 0) or bf16, [rows, cols] contiguous; cols % 4 == 0 (8 for bf16 input), <= 1024. */
int dab_linear_bf16(const void* A, const void* W, const float* bias, int relu, int M, int N, int K, float* C_f32, void* C_bf16,
                    void* stream);
int dab_bias_grad(const void* g, int g_is_bf16, const void* y_bf16, int64_t rows, int cols, float* db, void* g_out_bf16,
                  void* stream);
#ifdef DAB_DEBUG_HOOKS /* debug build only */
int dab_debug_set_timeline(long long* device_buf /* 64 slots per tile of the attention core, or NULL */);
#endif
/* fp32 -> bf16 conversion of the pair tensor (once per patch; round-to-nearest-even). */
int dab_cast_f32_to_bf16(const float* in, void* out, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIFFAB_B200_H */
