"""Oracle of the amino-acid bias of sampling (``DiffAb.sample(aa_bias=)``) for the tests.

UNPINNED BY THE REFERENCE, which has no sampler.  The weighted draw is stated here in fp32 torch on the CPU, on top of
``oracle.sampler.reverse_step`` (pinned by our goldens), whose positions and orientations it keeps.  The rule, with
``w`` = the per-type weights (``exp(b - max_k b)``) and ``q`` = the step's Exp(1) draw ``seq_exp``:

  eligible types: w_k > 0;  key_k = fl(fl(p_k * w_k) / q_k);  s' = first eligible k with the largest key
  every eligible key 0 (posterior mass on the allowed types underflowed): key_k = w_k / q_k over the eligible types
  no eligible type: s' = s (the residue keeps its type)

With all-ones weights, p_k * 1 = p_k and the draw is ``oracle.sampler``'s, bit for bit (unless a posterior row is zero
throughout, which a softmax never is).
"""
import torch

from oracle import diffusion as odiff
from oracle import sampler as osamp


def weights(aa_bias):
    """exp(b - max_k b) in fp32 (the conversion of ``aa_bias_weights`` without its checks)."""
    b = torch.as_tensor(aa_bias, dtype=torch.float32)
    return torch.exp(b - b.amax(-1, keepdim=True).clamp_min(torch.finfo(torch.float32).min))


def weighted_draw(post, q, w, s_old):
    """The sequence draw of one reverse step: post, q, w (N, 21) fp32, s_old (N,) int64 -> (N,) int64."""
    elig = w > 0
    neg = torch.full_like(post, -1.0)
    key = torch.where(elig, (post * w) / q, neg)
    idx = key.argmax(-1)
    redraw = key.amax(-1) == 0
    idx_w = torch.where(elig, w / q, neg).argmax(-1)
    idx = torch.where(redraw, idx_w, idx)
    return torch.where(elig.any(-1), idx, s_old)


def reverse_step(sched, hist_rev, s_t, x_t, O_t, eps_theta, O0_theta, seq_post, generation_mask, t, noise, w):
    """``oracle.sampler.reverse_step`` with the sequence drawn by ``weighted_draw``; ``w`` (B, L, 21)."""
    out = osamp.reverse_step(sched, hist_rev, s_t, x_t, O_t, eps_theta, O0_theta, seq_post, generation_mask, t, noise)
    B, L = s_t.shape
    V = odiff.V
    s_new = weighted_draw(seq_post.reshape(-1, V).float(), noise["seq_exp"].view(-1, V).float(),
                          w.reshape(-1, V).float(), s_t.reshape(-1)).view(B, L)
    out["seq_idx"] = torch.where(generation_mask, s_new, s_t)
    return out


def prior_draw(w, E):
    """The t = T prior of the sequence under weights: argmax_k w_k / E_k; w, E (N, 21)."""
    return (w / E).argmax(-1)
