"""``DiffAb`` and its epsilon network on the GPU - mirror of ``diffab_pytorch/diffab_pytorch.py``.

Drop-in boundary (SURVEY §8b): same class names, constructor signatures, method names, return
dict keys and the same 106 state-dict keys/shapes as the reference, so a reference checkpoint
loads with ``load_state_dict``.  What runs where:

* per-timestep hot path - IPA layers, SO(3) maps, forward noising, reverse step: hand-written
  sm_100a kernels behind the C ABI (``csrc/``);
* context encoders (``ResidueEmbedding``, ``PairEmbedding``; once per patch, out of scope per
  SURVEY §2) and the small dense glue of ``Denoiser`` (embedding + MLP heads, "next" row N1): PyTorch
  modules on the GPU (library GEMMs) on the exact fp32 path and in training; on the bf16 sampling path the
  glue runs in ``csrc/heads_sm100.cu`` and ``PairEmbedding`` in ``csrc/pair_embed_sm100.cu`` ("next" rows N1, N3);
* ``sample()`` - an empty stub in the reference (``diffab_pytorch.py:770-776``) - is implemented
  here following oracle/sampler.py.

Not a LightningModule: ``pytorch_lightning`` is not a dependency; ``training_step`` /
``validation_step`` / ``configure_optimizers`` keep their names and return values.
"""
import contextlib
import ctypes
import types
import math
from typing import Dict, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib
from . import diffusion as _diffusion
from . import so3 as _so3
from ._lib import ptr
from .diffusion import (CoordinateDiffuser, OrientationDiffuser, SequenceDiffuser,  # noqa: F401
                        cosine_variance_schedule)
from .so3 import vector_to_rotation_matrix

CA_IDX = 1     # protstruc.general.ATOM.CA (diffab_pytorch.py:110,249,820)
AA_UNK = 20    # protstruc.general.AA.UNK  (diffab_pytorch.py:115,273; assumed, SURVEY §8c O2)


@contextlib.contextmanager
def _tf32_matmuls(enabled):
    """TF32 for the library GEMMs of the PyTorch glue (context encoders, embedding / head MLPs).  The
    reference's own GPU entry point asks for the same (train.py:47, set_float32_matmul_precision("high"));
    used only by the bf16 sampling path, the fp32 path keeps full-precision matmuls."""
    if not enabled:
        yield
        return
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        yield
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


# =============================================================================================
# Context encoders (out of the hot path; forward-identical PyTorch restatements)
# =============================================================================================
class AngularEncoding(nn.Module):
    """diffab_pytorch.py:20-54: [x, sin(f x), cos(f x)] for f in (1..n, 1/1..1/n)."""

    def __init__(self, num_funcs=3):
        super().__init__()
        self.num_funcs = num_funcs
        # a non-persistent buffer: follows the module's device (no per-call host-to-device copy, CUDA-graph safe)
        # without appearing in the state dict
        self.register_buffer("freq_bands", torch.tensor([float(i + 1) for i in range(num_funcs)] +
                                                        [1.0 / (i + 1) for i in range(num_funcs)]), persistent=False)

    def get_output_dimension(self, d_in):
        return d_in * (4 * self.num_funcs + 1)

    def forward(self, x):
        f = self.freq_bands.to(x.device)
        x = x.unsqueeze(-1)
        return torch.cat([x, torch.sin(f * x), torch.cos(f * x)], dim=-1).flatten(-2)


def _mlp(dims, final_relu=False):
    layers = []
    for i in range(len(dims) - 1):
        layers.append(nn.Linear(dims[i], dims[i + 1]))
        if i + 2 < len(dims) or final_relu:
            layers.append(nn.ReLU())
    return nn.Sequential(*layers)


class _LinearFunction(torch.autograd.Function):
    """``F.linear`` whose bias gradient is the library's column-sum kernel (``dab_colsum_f32``): autograd's own is a strided
    at::reduce kernel, ~14 us per layer for the 8192 x 128 activations of a training batch, fifteen of them per step."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        return F.linear(x, weight, bias)

    @staticmethod
    def backward(ctx, g):
        x, weight = ctx.saved_tensors
        g2 = g.reshape(-1, g.shape[-1])
        dx = (g2 @ weight).view(x.shape) if ctx.needs_input_grad[0] else None
        dw = g2.t() @ x.reshape(-1, x.shape[-1]) if ctx.needs_input_grad[1] else None
        db = None
        if ctx.needs_input_grad[2]:
            n = g2.shape[1]
            if g2.dtype == torch.float32 and g2.is_contiguous() and n % 4 == 0 and n <= 1024 and g2.data_ptr() % 16 == 0:
                db = torch.empty(n, device=g2.device, dtype=torch.float32)
                _lib.check(_lib.lib().dab_colsum_f32(ptr(g2), g2.shape[0], n, ptr(db), None, _lib.stream_ptr()), "dab_colsum_f32")
            else:
                db = g2.sum(0)
        return dx, dw, db


class _MixedMlpFunction(torch.autograd.Function):
    """A run of nn.Linear (+ ReLU) layers on the library's kernels in mixed precision (bf16 operands and activations, fp32
    accumulation and results): forward ``dab_linear_bf16`` per layer with the bias / ReLU / bf16 epilogue fused; backward per
    layer ONE pass for ReLU backward + bias gradient + the bf16 operand (``dab_bias_grad``), the weight gradient on the
    MN-major GEMM (``dab_gemm_bf16_tn``) and the data gradient on the K-major one against the transposed weight.
    ``spec`` = tuple of booleans: ReLU behind layer k.  Every layer: in / out features multiples of 64, rows of 128."""

    @staticmethod
    def forward(ctx, x, spec, *params):
        lib, st = _lib.lib(), _lib.stream_ptr()
        bf, f32 = torch.bfloat16, torch.float32
        n = len(spec)
        lead, M = x.shape[:-1], x.numel() // x.shape[-1]
        a = torch.empty(M, x.shape[-1], device=x.device, dtype=bf)
        xc = _lib.dev(x.reshape(M, -1), f32, "x")
        _lib.check(lib.dab_cast_f32_to_bf16(ptr(xc), ptr(a), xc.numel(), st), "dab_cast_f32_to_bf16")
        acts, w16 = [a], []
        out = None
        for k in range(n):
            w, b = params[2 * k], params[2 * k + 1]
            wk = w.detach().to(bf).contiguous()
            w16.append(wk)
            N, K = w.shape
            last = k == n - 1
            y = torch.empty(M, N, device=x.device, dtype=f32 if last else bf)
            _lib.check(lib.dab_linear_bf16(ptr(acts[-1]), ptr(wk), ptr(_lib.dev(b.detach(), f32, "bias")), int(spec[k]), M, N, K,
                                           ptr(y) if last else None, None if last else ptr(y), st), "dab_linear_bf16")
            if last:
                out = y
                if spec[k]:                       # the ReLU mask of the last layer (its output leaves as fp32)
                    acts.append(y)
            else:
                acts.append(y)
        ctx.save_for_backward(*acts, *w16)
        ctx.spec, ctx.n = spec, n
        return out.view(*lead, out.shape[-1])

    @staticmethod
    def backward(ctx, g):
        lib, st = _lib.lib(), _lib.stream_ptr()
        bf, f32 = torch.bfloat16, torch.float32
        n, spec = ctx.n, ctx.spec
        saved = ctx.saved_tensors
        n_act = len(saved) - n
        acts, w16 = saved[:n_act], saved[n_act:]
        M = acts[0].shape[0]
        grads = [None] * (2 * n)
        gk = _lib.dev(g.reshape(M, -1), f32, "grad")
        g_is_bf16 = 0
        dx = None
        for k in range(n - 1, -1, -1):
            N, K = w16[k].shape
            mask = None
            if spec[k]:
                y = acts[k + 1]                 # ReLU output of layer k (bf16; fp32 for the last layer)
                mask = y if y.dtype == bf else y.to(bf)
            db = torch.empty(N, device=g.device, dtype=f32)
            g16 = torch.empty(M, N, device=g.device, dtype=bf)
            _lib.check(lib.dab_bias_grad(ptr(gk), g_is_bf16, ptr(mask), M, N, ptr(db), ptr(g16), st), "dab_bias_grad")
            dw = torch.empty(N, K, device=g.device, dtype=f32)
            _lib.check(lib.dab_gemm_bf16_tn(ptr(g16), N, ptr(acts[k]), K, ptr(dw), K, N, K, M, st), "dab_gemm_bf16_tn")
            grads[2 * k], grads[2 * k + 1] = dw, db
            if k > 0 or ctx.needs_input_grad[0]:
                wt = w16[k].t().contiguous()    # [K, N]: dx = g W as a K-major GEMM against W^T
                first = k == 0
                gx = torch.empty(M, K, device=g.device, dtype=f32 if first else bf)
                _lib.check(lib.dab_linear_bf16(ptr(g16), ptr(wt), None, 0, M, K, N, ptr(gx) if first else None,
                                               None if first else ptr(gx), st), "dab_linear_bf16 (dx)")
                if first:
                    dx = gx
                else:
                    gk, g_is_bf16 = gx, 1
        if dx is not None:
            dx = dx.view(*g.shape[:-1], dx.shape[-1])
        return (dx, None, *grads)


_MIXED_GLUE = [False]     # set for the duration of a mixed-precision training forward (DiffAb._shared_step)


@contextlib.contextmanager
def _mixed_glue(enabled):
    prev = _MIXED_GLUE[0]
    _MIXED_GLUE[0] = bool(enabled)
    try:
        yield
    finally:
        _MIXED_GLUE[0] = prev


def _run_mlp(mlp, x):
    """``mlp(x)`` for an ``_mlp`` Sequential.  On CUDA tensors that record gradients: in a mixed-precision training step,
    runs of layers whose shapes the tcgen05 GEMM takes (features multiples of 64, rows of 128) go through
    ``_MixedMlpFunction``; other Linear layers through ``_LinearFunction`` (same forward call, cheaper bias gradient)."""
    if not (x.is_cuda and torch.is_grad_enabled()):
        return mlp(x)
    mods = list(mlp)
    rows = x.numel() // x.shape[-1]
    ok = lambda m: (_MIXED_GLUE[0] and isinstance(m, nn.Linear) and m.bias is not None and m.in_features % 64 == 0 and
                    m.out_features % 64 == 0 and rows % 128 == 0 and x.dtype == torch.float32)
    i = 0
    while i < len(mods):
        m = mods[i]
        if ok(m):
            spec, params = [], []
            while i < len(mods) and ok(mods[i]):
                relu = i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU)
                spec.append(relu)
                params += [mods[i].weight, mods[i].bias]
                i += 2 if relu else 1
            x = _MixedMlpFunction.apply(x, tuple(spec), *params)
        elif isinstance(m, nn.Linear) and m.bias is not None:
            x = _LinearFunction.apply(x, m.weight, m.bias)
            i += 1
        else:
            x = m(x)
            i += 1
    return x


class _SmallVocabEmbedding(torch.autograd.Function):
    """nn.Embedding lookup whose weight gradient is one_hot(idx)^T @ grad (a small GEMM) instead of PyTorch's
    sort-and-segment kernels (~100 us per call for the 8192 residues of a training batch).  Same values."""

    @staticmethod
    def forward(ctx, idx, weight, padding_idx):
        ctx.save_for_backward(idx)
        ctx.vocab, ctx.padding_idx = weight.shape[0], padding_idx
        return F.embedding(idx, weight)

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        onehot = F.one_hot(idx.reshape(-1), ctx.vocab).to(g.dtype)
        dw = onehot.t() @ g.reshape(-1, g.shape[-1])
        if ctx.padding_idx is not None:
            dw[ctx.padding_idx] = 0          # nn.Embedding(padding_idx=...) never updates that row
        return None, dw, None


def _embed(module, idx):
    """``module(idx)`` for a small-vocabulary nn.Embedding; on the GPU with the gradient through a one-hot GEMM."""
    if idx.is_cuda and torch.is_grad_enabled() and module.weight.requires_grad:
        return _SmallVocabEmbedding.apply(idx, module.weight, module.padding_idx)
    return module(idx)


class ResidueEmbedding(nn.Module):
    """diffab_pytorch.py:57-183."""

    def __init__(self, max_n_atoms_per_residue, d_feat):
        super().__init__()
        self.max_n_aa_types = 21
        self.max_n_atoms_per_residue = max_n_atoms_per_residue
        self.amino_acid_type_embedding = nn.Embedding(self.max_n_aa_types, d_feat)
        self.dihedral_embedding = AngularEncoding(num_funcs=3)
        self.chain_embedding = nn.Embedding(10, d_feat, padding_idx=0)
        d_coord = self.max_n_aa_types * max_n_atoms_per_residue * 3
        d_dihedral = self.dihedral_embedding.get_output_dimension(3)
        self.mlp = _mlp([d_feat + d_coord + d_dihedral + d_feat, d_feat * 2, d_feat, d_feat, d_feat])

    def forward(self, seq_idx, xyz, orientation, dihedrals, chain_idx, atom_mask, structure_context_mask=None,
                sequence_context_mask=None):
        B, L = seq_idx.shape
        A = self.max_n_atoms_per_residue
        if sequence_context_mask is not None:
            seq_idx = torch.where(sequence_context_mask.bool(), seq_idx, torch.full_like(seq_idx, AA_UNK))
        aa = _embed(self.amino_acid_type_embedding, seq_idx)
        rel = xyz - xyz[:, :, CA_IDX:CA_IDX + 1, :]
        if xyz.is_cuda:
            local = _so3.small_matmul(rel, orientation) * atom_mask[..., None]             # O^T (x - x_CA), row vectors
        else:
            local = torch.einsum("blji,blaj->blai", orientation, rel) * atom_mask[..., None]
        # place the (A,3) local block in the slot of the residue's amino-acid type, zeros elsewhere
        coord = torch.zeros(B, L, self.max_n_aa_types, A * 3, device=xyz.device, dtype=local.dtype)
        coord.scatter_(2, seq_idx[:, :, None, None].expand(B, L, 1, A * 3), local.reshape(B, L, 1, A * 3))
        coord = coord.reshape(B, L, -1)
        dih = self.dihedral_embedding(dihedrals)
        if structure_context_mask is not None:
            sm = structure_context_mask
            coord = coord * sm[:, :, None]
            dih = dih * (sm & torch.roll(sm, shifts=-1, dims=1))[:, :, None]
        chain = _embed(self.chain_embedding, chain_idx)
        return _run_mlp(self.mlp, torch.cat([aa, coord, dih, chain], dim=-1))


class _RbfFunction(torch.autograd.Function):
    """exp(-softplus(C[pair type]) d^2) * atom-pair mask as ONE pass forward (bf16 out, 232 columns) and one pass
    backward (``dab_rbf_fwd`` / ``dab_rbf_bwd``); gradient w.r.t. the coefficient table only (distances are data)."""

    @staticmethod
    def forward(ctx, distmat, seq_idx, atom_mask, coef, squared):
        B, L = seq_idx.shape
        d = _lib.dev(distmat, torch.float32, "distmat").view(B, L, L, -1)
        s = _lib.dev(seq_idx, torch.int64, "seq_idx")
        m = _lib.mask_u8(atom_mask, "atom_mask")
        c = _lib.dev(coef.detach(), torch.float32, "pair2distcoef.weight")
        if d.shape[-1] != 225 or tuple(c.shape) != (441, 225):
            raise ValueError("fused RBF needs 15 atoms per residue and a (441, 225) coefficient table")
        out = torch.empty(B, L, L, 232, device=d.device, dtype=torch.bfloat16)
        ws = torch.empty(_lib.lib().dab_rbf_workspace_bytes(B, L), device=d.device, dtype=torch.uint8)
        _lib.check(_lib.lib().dab_rbf_fwd(ptr(d), ptr(s), ptr(m), ptr(c), B, L, int(squared), ptr(out), ptr(ws),
                                          ws.numel(), _lib.stream_ptr()), "dab_rbf_fwd")
        ctx.save_for_backward(d, s, m, c)
        ctx.squared = int(squared)
        return out

    @staticmethod
    def backward(ctx, g):
        d, s, m, c = ctx.saved_tensors
        B, L = s.shape
        dc = torch.zeros_like(c)
        g = _lib.dev(g, torch.bfloat16, "grad")
        ws = torch.empty(_lib.lib().dab_rbf_workspace_bytes(B, L), device=d.device, dtype=torch.uint8)
        _lib.check(_lib.lib().dab_rbf_bwd(ptr(g), ptr(d), ptr(s), ptr(m), ptr(c), B, L, ctx.squared, ptr(dc), ptr(ws),
                                          ws.numel(), _lib.stream_ptr()), "dab_rbf_bwd")
        return None, None, None, dc, None


class _PairMlpFunction(torch.autograd.Function):
    """PairEmbedding's two MLPs with bf16 activations and hand-written gradients (mixed-precision training).

    Forward: tensor-core GEMMs with fused bias / ReLU epilogues on bf16 activations (fp32 accumulation).  The first
    mlp layer acts on cat[f_type | f_rel | f_dist | f_dih] (diffab_pytorch.py:307 of the reference): its embedding
    blocks are applied to the TABLES (441 and 65 rows) and ``dab_pair_base_fwd`` turns them, the residue-level index
    vectors and the pairwise dihedrals into the per-pair pre-activation in one pass, so neither the (B, L, L) index
    tensors nor the 210-wide concat exist.
    Backward: every parameter gradient is a bf16 GEMM contracted over the B*L*L pairs with an fp32 result (bias
    gradients included: a GEMM against the 0/1 residue-pair mask); the two embedding tables receive theirs through
    ``dab_pair_table_grad`` (class sums in shared memory) instead of sorting 10^6 indices per table.  Only ``rbf``
    among the inputs carries a gradient (-> ``_RbfFunction`` -> pair2distcoef)."""

    fused_forward = True     # False: the layer-by-layer form of the forward pass (any L; tests compare the two)

    @staticmethod
    def forward(ctx, rbf, dihedrals, seq_idx, residue_idx, chain_idx, res_mask, max_dist, e_type, e_rel, wd1, bd1, wd2,
                bd2, w1, b1, w2, b2, w3, b3):
        bf = torch.bfloat16
        B, L = seq_idx.shape
        P = B * L * L
        D = w2.shape[0]
        lib, st = _lib.lib(), _lib.stream_ptr()
        if D != 64 or w1.shape[1] != 3 * D + 18 or e_type.shape[0] != 441 or e_rel.shape[0] != 2 * max_dist + 1:
            raise ValueError("mixed-precision PairEmbedding needs d_feat = 64, 21 residue types and 2 pairwise dihedrals")
        seq_idx = _lib.dev(seq_idx, torch.int64, "seq_idx")
        residue_idx = _lib.dev(residue_idx, torch.int64, "residue_idx")
        chain_idx = _lib.dev(chain_idx, torch.int64, "chain_idx")
        res_mask = _lib.mask_u8(res_mask, "residue mask")
        x0 = rbf.reshape(P, -1)
        kpad = x0.shape[1] - wd1.shape[1]
        wd1p = F.pad(wd1, (0, kpad)).to(bf)
        a1 = torch._addmm_activation(bd1.to(bf), x0, wd1p.t())                     # relu(rbf Wd1^T + bd1)
        t_type = (e_type @ w1[:, :D].t() + b1).to(bf)                               # (441, D): W1 on the table, bias folded in
        t_rel = (e_rel @ w1[:, D:2 * D].t()).to(bf)                                 # (65, D)
        dih = _lib.dev(dihedrals, torch.float32, "pairwise_dihedrals")
        xh = torch.empty(P, 32, device=rbf.device, dtype=bf)
        if L == 128 and max_dist == 32 and _PairMlpFunction.fused_forward:
            # everything behind the first distance layer in ONE kernel (csrc/pair_mlp_fwd_sm100.cu): reads a1 once and
            # writes fd, h1, h2, out and the angular features once; the per-pair base row of h1 never exists in HBM
            w5 = torch.stack([wd2, w1[:, 2 * D:3 * D], F.pad(w1[:, 3 * D:], (0, D - (w1.shape[1] - 3 * D))), w2, w3]).to(bf)
            bias3 = torch.stack([bd2, b2, b3]).float()
            fd, h1, h2, out = (torch.empty(P, D, device=rbf.device, dtype=bf) for _ in range(4))
            _lib.check(lib.dab_pair_mlp_fwd_train_sm100(
                ptr(a1), ptr(dih), ptr(seq_idx), ptr(residue_idx), ptr(chain_idx), ptr(res_mask), ptr(t_type), ptr(t_rel),
                ptr(w5.contiguous()), ptr(bias3.contiguous()), B, L, max_dist, ptr(fd), ptr(h1), ptr(h2), ptr(out), ptr(xh),
                st), "dab_pair_mlp_fwd_train_sm100")
        else:
            fd = torch._addmm_activation(bd2.to(bf), a1, wd2.to(bf).t())            # f_dist
            base = torch.empty(P, D, device=rbf.device, dtype=bf)
            _lib.check(lib.dab_pair_base_fwd(ptr(seq_idx), ptr(residue_idx), ptr(chain_idx), ptr(dih), ptr(t_type), ptr(t_rel),
                                             B, L, max_dist, ptr(base), ptr(xh), st), "dab_pair_base_fwd")
            w1h = F.pad(w1[:, 3 * D:], (0, xh.shape[1] - (w1.shape[1] - 3 * D))).to(bf)
            h1 = base.addmm_(fd, w1[:, 2 * D:3 * D].to(bf).t()).addmm_(xh, w1h.t()).relu_()
            h2 = torch._addmm_activation(b2.to(bf), h1, w2.to(bf).t())
            out = torch.addmm(b3.to(bf), h2, w3.to(bf).t())
            # `* pair_mask` (:309-311): masked rows of the output are zeroed, and so are those of h2 - its only other use is
            # the backward pass, where zero rows switch the whole pair off (ReLU backward, weight-gradient contractions)
            _lib.check(lib.dab_pair_zero_masked(ptr(out), ptr(res_mask), B, L, st), "dab_pair_zero_masked")
            _lib.check(lib.dab_pair_zero_masked(ptr(h2), ptr(res_mask), B, L, st), "dab_pair_zero_masked")
        ctx.save_for_backward(x0, xh, a1, fd, h1, h2, seq_idx, residue_idx, chain_idx, res_mask, e_type, e_rel, wd1p, wd2,
                              w1, w2, w3)
        ctx.kpad, ctx.max_dist = kpad, max_dist
        return out.view(B, L, L, D)

    @staticmethod
    def backward(ctx, g):
        bf, f32 = torch.bfloat16, torch.float32
        (x0, xh, a1, fd, h1, h2, seq_idx, residue_idx, chain_idx, res_mask, e_type, e_rel, wd1p, wd2, w1, w2,
         w3) = ctx.saved_tensors
        B, L = seq_idx.shape
        P, D = h2.shape
        lib, st = _lib.lib(), _lib.stream_ptr()
        mm32 = lambda a, b: torch.mm(a, b, out_dtype=f32)

        def wgrad_t(act, grad):
            """(grad^T act)^T = act^T grad, [act columns, 64] fp32: the library's weight-gradient GEMM, both operands read
            as they lie in memory (one row per pair)."""
            if P % 64 != 0:
                return mm32(act.t(), grad)
            out = torch.empty(act.shape[1], D, device=g.device, dtype=f32)
            _lib.check(lib.dab_gemm_bf16_tn(ptr(act), act.shape[1], ptr(grad), D, ptr(out), D, act.shape[1], D, P, st),
                       "dab_gemm_bf16_tn")
            return out

        # The four 64-channel layers: weight, bias and data gradient of a layer (and the ReLU before it) in ONE pass over
        # the pairs each (dab_pair_mlp_bwd_layer_sm100) - g and the layer input are read once, the next gradient written once.
        acc = torch.zeros(4 * D * D + 5 * D, device=g.device, dtype=f32)      # one fill: dW of the four layers, five biases
        dWs, dbs = acc[:4 * D * D].view(4, D, D), acc[4 * D * D:].view(5, D)

        def layer_bwd(k, grad, act_in, w, mask=None, db_prev=None):
            g_prev = torch.empty_like(act_in)
            _lib.check(lib.dab_pair_mlp_bwd_layer_sm100(ptr(grad), ptr(act_in), ptr(w.to(bf).contiguous()), ptr(mask), B, L,
                                                        ptr(g_prev), ptr(dWs[k]), ptr(dbs[k]), ptr(db_prev), st),
                       "dab_pair_mlp_bwd_layer_sm100")
            return g_prev

        g3 = _lib.dev(g.reshape(P, D), bf, "grad")         # masked pairs: rows of h2 are zero, the kernel leaves them out of d_b3
        g2 = layer_bwd(0, g3, h2, w3, mask=res_mask)
        g1 = layer_bwd(1, g2, h1, w2)
        del g2
        gd2 = layer_bwd(2, g1, fd, w1[:, 2 * D:3 * D])
        d_w3, d_b3, d_w2, d_b2, d_b1 = dWs[0], dbs[0], dWs[1], dbs[1], dbs[2]
        d_w1 = torch.empty_like(w1)
        d_w1[:, 2 * D:3 * D] = dWs[2]
        d_w1[:, 3 * D:] = wgrad_t(xh, g1).t()[:, :w1.shape[1] - 3 * D]
        # embedding tables: S_type[s_i*21 + s_j] / S_rel[offset] = class sums of g1 over the pairs
        s_type = torch.zeros(e_type.shape[0], D, device=g.device, dtype=f32)
        s_rel = torch.zeros(e_rel.shape[0], D, device=g.device, dtype=f32)
        if L == 128 and ctx.max_dist <= 63:      # one-hot GEMMs on the tensor cores (csrc/pair_table_grad_sm100.cu)
            _lib.check(lib.dab_pair_table_grad_sm100(ptr(g1), ptr(seq_idx), ptr(residue_idx), ptr(chain_idx), B, L,
                                                     ctx.max_dist, ptr(s_type), ptr(s_rel), st), "dab_pair_table_grad_sm100")
        else:
            ws = torch.empty(lib.dab_pair_table_grad_workspace_bytes(B, L, ctx.max_dist) // 4, device=g.device, dtype=f32)
            _lib.check(lib.dab_pair_table_grad(ptr(g1), ptr(seq_idx), ptr(residue_idx), ptr(chain_idx), B, L, ctx.max_dist,
                                               ptr(s_type), ptr(s_rel), ptr(ws), ws.numel() * 4, st), "dab_pair_table_grad")
        d_w1[:, :D] = s_type.t() @ e_type
        d_w1[:, D:2 * D] = s_rel.t() @ e_rel
        d_type, d_rel = s_type @ w1[:, :D], s_rel @ w1[:, D:2 * D]
        del g1
        gd1 = layer_bwd(3, gd2, a1, wd2, db_prev=dbs[4])
        del gd2
        d_wd2, d_bd2, d_bd1 = dWs[3], dbs[3], dbs[4]
        d_wd1 = wgrad_t(x0, gd1).t()[:, :x0.shape[1] - ctx.kpad]
        d_rbf = torch.mm(gd1, wd1p).view(B, L, L, -1) if ctx.needs_input_grad[0] else None
        return (d_rbf, None, None, None, None, None, None, d_type, d_rel, d_wd1, d_bd1, d_wd2, d_bd2, d_w1, d_b1, d_w2,
                d_b2, d_w3, d_b3)


class PairEmbedding(nn.Module):
    """diffab_pytorch.py:186-312.  The two in-place ``distmat *= mask`` lines (:296,:301) do not
    affect the forward result (``dist_feat`` is computed before them) and break autograd in the
    reference (SURVEY F5a); they are dropped, which is forward-identical."""

    def __init__(self, max_n_atoms_per_residue, d_feat, max_dist_to_consider=32):
        super().__init__()
        self.d_feat = d_feat
        self.max_dist_to_consider = max_dist_to_consider
        self.max_n_aa_types = 21
        self.aa_pair_type_embedding = nn.Embedding(self.max_n_aa_types**2, d_feat)
        self.relpos_embedding = nn.Embedding(2 * max_dist_to_consider + 1, d_feat)
        self.pair2distcoef = nn.Embedding(self.max_n_aa_types**2, max_n_atoms_per_residue**2)
        nn.init.zeros_(self.pair2distcoef.weight)
        self.distance_embedding = _mlp([max_n_atoms_per_residue**2, d_feat, d_feat], final_relu=True)
        self.dihedral_embedding = AngularEncoding(2)
        d_dihedral = self.dihedral_embedding.get_output_dimension(2)
        self.mlp = _mlp([3 * d_feat + d_dihedral, d_feat, d_feat, d_feat])

    def fused_supported(self, L, A):
        """Shapes the fused tcgen05 kernel (csrc/pair_embed_sm100.cu) covers."""
        return (L in (128, 256) and A == 15 and self.d_feat == 64 and self.max_dist_to_consider == 32 and
                self.pair2distcoef.weight.shape[1] == 225)

    @torch.no_grad()
    def forward_fused_bf16(self, seq_idx, xyz, dihedrals, residue_idx, chain_idx, atom_mask, sequence_context_mask):
        """The whole module in one kernel, distances computed from ``xyz`` on the fly, output in bf16 (sampling)."""
        B, L = seq_idx.shape
        A = xyz.shape[2]
        if sequence_context_mask is not None:
            seq_idx = torch.where(sequence_context_mask.bool(), seq_idx, torch.full_like(seq_idx, AA_UNK))
        lib = _lib.lib()
        ws = (self.aa_pair_type_embedding.weight, self.relpos_embedding.weight, self.pair2distcoef.weight,
              self.distance_embedding[0].weight, self.distance_embedding[0].bias, self.distance_embedding[2].weight,
              self.distance_embedding[2].bias, self.mlp[0].weight, self.mlp[0].bias, self.mlp[2].weight,
              self.mlp[2].bias, self.mlp[4].weight, self.mlp[4].bias)
        key = _lib.weight_key(ws)
        if getattr(self, "_packed", None) is None or self._packed[0] != key:
            buf = _lib.aligned_empty(lib.dab_pair_embed_packed_bytes(), xyz.device)
            wd = [_lib.dev(w.detach(), torch.float32, "pair embedding weight") for w in ws]
            st = _lib.DabPairEmbedWeights(*(w.data_ptr() for w in wd))
            _lib.check(lib.dab_pair_embed_pack_weights(ctypes.byref(st), ptr(buf), _lib.stream_ptr()),
                       "dab_pair_embed_pack_weights")
            self._packed = (key, buf)
        out = torch.empty(B, L, L, self.d_feat, device=xyz.device, dtype=torch.bfloat16)
        _lib.check(lib.dab_pair_embed_fwd_sm100(
            ptr(self._packed[1]), ptr(_lib.dev(seq_idx, torch.int64, "seq_idx")),
            ptr(_lib.dev(xyz, torch.float32, "xyz")), ptr(_lib.dev(dihedrals, torch.float32, "pairwise_dihedrals")),
            ptr(_lib.dev(residue_idx, torch.int64, "residue_idx")), ptr(_lib.dev(chain_idx, torch.int64, "chain_idx")),
            ptr(_lib.mask_u8(atom_mask, "atom_mask")), B, L, A, ptr(out), _lib.stream_ptr()), "dab_pair_embed_fwd_sm100")
        return out

    def forward(self, seq_idx, distmat, dihedrals, residue_idx, chain_idx, atom_mask, structure_context_mask,
                sequence_context_mask, distmat_is_squared=False):
        B, L = seq_idx.shape
        am = atom_mask
        res_mask = am[:, :, CA_IDX]
        if sequence_context_mask is not None:
            seq_idx = torch.where(sequence_context_mask.bool(), seq_idx, torch.full_like(seq_idx, AA_UNK))
        if getattr(self, "fused_rbf", False) and distmat.is_cuda and distmat.shape[-1] * distmat.shape[-2] == 225:
            # Mixed-precision training.  (1) The six (B, L, L, 225) passes collapse into one kernel each way; the first
            # distance layer then runs as an aligned bf16 GEMM (K padded 225 -> 232) with fp32 accumulation.
            rbf = _RbfFunction.apply(distmat, seq_idx, atom_mask, self.pair2distcoef.weight, distmat_is_squared)
            # (2) Both MLPs on bf16 activations with hand-written gradients (_PairMlpFunction); the result is the bf16
            # pair tensor the tensor-core IPA layers stream.
            de, mlp = self.distance_embedding, self.mlp
            return _PairMlpFunction.apply(
                rbf, dihedrals, seq_idx, residue_idx, chain_idx, res_mask, self.max_dist_to_consider,
                self.aa_pair_type_embedding.weight, self.relpos_embedding.weight, de[0].weight, de[0].bias, de[2].weight,
                de[2].bias, mlp[0].weight, mlp[0].bias, mlp[2].weight, mlp[2].bias, mlp[4].weight, mlp[4].bias)
        res_pair = res_mask[:, :, None] * res_mask[:, None, :]
        pair_type = seq_idx[:, :, None] * self.max_n_aa_types + seq_idx[:, None, :]
        # note: the reference multiplies by the PRODUCT of chain indices, not an equality mask (:279,285)
        chain_prod = chain_idx[:, :, None] * chain_idx[:, None, :]
        rel = (residue_idx[:, :, None] - residue_idx[:, None, :]).clamp(-self.max_dist_to_consider,
                                                                         self.max_dist_to_consider)
        f_type = self.aa_pair_type_embedding(pair_type)
        f_rel = self.relpos_embedding(rel + self.max_dist_to_consider) * chain_prod[..., None]
        coef = F.softplus(self.pair2distcoef(pair_type))
        d = distmat.flatten(-2)
        d2 = d if distmat_is_squared else d**2   # sample() hands over squared distances it computed itself
        atom_pair = (am[:, :, None, :, None] * am[:, None, :, None, :]).flatten(-2)
        f_dist = self.distance_embedding(torch.exp(-1 * coef * d2) * atom_pair)
        f_dih = self.dihedral_embedding(dihedrals)
        return self.mlp(torch.cat([f_type, f_rel, f_dist, f_dih], dim=-1)) * res_pair[..., None]


# =============================================================================================
# Invariant point attention
# =============================================================================================
def euclidean_transform(x, r, t):
    """diffab_pytorch.py:315-324: (b,n,l,p,3) local points -> global, row vectors: x @ R + t."""
    return torch.einsum("bnlpk,blkc->bnlpc", x, r) + t[:, None, :, None, :]


def inverse_euclidean_transform(x, r, t):
    """diffab_pytorch.py:327-336: (x - t) @ R^T."""
    return torch.einsum("bnlpk,blck->bnlpc", x - t[:, None, :, None, :], r)


FAST_L = 128   # patch length of the tensor-core kernels (keys sit on the 128 TMEM lanes)
FAST_L2 = 256  # inference only: two blocks of 128 (block-wise projections, the core per (query block, key block), merged)


def _fast_len(L, inference):
    """Length a patch of L residues is padded to for the tensor-core kernels (None: not covered)."""
    if L <= FAST_L:
        return FAST_L
    return FAST_L2 if inference and L <= FAST_L2 else None


def _pad_patch(x, e, r, t, planes, L_to, make_planes):
    """Pad a patch batch of L < L_to residues to the tensor-core kernels' length: zero residues / pair rows, identity
    frames, and the pair-bias planes (one per layer; None: ``make_planes`` builds them from the padded pair tensor) with
    the padded keys masked.  Differentiable (F.pad / cat), so gradients reach the unpadded tensors."""
    L = x.shape[1]
    n = L_to - L
    xp = F.pad(x, (0, 0, 0, n))
    ep = F.pad(e, (0, 0, 0, n, 0, n))
    eye = torch.eye(3, device=r.device, dtype=r.dtype).expand(r.shape[0], n, 3, 3)
    rp, tp = torch.cat([r, eye], dim=1), F.pad(t, (0, 0, 0, n))
    with torch.no_grad():
        planes = make_planes(ep.detach()) if planes is None else [F.pad(p_, (0, 0, 0, n, 0, n)) for p_ in planes]
        _mask_padded_keys(planes, L)
    return xp, ep, rp, tp, planes


def _mask_padded_keys(planes, L):
    """Pair-bias planes (.., L_pad(i), L_pad(j), H) of a padded batch: keys j >= L get -inf, so their probability is exactly
    zero - the layer then computes what the reference computes on the L real residues (it has no masks of its own)."""
    for p_ in planes:
        p_[:, :, L:, :] = float("-inf")
    return planes


_SIDE_STREAMS = {}


def _side_stream(device, which=0):
    """Auxiliary streams (per device) for the independent branches of the backward."""
    key = (torch.device(device).index, which)
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _SIDE_STREAMS[key]


def _ipa_structs(layer, B, L):
    dims = _lib.DabIpaDims(B, L, layer.d_residue_emb, layer.d_pair_emb, layer.n_head, layer.d_scalar_per_head,
                           layer.n_query_point_per_head, layer.n_value_point_per_head)
    return dims


def _weights_struct(tensors):
    return _lib.DabIpaWeights(*(t.data_ptr() for t in tensors))


def _fwd_stages(dims, packed, x, e, bias, r, t, y, ws, stages, st):
    """``dab_ipa_fwd_sm100_stages`` with the residue stream x / y in fp32, or in bf16 when that is their dtype."""
    x32, x16 = (None, x) if x.dtype == torch.bfloat16 else (x, None)
    y32, y16 = (None, y) if y.dtype == torch.bfloat16 else (y, None)
    _lib.check(_lib.lib().dab_ipa_fwd_sm100_stages(ctypes.byref(dims), ptr(packed), ptr(x32), ptr(x16), ptr(e), ptr(bias),
                                                   ptr(r), ptr(t), ptr(y32), ptr(y16), ptr(ws), ws.numel(), stages, st),
               "dab_ipa_fwd_sm100_stages")


def live_query_tiles(generation_mask, out=None):
    """The 16-row query tiles (tile = row / 16 of the flattened B x L rows) that hold a generated residue, on the device and
    without a host synchronisation: (int32 tile ids, the live ones first in ascending order; int32 (1,) their count).
    Sampling computes the last IPA layer's attention core and the heads on these tiles only: the reverse update keeps
    every other residue as it is.  ``out`` = a previous result, refilled in place (static buffers of a captured graph)."""
    flags = generation_mask.reshape(-1, 16).ne(0).any(-1)
    tiles = torch.argsort((~flags).to(torch.int32), stable=True).to(torch.int32)
    count = flags.sum(dtype=torch.int32).view(1)
    if out is None:
        return tiles, count
    out[0].copy_(tiles)
    out[1].copy_(count)
    return out


def aa_bias_weights(aa_bias, generation_mask, generate_sequence=True):
    """The per-type weights of the sequence draw, (B, L, 21) fp32 on ``generation_mask``'s device, from ``aa_bias`` (see
    ``DiffAb.sample``): ``w = exp(b - max_k b)``, so ``w`` is in [0, 1], exactly 0 where ``b = -inf`` and all ones for a
    bias that is constant over the types.  None stays None.  Raises ``ValueError`` on NaN or +inf, on a shape that does
    not broadcast to (B, L, 21), on a generated residue with every type at -inf, and when the sequence is not generated
    (``generate_sequence`` False: the bias would do nothing)."""
    if aa_bias is None:
        return None
    if not generate_sequence:
        raise ValueError("aa_bias: this design mode does not generate the sequence (generate_sequence is False)")
    B, L = generation_mask.shape
    b = torch.as_tensor(aa_bias, device=generation_mask.device)
    b = b.to(torch.promote_types(b.dtype, torch.float32))
    try:
        b = b.expand(B, L, 21)
    except RuntimeError:
        raise ValueError(f"aa_bias: shape {tuple(b.shape)} does not broadcast to (B, L, 21) = {(B, L, 21)}") from None
    if bool((torch.isnan(b) | (b == float("inf"))).any()):
        raise ValueError("aa_bias: NaN or +inf (use -inf to forbid a type, finite values to bias it)")
    if bool(((b == float("-inf")).all(-1) & generation_mask.bool()).any()):
        raise ValueError("aa_bias: a generated residue has every residue type at -inf")
    # a row at -inf throughout (a context residue) gets w = 0 instead of exp(-inf + inf) = NaN
    mx = b.amax(-1, keepdim=True).clamp_min(torch.finfo(b.dtype).min)
    return torch.exp(b - mx).to(torch.float32).contiguous()


def _pair_bias_planes(layers, e, out):
    """The pair-bias planes of ``layers`` into ``out`` (fp16 (n_layers, B, L, L, H), contiguous) from the bf16 pair
    tensor ``e``: one pass over it per six layers."""
    dims = _ipa_structs(layers[0], e.shape[0], e.shape[1])
    for lo in range(0, len(layers), 6):   # the kernel takes up to six layers per pass
        hi = min(len(layers), lo + 6)
        ws = [_lib.dev(l.to_pair_bias.weight.detach(), torch.float32, "to_pair_bias.weight") for l in layers[lo:hi]]
        w = ws[0] if len(ws) == 1 else torch.stack(ws)
        _lib.check(_lib.lib().dab_ipa_pair_bias_multi(ctypes.byref(dims), ptr(e), ptr(w), hi - lo, ptr(out[lo:hi]),
                                                      _lib.stream_ptr()), "dab_ipa_pair_bias_multi")


class _IpaFunction(torch.autograd.Function):
    """fp32 IPA layer: ``dab_ipa_fwd_f32`` / ``dab_ipa_bwd_f32``."""

    @staticmethod
    def forward(ctx, layer, need_bwd, x, e, r, t, *weights):
        x = _lib.dev(x, torch.float32, "x")
        e = _lib.dev(e, torch.float32, "e")
        r = _lib.dev(r, torch.float32, "r")
        t = _lib.dev(t, torch.float32, "t")
        weights = tuple(_lib.dev(w.detach(), torch.float32, "weight") for w in weights)
        B, L, D = x.shape
        if e.shape != (B, L, L, layer.d_pair_emb) or r.shape != (B, L, 3, 3) or t.shape != (B, L, 3):
            raise ValueError(f"IPA shape mismatch: x {tuple(x.shape)} e {tuple(e.shape)} r {tuple(r.shape)} t {tuple(t.shape)}")
        dims = _ipa_structs(layer, B, L)
        lib = _lib.lib()
        nbytes = lib.dab_ipa_f32_workspace_bytes(ctypes.byref(dims), 1 if need_bwd else 0)
        if need_bwd:   # kept for the backward pass: must be private to this call
            ws = torch.empty(max(nbytes, 16) // 4, device=x.device, dtype=torch.float32)
        else:          # inference: one persistent workspace per layer (stable address, graph friendly)
            ws = layer._workspace(max(nbytes, 16), x.device).view(torch.float32)
        y = torch.empty(B, L, D, device=x.device, dtype=torch.float32)
        wstruct = _weights_struct(weights)
        _lib.check(lib.dab_ipa_fwd_f32(ctypes.byref(dims), ctypes.byref(wstruct), ptr(x), ptr(e), ptr(r), ptr(t),
                                       ptr(y), ptr(ws), ws.numel() * 4, int(need_bwd), _lib.stream_ptr()),
                   "dab_ipa_fwd_f32")
        if need_bwd:
            ctx.save_for_backward(x, e, r, t, ws, *weights)
            ctx.layer = layer
        return y

    @staticmethod
    def backward(ctx, dy):
        x, e, r, t, ws, *weights = ctx.saved_tensors
        layer = ctx.layer
        if ctx.needs_input_grad[4] or ctx.needs_input_grad[5]:
            raise NotImplementedError("gradients w.r.t. the frames (r, t) are not provided: in DiffAb they are the "
                                      "noised frames and carry no gradient (diffab_pytorch.py:824-854)")
        B, L, D = x.shape
        dims = _ipa_structs(layer, B, L)
        dy = _lib.dev(dy, torch.float32, "dy")
        dx = torch.empty_like(x)
        de = torch.empty_like(e)
        grads = [torch.zeros_like(w) for w in weights]
        wstruct = _weights_struct(weights)
        gstruct = _lib.DabIpaGrads(*(g.data_ptr() for g in grads))
        _lib.check(_lib.lib().dab_ipa_bwd_f32(ctypes.byref(dims), ctypes.byref(wstruct), ptr(x), ptr(e), ptr(r),
                                              ptr(t), ptr(dy), ptr(dx), ptr(de), ctypes.byref(gstruct), ptr(ws),
                                              ws.numel() * 4, _lib.stream_ptr()), "dab_ipa_bwd_f32")
        return (None, None, dx, de, None, None, *grads)


class _PairFanOut(torch.autograd.Function):
    """The bf16 pair tensor handed to n layers as n aliases: the n gradients come back together and are summed in ONE
    pass with fp32 accumulation (``dab_sum_bf16``) instead of autograd's n - 1 pairwise bf16 adds."""

    @staticmethod
    def forward(ctx, e, n):
        return tuple(e.view_as(e) for _ in range(n))

    @staticmethod
    def backward(ctx, *grads):
        gs = [_lib.dev(g, torch.bfloat16, "pair gradient") for g in grads if g is not None]
        if not gs:
            return None, None
        if len(gs) == 1:
            return gs[0], None
        out = torch.empty_like(gs[0])
        total = None
        for lo in range(0, len(gs), 7):       # up to 8 sources per launch (the running total is one of them)
            part = ([total] if total is not None else []) + gs[lo:lo + 7]
            ptrs = (ctypes.c_void_p * len(part))(*(t.data_ptr() for t in part))
            _lib.check(_lib.lib().dab_sum_bf16(ptrs, len(part), out.numel(), ptr(out), _lib.stream_ptr()), "dab_sum_bf16")
            total = out
        return out, None


class _IpaFastFunction(torch.autograd.Function):
    """bf16 tensor-core IPA layer with gradients: ``dab_ipa_fwd_sm100_train`` / ``dab_ipa_bwd_sm100_main`` + ``_finish``.
    Every GEMM of the backward runs in the library's tcgen05 kernels too: the data gradients through ``to_out`` and the
    six projections on the K-major GEMM (``dab_linear_bf16``), the weight gradients on the MN-major split-K GEMM
    (``dab_gemm_bf16_tn``) - bf16 operands, fp32 accumulation."""

    @staticmethod
    def forward(ctx, layer, pair_bias, x, e, r, t, *weights):
        x = _lib.dev(x, torch.float32, "x")
        e = _lib.dev(e, torch.bfloat16, "e")
        r = _lib.dev(r, torch.float32, "r")
        t = _lib.dev(t, torch.float32, "t")
        B, L, D = x.shape
        dims = _ipa_structs(layer, B, L)
        lib = _lib.lib()
        packed = layer._packed_weights(dims)
        nbytes = lib.dab_ipa_sm100_workspace_bytes(ctypes.byref(dims))
        saved = _lib.aligned_empty(max(nbytes, 16), x.device)   # private: kept for the backward
        y = torch.empty(B, L, D, device=x.device, dtype=torch.float32)
        if pair_bias is not None:
            pair_bias = _lib.dev(pair_bias, torch.float16, "pair_bias")
            if tuple(pair_bias.shape) != (B, L, L, layer.n_head):
                raise ValueError(f"pair_bias shape {tuple(pair_bias.shape)} != {(B, L, L, layer.n_head)}")
        _lib.check(lib.dab_ipa_fwd_sm100_train(ctypes.byref(dims), ptr(packed), ptr(x), ptr(e), ptr(pair_bias), ptr(r),
                                               ptr(t), ptr(y), ptr(saved), saved.numel(), _lib.stream_ptr()),
                   "dab_ipa_fwd_sm100_train")
        ctx.save_for_backward(x, e, r, saved, packed, *[w.detach() for w in weights])
        ctx.layer = layer
        return y

    @staticmethod
    def backward(ctx, dy):
        x, e, r, saved, packed, *weights = ctx.saved_tensors
        layer = ctx.layer
        if ctx.needs_input_grad[4] or ctx.needs_input_grad[5]:
            raise NotImplementedError("gradients w.r.t. the frames (r, t) are not provided: in DiffAb they are the "
                                      "noised frames and carry no gradient (diffab_pytorch.py:824-854)")
        B, L, D = x.shape
        M = B * L
        dims = _ipa_structs(layer, B, L)
        lib = _lib.lib()
        offs = (ctypes.c_size_t * 8)()
        _lib.check(lib.dab_ipa_sm100_workspace_layout(ctypes.byref(dims), offs), "dab_ipa_sm100_workspace_layout")
        w_out = weights[8]
        ncat = w_out.shape[1]
        dev_ = x.device
        bf, f32 = torch.bfloat16, torch.float32
        st = _lib.stream_ptr()
        cat = saved[offs[4]: offs[4] + M * ncat * 2].view(bf).view(M, ncat)
        dy2 = _lib.dev(dy, f32, "dy").view(M, D)
        # bf16 copies of the weights as the forward used them, and their transposes (rows of Wcat: q/k/v scalars, q/k/v points)
        poffs = (ctypes.c_size_t * 7)()
        _lib.check(lib.dab_ipa_packed_layout(ctypes.byref(dims), poffs), "dab_ipa_packed_layout")
        n_proj = sum(w.shape[0] for w in weights[:6])
        w_cat_t = packed[poffs[5]: poffs[5] + D * n_proj * 2]        # Wcat^T [D][n_proj] bf16
        w_out_t = packed[poffs[6]: poffs[6] + ncat * D * 2]          # Wout^T [ncat][D] bf16

        def cast(t_):
            out_ = torch.empty(t_.shape, device=dev_, dtype=bf)
            _lib.check(lib.dab_cast_f32_to_bf16(ptr(t_), ptr(out_), t_.numel(), st), "dab_cast_f32_to_bf16")
            return out_

        # The plain GEMMs of the backward all run in the library on bf16 operands with fp32 accumulation and output (the
        # forward ran the same products on bf16 operands): data gradients on the K-major tcgen05 GEMM against the
        # transposed weight copies, weight gradients on the MN-major split-K GEMM straight from the activations.
        # The weight-gradient GEMMs depend only on dy / dproj and the saved activations, and at training batch sizes every
        # kernel of the backward is a single under-filled wave: they run on a side stream beside the main chain
        # (dcat -> prep -> backward core -> key side -> dx) and join before the gradients are returned (fork / join is
        # captured as parallel branches when the step is recorded into a CUDA graph).
        main = torch.cuda.current_stream(dev_)
        side = _side_stream(dev_)
        side2 = _side_stream(dev_, 1)
        dy_bf = torch.empty(M, D, device=dev_, dtype=bf)
        d_b_out = torch.empty(D, device=dev_, dtype=f32)
        d_w_out = torch.empty(D, ncat, device=dev_, dtype=f32)
        d_w_cat = torch.empty(n_proj, D, device=dev_, dtype=f32)
        zeros = torch.empty(weights[6].numel() + weights[7].numel(), device=dev_, dtype=f32)
        d_wpb = zeros[: weights[6].numel()].view_as(weights[6])
        d_gamma = zeros[weights[6].numel():].view_as(weights[7])
        x2 = x.view(M, D)
        x_bf = torch.empty(M, D, device=dev_, dtype=bf)
        # Everything that does not feed the main chain starts on the side streams right away: the fills of the split-K
        # accumulators (a fill node between two kernels of a graph costs several microseconds of hand-over), the bias
        # gradient, the bf16 copy of x.  The main chain begins with the one thing dcat needs: the bf16 copy of dy.
        side.wait_stream(main)
        side2.wait_stream(main)
        with torch.cuda.stream(side2):
            zeros.zero_()
            d_w_cat.zero_()
            ev_fill = side2.record_event()
            _lib.check(lib.dab_colsum_f32(ptr(dy2), M, D, ptr(d_b_out), None, _lib.stream_ptr()), "dab_colsum_f32")
        _lib.check(lib.dab_cast_f32_to_bf16(ptr(dy2), ptr(dy_bf), dy2.numel(), st), "dab_cast_f32_to_bf16")
        with torch.cuda.stream(side):
            sst = _lib.stream_ptr()
            d_w_out.zero_()
            _lib.check(lib.dab_cast_f32_to_bf16(ptr(x2), ptr(x_bf), x2.numel(), sst), "dab_cast_f32_to_bf16")
            ev_xbf = side.record_event()
            side.wait_stream(main)      # dy_bf
            _lib.check(lib.dab_gemm_bf16_tn_acc(ptr(dy_bf), D, ptr(cat), ncat, ptr(d_w_out), ncat, D, ncat, M, sst),
                       "dab_gemm_bf16_tn_acc (dWout)")
        dcat = torch.empty(M, ncat, device=dev_, dtype=f32)
        _lib.check(lib.dab_linear_bf16(ptr(dy_bf), ptr(w_out_t), None, 0, M, ncat, D, ptr(dcat), None, st),
                   "dab_linear_bf16 (dcat)")
        dproj = torch.empty(M, n_proj, device=dev_, dtype=bf)
        de = torch.empty_like(e)
        bws = _lib.aligned_empty(max(lib.dab_ipa_bwd_sm100_workspace_bytes(ctypes.byref(dims)), 16), dev_)
        bwd_args = (ctypes.byref(dims), ptr(packed), ptr(e), ptr(r), ptr(dcat), ptr(saved), saved.numel(), ptr(dproj), ptr(de),
                    ptr(d_wpb), ptr(d_gamma), ptr(bws), bws.numel())
        _lib.check(lib.dab_ipa_bwd_sm100_main(*bwd_args, st), "dab_ipa_bwd_sm100_main")
        layer._last_bwd_ws = bws   # kept for tools/debug_bwd.py (intermediate buffers of the last backward)
        # dproj is complete: three independent branches - dx (side), the to_pair_bias / gamma reductions (second side
        # stream), dWcat (main)
        side.wait_stream(main)
        side2.wait_stream(main)
        # the longer of the two GEMMs (dWcat, split over K) continues on the main stream without a stream hand-over
        dx = torch.empty(B, L, D, device=dev_, dtype=f32)
        with torch.cuda.stream(side):
            _lib.check(lib.dab_linear_bf16(ptr(dproj), ptr(w_cat_t), None, 0, M, D, n_proj, ptr(dx), None,
                                           _lib.stream_ptr()), "dab_linear_bf16 (dx)")
        with torch.cuda.stream(side2):
            _lib.check(lib.dab_ipa_bwd_sm100_finish(*bwd_args, _lib.stream_ptr()), "dab_ipa_bwd_sm100_finish")
        main.wait_event(ev_fill)        # the fill of d_w_cat and the bf16 copy of x: long done
        main.wait_event(ev_xbf)
        _lib.check(lib.dab_gemm_bf16_tn_acc(ptr(dproj), n_proj, ptr(x_bf), D, ptr(d_w_cat), D, n_proj, D, M, st),
                   "dab_gemm_bf16_tn_acc (dWcat)")
        main.wait_stream(side)
        main.wait_stream(side2)
        d_proj_w = torch.split(d_w_cat, [w.shape[0] for w in weights[:6]], dim=0)
        return (None, None, dx, de, None, None, *d_proj_w, d_wpb, d_gamma, d_w_out, d_b_out)


class InvariantPointAttentionLayer(nn.Module):
    """diffab_pytorch.py:339-465.  Parameters keep the reference's names and shapes."""

    def __init__(self, d_residue_emb, d_pair_emb, d_scalar_per_head=16, n_query_point_per_head=4,
                 n_value_point_per_head=4, n_head=8, use_pair_bias=True):
        super().__init__()
        self.d_residue_emb, self.d_pair_emb = d_residue_emb, d_pair_emb
        self.d_scalar_per_head = d_scalar_per_head
        self.n_query_point_per_head, self.n_value_point_per_head = n_query_point_per_head, n_value_point_per_head
        self.n_head = n_head
        self.use_pair_bias = use_pair_bias
        d_scalar = d_scalar_per_head * n_head
        self.to_q_scalar = nn.Linear(d_residue_emb, d_scalar, bias=False)
        self.to_k_scalar = nn.Linear(d_residue_emb, d_scalar, bias=False)
        self.to_v_scalar = nn.Linear(d_residue_emb, d_scalar, bias=False)
        self.scale_scalar = d_scalar_per_head**-0.5
        if use_pair_bias:                                                   # :362-363
            self.to_pair_bias = nn.Linear(d_pair_emb, n_head, bias=False)
        d_query_point = n_query_point_per_head * 3 * n_head
        d_value_point = n_value_point_per_head * 3 * n_head
        self.to_q_point = nn.Linear(d_residue_emb, d_query_point, bias=False)
        self.to_k_point = nn.Linear(d_residue_emb, d_query_point, bias=False)
        self.to_v_point = nn.Linear(d_residue_emb, d_value_point, bias=False)
        self.scale_point = (4.5 * n_query_point_per_head) ** -0.5
        self.gamma = nn.Parameter(torch.log(torch.exp(torch.ones(n_head)) - 1.0))  # used raw (:373,429)
        d_pair = d_pair_emb * n_head if use_pair_bias else 0                # :374-383
        self.to_out = nn.Linear(d_scalar + d_pair + d_value_point + n_value_point_per_head * n_head, d_residue_emb)
        self.num_independent_logits = 3 if use_pair_bias else 2            # :385
        self.scale_total = self.num_independent_logits**-0.5
        self._packed = None  # (version key, packed weights) for the sm_100a fast path

    def _workspace(self, nbytes, device):
        ws = getattr(self, "_ws", None)
        if ws is None or ws.numel() < nbytes or ws.device != device:
            ws = _lib.aligned_empty((nbytes + 255) // 256 * 256, device)
            self._ws = ws
        return ws[: (nbytes // 4) * 4]

    # dummy pair width of the use_pair_bias=False re-expression (16-byte rows for the fp32 kernels)
    _NOPB_C = 4

    def _weights_no_pair_bias(self):
        """``use_pair_bias=False`` (:374-387,438-462) expressed EXACTLY on the kernels of the pair-bias layer: a zero pair
        tensor of width 4 and a zero ``to_pair_bias`` contribute nothing to the logits or the features; the kernels' fixed
        scale_total = 3^-1/2 becomes the layer's 2^-1/2 by scaling ``to_q_scalar`` and ``gamma`` (both logit terms are
        linear in them) by sqrt(3/2); ``to_out`` gets zero columns where the (all-zero) pair features sit.  Built from the
        parameters with differentiable PyTorch ops, so autograd carries the kernels' gradients back to them."""
        r = (3.0 / 2.0) ** 0.5
        H, ns = self.n_head, self.d_scalar_per_head * self.n_head
        w_out = self.to_out.weight
        w_out = torch.cat([w_out[:, :ns], w_out.new_zeros(w_out.shape[0], H * self._NOPB_C), w_out[:, ns:]], dim=1)
        return (self.to_q_scalar.weight * r, self.to_k_scalar.weight, self.to_v_scalar.weight, self.to_q_point.weight,
                self.to_k_point.weight, self.to_v_point.weight, w_out.new_zeros(H, self._NOPB_C), self.gamma * r, w_out,
                self.to_out.bias)

    def _weights(self):
        return (self.to_q_scalar.weight, self.to_k_scalar.weight, self.to_v_scalar.weight, self.to_q_point.weight,
                self.to_k_point.weight, self.to_v_point.weight, self.to_pair_bias.weight, self.gamma,
                self.to_out.weight, self.to_out.bias)

    def forward(self, x, e, r, t, pair_bias=None):
        if not self.use_pair_bias:
            # the pair tensor is accepted and unused, as in the reference (:389, :438-441); fp32 kernels
            x = _lib.dev(x, torch.float32, "x")
            B, L = x.shape[0], x.shape[1]
            ws = self._weights_no_pair_bias()
            e0 = x.new_zeros(B, L, L, self._NOPB_C)
            need_bwd = torch.is_grad_enabled() and (x.requires_grad or any(w.requires_grad for w in ws))
            return _IpaFunction.apply(self._nopb_view(), need_bwd, x, e0, r, t, *ws)
        if e.dtype == torch.bfloat16:
            L = x.shape[1]
            no_grad = not (torch.is_grad_enabled() and (x.requires_grad or e.requires_grad or
                                                        any(w.requires_grad for w in self._weights())))
            Lp = _fast_len(L, no_grad)
            if Lp is None or not self.fast_path_supported(Lp, no_grad):
                raise RuntimeError("bf16 pair tensor given but the sm_100a path only supports the train.py configuration "
                                   "(D=128, C=64, H=8, ds=32, Pq=Pv=8; L <= 128, without gradients L <= 256)")
            if L < Lp:
                # shorter patch on the tensor-core kernels: padded to 128 (without gradients: 256) residues, padded keys
                # masked through the bias plane
                x, e, r, t, (pair_bias,) = _pad_patch(x, e, r, t, None if pair_bias is None else [pair_bias], Lp,
                                                      lambda ep: [self.pair_bias(ep)])
            if no_grad:
                y = self.forward_fast_io(x, e, r, t, pair_bias, torch.float32)
            else:
                y = _IpaFastFunction.apply(self, pair_bias, x, e, r, t, *self._weights())
            return y[:, :L] if L < Lp else y
        ws = self._weights()
        need_bwd = torch.is_grad_enabled() and (x.requires_grad or e.requires_grad or r.requires_grad or
                                                t.requires_grad or any(w.requires_grad for w in ws))
        return _IpaFunction.apply(self, need_bwd, x, e, r, t, *ws)

    def _nopb_view(self):
        """What ``_ipa_structs`` / the workspace cache see for the use_pair_bias=False re-expression: this layer with the
        dummy pair width."""
        v = getattr(self, "_nopb", None)
        if v is None:
            v = types.SimpleNamespace(d_residue_emb=self.d_residue_emb, d_pair_emb=self._NOPB_C, n_head=self.n_head,
                                      d_scalar_per_head=self.d_scalar_per_head,
                                      n_query_point_per_head=self.n_query_point_per_head,
                                      n_value_point_per_head=self.n_value_point_per_head, _workspace=self._workspace)
            self._nopb = v
        return v

    # ---- sm_100a fast path (inference; train.py configuration only) ----
    def fast_path_supported(self, L, inference=False):
        """Shapes of the tensor-core kernels: the train.py configuration at L = 128; without gradients also L = 256."""
        return (self.use_pair_bias and (L == FAST_L or (inference and L == FAST_L2)) and self.d_residue_emb == 128 and
                self.d_pair_emb == 64 and self.n_head == 8 and self.d_scalar_per_head == 32 and
                self.n_query_point_per_head == 8 and self.n_value_point_per_head == 8)

    def _packed_weights(self, dims):
        ws = self._weights()
        key = _lib.weight_key(ws)
        # While a training step is being captured into a CUDA graph (distributed.GraphedTrainStep): always repack, so that
        # the pack is part of the graph - its replays follow optimizer steps that no Python-side version counter sees.
        capturing = (_lib.repack_when_capturing and torch.is_grad_enabled() and ws[0].is_cuda
                     and torch.cuda.is_current_stream_capturing())
        if capturing or self._packed is None or self._packed[0] != key:
            lib = _lib.lib()
            nbytes = lib.dab_ipa_packed_bytes(ctypes.byref(dims))
            if self._packed is not None and self._packed[1].device == ws[0].device:
                buf = self._packed[1]          # repack in place (stable address: graph captures keep pointing at it)
            else:
                buf = _lib.aligned_empty(max(nbytes, 16), ws[0].device)
            wstruct = _weights_struct([_lib.dev(w.detach(), torch.float32, "weight") for w in ws])
            _lib.check(lib.dab_ipa_pack_weights(ctypes.byref(dims), ctypes.byref(wstruct), ptr(buf), _lib.stream_ptr()),
                       "dab_ipa_pack_weights")
            self._packed = (key, buf)
        return self._packed[1]

    def pair_bias(self, e_bf16, out=None):
        """This layer's pair bias for every (i, j) as fp16 (B, L, L, H), scale_total and log2(e) folded in.
        The pair tensor is constant over the sampling loop, so ``DiffAb.sample`` computes this once per run."""
        e = _lib.dev(e_bf16, torch.bfloat16, "e")
        B, L = e.shape[0], e.shape[1]
        if out is None:
            out = torch.empty(B, L, L, self.n_head, device=e.device, dtype=torch.float16)
        elif out.dtype != torch.float16 or tuple(out.shape) != (B, L, L, self.n_head) or not out.is_contiguous():
            raise ValueError("pair_bias: `out` must be a contiguous fp16 (B, L, L, H) tensor")
        _pair_bias_planes([self], e, out[None])
        return out

    @torch.no_grad()
    def forward_fast_io(self, x, e_bf16, r, t, pair_bias, out_dtype):
        """Inference on the sm_100a path with the residue stream in fp32 or bf16 on either side (``x.dtype`` /
        ``out_dtype``): the layers of a stack hand it over already rounded to bf16 - what the next layer's projections
        consume anyway, so no bit of the result changes.  ``pair_bias`` None: the library builds this layer's plane."""
        B, L, D = x.shape
        if not self.fast_path_supported(L, True):
            raise RuntimeError("the sm_100a fast path only supports the train.py configuration")
        x = _lib.dev(x, x.dtype if x.dtype == torch.bfloat16 else torch.float32, "x")
        e = _lib.dev(e_bf16, torch.bfloat16, "e")
        r = _lib.dev(r, torch.float32, "r")
        t = _lib.dev(t, torch.float32, "t")
        bias = None if pair_bias is None else _lib.dev(pair_bias, torch.float16, "pair_bias")
        if bias is not None and tuple(bias.shape) != (B, L, L, self.n_head):
            raise ValueError(f"pair_bias shape {tuple(bias.shape)} != {(B, L, L, self.n_head)}")
        dims = _ipa_structs(self, B, L)
        packed = self._packed_weights(dims)
        ws = self._workspace(max(_lib.lib().dab_ipa_sm100_workspace_bytes(ctypes.byref(dims)), 16), x.device)
        y = torch.empty(B, L, D, device=x.device, dtype=out_dtype)
        if B > 0:   # (an empty tensor's data pointer is NULL: the library would read x / y as not given)
            _fwd_stages(dims, packed, x, e, bias, r, t, y, ws, 7, _lib.stream_ptr())
        return y


class InvariantPointAttentionModule(nn.Module):
    """diffab_pytorch.py:468-498: plain chain, same (pair_emb, R, t) for every layer."""

    def __init__(self, n_layers, d_residue_emb, d_pair_emb, d_scalar_per_head, n_query_point_per_head,
                 n_value_point_per_head, n_head):
        super().__init__()
        self.layers = nn.ModuleList([
            InvariantPointAttentionLayer(d_residue_emb, d_pair_emb, d_scalar_per_head, n_query_point_per_head,
                                         n_value_point_per_head, n_head) for _ in range(n_layers)])

    def forward(self, res_emb, pair_emb, orientations, translations, pair_bias=None):
        L = res_emb.shape[1]
        needs_grad = torch.is_grad_enabled() and (res_emb.requires_grad or pair_emb.requires_grad or
                                                  any(p.requires_grad for p in self.parameters()))
        Lp = _fast_len(L, not needs_grad)
        if (pair_emb.dtype == torch.bfloat16 and Lp is not None and L < Lp and
                self.layers[0].fast_path_supported(Lp, not needs_grad)):
            # shorter patches on the tensor-core kernels: pad once for the whole stack (to 128, without gradients to 256
            # residues), mask the padded keys in every layer's bias plane, slice the result
            padded = _pad_patch(res_emb, pair_emb, orientations, translations, pair_bias, Lp, self.precompute_pair_bias)
            return self.forward(*padded)[:, :L]
        if (pair_bias is None and pair_emb.dtype == torch.bfloat16 and
                self.layers[0].fast_path_supported(pair_emb.shape[1], not needs_grad)):
            # tensor-core path: the bias planes of all layers in one pass over the pair tensor (their gradient
            # w.r.t. to_pair_bias and the pair tensor is produced by the layers' own backward kernels)
            pair_bias = self.precompute_pair_bias(pair_emb.detach())
        if (not needs_grad and pair_bias is not None and pair_emb.dtype == torch.bfloat16 and len(self.layers) > 1 and
                self.layers[0].fast_path_supported(pair_emb.shape[1], True)):
            # inference on the tensor-core path: the residue stream travels between the layers as bf16
            n = len(self.layers)
            if self.fused_stack_applicable(res_emb.shape[0], L, pair_emb, pair_bias):
                # large batches (one projection CTA per patch): each layer's to_out is fused into the next layer's
                # projection kernel, the stream between the layers never exists in HBM (bit-identical)
                return self._forward_fused_stack(res_emb, pair_emb, orientations, translations, pair_bias)
            for k, layer in enumerate(self.layers):
                res_emb = layer.forward_fast_io(res_emb, pair_emb, orientations, translations, pair_bias[k],
                                                torch.float32 if k == n - 1 else torch.bfloat16)
            return res_emb
        pairs = [pair_emb] * len(self.layers)
        if (pair_emb.is_cuda and pair_emb.dtype == torch.bfloat16 and pair_emb.requires_grad and torch.is_grad_enabled()
                and pair_emb.numel() % 8 == 0 and len(self.layers) > 1):
            pairs = _PairFanOut.apply(pair_emb, len(self.layers))    # one fused sum of the layers' pair gradients
        for k, layer in enumerate(self.layers):
            if pair_bias is not None:
                res_emb = layer(res_emb, pairs[k], orientations, translations, pair_bias[k])
            else:
                res_emb = layer(res_emb, pairs[k], orientations, translations)
        return res_emb

    def fused_stack_applicable(self, B, L, pair_emb, pair_bias):
        """Inference on the tensor-core path with enough 128-residue blocks for one projection CTA per block."""
        return (pair_bias is not None and pair_emb.dtype == torch.bfloat16 and len(self.layers) > 1 and
                self.layers[0].fast_path_supported(L, True) and B * (L // FAST_L) >= 128)

    @torch.no_grad()
    def _forward_fused_stack(self, res_emb, pair_emb, orientations, translations, pair_bias, front=None, heads=None,
                             live=None):
        """The layer stack launch by launch on ONE shared workspace: projections of layer 0, then per layer the attention
        core followed by ``dab_ipa_mid_sm100`` (its to_out + the next layer's projections in one kernel), to_out of the
        last layer.  2 n launches instead of 3 n; results bit-identical to ``forward_fast_io`` layer by layer.
        ``front`` = (sampling cache of the Denoiser, seq_idx_t) instead of ``res_emb``: the epsilon network's front MLP
        runs inside the first projection kernel (``dab_ipa_front_proj_sm100``).  ``heads`` = (packed head weights, beta per
        block): the last layer's to_out runs inside the heads kernel (``dab_out_heads_fwd_sm100``) and the call returns
        (eps, rotvec, posterior) instead of the stack's output.  ``live`` (``live_query_tiles``): the last layer's attention
        core and the heads compute only the rows of these tiles, the other rows of the result are undefined."""
        layers = self.layers
        n = len(layers)
        e = _lib.dev(pair_emb, torch.bfloat16, "e")
        B, L = e.shape[0], e.shape[1]
        D = layers[0].d_residue_emb
        r = _lib.dev(orientations, torch.float32, "r")
        t = _lib.dev(translations, torch.float32, "t")
        bias = [_lib.dev(p_, torch.float16, "pair_bias") for p_ in pair_bias]
        dims = _ipa_structs(layers[0], B, L)
        lib = _lib.lib()
        st = _lib.stream_ptr()
        packed = [layer._packed_weights(dims) for layer in layers]
        ws = layers[0]._workspace(max(lib.dab_ipa_sm100_workspace_bytes(ctypes.byref(dims)), 16), e.device)
        y = torch.empty(B, L, D, device=e.device, dtype=torch.float32)
        if front is None:
            x = _lib.dev(res_emb, res_emb.dtype if res_emb.dtype == torch.bfloat16 else torch.float32, "x")
        else:
            x = ws                  # (stages 2 / 4 do not read x: any non-null pointer satisfies the argument check)

        def stage(k, stages):     # (x is read by stage 1 only, y written by stage 4 only)
            _fwd_stages(dims, packed[k], x, e, bias[k], r, t, y, ws, stages, st)

        if front is None:
            stage(0, 1)
        else:
            cache, seq = front
            _lib.check(lib.dab_ipa_front_proj_sm100(
                ctypes.byref(dims), ptr(packed[0]), ptr(cache["c"]), ptr(cache["t1"]), ptr(_lib.dev(seq, torch.int64, "seq_idx")),
                ptr(cache["w2_bf16"]), ptr(cache["b2"]), ptr(r), ptr(t), ptr(ws), ws.numel(), st), "dab_ipa_front_proj_sm100")
        for k in range(n):
            if k == n - 1 and live is not None:     # (earlier layers: every row feeds the next layer's keys and values)
                _lib.check(lib.dab_ipa_core_sm100_live(ctypes.byref(dims), ptr(packed[k]), ptr(e), ptr(bias[k]), ptr(r), ptr(t),
                                                       ptr(ws), ws.numel(), ptr(live[0]), ptr(live[1]), st),
                           "dab_ipa_core_sm100_live")
            else:
                stage(k, 2)
            if k + 1 < n:
                _lib.check(lib.dab_ipa_mid_sm100(ctypes.byref(dims), ptr(packed[k]), ptr(packed[k + 1]), ptr(r), ptr(t), ptr(ws),
                                                 ws.numel(), st), "dab_ipa_mid_sm100")
            elif heads is None:
                stage(k, 4)
        if heads is None:
            return y
        heads_packed, beta_blk = heads
        nblk = B * (L // FAST_L)
        bdims = _ipa_structs(layers[0], nblk, FAST_L)          # the workspace sections are laid out per 128-residue block
        offs = (ctypes.c_size_t * 8)()
        _lib.check(lib.dab_ipa_sm100_workspace_layout(ctypes.byref(bdims), offs), "dab_ipa_sm100_workspace_layout")
        poffs = (ctypes.c_size_t * 7)()
        _lib.check(lib.dab_ipa_packed_layout(ctypes.byref(dims), poffs), "dab_ipa_packed_layout")
        eps = torch.empty(B, L, 3, device=e.device)
        rot = torch.empty(B, L, 3, device=e.device)
        post = torch.empty(B, L, 21, device=e.device)
        pk_last = packed[n - 1]
        _lib.check(lib.dab_out_heads_fwd_sm100(ptr(heads_packed), ws.data_ptr() + offs[4], pk_last.data_ptr() + poffs[1],
                                               pk_last.data_ptr() + poffs[3], ptr(beta_blk), nblk, FAST_L, ptr(eps), ptr(rot),
                                               ptr(post), None if live is None else ptr(live[0]),
                                               None if live is None else ptr(live[1]), st), "dab_out_heads_fwd_sm100")
        return eps, rot, post

    def precompute_pair_bias(self, pair_emb_bf16, out=None):
        """Per-layer pair-bias planes for the sm_100a path: one pass over the pair tensor for all layers
        (once per sampling run / once per training step).  Returns a list of (B, L, L, H) fp16 views of one
        (n_layers, B, L, L, H) tensor (``out`` if given)."""
        e = _lib.dev(pair_emb_bf16, torch.bfloat16, "e")
        B, L = e.shape[0], e.shape[1]
        n, H = len(self.layers), self.layers[0].n_head
        if out is None:
            out = torch.empty(n, B, L, L, H, device=e.device, dtype=torch.float16)
        elif out.dtype != torch.float16 or tuple(out.shape) != (n, B, L, L, H) or not out.is_contiguous():
            raise ValueError("precompute_pair_bias: `out` must be a contiguous fp16 (n_layers, B, L, L, H) tensor")
        _pair_bias_planes(self.layers, e, out)
        return list(out.unbind(0))


def cast_pair_to_bf16(pair_emb):
    """fp32 (B,L,L,C) -> bf16 once per patch (the pair tensor is constant over layers and steps)."""
    e = _lib.dev(pair_emb, torch.float32, "pair_emb")
    out = torch.empty(e.shape, device=e.device, dtype=torch.bfloat16)
    _lib.check(_lib.lib().dab_cast_f32_to_bf16(ptr(e), ptr(out), e.numel(), _lib.stream_ptr()), "dab_cast_f32_to_bf16")
    return out


class Denoiser(nn.Module):
    """diffab_pytorch.py:501-607."""

    def __init__(self, d_residue_emb, d_pair_emb, n_ipa_layers, d_scalar_per_head, n_query_point_per_head,
                 n_value_point_per_head, n_head, aa_vocab_size):
        super().__init__()
        D = d_residue_emb
        self.sequence_embedding = nn.Embedding(25, D)
        self.to_res_emb = _mlp([2 * D, D, D])
        self.ipa = InvariantPointAttentionModule(n_ipa_layers, D, d_pair_emb, d_scalar_per_head,
                                                 n_query_point_per_head, n_value_point_per_head, n_head)
        self.coordinate_denoising = _mlp([D + 3, D, D, 3])
        self.orientation_denoising = _mlp([D + 3, D, D, 3])
        self.sequence_denoising = _mlp([D + 3, D, D, aa_vocab_size])
        self.sequence_denoising.append(nn.Softmax(dim=-1))

    def heads(self, seq_idx_t, translations_t, orientations_t, res_context_emb, pair_context_emb, beta,
              pair_bias=None):
        """Everything up to the three head outputs; returns (eps, rotvec, seq_posterior)."""
        n_residues = seq_idx_t.shape[1]
        h = torch.cat([res_context_emb, _embed(self.sequence_embedding, seq_idx_t)], dim=-1)
        h = _run_mlp(self.to_res_emb, h)
        h = self.ipa(h, pair_context_emb, orientations_t, translations_t, pair_bias)
        t_emb = torch.stack([beta, torch.sin(beta), torch.cos(beta)], dim=-1)
        # (h is a CUDA tensor here: the IPA layers above raise on CPU tensors - there is no CPU path)
        # [h | t_emb] @ W1^T = h @ W1[:, :D]^T + (t_emb @ W1[:, D:]^T): the three time columns are a per-patch bias,
        # and the residue part is a K = 128 GEMM (K = 131 sends forward and both backward GEMMs to unaligned kernels)
        D = h.shape[-1]
        outs = []
        heads = (self.coordinate_denoising, self.orientation_denoising, self.sequence_denoising)
        # the three heads are independent chains of small kernels: when gradients are recorded (a training step, replayed
        # from a CUDA graph) each runs on its own stream, forward and - autograd replays a node on its forward stream - backward
        fork = torch.is_grad_enabled() and h.requires_grad
        main = torch.cuda.current_stream(h.device)
        for k, head in enumerate(heads):
            side = _side_stream(h.device, 3 + k) if fork else None
            if fork:
                side.wait_stream(main)
            with torch.cuda.stream(side) if fork else contextlib.nullcontext():
                w1, b1 = head[0].weight, head[0].bias
                pb = torch.addmm(b1, t_emb, w1[:, D:].t())                                  # (B, D)
                a = torch.relu(F.linear(h, w1[:, :D].contiguous()) + pb[:, None, :])
                outs.append(_run_mlp(head[2:], a))
        if fork:
            for k, o in enumerate(outs):
                main.wait_stream(_side_stream(h.device, 3 + k))
                o.record_stream(main)
        return tuple(outs)

    # ---- sampling fast path of the dense glue (same arithmetic, regrouped; inference only) ----
    @torch.no_grad()
    def sampling_cache(self, res_context_emb, cache=None):
        """Everything of the glue that does not change over the T reverse steps, computed once per run:
        * to_res_emb layer 1 (:572-574) acts on [res_ctx | emb(s_t)]: its res_ctx half (+ bias) is a constant
          (B, L, D) tensor and its embedding half a 25-row table, so per step layer 1 is a gather + add + relu;
        * the three heads (:591-599) act on [h | beta, sin beta, cos beta]: their first layers are concatenated
          into one (3D, D) matrix, the 3 time columns become a per-patch bias; layers 2 / 3 run as one batched GEMM each.
        ``cache`` (a previous result) is refreshed in place so CUDA graphs keep their addresses."""
        D = self.to_res_emb[0].out_features
        w1, b1 = self.to_res_emb[0].weight, self.to_res_emb[0].bias
        c = torch.addmm(b1, res_context_emb.reshape(-1, D), w1[:, :D].t()).view(res_context_emb.shape)
        if cache is not None:
            cache["c"].copy_(c)
            return cache
        heads = (self.coordinate_denoising, self.orientation_denoising, self.sequence_denoising)
        n_out = max(h[4].out_features for h in heads)
        w3 = torch.zeros(3, D, n_out, device=c.device)
        b3 = torch.zeros(3, 1, n_out, device=c.device)
        for k, h in enumerate(heads):
            w3[k, :, : h[4].out_features] = h[4].weight.t()
            b3[k, 0, : h[4].out_features] = h[4].bias
        wc1 = torch.cat([h[0].weight for h in heads], dim=0)             # (3D, D + 3)
        packed = None
        if (D == 128 and res_context_emb.shape[1] == 128 and [h[4].out_features for h in heads] == [3, 3, 21] and
                all(h[0].in_features == D + 3 for h in heads)):
            # fused tcgen05 heads kernel (csrc/heads_sm100.cu): weights packed once per run
            lib = _lib.lib()
            packed = _lib.aligned_empty(lib.dab_heads_packed_bytes(), c.device)
            ws = [_lib.dev(p.detach(), torch.float32, "head weight") for h in heads
                  for p in (h[0].weight, h[0].bias, h[2].weight, h[2].bias, h[4].weight, h[4].bias)]
            hw = _lib.DabHeadWeights(*(w.data_ptr() for w in ws))
            _lib.check(lib.dab_heads_pack_weights(ctypes.byref(hw), ptr(packed), _lib.stream_ptr()),
                       "dab_heads_pack_weights")
        return {
            "heads_packed": packed,
            "w2_bf16": self.to_res_emb[2].weight.detach().to(torch.bfloat16).contiguous() if packed is not None else None,
            "a_scratch": torch.empty(c.shape, device=c.device, dtype=torch.bfloat16) if packed is not None else None,
            "c": c, "t1": (self.sequence_embedding.weight @ w1[:, D:].t()).contiguous(),        # (25, D)
            "w2t": self.to_res_emb[2].weight.t().contiguous(), "b2": self.to_res_emb[2].bias,
            "wh1": wc1[:, :D].t().contiguous(),                                                  # (D, 3D)
            "wt1": wc1[:, D:].t().contiguous(), "bh1": torch.cat([h[0].bias for h in heads]),   # (3, 3D), (3D)
            "wh2": torch.stack([h[2].weight.t() for h in heads]).contiguous(),                  # (3, D, D)
            "bh2": torch.stack([h[2].bias for h in heads])[:, None, :].contiguous(),            # (3, 1, D)
            "wh3": w3, "bh3": b3, "n_out": [h[4].out_features for h in heads],
        }

    @torch.no_grad()
    def heads_fast(self, seq_idx_t, translations_t, orientations_t, cache, pair_context_emb, beta, pair_bias=None,
                   live=None):
        """``heads`` with the per-run constants of ``sampling_cache``; returns (eps, rotvec, seq_posterior).
        ``live`` (``live_query_tiles``, large batches only): the rows outside these tiles are left undefined."""
        B, L = seq_idx_t.shape
        D = cache["c"].shape[-1]
        if self.fused_heads_applicable(cache, B, L, pair_context_emb, pair_bias):
            # large batches: the front MLP runs inside the first layer's projection kernel (same bits as the branch below)
            front = (cache, seq_idx_t.contiguous())
            if cache.get("heads_packed") is not None:
                # ... and the last layer's to_out inside the heads kernel: the stack's output never exists in HBM either
                nb = L // FAST_L
                beta_blk = beta.contiguous() if nb == 1 else beta.repeat_interleave(nb)
                return self.ipa._forward_fused_stack(None, pair_context_emb, orientations_t, translations_t, pair_bias,
                                                     front=front, heads=(cache["heads_packed"], beta_blk), live=live)
            h = self.ipa._forward_fused_stack(None, pair_context_emb, orientations_t, translations_t, pair_bias, front=front,
                                              live=live)
            return self._heads_from(h, cache, pair_context_emb, beta)
        if cache.get("w2_bf16") is not None and pair_context_emb.dtype == torch.bfloat16 and (B * L) % 128 == 0:
            # bf16 out when the layer stack takes it (its first projection kernel rounds an fp32 input the same way)
            h16 = pair_bias is not None and len(self.ipa.layers) > 1 and self.ipa.layers[0].fast_path_supported(L, True)
            h = torch.empty(B, L, D, device=seq_idx_t.device, dtype=torch.bfloat16 if h16 else torch.float32)
            _lib.check(_lib.lib().dab_front_fwd_sm100(ptr(cache["c"]), ptr(cache["t1"]), ptr(seq_idx_t.contiguous()),
                                                      B * L, ptr(cache["w2_bf16"]), ptr(cache["b2"]),
                                                      ptr(cache["a_scratch"]), None if h16 else ptr(h),
                                                      ptr(h) if h16 else None, _lib.stream_ptr()),
                       "dab_front_fwd_sm100")
        else:
            h = torch.relu_(cache["c"] + F.embedding(seq_idx_t, cache["t1"]))
            h = torch.addmm(cache["b2"], h.view(-1, D), cache["w2t"]).view(B, L, D)
        h = self.ipa(h, pair_context_emb, orientations_t, translations_t, pair_bias)
        return self._heads_from(h, cache, pair_context_emb, beta)

    def fused_heads_applicable(self, cache, B, L, pair_context_emb, pair_bias):
        """``heads_fast`` runs the fused stack (front MLP in the first projections) - the path that takes ``live``."""
        return (cache.get("w2_bf16") is not None and cache["c"].dtype == torch.float32 and cache["c"].is_contiguous() and
                self.ipa.fused_stack_applicable(B, L, pair_context_emb, pair_bias))

    def _heads_from(self, h, cache, pair_context_emb, beta):
        """The three heads on the stack's output (sampling)."""
        B, L, D = h.shape
        if cache.get("heads_packed") is not None and pair_context_emb.dtype == torch.bfloat16:
            eps = torch.empty(B, L, 3, device=h.device)
            rot = torch.empty(B, L, 3, device=h.device)
            post = torch.empty(B, L, 21, device=h.device)
            nb = L // FAST_L if L % FAST_L == 0 else 1     # the kernel works on blocks of 128 residues (CTA = block)
            beta_blk = beta.contiguous() if nb == 1 else beta.repeat_interleave(nb)
            _lib.check(_lib.lib().dab_heads_fwd_sm100(ptr(cache["heads_packed"]), ptr(h.contiguous()), ptr(beta_blk),
                                                      B * nb, L // nb, ptr(eps), ptr(rot), ptr(post), _lib.stream_ptr()),
                       "dab_heads_fwd_sm100")
            return eps, rot, post
        t_emb = torch.stack([beta, torch.sin(beta), torch.cos(beta)], dim=-1)                   # (B, 3)
        pb = torch.addmm(cache["bh1"], t_emb, cache["wt1"])                                      # (B, 3D)
        a = torch.baddbmm(pb[:, None, :], h, cache["wh1"][None].expand(B, D, 3 * D)).relu_()     # (B, L, 3D)
        a = a.view(B * L, 3, D).transpose(0, 1)                                                  # (3, B L, D) strided
        a = torch.baddbmm(cache["bh2"], a, cache["wh2"]).relu_()                                 # (3, B L, D)
        o = torch.baddbmm(cache["bh3"], a, cache["wh3"])                                         # (3, B L, n_out)
        n = cache["n_out"]
        return (o[0, :, : n[0]].reshape(B, L, n[0]), o[1, :, : n[1]].reshape(B, L, n[1]),
                torch.softmax(o[2, :, : n[2]], dim=-1).view(B, L, n[2]))

    def forward(self, seq_idx_t, translations_t, orientations_t, res_context_emb, pair_context_emb, beta,
                generation_mask=None, residue_mask=None):
        # the two masks are accepted and unused, as in the reference (:566-567)
        eps, v_eps, post = self.heads(seq_idx_t, translations_t, orientations_t, res_context_emb, pair_context_emb,
                                      beta)
        o_denoised = _so3.small_matmul(orientations_t, vector_to_rotation_matrix(v_eps))   # :594-596
        return {"translations_eps": eps, "orientations_t0": o_denoised, "seq_posterior": post}


class OrientationLoss(nn.Module):
    """diffab_pytorch.py:610-625: MSE(R_pred^T R_true, I)."""

    def __init__(self, reduction="mean"):
        super().__init__()
        self.reduction = reduction

    def forward(self, pred_rotmat, target_rotmat):
        if pred_rotmat.is_cuda:
            d = _so3.small_matmul(pred_rotmat.transpose(-1, -2), target_rotmat)
        else:
            d = torch.einsum("blij,blik->bljk", pred_rotmat, target_rotmat)
        eye = torch.eye(3, device=d.device, dtype=d.dtype).expand_as(d)
        return F.mse_loss(d, eye, reduction=self.reduction)


class _FusedLosses(torch.autograd.Function):
    """The three masked losses of ``_shared_step`` (:856-880) in one kernel each way: ``dab_losses_fwd`` /
    ``dab_losses_bwd`` (gradients with respect to the three predictions only; targets are data)."""

    @staticmethod
    def forward(ctx, post_pred, post_tgt, eps_pred, eps_tgt, o_pred, o_true, mask, generate=3):
        f32 = torch.float32
        tensors = [_lib.dev(t.detach(), f32, n) for t, n in ((post_pred, "seq_posterior"), (post_tgt, "seq_posterior target"),
                                                             (eps_pred, "translations_eps"), (eps_tgt, "translations_eps target"),
                                                             (o_pred, "orientations_t0"), (o_true, "orientations target"))]
        m = _lib.mask_u8(mask, "loss mask")
        n = m.numel()
        if tensors[0].numel() != n * 21 or tensors[2].numel() != n * 3 or tensors[4].numel() != n * 9:
            raise ValueError("fused losses: shapes must be (B, L, 21), (B, L, 3), (B, L, 3, 3) and a (B, L) mask")
        acc = torch.zeros(8, device=m.device, dtype=f32)
        out = torch.empty(4, device=m.device, dtype=f32)
        _lib.check(_lib.lib().dab_losses_fwd(*(ptr(t) for t in tensors), ptr(m), n, generate, ptr(acc), ptr(out),
                                             _lib.stream_ptr()), "dab_losses_fwd")
        ctx.save_for_backward(*tensors, m, out)
        ctx.generate = generate
        return out[0], out[1], out[2]

    @staticmethod
    def backward(ctx, g_seq, g_pos, g_rot):
        *tensors, m, out = ctx.saved_tensors
        zero = out.new_zeros(())
        g = torch.stack([x.to(out.dtype) if x is not None else zero for x in (g_seq, g_pos, g_rot)]).contiguous()
        d_post, d_eps, d_o = torch.empty_like(tensors[0]), torch.empty_like(tensors[2]), torch.empty_like(tensors[4])
        _lib.check(_lib.lib().dab_losses_bwd(*(ptr(t) for t in tensors), ptr(m), m.numel(), ctx.generate, ptr(g), ptr(out),
                                             ptr(d_post), ptr(d_eps), ptr(d_o), _lib.stream_ptr()), "dab_losses_bwd")
        return d_post, None, d_eps, None, d_o, None, None, None


# =============================================================================================
# DiffAb
# =============================================================================================
class DiffAb(nn.Module):
    """diffab_pytorch.py:628-931.  ``device`` is where the schedules / IGSO(3) tables are built; they
    follow ``.to()`` / ``.cuda()`` and are not part of the state dict (106 keys, as in the reference).

    Design mode: ``generate_sequence`` / ``generate_structure`` (plain attributes, not in the state dict) say which
    modalities the masked residues generate in training and sampling.  Both True (default) is the reference's
    sequence-structure co-design; sequence only is fixed-backbone sequence design; structure only is structure
    prediction.  A modality that is not generated is shown to the context encoders on every residue, is neither noised
    nor denoised, and adds nothing to the loss."""

    generate_sequence = True
    generate_structure = True

    def __init__(self, d_residue_emb, d_pair_emb, n_ipa_layers, d_scalar_per_head, n_query_point_per_head,
                 n_value_point_per_head, n_head, T=100, s=0.01, beta_max=0.999, n_atoms=15, aa_vocab_size=21,
                 max_dist_to_consider=32, lr=1e-4, weight_decay=0.0, betas=(0.9, 0.999), device="cuda"):
        super().__init__()
        self.sched = cosine_variance_schedule(T=T, s=s, beta_max=beta_max)
        self.residue_context_embedding = ResidueEmbedding(n_atoms, d_residue_emb)
        self.pair_context_embedding = PairEmbedding(n_atoms, d_pair_emb, max_dist_to_consider)
        self.denoiser = Denoiser(d_residue_emb, d_pair_emb, n_ipa_layers, d_scalar_per_head,
                                 n_query_point_per_head, n_value_point_per_head, n_head, aa_vocab_size)
        self.seq_diffuser = SequenceDiffuser(T, s, beta_max, aa_vocab_size, device=device)
        self.coordinate_diffuser = CoordinateDiffuser(T, s, beta_max, device=device)
        self.orientation_diffuser = OrientationDiffuser(T, s, beta_max, device=device)
        # reverse-step IGSO(3) table at sigma = sqrt(beta_t) (SURVEY §3.3); built lazily by sample()
        self._so3_reverse = None
        self.aa_loss = nn.KLDivLoss(reduction="none")
        self.coordinate_loss = nn.MSELoss(reduction="none")
        self.orientation_loss = OrientationLoss(reduction="none")
        self.T, self.lr, self.weight_decay, self.betas = T, lr, weight_decay, betas
        self._device = torch.device(device)
        self._dsched = None
        if self._device.type == "cuda" and torch.cuda.is_available():
            if self._device.index is None:
                self._device = torch.device("cuda", torch.cuda.current_device())
            self.to(self._device)
        # without a GPU the module can still be constructed (state-dict inspection); every op raises

    # ---- device plumbing: non-buffer tables follow the module ----
    def _apply(self, fn, *args, **kwargs):
        super()._apply(fn, *args, **kwargs)
        probe = fn(torch.empty(0, device=self._device))
        if probe.device != self._device:
            if probe.device.type != "cuda":
                raise RuntimeError("DiffAb lives on the GPU - diffab_pytorch_b200 has no CPU path")
            self._device = probe.device
            self._dsched = None
            for d in (self.seq_diffuser, self.coordinate_diffuser, self.orientation_diffuser):
                d.to(self._device)
            if self._so3_reverse is not None:
                self._so3_reverse.to(self._device)
        return self

    @property
    def dsched(self):
        if self._dsched is None:
            self._dsched = _lib.Schedule(self.sched, self._device)
        return self._dsched

    def _generate(self):
        """The ``generate`` bits of the fused kernels for the current design mode (ValueError if it generates nothing)."""
        return _diffusion.generate_bits(self.generate_sequence, self.generate_structure)

    @property
    def so3_reverse(self):
        if self._so3_reverse is None:
            self._so3_reverse = _so3.SO3(self.sched["beta"].sqrt(), sigma_threshold=0.1, n_bins=8192, num_iters=1024,
                                         device=self._device)
        return self._so3_reverse

    # ---- reference API ----
    def encode_context(self, seq_idx_t0, xyz_t0, orientations_t0, backbone_dihedrals, distmat, pairwise_dihedrals,
                       atom_mask, chain_idx, residue_idx, generation_mask, residue_mask, generate_structure=True,
                       generate_sequence=True, distmat_is_squared=False):
        """diffab_pytorch.py:680-724 (``distmat_is_squared`` is ours: lets ``sample`` skip a sqrt / square pair)."""
        context_mask = residue_mask & (~generation_mask)
        structure_context_mask = context_mask if generate_structure else None
        sequence_context_mask = context_mask if generate_sequence else None
        fork = seq_idx_t0.is_cuda and torch.is_grad_enabled() and getattr(self, "train_precision", "fp32") == "bf16"
        if fork:
            # Training: the two context encoders are independent - the small residue encoder (a few dozen small kernels,
            # forward and, because autograd replays a node on the stream of its forward, backward) runs on a side stream
            # beside the pair encoder (parallel branches of the captured graph).
            main, side = torch.cuda.current_stream(seq_idx_t0.device), _side_stream(seq_idx_t0.device, 2)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                res = self.residue_context_embedding(seq_idx_t0, xyz_t0, orientations_t0, backbone_dihedrals, chain_idx,
                                                     atom_mask, structure_context_mask, sequence_context_mask)
        else:
            res = self.residue_context_embedding(seq_idx_t0, xyz_t0, orientations_t0, backbone_dihedrals, chain_idx,
                                                 atom_mask, structure_context_mask, sequence_context_mask)
        pair = self.pair_context_embedding(seq_idx_t0, distmat, pairwise_dihedrals, residue_idx, chain_idx, atom_mask,
                                           structure_context_mask, sequence_context_mask,
                                           distmat_is_squared=distmat_is_squared)
        if fork:
            main.wait_stream(side)
            res.record_stream(main)
        return res, pair

    def denoise(self, seq_idx_t, translations_t, orientations_t, res_context_emb, pair_context_emb, beta,
                generation_mask, residue_mask) -> Dict[str, torch.Tensor]:
        """diffab_pytorch.py:726-768."""
        return self.denoiser(seq_idx_t, translations_t, orientations_t, res_context_emb, pair_context_emb, beta,
                             generation_mask, residue_mask)

    def _add_noise(self, seq_idx_t0, translations_t0, orientations_t0, generation_mask, t, noise=None, generate=3):
        """diffab_pytorch.py:778-806, fused (two launches).  ``noise`` = the six draws of
        ``diffusion.draw_add_noise_tensors``; drawn on the device in that order when omitted (in every design mode).
        ``generate`` (``diffusion.generate_bits``): a modality that is not generated is returned as given."""
        B, L = seq_idx_t0.shape
        if noise is None:
            noise = _diffusion.draw_add_noise_tensors(B, L, device=seq_idx_t0.device)
        return _diffusion.fused_add_noise(self.dsched, self.orientation_diffuser.so3, seq_idx_t0, translations_t0,
                                          orientations_t0, generation_mask, t, noise, generate=generate)

    def _losses(self, denoised, noised, orientations_t0, generation_mask, residue_mask, generate=3):
        """diffab_pytorch.py:856-880.  On the GPU the three masked means are one fused kernel each way (SURVEY §8f N2).
        ``generate`` (``diffusion.generate_bits``): the term of a modality that is not generated is exactly 0, with a zero
        gradient; the denominator is the same in every mode."""
        if denoised["seq_posterior"].is_cuda and denoised["seq_posterior"].dtype == torch.float32:
            return _FusedLosses.apply(denoised["seq_posterior"], noised["seq_posterior"], denoised["translations_eps"],
                                      noised["translations_eps"], denoised["orientations_t0"], orientations_t0,
                                      generation_mask & residue_mask, generate)
        seq_loss = self.aa_loss(denoised["seq_posterior"].log(), noised["seq_posterior"])
        translations_loss = self.coordinate_loss(denoised["translations_eps"], noised["translations_eps"])
        orientations_loss = self.orientation_loss(denoised["orientations_t0"], orientations_t0)
        loss_mask = generation_mask & residue_mask
        denom = loss_mask.sum()
        seq_mask = loss_mask & bool(generate & _diffusion.GEN_SEQUENCE)
        str_mask = loss_mask & bool(generate & _diffusion.GEN_STRUCTURE)
        return ((seq_loss * seq_mask[..., None]).sum() / denom,
                (translations_loss * str_mask[..., None]).sum() / denom,
                (orientations_loss * str_mask[..., None, None]).sum() / denom)

    def _shared_step(self, batch, batch_idx, t=None, noise=None):
        """diffab_pytorch.py:808-880.  ``t`` / ``noise`` may be injected (tests); otherwise drawn on the
        device in the reference's order (#1 t, then the six noising draws).  ``self.train_precision``
        ("fp32" default, "bf16") picks the IPA path: with "bf16" the pair embedding is cast once per step and
        the six IPA layers run forward and backward on the tensor-core kernels.  ``generate_sequence`` /
        ``generate_structure`` pick the design mode (class docstring); the draws are the same in every mode."""
        generate = self._generate()
        device = batch["generation_mask"].device
        bsz = batch["generation_mask"].size(0)
        if t is None:
            t = torch.randint(low=1, high=self.T + 1, size=(bsz,), device=device)
        beta = self.dsched.tensors["beta"][t]
        seq_idx_t0 = batch["seq_idx"]
        xyz_t0 = batch["xyz"]
        translations_t0 = xyz_t0[:, :, CA_IDX].contiguous()
        orientations_t0 = batch["orientations"]
        generation_mask = batch["generation_mask"]
        bf16 = (getattr(self, "train_precision", "fp32") == "bf16" and
                self.denoiser.ipa.layers[0].fast_path_supported(seq_idx_t0.shape[1]))
        # forward noising is independent of the context encoders: in a (graph-captured) mixed-precision training step it runs
        # on a side stream beside them
        fork = bf16 and torch.is_grad_enabled() and seq_idx_t0.is_cuda
        if fork:
            main, nside = torch.cuda.current_stream(device), _side_stream(device, 6)
            nside.wait_stream(main)
        with torch.cuda.stream(nside) if fork else contextlib.nullcontext():
            noised = self._add_noise(seq_idx_t0, translations_t0, orientations_t0, generation_mask, t, noise=noise,
                                     generate=generate)
        self.pair_context_embedding.fused_rbf = bf16
        with _tf32_matmuls(bf16), _mixed_glue(bf16):   # mixed-precision step: the context encoders' GEMMs on the tensor cores too
            res_context_emb, pair_context_emb = self.encode_context(
                seq_idx_t0, xyz_t0, orientations_t0, batch["backbone_dihedrals"], batch["distmat"],
                batch["pairwise_dihedrals"], batch["atom_mask"], batch["chain_idx"], batch["residue_idx"],
                batch["generation_mask"], batch["residue_mask"],
                generate_structure=bool(generate & _diffusion.GEN_STRUCTURE),
                generate_sequence=bool(generate & _diffusion.GEN_SEQUENCE))
        if fork:
            main.wait_stream(nside)
            for v in noised.values():
                v.record_stream(main)
        if bf16:
            pair_context_emb = pair_context_emb.to(torch.bfloat16)   # autograd-aware cast (grad comes back as bf16)
        with _tf32_matmuls(bf16), _mixed_glue(bf16):
            denoised = self.denoise(noised["seq_idx_t"], noised["translations_t"], noised["orientations_t"],
                                    res_context_emb, pair_context_emb, beta, batch["generation_mask"],
                                    batch["residue_mask"])
        return self._losses(denoised, noised, batch["orientations"], batch["generation_mask"], batch["residue_mask"],
                            generate=generate)

    def training_step(self, batch, batch_idx):
        seq_loss, translations_loss, orientations_loss = self._shared_step(batch, batch_idx)
        loss = seq_loss + translations_loss + orientations_loss
        self.log_dict({"train/seq_loss": seq_loss, "train/translations_loss": translations_loss,
                       "train/orientations_loss": orientations_loss, "train/loss": loss})
        return loss

    def validation_step(self, batch, batch_idx):
        seq_loss, translations_loss, orientations_loss = self._shared_step(batch, batch_idx)
        loss = seq_loss + translations_loss + orientations_loss
        self.log_dict({"val/seq_loss": seq_loss, "val/translations_loss": translations_loss,
                       "val/orientations_loss": orientations_loss, "val/loss": loss})
        return loss

    def log_dict(self, metrics, *args, **kwargs):
        """Lightning's logging hook; here the last metrics are kept on the module."""
        self.last_metrics = {k: v.detach() for k, v in metrics.items()}

    def configure_optimizers(self):
        """diffab_pytorch.py:925-931: Adam(lr, weight_decay, betas).  On CUDA parameters PyTorch's single-kernel (``fused``)
        implementation of the same update: the default multi-tensor one is ~0.3 ms of small kernels per step here."""
        on_gpu = all(p.is_cuda for p in self.parameters())
        return torch.optim.Adam(self.parameters(), lr=self.lr, weight_decay=self.weight_decay, betas=self.betas,
                                fused=True if on_gpu else None)

    # ---- sampling (a stub in the reference, diffab_pytorch.py:770-776) ----
    @staticmethod
    def draw_step_noise(B, L, device, n_bins=8192, generator=None):
        """Per-step draws in the order fixed by oracle/sampler.py."""
        g = generator
        return {
            "seq_exp": torch.empty(B * L, 21, device=device).exponential_(generator=g),
            "z": torch.randn(B, L, 3, device=device, generator=g),
            "axis": torch.randn(B, L, 3, device=device, generator=g),
            "hist_exp": torch.empty(B, n_bins, device=device).exponential_(generator=g),
            "jitter": torch.rand(B, L, device=device, generator=g),
            "gauss": torch.randn(B, L, device=device, generator=g),
        }

    @staticmethod
    def draw_block_noise(n_steps, B, L, device, n_bins=8192):
        """The draws of ``n_steps`` consecutive reverse steps in six launches (leading dimension = step); used by the
        multi-step CUDA graph of ``sample``.  Same distributions as ``draw_step_noise``, another stream order."""
        return {
            "seq_exp": torch.empty(n_steps, B * L, 21, device=device).exponential_(),
            "z": torch.randn(n_steps, B, L, 3, device=device),
            "axis": torch.randn(n_steps, B, L, 3, device=device),
            "hist_exp": torch.empty(n_steps, B, n_bins, device=device).exponential_(),
            "jitter": torch.rand(n_steps, B, L, device=device),
            "gauss": torch.randn(n_steps, B, L, device=device),
        }

    @staticmethod
    def draw_prior_sequence(B, L, device, generator=None, seq_weight=None):
        """The t = T prior of the sequence, (B, L) int64: uniform over the 21 types, or with per-type weights
        (``aa_bias_weights``) the categorical draw of w / sum(w) as ``argmax_k w_k / E_k``, E ~ Exp(1) of shape (B*L, 21)."""
        if seq_weight is None:
            return torch.randint(0, 21, (B, L), device=device, generator=generator)
        E = torch.empty(B * L, 21, device=device).exponential_(generator=generator)
        return (seq_weight.reshape(B * L, 21) / E).argmax(-1).view(B, L)

    graph_block_steps = 20   # reverse steps per replay of the multi-step graph (static noise: ~12 MB per step at B = 256)

    @torch.no_grad()
    def reverse_step(self, seq_idx_t, translations_t, orientations_t, res_context_emb, pair_context_emb,
                     generation_mask, t, noise, inplace=False, pair_bias=None, glue_cache=None, beta=None, generate=3,
                     live=None, seq_weight=None):
        """One reverse-diffusion step: epsilon network + fused update kernel.  ``t`` is (B,) int64.
        ``glue_cache`` (``Denoiser.sampling_cache``) switches the dense glue to its regrouped form; ``beta`` = the
        schedule's beta at ``t`` when the caller has already gathered it.  ``generate`` (``diffusion.generate_bits``):
        a modality that is not generated keeps its value.  ``live`` = ``live_query_tiles(generation_mask)`` (with
        ``glue_cache``): the epsilon network's last layer and heads skip the tiles without a generated residue.
        ``seq_weight`` = ``aa_bias_weights(...)`` or None: per-type weights of the sequence draw."""
        if beta is None:
            beta = self.dsched.tensors["beta"][t]
        rotvec = None
        if glue_cache is not None:
            # the step's IGSO(3) draw depends on t and the noise only: it runs on a side stream beside the epsilon network
            # (a parallel branch of the step graph) instead of between the heads and the update
            B, L = seq_idx_t.shape
            rotvec = torch.empty(B, L, 3, device=seq_idx_t.device, dtype=torch.float32)
            main, side = torch.cuda.current_stream(seq_idx_t.device), _side_stream(seq_idx_t.device, 2)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                self.so3_reverse.sample_isotropic_gaussian(t, L, noise=noise, out=rotvec)
            eps, v_eps, post = self.denoiser.heads_fast(seq_idx_t, translations_t, orientations_t, glue_cache,
                                                        pair_context_emb, beta, pair_bias, live=live)
            main.wait_stream(side)
        else:
            eps, v_eps, post = self.denoiser.heads(seq_idx_t, translations_t, orientations_t, res_context_emb,
                                                   pair_context_emb, beta, pair_bias)
        return _diffusion.fused_reverse_step(self.dsched, self.so3_reverse, seq_idx_t, translations_t,
                                             orientations_t, eps, v_eps, post, generation_mask, t, noise,
                                             inplace=inplace, rotvec=rotvec, generate=generate, seq_weight=seq_weight)

    @torch.no_grad()
    def sample_from_context(self, seq_idx, translations, orientations, res_context_emb, pair_context_emb,
                            generation_mask, noises=None, generator=None, t_start=None, t_stop=1,
                            use_cuda_graph=False, _valid_len=None, seq_weight=None):
        """The reverse loop t_start..t_stop on resident tensors (this is what bench.py's ``value`` times).
        ``pair_context_emb`` may be fp32 (exact path) or bf16 (tensor-core path).  ``noises`` = {t: draws of step t}
        (``draw_step_noise``) injects every random draw (parity tests); it works with and without CUDA graphs.
        Only the modalities of the design mode (``generate_sequence`` / ``generate_structure``) change.  ``seq_weight``
        (``aa_bias_weights``, already validated) weighs the sequence draw of every step."""
        generate = self._generate()
        T = self.T
        t_start = T if t_start is None else t_start
        L0 = seq_idx.shape[1]
        Lp = _fast_len(L0, True)
        if (pair_context_emb.dtype == torch.bfloat16 and Lp is not None and L0 < Lp and _valid_len is None
                and self.denoiser.ipa.layers[0].fast_path_supported(Lp, True)):
            # Shorter patches on the tensor-core path: the state and the context are padded to 128 (or 256) residues (never
            # generated, never attended to: their keys are masked in every layer's bias plane), the loop runs on the
            # padded batch and the result is cut back.
            n = Lp - L0
            eye = torch.eye(3, device=orientations.device, dtype=orientations.dtype).expand(orientations.shape[0], n, 3, 3)
            pad_noise = None
            if noises is not None:
                B_ = seq_idx.shape[0]
                def pn(d):
                    return {"seq_exp": F.pad(d["seq_exp"].view(B_, L0, -1), (0, 0, 0, n), value=1.0).reshape(B_ * Lp, -1),
                            "z": F.pad(d["z"], (0, 0, 0, n)), "axis": F.pad(d["axis"], (0, 0, 0, n), value=1.0),
                            "hist_exp": d["hist_exp"], "jitter": F.pad(d["jitter"], (0, n)), "gauss": F.pad(d["gauss"], (0, n))}
                pad_noise = {k: pn(v) for k, v in noises.items()}
            out = self.sample_from_context(
                F.pad(seq_idx, (0, n)), F.pad(translations, (0, 0, 0, n)), torch.cat([orientations, eye], dim=1),
                F.pad(res_context_emb, (0, 0, 0, n)), F.pad(pair_context_emb, (0, 0, 0, n, 0, n)),
                F.pad(generation_mask, (0, n)), noises=pad_noise, generator=generator, t_start=t_start, t_stop=t_stop,
                use_cuda_graph=use_cuda_graph, _valid_len=L0,
                seq_weight=None if seq_weight is None else F.pad(seq_weight, (0, 0, 0, n), value=1.0))
            return {k: v[:, :L0].contiguous() for k, v in out.items()}
        s, x, O = seq_idx.clone(), translations.clone().contiguous(), orientations.clone().contiguous()
        B, L = s.shape
        dev = s.device
        _ = self.so3_reverse.histograms  # build the table outside any capture
        with _tf32_matmuls(pair_context_emb.dtype == torch.bfloat16):
            if use_cuda_graph and generator is None:
                return self._sample_graphed(s, x, O, res_context_emb, pair_context_emb, generation_mask, t_start,
                                            t_stop, noises, _valid_len, generate, seq_weight)
            pair_bias = self._pair_bias_planes(pair_context_emb)
            if pair_bias is not None and _valid_len is not None:
                _mask_padded_keys(pair_bias, _valid_len)
            glue = self.denoiser.sampling_cache(res_context_emb) if pair_context_emb.dtype == torch.bfloat16 else None
            live = self._live_tiles(generation_mask, pair_context_emb, pair_bias, glue)
            for step in range(t_start, t_stop - 1, -1):
                t = torch.full((B,), step, device=dev, dtype=torch.int64)
                noise = noises[step] if noises is not None else self.draw_step_noise(B, L, dev, generator=generator)
                out = self.reverse_step(s, x, O, res_context_emb, pair_context_emb, generation_mask, t, noise,
                                        inplace=True, pair_bias=pair_bias, glue_cache=glue, generate=generate, live=live,
                                        seq_weight=seq_weight)
                s, x, O = out["seq_idx"], out["translations"], out["orientations"]
            return {"seq_idx": s, "translations": x, "orientations": O}

    def _live_tiles(self, generation_mask, pair_ctx, pair_bias, glue, out=None):
        """``live_query_tiles`` of the mask where the reverse step runs the fused stack (the only path that takes them),
        else None."""
        B, L = generation_mask.shape
        if glue is None or not self.denoiser.fused_heads_applicable(glue, B, L, pair_ctx, pair_bias):
            return None
        return live_query_tiles(generation_mask, out=out)

    def _pair_bias_planes(self, pair_ctx):
        """Per-layer pair-bias planes of the tensor-core path (None on the fp32 path): the e . Wpb contraction
        depends on neither the step nor the state, so it is hoisted out of the T-step loop."""
        if pair_ctx.dtype != torch.bfloat16:
            return None
        return self.denoiser.ipa.precompute_pair_bias(pair_ctx)

    @staticmethod
    def _fill_noise_(bufs):
        """Redraw static noise buffers in place (same distributions as ``draw_step_noise``)."""
        bufs["seq_exp"].exponential_(); bufs["z"].normal_(); bufs["axis"].normal_()
        bufs["hist_exp"].exponential_(); bufs["jitter"].uniform_(); bufs["gauss"].normal_()

    def _sample_graphed(self, s, x, O, res_ctx, pair_ctx, generation_mask, t_start, t_stop, noises=None, valid_len=None,
                        generate=3, seq_weight=None):
        """Reverse steps captured in CUDA graphs and replayed; the step index lives in a device tensor.
        The graphs work on static buffers (state, context, mask, pair-bias planes, noise) and are cached per shape and
        ``_lib.weight_key``, so repeated ``sample()`` calls only copy their context in (~1 GB device-to-device, well
        under a millisecond).  Two step graphs: one reverse step, and a block of ``graph_block_steps`` consecutive
        steps; each reads its random draws from static buffers that a small companion graph redraws before every
        replay - or that the caller's ``noises`` are copied into (injected draws, parity tests).  The ``generate`` bits of
        the design mode are baked into the captured update kernels, so they are part of the cache key.  So is whether
        ``seq_weight`` is given: the weights are copied into a static buffer on every call, like the mask, so new values
        need no recapture; without them the graphs are those of the unweighted draw."""
        B, L = s.shape
        dev = s.device
        # the captured graphs bake in packed weights and per-run weight products: recapture when any parameter may have
        # changed (see _lib.weight_key for which updates are noticed on their own)
        key = (B, L, tuple(res_ctx.shape), tuple(pair_ctx.shape), pair_ctx.dtype, str(dev), generate,
               seq_weight is not None, _lib.weight_key(self.denoiser.parameters()))
        cache = getattr(self, "_graph_cache", None)
        fresh = cache is None or cache["key"] != key
        if fresh:
            cache = {"key": key, "s": torch.empty_like(s), "x": torch.empty_like(x), "O": torch.empty_like(O),
                     "t": torch.full((B,), t_start, device=dev, dtype=torch.int64),
                     "res": torch.empty_like(res_ctx), "pair": torch.empty_like(pair_ctx),
                     "mask": torch.empty_like(generation_mask), "bias": None, "graph": None, "glue": None, "live": None,
                     "graph_block": None, "noise1": self.draw_step_noise(B, L, dev),
                     "w": None if seq_weight is None else torch.empty_like(seq_weight)}
        st = cache
        st["res"].copy_(res_ctx); st["pair"].copy_(pair_ctx); st["mask"].copy_(generation_mask)
        if seq_weight is not None:
            st["w"].copy_(seq_weight)
        if pair_ctx.dtype == torch.bfloat16:   # per-layer pair-bias planes, written straight into the static buffers
            layers = self.denoiser.ipa.layers
            if st["bias"] is None:
                st["bias_all"] = torch.empty(len(layers), B, L, L, layers[0].n_head, device=dev, dtype=torch.float16)
                st["bias"] = list(st["bias_all"].unbind(0))
            self.denoiser.ipa.precompute_pair_bias(st["pair"], out=st["bias_all"])
            if valid_len is not None:          # padded batch of shorter patches: the padded keys are never attended to
                st["bias_all"][:, :, :, valid_len:, :] = float("-inf")
            st["glue"] = self.denoiser.sampling_cache(st["res"], cache=st["glue"])
            # the graphs are cached per shape, not per mask: the tile list is rebuilt into its static buffers on every call
            st["live"] = self._live_tiles(st["mask"], st["pair"], st["bias"], st["glue"], out=st["live"])
        if fresh:
            st["s"].copy_(s); st["x"].copy_(x); st["O"].copy_(O)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for _ in range(2):  # warm-up outside capture (allocator, lazy init, weight packing)
                    self._fill_noise_(st["noise1"])
                    self.reverse_step(st["s"].clone(), st["x"].clone(), st["O"].clone(), st["res"], st["pair"],
                                      st["mask"], st["t"], st["noise1"], pair_bias=st["bias"], glue_cache=st["glue"],
                                      generate=generate, live=st["live"], seq_weight=st["w"])
            torch.cuda.current_stream(dev).wait_stream(side)
            draw, graph = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(draw):
                self._fill_noise_(st["noise1"])
            with torch.cuda.graph(graph, pool=draw.pool()):
                self.reverse_step(st["s"], st["x"], st["O"], st["res"], st["pair"], st["mask"], st["t"], st["noise1"],
                                  inplace=True, pair_bias=st["bias"], glue_cache=st["glue"], generate=generate,
                                  live=st["live"], seq_weight=st["w"])
                st["t"].sub_(1)
            st["graph"], st["draw"] = graph, draw
            self._graph_cache = st
        # Long runs replay a second graph that holds `graph_block_steps` consecutive steps: their random draws are six
        # launches per block instead of six per step (9 of the 32 launches of a step are PyTorch RNG / index kernels).
        U = int(self.graph_block_steps)
        n_steps = t_start - t_stop + 1
        n_blocks = n_steps // U if U > 1 else 0
        if n_blocks > 0 and (st["graph_block"] is None or st["graph_block"][0] != U):
            st["s"].copy_(s); st["x"].copy_(x); st["O"].copy_(O)
            st["t"].fill_(t_start)
            # (graph inputs: must live as long as the graphs, so they are kept in the cache next to them)
            st["steps_back"] = steps_back = torch.arange(U, device=dev, dtype=torch.int64)[:, None]
            st["noiseU"] = noiseU = self.draw_block_noise(U, B, L, dev)
            draw_block, block = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(draw_block, pool=st["draw"].pool()):
                self._fill_noise_(noiseU)
            with torch.cuda.graph(block, pool=st["draw"].pool()):
                t_blk = st["t"][None, :] - steps_back                  # (U, B): the block's step indices ...
                beta_blk = self.dsched.tensors["beta"][t_blk]          # ... and betas, one gather per block
                for u in range(U):
                    self.reverse_step(st["s"], st["x"], st["O"], st["res"], st["pair"], st["mask"], t_blk[u],
                                      {k: v[u] for k, v in noiseU.items()}, inplace=True, pair_bias=st["bias"],
                                      glue_cache=st["glue"], beta=beta_blk[u], generate=generate, live=st["live"],
                                      seq_weight=st["w"])
                st["t"].sub_(U)
            st["graph_block"] = (U, block, draw_block)
        st["s"].copy_(s); st["x"].copy_(x); st["O"].copy_(O)
        st["t"].fill_(t_start)
        step = t_start
        for _ in range(n_blocks):
            if noises is None:
                st["graph_block"][2].replay()
            else:
                for k, buf in st["noiseU"].items():
                    for u in range(U):
                        buf[u].copy_(noises[step - u][k].view_as(buf[u]))
            st["graph_block"][1].replay()
            step -= U
        for _ in range(n_steps - n_blocks * U):
            if noises is None:
                st["draw"].replay()
            else:
                for k, buf in st["noise1"].items():
                    buf.copy_(noises[step][k].view_as(buf))
            st["graph"].replay()
            step -= 1
        return {"seq_idx": st["s"].clone(), "translations": st["x"].clone(), "orientations": st["O"].clone()}

    def invalidate_weight_caches(self):
        """Forget every weight-derived cache (packed bf16 weights, glue constants, captured sampling graphs).  Needed after
        weight updates PyTorch cannot see - raw ``.data`` writes, optimizer steps replayed from a CUDA graph outside
        ``distributed.GraphedTrainStep`` (which calls the library-wide equivalent, ``_lib.bump_weight_generation``, at
        every replay).  Noticed without this call: eager in-place updates of the parameters, and eager optimizer steps on
        the flat parameter of ``GradientBucket.flatten_parameters`` (``torch.optim`` optimizers and ``FlatAdam``)."""
        _lib.bump_weight_generation()
        self._graph_cache = None

    def load_state_dict(self, *args, **kwargs):
        out = super().load_state_dict(*args, **kwargs)
        self.invalidate_weight_caches()
        return out

    @torch.no_grad()
    def sample(self, seq_idx, xyz, orientations, backbone_dihedrals=None, distmat=None, pairwise_dihedrals=None,
               atom_mask=None, chain_idx=None, residue_idx=None, generation_mask=None, residue_mask=None,
               generator=None, precision="bf16", use_cuda_graph=True, context_chunk=32, t_start=None, t_stop=1,
               init="prior", aa_bias=None):
        """Reverse-diffusion sampling of the masked residues (the reference's stub, made real).

        Accepts host or device tensors (host tensors are copied to the model's device; pinned memory
        makes that asynchronous).  Features not given are derived: ``distmat`` from ``xyz`` on the
        device, masks default to "all residues valid / generation mask required".  Returns a dict
        ``{seq_idx, translations, orientations}`` on the model's device.

        Only the modalities of the design mode (``generate_sequence`` / ``generate_structure``) are generated; the
        other one is context on every residue and comes back unchanged.  ``init="prior"`` starts the generated
        residues from the t = T prior; ``init="native"`` (optimisation of an existing antibody) starts from the given
        sequence and structure noised to step ``t_start`` (in [1, T], default T) by the forward process, then
        denoises from there.

        ``aa_bias`` constrains the designed sequence: a float log-space bias on the residue types, broadcastable to
        (B, L, 21) - (21,), (L, 21) or (B, L, 21); column k is type k of ``seq_idx``, 20 = UNK.  ``-inf`` forbids a
        type, 0 everywhere is no bias; on the generated residues it acts as a bias added to the sequence head's logits.
        It is turned once into weights ``w = exp(b - max_k b)`` (``aa_bias_weights``), and every reverse step draws
        ``argmax_k p_k w_k / E_k`` over the types with ``w_k > 0`` (E = the step's Exp(1) draw; when the posterior mass
        on the allowed types underflows, ``argmax_k w_k / E_k``).  The t = T prior becomes ``argmax_k w_k / E_k`` with
        E ~ Exp(1) of shape (B*L, 21) from ``generator``, in place of the uniform draw.  Every generated residue of the
        returned ``seq_idx`` has ``w > 0``; context residues keep their type even where it is forbidden; translations
        and orientations follow the same draws as without the bias.  Refused with ``ValueError``: NaN or +inf, a shape
        that does not broadcast, a generated residue with every type at -inf, and a design mode that does not generate
        the sequence."""
        generate = self._generate()
        gen_seq, gen_str = bool(generate & _diffusion.GEN_SEQUENCE), bool(generate & _diffusion.GEN_STRUCTURE)
        if init not in ("prior", "native"):
            raise ValueError(f"sample(): init must be 'prior' or 'native', got {init!r}")
        if init == "native":
            t_start = self.T if t_start is None else t_start
            if not 1 <= t_start <= self.T:
                raise ValueError(f"sample(init='native'): t_start must be in [1, {self.T}], got {t_start}")
        dev = self._device
        mv = lambda v: None if v is None else v.to(dev, non_blocking=True)
        seq_idx, xyz, orientations = mv(seq_idx), mv(xyz), mv(orientations)
        B, L = seq_idx.shape
        A = xyz.shape[2]
        if generation_mask is None:
            raise ValueError("sample() needs generation_mask: which residues to generate")
        generation_mask = mv(generation_mask).bool()
        seq_weight = aa_bias_weights(aa_bias, generation_mask, gen_seq)
        residue_mask = torch.ones(B, L, dtype=torch.bool, device=dev) if residue_mask is None else mv(residue_mask).bool()
        atom_mask = torch.ones(B, L, A, dtype=torch.bool, device=dev) if atom_mask is None else mv(atom_mask)
        chain_idx = torch.ones(B, L, dtype=torch.long, device=dev) if chain_idx is None else mv(chain_idx)
        residue_idx = torch.arange(L, device=dev)[None].expand(B, L) if residue_idx is None else mv(residue_idx)
        backbone_dihedrals = torch.zeros(B, L, 3, device=dev) if backbone_dihedrals is None else mv(backbone_dihedrals)
        pairwise_dihedrals = torch.zeros(B, L, L, 2, device=dev) if pairwise_dihedrals is None else mv(pairwise_dihedrals)
        distmat = mv(distmat)
        layer0 = self.denoiser.ipa.layers[0]
        Lp = _fast_len(L, True)                       # tensor-core path: L <= 256 (padded to 128 or 256 residues)
        use_bf16 = precision == "bf16" and Lp is not None and layer0.fast_path_supported(Lp, True)
        res_parts, pair_parts = [], []
        fused_pair = (use_bf16 and distmat is None and self.pair_context_embedding.fused_supported(Lp, A))
        from .synth import pairwise_atom_distances, pairwise_atom_sq_distances
        # distances derived on the device: exact differences on the fp32 path, the cheaper Gram-matrix form
        # (|a|^2 + |b|^2 - 2 a.b, ~1e-3 A^2 absolute error) on the bf16 path
        derive = pairwise_atom_sq_distances if use_bf16 else (lambda v: pairwise_atom_distances(v).pow(2))
        with _tf32_matmuls(use_bf16):
            if fused_pair:
                # pair context from one fused tcgen05 kernel (bf16, distances from xyz inside the kernel); the small
                # residue encoder stays a PyTorch module
                ctx_mask = residue_mask & (~generation_mask)
                seq_ctx = ctx_mask if gen_seq else None        # encode_context's generate_* flags
                res_ctx = self.residue_context_embedding(seq_idx, xyz, orientations, backbone_dihedrals, chain_idx,
                                                         atom_mask, ctx_mask if gen_str else None, seq_ctx)
                if L < Lp:    # ragged length: the fused kernel works on 128 / 256 residues - pad with absent residues, cut back
                    n = Lp - L
                    pad1 = lambda v: F.pad(v, (0, n))
                    pair_ctx = self.pair_context_embedding.forward_fused_bf16(
                        pad1(seq_idx), F.pad(xyz, (0, 0, 0, 0, 0, n)), F.pad(pairwise_dihedrals, (0, 0, 0, n, 0, n)),
                        pad1(residue_idx), pad1(chain_idx), F.pad(atom_mask, (0, 0, 0, n)),
                        None if seq_ctx is None else pad1(seq_ctx))
                    pair_ctx = pair_ctx[:, :L, :L].contiguous()
                else:
                    pair_ctx = self.pair_context_embedding.forward_fused_bf16(seq_idx, xyz, pairwise_dihedrals, residue_idx,
                                                                              chain_idx, atom_mask, seq_ctx)
            else:
                for lo in range(0, B, context_chunk):
                    sl = slice(lo, min(B, lo + context_chunk))
                    dm = distmat[sl] if distmat is not None else derive(xyz[sl])
                    r, p = self.encode_context(seq_idx[sl], xyz[sl], orientations[sl], backbone_dihedrals[sl], dm,
                                               pairwise_dihedrals[sl], atom_mask[sl], chain_idx[sl], residue_idx[sl],
                                               generation_mask[sl], residue_mask[sl], generate_structure=gen_str,
                                               generate_sequence=gen_seq, distmat_is_squared=distmat is None)
                    res_parts.append(r)
                    pair_parts.append(cast_pair_to_bf16(p) if use_bf16 else p)
                res_ctx, pair_ctx = torch.cat(res_parts), torch.cat(pair_parts)
        m = generation_mask
        x0 = xyz[:, :, CA_IDX]
        if init == "native":
            # the native state noised to t_start on the generated modalities (the forward process of training)
            noise = _diffusion.draw_add_noise_tensors(B, L, device=dev, generator=generator)
            t = torch.full((B,), t_start, device=dev, dtype=torch.int64)
            noised = self._add_noise(seq_idx, x0, orientations, m, t, noise=noise, generate=generate)
            s, x, O = noised["seq_idx_t"], noised["translations_t"], noised["orientations_t"]
        else:
            # t = T prior on generated residues: s ~ U{0..20}, x ~ N(0, I), O ~ uniform SO(3); drawn in every mode,
            # a modality that is not generated starts (and stays) at its native value
            from .synth import uniform_rotations
            sT = self.draw_prior_sequence(B, L, dev, generator=generator, seq_weight=seq_weight)
            xT = torch.randn(B, L, 3, device=dev, generator=generator)
            OT = uniform_rotations(B, L, generator=generator, device=dev)
            ms, mx = m & gen_seq, m & gen_str
            s = torch.where(ms, sT, seq_idx)
            x = torch.where(mx[..., None], xT, x0)
            O = torch.where(mx[..., None, None], OT, orientations)
        return self.sample_from_context(s, x, O, res_ctx, pair_ctx, m, generator=generator, t_start=t_start,
                                        t_stop=t_stop, use_cuda_graph=use_cuda_graph and generator is None,
                                        seq_weight=seq_weight)
