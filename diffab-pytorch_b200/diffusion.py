"""Variance schedule and the three diffusers on the GPU - mirror of ``diffab_pytorch/diffusion.py``.

Same class / method names and argument meaning as the reference (``diffusion.py:11-294``).  The
per-residue arithmetic runs in ``csrc/diffusion_kernels.cu``.  Every sampling method takes an
optional ``noise=`` argument; when omitted the draws are made with torch on the device in the
reference's order.  CUDA tensors only.
"""
import math

import torch

from . import _lib
from . import so3
from ._lib import ptr

V = 21  # diffusion.py:47 (``aa_vocab_size`` is ignored there)
GEN_SEQUENCE, GEN_STRUCTURE = 1, 2   # ``generate`` bits of the fused kernels (DAB_GEN_* in include/diffab_b200.h)


def generate_bits(generate_sequence, generate_structure):
    """The ``generate`` argument of the fused kernels for a design mode: 3 co-design, 1 fixed-backbone sequence design,
    2 structure prediction.  Generating neither modality is refused."""
    if not (generate_sequence or generate_structure):
        raise ValueError("generate_sequence and generate_structure are both False: nothing to generate")
    return (GEN_SEQUENCE if generate_sequence else 0) | (GEN_STRUCTURE if generate_structure else 0)


def cosine_variance_schedule(T, s=8e-3, beta_max=0.999):
    """diffusion.py:11-35.  Host-side (T+1 floats, computed once); returns CPU fp32 tensors with the
    reference's keys - ``DiffAb.sched`` keeps this dict for API compatibility."""
    t = torch.arange(T + 1)
    f_t = torch.cos((t / T + s) / (1 + s) * math.pi / 2.0).square()
    alpha_bar = f_t / f_t[0]
    beta = torch.cat([torch.zeros(1), torch.clip(1 - alpha_bar[1:] / alpha_bar[:-1], min=1e-5, max=beta_max)])
    return {
        "alpha": 1 - beta,
        "alpha_bar": alpha_bar,
        "alpha_bar_sqrt": alpha_bar.sqrt(),
        "one_minus_alpha_bar_sqrt": (1 - alpha_bar).sqrt(),
        "beta": beta,
    }


class _Diffuser(object):
    def __init__(self, T, s=0.01, beta_max=0.999, device="cuda"):
        self.T = T
        self.sched = cosine_variance_schedule(T, s=s, beta_max=beta_max)
        self.device = torch.device(device)
        self._dsched = None

    def to(self, device):
        self.device = torch.device(device)
        self._dsched = None
        return self

    @property
    def dsched(self):
        if self._dsched is None:
            if self.device.type != "cuda":
                raise RuntimeError("diffusers run on the GPU - diffab_pytorch_b200 has no CPU path")
            self._dsched = _lib.Schedule(self.sched, self.device)
        return self._dsched


class SequenceDiffuser(_Diffuser):
    def __init__(self, T, s=0.01, beta_max=0.999, aa_vocab_size=21, device="cuda"):
        super().__init__(T, s, beta_max, device)
        self.aa_vocab_size = V

    def _probs(self, kind, seq, seq0, t, generation_mask):
        seq = _lib.dev(seq, torch.int64, "seq_idx")
        t = _lib.dev(t, torch.int64, "t")
        m = _lib.mask_u8(generation_mask, "generation_mask")
        B, L = seq.shape
        out = torch.empty(B, L, V, device=seq.device, dtype=torch.float32)
        s0 = _lib.dev(seq0, torch.int64, "seq_idx_t0") if seq0 is not None else None
        _lib.check(_lib.lib().dab_seq_probs(self.dsched.ref(), kind, ptr(seq), ptr(s0), ptr(m), ptr(t), B, L, ptr(out),
                                            _lib.stream_ptr()), "dab_seq_probs")
        return out

    def forward_prob_single_step(self, seq_idx, t, generation_mask):
        """diffusion.py:49-79."""
        return self._probs(0, seq_idx, None, t, generation_mask)

    def forward_prob_from_t0(self, seq_idx_t0, t, generation_mask):
        """diffusion.py:105-135."""
        return self._probs(1, seq_idx_t0, None, t, generation_mask)

    def posterior_single_step(self, seq_idx_t, seq_idx_t0, t, generation_mask):
        """diffusion.py:168-192."""
        return self._probs(2, seq_idx_t, seq_idx_t0, t, generation_mask)

    @staticmethod
    def _multinomial(p, exp_noise):
        # torch.multinomial(p, 1) == argmax(p / Exp(1)); kept as two torch ops here because the fused
        # noising kernel (DiffAb._add_noise) is the hot path, this method is API surface only.
        if exp_noise is None:
            exp_noise = torch.empty_like(p).exponential_()
        return (p / exp_noise.view_as(p)).argmax(dim=-1)

    def diffuse_single_step(self, seq_idx, t, generation_mask, noise=None):
        """diffusion.py:81-103 (without the stray print at :100)."""
        p = self.forward_prob_single_step(seq_idx, t, generation_mask)
        return self._multinomial(p, noise)

    def diffuse_from_t0(self, seq_idx_t0, t, generation_mask, return_posterior=True, noise=None):
        """diffusion.py:137-166."""
        p = self.forward_prob_from_t0(seq_idx_t0, t, generation_mask)
        seq_idx_t = self._multinomial(p, noise)
        if return_posterior:
            return seq_idx_t, self.posterior_single_step(seq_idx_t, seq_idx_t0, t, generation_mask)
        return seq_idx_t


class CoordinateDiffuser(_Diffuser):
    def diffuse_from_t0(self, translations_t0, t, generation_mask, return_eps=True, noise=None):
        """diffusion.py:199-236.  Plain torch elementwise ops (API surface; the fused path is
        ``DiffAb._add_noise``)."""
        x0 = _lib.dev(translations_t0, torch.float32, "translations_t0")
        d = self.dsched.tensors
        a = d["alpha_bar_sqrt"][t][:, None, None]
        b = d["one_minus_alpha_bar_sqrt"][t][:, None, None]
        eps = torch.randn_like(x0) if noise is None else noise
        x_t = torch.where(generation_mask.bool().unsqueeze(-1), a * x0 + b * eps, x0)
        return (x_t, eps) if return_eps else x_t


class OrientationDiffuser(_Diffuser):
    def __init__(self, T, s=0.01, beta_max=0.999, device="cuda"):
        """diffusion.py:240-260: IGSO(3) table at sigma_t = sqrt(1 - abar_t), built on the device."""
        super().__init__(T, s, beta_max, device)
        self.so3 = so3.SO3(sigmas_to_consider=self.sched["one_minus_alpha_bar_sqrt"], sigma_threshold=0.1,
                           n_bins=8192, num_iters=1024, device=device)

    def to(self, device):
        super().to(device)
        self.so3.to(device)
        return self

    def diffuse_from_t0(self, orientations_t0, generation_mask, t, noise=None):
        """diffusion.py:262-294."""
        O0 = _lib.dev(orientations_t0, torch.float32, "orientations_t0")
        mean = so3.scale_rot(O0, self.dsched.tensors["alpha_bar_sqrt"][t])
        rotvec = self.so3.sample_isotropic_gaussian(t, num_samples=O0.shape[1], noise=noise)
        O_t = mean @ so3.vector_to_rotation_matrix(rotvec)
        return torch.where(generation_mask.bool()[..., None, None], O_t, O0)


def draw_add_noise_tensors(bsz, L, n_bins=8192, device="cuda", generator=None):
    """The six draws of ``DiffAb._add_noise`` in the reference's order (SURVEY §3.1 #2-#7)."""
    g = generator
    return {
        "seq_exp": torch.empty(bsz * L, V, device=device).exponential_(generator=g),
        "eps": torch.randn(bsz, L, 3, device=device, generator=g),
        "axis": torch.randn(bsz, L, 3, device=device, generator=g),
        "hist_exp": torch.empty(bsz, n_bins, device=device).exponential_(generator=g),
        "jitter": torch.rand(bsz, L, device=device, generator=g),
        "gauss": torch.randn(bsz, L, device=device, generator=g),
    }


def fused_add_noise(dsched, so3_table, seq0, x0, O0, generation_mask, t, noise, generate=3):
    """``DiffAb._add_noise`` (diffab_pytorch.py:778-806) as two launches: IGSO(3) sampler + one fused
    per-residue kernel.  ``generate`` (``generate_bits``): a modality that is not generated comes back as its input."""
    seq0 = _lib.dev(seq0, torch.int64, "seq_idx_t0")
    x0 = _lib.dev(x0, torch.float32, "translations_t0")
    O0 = _lib.dev(O0, torch.float32, "orientations_t0")
    t = _lib.dev(t, torch.int64, "t")
    m = _lib.mask_u8(generation_mask, "generation_mask")
    B, L = seq0.shape
    rotvec = so3_table.sample_isotropic_gaussian(t, L, noise=noise)
    seq_exp = _lib.dev(noise["seq_exp"], torch.float32, "seq_exp")
    eps = _lib.dev(noise["eps"], torch.float32, "eps")
    dev = seq0.device
    seq_t = torch.empty(B, L, device=dev, dtype=torch.int64)
    post = torch.empty(B, L, V, device=dev, dtype=torch.float32)
    x_t = torch.empty(B, L, 3, device=dev, dtype=torch.float32)
    O_t = torch.empty(B, L, 3, 3, device=dev, dtype=torch.float32)
    _lib.check(_lib.lib().dab_forward_noise(dsched.ref(), ptr(seq0), ptr(x0), ptr(O0), ptr(m), ptr(t), B, L,
                                            ptr(seq_exp), ptr(eps), ptr(rotvec), generate, ptr(seq_t), ptr(post), ptr(x_t),
                                            ptr(O_t), _lib.stream_ptr()), "dab_forward_noise")
    return {"seq_idx_t": seq_t, "seq_posterior": post, "translations_t": x_t, "translations_eps": eps,
            "orientations_t": O_t}


def fused_reverse_step(dsched, so3_rev, seq_t, x_t, O_t, eps_theta, v_theta, seq_post, generation_mask, t, noise,
                       inplace=False, return_O0=False, rotvec=None, generate=3, seq_weight=None):
    """Reverse step (oracle/sampler.py; not in the reference): IGSO(3) sampler + one fused kernel.  ``rotvec``: the step's
    IGSO(3) draw when the caller has already made it (it depends on t and the noise only, not on the network).
    ``generate`` (``generate_bits``): a modality that is not generated keeps its old value.  ``seq_weight``: (B, L, 21)
    fp32 per-type weights of the sequence draw in [0, 1], 0 = forbidden (``DiffAb.sample``'s ``aa_bias``; rule in
    ``dab_reverse_step_weighted``), or None."""
    seq_t = _lib.dev(seq_t, torch.int64, "seq_idx_t")
    x_t = _lib.dev(x_t, torch.float32, "translations_t")
    O_t = _lib.dev(O_t, torch.float32, "orientations_t")
    eps_theta = _lib.dev(eps_theta, torch.float32, "eps_theta")
    v_theta = _lib.dev(v_theta, torch.float32, "v_theta")
    seq_post = _lib.dev(seq_post, torch.float32, "seq_posterior")
    t = _lib.dev(t, torch.int64, "t")
    m = _lib.mask_u8(generation_mask, "generation_mask")
    B, L = seq_t.shape
    seq_exp = _lib.dev(noise["seq_exp"], torch.float32, "seq_exp")
    z = _lib.dev(noise["z"], torch.float32, "z")
    if inplace:
        s_out, x_out, O_out = seq_t, x_t, O_t
    else:
        s_out, x_out, O_out = torch.empty_like(seq_t), torch.empty_like(x_t), torch.empty_like(O_t)
    if rotvec is None:
        rotvec = so3_rev.sample_isotropic_gaussian(t, L, noise=noise)
    rotvec = _lib.dev(rotvec, torch.float32, "rotvec")
    if seq_weight is not None:
        seq_weight = _lib.dev(seq_weight, torch.float32, "seq_weight")
        if seq_weight.shape != (B, L, V):
            raise ValueError(f"seq_weight: expected shape {(B, L, V)}, got {tuple(seq_weight.shape)}")
    O0 = torch.empty_like(O_t) if return_O0 else None
    _lib.check(_lib.lib().dab_reverse_step_weighted(dsched.ref(), ptr(seq_t), ptr(x_t), ptr(O_t), ptr(eps_theta),
                                                    ptr(v_theta), ptr(seq_post), ptr(m), ptr(t), B, L, ptr(seq_exp),
                                                    ptr(z), ptr(rotvec), ptr(seq_weight), generate, ptr(s_out),
                                                    ptr(x_out), ptr(O_out), ptr(O0), _lib.stream_ptr()),
               "dab_reverse_step_weighted")
    out = {"seq_idx": s_out, "translations": x_out, "orientations": O_out}
    if return_O0:
        out["orientations_t0"] = O0
    return out
