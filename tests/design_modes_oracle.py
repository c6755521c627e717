"""Oracle of the design modes (fixed-backbone sequence design, structure prediction) for the tests.

UNPINNED BY THE REFERENCE beyond its ``encode_context(generate_structure, generate_sequence)`` flags
(diffab_pytorch.py:680-724): nothing after the encoder honours them there.  The modes are composed here from primitives
of ``oracle/`` that ARE pinned (the three ``*_diffuse_from_t0``, the sampler's reverse step and initial state, the
orientation loss), by giving each modality its own set of generated residues: ``generation_mask`` when the modality is
on, no residue when it is off.  With both switches on every function equals its co-design counterpart in ``oracle/``.
The random draws are the same in every mode.
"""
import torch

from oracle import diffusion as odiff
from oracle import ipa as oipa
from oracle import sampler as osamp


def modality_masks(generation_mask, generate_sequence=True, generate_structure=True):
    """(residues that generate the sequence, residues that generate the structure)."""
    if not (generate_sequence or generate_structure):
        raise ValueError("generate_sequence and generate_structure are both False")
    none = torch.zeros_like(generation_mask)
    return (generation_mask if generate_sequence else none), (generation_mask if generate_structure else none)


def add_noise(sched, hist, seq_idx_t0, x0, O0, generation_mask, t, noise, generate_sequence=True,
              generate_structure=True):
    """``oracle.diffusion.add_noise`` with a modality that is off left as its input on every residue."""
    m_seq, m_str = modality_masks(generation_mask, generate_sequence, generate_structure)
    s_t, post = odiff.seq_diffuse_from_t0(sched, seq_idx_t0, t, m_seq, noise["seq_exp"])
    x_t, eps = odiff.coord_diffuse_from_t0(sched, x0, t, m_str, noise["eps"])
    O_t = odiff.orient_diffuse_from_t0(sched, hist, O0, m_str, t, noise["axis"], noise["hist_exp"], noise["jitter"],
                                       noise["gauss"])
    return {"seq_idx_t": s_t, "seq_posterior": post, "translations_t": x_t, "translations_eps": eps,
            "orientations_t": O_t}


def reverse_step(sched, hist_rev, s_t, x_t, O_t, eps_theta, O0_theta, seq_post, generation_mask, t, noise,
                 generate_sequence=True, generate_structure=True):
    """``oracle.sampler.reverse_step`` with a modality that is off keeping its old value on every residue."""
    m_seq, m_str = modality_masks(generation_mask, generate_sequence, generate_structure)
    seq = osamp.reverse_step(sched, hist_rev, s_t, x_t, O_t, eps_theta, O0_theta, seq_post, m_seq, t, noise)
    st = osamp.reverse_step(sched, hist_rev, s_t, x_t, O_t, eps_theta, O0_theta, seq_post, m_str, t, noise)
    return {"seq_idx": seq["seq_idx"], "translations": st["translations"], "orientations": st["orientations"]}


def draw_initial_state(seq_idx, x, O, generation_mask, generator=None, generate_sequence=True,
                       generate_structure=True):
    """``oracle.sampler.draw_initial_state`` (same draws) with a modality that is off starting at its native value."""
    s, xT, OT = osamp.draw_initial_state(seq_idx, x, O, generation_mask, generator=generator)
    m_seq, m_str = modality_masks(generation_mask, generate_sequence, generate_structure)
    return (torch.where(m_seq, s, seq_idx), torch.where(m_str[..., None], xT, x),
            torch.where(m_str[..., None, None], OT, O))


def losses(denoised, noised, orientations_t0, generation_mask, residue_mask, generate_sequence=True,
           generate_structure=True):
    """``oracle.ipa.losses`` with the terms of a modality that is off summed over no residue; same denominator."""
    denom = (generation_mask & residue_mask).sum()
    m_seq, m_str = (m & residue_mask for m in modality_masks(generation_mask, generate_sequence, generate_structure))
    kl = torch.nn.functional.kl_div(denoised["seq_posterior"].log(), noised["seq_posterior"], reduction="none")
    mse = (denoised["translations_eps"] - noised["translations_eps"]).pow(2)
    rot = oipa.orientation_loss(denoised["orientations_t0"], orientations_t0)
    return ((kl * m_seq[..., None]).sum() / denom, (mse * m_str[..., None]).sum() / denom,
            (rot * m_str[..., None, None]).sum() / denom)
