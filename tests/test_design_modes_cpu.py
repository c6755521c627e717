"""CPU: the design-mode oracle (design_modes_oracle.py: fixed-backbone sequence design, structure prediction) against
the pinned co-design oracle, the argument checks of DiffAb's switches and of sample(init="native"), and the library's
refusal of a `generate` value outside 1..3."""
import ctypes

import pytest
import torch

import design_modes_oracle as mo
from diffab_pytorch_b200 import _lib, diffusion, synth
from diffab_pytorch_b200.diffab_pytorch import DiffAb
from oracle import diffusion as odiff
from oracle import ipa as oipa
from oracle import sampler as osamp
from oracle import so3 as oso3

MODES = [(True, False), (False, True)]      # (generate_sequence, generate_structure) besides co-design
SCHED = odiff.cosine_schedule(100, s=0.01, beta_max=0.999)


def _mode_id(mode):
    return {(True, False): "sequence", (False, True): "structure"}[mode]


@pytest.fixture(scope="module")
def noising():
    batch = synth.make_patches(3, 40, seed=21, cdr=(10, 25), with_distmat=False)
    hist = oso3.igso3_table(SCHED["one_minus_alpha_bar_sqrt"], n_bins=256, n_terms=64)
    t = torch.tensor([1, 37, 100])
    noise = odiff.draw_add_noise_tensors(3, 40, n_bins=256, generator=torch.Generator().manual_seed(5))
    args = (SCHED, hist, batch["seq_idx"], batch["xyz"][:, :, 1], batch["orientations"], batch["generation_mask"], t, noise)
    return batch, args


@pytest.mark.parametrize("mode", MODES, ids=_mode_id)
def test_oracle_add_noise_keeps_the_off_modality(noising, mode):
    batch, args = noising
    gs, gx = mode
    both = odiff.add_noise(*args)
    out = mo.add_noise(*args, generate_sequence=gs, generate_structure=gx)
    m = batch["generation_mask"]
    if gs:
        for k in ("seq_idx_t", "seq_posterior"):
            assert torch.equal(out[k], both[k]), k
        assert torch.equal(out["translations_t"], batch["xyz"][:, :, 1])
        assert torch.equal(out["orientations_t"], batch["orientations"])
        assert not torch.equal(both["translations_t"][m], batch["xyz"][:, :, 1][m])      # co-design does move them
    else:
        assert torch.equal(out["seq_idx_t"], batch["seq_idx"])
        assert torch.equal(out["seq_posterior"], torch.nn.functional.one_hot(batch["seq_idx"], 21).float())
        for k in ("translations_t", "orientations_t"):
            assert torch.equal(out[k], both[k]), k
    assert torch.equal(out["translations_eps"], both["translations_eps"])


def test_oracle_refuses_generating_nothing(noising):
    _, args = noising
    with pytest.raises(ValueError):
        mo.add_noise(*args, generate_sequence=False, generate_structure=False)
    with pytest.raises(ValueError):
        mo.modality_masks(torch.ones(2, 3, dtype=torch.bool), False, False)


@pytest.mark.parametrize("mode", MODES, ids=_mode_id)
def test_oracle_reverse_step_keeps_the_off_modality(mode):
    gs, gx = mode
    B, L = 3, 40
    g = torch.Generator().manual_seed(8)
    batch = synth.make_patches(B, L, seed=22, cdr=(5, 30), with_distmat=False)
    s, x, O = batch["seq_idx"], batch["xyz"][:, :, 1], batch["orientations"]
    eps = torch.randn(B, L, 3, generator=g)
    O0 = oso3.exp_vec(0.3 * torch.randn(B, L, 3, generator=g)) @ O
    post = torch.softmax(torch.randn(B, L, 21, generator=g), -1)
    hist_rev = oso3.igso3_table(osamp.reverse_sigmas(SCHED), n_bins=256, n_terms=64)
    noise = osamp.draw_step_noise(B, L, n_bins=256, generator=g)
    t = torch.tensor([1, 2, 60])
    args = (SCHED, hist_rev, s, x, O, eps, O0, post, batch["generation_mask"], t, noise)
    both = osamp.reverse_step(*args)
    out = mo.reverse_step(*args, generate_sequence=gs, generate_structure=gx)
    on, off = (("seq_idx",), ("translations", "orientations")) if gs else (("translations", "orientations"), ("seq_idx",))
    for k in on:
        assert torch.equal(out[k], both[k]), k
    old = {"seq_idx": s, "translations": x, "orientations": O}
    for k in off:
        assert torch.equal(out[k], old[k]), k
    with pytest.raises(ValueError):
        mo.reverse_step(*args, generate_sequence=False, generate_structure=False)


@pytest.mark.parametrize("mode", MODES, ids=_mode_id)
def test_oracle_losses_zero_the_off_terms(mode):
    gs, gx = mode
    B, L = 2, 30
    g = torch.Generator().manual_seed(9)
    pred = {"seq_posterior": torch.softmax(torch.randn(B, L, 21, generator=g, dtype=torch.float64), -1),
            "translations_eps": torch.randn(B, L, 3, generator=g, dtype=torch.float64),
            "orientations_t0": oso3.exp_vec(torch.randn(B, L, 3, generator=g, dtype=torch.float64))}
    noised = {"seq_posterior": torch.softmax(3 * torch.randn(B, L, 21, generator=g, dtype=torch.float64), -1),
              "translations_eps": torch.randn(B, L, 3, generator=g, dtype=torch.float64)}
    O_true = oso3.exp_vec(torch.randn(B, L, 3, generator=g, dtype=torch.float64))
    gm = torch.zeros(B, L, dtype=torch.bool)
    gm[:, 8:20] = True
    rm = torch.ones(B, L, dtype=torch.bool)
    rm[1, 10:12] = False
    both = oipa.losses(pred, noised, O_true, gm, rm)
    leaves = {k: v.clone().requires_grad_(True) for k, v in pred.items()}
    out = mo.losses(leaves, noised, O_true, gm, rm, generate_sequence=gs, generate_structure=gx)
    sum(out).backward()
    on, off = ((0,), (1, 2)) if gs else ((1, 2), (0,))
    for i in on:
        assert torch.equal(out[i].detach(), both[i]), i
    for i in off:
        assert float(out[i].detach()) == 0.0, i
    grads_off = ("translations_eps", "orientations_t0") if gs else ("seq_posterior",)
    for k in grads_off:
        assert bool((leaves[k].grad == 0).all()), k


def test_generate_bits():
    assert diffusion.generate_bits(True, True) == 3
    assert diffusion.generate_bits(True, False) == 1
    assert diffusion.generate_bits(False, True) == 2
    with pytest.raises(ValueError):
        diffusion.generate_bits(False, False)


def _cpu_model():
    return DiffAb(32, 16, 2, 8, 4, 4, 4, device="cpu")


def test_switches_are_plain_attributes_outside_the_state_dict():
    model = _cpu_model()
    keys = set(model.state_dict())
    assert model.generate_sequence is True and model.generate_structure is True
    model.generate_sequence = False
    assert set(model.state_dict()) == keys
    assert not any("generate" in k for k in keys)
    assert DiffAb.generate_sequence is True         # set per model, like train_precision


def test_generating_nothing_is_refused_where_the_switches_are_read():
    model = _cpu_model()
    model.generate_sequence = model.generate_structure = False
    batch = synth.make_patches(1, 8, seed=1, cdr=(2, 5))
    with pytest.raises(ValueError):
        model._shared_step(batch, 0)
    with pytest.raises(ValueError):
        model.sample(batch["seq_idx"], batch["xyz"], batch["orientations"], generation_mask=batch["generation_mask"])
    with pytest.raises(ValueError):
        model.sample_from_context(batch["seq_idx"], batch["xyz"][:, :, 1], batch["orientations"], None, None,
                                  batch["generation_mask"])


@pytest.mark.parametrize("kw", [dict(init="native", t_start=0), dict(init="native", t_start=101),
                                dict(init="native", t_start=-3), dict(init="posterior")])
def test_sample_refuses_a_bad_native_start(kw):
    model = _cpu_model()
    batch = synth.make_patches(1, 8, seed=1, cdr=(2, 5))
    with pytest.raises(ValueError):
        model.sample(batch["seq_idx"], batch["xyz"], batch["orientations"], generation_mask=batch["generation_mask"], **kw)


@pytest.mark.parametrize("generate", [0, 4, -1])
def test_library_refuses_generate_outside_1_to_3(generate):
    """The checks run before anything touches a device, so they are exercised here without a GPU."""
    lib = _lib.lib()
    fake = [ctypes.c_void_p(16 * (i + 1)) for i in range(5)]
    sched = _lib.DabSchedule(100, *fake)
    calls = {
        "dab_forward_noise": lambda: lib.dab_forward_noise(ctypes.byref(sched), *[None] * 5, 0, 0, *[None] * 3, generate,
                                                           *[None] * 5),
        "dab_reverse_step": lambda: lib.dab_reverse_step(ctypes.byref(sched), *[None] * 8, 0, 0, *[None] * 3, generate,
                                                         *[None] * 5),
        "dab_losses_fwd": lambda: lib.dab_losses_fwd(*[None] * 7, 1, generate, None, None, None),
        "dab_losses_bwd": lambda: lib.dab_losses_bwd(*[None] * 7, 1, generate, *[None] * 6),
    }
    for name, call in calls.items():
        assert call() == -1, name                                                   # DAB_EINVAL
        msg = lib.dab_last_error().decode()
        assert msg.startswith(name) and "generate must be 1 (sequence), 2 (structure) or 3 (both)" in msg, msg
    assert lib.dab_version() >= 101
