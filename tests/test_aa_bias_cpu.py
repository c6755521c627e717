"""CPU: the amino-acid bias of sampling (DiffAb.sample(aa_bias=)) - the oracle's weighted draw against the pinned
sampler, the conversion and checks of aa_bias_weights, the argument checks of dab_reverse_step_weighted (they run before
anything touches a device) and the sharding of a per-patch bias by distributed.sample_sharded."""
import ctypes

import pytest
import torch

import aa_bias_oracle as ao
from diffab_pytorch_b200 import _lib, synth
from diffab_pytorch_b200 import distributed as dd
from diffab_pytorch_b200.diffab_pytorch import DiffAb, aa_bias_weights
from oracle import diffusion as odiff
from oracle import sampler as osamp
from oracle import so3 as oso3

SCHED = odiff.cosine_schedule(100, s=0.01, beta_max=0.999)
INF = float("inf")


def _step_args(B=3, L=40, seed=8):
    g = torch.Generator().manual_seed(seed)
    batch = synth.make_patches(B, L, seed=22, cdr=(5, 30), with_distmat=False)
    s, x, O = batch["seq_idx"], batch["xyz"][:, :, 1], batch["orientations"]
    eps = torch.randn(B, L, 3, generator=g)
    O0 = oso3.exp_vec(0.3 * torch.randn(B, L, 3, generator=g)) @ O
    post = torch.softmax(3 * torch.randn(B, L, 21, generator=g), -1)
    hist_rev = oso3.igso3_table(osamp.reverse_sigmas(SCHED), n_bins=256, n_terms=64)
    noise = osamp.draw_step_noise(B, L, n_bins=256, generator=g)
    t = torch.tensor([1, 2, 60])[:B]
    return [SCHED, hist_rev, s, x, O, eps, O0, post, batch["generation_mask"], t, noise]


def _random_weights(B, L, seed, p_zero=0.5):
    g = torch.Generator().manual_seed(seed)
    b = torch.randn(B, L, 21, generator=g)
    b[torch.rand(B, L, 21, generator=g) < p_zero] = -INF
    b[..., 3] = 0.0                          # at least one allowed type per residue
    return ao.weights(b)


# ------------------------------------------------------------------------------------------------------------ oracle
def test_oracle_with_all_ones_weights_is_the_sampler_bit_for_bit():
    args = _step_args()
    B, L = args[2].shape
    ref = osamp.reverse_step(*args)
    out = ao.reverse_step(*args, torch.ones(B, L, 21))
    for k in ref:
        assert torch.equal(out[k], ref[k]), k


def test_oracle_never_draws_a_forbidden_type_and_keeps_positions():
    args = _step_args()
    B, L = args[2].shape
    w = _random_weights(B, L, seed=3)
    ref = osamp.reverse_step(*args)
    out = ao.reverse_step(*args, w)
    m = args[8]
    drawn = w.gather(-1, out["seq_idx"][..., None])[..., 0]
    assert bool((drawn[m] > 0).all())
    assert torch.equal(out["seq_idx"][~m], args[2][~m])
    assert torch.equal(out["translations"], ref["translations"]) and torch.equal(out["orientations"], ref["orientations"])
    assert not torch.equal(out["seq_idx"], ref["seq_idx"])          # the weights do change the draw


def test_oracle_weighted_draw_is_argmax_of_p_w_over_q():
    g = torch.Generator().manual_seed(1)
    N = 4096
    post = torch.softmax(2 * torch.randn(N, 21, generator=g), -1)
    q = torch.empty(N, 21).exponential_(generator=g)
    w = _random_weights(1, N, seed=2)[0]
    got = ao.weighted_draw(post, q, w, torch.full((N,), -7))
    ref = torch.where(w > 0, post * w / q, torch.tensor(-1.0)).argmax(-1)
    assert torch.equal(got, ref)


def test_oracle_fallback_draws_from_the_weights_alone():
    """A posterior one-hot on a forbidden type leaves every eligible key at 0: the draw is redone with w / q."""
    g = torch.Generator().manual_seed(4)
    N = 512
    w = _random_weights(1, N, seed=5)[0]
    forbidden = (w == 0).float().argmax(-1)                  # one forbidden type per row
    assert bool((w.gather(-1, forbidden[:, None]) == 0).all())
    post = torch.nn.functional.one_hot(forbidden, 21).float()
    q = torch.empty(N, 21).exponential_(generator=g)
    got = ao.weighted_draw(post, q, w, torch.full((N,), -7))
    assert bool((w.gather(-1, got[:, None]) > 0).all())
    assert torch.equal(got, torch.where(w > 0, w / q, torch.tensor(-1.0)).argmax(-1))
    assert not bool((got == 0).all())                         # not "index 0 by tie-break"


def test_oracle_row_without_an_eligible_type_keeps_its_type():
    post = torch.softmax(torch.randn(4, 21), -1)
    q = torch.ones(4, 21)
    w = torch.ones(4, 21)
    w[1] = 0.0
    w[3] = 0.0
    old = torch.tensor([5, 6, 7, 8])
    got = ao.weighted_draw(post, q, w, old)
    assert int(got[1]) == 6 and int(got[3]) == 8
    assert torch.equal(got[[0, 2]], post[[0, 2]].argmax(-1))


# ------------------------------------------------------------------------------------------------- aa_bias_weights
@pytest.mark.parametrize("shape", [(21,), (7, 21), (2, 7, 21)])
def test_weights_of_every_accepted_shape(shape):
    B, L = 2, 7
    g = torch.Generator().manual_seed(len(shape))
    b = torch.randn(*shape, generator=g)
    b[..., 4] = -INF
    m = torch.zeros(B, L, dtype=torch.bool)
    m[:, 2:5] = True
    w = aa_bias_weights(b, m)
    assert w.shape == (B, L, 21) and w.dtype == torch.float32 and w.is_contiguous()
    full = b.expand(B, L, 21)
    assert torch.equal(w, torch.exp(full - full.amax(-1, keepdim=True)))
    assert bool((w[..., 4] == 0).all())
    assert bool((w.amax(-1) == 1).all()) and bool((w >= 0).all())


def test_weights_of_a_constant_bias_are_ones_and_none_stays_none():
    m = torch.ones(3, 5, dtype=torch.bool)
    assert aa_bias_weights(None, m) is None
    assert torch.equal(aa_bias_weights(torch.zeros(21), m), torch.ones(3, 5, 21))
    assert torch.equal(aa_bias_weights(torch.full((5, 21), -3.5, dtype=torch.float64), m), torch.ones(3, 5, 21))


def test_context_residue_may_forbid_everything():
    m = torch.zeros(1, 4, dtype=torch.bool)
    m[0, :2] = True
    b = torch.zeros(1, 4, 21)
    b[0, 3] = -INF                        # a context residue: never drawn, so it is no error
    w = aa_bias_weights(b, m)
    assert bool(torch.isfinite(w).all()) and bool((w[0, 3] == 0).all()) and bool((w[0, :3] == 1).all())


def _bad_bias(kind, B=2, L=6):
    b = torch.zeros(B, L, 21)
    if kind == "nan":
        b[1, 2, 5] = float("nan")
    elif kind == "+inf":
        b[0, 0, 0] = INF
    elif kind == "all -inf":
        b[1, 3] = -INF                    # residue 3 is generated
    elif kind == "short":
        b = torch.zeros(20)
    elif kind == "long L":
        b = torch.zeros(L + 1, 21)
    elif kind == "wrong B":
        b = torch.zeros(B + 1, L, 21)
    elif kind == "4-d":
        b = torch.zeros(2, B, L, 21)
    return b


@pytest.mark.parametrize("kind", ["nan", "+inf", "all -inf", "short", "long L", "wrong B", "4-d"])
def test_weights_refuse(kind):
    m = torch.zeros(2, 6, dtype=torch.bool)
    m[:, 2:5] = True
    with pytest.raises(ValueError, match="aa_bias"):
        aa_bias_weights(_bad_bias(kind), m)


def test_weights_refuse_a_mode_without_sequence_generation():
    m = torch.ones(2, 6, dtype=torch.bool)
    with pytest.raises(ValueError, match="generate_sequence"):
        aa_bias_weights(torch.zeros(21), m, generate_sequence=False)


def _cpu_model():
    return DiffAb(32, 16, 2, 8, 4, 4, 4, device="cpu")


def test_sample_checks_aa_bias_before_any_work():
    """sample() validates the bias first: these raise on a CPU model, before anything would need a device."""
    batch = synth.make_patches(1, 8, seed=1, cdr=(2, 5))
    args = (batch["seq_idx"], batch["xyz"], batch["orientations"])
    model = _cpu_model()
    bad = torch.zeros(8, 21)
    bad[3] = -INF                                                    # residue 3 is generated (cdr 2..5)
    with pytest.raises(ValueError, match="every residue type"):
        model.sample(*args, generation_mask=batch["generation_mask"], aa_bias=bad)
    model.generate_sequence = False                                  # structure prediction
    with pytest.raises(ValueError, match="generate_sequence"):
        model.sample(*args, generation_mask=batch["generation_mask"], aa_bias=torch.zeros(21))


# ------------------------------------------------------------------------------------------ dab_reverse_step_weighted
def _weighted_call(generate=3, B=0, L=0, pointers=None, weight=None):
    lib = _lib.lib()
    fake = [ctypes.c_void_p(16 * (i + 1)) for i in range(5)]
    sched = _lib.DabSchedule(100, *fake)
    p = pointers if pointers is not None else [None] * 15
    return lib.dab_reverse_step_weighted(ctypes.byref(sched), *p[:8], B, L, *p[8:11], weight, generate, *p[11:15], None)


@pytest.mark.parametrize("generate", [0, 4, -1])
def test_weighted_entry_refuses_a_bad_generate(generate):
    assert _weighted_call(generate) == -1
    msg = _lib.lib().dab_last_error().decode()
    assert msg.startswith("dab_reverse_step_weighted") and "generate must be 1 (sequence), 2 (structure) or 3" in msg
    assert _lib.lib().dab_version() >= 102


@pytest.mark.parametrize("B,L", [(-1, 4), (2, -3)])
def test_weighted_entry_refuses_negative_sizes(B, L):
    assert _weighted_call(B=B, L=L) == -1
    assert "dab_reverse_step_weighted: negative size" in _lib.lib().dab_last_error().decode()


@pytest.mark.parametrize("missing", range(14))
def test_weighted_entry_refuses_null_pointers(missing):
    """Each of the 14 required tensors (O0_out, the 15th, and seq_weight are optional) missing with B * L > 0."""
    p = [ctypes.c_void_p(256 * (i + 1)) for i in range(15)]
    p[14] = None
    p[missing] = None
    assert _weighted_call(B=2, L=3, pointers=p, weight=ctypes.c_void_p(4096)) == -1
    assert "dab_reverse_step_weighted: null pointer" in _lib.lib().dab_last_error().decode()


@pytest.mark.parametrize("B,L", [(0, 128), (5, 0), (0, 0)])
def test_weighted_entry_accepts_an_empty_batch(B, L):
    assert _weighted_call(B=B, L=L) == 0
    assert _weighted_call(B=B, L=L, weight=ctypes.c_void_p(4096)) == 0


def test_weighted_entry_refuses_an_incomplete_schedule():
    lib = _lib.lib()
    sched = _lib.DabSchedule(100, None, None, None, None, None)
    assert lib.dab_reverse_step_weighted(ctypes.byref(sched), *[None] * 8, 0, 0, *[None] * 4, 3, *[None] * 5) == -1
    assert "dab_reverse_step_weighted: incomplete schedule" in lib.dab_last_error().decode()


# ------------------------------------------------------------------------------------------------- sample_sharded
class _RecordingModel:
    def __init__(self):
        self.calls = []

    def sample(self, *args, **kwargs):
        self.calls.append((args, kwargs))
        return {"seq_idx": args[0].clone()}


@pytest.mark.parametrize("world", [2, 3])
def test_sample_sharded_hands_each_rank_its_slice_of_the_bias(monkeypatch, world):
    n, L = 7, 5
    batch = synth.make_patches(n, L, seed=2, cdr=(1, 3), with_distmat=False)
    batch["aa_bias"] = torch.randn(n, L, 21)
    monkeypatch.setattr(dd, "all_gather_samples", lambda out, n_total, group=None: out)
    seen = []
    for rank in range(world):
        monkeypatch.setattr(dd, "world_info", lambda group=None, r=rank: (r, world))
        model = _RecordingModel()
        dd.sample_sharded(model, batch, precision="fp32")
        (args, kwargs), = model.calls
        lo, hi = dd.shard_bounds(n, world)[rank]
        assert torch.equal(kwargs["aa_bias"], batch["aa_bias"][lo:hi])
        assert torch.equal(args[0], batch["seq_idx"][lo:hi])
        assert kwargs["precision"] == "fp32"
        seen.append(kwargs["aa_bias"])
    assert torch.equal(torch.cat(seen), batch["aa_bias"])


def test_sample_sharded_passes_a_shared_bias_through():
    batch = synth.make_patches(4, 5, seed=2, cdr=(1, 3), with_distmat=False)
    shared = torch.randn(21)
    model = _RecordingModel()
    dd.sample_sharded(model, batch, aa_bias=shared)
    assert model.calls[0][1]["aa_bias"] is shared
    model = _RecordingModel()
    dd.sample_sharded(model, batch)
    assert "aa_bias" not in model.calls[0][1]
    with pytest.raises(ValueError):
        dd.sample_sharded(_RecordingModel(), dict(batch, aa_bias=torch.zeros(4, 5, 21)), aa_bias=shared)


def test_prior_under_weights_is_the_oracle_draw_and_never_forbidden():
    B, L = 64, 40
    w = _random_weights(B, L, seed=9)
    got = DiffAb.draw_prior_sequence(B, L, "cpu", generator=torch.Generator().manual_seed(3), seq_weight=w)
    E = torch.empty(B * L, 21).exponential_(generator=torch.Generator().manual_seed(3))
    assert torch.equal(got.view(-1), ao.prior_draw(w.view(-1, 21), E))
    assert bool((w.gather(-1, got[..., None]) > 0).all())
    plain = DiffAb.draw_prior_sequence(B, L, "cpu", generator=torch.Generator().manual_seed(3))
    assert torch.equal(plain, torch.randint(0, 21, (B, L), generator=torch.Generator().manual_seed(3)))
