"""GPU: the amino-acid bias of sampling (DiffAb.sample(aa_bias=)) - the weighted draw of the reverse-step kernel against
the oracle rule (aa_bias_oracle.py), its statistics, sampling with weights against the oracle sampler (fp32 free running,
bf16 teacher-forced), graphed against eager, and full-size invariants of sample()."""
import pytest
import torch
from scipy import stats

import aa_bias_oracle as ao
import design_modes_oracle as mo
from conftest import load_golden
from diffab_pytorch_b200 import _lib, diffusion, so3, synth
from diffab_pytorch_b200.diffab_pytorch import DiffAb, aa_bias_weights, cast_pair_to_bf16
from oracle import diffusion as odiff
from oracle import ipa as oipa
from oracle import sampler as osamp
from oracle import so3 as oso3

pytestmark = pytest.mark.gpu
DEV = "cuda"
TRAIN = (128, 64, 6, 32, 8, 8, 8)
SCHED = odiff.cosine_schedule(100, s=0.01, beta_max=0.999)
INF = float("inf")
CTX_KEYS = ("seq_idx", "xyz", "orientations", "backbone_dihedrals", "distmat", "pairwise_dihedrals", "atom_mask",
            "chain_idx", "residue_idx", "generation_mask", "residue_mask")
CYS, UNK = 1, 20        # a fixed type standing in for cysteine (the letter order is not this package's), and AA_UNK


def _to(d):
    return {k: v.to(DEV) for k, v in d.items()}


def _model(generate_sequence=True, generate_structure=True, seed=0):
    model = DiffAb(*TRAIN, device=DEV)
    model.load_state_dict(synth.synthetic_state(load_golden("state_shapes.pt"), seed=seed))
    model.generate_sequence, model.generate_structure = generate_sequence, generate_structure
    return model.eval()


def _random_bias(B, L, seed, p_forbid=0.5):
    """Log-space bias: random values, a random share of the types forbidden per residue (type 3 always allowed)."""
    g = torch.Generator().manual_seed(seed)
    b = torch.randn(B, L, 21, generator=g)
    b[torch.rand(B, L, 21, generator=g) < p_forbid] = -INF
    b[..., 3] = 0.0
    return b


def _design_bias(B, L, seed):
    """C and UNK excluded everywhere, and a random half of the other types per residue."""
    b = _random_bias(B, L, seed)
    b[..., [CYS, UNK]] = -INF
    return b


# ---------------------------------------------------------------------------------------------------- kernel
@pytest.fixture(scope="module")
def tables():
    rev = so3.SO3(SCHED["beta"].sqrt(), device=DEV)
    return _lib.Schedule(SCHED, DEV), rev


@pytest.mark.parametrize("B,L", [(1, 128), (3, 37), (0, 128)])
@pytest.mark.parametrize("generate", [1, 3])
def test_weighted_reverse_step_vs_oracle(tables, generate, B, L):
    dsched, rev = tables
    lib = _lib.lib()
    if B == 0:
        w_ptr = _lib.ptr(torch.ones(1, 21, device=DEV))
        assert lib.dab_reverse_step_weighted(dsched.ref(), *[None] * 8, 0, L, *[None] * 3, w_ptr, generate,
                                             *[None] * 4, _lib.stream_ptr()) == 0
        assert lib.dab_reverse_step_weighted(dsched.ref(), *[None] * 8, 0, L, *[None] * 3, w_ptr, 0,
                                             *[None] * 4, _lib.stream_ptr()) == -1
        return
    g = torch.Generator().manual_seed(300 + B)
    batch = synth.make_patches(B, L, seed=33, cdr=(5, 30), with_distmat=False)
    s, x, O, m = batch["seq_idx"], batch["xyz"][:, :, 1].contiguous(), batch["orientations"], batch["generation_mask"]
    eps = torch.randn(B, L, 3, generator=g)
    v = 0.3 * torch.randn(B, L, 3, generator=g)
    post = torch.softmax(2 * torch.randn(B, L, 21, generator=g), -1)
    w = ao.weights(_random_bias(B, L, seed=B))
    gen_rows = m.nonzero()
    # fallback: posterior one-hot on a forbidden type; no eligible type: the old type stays
    r0, r1 = gen_rows[0], gen_rows[1]
    forb = int((w[r0[0], r0[1]] == 0).float().argmax())
    post[r0[0], r0[1]] = torch.nn.functional.one_hot(torch.tensor(forb), 21).float()
    w[r1[0], r1[1]] = 0.0
    t = torch.randint(1, 101, (B,), generator=g)
    t[0] = 1
    noise = osamp.draw_step_noise(B, L, generator=g)

    def run(weight):
        return {k: val.cpu() for k, val in diffusion.fused_reverse_step(
            dsched, rev, s.to(DEV), x.to(DEV), O.to(DEV), eps.to(DEV), v.to(DEV), post.to(DEV), m.to(DEV), t.to(DEV),
            _to(noise), return_O0=True, generate=generate,
            seq_weight=None if weight is None else weight.to(DEV)).items()}

    out, plain, ones = run(w), run(None), run(torch.ones(B, L, 21))
    for k in plain:
        assert torch.equal(ones[k], plain[k]), k                      # all-ones weights = no weights, bit for bit
        if k != "seq_idx":
            assert torch.equal(out[k], plain[k]), k                   # the weights change the sequence only
    gm = m if generate & 1 else torch.zeros_like(m)
    O0 = O @ oso3.exp_vec(v)
    ref = ao.reverse_step(SCHED, rev.histograms.cpu(), s, x, O, eps, O0, post, gm, t, noise, w)
    assert torch.equal(out["seq_idx"], ref["seq_idx"])
    assert torch.equal(out["seq_idx"][~gm], s[~gm])
    if generate & 1:
        drawn = w.gather(-1, out["seq_idx"][..., None])[..., 0]
        r0m = torch.zeros_like(m)
        r0m[r0[0], r0[1]] = True
        r1m = torch.zeros_like(m)
        r1m[r1[0], r1[1]] = True
        assert bool((drawn[m & ~r1m] > 0).all())
        assert int(out["seq_idx"][r0[0], r0[1]]) != forb                     # the fallback lands on an allowed type
        assert int(out["seq_idx"][r1[0], r1[1]]) == int(s[r1[0], r1[1]])     # no eligible type: keeps its type
        assert not torch.equal(out["seq_idx"], plain["seq_idx"])


def _chi_square(counts, probs):
    keep = probs > 0
    assert int(counts[~keep].sum()) == 0
    n = int(counts.sum())
    exp = probs[keep] / probs[keep].sum() * n
    return stats.chisquare(counts[keep].double().numpy(), exp.double().numpy()).pvalue


def test_weighted_draw_is_a_sample_of_p_w(tables):
    """~10^6 residues sharing one posterior and one weight row: the frequencies match p w / sum(p w)."""
    dsched, rev = tables
    B, L = 8192, 128
    g = torch.Generator(device=DEV).manual_seed(7)
    p = torch.softmax(torch.linspace(-2.0, 1.5, 21), -1)
    b = torch.linspace(0.0, -2.0, 21)
    b[[CYS, UNK, 7, 12]] = -INF
    w = ao.weights(b)
    post = p.to(DEV).expand(B, L, 21).contiguous()
    weight = w.to(DEV).expand(B, L, 21).contiguous()
    s = torch.zeros(B, L, dtype=torch.int64, device=DEV)
    x = torch.zeros(B, L, 3, device=DEV)
    O = torch.eye(3, device=DEV).expand(B, L, 3, 3).contiguous()
    noise = {"seq_exp": torch.empty(B * L, 21, device=DEV).exponential_(generator=g),
             "z": torch.zeros(B, L, 3, device=DEV)}
    out = diffusion.fused_reverse_step(dsched, rev, s, x, O, x, x, post, torch.ones(B, L, dtype=torch.bool, device=DEV),
                                       torch.full((B,), 50, device=DEV), noise, rotvec=torch.zeros(B, L, 3, device=DEV),
                                       generate=1, seq_weight=weight)
    counts = torch.bincount(out["seq_idx"].view(-1), minlength=21).cpu()
    assert _chi_square(counts, (p * w).double()) > 1e-3
    # the prior under the same weights: w / sum(w)
    prior = DiffAb.draw_prior_sequence(B, L, DEV, generator=torch.Generator(device=DEV).manual_seed(8),
                                       seq_weight=weight)
    counts = torch.bincount(prior.view(-1), minlength=21).cpu()
    assert _chi_square(counts, w.double()) > 1e-3


# ---------------------------------------------------------------------------------------------------- sampling
def _context(model, b):
    with torch.no_grad():
        return model.encode_context(*[b[k] for k in CTX_KEYS])


def test_free_running_fp32_steps_vs_oracle_sampler_with_weights():
    model = _model()
    batch = synth.make_patches(2, 128, seed=9)
    res, pair = _context(model, _to(batch))
    gen = torch.Generator().manual_seed(4)
    m = batch["generation_mask"]
    w = ao.weights(_design_bias(2, 128, seed=5))
    s, x, O = osamp.draw_initial_state(batch["seq_idx"], batch["xyz"][:, :, 1], batch["orientations"], m, generator=gen)
    noises = {t: osamp.draw_step_noise(2, 128, generator=gen) for t in range(100, 95, -1)}
    state = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    hist_rev = model.so3_reverse.histograms.cpu()
    near_tie = torch.zeros(2, dtype=torch.bool)
    rs, rx, rO = s, x, O
    for step in range(100, 95, -1):
        tt = torch.full((2,), step, dtype=torch.long)
        den = oipa.denoiser_forward(state, rs, rx, rO, res.cpu(), pair.cpu(), SCHED["beta"][tt], 6, 8)
        key = torch.where(w > 0, den["seq_posterior"] * w, torch.tensor(0.0)).reshape(-1, 21) / noises[step]["seq_exp"]
        top2 = key.topk(2, dim=-1).values
        near_tie |= (((top2[:, 0] - top2[:, 1]) / top2[:, 0]).view(2, -1) < 1e-4).logical_and(m).any(dim=1)
        nxt = ao.reverse_step(SCHED, hist_rev, rs, rx, rO, den["translations_eps"], den["orientations_t0"],
                              den["seq_posterior"], m, tt, noises[step], w)
        rs, rx, rO = nxt["seq_idx"], nxt["translations"], nxt["orientations"]
    got = model.sample_from_context(s.to(DEV), x.to(DEV), O.to(DEV), res, pair, m.to(DEV),
                                    noises={t: _to(n) for t, n in noises.items()}, t_start=100, t_stop=96,
                                    seq_weight=w.to(DEV))
    got = {k: v.cpu() for k, v in got.items()}
    assert torch.equal(got["seq_idx"][~m], s[~m])
    assert bool((w.gather(-1, got["seq_idx"][..., None])[..., 0][m] > 0).all())
    same = (got["seq_idx"] == rs).all(dim=1)
    assert bool((same | near_tie).all()), "sequence differs in a patch without any near-tie in the oracle"
    assert bool(same.any())
    for p_ in range(2):
        if bool(same[p_]):
            assert float((got["translations"][p_] - rx[p_]).norm(dim=-1)[m[p_]].max()) < 1e-2
            assert float((got["orientations"][p_] - rO[p_]).abs().amax(dim=(-1, -2))[m[p_]].max()) < 1e-2


def test_bf16_graph_steps_teacher_forced_with_weights():
    """The t = 10..6 window of tests/test_gpu_sampling_parity.py with weights: fp64 oracle on the bf16-rounded pair
    tensor, teacher-forced, injected draws; a sequence may differ only where the oracle's weighted top-2 margin is within
    what the bf16 posterior error allows."""
    model = _model()
    batch = synth.make_patches(2, 128, seed=9)
    b = _to(batch)
    B, L = 2, 128
    m = batch["generation_mask"]
    w = ao.weights(_design_bias(B, L, seed=6))
    res, pair = _context(model, b)
    pair16 = cast_pair_to_bf16(pair)
    state64 = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
    res64, pair64 = res.cpu().double(), pair16.float().cpu().double()
    hist_rev = model.so3_reverse.histograms.cpu()
    torch.manual_seed(7)
    noised = odiff.add_noise(SCHED, model.orientation_diffuser.so3.histograms.cpu(), batch["seq_idx"],
                             batch["xyz"][:, :, 1], batch["orientations"], m, torch.full((B,), 10),
                             odiff.draw_add_noise_tensors(B, L))
    s, x, O = noised["seq_idx_t"], noised["translations_t"], noised["orientations_t"]
    glue = model.denoiser.sampling_cache(res)
    planes = model._pair_bias_planes(pair16)
    gen = torch.Generator().manual_seed(50)
    for step in range(10, 5, -1):
        noise = osamp.draw_step_noise(B, L, generator=gen)
        tt = torch.full((B,), step, dtype=torch.long)
        den = oipa.denoiser_forward(state64, s, x.double(), O.double(), res64, pair64, SCHED["beta"][tt].double(), 6, 8)
        ref = ao.reverse_step(SCHED, hist_rev, s, x.double(), O.double(), den["translations_eps"],
                              den["orientations_t0"], den["seq_posterior"], m, tt,
                              {k: v.double() if v.dtype.is_floating_point else v for k, v in noise.items()}, w)
        key = (den["seq_posterior"] * w.double()).reshape(-1, 21) / noise["seq_exp"].double()
        top2 = key.topk(2, dim=-1).values
        margin = ((top2[:, 0] - top2[:, 1]) / top2[:, 0]).view(B, -1)
        args = (s.to(DEV), x.float().to(DEV), O.float().to(DEV), res, pair16, b["generation_mask"])
        kw = dict(noises={step: _to(noise)}, t_start=step, t_stop=step, seq_weight=w.to(DEV))
        eager = model.sample_from_context(*args, use_cuda_graph=False, **kw)
        graph = model.sample_from_context(*args, use_cuda_graph=True, **kw)
        for k in eager:
            assert torch.equal(eager[k], graph[k]), (step, k)
        with torch.no_grad():
            _, _, post = model.denoiser.heads_fast(args[0], args[1], args[2], glue, pair16,
                                                   model.dsched.tensors["beta"][tt.to(DEV)], planes)
        p_ref = den["seq_posterior"]
        d_rel = float(((post.cpu().double() - p_ref).abs() / p_ref)[p_ref > 1e-3].max())
        assert d_rel < 2e-2, (step, d_rel)
        got = {k: v.cpu() for k, v in eager.items()}
        diff = got["seq_idx"] != ref["seq_idx"]
        assert not diff[~m].any()
        assert not (diff & ~(margin <= 2 * d_rel / (1 - d_rel))).any(), step
        assert bool((w.gather(-1, got["seq_idx"][..., None])[..., 0][m] > 0).all())
        step_len = (ref["translations"] - x.double()).norm(dim=-1)[m]
        dx = (got["translations"].double() - ref["translations"]).norm(dim=-1)[m]
        assert float(dx.max() / step_len.mean()) < 1e-2, step
        s, x, O = ref["seq_idx"], ref["translations"].float(), ref["orientations"].float()     # teacher forcing


def _bf16_setup(seed=11):
    model = _model()
    batch = synth.make_patches(2, 128, seed=seed)
    res, pair = _context(model, _to(batch))
    gen = torch.Generator().manual_seed(3)
    s, x, O = osamp.draw_initial_state(batch["seq_idx"], batch["xyz"][:, :, 1], batch["orientations"],
                                       batch["generation_mask"], generator=gen)
    noises = {t: _to(osamp.draw_step_noise(2, 128, generator=gen)) for t in range(100, 78, -1)}
    return model, batch, (s.to(DEV), x.to(DEV), O.to(DEV), res, cast_pair_to_bf16(pair),
                          batch["generation_mask"].to(DEV)), noises


def test_graphed_loop_equals_eager_loop_with_weights():
    """22 steps (one replay of the 20-step block graph, two single-step replays); a second graphed call with other
    weight values follows them without a recapture."""
    model, batch, args, noises = _bf16_setup()
    kw = dict(noises=noises, t_start=100, t_stop=79)
    m = batch["generation_mask"]
    for i, seed in enumerate((1, 2)):
        w = ao.weights(_design_bias(2, 128, seed=seed)).to(DEV)
        eager = model.sample_from_context(*args, use_cuda_graph=False, seq_weight=w, **kw)
        graph = model.sample_from_context(*args, use_cuda_graph=True, seq_weight=w, **kw)
        if i == 0:
            captured = (model._graph_cache["graph"], model._graph_cache["graph_block"])
        else:
            assert (model._graph_cache["graph"], model._graph_cache["graph_block"]) == captured     # no recapture
        for k in eager:
            assert torch.equal(eager[k], graph[k]), (seed, k)
        assert bool((w.cpu().gather(-1, graph["seq_idx"].cpu()[..., None])[..., 0][m] > 0).all())
        assert torch.equal(graph["seq_idx"].cpu()[~m], args[0].cpu()[~m])


def test_alternating_weights_and_no_weights_equal_fresh_runs():
    model, batch, args, noises = _bf16_setup()
    kw = dict(noises=noises, t_start=100, t_stop=79, use_cuda_graph=True)
    w = ao.weights(_design_bias(2, 128, seed=3)).to(DEV)
    fresh = {"w": _model().sample_from_context(*args, seq_weight=w, **kw),
             "none": _model().sample_from_context(*args, **kw)}
    assert not torch.equal(fresh["w"]["seq_idx"], fresh["none"]["seq_idx"])
    for which in ("w", "none", "w", "none"):
        got = model.sample_from_context(*args, seq_weight=w if which == "w" else None, **kw)
        for k in got:
            assert torch.equal(got[k], fresh[which][k]), (which, k)


def test_launches_per_reverse_step_do_not_depend_on_the_weights():
    counts = {}
    model, batch, args, noises = _bf16_setup()
    w = ao.weights(_design_bias(2, 128, seed=4)).to(DEV)
    for which, weight in (("none", None), ("w", w)):
        model.sample_from_context(*args, noises=noises, t_start=100, t_stop=100, seq_weight=weight)     # warm caches
        torch.cuda.synchronize()
        n0 = _lib.lib().dab_launch_count()
        model.sample_from_context(*args, noises=noises, t_start=99, t_stop=99, seq_weight=weight)
        torch.cuda.synchronize()
        counts[which] = _lib.lib().dab_launch_count() - n0
    assert counts["none"] == counts["w"], counts


# ---------------------------------------------------------------------------------------------------- full size
def _check_invariants(out, batch, bias, structure_moves=True):
    m = batch["generation_mask"]
    allowed = (bias > -INF).expand(*out["seq_idx"].shape, 21)
    assert bool(allowed.gather(-1, out["seq_idx"][..., None])[..., 0][m].all())
    assert torch.equal(out["seq_idx"][~m], batch["seq_idx"][~m])
    assert torch.equal(out["translations"][~m], batch["xyz"][:, :, 1][~m])
    assert torch.equal(out["orientations"][~m], batch["orientations"][~m])
    if structure_moves:
        O = out["orientations"][m].double()
        assert float((O.transpose(-1, -2) @ O - torch.eye(3, dtype=torch.float64)).abs().max()) < 1e-4
        assert float((torch.linalg.det(O) - 1).abs().max()) < 1e-4
        assert torch.isfinite(out["translations"]).all()
    else:
        assert torch.equal(out["translations"], batch["xyz"][:, :, 1])
        assert torch.equal(out["orientations"], batch["orientations"])


@pytest.mark.parametrize("L", [128, 100, 200])
def test_full_size_sampling_obeys_the_bias(L):
    """B = 256 at L = 128, L = 100 (padded to 128) and L = 200 (two 128-residue key blocks)."""
    B = 256
    model = _model()
    batch = synth.make_patches(B, L, seed=77, with_distmat=False, cdr=(56, 72))
    args = [batch[k] if k != "distmat" else None for k in CTX_KEYS]
    bias = _design_bias(B, L, seed=L)
    torch.manual_seed(5)
    out = {k: v.cpu() for k, v in model.sample(*args, precision="bf16", aa_bias=bias).items()}
    _check_invariants(out, batch, bias)


def test_native_start_and_fixed_backbone_obey_the_bias():
    B, L = 256, 128
    batch = synth.make_patches(B, L, seed=78, with_distmat=False, cdr=(56, 72))
    args = [batch[k] if k != "distmat" else None for k in CTX_KEYS]
    bias = _design_bias(B, L, seed=9)[0]                 # (L, 21): one bias shared by the patches
    torch.manual_seed(6)
    model = _model()
    out = {k: v.cpu() for k, v in model.sample(*args, precision="bf16", aa_bias=bias, init="native", t_start=30).items()}
    _check_invariants(out, batch, bias)
    model = _model(generate_structure=False)
    out = {k: v.cpu() for k, v in model.sample(*args, precision="bf16", aa_bias=bias).items()}
    _check_invariants(out, batch, bias, structure_moves=False)
    model = _model(generate_sequence=False)
    with pytest.raises(ValueError, match="generate_sequence"):
        model.sample(*args, precision="bf16", aa_bias=bias)


def test_sample_without_bias_is_unchanged_and_zero_bias_matches_it():
    """aa_bias = 0 everywhere gives the weights 1: the reverse steps are the unweighted ones, only the prior draws
    differently (Exp(1) race instead of randint).  With a seeded generator and init="native" (no prior draw) the
    results are identical."""
    B, L = 4, 128
    batch = synth.make_patches(B, L, seed=79, with_distmat=False, cdr=(56, 72))
    args = [batch[k] if k != "distmat" else None for k in CTX_KEYS]
    model = _model()
    run = lambda **kw: model.sample(*args, precision="fp32", init="native", t_start=5,
                                    generator=torch.Generator(device=DEV).manual_seed(2), **kw)
    plain, zero = run(), run(aa_bias=torch.zeros(21))
    for k in plain:
        assert torch.equal(plain[k], zero[k]), k
    assert aa_bias_weights(torch.zeros(21), torch.ones(1, 1, dtype=torch.bool, device=DEV)).is_cuda
