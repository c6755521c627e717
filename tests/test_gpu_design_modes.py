"""GPU: design modes - fixed-backbone sequence design (generate = 1), structure prediction (2) and co-design (3) - through
the fused kernels, the training step (eager, mixed precision, graphed), sampling (eager, graphed, full size) and the
optimisation of a native design (sample(init="native")), against the moded oracle and against co-design."""
import pytest
import torch

import design_modes_oracle as mo
from conftest import load_golden
from diffab_pytorch_b200 import _lib, diffusion, so3, synth
from diffab_pytorch_b200.diffab_pytorch import DiffAb, _FusedLosses, cast_pair_to_bf16
from oracle import diffusion as odiff
from oracle import ipa as oipa
from oracle import sampler as osamp
from oracle import so3 as oso3

pytestmark = pytest.mark.gpu
DEV = "cuda"
TRAIN = (128, 64, 6, 32, 8, 8, 8)
SMALL = (32, 16, 2, 8, 4, 4, 4)
FLAGS = {1: (True, False), 2: (False, True), 3: (True, True)}    # generate -> (generate_sequence, generate_structure)
MODES = [1, 2, 3]
SCHED = odiff.cosine_schedule(100, s=0.01, beta_max=0.999)
HEADS = {"seq": ("sequence_denoising",), "str": ("coordinate_denoising", "orientation_denoising")}
CTX_KEYS = ("seq_idx", "xyz", "orientations", "backbone_dihedrals", "distmat", "pairwise_dihedrals", "atom_mask",
            "chain_idx", "residue_idx", "generation_mask", "residue_mask")


def _to(d):
    return {k: v.to(DEV) for k, v in d.items()}


def _flags(generate):
    gs, gx = FLAGS[generate]
    return {"generate_sequence": gs, "generate_structure": gx}


def _set_mode(model, generate):
    model.generate_sequence, model.generate_structure = FLAGS[generate]
    return model


def _model(generate, cfg=TRAIN, seed=0):
    model = DiffAb(*cfg, device=DEV)
    if cfg == TRAIN:
        model.load_state_dict(synth.synthetic_state(load_golden("state_shapes.pt"), seed=seed))
    return _set_mode(model.eval(), generate)


def _context(model, b, generate):
    with torch.no_grad():
        return model.encode_context(*[b[k] for k in CTX_KEYS], **_flags(generate))


def _off_heads(generate):
    gs, gx = FLAGS[generate]
    return (() if gs else HEADS["seq"]) + (() if gx else HEADS["str"])


def _assert_off_heads_zero(model, generate):
    for name, p in model.denoiser.named_parameters():
        if name.split(".")[0] in _off_heads(generate):
            assert p.grad is None or bool((p.grad == 0).all()), name


# ---------------------------------------------------------------------------------------------------- kernels
@pytest.fixture(scope="module")
def tables():
    od = diffusion.OrientationDiffuser(T=100, s=0.01, beta_max=0.999, device=DEV)
    rev = so3.SO3(SCHED["beta"].sqrt(), device=DEV)
    return _lib.Schedule(SCHED, DEV), od.so3, rev


SIZES = [(1, 128), (3, 37), (0, 128)]      # B = 1; B * L = 111, not a multiple of the 128-residue block; empty batch


def _check_empty_batch(dsched, generate, L):
    """B = 0 at the C entry points (the IGSO(3) draw in front of them refuses an empty batch): nothing to launch, so the
    call succeeds without touching its (null) tensors - and a bad `generate` is still refused."""
    lib = _lib.lib()
    for bits, rc in ((generate, 0), (0, -1)):
        assert lib.dab_forward_noise(dsched.ref(), *[None] * 5, 0, L, *[None] * 3, bits, *[None] * 4,
                                     _lib.stream_ptr()) == rc
        assert lib.dab_reverse_step(dsched.ref(), *[None] * 8, 0, L, *[None] * 3, bits, *[None] * 4,
                                    _lib.stream_ptr()) == rc


@pytest.mark.parametrize("B,L", SIZES)
@pytest.mark.parametrize("generate", MODES)
def test_forward_noise_per_mode(tables, generate, B, L):
    dsched, table, _ = tables
    if B == 0:
        _check_empty_batch(dsched, generate, L)
        return
    g = torch.Generator().manual_seed(100 + B)
    batch = {k: v[:B] for k, v in synth.make_patches(max(B, 1), L, seed=31, cdr=(5, 30), with_distmat=False).items()}
    seq0, x0, O0, m = batch["seq_idx"], batch["xyz"][:, :, 1].contiguous(), batch["orientations"], batch["generation_mask"]
    t = torch.randint(1, 101, (B,), generator=g)
    if B:
        t[0] = 1
    noise = odiff.draw_add_noise_tensors(B, L, generator=g)
    run = lambda gen: {k: v.cpu() for k, v in diffusion.fused_add_noise(
        dsched, table, seq0.to(DEV), x0.to(DEV), O0.to(DEV), m.to(DEV), t.to(DEV), _to(noise), generate=gen).items()}
    out, both = run(generate), run(3)
    gs, gx = FLAGS[generate]
    if gs:
        assert torch.equal(out["seq_idx_t"], both["seq_idx_t"]) and torch.equal(out["seq_posterior"], both["seq_posterior"])
    else:
        assert torch.equal(out["seq_idx_t"], seq0)
        assert torch.equal(out["seq_posterior"], torch.nn.functional.one_hot(seq0, 21).float())     # exactly one-hot
    if gx:
        assert torch.equal(out["translations_t"], both["translations_t"])
        assert torch.equal(out["orientations_t"], both["orientations_t"])
    else:
        assert torch.equal(out["translations_t"], x0) and torch.equal(out["orientations_t"], O0)
    ref = mo.add_noise(SCHED, table.histograms.cpu(), seq0, x0, O0, m, t, noise, **_flags(generate))
    assert torch.equal(out["seq_idx_t"], ref["seq_idx_t"])
    for k in ("seq_posterior", "translations_t", "orientations_t"):
        assert float((out[k] - ref[k]).abs().max()) < 1e-4, k


@pytest.mark.parametrize("B,L", SIZES)
@pytest.mark.parametrize("generate", MODES)
def test_reverse_step_per_mode(tables, generate, B, L):
    dsched, _, rev = tables
    if B == 0:
        _check_empty_batch(dsched, generate, L)
        return
    g = torch.Generator().manual_seed(200 + B)
    batch = {k: v[:B] for k, v in synth.make_patches(max(B, 1), L, seed=32, cdr=(5, 30), with_distmat=False).items()}
    s, x, O, m = batch["seq_idx"], batch["xyz"][:, :, 1].contiguous(), batch["orientations"], batch["generation_mask"]
    eps = torch.randn(B, L, 3, generator=g)
    v = 0.3 * torch.randn(B, L, 3, generator=g)
    post = torch.softmax(2 * torch.randn(B, L, 21, generator=g), -1)
    t = torch.randint(1, 101, (B,), generator=g)
    if B:
        t[0] = 1                  # the noise-free last step
    noise = osamp.draw_step_noise(B, L, generator=g)
    run = lambda gen: {k: val.cpu() for k, val in diffusion.fused_reverse_step(
        dsched, rev, s.to(DEV), x.to(DEV), O.to(DEV), eps.to(DEV), v.to(DEV), post.to(DEV), m.to(DEV), t.to(DEV),
        _to(noise), return_O0=True, generate=gen).items()}
    out, both = run(generate), run(3)
    gs, gx = FLAGS[generate]
    assert torch.equal(out["orientations_t0"], both["orientations_t0"])
    assert torch.equal(out["seq_idx"], both["seq_idx"] if gs else s)
    assert torch.equal(out["translations"], both["translations"] if gx else x)
    assert torch.equal(out["orientations"], both["orientations"] if gx else O)
    O0 = O @ oso3.exp_vec(v)
    ref = mo.reverse_step(SCHED, rev.histograms.cpu(), s, x, O, eps, O0, post, m, t, noise, **_flags(generate))
    assert torch.equal(out["seq_idx"], ref["seq_idx"])
    assert float((out["translations"] - ref["translations"]).abs().max()) < 1e-4
    assert float((out["orientations"] - ref["orientations"]).abs().max()) < 2e-4


@pytest.mark.parametrize("B,L", [(1, 128), (3, 37)])
@pytest.mark.parametrize("generate", MODES)
def test_fused_losses_per_mode(generate, B, L):
    gen = torch.Generator().manual_seed(17 + B)
    post = torch.softmax(torch.randn(B, L, 21, generator=gen), -1)
    tgt = torch.softmax(4 * torch.randn(B, L, 21, generator=gen), -1)
    tgt[:, ::3] = torch.nn.functional.one_hot(torch.randint(0, 21, (B, (L + 2) // 3), generator=gen), 21).float()
    eps, eps_t = torch.randn(B, L, 3, generator=gen), torch.randn(B, L, 3, generator=gen)
    o_pred = synth.uniform_rotations(B, L) + 0.05 * torch.randn(B, L, 3, 3, generator=gen)
    o_true = synth.uniform_rotations(B, L)
    mask = torch.zeros(B, L, dtype=torch.bool)
    mask[:, 10:30] = True
    mask[-1, 12:15] = False
    w = torch.tensor([0.7, 1.3, 2.1])

    def run(g_):
        p, e, o = (t_.clone().to(DEV).requires_grad_(True) for t_ in (post, eps, o_pred))
        ls = _FusedLosses.apply(p, tgt.to(DEV), e, eps_t.to(DEV), o, o_true.to(DEV), mask.to(DEV), g_)
        sum(wi * li for wi, li in zip(w.to(DEV), ls)).backward()
        return [l_.detach().cpu() for l_ in ls], [p.grad.cpu(), e.grad.cpu(), o.grad.cpu()]

    (vals, grads), (vals3, grads3) = run(generate), run(3)
    gs, gx = FLAGS[generate]
    on = [gs, gx, gx]
    for i in range(3):
        if on[i]:
            assert torch.equal(vals[i], vals3[i]) and torch.equal(grads[i], grads3[i]), i
        else:
            assert float(vals[i]) == 0.0 and bool((grads[i] == 0).all()), i
    # against fp64 autograd of the moded oracle
    leaves = [t_.double().requires_grad_(True) for t_ in (post, eps, o_pred)]
    ref = mo.losses({"seq_posterior": leaves[0], "translations_eps": leaves[1], "orientations_t0": leaves[2]},
                      {"seq_posterior": tgt.double(), "translations_eps": eps_t.double()}, o_true.double(), mask,
                      torch.ones_like(mask), **_flags(generate))
    sum(wi * li for wi, li in zip(w.double(), ref)).backward()
    for i in range(3):
        r0 = float(ref[i].detach())
        assert abs(float(vals[i]) - r0) <= 1e-5 * max(abs(r0), 1e-30), i
        r = leaves[i].grad
        assert float((grads[i].double() - r).abs().max()) <= 1e-5 * float(r.abs().max()), i


def test_generate_outside_1_to_3_is_refused(tables):
    dsched, table, rev = tables
    batch = synth.make_patches(1, 16, seed=3, cdr=(2, 8), with_distmat=False)
    s, x, O, m = (batch[k].to(DEV) for k in ("seq_idx", "xyz", "orientations", "generation_mask"))
    x = x[:, :, 1].contiguous()
    t = torch.tensor([5], device=DEV)
    for bad in (0, 4):
        with pytest.raises(RuntimeError, match="dab_forward_noise.*generate must be 1"):
            diffusion.fused_add_noise(dsched, table, s, x, O, m, t, _to(odiff.draw_add_noise_tensors(1, 16)), generate=bad)
        with pytest.raises(RuntimeError, match="dab_reverse_step.*generate must be 1"):
            diffusion.fused_reverse_step(dsched, rev, s, x, O, torch.zeros_like(x), torch.full_like(x, 0.1),
                                         torch.full((1, 16, 21), 1 / 21, device=DEV), m, t,
                                         _to(osamp.draw_step_noise(1, 16)), generate=bad)
        p = torch.full((1, 16, 21), 1 / 21, device=DEV)
        with pytest.raises(RuntimeError, match="dab_losses_fwd.*generate must be 1"):
            _FusedLosses.apply(p, p, x, x, O, O, m, bad)


# ---------------------------------------------------------------------------------------------------- training
@pytest.mark.parametrize("generate", MODES)
def test_training_step_vs_oracle_grads_per_mode(generate):
    model = _set_mode(DiffAb(*SMALL, device=DEV), generate)
    batch = synth.make_patches(2, 24, seed=5, cdr=(8, 16))
    torch.manual_seed(3)
    t = torch.randint(1, 101, (2,))
    noise = odiff.draw_add_noise_tensors(2, 24)
    model.zero_grad()
    losses = model._shared_step(_to(batch), 0, t=t.to(DEV), noise=_to(noise))
    sum(losses).backward()
    _assert_off_heads_zero(model, generate)
    state = {k: v.detach().cpu().double().requires_grad_(True) for k, v in model.state_dict().items()}
    hist = model.orientation_diffuser.so3.histograms.cpu()
    noised = mo.add_noise(SCHED, hist, batch["seq_idx"], batch["xyz"][:, :, 1], batch["orientations"],
                             batch["generation_mask"], t, noise, **_flags(generate))
    res, pair = _context(model, _to(batch), generate)
    den = oipa.denoiser_forward(state, noised["seq_idx_t"], noised["translations_t"].double(),
                                noised["orientations_t"].double(), res.cpu().double(), pair.cpu().double(),
                                SCHED["beta"][t].double(), 2, 4)
    ol = mo.losses(den, {k: (v.double() if v.dtype.is_floating_point else v) for k, v in noised.items()},
                     batch["orientations"].double(), batch["generation_mask"], batch["residue_mask"], **_flags(generate))
    sum(ol).backward()
    assert torch.allclose(torch.stack(losses).detach().cpu().double(), torch.stack(ol).detach(), rtol=2e-4)
    for name, p in model.denoiser.named_parameters():
        ref = state["denoiser." + name].grad
        if ref is None:
            continue
        err = (p.grad.cpu().double() - ref).abs().max() / ref.abs().max().clamp_min(1e-12)
        assert err < 5e-3, (name, float(err))


@pytest.mark.parametrize("generate", MODES)
def test_bf16_training_step_matches_fp32_per_mode(generate):
    g = load_golden("shared_step.pt")
    batch = _to(synth.make_patches(2, 128, seed=g["seed_patches"]))
    torch.manual_seed(g["seed_step"])
    t = torch.randint(low=1, high=101, size=(2,)).to(DEV)
    noise = _to(odiff.draw_add_noise_tensors(2, 128))
    grads, losses = {}, {}
    for prec in ("fp32", "bf16"):
        model = _model(generate, seed=g["seed_state"]).train()
        model.train_precision = prec
        model.zero_grad()
        ls = model._shared_step(batch, 0, t=t, noise=noise)
        sum(ls).backward()
        _assert_off_heads_zero(model, generate)
        losses[prec] = torch.stack(ls).detach().cpu()
        grads[prec] = {n: p.grad.detach().cpu().double().flatten() for n, p in model.named_parameters()
                       if p.grad is not None}
    assert torch.allclose(losses["bf16"], losses["fp32"], rtol=2e-2), (losses["bf16"], losses["fp32"])
    for n, ref in grads["fp32"].items():
        got = grads["bf16"].get(n, torch.zeros_like(ref))
        assert torch.isfinite(got).all(), n
        if not bool(ref.any()):          # a head of the modality that is off: exactly zero on both paths
            assert not bool(got.any()), n
            continue
        cos = float(got @ ref / (got.norm() * ref.norm()).clamp_min(1e-300))
        assert cos >= 0.97, (n, cos)


@pytest.mark.parametrize("generate", MODES)
def test_graphed_training_step_with_flat_adam_per_mode(generate):
    from diffab_pytorch_b200 import distributed as dd
    batch = _to(synth.make_patches(2, 128, seed=51))
    torch.manual_seed(3)
    t = torch.randint(low=1, high=101, size=(2,)).to(DEV)
    noise = _to(odiff.draw_add_noise_tensors(2, 128))
    results = {}
    for how in ("eager", "graph"):
        model = _model(generate).train()
        model.train_precision = "bf16"
        bucket = dd.GradientBucket(model.parameters())
        opt = dd.FlatAdam(bucket, lr=0.0)                # lr = 0: the weights stay put
        terms = lambda: dd.diffab_loss_terms(model, batch, t=t, noise=noise)
        loss = dd.ddp_step(terms, bucket, opt) if how == "eager" else dd.GraphedTrainStep(terms, bucket, opt, warmup=2)()
        results[how] = (float(loss), bucket.flat.detach().clone())
    (le, ge), (lg, gg) = results["eager"], results["graph"]
    assert abs(le - lg) <= 1e-4 * abs(le)
    assert torch.isfinite(gg).all()
    assert float((ge - gg).norm() / ge.norm()) < 1e-3


# ---------------------------------------------------------------------------------------------------- sampling
def _oracle_free_run(model, res, pair, s, x, O, m, noises, t_start, t_stop, generate):
    """The oracle sampler step by step, with the smallest top-2 margin of p / Exp(1) seen per patch."""
    state = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    hist_rev = model.so3_reverse.histograms.cpu()
    B = s.shape[0]
    near_tie = torch.zeros(B, dtype=torch.bool)
    gs = FLAGS[generate][0]
    n_layers, n_head = len(model.denoiser.ipa.layers), model.denoiser.ipa.layers[0].n_head
    for step in range(t_start, t_stop - 1, -1):
        tt = torch.full((B,), step, dtype=torch.long)
        den = oipa.denoiser_forward(state, s, x, O, res.cpu(), pair.cpu(), SCHED["beta"][tt], n_layers, n_head)
        if gs:
            key = den["seq_posterior"].reshape(-1, 21) / noises[step]["seq_exp"]
            top2 = key.topk(2, dim=-1).values
            near_tie |= (((top2[:, 0] - top2[:, 1]) / top2[:, 0]).view(B, -1) < 1e-4).logical_and(m).any(dim=1)
        nxt = mo.reverse_step(SCHED, hist_rev, s, x, O, den["translations_eps"], den["orientations_t0"],
                                 den["seq_posterior"], m, tt, noises[step], **_flags(generate))
        s, x, O = nxt["seq_idx"], nxt["translations"], nxt["orientations"]
    return (s, x, O), near_tie


def _check_free_run(got, ref, near_tie, m, start, generate):
    """The bars of test_gpu_model.py::test_reverse_steps_vs_oracle_sampler, plus the off modality unchanged."""
    rs, rx, rO = ref
    s0, x0, O0 = start
    gs, gx = FLAGS[generate]
    got = {k: v.cpu() for k, v in got.items()}
    assert torch.equal(got["seq_idx"][~m], s0[~m])
    if not gs:
        assert torch.equal(got["seq_idx"], s0)
    if not gx:
        assert torch.equal(got["translations"], x0) and torch.equal(got["orientations"], O0)
    same = (got["seq_idx"] == rs).all(dim=1)
    assert bool((same | near_tie).all()), "sequence differs in a patch without any near-tie in the oracle"
    assert bool(same.any())
    for p_ in range(rs.shape[0]):
        if bool(same[p_]):
            assert float((got["translations"][p_] - rx[p_]).norm(dim=-1)[m[p_]].max()) < 1e-2
            assert float((got["orientations"][p_] - rO[p_]).abs().amax(dim=(-1, -2))[m[p_]].max()) < 1e-2


@pytest.mark.parametrize("generate", MODES)
def test_free_running_fp32_steps_vs_oracle_sampler_per_mode(generate):
    model = _model(generate)
    batch = synth.make_patches(2, 128, seed=9)
    res, pair = _context(model, _to(batch), generate)
    gen = torch.Generator().manual_seed(4)
    m = batch["generation_mask"]
    s, x, O = mo.draw_initial_state(batch["seq_idx"], batch["xyz"][:, :, 1], batch["orientations"], m,
                                       generator=gen, **_flags(generate))
    noises = {t: osamp.draw_step_noise(2, 128, generator=gen) for t in range(100, 95, -1)}
    ref, near_tie = _oracle_free_run(model, res, pair, s, x, O, m, noises, 100, 96, generate)
    got = model.sample_from_context(s.to(DEV), x.to(DEV), O.to(DEV), res, pair, m.to(DEV),
                                    noises={t: _to(n) for t, n in noises.items()}, t_start=100, t_stop=96)
    _check_free_run(got, ref, near_tie, m, (s, x, O), generate)


@pytest.mark.parametrize("generate", MODES)
def test_bf16_graph_steps_teacher_forced_per_mode(generate):
    """The t = 10..6 window of tests/test_gpu_sampling_parity.py (bf16 kernels + CUDA graph, fp64 oracle on the
    bf16-rounded pair tensor, teacher-forced, injected draws) with its bars, in each mode."""
    model = _model(generate)
    batch = synth.make_patches(2, 128, seed=9)
    b = _to(batch)
    B, L = 2, 128
    m = batch["generation_mask"]
    gs, gx = FLAGS[generate]
    res, pair = _context(model, b, generate)
    pair16 = cast_pair_to_bf16(pair)
    state64 = {k: v.detach().cpu().double() for k, v in model.state_dict().items()}
    res64, pair64 = res.cpu().double(), pair16.float().cpu().double()
    hist_rev = model.so3_reverse.histograms.cpu()
    torch.manual_seed(7)
    noised = mo.add_noise(SCHED, model.orientation_diffuser.so3.histograms.cpu(), batch["seq_idx"],
                             batch["xyz"][:, :, 1], batch["orientations"], m, torch.full((B,), 10),
                             odiff.draw_add_noise_tensors(B, L), **_flags(generate))
    s, x, O = noised["seq_idx_t"], noised["translations_t"], noised["orientations_t"]
    glue = model.denoiser.sampling_cache(res)
    planes = model._pair_bias_planes(pair16)
    gen = torch.Generator().manual_seed(50)
    for step in range(10, 5, -1):
        noise = osamp.draw_step_noise(B, L, generator=gen)
        tt = torch.full((B,), step, dtype=torch.long)
        den = oipa.denoiser_forward(state64, s, x.double(), O.double(), res64, pair64, SCHED["beta"][tt].double(), 6, 8)
        ref = mo.reverse_step(SCHED, hist_rev, s, x.double(), O.double(), den["translations_eps"],
                                 den["orientations_t0"], den["seq_posterior"], m, tt,
                                 {k: v.double() if v.dtype.is_floating_point else v for k, v in noise.items()},
                                 **_flags(generate))
        key = den["seq_posterior"].reshape(-1, 21) / noise["seq_exp"].double()
        top2 = key.topk(2, dim=-1).values
        margin = ((top2[:, 0] - top2[:, 1]) / top2[:, 0]).view(B, -1)
        args = (s.to(DEV), x.float().to(DEV), O.float().to(DEV), res, pair16, b["generation_mask"])
        kw = dict(noises={step: _to(noise)}, t_start=step, t_stop=step)
        eager = model.sample_from_context(*args, use_cuda_graph=False, **kw)
        graph = model.sample_from_context(*args, use_cuda_graph=True, **kw)
        for k in eager:
            assert torch.equal(eager[k], graph[k]), (step, k)
        with torch.no_grad():
            eps_g, v_g, post = model.denoiser.heads_fast(args[0], args[1], args[2], glue, pair16,
                                                         model.dsched.tensors["beta"][tt.to(DEV)], planes)
        p_ref = den["seq_posterior"]
        d_rel = float(((post.cpu().double() - p_ref).abs() / p_ref)[p_ref > 1e-3].max())
        assert d_rel < 2e-2, (step, d_rel)
        got = {k: v.cpu() for k, v in eager.items()}
        diff = got["seq_idx"] != ref["seq_idx"]
        assert not diff[~m].any()
        if gs:
            assert not (diff & ~(margin <= 2 * d_rel / (1 - d_rel))).any(), step
        else:
            assert torch.equal(got["seq_idx"], s)
        if gx:
            step_len = (ref["translations"] - x.double()).norm(dim=-1)[m]
            dx = (got["translations"].double() - ref["translations"]).norm(dim=-1)[m]
            assert float(dx.max() / step_len.mean()) < 1e-2, step
            dO = (got["orientations"].double() - ref["orientations"]).abs().amax(dim=(-1, -2))[m]
            assert float(dO.max()) < 2e-2, step
            dv = float((v_g.cpu().double() - den["rotvec"]).abs().max() / den["rotvec"].abs().max())
            de = float((eps_g.cpu().double() - den["translations_eps"]).abs().max() / den["translations_eps"].abs().max())
            assert dv < 2e-2 and de < 2e-2, (step, dv, de)
        else:
            assert torch.equal(got["translations"], x.float()) and torch.equal(got["orientations"], O.float())
        assert torch.equal(got["translations"][~m], x.float()[~m])
        s, x, O = ref["seq_idx"], ref["translations"].float(), ref["orientations"].float()     # teacher forcing


def _bf16_setup(generate, seed=11):
    model = _model(generate)
    batch = synth.make_patches(2, 128, seed=seed)
    res, pair = _context(model, _to(batch), generate)
    gen = torch.Generator().manual_seed(3)
    s, x, O = mo.draw_initial_state(batch["seq_idx"], batch["xyz"][:, :, 1], batch["orientations"],
                                       batch["generation_mask"], generator=gen, **_flags(generate))
    noises = {t: _to(osamp.draw_step_noise(2, 128, generator=gen)) for t in range(100, 78, -1)}
    return model, batch, (s.to(DEV), x.to(DEV), O.to(DEV), res, cast_pair_to_bf16(pair),
                          batch["generation_mask"].to(DEV)), noises


@pytest.mark.parametrize("generate", MODES)
def test_graphed_loop_equals_eager_loop_per_mode(generate):
    """22 steps: one replay of the 20-step block graph and two single-step replays against the eager loop."""
    model, batch, args, noises = _bf16_setup(generate)
    kw = dict(noises=noises, t_start=100, t_stop=79)
    eager = model.sample_from_context(*args, use_cuda_graph=False, **kw)
    graph = model.sample_from_context(*args, use_cuda_graph=True, **kw)
    for k in eager:
        assert torch.equal(eager[k], graph[k]), k
    gs, gx = FLAGS[generate]
    if not gs:
        assert torch.equal(graph["seq_idx"], args[0])
    if not gx:
        assert torch.equal(graph["translations"], args[1]) and torch.equal(graph["orientations"], args[2])


@pytest.mark.parametrize("first,second", [(3, 1), (1, 2), (2, 3)])
def test_switching_mode_between_calls_recaptures(first, second):
    model, batch, args, noises = _bf16_setup(first)
    kw = dict(noises=noises, t_start=100, t_stop=79, use_cuda_graph=True)
    model.sample_from_context(*args, **kw)
    _set_mode(model, second)
    got = model.sample_from_context(*args, **kw)
    fresh = _model(second).sample_from_context(*args, **kw)
    for k in got:
        assert torch.equal(got[k], fresh[k]), k


@pytest.mark.parametrize("B,L,generate", [(256, 128, 1), (256, 128, 2), (256, 128, 3), (64, 200, 1), (64, 200, 2),
                                          (64, 200, 3)])
def test_full_size_sampling_invariants_per_mode(B, L, generate):
    model = _model(generate)
    batch = synth.make_patches(B, L, seed=77, with_distmat=False, cdr=(56, 72))
    args = [batch[k] if k != "distmat" else None for k in CTX_KEYS]
    torch.manual_seed(5)
    out = {k: v.cpu() for k, v in model.sample(*args, precision="bf16").items()}
    m = batch["generation_mask"]
    gs, gx = FLAGS[generate]
    assert out["seq_idx"].shape == (B, L)
    assert int(out["seq_idx"].min()) >= 0 and int(out["seq_idx"].max()) <= 20
    assert torch.equal(out["seq_idx"][~m], batch["seq_idx"][~m])
    assert torch.equal(out["translations"][~m], batch["xyz"][:, :, 1][~m])
    assert torch.equal(out["orientations"][~m], batch["orientations"][~m])
    if not gs:
        assert torch.equal(out["seq_idx"], batch["seq_idx"])
    if not gx:
        assert torch.equal(out["translations"], batch["xyz"][:, :, 1])
        assert torch.equal(out["orientations"], batch["orientations"])
    else:
        O = out["orientations"][m].double()
        assert float((O.transpose(-1, -2) @ O - torch.eye(3, dtype=torch.float64)).abs().max()) < 1e-4
        assert float((torch.linalg.det(O) - 1).abs().max()) < 1e-4
        assert torch.isfinite(out["translations"]).all()


def test_launches_per_reverse_step_do_not_depend_on_the_mode():
    counts = {}
    for generate in MODES:
        model, batch, args, noises = _bf16_setup(generate)
        model.sample_from_context(*args, noises=noises, t_start=100, t_stop=100)       # warm caches
        torch.cuda.synchronize()
        n0 = _lib.lib().dab_launch_count()
        model.sample_from_context(*args, noises=noises, t_start=99, t_stop=99)
        torch.cuda.synchronize()
        counts[generate] = _lib.lib().dab_launch_count() - n0
    assert counts[1] == counts[2] == counts[3], counts


# ---------------------------------------------------------------------------------------------------- optimisation
@pytest.mark.parametrize("generate", MODES)
def test_native_start_vs_oracle(generate):
    """sample(init="native", t_start=k) under a seeded generator = the oracle's add_noise at k followed by its sampling
    loop, fed the same draws (fp32 path); and the same composition on the GPU, eager and graphed, is bit-identical."""
    model = _model(generate)
    batch = synth.make_patches(2, 128, seed=13)
    b = _to(batch)
    B, L, k = 2, 128, 5
    m = batch["generation_mask"]
    args = [b[n] for n in CTX_KEYS]
    out = model.sample(*args, precision="fp32", generator=torch.Generator(device=DEV).manual_seed(21), init="native",
                       t_start=k)
    g2 = torch.Generator(device=DEV).manual_seed(21)                   # the same draws, in sample()'s order
    noise = diffusion.draw_add_noise_tensors(B, L, device=DEV, generator=g2)
    noises = {t: DiffAb.draw_step_noise(B, L, DEV, generator=g2) for t in range(k, 0, -1)}
    # the composition on the GPU: native start, then the reverse loop, eager and graphed
    res, pair = _context(model, b, generate)
    start = model._add_noise(b["seq_idx"], b["xyz"][:, :, 1], b["orientations"], b["generation_mask"],
                             torch.full((B,), k, device=DEV), noise=noise, generate=model._generate())
    st = (start["seq_idx_t"], start["translations_t"], start["orientations_t"])
    eager = model.sample_from_context(*st, res, pair, b["generation_mask"], noises=noises, t_start=k)
    for key in out:
        assert torch.equal(out[key], eager[key]), key
    pair16 = cast_pair_to_bf16(pair)
    kw = dict(noises=noises, t_start=k)
    e16 = model.sample_from_context(*st, res, pair16, b["generation_mask"], use_cuda_graph=False, **kw)
    g16 = model.sample_from_context(*st, res, pair16, b["generation_mask"], use_cuda_graph=True, **kw)
    for key in e16:
        assert torch.equal(e16[key], g16[key]), key
    # the oracle: add_noise at k, then sample_loop
    cpu = lambda d: {n: v.cpu() for n, v in d.items()}
    ref0 = mo.add_noise(SCHED, model.orientation_diffuser.so3.histograms.cpu(), batch["seq_idx"],
                           batch["xyz"][:, :, 1], batch["orientations"], m, torch.full((B,), k), cpu(noise),
                           **_flags(generate))
    assert torch.equal(start["seq_idx_t"].cpu(), ref0["seq_idx_t"])
    assert float((start["translations_t"].cpu() - ref0["translations_t"]).abs().max()) < 1e-4
    assert float((start["orientations_t"].cpu() - ref0["orientations_t"]).abs().max()) < 1e-4
    s0, x0, O0 = ref0["seq_idx_t"], ref0["translations_t"], ref0["orientations_t"]
    ref, near_tie = _oracle_free_run(model, res, pair, s0, x0, O0, m, {t: cpu(n) for t, n in noises.items()}, k, 1,
                                     generate)
    native = (batch["seq_idx"], batch["xyz"][:, :, 1], batch["orientations"])
    _check_free_run(out, ref, near_tie, m, native, generate)


def test_native_start_refuses_t_start_outside_1_to_T():
    model = _model(3, cfg=SMALL)
    batch = synth.make_patches(1, 32, seed=1, cdr=(10, 20))
    for bad in (0, 101):
        with pytest.raises(ValueError):
            model.sample(batch["seq_idx"], batch["xyz"], batch["orientations"], generation_mask=batch["generation_mask"],
                         init="native", t_start=bad)
