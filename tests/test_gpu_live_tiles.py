"""Sampling on live tiles: the last IPA layer's attention core and the heads (with the last to_out) run only on the 16-row
query tiles that hold a generated residue (``live_query_tiles``).  Every value that reaches the output must be the same bit
as with all rows computed: the head outputs on every row of a live tile, and the sampled state of eager and graphed loops
against a plain loop of ``reverse_step`` without the list - also when the cached graphs are replayed with another mask,
with fewer live tiles than SMs, and with none at all."""
import pytest
import torch

from conftest import load_golden
from diffab_pytorch_b200 import synth
from diffab_pytorch_b200.diffab_pytorch import DiffAb, _tf32_matmuls, live_query_tiles

DEV = "cuda"
TRAIN = (128, 64, 6, 32, 8, 8, 8)
# the fused stack (and so the live tiles) needs >= 128 blocks of 128 residues; patches of 256 sample without the fused heads
# (and so without the list), their stack is checked with it directly
SHAPES = [(128, 128), (64, 256)]


def _masks(B, L, seed, kind):
    """Per-patch generation masks: CDR-like stretches at random offsets and lengths (some on 16-row boundaries), single
    residues, all-true and all-false patches ("mixed"); a few single residues, far fewer live tiles than SMs ("sparse");
    nothing generated ("none")."""
    g = torch.Generator().manual_seed(seed)
    m = torch.zeros(B, L, dtype=torch.bool)
    if kind == "none":
        return m
    if kind == "sparse":
        for b in torch.randperm(B, generator=g)[:37].tolist():
            m[b, int(torch.randint(L, (1,), generator=g))] = True
        return m
    for b in range(B):
        k = b % 5
        if k == 0:                                     # stretch at a random offset
            n = int(torch.randint(1, 40, (1,), generator=g))
            a = int(torch.randint(0, L - n + 1, (1,), generator=g))
            m[b, a:a + n] = True
        elif k == 1:                                   # stretch starting and ending on tile boundaries
            a = 16 * int(torch.randint(0, L // 16, (1,), generator=g))
            n = 16 * int(torch.randint(1, (L - a) // 16 + 1, (1,), generator=g))
            m[b, a:a + n] = True
        elif k == 2:                                   # one residue
            m[b, int(torch.randint(L, (1,), generator=g))] = True
        elif k == 3 and b % 2 == 0:
            m[b] = True
    return m


def _row_flags(mask):
    return mask.reshape(-1, 16).any(-1).repeat_interleave(16).view(mask.shape)


def test_live_query_tiles_lists_the_tiles_of_generated_residues():
    for kind in ("mixed", "sparse", "none"):
        m = _masks(16, 128, 5, kind)
        tiles, count = live_query_tiles(m)
        flags = m.view(-1, 16).any(-1)
        n = int(count)
        assert tiles.dtype == count.dtype == torch.int32 and count.shape == (1,) and tiles.numel() == flags.numel()
        assert n == int(flags.sum())
        assert torch.equal(tiles[:n].long(), flags.nonzero().flatten())          # ascending, live ones first
        assert sorted(tiles.tolist()) == list(range(flags.numel()))


def _setup(B, L, seed=0):
    model = DiffAb(*TRAIN, device=DEV).eval()
    model.load_state_dict(synth.synthetic_state(load_golden("state_shapes.pt"), seed=0))
    g = torch.Generator(device=DEV).manual_seed(seed + 3)
    res = torch.randn(B, L, 128, device=DEV, generator=g)
    pair = torch.randn(B, L, L, 64, device=DEV, generator=g).bfloat16()
    batch = {k: v.to(DEV) for k, v in synth.make_patches(B, L, seed=seed + 4, with_distmat=False).items()}
    return model, res, pair, batch["seq_idx"], batch["xyz"][:, :, 1].contiguous(), batch["orientations"].contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("B,L", SHAPES)
def test_heads_on_live_tiles_equal_all_rows(B, L):
    """The layer stack with its last attention core on the live tiles (both core modes: 128 and 256 residues per patch),
    and the heads with the last to_out on them (patches of 128: the sampling path with the fused heads)."""
    model, res, pair, s, x, O = _setup(B, L)
    ipa = model.denoiser.ipa
    with torch.no_grad():
        planes = model._pair_bias_planes(pair)
        cache = model.denoiser.sampling_cache(res)
        beta = model.dsched.tensors["beta"][torch.randint(1, 100, (B,), device=DEV)]
        h = res.bfloat16()
        assert ipa.fused_stack_applicable(B, L, pair, planes)
        assert model.denoiser.fused_heads_applicable(cache, B, L, pair, planes) == (L == 128)
        full_y = ipa._forward_fused_stack(h, pair, O, x, planes).clone()
        full = model.denoiser.heads_fast(s, x, O, cache, pair, beta, planes)
        for kind in ("mixed", "sparse", "none"):
            m = _masks(B, L, 1, kind).to(DEV)
            live = live_query_tiles(m)
            rows = _row_flags(m)
            y = ipa._forward_fused_stack(h, pair, O, x, planes, live=live)
            got = model.denoiser.heads_fast(s, x, O, cache, pair, beta, planes, live=live)
            torch.cuda.synchronize()
            assert torch.equal(y[rows], full_y[rows]), kind
            for a, b in zip(got, full):
                assert a.shape == b.shape and torch.equal(a[rows], b[rows]), kind


def _plain_loop(model, s, x, O, res, pair, mask, noises, t_start, t_stop):
    """Eager reverse steps with every row computed (no live-tile list), TF32 glue GEMMs as in ``sample_from_context``."""
    B = s.shape[0]
    s, x, O = s.clone(), x.clone(), O.clone()
    with torch.no_grad(), _tf32_matmuls(True):
        planes = model._pair_bias_planes(pair)
        glue = model.denoiser.sampling_cache(res)
        for step in range(t_start, t_stop - 1, -1):
            t = torch.full((B,), step, device=DEV, dtype=torch.int64)
            out = model.reverse_step(s, x, O, res, pair, mask, t, noises[step], inplace=True, pair_bias=planes,
                                     glue_cache=glue, generate=model._generate())
            s, x, O = out["seq_idx"], out["translations"], out["orientations"]
    return {"seq_idx": s, "translations": x, "orientations": O}


@pytest.mark.gpu
@pytest.mark.parametrize("B,L", SHAPES)
def test_sampling_on_live_tiles_equals_all_rows(B, L):
    """25 steps (one replay of the 20-step block graph + five single steps) under injected draws, eager and graphed, then
    the cached graphs again with another mask and with no generated residue."""
    model, res, pair, s, x, O = _setup(B, L, seed=1)
    g = torch.Generator(device=DEV).manual_seed(11)
    noises = {t: model.draw_step_noise(B, L, DEV, generator=g) for t in range(100, 75, -1)}
    kw = dict(noises=noises, t_start=100, t_stop=76)
    m = _masks(B, L, 2, "mixed").to(DEV)
    ref = _plain_loop(model, s, x, O, res, pair, m, noises, 100, 76)
    eager = model.sample_from_context(s, x, O, res, pair, m, use_cuda_graph=False, **kw)
    graph = model.sample_from_context(s, x, O, res, pair, m, use_cuda_graph=True, **kw)
    for k in ref:
        assert torch.equal(eager[k], ref[k]), k
        assert torch.equal(graph[k], ref[k]), k
    assert not torch.equal(graph["translations"], x)
    # the graphs are cached per shape: the tile list must follow the mask of each call
    m2 = _masks(B, L, 3, "sparse").to(DEV)
    ref2 = _plain_loop(model, s, x, O, res, pair, m2, noises, 100, 76)
    again = model.sample_from_context(s, x, O, res, pair, m2, use_cuda_graph=True, **kw)
    for k in ref2:
        assert torch.equal(again[k], ref2[k]), k
    none = model.sample_from_context(s, x, O, res, pair, torch.zeros_like(m), use_cuda_graph=True, **kw)
    torch.cuda.synchronize()
    for k, v in (("seq_idx", s), ("translations", x), ("orientations", O)):
        assert torch.equal(none[k], v), k
