"""GPU parity: IPA layer forward/backward vs the reference goldens (fp32 and fp64 arbiters).
Tolerance (north_star): fp32 path <= 1e-4 relative (max-normalised, as SURVEY §3.2 measures the
reference's own fp32-vs-fp64 gap); bf16 tensor-core path <= 2e-2 on logits -> checked on outputs."""
import pytest
import torch

from conftest import checksum, load_golden
from diffab_pytorch_b200 import synth
from diffab_pytorch_b200.diffab_pytorch import (Denoiser, InvariantPointAttentionLayer,
                                                InvariantPointAttentionModule, cast_pair_to_bf16)
from oracle import ipa as oipa

pytestmark = pytest.mark.gpu
DEV = "cuda"
REL = 1e-4


def _rel(a, b):
    return float((a.double().cpu() - b.double()).abs().max() / b.double().abs().max().clamp_min(1e-30))


def _case(name):
    g = load_golden(f"ipa_{name}.pt")
    c = g["cfg"]
    w = synth.synthetic_state(synth.ipa_layer_shapes(c["D"], c["C"], c["H"], c["ds"], c["Pq"], c["Pv"]), seed=c["seed"])
    x, e, R, t = synth.make_ipa_inputs(c["B"], c["L"], c["D"], c["C"], seed=c["seed"] + 100)
    assert checksum(e) == pytest.approx(g["chk"]["e"], rel=1e-12)
    gy = torch.randn(c["B"], c["L"], c["D"], generator=torch.Generator().manual_seed(c["seed"] + 200))
    layer = InvariantPointAttentionLayer(c["D"], c["C"], c["ds"], c["Pq"], c["Pv"], c["H"]).to(DEV)
    layer.load_state_dict(w)
    return g, c, layer, x, e, R, t, gy


@pytest.mark.parametrize("name", ["train", "tiny", "ragged"])
def test_forward_and_backward_vs_reference(name):
    g, c, layer, x, e, R, t, gy = _case(name)
    xg, eg = x.to(DEV).requires_grad_(True), e.to(DEV).requires_grad_(True)
    y = layer(xg, eg, R.to(DEV), t.to(DEV))
    (y * gy.to(DEV)).sum().backward()
    ref = g["f64"]
    assert _rel(y, ref["y"]) < REL
    assert _rel(xg.grad, ref["dx"]) < REL
    idx = tuple(slice(None, None, s) for s in ref["de"]["stride"])
    assert _rel(eg.grad[idx], ref["de"]["sub"]) < REL
    assert float(eg.grad.double().sum()) == pytest.approx(ref["de"]["sum"], rel=1e-3, abs=1e-3)
    assert float(eg.grad.double().abs().sum()) == pytest.approx(ref["de"]["abssum"], rel=1e-4)
    params = dict(layer.named_parameters())
    for n, gr in ref["dw"].items():
        mine = params[n].grad
        if isinstance(gr, dict):
            idx = tuple(slice(None, None, s) for s in gr["stride"])
            assert _rel(mine[idx], gr["sub"]) < 5 * REL, n
            assert float(mine.double().abs().sum()) == pytest.approx(gr["abssum"], rel=1e-4), n
        else:
            assert _rel(mine, gr) < 5 * REL, n


def test_forward_is_deterministic_and_no_grad_path_matches():
    g, c, layer, x, e, R, t, gy = _case("tiny")
    a = [v.to(DEV) for v in (x, e, R, t)]
    with torch.no_grad():
        y1, y2 = layer(*a), layer(*a)
    assert torch.equal(y1, y2)
    assert _rel(y1, g["f32"]["y"]) < REL


def test_reference_shape_tests():
    # tests/test_modules.py:143-248 of the reference (rand inputs, r not a rotation)
    ipa = InvariantPointAttentionLayer(32, 16, 16, 4, 4, 8).to(DEV)
    bsz, n_res = 32, 16
    x, e = torch.rand(bsz, n_res, 32, device=DEV), torch.rand(bsz, n_res, n_res, 16, device=DEV)
    r, t = torch.rand(bsz, n_res, 3, 3, device=DEV), torch.rand(bsz, n_res, 3, device=DEV)
    out = ipa(x, e, r, t)
    assert out.shape == (bsz, n_res, 32)
    w = {k: v.detach().cpu().double() for k, v in ipa.state_dict().items()}
    ref = oipa.ipa_layer(w, x.cpu().double(), e.cpu().double(), r.cpu().double(), t.cpu().double(), 8)
    assert _rel(out.detach(), ref) < REL
    mod = InvariantPointAttentionModule(4, 32, 16, 16, 4, 4, 8).to(DEV)
    assert mod(x, torch.randn(bsz, n_res, n_res, 16, device=DEV), r, t).shape == (bsz, n_res, 32)
    den = Denoiser(32, 16, 4, 12, 4, 4, 8, aa_vocab_size=21).to(DEV)
    o = den(torch.randint(0, 20, (bsz, n_res), device=DEV), t, r, x, torch.randn(bsz, n_res, n_res, 16, device=DEV),
            torch.rand(bsz, device=DEV), torch.randint(0, 2, (bsz, n_res), device=DEV),
            torch.randint(0, 2, (bsz, n_res), device=DEV))
    assert o["translations_eps"].shape == (bsz, n_res, 3)
    assert o["orientations_t0"].shape == (bsz, n_res, 3, 3)
    assert o["seq_posterior"].shape == (bsz, n_res, 21)


def test_batch_independence_and_empty_batch():
    g, c, layer, x, e, R, t, gy = _case("tiny")
    a = [v.to(DEV) for v in (x, e, R, t)]
    with torch.no_grad():
        full = layer(*a)
        one = layer(*[v[2:3].contiguous() for v in a])
        empty = layer(*[v[:0].contiguous() for v in a])
    assert torch.equal(full[2:3], one)          # patches never mix (basis of the multi-GPU sharding)
    assert empty.shape == (0, c["L"], c["D"])


def test_frames_requiring_grad_are_rejected():
    g, c, layer, x, e, R, t, gy = _case("tiny")
    tt = t.to(DEV).requires_grad_(True)
    y = layer(x.to(DEV).requires_grad_(True), e.to(DEV), R.to(DEV), tt)
    with pytest.raises(NotImplementedError):
        y.sum().backward()


def test_tensor_core_path_vs_fp32_kernel_and_reference():
    g, c, layer, x, e, R, t, gy = _case("train")
    a = [v.to(DEV) for v in (x, e, R, t)]
    with torch.no_grad():
        y32 = layer(*a)
        try:
            yb = layer(a[0], cast_pair_to_bf16(a[1]), a[2], a[3])
        except RuntimeError as exc:
            if "not built" in str(exc):
                pytest.skip("sm_100a fast path not built yet")
            raise
        # reference evaluated on the bf16-rounded pair tensor isolates the kernel's own error
        w = {k: v.detach().cpu().double() for k, v in layer.state_dict().items()}
        e_r = e.to(torch.bfloat16).double()
        ref_r = oipa.ipa_layer(w, x.double(), e_r, R.double(), t.double(), 8)
    assert _rel(yb, ref_r) < 2e-2
    assert _rel(yb, g["f64"]["y"]) < 3e-2
    assert _rel(y32, g["f64"]["y"]) < REL


def test_tensor_core_backward_vs_reference_autograd():
    """bf16 tcgen05 training path (dab_ipa_fwd_sm100_train / dab_ipa_bwd_sm100_main + _finish): every gradient against
    the fp64 autograd of the oracle evaluated on the bf16-rounded pair tensor.  Tolerance: 2e-2 max-normalised per tensor
    (north_star's bound for the bf16 path); measured ~1e-2 on the point-projection weights, ~5e-3 elsewhere."""
    g, c, layer, x, e, R, t, gy = _case("train")
    e16 = e.to(torch.bfloat16)
    w = {k: v.detach().cpu().double().requires_grad_(True) for k, v in layer.state_dict().items()}
    xd, ed = x.double().requires_grad_(True), e16.double().requires_grad_(True)
    yd = oipa.ipa_layer(w, xd, ed, R.double(), t.double(), 8)
    (yd * gy.double()).sum().backward()

    xg, eg = x.to(DEV).requires_grad_(True), e16.to(DEV).requires_grad_(True)
    y = layer(xg, eg, R.to(DEV), t.to(DEV))
    (y * gy.to(DEV)).sum().backward()
    assert eg.grad.dtype == torch.bfloat16 and eg.grad.shape == e.shape
    assert _rel(y.detach(), yd.detach()) < 2e-2
    assert _rel(xg.grad, xd.grad) < 2e-2
    assert _rel(eg.grad, ed.grad) < 2e-2
    for n, p in layer.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), n
        assert _rel(p.grad, w[n].grad) < 2e-2, n
    # gradient scale invariance of the fp16 staging: a 1e-6 smaller upstream gradient gives 1e-6 smaller grads
    xs, es = x.to(DEV).requires_grad_(True), e16.to(DEV).requires_grad_(True)
    for p in layer.parameters():
        p.grad = None
    (layer(xs, es, R.to(DEV), t.to(DEV)) * gy.to(DEV) * 1e-6).sum().backward()
    assert _rel(xs.grad * 1e6, xd.grad) < 2e-2
    assert _rel(es.grad.float() * 1e6, ed.grad) < 2e-2
    assert _rel(layer.gamma.grad * 1e6, w["gamma"].grad) < 2e-2


def test_tensor_core_backward_rejects_frame_grads():
    g, c, layer, x, e, R, t, gy = _case("train")
    tt = t.to(DEV).requires_grad_(True)
    y = layer(x.to(DEV).requires_grad_(True), e.to(torch.bfloat16).to(DEV), R.to(DEV), tt)
    with pytest.raises(NotImplementedError):
        y.sum().backward()


def test_pair_bias_planes_single_pass_for_all_layers():
    """dab_ipa_pair_bias_multi: the planes of six layers from one pass over the pair tensor (tensor cores, weights
    as bf16 hi + lo) against e . Wpb^T in fp64; and the single-layer entry point gives the same bits."""
    torch.manual_seed(0)
    B = 2
    mod = InvariantPointAttentionModule(6, 128, 64, 32, 8, 8, 8).to(DEV)
    e = torch.randn(B, 128, 128, 64, device=DEV).bfloat16()
    planes = mod.precompute_pair_bias(e)
    assert len(planes) == 6
    sc = 3 ** -0.5 * 1.4426950408889634
    for k, layer in enumerate(mod.layers):
        ref = torch.einsum("bijc,hc->bijh", e.double(), layer.to_pair_bias.weight.detach().double()) * sc
        assert planes[k].dtype == torch.float16 and planes[k].shape == (B, 128, 128, 8)
        assert float((planes[k].double() - ref).abs().max()) < 2e-3 * float(ref.abs().max())   # fp16 storage
        assert torch.equal(layer.pair_bias(e), planes[k])


def test_tensor_core_layer_full_size_properties():
    """Size-independent properties of the tensor-core IPA layer at the benchmark size (B = 256 patches, BASELINE config 3):
    patches never mix (a sub-batch gives the same rows, a permuted batch permuted rows - other launch shapes, so only
    within accumulation-order noise) and the layer is invariant under a global rigid motion of all frames."""
    torch.manual_seed(0)
    B = 256
    layer = InvariantPointAttentionLayer(128, 64, 32, 8, 8, 8).to(DEV)
    layer.load_state_dict(synth.synthetic_state(synth.ipa_layer_shapes(128, 64, 8, 32, 8, 8), seed=0))
    x, e, R, t = (v.to(DEV) for v in synth.make_ipa_inputs(B, 128, 128, 64, seed=9))
    e = e.bfloat16()
    with torch.no_grad():
        y = layer(x, e, R, t)
        assert torch.isfinite(y).all()
        assert torch.equal(y, layer(x, e, R, t))                                 # deterministic
        sub = slice(100, 108)
        ys = layer(x[sub], e[sub].contiguous(), R[sub], t[sub])
        assert _rel(ys, y[sub].cpu()) < 1e-5                                      # patches are independent
        perm = torch.randperm(B, device=DEV)
        yp = layer(x[perm], e[perm].contiguous(), R[perm], t[perm])
        assert torch.equal(yp, y[perm])                                           # same launch shape: same bits
        # global rigid motion: frames (R, t) -> (R G, t G + s) (row-vector convention of the reference)
        G = synth.uniform_rotations(1, 1, device=DEV)[0, 0]
        shift = torch.tensor([3.0, -7.0, 11.0], device=DEV)
        ym = layer(x, e, R @ G, t @ G + shift)
        assert _rel(ym, y.cpu()) < 2e-2                                           # bf16 operands: tolerance of the path


def test_layer_stack_bf16_handoff_changes_no_bit():
    """Inference through InvariantPointAttentionModule hands the residue stream from layer to layer as bf16
    (dab_ipa_fwd_sm100_stages with y_bf16: the to_out GEMM rounds, the next projections copy); the projections round
    their fp32 input the same way, so the result must equal the layer-by-layer fp32 hand-off bit for bit."""
    torch.manual_seed(2)
    B = 4
    mod = InvariantPointAttentionModule(4, 128, 64, 32, 8, 8, 8).to(DEV)
    for layer in mod.layers:
        layer.load_state_dict(synth.synthetic_state(synth.ipa_layer_shapes(128, 64, 8, 32, 8, 8), seed=3))
    x, e, R, t = (v.to(DEV) for v in synth.make_ipa_inputs(B, 128, 128, 64, seed=6))
    e = e.bfloat16()
    with torch.no_grad():
        y = mod(x, e, R, t)                          # bf16 hand-off (planes precomputed inside)
        planes = mod.precompute_pair_bias(e)
        ref = x
        for k, layer in enumerate(mod.layers):       # fp32 hand-off, one public layer call at a time
            ref = layer(ref, e, R, t, planes[k])
    assert y.dtype == torch.float32 and torch.isfinite(y).all()
    assert torch.equal(y, ref)


def test_pair_gradient_of_the_layer_stack_is_one_fused_sum():
    """InvariantPointAttentionModule hands the bf16 pair tensor to its layers through _PairFanOut: the layers' pair
    gradients are summed in one fp32-accumulated pass (dab_sum_bf16).  Against the fp32 sum of the per-layer gradients
    (captured with hooks) the result is within one bf16 rounding; autograd's pairwise bf16 adds are not."""
    from diffab_pytorch_b200 import diffab_pytorch as dp
    torch.manual_seed(1)
    B = 2
    mod = InvariantPointAttentionModule(3, 128, 64, 32, 8, 8, 8).to(DEV)
    x, e, R, t = (v.to(DEV) for v in synth.make_ipa_inputs(B, 128, 128, 64, seed=5))
    e = e.bfloat16().requires_grad_(True)
    gy = torch.randn(B, 128, 128, device=DEV)
    per_layer = []
    orig = dp._PairFanOut.backward

    def spy(ctx, *grads):
        per_layer.extend(g.detach().float().clone() for g in grads)
        return orig(ctx, *grads)

    dp._PairFanOut.backward = staticmethod(spy)
    try:
        mod(x, e, R, t).backward(gy)
    finally:
        dp._PairFanOut.backward = staticmethod(orig)
    assert len(per_layer) == 3
    ref = sum(per_layer)
    got = e.grad.float()
    assert torch.equal(got, ref.bfloat16().float())                 # exactly the rounded fp32 sum
    assert torch.isfinite(got).all()


@pytest.mark.parametrize("B", [1, 3, 65])
def test_tensor_core_training_pair_other_batch_sizes(B):
    """Batch sizes that exercise the small-batch launch variants (projection tiles split over 4 / 2 CTAs per patch,
    32-wide to_out tiles, partial-reduction blocks without work): bf16 forward + backward against the fp32 kernels on
    the same bf16-rounded pair tensor."""
    torch.manual_seed(B)
    layer = InvariantPointAttentionLayer(128, 64, 32, 8, 8, 8).to(DEV)
    layer.load_state_dict(synth.synthetic_state(synth.ipa_layer_shapes(128, 64, 8, 32, 8, 8), seed=1))
    x, e, R, t = (v.to(DEV) for v in synth.make_ipa_inputs(B, 128, 128, 64, seed=7 + B))
    e16 = e.to(torch.bfloat16)
    gy = torch.randn(B, 128, 128, device=DEV)
    grads = {}
    for name, pair in (("fp32", e16.float()), ("bf16", e16)):
        for p in layer.parameters():
            p.grad = None
        xg, eg = x.clone().requires_grad_(True), pair.clone().requires_grad_(True)
        y = layer(xg, eg, R, t)
        (y * gy).sum().backward()
        grads[name] = {"y": y.detach(), "dx": xg.grad, "de": eg.grad.float(),
                       **{n: p.grad.clone() for n, p in layer.named_parameters()}}
    for k, ref in grads["fp32"].items():
        assert torch.isfinite(grads["bf16"][k]).all(), k
        assert _rel(grads["bf16"][k], ref.cpu()) < 2e-2, k


def test_tensor_core_path_empty_batch_and_wrong_shape():
    layer = InvariantPointAttentionLayer(128, 64, 32, 8, 8, 8).to(DEV)
    x = torch.zeros(0, 128, 128, device=DEV)
    e = torch.zeros(0, 128, 128, 64, device=DEV, dtype=torch.bfloat16)
    R = torch.zeros(0, 128, 3, 3, device=DEV)
    t = torch.zeros(0, 128, 3, device=DEV)
    with torch.no_grad():
        assert layer(x, e, R, t).shape == (0, 128, 128)
    small = InvariantPointAttentionLayer(32, 16, 16, 4, 4, 8).to(DEV)
    with pytest.raises(RuntimeError, match="train.py"):
        with torch.no_grad():
            small(torch.rand(2, 16, 32, device=DEV), torch.rand(2, 16, 16, 16, device=DEV).bfloat16(),
                  torch.rand(2, 16, 3, 3, device=DEV), torch.rand(2, 16, 3, device=DEV))


def test_layer_without_pair_bias_vs_reference():
    """use_pair_bias=False (diffab_pytorch.py:374-387,438-462; never constructed by the reference model, but part of the
    layer's interface): same state-dict keys as the reference, forward and every gradient vs its fp64 result."""
    g = load_golden("ipa_nopb.pt")
    c = g["cfg"]
    layer = InvariantPointAttentionLayer(c["D"], c["C"], c["ds"], c["Pq"], c["Pv"], c["H"], use_pair_bias=False).to(DEV)
    assert sorted(layer.state_dict()) == sorted(g["state"])
    layer.load_state_dict({k: v.float() for k, v in g["state"].items()})
    x, e, R, t = synth.make_ipa_inputs(c["B"], c["L"], c["D"], c["C"], seed=c["seed"] + 100)
    gy = torch.randn(c["B"], c["L"], c["D"], generator=torch.Generator().manual_seed(c["seed"] + 200))
    xg = x.to(DEV).requires_grad_(True)
    y = layer(xg, e.to(DEV), R.to(DEV), t.to(DEV))
    (y * gy.to(DEV)).sum().backward()
    assert _rel(y, g["y"]) < REL
    assert _rel(xg.grad, g["dx"]) < REL
    params = dict(layer.named_parameters())
    for n, gr in g["dw"].items():
        assert _rel(params[n].grad, gr) < 5 * REL, n
    with torch.no_grad():
        assert torch.equal(layer(xg, e.to(DEV), R.to(DEV), t.to(DEV)), y)


@pytest.mark.parametrize("L", [100, 37])
def test_tensor_core_path_for_shorter_patches(L):
    """Patches of L < 128 residues (train.py head configuration) on the tensor-core kernels: padded to 128 residues, the
    padded keys masked through the bias plane (-inf), so the layer computes exactly what the reference computes on the L
    real residues.  Forward and every gradient vs the fp64 autograd of the oracle on the bf16-rounded pair tensor
    (2e-2 max-normalised, the bf16 bar); a three-layer stack (inference hand-off and training) against the oracle chain."""
    shp = synth.ipa_layer_shapes(128, 64, 8, 32, 8, 8)
    layer = InvariantPointAttentionLayer(128, 64, 32, 8, 8, 8).to(DEV)
    layer.load_state_dict(synth.synthetic_state(shp, seed=3))
    x, e, R, t = synth.make_ipa_inputs(2, L, 128, 64, seed=300 + L)
    gy = torch.randn(2, L, 128, generator=torch.Generator().manual_seed(L))
    e16 = e.to(torch.bfloat16)
    w = {k: v.detach().cpu().double().requires_grad_(True) for k, v in layer.state_dict().items()}
    xd, ed = x.double().requires_grad_(True), e16.double().requires_grad_(True)
    yd = oipa.ipa_layer(w, xd, ed, R.double(), t.double(), 8)
    (yd * gy.double()).sum().backward()
    xg, eg = x.to(DEV).requires_grad_(True), e16.to(DEV).requires_grad_(True)
    y = layer(xg, eg, R.to(DEV), t.to(DEV))
    assert y.shape == (2, L, 128)
    (y * gy.to(DEV)).sum().backward()
    assert _rel(y.detach(), yd.detach()) < 2e-2
    assert _rel(xg.grad, xd.grad) < 2e-2
    assert eg.grad.shape == e.shape and _rel(eg.grad, ed.grad) < 2e-2
    for n, p in layer.named_parameters():
        assert _rel(p.grad, w[n].grad) < 2e-2, n
    with torch.no_grad():
        assert _rel(layer(x.to(DEV), e16.to(DEV), R.to(DEV), t.to(DEV)), yd.detach()) < 2e-2
    # layer stack: one padding for the whole chain
    mod = InvariantPointAttentionModule(3, 128, 64, 32, 8, 8, 8).to(DEV)
    state = {}
    for k_, lay in enumerate(mod.layers):
        sd = synth.synthetic_state(shp, seed=10 + k_)
        lay.load_state_dict(sd)
        state.update({f"l.{k_}.{n}": v.double() for n, v in sd.items()})
    ref = oipa.ipa_module(state, x.double(), e16.double(), R.double(), t.double(), 3, 8, prefix="l.")
    with torch.no_grad():
        got = mod(x.to(DEV), e16.to(DEV), R.to(DEV), t.to(DEV))
    assert got.shape == (2, L, 128) and _rel(got, ref) < 3e-2
    got_t = mod(x.to(DEV).requires_grad_(True), e16.to(DEV), R.to(DEV), t.to(DEV))     # training path of the stack
    assert _rel(got_t.detach(), ref) < 3e-2


def test_fused_stack_is_bit_identical_to_the_layerwise_stack():
    """dab_ipa_mid_sm100 (a layer's to_out fused into the next layer's projection kernel, used for batches >= 128): the
    six-layer stack gives the same bits as the layer-by-layer bf16 hand-off, for fp32 and for bf16 input."""
    torch.manual_seed(0)
    B = 128
    mod = InvariantPointAttentionModule(6, 128, 64, 32, 8, 8, 8).to(DEV)
    shp = synth.ipa_layer_shapes(128, 64, 8, 32, 8, 8)
    for k_, lay in enumerate(mod.layers):
        lay.load_state_dict(synth.synthetic_state(shp, seed=20 + k_))
    g = torch.Generator(device=DEV).manual_seed(1)
    x = torch.randn(B, 128, 128, device=DEV, generator=g)
    e = torch.randn(B, 128, 128, 64, device=DEV, generator=g).bfloat16()
    R = synth.uniform_rotations(B, 128, device=DEV)
    t = 10 * torch.randn(B, 128, 3, device=DEV, generator=g)
    with torch.no_grad():
        planes = mod.precompute_pair_bias(e)
        for xin in (x, x.bfloat16()):
            fused = mod._forward_fused_stack(xin, e, R, t, planes)
            h = xin
            for k_, lay in enumerate(mod.layers):
                h = lay.forward_fast_io(h, e, R, t, planes[k_], torch.float32 if k_ == 5 else torch.bfloat16)
            assert torch.isfinite(fused).all()
            assert torch.equal(fused, h)
        assert torch.equal(mod(x, e, R, t, planes), fused)          # the module picks the fused stack at this batch size


@pytest.mark.parametrize("L", [256, 200, 129])
def test_tensor_core_inference_for_patches_up_to_256_residues(L):
    """Inference on patches of 128 < L <= 256 residues - what the reference's preprocessing produces (the union of two
    128-nearest-residue sets, preprocess_pdb.py:48-58) - on the tensor-core kernels: two blocks of 128 (block-wise
    projections on the patch centroid, the attention core per (query block, key block), the key blocks merged by their
    softmax statistics), ragged lengths padded to 256 with the padded keys masked.  One layer and a three-layer stack
    against the fp64 oracle on the bf16-rounded pair tensor (2e-2 / 3e-2 max-normalised, the bf16 bars of L = 128)."""
    shp = synth.ipa_layer_shapes(128, 64, 8, 32, 8, 8)
    layer = InvariantPointAttentionLayer(128, 64, 32, 8, 8, 8).to(DEV)
    layer.load_state_dict(synth.synthetic_state(shp, seed=5))
    x, e, R, t = synth.make_ipa_inputs(2, L, 128, 64, seed=500 + L)
    e16 = e.to(torch.bfloat16)
    w = {k: v.detach().cpu().double() for k, v in layer.state_dict().items()}
    ref = oipa.ipa_layer(w, x.double(), e16.double(), R.double(), t.double(), 8)
    with torch.no_grad():
        got = layer(x.to(DEV), e16.to(DEV), R.to(DEV), t.to(DEV))
        assert got.shape == (2, L, 128) and torch.isfinite(got).all()
        assert _rel(got, ref) < 2e-2
        if L == 256:   # with the bias plane given (as the sampling loop does)
            assert torch.equal(layer(x.to(DEV), e16.to(DEV), R.to(DEV), t.to(DEV), layer.pair_bias(e16.to(DEV))), got)
    mod = InvariantPointAttentionModule(3, 128, 64, 32, 8, 8, 8).to(DEV)
    state = {}
    for k_, lay in enumerate(mod.layers):
        sd = synth.synthetic_state(shp, seed=30 + k_)
        lay.load_state_dict(sd)
        state.update({f"l.{k_}.{n}": v.double() for n, v in sd.items()})
    refm = oipa.ipa_module(state, x.double(), e16.double(), R.double(), t.double(), 3, 8, prefix="l.")
    with torch.no_grad():
        gotm = mod(x.to(DEV), e16.to(DEV), R.to(DEV), t.to(DEV))
    assert gotm.shape == (2, L, 128) and _rel(gotm, refm) < 3e-2


def test_fused_stack_at_256_residues_matches_the_layerwise_stack():
    """Batches of >= 64 patches of 256 residues take the fused stack (to_out of a layer inside the next layer's projection
    kernel, 128 blocks of 128 residues): same bits as the layer-by-layer bf16 hand-off."""
    B, L = 64, 256
    mod = InvariantPointAttentionModule(3, 128, 64, 32, 8, 8, 8).to(DEV)
    shp = synth.ipa_layer_shapes(128, 64, 8, 32, 8, 8)
    for k_, lay in enumerate(mod.layers):
        lay.load_state_dict(synth.synthetic_state(shp, seed=40 + k_))
    g = torch.Generator(device=DEV).manual_seed(2)
    x = torch.randn(B, L, 128, device=DEV, generator=g)
    e = torch.randn(B, L, L, 64, device=DEV, generator=g).bfloat16()
    R = synth.uniform_rotations(B, L, device=DEV)
    t = 10 * torch.randn(B, L, 3, device=DEV, generator=g)
    with torch.no_grad():
        planes = mod.precompute_pair_bias(e)
        fused = mod._forward_fused_stack(x, e, R, t, planes)
        h = x
        for k_, lay in enumerate(mod.layers):
            h = lay.forward_fast_io(h, e, R, t, planes[k_], torch.float32 if k_ == 2 else torch.bfloat16)
        assert torch.isfinite(fused).all() and torch.equal(fused, h)
        assert torch.equal(mod(x, e, R, t, planes), fused)
