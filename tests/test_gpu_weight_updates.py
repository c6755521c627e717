"""Every way of updating the weights reaches the weight-derived caches.

Three caches hold data derived from the weights: the packed bf16 weights of each tensor-core IPA layer
(``InvariantPointAttentionLayer._packed_weights``), the packed weights of the fused pair embedding
(``PairEmbedding.forward_fused_bf16``) and the captured sampling graphs (``DiffAb._sample_graphed``, with the packed heads
weights and the glue constants baked in).  After each update, every kernel that reads one of them must compute what a
freshly built model holding the same weights computes.

Probes, one per cache reader:
  P1  fused pair embedding (bf16)                         pair-embedding pack                 bitwise
  P2  IPA stack, inference, bf16 pair                     IPA pack (inference)                bitwise
  P3  bf16 training forward + backward                    IPA pack (training fwd / bwd)       losses 1e-6 rel, grads 1e-3
  P4  graphed reverse steps 100..96, bf16 pair            sampling graph, heads pack, planes  bitwise
  P5  graphed reverse steps 100..96, fp32 pair            sampling graph, fp32 glue           bitwise
(P3's gradient bar is that of test_graphed_training_step_matches_eager_step: fp32 atomics in the table-gradient kernels.)
"""
import pytest
import torch

from conftest import load_golden
from diffab_pytorch_b200 import distributed as dd
from diffab_pytorch_b200 import synth
from diffab_pytorch_b200.diffab_pytorch import DiffAb, cast_pair_to_bf16
from oracle import diffusion as odiff
from oracle import ipa as oipa
from oracle import sampler as osamp

pytestmark = pytest.mark.gpu
DEV = "cuda"
TRAIN = (128, 64, 6, 32, 8, 8, 8)
LR = 1e-3
ROUTES = [
    "inplace_mul",           # control: p.mul_ under no_grad
    "load_state_dict",       # control: another synthetic state
    "adam_per_tensor",       # torch.optim.Adam(model.parameters()), eager ddp_step
    "adam_flat",             # torch.optim.Adam([bucket.flatten_parameters()]), eager ddp_step
    "flat_adam",             # distributed.FlatAdam, eager ddp_step
    "graphed_flat_adam",     # GraphedTrainStep with FlatAdam
    "graphed_adam_flat",     # GraphedTrainStep with torch.optim.Adam([flat parameter], capturable=True)
]


def _model(seed):
    model = DiffAb(*TRAIN, device=DEV)
    model.load_state_dict(synth.synthetic_state(load_golden("state_shapes.pt"), seed=seed))
    model.train_precision = "bf16"
    return model.train()


def _rel(a, b):
    return float((a.double().cpu() - b.double().cpu()).abs().max() / b.double().cpu().abs().max())


def _inputs(model):
    """Fixed inputs of every probe.  The contexts come from ``model`` on the fp32 path, before any training step."""
    cpu = synth.make_patches(2, 128, seed=61)
    b = {k: v.to(DEV) for k, v in cpu.items()}
    torch.manual_seed(62)
    t = torch.randint(low=1, high=101, size=(2,)).to(DEV)
    noise = {k: v.to(DEV) for k, v in odiff.draw_add_noise_tensors(2, 128).items()}
    x, e, R, tr = (v.to(DEV) for v in synth.make_ipa_inputs(2, seed=63))
    with torch.no_grad():
        res, pair = model.encode_context(b["seq_idx"], b["xyz"], b["orientations"], b["backbone_dihedrals"],
                                         b["distmat"], b["pairwise_dihedrals"], b["atom_mask"], b["chain_idx"],
                                         b["residue_idx"], b["generation_mask"], b["residue_mask"])
    assert pair.dtype == torch.float32
    gen = torch.Generator().manual_seed(64)
    state = osamp.draw_initial_state(cpu["seq_idx"], cpu["xyz"][:, :, 1], cpu["orientations"], cpu["generation_mask"],
                                     generator=gen)
    noises = {s: {k: v.to(DEV) for k, v in osamp.draw_step_noise(2, 128, generator=gen).items()} for s in range(100, 95, -1)}
    return {"batch": b, "t": t, "noise": noise, "ipa": (x, e.to(torch.bfloat16), R, tr),
            "ctx_mask": b["residue_mask"] & ~b["generation_mask"], "res": res, "pair": pair,
            "pair16": cast_pair_to_bf16(pair), "state": tuple(v.to(DEV) for v in state), "noises": noises}


def _probes(model, inp, sampling_order):
    b = inp["batch"]
    out = {}
    with torch.no_grad():
        out["P1"] = (model.pair_context_embedding.forward_fused_bf16(
            b["seq_idx"], b["xyz"], b["pairwise_dihedrals"], b["residue_idx"], b["chain_idx"], b["atom_mask"],
            inp["ctx_mask"]),)
        out["P2"] = (model.denoiser.ipa(*inp["ipa"]),)
    params = list(model.parameters())
    losses = model._shared_step(b, 0, t=inp["t"], noise=inp["noise"])
    # autograd.grad leaves every .grad (the gradient bucket views of the training routes) alone
    grads = torch.autograd.grad(sum(losses), params, allow_unused=True)
    out["P3"] = (torch.stack([l.detach() for l in losses]),
                 torch.cat([(torch.zeros_like(p) if g is None else g).flatten() for p, g in zip(params, grads)]))
    for name in sampling_order:
        o = model.sample_from_context(*inp["state"], inp["res"], inp["pair16"] if name == "P4" else inp["pair"],
                                      b["generation_mask"], noises=inp["noises"], t_start=100, t_stop=96,
                                      use_cuda_graph=True)
        out[name] = (o["seq_idx"], o["translations"], o["orientations"])
    for k, vs in out.items():
        for v in vs:
            assert torch.isfinite(v.float()).all(), k
    return out


def _sampling_order(k):
    """The graph cache holds one entry, so only the sampling probe whose pair dtype was captured LAST before an update
    can meet a graph captured with the old weights, and only if it runs FIRST after the update.  Alternate which one that
    is from update to update so that both graphs are tested."""
    return ("P4", "P5") if k % 2 else ("P5", "P4")


def _unmoved(got, before):
    """Probes whose floating-point outputs moved by less than 1e-3 max-normalised (1000x the P3 loss bar)."""
    out = {}
    for k, vs in got.items():
        moved = min(_rel(a, r) for a, r in zip(vs, before[k]) if a.dtype.is_floating_point)
        if not moved >= 1e-3:
            out[k] = moved
    return out


def _mismatches(got, ref):
    """Probes that differ from the reference beyond their bars (see the module docstring)."""
    out = {}
    for k in ("P1", "P2", "P4", "P5"):
        if not all(torch.equal(a, r) for a, r in zip(got[k], ref[k])):
            out[k] = max(float((a.double() - r.double()).abs().max()) for a, r in zip(got[k], ref[k]))
    (la, ga), (lr, gr) = got["P3"], ref["P3"]
    err = float((ga - gr).norm() / gr.norm())
    if not (((la - lr).abs() <= 1e-6 * lr.abs()).all() and err < 1e-3):
        out["P3"] = (float(((la - lr).abs() / lr.abs()).max()), err)
    return out


def _updater(route, model, terms):
    """Builds what the route needs and returns update(k).  Flattening the parameters moves every weight to a new address
    (which alone forces every cache to rebuild), so the bucket and the optimizer come before the first probes."""
    if route == "inplace_mul":
        def update(k):
            with torch.no_grad():
                for p in model.parameters():
                    p.mul_(0.95)
        return update
    if route == "load_state_dict":
        return lambda k: model.load_state_dict(synth.synthetic_state(load_golden("state_shapes.pt"), seed=10 + k))
    bucket = dd.GradientBucket(model.parameters())
    if route == "adam_per_tensor":
        opt = torch.optim.Adam(model.parameters(), lr=LR)
    elif route in ("adam_flat", "graphed_adam_flat"):
        opt = torch.optim.Adam([bucket.flatten_parameters()], lr=LR, capturable=route.startswith("graphed"))
    else:
        opt = dd.FlatAdam(bucket, lr=LR)
    if route.startswith("graphed"):
        step = dd.GraphedTrainStep(terms, bucket, opt, warmup=2)
        return lambda k: step()
    return lambda k: dd.ddp_step(terms, bucket, opt)


@pytest.mark.parametrize("route", ROUTES)
def test_kernels_compute_with_the_updated_weights(route):
    model = _model(0)
    inp = _inputs(model)
    update = _updater(route, model,
                      lambda: dd.diffab_loss_terms(model, inp["batch"], t=inp["t"], noise=inp["noise"]))
    before = _probes(model, inp, _sampling_order(0))         # fills every cache
    for k in (1, 2):
        update(k)
        got = _probes(model, inp, _sampling_order(k))
        # The order matters.  The reference model is built only AFTER the updated model has been probed:
        # DiffAb.load_state_dict calls invalidate_weight_caches(), which bumps the library-wide weight generation and
        # would make the updated model rebuild stale caches before they were ever read.
        snap = {n: v.detach().cpu().clone() for n, v in model.state_dict().items()}
        fresh = _model(0)
        fresh.load_state_dict(snap)
        ref = _probes(fresh, inp, _sampling_order(k))
        del fresh
        # every probe moved (a route that leaves the weights alone cannot pass) and matches the fresh model
        unmoved, wrong = _unmoved(got, before), _mismatches(got, ref)
        assert not unmoved and not wrong, f"{route}, update {k}: moved < 1e-3: {unmoved}; differ from a fresh model " \
                                          f"holding the same weights: {wrong}"
        # That bump has invalidated the updated model's caches: probe it once more, so that the next update meets caches
        # built under the current generation (and holds the sampling graph the next round's first probe reads).
        before = _probes(model, inp, _sampling_order(k))
        wrong = _mismatches(before, ref)
        assert not wrong, f"{route}, update {k}, rebuilt caches: {wrong}"
    # the snapshot is what the model computes with: the fp32 path (no caches) against the fp64 reference on it
    s, x, O = inp["state"]
    beta = model.dsched.tensors["beta"][inp["t"]]
    b = inp["batch"]
    with torch.no_grad():
        den = model.denoise(s, x, O, inp["res"], inp["pair"], beta, b["generation_mask"], b["residue_mask"])
    state64 = {n: v.double() for n, v in snap.items()}
    ref = oipa.denoiser_forward(state64, s.cpu(), x.cpu().double(), O.cpu().double(), inp["res"].cpu().double(),
                                inp["pair"].cpu().double(), beta.cpu().double(), TRAIN[2], TRAIN[-1])
    for key in ("translations_eps", "orientations_t0", "seq_posterior"):
        assert _rel(den[key], ref[key]) < 1e-4, (route, key, _rel(den[key], ref[key]))
