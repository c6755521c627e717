"""CPU: host-side logic of the mirror - state-dict compatibility, schedule, context encoders
(PyTorch modules, bit-identical to the reference's on the golden inputs), API surface."""
import inspect

import torch

from conftest import load_golden
from diffab_pytorch_b200 import diffusion, synth
from diffab_pytorch_b200.diffab_pytorch import (DiffAb, Denoiser, InvariantPointAttentionLayer,
                                                InvariantPointAttentionModule, OrientationLoss)

TRAIN = (128, 64, 6, 32, 8, 8, 8)


def test_state_dict_matches_reference_keys_and_shapes():
    shapes = load_golden("state_shapes.pt")
    model = DiffAb(*TRAIN)
    sd = model.state_dict()
    assert list(sd.keys()) == list(shapes.keys())
    for k, shp in shapes.items():
        assert tuple(sd[k].shape) == tuple(shp), k
    assert sum(v.numel() for v in sd.values()) == 2538468
    # schedules / tables are not in the state dict (the only buffers are non-persistent constants)
    assert not set(n for n, _ in model.named_buffers()) & set(sd.keys())
    model.load_state_dict(synth.synthetic_state(shapes, seed=0))  # "reference checkpoint" loads unchanged


def test_constructor_signature_and_methods():
    params = list(inspect.signature(DiffAb.__init__).parameters)
    assert params[1:17] == ["d_residue_emb", "d_pair_emb", "n_ipa_layers", "d_scalar_per_head",
                            "n_query_point_per_head", "n_value_point_per_head", "n_head", "T", "s", "beta_max",
                            "n_atoms", "aa_vocab_size", "max_dist_to_consider", "lr", "weight_decay", "betas"]
    for name in ("encode_context", "denoise", "sample", "_add_noise", "_shared_step", "training_step",
                 "validation_step", "configure_optimizers"):
        assert callable(getattr(DiffAb, name))
    model = DiffAb(*TRAIN)
    assert model.T == 100 and set(model.sched) == {"alpha", "alpha_bar", "alpha_bar_sqrt",
                                                    "one_minus_alpha_bar_sqrt", "beta"}
    assert isinstance(model.configure_optimizers(), torch.optim.Adam)
    assert len(model.denoiser.ipa.layers) == 6
    layer = model.denoiser.ipa.layers[0]
    assert abs(float(layer.gamma[0]) - 0.5413) < 1e-3            # softplus^-1(1), used raw
    assert layer.scale_total == 3 ** -0.5 and layer.scale_point == (4.5 * 8) ** -0.5


def test_schedule_matches_reference():
    g = load_golden("schedule.pt")
    s = diffusion.cosine_variance_schedule(100, s=0.01, beta_max=0.999)
    for k in g:
        assert torch.equal(s[k], g[k]), k


def test_context_encoders_match_reference_bitwise():
    g = load_golden("denoiser.pt")
    model = DiffAb(*TRAIN, device="cpu")     # CPU modules on CPU inputs, also on a machine with a GPU
    model.load_state_dict(synth.synthetic_state(load_golden("state_shapes.pt"), seed=g["seed_state"]))
    b = synth.make_patches(2, 128, seed=g["seed_patches"])
    with torch.no_grad():
        res, pair = model.encode_context(b["seq_idx"], b["xyz"], b["orientations"], b["backbone_dihedrals"],
                                         b["distmat"], b["pairwise_dihedrals"], b["atom_mask"], b["chain_idx"],
                                         b["residue_idx"], b["generation_mask"], b["residue_mask"])
    assert torch.equal(res, g["res_ctx"])
    assert torch.equal(pair[:, ::8, ::8], g["pair_ctx"]["sub"])
    assert abs(float(pair.double().sum()) - g["pair_ctx"]["sum"]) < 1e-6
    # mask logic (A19): context = residue & ~generation
    assert int((b["residue_mask"] & ~b["generation_mask"]).sum()) == 2 * (128 - 16)


def test_pair_embedding_backward_works():
    # the reference's in-place distmat ops break autograd (SURVEY F5a); ours must not
    model = DiffAb(32, 16, 1, 8, 4, 4, 4, device="cpu")
    b = synth.make_patches(1, 12, seed=2, cdr=(4, 8))
    res, pair = model.encode_context(b["seq_idx"], b["xyz"], b["orientations"], b["backbone_dihedrals"],
                                     b["distmat"], b["pairwise_dihedrals"], b["atom_mask"], b["chain_idx"],
                                     b["residue_idx"], b["generation_mask"], b["residue_mask"])
    (res.sum() + pair.sum()).backward()
    assert model.pair_context_embedding.mlp[0].weight.grad.abs().sum() > 0


def test_orientation_loss_known_answer():
    # tests/test_loss.py:9-21 of the reference
    R = synth.uniform_rotations(16, 20, dtype=torch.float64)
    assert float(OrientationLoss(reduction="mean")(R, R)) < 1e-20


def test_module_ctor_shapes_from_reference_tests():
    # tests/test_modules.py:143-221 instantiate these shapes
    InvariantPointAttentionLayer(32, 16, 16, 4, 4, 8)
    InvariantPointAttentionModule(4, 32, 16, 16, 4, 4, 8)
    d = Denoiser(32, 16, 4, 12, 4, 4, 8, aa_vocab_size=21)
    assert d.sequence_embedding.weight.shape == (25, 32)
