#!/usr/bin/env python
"""Device time of one graphed reverse step with and without per-residue amino-acid weights (sample()'s aa_bias) at
B patches of L = 128 residues, residues 56..71 generated, on the bf16 tensor-core path, with the GPU's name and power
limit.

    python tools/time_aa_bias.py [B] [repeats]

Each variant runs 50 steps (t = 100..51: two replays of the 20-step block graph and ten single-step replays) between
two CUDA events after a warm-up that captures its graphs; the two run on two models in one process, alternating
`repeats` times, so the spread of the repeats is the noise to compare them against.  The weights forbid types 1 and 20
everywhere and a random half of the types per residue."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402

import diffab_pytorch_b200  # noqa: E402,F401
from diffab_pytorch_b200 import synth  # noqa: E402
from diffab_pytorch_b200.diffab_pytorch import DiffAb, aa_bias_weights  # noqa: E402
from time_design_modes import gpu_label  # noqa: E402


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
    repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    L = 128
    dev = torch.device("cuda")
    shapes = torch.load(os.path.join(ROOT, "tests", "golden", "state_shapes.pt"), weights_only=False)
    g = torch.Generator(device=dev).manual_seed(0)
    res = torch.randn(B, L, 128, device=dev, generator=g)
    pair = torch.randn(B, L, L, 64, device=dev, generator=g).bfloat16()
    batch = {k: v.to(dev) for k, v in synth.make_patches(B, L, seed=1, with_distmat=False, cdr=(56, 72)).items()}
    s, x, O, m = batch["seq_idx"], batch["xyz"][:, :, 1].contiguous(), batch["orientations"], batch["generation_mask"]
    bias = torch.where(torch.rand(B, L, 21, device=dev, generator=g) < 0.5, float("-inf"), 0.0)
    bias[..., 3] = 0.0
    bias[..., [1, 20]] = float("-inf")
    weights = {"no weights": None, "weights": aa_bias_weights(bias, m)}
    models = {}
    for name, w in weights.items():
        model = DiffAb(128, 64, 6, 32, 8, 8, 8, device=dev).eval()
        model.load_state_dict(synth.synthetic_state(shapes, seed=0))
        for _ in range(2):
            model.sample_from_context(s, x, O, res, pair, m, use_cuda_graph=True, t_start=100, t_stop=51, seq_weight=w)
        models[name] = model
    times = {name: [] for name in weights}
    for _ in range(repeats):
        for name, model in models.items():
            torch.cuda.synchronize()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            model.sample_from_context(s, x, O, res, pair, m, use_cuda_graph=True, t_start=100, t_stop=51,
                                      seq_weight=weights[name])
            b_.record()
            torch.cuda.synchronize()
            times[name].append(a.elapsed_time(b_) * 1000 / 50)
    print(f"{gpu_label()}; B = {B}, L = {L}, residues 56..71 generated, bf16, CUDA graphs; "
          f"us per reverse step over {repeats} alternating repeats")
    for name, ts in times.items():
        print(f"  {name:12s} median {sorted(ts)[len(ts) // 2]:8.1f}   min {min(ts):8.1f}   max {max(ts):8.1f}")


if __name__ == "__main__":
    main()
