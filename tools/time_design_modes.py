#!/usr/bin/env python
"""Device time of one graphed reverse step per design mode (co-design, fixed-backbone sequence design, structure
prediction) at B patches of L = 128 residues on the bf16 tensor-core path, with the GPU's name and power limit.

    python tools/time_design_modes.py [B] [repeats]

Each mode runs 50 steps (t = 100..51: two replays of the 20-step block graph and ten single-step replays) between two
CUDA events after a warm-up that captures its graphs; the modes are interleaved `repeats` times, so the spread of the
repeats is the noise to compare the modes against."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import diffab_pytorch_b200  # noqa: E402,F401
from diffab_pytorch_b200 import synth  # noqa: E402
from diffab_pytorch_b200.diffab_pytorch import DiffAb  # noqa: E402

MODES = {"co-design": (True, True), "sequence (fixed backbone)": (True, False), "structure": (False, True)}


def gpu_label():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return f"{name}, power limit {limit or 'unknown'}"


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
    repeats = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    dev = torch.device("cuda")
    shapes = torch.load(os.path.join(ROOT, "tests", "golden", "state_shapes.pt"), weights_only=False)
    g = torch.Generator(device=dev).manual_seed(0)
    res = torch.randn(B, 128, 128, device=dev, generator=g)
    pair = torch.randn(B, 128, 128, 64, device=dev, generator=g).bfloat16()
    batch = {k: v.to(dev) for k, v in synth.make_patches(B, 128, seed=1, with_distmat=False).items()}
    s, x, O, m = batch["seq_idx"], batch["xyz"][:, :, 1].contiguous(), batch["orientations"], batch["generation_mask"]
    models = {}
    for mode, (gs, gx) in MODES.items():
        model = DiffAb(128, 64, 6, 32, 8, 8, 8, device=dev).eval()
        model.load_state_dict(synth.synthetic_state(shapes, seed=0))
        model.generate_sequence, model.generate_structure = gs, gx
        for _ in range(2):
            model.sample_from_context(s, x, O, res, pair, m, use_cuda_graph=True, t_start=100, t_stop=51)
        models[mode] = model
    times = {mode: [] for mode in MODES}
    for _ in range(repeats):
        for mode, model in models.items():
            torch.cuda.synchronize()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            model.sample_from_context(s, x, O, res, pair, m, use_cuda_graph=True, t_start=100, t_stop=51)
            b_.record()
            torch.cuda.synchronize()
            times[mode].append(a.elapsed_time(b_) * 1000 / 50)
    print(f"{gpu_label()}; B = {B}, L = 128, bf16, CUDA graphs; us per reverse step over {repeats} interleaved repeats")
    for mode, ts in times.items():
        print(f"  {mode:28s} median {sorted(ts)[len(ts) // 2]:8.1f}   min {min(ts):8.1f}   max {max(ts):8.1f}")


if __name__ == "__main__":
    main()
