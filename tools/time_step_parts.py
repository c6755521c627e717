#!/usr/bin/env python
"""Where one graphed reverse step spends its time (GPU only): the step's sub-chains captured as separate CUDA graphs
(ten repetitions each) and replayed - front MLP, the IPA stack, heads, IGSO(3) draw + update kernel - next to the whole
step.  The difference between the whole and the sum of the parts is what the hand-offs between the parts cost.
Then the whole step, the fused IPA stack and the last to_out + heads kernel with and without the live-tile list of the
batch's generation mask (the last layer's core and the heads on the tiles of generated residues only), alternating.

    python tools/time_step_parts.py [B]
"""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import diffab_pytorch_b200  # noqa: E402,F401
from diffab_pytorch_b200 import _lib, synth  # noqa: E402
from diffab_pytorch_b200 import diffusion as _diffusion  # noqa: E402
from diffab_pytorch_b200._lib import ptr  # noqa: E402
from diffab_pytorch_b200.diffab_pytorch import FAST_L, DiffAb, _ipa_structs, live_query_tiles  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 256
REP = 10
dev = torch.device("cuda")
shapes = torch.load(os.path.join(ROOT, "tests", "golden", "state_shapes.pt"), weights_only=False)
g = torch.Generator(device=dev).manual_seed(0)
res = torch.randn(B, 128, 128, device=dev, generator=g)
pair = torch.randn(B, 128, 128, 64, device=dev, generator=g).bfloat16()
batch = {k: v.to(dev) for k, v in synth.make_patches(B, 128, seed=1, with_distmat=False).items()}
s, x, O, m = batch["seq_idx"], batch["xyz"][:, :, 1].contiguous(), batch["orientations"], batch["generation_mask"]
model = DiffAb(128, 64, 6, 32, 8, 8, 8, device=dev).eval()
model.load_state_dict(synth.synthetic_state(shapes, seed=0))
den = model.denoiser


def timed(fn, label):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(REP):
            fn()
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    ts = []
    for _ in range(10):
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); graph.replay(); b_.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b_) * 1000 / REP)
    ts.sort()
    print(f"  {label:34s} {ts[len(ts) // 2]:8.1f} us")
    return ts[len(ts) // 2]


with torch.no_grad():
    _ = model.so3_reverse.histograms
    bias = model._pair_bias_planes(pair)
    glue = den.sampling_cache(res)
    t = torch.full((B,), 50, device=dev, dtype=torch.int64)
    beta = model.dsched.tensors["beta"][t]
    noise = model.draw_step_noise(B, 128, dev)
    D = 128
    h16 = torch.empty(B, 128, D, device=dev, dtype=torch.bfloat16)

    def front():
        _lib.check(_lib.lib().dab_front_fwd_sm100(ptr(glue["c"]), ptr(glue["t1"]), ptr(s), B * 128, ptr(glue["w2_bf16"]),
                                                  ptr(glue["b2"]), ptr(glue["a_scratch"]), None, ptr(h16),
                                                  _lib.stream_ptr()), "front")

    hs = {}

    def stack():
        hs["h"] = den.ipa(h16, pair, O, x, bias)

    front(); stack()
    h = hs["h"].contiguous()
    eps = torch.empty(B, 128, 3, device=dev); rot = torch.empty(B, 128, 3, device=dev); post = torch.empty(B, 128, 21, device=dev)

    def heads():
        _lib.check(_lib.lib().dab_heads_fwd_sm100(ptr(glue["heads_packed"]), ptr(h), ptr(beta), B, 128, ptr(eps), ptr(rot),
                                                  ptr(post), _lib.stream_ptr()), "heads")

    heads()
    s1, x1, O1 = s.clone(), x.clone(), O.clone()

    def update():
        _diffusion.fused_reverse_step(model.dsched, model.so3_reverse, s1, x1, O1, eps, rot, post, m, t, noise, inplace=True)

    def eps_net():
        den.heads_fast(s1, x1, O1, glue, pair, beta, bias)

    def whole():
        model.reverse_step(s1, x1, O1, res, pair, m, t, noise, inplace=True, pair_bias=bias, glue_cache=glue, beta=beta)

    print(f"B={B}: device time per repetition (graph of {REP} repetitions)")
    parts = [timed(front, "front MLP (act + GEMM)"), timed(stack, "IPA stack (6 layers)"), timed(heads, "heads"),
             timed(update, "IGSO(3) draw + reverse-step update")]
    e = timed(eps_net, "epsilon network (front+stack+heads)")
    w = timed(whole, "whole reverse step")
    print(f"  sum of the four parts {sum(parts):.1f} us; epsilon network {e:.1f}; whole step {w:.1f}")

    live = live_query_tiles(m)
    n_live = int(live[1])
    print(f"live tiles: {n_live} of {B * 128 // 16} (generation mask of the batch)")
    ipa = den.ipa
    front_arg = (glue, s)

    def stack_fused(lv):
        return lambda: ipa._forward_fused_stack(None, pair, O, x, bias, front=front_arg, live=lv)

    # the last layer's to_out + heads alone, on the concat features the stack leaves in the shared workspace
    lib = _lib.lib()
    layers = ipa.layers
    dims = _ipa_structs(layers[0], B, 128)
    ws = layers[0]._workspace(max(lib.dab_ipa_sm100_workspace_bytes(ctypes.byref(dims)), 16), dev)
    pk_last = layers[-1]._packed_weights(dims)
    offs = (ctypes.c_size_t * 8)(); poffs = (ctypes.c_size_t * 7)()
    _lib.check(lib.dab_ipa_sm100_workspace_layout(ctypes.byref(dims), offs), "layout")
    _lib.check(lib.dab_ipa_packed_layout(ctypes.byref(dims), poffs), "packed layout")

    def out_heads(lv):
        return lambda: _lib.check(lib.dab_out_heads_fwd_sm100(
            ptr(glue["heads_packed"]), ws.data_ptr() + offs[4], pk_last.data_ptr() + poffs[1], pk_last.data_ptr() + poffs[3],
            ptr(beta), B, FAST_L, ptr(eps), ptr(rot), ptr(post), None if lv is None else ptr(lv[0]),
            None if lv is None else ptr(lv[1]), _lib.stream_ptr()), "out_heads")

    def whole_step(lv):
        return lambda: model.reverse_step(s1, x1, O1, res, pair, m, t, noise, inplace=True, pair_bias=bias, glue_cache=glue,
                                          beta=beta, live=lv)

    rows = []
    for name, mk in (("whole reverse step", whole_step), ("IPA stack (fused, 6 layers)", stack_fused),
                     ("last to_out + heads", out_heads)):
        a, b_ = [], []
        for _ in range(3):   # alternating
            a.append(timed(mk(None), f"{name}: all tiles"))
            b_.append(timed(mk(live), f"{name}: live tiles"))
        a.sort(); b_.sort()
        rows.append((name, a[1], b_[1]))
    print("medians of three alternating runs:")
    for name, a, b_ in rows:
        print(f"  {name:30s} all {a:8.1f} us  live {b_:8.1f} us  saved {a - b_:7.1f} us ({100 * (a - b_) / a:.1f} %)")
