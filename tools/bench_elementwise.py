#!/usr/bin/env python
"""Achieved HBM bandwidth of the SO(3) / diffusion kernels at sizes where they are bandwidth-bound (GPU only).
At benchmark sizes (32,768 rotations) they are launch-latency-bound (SURVEY H7); here N is large enough that each
launch moves >= 1 GB.  CUDA events on the launching stream, 3 warm-ups, median of 10; algorithmic bytes per unit as in
DESIGN.md 4.5; peak = MEASURED_PEAKS.json."""
import ctypes, json, os, statistics, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import diffab_pytorch_b200  # noqa
from diffab_pytorch_b200 import _lib, so3, synth
from diffab_pytorch_b200._lib import ptr

dev = "cuda"
lib = _lib.lib()
peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 6650.0
N = 16 * 1024 * 1024          # rotations


def timed(fn):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(10):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return statistics.median(ts)


rows = []
g = torch.Generator(device=dev).manual_seed(0)
v = torch.randn(N, 3, device=dev, generator=g)
R = torch.empty(N, 3, 3, device=dev)
s = lib.dab_so3_exp
rows.append(("so3 exp (vector_to_rotation_matrix)", 48 * N, timed(lambda: s(ptr(v), ptr(R), N, _lib.stream_ptr()))))
v2 = torch.empty_like(v)
rows.append(("so3 log (rotation_matrix_to_vector)", 48 * N, timed(lambda: lib.dab_so3_log(ptr(R), ptr(v2), N, _lib.stream_ptr()))))
S = torch.empty_like(R)
rows.append(("so3 log_skew (log_rotmat)", 72 * N, timed(lambda: lib.dab_so3_log_skew(ptr(R), ptr(S), N, _lib.stream_ptr()))))
R2 = torch.empty_like(R)
rows.append(("so3 exp_skew (exp_skew_symmetric_mat)", 72 * N, timed(lambda: lib.dab_so3_exp_skew(ptr(S), ptr(R2), N, _lib.stream_ptr()))))
k = torch.rand(N // 128, device=dev, generator=g)
rows.append(("so3 scale_rot", (72 + 4 / 128) * N, timed(lambda: lib.dab_so3_scale_rot(ptr(R), ptr(k), N, 128, ptr(R2), _lib.stream_ptr()))))
x32 = torch.randn(N * 16, device=dev, generator=g)
x16 = torch.empty(N * 16, device=dev, dtype=torch.bfloat16)
rows.append(("cast fp32 -> bf16 (pair tensor)", 6 * N * 16, timed(lambda: lib.dab_cast_f32_to_bf16(ptr(x32), ptr(x16), N * 16, _lib.stream_ptr()))))
del x32, x16, S, R2, v2

# forward noising / reverse step through the Python mirror (one fused launch each + the IGSO(3) sampler)
from diffab_pytorch_b200.diffab_pytorch import DiffAb
from diffab_pytorch_b200 import diffusion
B, L = 16384, 128
model = DiffAb(32, 16, 1, 8, 4, 4, 4, device=dev)
seq = torch.randint(0, 20, (B, L), device=dev, generator=g)
x0 = torch.randn(B, L, 3, device=dev, generator=g)
O0 = synth.uniform_rotations(B, L, device=dev)
mask = torch.zeros(B, L, dtype=torch.bool, device=dev); mask[:, 56:72] = True
t = torch.randint(1, 101, (B,), device=dev, generator=g)
noise = diffusion.draw_add_noise_tensors(B, L, device=dev)
rotvec = torch.randn(B, L, 3, device=dev, generator=g)
seq_t = torch.empty_like(seq); post = torch.empty(B, L, 21, device=dev); x_t = torch.empty_like(x0); O_t = torch.empty_like(O0)
sched = model.dsched
m8 = mask.to(torch.uint8)
fn = lambda: lib.dab_forward_noise(sched.ref(), ptr(seq), ptr(x0), ptr(O0), ptr(m8), ptr(t), B, L, ptr(noise["seq_exp"]),
                                   ptr(noise["eps"]), ptr(rotvec), 3, ptr(seq_t), ptr(post), ptr(x_t), ptr(O_t), _lib.stream_ptr())
rows.append(("forward_noise (DiffAb._add_noise, fused)", 317 * B * L, timed(fn)))
eps = torch.randn(B, L, 3, device=dev, generator=g); vth = 0.1 * torch.randn(B, L, 3, device=dev, generator=g)
z = torch.randn(B, L, 3, device=dev, generator=g)
so = torch.empty_like(seq); xo = torch.empty_like(x0); Oo = torch.empty_like(O0)
fn = lambda: lib.dab_reverse_step(sched.ref(), ptr(seq), ptr(x0), ptr(O0), ptr(eps), ptr(vth), ptr(post), ptr(m8), ptr(t), B, L,
                                  ptr(noise["seq_exp"]), ptr(z), ptr(rotvec), 3, ptr(so), ptr(xo), ptr(Oo), None, _lib.stream_ptr())
rows.append(("reverse_step (fused update)", 330 * B * L, timed(fn)))

print(f"{'kernel':44s} {'GB moved':>9s} {'ms':>8s} {'GB/s':>8s} {'of measured HBM peak':>22s}")
out = []
for name, nbytes, sec in rows:
    gbs = nbytes / sec / 1e9
    print(f"{name:44s} {nbytes/1e9:9.2f} {sec*1e3:8.3f} {gbs:8.0f} {gbs/peak:22.2f}")
    out.append({"kernel": name, "algorithmic_bytes": nbytes, "ms": sec * 1e3, "gbs": gbs, "frac_of_measured_peak": gbs / peak})
json.dump({"peak_gbs": peak, "rows": out}, open(os.path.join(ROOT, "gpurun_out", "elementwise_bw.json"), "w"), indent=1)
