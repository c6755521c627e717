#!/usr/bin/env python
"""Headline benchmark: reverse-diffusion patches/s (K=128 residues, T=100 steps) on N B200.

    python bench.py --gpus N --steps K --warmup W            # this repo (sm_100a kernels)
    python bench.py --impl reference --steps K --warmup W    # CPU arm: the reference's own modules on the host cores
    python bench.py --steps K --warmup W --dump-outputs DIR  # + the sampled structures of the last timed step as .npy

One "step" = one full reverse-diffusion pass (T=100 denoise + update steps) over the rank's batch of
synthetic 128-residue CDR-H3 patches (BASELINE config 3: 256 patches per GPU; weak scaling: every
rank owns 256 independent patches, results are all-gathered with NCCL inside the timed region).
`value` times the loop with context embeddings and the t=T state resident in HBM; `e2e` times
`DiffAb.sample()` from pinned host buffers to host results (H2D, context encoding, loop, D2H).
Prints ONE JSON line (see DESIGN.md "Measurement" for every field).
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "reverse-diffusion patches/s (K=128, T=100)"
TRAIN_CFG = (128, 64, 6, 32, 8, 8, 8)  # train.py:62-70 of the reference = "DiffAb default config"
L, T = 128, 100


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--patches", type=int, default=256, help="patches per GPU")
    ap.add_argument("--precision", default="auto", choices=["auto", "bf16", "fp32"])
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-extras", action="store_true", help="skip e2e / roofline / cpu_baseline passes")
    ap.add_argument("--full-pass", action="store_true",
                    help="--impl reference only: every timed step runs all T reverse steps (minutes per step)")
    ap.add_argument("--reverse-steps", type=int, default=T,
                    help="PROFILING ONLY: run this many of the T reverse steps per pass (ncu launch lists); "
                         "the JSON line is then marked profile_only and is not a bench value")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as DIR/<name>.npy (float32; a seeded sample of the "
                         "patches above 64 MB); the same arguments give the same inputs and random draws on every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


DUMP_BYTES = 64 << 20


def dump_outputs(out, dirname, limit=DUMP_BYTES):
    """Write every array of `out` (leading dimension = patches) as `dirname`/<name>.npy in float32 (seq_idx holds
    integers < 21, exact in float32).  When all patches would exceed `limit` bytes, a fixed sample of them (seeded
    permutation, in ascending order) is written instead, with their indices in patch_index.npy (float64)."""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in out.items()}
    n = len(next(iter(arrays.values())))
    per_patch = sum(a[0].nbytes for a in arrays.values())
    if n * per_patch > limit:
        keep = (limit - 4096) // (per_patch + 8)          # 4 KB: room for the .npy headers
        idx = np.sort(np.random.default_rng(0).permutation(n)[:keep])
        arrays = {k: a[idx] for k, a in arrays.items()}
        arrays["patch_index"] = idx.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, f"{k}.npy"), a)


# ------------------------------------------------------------------------------------------------
# CPU arm (the only place bench.py executes oracle/): the UNMODIFIED reference from baseline/_ref when it is installed
# (its encode_context + denoise, stock fp32 CPU path, all host threads; the reverse update itself is the oracle's because
# the reference's sample() is a stub), else the oracle port.
# ------------------------------------------------------------------------------------------------
REF_PATCHES = int(os.environ.get("DIFFAB_REF_PATCHES", "32"))   # patches per bounded sample (threads saturate at ~32)
REF_STEPS = (T, 5)    # reverse steps of a bounded sample: one on the Gaussian IGSO(3) branch, one on the histogram branch


def cpu_sample(n_patches, steps, threads, seed=0, with_context=True):
    """One bounded sample of the workload on the host: context encoding of `n_patches` synthetic patches + the reverse
    steps `steps`; returns the runner's timing record with the T=100 rate it implies."""
    from diffab_pytorch_b200 import synth
    from oracle import reference_runner as rr

    shapes = torch.load(os.path.join(ROOT, "tests", "golden", "state_shapes.pt"), weights_only=False)
    state = synth.synthetic_state(shapes, seed=0)
    batch = synth.make_patches(n_patches, L, seed=seed, with_distmat=False)
    r = rr.timed_pass(state, batch, list(steps), threads, with_context=with_context, seed=seed)
    r["patches_per_s"] = rr.patches_per_s(r, T)
    return r


def cpu_sample_text(r):
    what = ("the UNMODIFIED reference (baseline/_ref: DiffAb.encode_context + DiffAb.denoise, stock fp32 CPU path) + the "
            "oracle's reverse update (the reference's sample() is a stub)" if r["kind"] == "reference" else
            "oracle port of the reference's PyTorch CPU path, fp32 (reference not installed); context encoders not run")
    which = "every step" if r["n_steps"] >= T else "one Gaussian-branch step, one histogram-branch step"
    return (f"{r['n_patches']} patches: context encoding once ({r['t_context_s']:.2f} s) + {r['n_steps']} of {T} reverse steps "
            f"({r['t_steps_s'] / max(r['n_steps'], 1):.2f} s each; {which}) on "
            f"{r['threads']} threads; patches/s = patches / (t_context + {T} x t_step); {what}")


def workload_name(patches_per_gpu):
    """The workload both arms are quoted on (BASELINE config 3)."""
    return (f"full reverse sampling T={T} over {patches_per_gpu} synthetic 128-residue CDR-H3 patches per GPU "
            "(BASELINE config 3), train.py model config, random-init weights")


def bench_config(patches_per_gpu, world):
    """`config` of the JSON line: identical for both arms (the workload the metric is quoted on, and how each arm
    samples it); arm-specific facts live under `arm`."""
    return {"workload": workload_name(patches_per_gpu), "patches_per_gpu": patches_per_gpu, "L": L, "T": T,
            "l2": f"pair tensor {patches_per_gpu * L * L * 64 * 2 / 1e6:.0f} MB per GPU (bf16) > 126 MB L2 "
                  "(inputs larger than L2, no flush)",
            "gather": "nccl all_gather of results inside the timed region" if world > 1 else "none",
            "reference_arm_sample": f"--impl reference times a BOUNDED sample per step: {REF_PATCHES} patches, context "
                                    f"encoding + reverse steps t={list(REF_STEPS)}, rate extrapolated to T={T} "
                                    "(every reverse step costs the same on the CPU); --full-pass runs all T steps"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    steps = list(range(T, 0, -1)) if args.full_pass else list(REF_STEPS)
    for _ in range(args.warmup if not args.full_pass else 0):
        cpu_sample(REF_PATCHES, REF_STEPS, threads)
    if args.warmup == 0 or args.full_pass:
        cpu_sample(min(REF_PATCHES, 4), (T,), threads)      # model construction (IGSO(3) table) is not timed
    t0 = time.perf_counter()
    recs = [cpu_sample(REF_PATCHES, steps, threads, seed=k) for k in range(args.steps)]
    elapsed = time.perf_counter() - t0
    value = statistics.mean(r["patches_per_s"] for r in recs)
    r = recs[-1]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "patches/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * elapsed / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.patches, args.gpus),
        "arm": {"impl": r["kind"], "reference_root": r["root"], "patches_run": r["n_patches"],
                "reverse_steps_run": r["n_steps"], "context_encoding_in_timed_region": r["with_context"],
                "full_pass": bool(args.full_pass), "precision": "fp32 (CPU)", "finite": r["finite"]},
        "cpu_baseline": {"value": value, "unit": "patches/s", "cores": threads, "kind": r["kind"],
                         "sample": cpu_sample_text(r)},
        "e2e": {"value": value, "unit": "patches/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self, skip=0):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        rows = self.rows[skip:] if len(self.rows) > skip else self.rows[-3:]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_arm(args)
    # stdout must carry exactly ONE JSON line: libraries that write to fd 1 (NCCL prints its version banner there)
    # are sent to stderr for the whole run and the line is written to the saved descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import diffab_pytorch_b200  # noqa: F401
    from diffab_pytorch_b200 import _lib, synth
    from diffab_pytorch_b200.diffab_pytorch import DiffAb, cast_pair_to_bf16

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # ---- CPU baseline on this box's host cores: rank 0 alone, BEFORE the process group exists (the other ranks sit idle
    # in the rendezvous instead of spinning in NCCL), on a bounded sample of the same workload ----
    cpu_line = None
    if rank == 0 and not args.skip_extras:
        threads = os.cpu_count() or 1
        cpu_sample(min(REF_PATCHES, 4), (T,), threads)          # model construction / first-touch, not timed
        r = cpu_sample(REF_PATCHES, REF_STEPS, threads)
        cpu_line = {"value": r["patches_per_s"], "unit": "patches/s", "cores": threads, "kind": r["kind"],
                    "sample": cpu_sample_text(r)}
    dist = None
    if world > 1:
        import datetime
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(minutes=20))
    n_gpus = world
    lib = _lib.lib()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak, peak_src = (peaks["hbm_gbs"], "measured") if "hbm_gbs" in peaks else (6650.0, "fallback")

    # ---- model + resident inputs ------------------------------------------------------------
    B = args.patches
    shapes = torch.load(os.path.join(ROOT, "tests", "golden", "state_shapes.pt"), weights_only=False)
    model = DiffAb(*TRAIN_CFG, device=dev).eval()
    model.load_state_dict(synth.synthetic_state(shapes, seed=0))   # random-init stand-in weights
    layer0 = model.denoiser.ipa.layers[0]
    precision = args.precision
    if precision == "auto":
        d = _lib.DabIpaDims(1, L, *TRAIN_CFG[:2], 8, 32, 8, 8)
        precision = "bf16" if lib.dab_ipa_packed_bytes(ctypes.byref(d)) > 0 else "fp32"
    batch = synth.make_patches(B, L, seed=1000 + rank, with_distmat=False)
    host = {k: v.pin_memory() for k, v in batch.items()}
    h2d_bytes = sum(v.numel() * v.element_size() for v in host.values())

    def sample_e2e():
        out = model.sample(host["seq_idx"], host["xyz"], host["orientations"], host["backbone_dihedrals"], None,
                           host["pairwise_dihedrals"], host["atom_mask"], host["chain_idx"], host["residue_idx"],
                           host["generation_mask"], host["residue_mask"], precision=precision,
                           use_cuda_graph=not args.no_graph)
        return {k: v.to("cpu", non_blocking=False) for k, v in out.items()}

    # resident context for the kernel-path number
    with torch.no_grad():
        b = {k: v.to(dev) for k, v in batch.items()}
        res_parts, pair_parts = [], []
        for lo in range(0, B, 32):
            sl = slice(lo, min(B, lo + 32))
            r, p = model.encode_context(b["seq_idx"][sl], b["xyz"][sl], b["orientations"][sl],
                                        b["backbone_dihedrals"][sl], synth.pairwise_atom_distances(b["xyz"][sl]),
                                        b["pairwise_dihedrals"][sl], b["atom_mask"][sl], b["chain_idx"][sl],
                                        b["residue_idx"][sl], b["generation_mask"][sl], b["residue_mask"][sl])
            res_parts.append(r)
            pair_parts.append(cast_pair_to_bf16(p) if precision == "bf16" else p)
        res_ctx, pair_ctx = torch.cat(res_parts), torch.cat(pair_parts)
        del res_parts, pair_parts
        m = b["generation_mask"]
        # the t = T state from its own seeded generator: it does not depend on what model construction drew before
        g = torch.Generator(device=dev).manual_seed(3000 + rank)
        s0 = torch.where(m, torch.randint(0, 21, (B, L), device=dev, generator=g), b["seq_idx"])
        x0 = torch.where(m[..., None], torch.randn(B, L, 3, device=dev, generator=g), b["xyz"][:, :, 1])
        O0 = torch.where(m[..., None, None], synth.uniform_rotations(B, L, generator=g, device=dev), b["orientations"])

    t_stop = T - args.reverse_steps + 1
    n_warm = max(args.warmup, 3) if args.reverse_steps == T else args.warmup

    def one_step():
        # every step restarts the sampler's random draws from one seed: a step's result depends on neither --steps nor
        # --warmup, nor on how many draws anything before it took
        torch.cuda.manual_seed(4000 + rank)
        out = model.sample_from_context(s0, x0, O0, res_ctx, pair_ctx, m, use_cuda_graph=not args.no_graph,
                                        t_stop=t_stop)
        if dist is not None:   # gather the sampled structures on every rank (7,168 B per patch)
            gathered = {}
            for k in ("seq_idx", "translations", "orientations"):
                buf = torch.empty((world,) + out[k].shape, device=dev, dtype=out[k].dtype)
                dist.all_gather_into_tensor(buf, out[k].contiguous())
                gathered[k] = buf.flatten(0, 1)
            out = gathered
        return out

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local_rank)
    clocks.start()                     # nvidia-smi needs ~1 s to start: begin before the warm-up steps
    for _ in range(n_warm):
        one_step()
    barrier()
    # launches of OUR kernels per step, counted on one eager step (graph replays do not pass through the host)
    c0 = lib.dab_launch_count()
    model.sample_from_context(s0, x0, O0, res_ctx, pair_ctx, m, use_cuda_graph=False, t_start=T, t_stop=T)
    launches_per_reverse_step = lib.dab_launch_count() - c0
    barrier()
    n_clock_warm = len(clocks.rows)    # samples taken before the timed region are dropped
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        out = one_step()
    ev1.record()
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    clock_info = clocks.stop(skip=n_clock_warm)
    if args.dump_outputs and rank == 0:
        dump_outputs(out, args.dump_outputs)
    del out
    if dist is not None:
        tmax = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        elapsed_ms = float(tmax)
    value = B * n_gpus * args.steps / (elapsed_ms / 1000.0)

    line = {
        "metric": METRIC, "value": value, "unit": "patches/s", "n_gpus": n_gpus, "steps": args.steps,
        "warmup": n_warm, "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32",
        "data": "synthetic",
        "config": bench_config(B, n_gpus),
        "arm": {"impl": "b200", "precision": precision, "cuda_graph": not args.no_graph},
        "clocks": clock_info,
        "gpu_launches": int(launches_per_reverse_step) * args.reverse_steps * args.steps,
    }
    if args.reverse_steps != T:
        line["profile_only"] = True

    if not args.skip_extras:
        # ---- roofline of the dominant kernel (IPA attention core), measured live ---------------
        if rank == 0:
            line["roofline"] = measure_roofline(model, layer0, res_ctx, pair_ctx, x0, O0, precision, hbm_peak, peak_src)
        # ---- e2e through DiffAb.sample() from pinned host memory, every rank on its own patches -----------------
        # (the resident tensors of the kernel-path measurement are released first: sample() builds its own)
        del res_ctx, pair_ctx, s0, x0, O0, b
        torch.cuda.empty_cache()
        sample_e2e()
        barrier()
        t0 = time.perf_counter()
        n_e2e = max(1, min(args.steps, 3))
        for _ in range(n_e2e):
            res = sample_e2e()
        torch.cuda.synchronize()
        e2e_s = (time.perf_counter() - t0) / n_e2e
        if dist is not None:
            tmax = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            e2e_s = float(tmax)
        d2h_bytes = sum(v.numel() * v.element_size() for v in res.values())
        line["e2e"] = {"value": B * n_gpus / e2e_s, "unit": "patches/s", "h2d_bytes_per_step": h2d_bytes,
                       "d2h_bytes_per_step": d2h_bytes, "ms_per_step": 1000 * e2e_s, "n_gpus_measured": n_gpus,
                       "note": "host wall clock around DiffAb.sample() on pinned host inputs, max over ranks; bytes are "
                               "per rank"}
    if rank == 0 and not args.skip_extras:
        line["bf16_vs_fp32"] = measure_drift(model, dev)
        line["ipa_fwd_bwd"] = measure_ipa_fwd_bwd_bf16(dev)
        line["ipa_fwd_bwd"]["fp32_path"] = measure_ipa_fwd_bwd(dev)

        line["cpu_baseline"] = cpu_line
    if not args.skip_extras and args.reverse_steps == T and dist is not None:
        # ---- BASELINE config 4: 4096 patches sharded over the ranks, T = 100, results gathered with NCCL ----
        c4 = measure_config4(model, dist, world, rank, dev, precision, not args.no_graph)
        if rank == 0:
            line["config4"] = c4
    if not args.skip_extras and args.reverse_steps == T:
        # ---- BASELINE config 5: training step, B=64 patches per GPU, all ranks (DDP all-reduce over NCCL) ------
        train = measure_train_step(dev, dist, world, shapes)
        if rank == 0:
            line["train_step"] = train
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    os.close(json_fd)


def measure_roofline(model, layer, res_ctx, pair_ctx, x0, O0, precision, hbm_peak, peak_src, iters=20):
    """Roofline of the dominant kernel (the IPA attention core) and of the whole IPA layer (the stack / n_layers), timed
    live with CUDA events on the launching stream; the input (pair tensor of all patches) is larger than L2.
    `achieved` uses SURVEY 8(d)'s ALGORITHMIC bytes of one IPA layer, B (L^2 C + 2 L D + 12 L) sz + params - what any
    implementation of the layer must move - over the kernel's / the layer's duration; the bytes the kernel's own operand
    list adds up to (which include this design's packed Q/K/V, bias planes and concat features) are reported beside it."""
    import ctypes
    from diffab_pytorch_b200 import _lib
    from diffab_pytorch_b200._lib import ptr
    from diffab_pytorch_b200.diffab_pytorch import _ipa_structs
    lib = _lib.lib()
    B = res_ctx.shape[0]
    x = res_ctx.contiguous()
    sz = pair_ctx.element_size()
    alg = B * (L * L * 64 + 2 * L * 128 + 12 * L) * sz + 303752 * 4          # SURVEY 8(d), per layer
    if precision != "bf16":
        call = lambda: layer(x, pair_ctx, O0, x0)
        with torch.no_grad():
            for _ in range(3):
                call()
            evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
            for a, b_ in evs:
                a.record(); call(); b_.record()
            torch.cuda.synchronize()
        us = statistics.mean(a.elapsed_time(b_) for a, b_ in evs) * 1000.0
        return {"bound": "hbm", "kernel": "ipa layer (fp32 CUDA-core path, all launches)", "achieved": alg / us / 1e3,
                "peak": hbm_peak, "peak_source": peak_src, "unit": "GB/s", "frac": alg / us / 1e3 / hbm_peak, "traffic": None,
                "us_per_launch": us, "algorithmic_bytes_per_launch": alg, "patches_per_launch": B}
    with torch.no_grad():
        bias = layer.pair_bias(pair_ctx)                                         # hoisted out of the loop, as in sample()
        dims = _ipa_structs(layer, B, L)
        packed = layer._packed_weights(dims)
        ws = layer._workspace(lib.dab_ipa_sm100_workspace_bytes(ctypes.byref(dims)), x.device)
        y = torch.empty(B, L, 128, device=x.device)

        def run(stages):
            _lib.check(lib.dab_ipa_fwd_sm100_stages(ctypes.byref(dims), ptr(packed), ptr(x), None, ptr(pair_ctx), ptr(bias),
                                                    ptr(O0), ptr(x0), ptr(y), None, ptr(ws), ws.numel(), stages,
                                                    _lib.stream_ptr()), "dab_ipa_fwd_sm100_stages")

        def timed(stages):
            for _ in range(3):
                run(7)                                        # a full layer first: the stage then sees the cache state
            evs = []                                          # it sees inside a stack of layers
            reps = 4                                          # launches per event pair: the queue hides the launch latency
            for _ in range(iters // reps + 1):
                run(1)
                a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(reps):
                    run(stages)
                b_.record()
                evs.append((a, b_))
                run(4)
            torch.cuda.synchronize()
            return statistics.mean(a.elapsed_time(b_) for a, b_ in evs) * 1000.0 / reps

        core_us = timed(2)
        # the whole layer as sample() runs it: the six-layer stack (per layer the attention core and ONE projection
        # kernel that carries the previous layer's to_out GEMM; 2 launches per layer + the first projection and the last
        # to_out), replayed from a CUDA graph, divided by the number of layers
        stack = model.denoiser.ipa
        planes = stack.precompute_pair_bias(pair_ctx)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            stack(x, pair_ctx, O0, x0, planes)
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            stack(x, pair_ctx, O0, x0, planes)
        for _ in range(2):
            g.replay()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(5):
            g.replay()
        b_.record()
        torch.cuda.synchronize()
        n_layers = len(stack.layers)
        layer_us = a.elapsed_time(b_) * 1000.0 / (5 * n_layers)
        del g, planes
    # bytes on the core kernel's own operand list: e row (bf16) + precomputed bias row (fp16, 8 heads) per (i, j) pair;
    # packed Q/K (2 x 768 bf16) + V (512 fp16) operands + centred t / R in, concat features (1024 bf16) out
    operand = B * L * (L * 64 * 2 + L * 8 * 2 + (768 + 768 + 512 + 1024) * 2 + 12 + 36)
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of the same launch shape from the committed ncu capture
        prof = json.load(open(os.path.join(ROOT, "profiles", "core_ncu_summary.json")))
        if prof.get("precision") == precision and prof.get("patches_per_launch") == B:
            traffic = prof["dram_bytes_per_launch"]
    except (OSError, ValueError, KeyError):
        pass
    achieved = alg / core_us / 1e3
    return {"bound": "hbm", "kernel": "ipa_core_kernel (attention core of one IPA layer, bf16 pair tensor)",
            "achieved": achieved, "peak": hbm_peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / hbm_peak,
            "traffic": traffic, "us_per_launch": core_us, "algorithmic_bytes_per_launch": alg,
            "algorithmic_bytes_source": "SURVEY 8(d): B (L^2 C + 2 L D + 12 L) 2 + params, one IPA layer",
            "patches_per_launch": B,
            "operand_list": {"bytes_per_launch": operand, "achieved": operand / core_us / 1e3,
                             "frac": operand / core_us / 1e3 / hbm_peak,
                             "note": "this design's own operands (packed Q/K/V, fp16 bias planes, concat features)"},
            "layer": {"launches": "%d-layer stack / %d: ipa_core_kernel + ipa_proj_kernel (with the previous layer's to_out "
                                  "fused) per layer, graph replay" % (n_layers, n_layers),
                      "us": layer_us, "achieved": alg / layer_us / 1e3, "frac": alg / layer_us / 1e3 / hbm_peak}}


def measure_config4(model, dist, world, rank, dev, precision, use_graph, total=4096, chunk=256):
    """BASELINE config 4: batch-sharded sampling of 4096 synthetic patches (T = 100) over the ranks of one box with an
    NCCL gather of the results.  Every rank samples its contiguous shard (4096 / N patches: 2048 / 1024 / 512 at
    N = 2 / 4 / 8) through DiffAb.sample() from pinned host buffers in chunks of 256 patches (the captured graphs of
    the main measurement are reused), then the sampled structures of all ranks are all-gathered; the time is the wall
    clock from the first H2D copy to the end of the gather, max over ranks."""
    from diffab_pytorch_b200 import synth
    from diffab_pytorch_b200.distributed import shard_bounds
    lo, hi = shard_bounds(total, world)[rank]
    chunks = []
    for c0 in range(lo, hi, chunk):
        n = min(chunk, hi - c0)
        batch = synth.make_patches(n, L, seed=500000 + c0, with_distmat=False)
        chunks.append({k: v.pin_memory() for k, v in batch.items()})

    def run():
        outs = []
        for h in chunks:
            o = model.sample(h["seq_idx"], h["xyz"], h["orientations"], h["backbone_dihedrals"], None,
                             h["pairwise_dihedrals"], h["atom_mask"], h["chain_idx"], h["residue_idx"],
                             h["generation_mask"], h["residue_mask"], precision=precision, use_cuda_graph=use_graph)
            outs.append(o)
        local = {k: torch.cat([o[k] for o in outs]) for k in outs[0]}
        gathered = {}
        for k, v in local.items():
            buf = torch.empty((world,) + v.shape, device=dev, dtype=v.dtype)
            dist.all_gather_into_tensor(buf, v.contiguous())
            gathered[k] = buf
        torch.cuda.synchronize()
        return gathered

    h = chunks[0]                                                # warm-up: graphs for this shape are captured / reused
    model.sample(h["seq_idx"], h["xyz"], h["orientations"], h["backbone_dihedrals"], None, h["pairwise_dihedrals"],
                 h["atom_mask"], h["chain_idx"], h["residue_idx"], h["generation_mask"], h["residue_mask"],
                 precision=precision, use_cuda_graph=use_graph)
    dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = run()
    dt = time.perf_counter() - t0
    tmax = torch.tensor([dt], device=dev, dtype=torch.float64)
    dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    dt = float(tmax)
    ok = bool(all(torch.isfinite(v.float()).all() for v in out.values()))
    return {"what": "BASELINE config 4: batch-sharded sampling, T=100, NCCL all-gather of {seq, x, O} inside the timed region",
            "patches_total": total, "patches_per_gpu": hi - lo, "n_gpus": world, "seconds": dt,
            "patches_per_s": total / dt, "timing": "host wall clock from first H2D to end of gather, max over ranks",
            "gathered_patches": int(out["seq_idx"].shape[0] * out["seq_idx"].shape[1]), "finite": ok}


def measure_ipa_fwd_bwd(dev, B=32, iters=5):
    """Secondary metric of BASELINE.json: one IPA layer fwd+bwd, B=32 patches x K=128 (config 2), fp32."""
    from diffab_pytorch_b200 import synth
    from diffab_pytorch_b200.diffab_pytorch import InvariantPointAttentionLayer
    layer = InvariantPointAttentionLayer(128, 64, 32, 8, 8, 8).to(dev)
    layer.load_state_dict(synth.synthetic_state(synth.ipa_layer_shapes(128, 64, 8, 32, 8, 8), seed=0))
    bufs = []
    for i in range(3):   # rotate 3 input sets (3 x 134 MB of e > L2)
        x, e, R, t = (v.to(dev) for v in synth.make_ipa_inputs(B, L, 128, 64, seed=i))
        bufs.append((x.requires_grad_(True), e.requires_grad_(True), R, t))
    gy = torch.randn(B, L, 128, device=dev)

    def run(i):
        x, e, R, t = bufs[i % 3]
        y = layer(x, e, R, t)
        y.backward(gy)
        x.grad = None; e.grad = None

    for i in range(3):
        run(i)
    torch.cuda.synchronize()
    a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        run(i)
    b_.record()
    torch.cuda.synchronize()
    us = a.elapsed_time(b_) * 1000 / iters
    alg = 3 * B * L * L * 64 * 4 + 6 * B * L * 128 * 4
    return {"metric": "IPA fwd+bwd us/layer (B=32, K=128, fp32)", "value": us, "unit": "us",
            "algorithmic_bytes": alg, "hbm_roofline_us": alg / 6528.4e9 * 1e6}


def measure_drift(model, dev, B=4):
    """north_star: "final C-alpha RMSD drift reported".  The full T=100 reverse pass of B patches through the fp32
    kernels and through the bf16 tensor-core path from the same initial state and the same injected noise (every draw of
    every step); reports the RMSD of the final C-alpha positions of the generated residues between the two paths, the
    rotation difference and the sequence agreement.  (The t ~ 100 steps divide by sqrt(alpha_t) ~ 0.03, so rounding
    differences are amplified early and then contracted; this is a property of the sampler, not of a kernel.)"""
    from diffab_pytorch_b200 import synth
    from diffab_pytorch_b200.diffab_pytorch import cast_pair_to_bf16
    g = torch.Generator(device=dev).manual_seed(1234)
    batch = {k: v.to(dev) for k, v in synth.make_patches(B, L, seed=4321, with_distmat=False).items()}
    with torch.no_grad():
        res, pair = model.encode_context(batch["seq_idx"], batch["xyz"], batch["orientations"],
                                         batch["backbone_dihedrals"], synth.pairwise_atom_distances(batch["xyz"]),
                                         batch["pairwise_dihedrals"], batch["atom_mask"], batch["chain_idx"],
                                         batch["residue_idx"], batch["generation_mask"], batch["residue_mask"])
        m = batch["generation_mask"]
        s0 = torch.where(m, torch.randint(0, 21, (B, L), device=dev, generator=g), batch["seq_idx"])
        x0 = torch.where(m[..., None], torch.randn(B, L, 3, device=dev, generator=g), batch["xyz"][:, :, 1])
        O0 = torch.where(m[..., None, None], synth.uniform_rotations(B, L, generator=g, device=dev), batch["orientations"])
        noises = {t: model.draw_step_noise(B, L, dev, generator=g) for t in range(T, 0, -1)}
        a = model.sample_from_context(s0, x0, O0, res, pair, m, noises=noises)
        b_ = model.sample_from_context(s0, x0, O0, res, cast_pair_to_bf16(pair), m, noises=noises)
        # one step from the SAME state (t = 50): isolates the per-step kernel error from the sampler's own sensitivity
        one = {t_: noises[t_] for t_ in (50,)}
        a1 = model.sample_from_context(s0, x0, O0, res, pair, m, noises=one, t_start=50, t_stop=50)
        b1 = model.sample_from_context(s0, x0, O0, res, cast_pair_to_bf16(pair), m, noises=one, t_start=50, t_stop=50)
    d1 = (a1["translations"] - b1["translations"])[m].norm(dim=-1)
    step_scale = float((a1["translations"] - x0)[m].norm(dim=-1).mean())
    d = (a["translations"] - b_["translations"])[m]
    rmsd = float(d.pow(2).sum(-1).mean().sqrt())
    rot = float((a["orientations"] - b_["orientations"])[m].abs().amax(dim=(-1, -2)).mean())
    same = float((a["seq_idx"] == b_["seq_idx"])[m].float().mean())
    spread = float((a["translations"][m] - a["translations"][m].mean(0)).pow(2).sum(-1).mean().sqrt())
    return {"what": "final state of the T=100 reverse pass, bf16 tensor-core path vs fp32 kernels, same initial state "
                    "and injected noise", "patches": B, "generated_residues": int(m.sum()),
            "ca_rmsd_angstrom": rmsd, "ca_spread_angstrom": spread, "mean_max_abs_rotation_entry_diff": rot,
            "sequence_identity": same, "finite": bool(torch.isfinite(b_["translations"]).all()),
            "one_step_t50": {"ca_max_diff_angstrom": float(d1.max()), "ca_mean_step_length_angstrom": step_scale,
                             "max_abs_rotation_entry_diff": float((a1["orientations"] - b1["orientations"])[m].abs().max()),
                             "sequence_identity": float((a1["seq_idx"] == b1["seq_idx"])[m].float().mean())},
            "note": "random-init weights: the epsilon network's outputs are not small, so the T=100 trajectory spreads "
                    "over thousands of Angstrom and orientations decorrelate; compare ca_rmsd to ca_spread, and see "
                    "one_step_t50 for the per-step error"}


def measure_train_step(dev, dist, world, shapes, B=64, steps=5, warmup=3):
    """BASELINE config 5: noising + context encoders + epsilon network forward + losses + backward + gradient
    all-reduce + Adam, B=64 synthetic patches per GPU, bf16 tensor-core IPA path (train_precision="bf16").
    Device time over `steps` steps (CUDA events), max over ranks; weak scaling (every rank has its own 64 patches)."""
    from diffab_pytorch_b200 import synth
    from diffab_pytorch_b200.diffab_pytorch import DiffAb
    from diffab_pytorch_b200.distributed import FlatAdam, GradientBucket, GraphedTrainStep, diffab_loss_terms
    rank = dist.get_rank() if dist is not None else 0
    model = DiffAb(*TRAIN_CFG, device=dev).train()
    model.load_state_dict(synth.synthetic_state(shapes, seed=0))
    model.train_precision = "bf16"
    # the reference's own training entry point runs its fp32 GEMMs as TF32 (train.py:47,
    # torch.set_float32_matmul_precision("high")); set globally so that autograd's backward GEMMs are covered too
    prev_prec = torch.get_float32_matmul_precision()
    torch.set_float32_matmul_precision("high")
    bucket = GradientBucket(model.parameters())
    # Adam over ONE flat parameter that aliases all 106 weight tensors (its gradient is the bucket): one elementwise pass
    # of the library's kernel (distributed.FlatAdam = torch.optim.Adam's update, step count on the device)
    opt = FlatAdam(bucket, lr=1e-4)
    batch = {k: v.to(dev) for k, v in synth.make_patches(B, L, seed=2000 + rank, with_distmat=False).items()}
    batch["distmat"] = torch.cat([synth.pairwise_atom_distances(batch["xyz"][i:i + 8]) for i in range(0, B, 8)])
    group = dist.group.WORLD if dist is not None else None
    # zero + forward + backward (+ Adam) captured in CUDA graphs; timesteps and noise are drawn inside the step, so every
    # replay is a different optimisation step on the resident batch
    step = GraphedTrainStep(lambda: diffab_loss_terms(model, batch), bucket, opt, group=group)

    for _ in range(warmup):
        loss = step()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        loss = step()
    b_.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b_) / steps
    if dist is not None:
        tmax = torch.tensor([ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax)
    finite = bool(torch.isfinite(loss))
    torch.set_float32_matmul_precision(prev_prec)
    del step, model, bucket, opt, batch
    torch.cuda.empty_cache()
    return {"metric": "training steps/s (config 5: B=64 patches per GPU, noising + fwd + losses + bwd + "
                      "all-reduce + Adam, bf16 tensor-core IPA)", "value": 1000.0 / ms, "unit": "steps/s",
            "patches_per_s": B * world * 1000.0 / ms, "ms_per_step": ms, "patches_per_gpu": B, "n_gpus": world,
            "cuda_graph": "whole step (zero, forward, backward, Adam) replayed from CUDA graphs; gradient all-reduce "
                          "between the backward and the optimizer graph when n_gpus > 1",
            "matmul_precision": "bf16 operands / fp32 accumulation in the library's kernels (IPA layers, pair context encoder, "
                                "aligned Linear layers of the dense glue); TF32 for the remaining PyTorch GEMMs (as the "
                                "reference's train.py:47); PyTorch's fused Adam", "loss_finite": finite}


def measure_ipa_fwd_bwd_bf16(dev, B=32, iters=20):
    """Secondary metric of BASELINE.json: one IPA layer fwd+bwd, B=32 patches x K=128 (config 2), bf16 pair tensor,
    tensor-core kernels (dab_ipa_fwd_sm100_train / dab_ipa_bwd_sm100 + the four library GEMMs).  The whole
    fwd+bwd is one CUDA graph; L2 is flushed (256 MB write) before every timed replay; also timed eagerly."""
    from diffab_pytorch_b200 import synth
    from diffab_pytorch_b200.diffab_pytorch import InvariantPointAttentionLayer
    layer = InvariantPointAttentionLayer(128, 64, 32, 8, 8, 8).to(dev)
    layer.load_state_dict(synth.synthetic_state(synth.ipa_layer_shapes(128, 64, 8, 32, 8, 8), seed=0))
    x, e, R, t = (v.to(dev) for v in synth.make_ipa_inputs(B, L, 128, 64, seed=0))
    x = x.requires_grad_(True)
    e = e.to(torch.bfloat16).requires_grad_(True)
    gy = torch.randn(B, L, 128, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        layer(x, e, R, t).backward(gy)

    def clear():
        x.grad = None; e.grad = None
        for p in layer.parameters():
            p.grad = None

    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(3):
            step(); clear()
    torch.cuda.current_stream(dev).wait_stream(side)

    def timed(fn):
        ts = []
        for _ in range(iters):
            flush.zero_()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b_.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b_) * 1000)
        ts.sort()
        return ts[len(ts) // 2]

    eager_us = timed(lambda: (step(), clear()))
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    us = timed(graph.replay)
    ok = bool(torch.isfinite(x.grad).all() and torch.isfinite(e.grad.float()).all())
    del graph
    clear()
    alg = 3 * B * L * L * 64 * 2 + 6 * B * L * 128 * 4
    return {"metric": "IPA fwd+bwd us/layer (B=32, K=128, bf16 pair tensor, tcgen05)", "value": us, "unit": "us",
            "eager_us": eager_us, "cuda_graph": True, "l2": "256 MB flush before every replay", "finite": ok,
            "algorithmic_bytes": alg, "hbm_roofline_us": alg / 6528.4e9 * 1e6}


if __name__ == "__main__":
    main()
