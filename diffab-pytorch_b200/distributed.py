"""Multi-GPU plumbing: one process per GPU, patches sharded across ranks (SURVEY §8e).

The reference is single-process (``train.py:98-100``, ``devices=1``).  Patches never interact
(every einsum keeps the batch index, ``diffab_pytorch.py:417-452``; losses sum over the batch,
``:868-878``), so both sampling and the training step shard over patches with no data-path
collective.  NCCL is used for exactly two things:

* sampling - one all-gather of the sampled structures (7,168 B per patch) at the end of a run;
* training - one all-reduce of the flat gradient bucket (2,538,468 fp32 = 10.15 MB) per step, plus
  a 1-element all-reduce of the loss-mask count so that the sharded step is EXACTLY the
  single-process large-batch step (the reference divides by the global mask count, ``:869``).

Everything here takes a ``torch.distributed`` process group, so the same code runs on ``gloo``
(CPU, used by the world_size-2 tests) and ``nccl``.
"""
import os
import warnings
from typing import Callable, Dict, Iterable, Optional

import torch
import torch.distributed as dist


def world_info(group=None):
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def shard_bounds(n: int, world: int):
    """Contiguous split of n patches over `world` ranks: sizes differ by at most one."""
    base, extra = divmod(n, world)
    bounds, lo = [], 0
    for r in range(world):
        hi = lo + base + (1 if r < extra else 0)
        bounds.append((lo, hi))
        lo = hi
    return bounds


def shard_batch(batch: Dict[str, torch.Tensor], rank: int, world: int) -> Dict[str, torch.Tensor]:
    n = next(iter(batch.values())).shape[0]
    lo, hi = shard_bounds(n, world)[rank]
    return {k: v[lo:hi] for k, v in batch.items()}


def all_gather_samples(samples: Dict[str, torch.Tensor], n_total: int, group=None) -> Dict[str, torch.Tensor]:
    """Gather per-rank sample dicts (leading dim = local patches) into the full batch on every rank.
    Shards may be ragged (n_total not divisible by world): every rank pads to the largest shard."""
    rank, world = world_info(group)
    if world == 1:
        return samples
    bounds = shard_bounds(n_total, world)
    width = max(hi - lo for lo, hi in bounds)
    out = {}
    for k, v in samples.items():
        v = v.contiguous()
        pad = torch.zeros((width,) + tuple(v.shape[1:]), dtype=v.dtype, device=v.device)
        pad[: v.shape[0]] = v
        buf = torch.empty((world * width,) + tuple(v.shape[1:]), dtype=v.dtype, device=v.device)
        dist.all_gather_into_tensor(buf, pad, group=group)
        buf = buf.view((world, width) + tuple(v.shape[1:]))
        out[k] = torch.cat([buf[r, : hi - lo] for r, (lo, hi) in enumerate(bounds)], dim=0)
    return out


def sample_sharded(model, batch: Dict[str, torch.Tensor], group=None, **sample_kwargs) -> Dict[str, torch.Tensor]:
    """``DiffAb.sample`` on this rank's contiguous shard of `batch`, then an all-gather of the results."""
    rank, world = world_info(group)
    n = batch["seq_idx"].shape[0]
    local = shard_batch(batch, rank, world)
    out = model.sample(local["seq_idx"], local["xyz"], local["orientations"], local.get("backbone_dihedrals"),
                       local.get("distmat"), local.get("pairwise_dihedrals"), local.get("atom_mask"),
                       local.get("chain_idx"), local.get("residue_idx"), local["generation_mask"],
                       local.get("residue_mask"), **sample_kwargs)
    return all_gather_samples(out, n, group=group)


class GradientBucket:
    """One flat fp32 bucket over all parameters; gradients are views into it, so the all-reduce
    needs no packing copies after the first step."""

    def __init__(self, params: Iterable[torch.nn.Parameter]):
        self.params = [p for p in params if p.requires_grad]
        total = sum(p.numel() for p in self.params)
        ref = self.params[0]
        self.flat = torch.zeros(total, dtype=ref.dtype, device=ref.device)
        off = 0
        for p in self.params:
            p.grad = self.flat[off: off + p.numel()].view_as(p)
            off += p.numel()

    def flatten_parameters(self) -> torch.nn.Parameter:
        """Move the parameters into ONE flat buffer - every parameter becomes a view of it; names, shapes and the
        state_dict are unchanged - and return the buffer as a single ``Parameter`` whose gradient is the bucket.  An
        optimizer built over ``[that parameter]`` updates all weights in one elementwise pass (PyTorch's fused Adam walks
        the 106 small tensors chunk by chunk: ~165 us per step against ~10 us).  Call it BEFORE constructing the optimizer,
        and only with elementwise optimizers (Adam / AdamW / SGD: the update of an element depends on that element alone,
        so the result is the per-tensor one, bit for bit).

        An in-place update of the flat parameter moves neither the version counter nor the data pointer of any parameter,
        so each parameter records the flat parameter (``_dab_flat_param``) and ``_lib.weight_key``, the key of the packed
        weights and captured sampling graphs, includes its version: eager optimizer steps on it need no
        ``DiffAb.invalidate_weight_caches()``.  Raw writes (``flat_param.data``, a pointer handed to a kernel) must bump
        it themselves (``torch.autograd.graph.increment_version``, as ``FlatAdam`` does) or call that method."""
        flat_p = torch.empty_like(self.flat)
        off = 0
        with torch.no_grad():
            for p in self.params:
                n = p.numel()
                flat_p[off: off + n].copy_(p.detach().reshape(-1))
                p.data = flat_p[off: off + n].view_as(p)
                off += n
        self.flat_param = torch.nn.Parameter(flat_p, requires_grad=True)
        self.flat_param.grad = self.flat
        for p in self.params:
            p._dab_flat_param = self.flat_param
        return self.flat_param

    def zero(self):
        self.flat.zero_()

    def rebind(self):
        """Optimizers / zero_grad(set_to_none=True) may drop .grad; point it back at the bucket."""
        off = 0
        for p in self.params:
            view = self.flat[off: off + p.numel()].view_as(p)
            if p.grad is None or p.grad.data_ptr() != view.data_ptr():
                if p.grad is not None:
                    view.copy_(p.grad)
                p.grad = view
            off += p.numel()

    def all_reduce(self, group=None):
        _, world = world_info(group)
        if world > 1:
            dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=group)


class FlatAdam:
    """Adam (``torch.optim.Adam`` semantics: L2 weight decay, bias corrections) on ``GradientBucket.flatten_parameters()``:
    ONE launch of the library's elementwise kernel (``dab_adam_flat``) per step - the step count lives on the device, so
    the step is CUDA-graph capturable.  PyTorch's fused Adam on the same flat tensor walks it in 64K-element chunks,
    one block each (39 blocks for DiffAb's 2.5 M weights: ~73 us); on the 106 separate tensors ~165 us."""

    def __init__(self, bucket: "GradientBucket", lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        if getattr(bucket, "flat_param", None) is None:
            bucket.flatten_parameters()
        self.bucket = bucket
        p = bucket.flat_param
        if not p.is_cuda or p.dtype != torch.float32 or p.numel() % 4 != 0:
            raise ValueError("FlatAdam: needs a CUDA fp32 flat parameter with a multiple of 4 elements")
        self.exp_avg, self.exp_avg_sq = torch.zeros_like(p.data), torch.zeros_like(p.data)
        self.step_count = torch.zeros((), device=p.device, dtype=torch.float32)
        self.param_groups = [{"params": [p], "lr": lr, "betas": betas, "eps": eps, "weight_decay": weight_decay,
                              "capturable": True}]

    def zero_grad(self, set_to_none=False):
        self.bucket.zero()

    @torch.no_grad()
    def step(self):
        from . import _lib
        g = self.param_groups[0]
        p = self.bucket.flat_param
        self.step_count.add_(1.0)
        _lib.check(_lib.lib().dab_adam_flat(_lib.ptr(p.data), _lib.ptr(self.bucket.flat), _lib.ptr(self.exp_avg),
                                            _lib.ptr(self.exp_avg_sq), _lib.ptr(self.step_count), float(g["lr"]),
                                            float(g["betas"][0]), float(g["betas"][1]), float(g["eps"]),
                                            float(g["weight_decay"]), p.numel(), _lib.stream_ptr()), "dab_adam_flat")
        # the kernel writes through a raw pointer: mark the update so weight-derived caches see it (_lib.weight_key)
        torch.autograd.graph.increment_version(p)

    def state_dict(self):
        return {"step": self.step_count.clone(), "exp_avg": self.exp_avg.clone(), "exp_avg_sq": self.exp_avg_sq.clone(),
                "param_groups": [{k: v for k, v in self.param_groups[0].items() if k != "params"}]}

    def load_state_dict(self, state):
        self.step_count.copy_(state["step"]); self.exp_avg.copy_(state["exp_avg"]); self.exp_avg_sq.copy_(state["exp_avg_sq"])
        self.param_groups[0].update(state["param_groups"][0])


def ddp_step(loss_terms: Callable[[], "tuple[torch.Tensor, torch.Tensor]"], bucket: GradientBucket,
             optimizer: Optional[torch.optim.Optimizer] = None, group=None) -> torch.Tensor:
    """One data-parallel step that reproduces the single-process large-batch step exactly.

    ``loss_terms()`` runs the local forward and returns ``(numerator, count)``: the SUM of the masked
    per-residue losses on this rank's shard and the number of masked residues (the reference's
    ``loss_denom``, ``diffab_pytorch.py:868-878``).  The global loss is sum(numerators) / sum(counts);
    each rank back-propagates numerator / global_count and the gradient bucket is summed over ranks.
    """
    bucket.rebind()
    bucket.zero()
    num, cnt = loss_terms()
    cnt = cnt.detach().to(num.dtype).reshape(1).clone()
    _, world = world_info(group)
    if world > 1:
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM, group=group)
    local = num / cnt[0]
    local.backward()
    bucket.all_reduce(group)
    if optimizer is not None:
        optimizer.step()
    total = local.detach().reshape(1).clone()
    if world > 1:
        dist.all_reduce(total, op=dist.ReduceOp.SUM, group=group)
    return total[0]


class GraphedTrainStep:
    """``ddp_step`` with the device work captured in CUDA graphs (a training step is ~550 kernel launches; issued
    eagerly the host, not the GPU, sets the step time).

    Graph A: zero the gradient bucket, forward, backward of the local loss NUMERATOR.  Between the graphs, eagerly:
    all-reduce of the mask count and of the flat bucket (``world > 1``), division by the global count - the gradient of
    numerator / global_count, exactly what ``ddp_step`` back-propagates.  Graph B: ``optimizer.step()`` (the optimizer
    must be constructed with ``capturable=True``).  With one rank everything is ONE graph; with
    ``capture_collectives=True`` (or ``DAB_GRAPH_COLLECTIVES=1``) also with several ranks - the NCCL collectives are then
    captured with the rest (measured on 2 GPUs: 4.416 ms against 4.422 ms: what the step pays for at N > 1 is the
    all-reduce itself, not the hand-over between the graphs, so the two-graph form stays the default).

    The tensors of ``batch`` (and of ``t`` / ``noise`` when given) are the graphs' static inputs: refill them in
    place (``tensor.copy_``) for the next batch.  Random draws made inside the step (timesteps, noise) advance with
    every replay, as in eager mode.  Shapes are fixed by the capture."""

    def __init__(self, loss_terms: Callable[[], "tuple[torch.Tensor, torch.Tensor]"], bucket: GradientBucket,
                 optimizer: torch.optim.Optimizer, group=None, warmup: int = 3, capture_collectives: Optional[bool] = None):
        self.bucket, self.optimizer, self.group = bucket, optimizer, group
        _, self.world = world_info(group)
        for pg in optimizer.param_groups:
            if not pg.get("capturable", False):
                raise ValueError("GraphedTrainStep: construct the optimizer with capturable=True")
        bucket.rebind()
        self._loss_terms = loss_terms
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):          # warm-up off the capture: lazy initialisations, autotuning, workspaces
            for _ in range(warmup):
                self._backward_part()
                self._reduce_part()
                optimizer.step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        from . import _lib
        self.graph_a = None
        self.graph_b = None
        if capture_collectives is None:
            capture_collectives = os.environ.get("DAB_GRAPH_COLLECTIVES", "0") == "1"
        _lib.repack_when_capturing = True     # weight-derived buffers (packed bf16 weights) are rebuilt inside the graph
        try:
            if self.world > 1 and capture_collectives:
                # The two NCCL all-reduces captured with the rest: the whole step is ONE graph on every rank.
                # NCCL's watchdog thread may touch CUDA during the capture: thread-local capture mode keeps it legal.
                try:
                    graph = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                        self._backward_part()
                        self._reduce_part()
                        optimizer.step()
                    self.graph_a, self.one_graph = graph, True
                except Exception as exc:   # noqa: BLE001 - any capture failure: fall back to the two-graph form below
                    warnings.warn(f"GraphedTrainStep: collectives not capturable here ({exc}); using two graphs")
                    torch.cuda.synchronize()
            if self.graph_a is None:
                self.one_graph = self.world == 1
                self.graph_a = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self.graph_a):
                    self._backward_part()
                    if self.world == 1:
                        self._reduce_part()
                        optimizer.step()
        finally:
            _lib.repack_when_capturing = False
        if not self.one_graph:
            self.graph_b = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_b, pool=self.graph_a.pool()):
                optimizer.step()

    def _backward_part(self):
        # Gradients are produced into fresh tensors (``.grad = None``: autograd assigns instead of launching one small
        # ``grad += new`` kernel per parameter into the bucket views) and gathered into the flat bucket by a multi-tensor
        # copy; parameters that received no gradient contribute zeros.
        bucket = self.bucket
        for p in bucket.params:
            p.grad = None
        num, cnt = self._loss_terms()
        num.backward()
        views, grads, off = [], [], 0
        for p in bucket.params:
            view = bucket.flat[off: off + p.numel()].view_as(p)
            off += p.numel()
            if p.grad is None:
                view.zero_()
            else:
                views.append(view)
                grads.append(p.grad)
            p.grad = view
        if views:
            torch._foreach_copy_(views, grads)
        self._num = num.detach().reshape(1)
        self._cnt = cnt.detach().to(num.dtype).reshape(1).clone()

    def _reduce_part(self):
        if self.world > 1:
            dist.all_reduce(self._cnt, op=dist.ReduceOp.SUM, group=self.group)
            self.bucket.all_reduce(self.group)
        self.bucket.flat.div_(self._cnt)
        self._loss = self._num / self._cnt

    def __call__(self) -> torch.Tensor:
        """One optimisation step; returns this rank's share of the global loss (sum over ranks = global loss), as a
        1-element device tensor that the next call overwrites."""
        from . import _lib
        _lib.bump_weight_generation()      # the replayed optimizer step changes weights without touching their versions
        self.graph_a.replay()
        if not self.one_graph:
            self._reduce_part()
            self.graph_b.replay()
        return self._loss


def diffab_loss_terms(model, batch, t=None, noise=None):
    """(numerator, count) of the DiffAb training loss on a local shard: the three masked-mean losses of
    ``_shared_step`` share one denominator, so numerator = (seq + pos + rot) * count."""
    seq_loss, pos_loss, rot_loss = model._shared_step(batch, 0, t=t, noise=noise)
    cnt = (batch["generation_mask"] & batch["residue_mask"]).sum()
    return (seq_loss + pos_loss + rot_loss) * cnt, cnt
