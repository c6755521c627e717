"""CPU, gloo, world_size 2: host-side logic of the multi-GPU path (sharding, ragged gather, exact
data-parallel step with a flat gradient bucket).  The model here is a small torch stand-in: the
product kernels have no CPU path, the plumbing is device-agnostic."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from diffab_pytorch_b200 import distributed as dd


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_shard_bounds_cover_everything():
    for n in (0, 1, 7, 256, 4096):
        for w in (1, 2, 3, 8):
            b = dd.shard_bounds(n, w)
            assert b[0][0] == 0 and b[-1][1] == n
            assert all(b[i][1] == b[i + 1][0] for i in range(w - 1))
            sizes = [hi - lo for lo, hi in b]
            assert max(sizes) - min(sizes) <= 1
    batch = {"a": torch.arange(10), "b": torch.arange(20).view(10, 2)}
    parts = [dd.shard_batch(batch, r, 3) for r in range(3)]
    assert torch.equal(torch.cat([p["a"] for p in parts]), batch["a"])


def _masked_loss_terms(model, x, y, mask):
    per = (model(x) - y).pow(2).sum(-1)          # (n, L)
    return (per * mask).sum(), mask.sum()


def _worker(rank, world, port, n_total, tmp):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(0)
        model = torch.nn.Sequential(torch.nn.Linear(6, 16), torch.nn.ReLU(), torch.nn.Linear(16, 3))
        g = torch.Generator().manual_seed(1)
        x, y = torch.randn(n_total, 5, 6, generator=g), torch.randn(n_total, 5, 3, generator=g)
        mask = torch.rand(n_total, 5, generator=g) < 0.4          # ragged mask counts per shard
        lo, hi = dd.shard_bounds(n_total, world)[rank]
        # --- exact data-parallel step
        bucket = dd.GradientBucket(model.parameters())
        opt = torch.optim.SGD(model.parameters(), lr=0.1)
        loss = dd.ddp_step(lambda: _masked_loss_terms(model, x[lo:hi], y[lo:hi], mask[lo:hi]), bucket, opt)
        # --- ragged gather of "samples"
        local = {"seq_idx": torch.arange(lo, hi)[:, None].expand(-1, 4).contiguous(),
                 "translations": torch.arange(lo, hi, dtype=torch.float32)[:, None, None].expand(-1, 4, 3).contiguous()}
        full = dd.all_gather_samples(local, n_total)
        if rank == 0:
            torch.save({"loss": loss, "state": model.state_dict(), "flat": bucket.flat.clone(), "full": full}, tmp)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n_total", [8, 7])
def test_ddp_step_and_gather_world2(tmp_path, n_total):
    tmp = str(tmp_path / "out.pt")
    mp.spawn(_worker, args=(2, _free_port(), n_total, tmp), nprocs=2, join=True)
    got = torch.load(tmp, weights_only=False)
    # single-process reference: same step on the whole batch
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(6, 16), torch.nn.ReLU(), torch.nn.Linear(16, 3))
    g = torch.Generator().manual_seed(1)
    x, y = torch.randn(n_total, 5, 6, generator=g), torch.randn(n_total, 5, 3, generator=g)
    mask = torch.rand(n_total, 5, generator=g) < 0.4
    num, cnt = _masked_loss_terms(model, x, y, mask)
    loss = num / cnt
    loss.backward()
    torch.optim.SGD(model.parameters(), lr=0.1).step()
    assert torch.allclose(got["loss"], loss.detach(), rtol=1e-5)
    for k, v in model.state_dict().items():
        assert torch.allclose(got["state"][k], v, rtol=1e-5, atol=1e-6), k
    assert torch.equal(got["full"]["seq_idx"][:, 0], torch.arange(n_total))
    assert got["full"]["translations"].shape == (n_total, 4, 3)
    assert torch.equal(got["full"]["translations"][:, 0, 0], torch.arange(n_total, dtype=torch.float32))


def test_single_process_paths_need_no_process_group():
    model = torch.nn.Linear(3, 2)
    bucket = dd.GradientBucket(model.parameters())
    x = torch.randn(4, 3)
    loss = dd.ddp_step(lambda: (model(x).pow(2).sum(), torch.tensor(4.0)), bucket)
    assert torch.isfinite(loss)
    assert model.weight.grad.data_ptr() == bucket.flat.data_ptr()
    assert dd.all_gather_samples({"a": x}, 4)["a"] is x


def test_graphed_step_rejects_a_non_capturable_optimizer():
    """GraphedTrainStep captures optimizer.step() in a CUDA graph: an optimizer built without capturable=True keeps
    its step counters on the host and must be refused before anything is captured."""
    model = torch.nn.Linear(3, 2)
    bucket = dd.GradientBucket(model.parameters())
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    with pytest.raises(ValueError, match="capturable"):
        dd.GraphedTrainStep(lambda: (model(torch.randn(4, 3)).pow(2).sum(), torch.tensor(4.0)), bucket, opt)


def test_flat_parameter_optimizer_equals_the_per_tensor_one():
    """GradientBucket.flatten_parameters: every parameter becomes a view of one flat buffer and an optimizer over that one
    tensor (its gradient = the bucket) makes the per-tensor update, bit for bit; names and the state_dict are unchanged."""
    torch.manual_seed(0)
    ref = torch.nn.Sequential(torch.nn.Linear(5, 7), torch.nn.ReLU(), torch.nn.Linear(7, 3))
    flat = torch.nn.Sequential(torch.nn.Linear(5, 7), torch.nn.ReLU(), torch.nn.Linear(7, 3))
    flat.load_state_dict(ref.state_dict())
    keys = list(flat.state_dict().keys())
    bucket = dd.GradientBucket(flat.parameters())
    fp = bucket.flatten_parameters()
    assert list(flat.state_dict().keys()) == keys and fp.numel() == sum(p.numel() for p in ref.parameters())
    assert all(torch.equal(a, b) for a, b in zip(flat.state_dict().values(), ref.state_dict().values()))
    opt_ref = torch.optim.Adam(ref.parameters(), lr=1e-2, weight_decay=1e-3)
    opt_flat = torch.optim.Adam([fp], lr=1e-2, weight_decay=1e-3)
    for step in range(3):
        x = torch.randn(6, 5)
        opt_ref.zero_grad()
        ref(x).pow(2).sum().backward()
        opt_ref.step()
        loss = dd.ddp_step(lambda: (flat(x).pow(2).sum(), torch.tensor(1.0)), bucket, opt_flat)
        assert torch.isfinite(loss)
    for (n, a), b in zip(flat.named_parameters(), ref.parameters()):
        assert torch.equal(a, b), n
    # a checkpoint loads in place: the views stay views of the flat buffer
    flat.load_state_dict(ref.state_dict())
    assert flat[0].weight.data_ptr() == fp.data_ptr()


def test_weight_key_follows_optimizer_steps_on_the_flat_parameter():
    """_lib.weight_key decides when packed weights and captured sampling graphs are rebuilt.  An optimizer step on the
    flat parameter of flatten_parameters() changes every weight but no per-parameter version or data pointer: the key
    must change all the same, and must stay put while nothing changes."""
    from diffab_pytorch_b200 import _lib
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(5, 7), torch.nn.ReLU(), torch.nn.Linear(7, 3))
    bucket = dd.GradientBucket(model.parameters())
    fp = bucket.flatten_parameters()
    opt = torch.optim.Adam([fp], lr=1e-3)
    params = list(model.parameters())
    key = _lib.weight_key(params)
    assert _lib.weight_key(params) == key
    for _ in range(2):
        before = [p.detach().clone() for p in params]
        versions, ptrs = [p._version for p in params], [p.data_ptr() for p in params]
        dd.ddp_step(lambda: (model(torch.randn(6, 5)).pow(2).sum(), torch.tensor(1.0)), bucket, opt)
        assert all(not torch.equal(a, p) for a, p in zip(before, params))
        assert [p._version for p in params] == versions and [p.data_ptr() for p in params] == ptrs
        new = _lib.weight_key(params)
        assert new != key
        assert _lib.weight_key(params) == new
        key = new
    # in-place updates of one parameter and declared updates change it too
    with torch.no_grad():
        params[0].mul_(2.0)
    assert _lib.weight_key(params) != key
    key = _lib.weight_key(params)
    _lib.bump_weight_generation()
    assert _lib.weight_key(params) != key
