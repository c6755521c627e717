"""CPU: what ``bench.py --dump-outputs`` writes - every returned array as float32 .npy, and above the size limit a fixed,
seeded sample of the patches together with their indices."""
import os

import numpy as np
import torch

import bench


def _outputs(n, L=5):
    g = torch.Generator().manual_seed(0)
    return {"seq_idx": torch.randint(0, 21, (n, L), generator=g), "translations": torch.randn(n, L, 3, generator=g),
            "orientations": torch.randn(n, L, 3, 3, generator=g)}


def _dir_bytes(d):
    return sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d))


def test_dump_writes_every_array_as_float32(tmp_path):
    out = _outputs(6)
    d = str(tmp_path / "dump")
    bench.dump_outputs(out, d)
    assert sorted(os.listdir(d)) == sorted(f"{k}.npy" for k in out)
    for k, v in out.items():
        a = np.load(os.path.join(d, f"{k}.npy"))
        assert a.dtype == np.float32 and np.array_equal(a, v.float().numpy()), k


def test_dump_above_the_limit_is_a_fixed_sample_of_patches(tmp_path):
    out = _outputs(1000)
    per_patch = 5 * (1 + 3 + 9) * 4
    limit = 4096 + 100 * (per_patch + 8)
    dirs = [str(tmp_path / f"dump{i}") for i in range(2)]
    for d in dirs:
        bench.dump_outputs(out, d, limit=limit)
        assert _dir_bytes(d) <= limit
    idx = [np.load(os.path.join(d, "patch_index.npy")) for d in dirs]
    assert idx[0].dtype == np.float64 and np.array_equal(idx[0], idx[1])
    assert len(idx[0]) == 100 and np.all(np.diff(idx[0]) > 0)
    rows = torch.from_numpy(idx[0]).long()
    for k, v in out.items():
        assert np.array_equal(np.load(os.path.join(dirs[0], f"{k}.npy")), v[rows].float().numpy()), k
