"""CPU: bench.py --dump-outputs — the seeded sample two builds are compared on, and the files it writes."""
import numpy as np
import torch

import bench


def _tensors():
    g = torch.Generator().manual_seed(0)
    return [torch.randn(3, 5, generator=g).bfloat16(), torch.randn(1000, generator=g), torch.randn(7, 11, 13, generator=g)]


def test_flat_sample_is_the_concatenation_at_seeded_sorted_positions():
    ts = _tensors()
    full = torch.cat([t.reshape(-1).float() for t in ts])
    idx = torch.randint(0, full.numel(), (500,), generator=torch.Generator().manual_seed(3)).sort().values
    s = bench.flat_sample(ts, n=500, seed=3)
    assert s.dtype == torch.float32 and torch.equal(s, full[idx])
    assert torch.equal(bench.flat_sample(ts, n=500, seed=3), s)          # same positions on every call
    assert torch.equal(bench.flat_sample(ts, n=full.numel()), full)       # small enough: everything, in order


def test_dump_outputs_writes_float32_keeping_small_shapes(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_ELEMS", 1000)
    ts = _tensors()
    loss = torch.tensor([1.5, 2.5])
    big = torch.randn(40, 40)
    bench.dump_outputs(tmp_path / "out", {"loss": loss, "params": ts, "big": big})
    got = {n: np.load(tmp_path / "out" / f"{n}.npy") for n in ("loss", "params", "big")}
    assert all(a.dtype == np.float32 for a in got.values())
    assert got["loss"].shape == (2,) and np.array_equal(got["loss"], loss.numpy())
    assert np.array_equal(got["params"], bench.flat_sample(ts, n=1000).numpy())
    assert np.array_equal(got["big"], bench.flat_sample([big], n=1000).numpy())
