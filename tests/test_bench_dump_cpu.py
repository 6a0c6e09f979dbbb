"""bench.py --dump-outputs on CPU tensors: float32 files, the same seeded sample on every run and for every array of one
length, the size cap, complex tensors as (re, im) pairs."""
import numpy as np
import torch

import bench


def _load(d, name):
    return np.load(d / (name + ".npy"))


def test_dump_is_float32_deterministic_and_capped(tmp_path):
    n = bench.DUMP_MAX_ELEMS + 12345
    big = torch.arange(n, dtype=torch.float64)
    small = torch.arange(6, dtype=torch.int32).reshape(2, 3)
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, {"params": big, "grads": -big, "calls": small})
    for name in ("params", "grads", "calls"):
        a, b = _load(tmp_path / "a", name), _load(tmp_path / "b", name)
        assert a.dtype == np.float32 and np.array_equal(a, b)
    p, g = _load(tmp_path / "a", "params"), _load(tmp_path / "a", "grads")
    assert p.shape == (bench.DUMP_MAX_ELEMS,) and np.array_equal(g, -p)     # same indices for arrays of one length
    assert np.all(np.diff(p) >= 0) and p.max() < n
    assert _load(tmp_path / "a", "calls").shape == (2, 3)                   # small arrays keep their shape
    assert 2 * 4 * bench.DUMP_MAX_ELEMS < 64 << 20


def test_flat_keeps_complex_parts():
    c = torch.tensor([1 + 2j, 3 - 4j], dtype=torch.complex64)
    r = torch.tensor([[5.0, 6.0]])
    assert bench.flat([r, c]).tolist() == [5.0, 6.0, 1.0, 2.0, 3.0, -4.0]
