"""bench.py --dump-outputs (CPU): the files two builds are compared by - the whole (D, I) when it fits the size cap,
otherwise the same seeded sample of query rows in both files, on every run."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
import bench  # noqa: E402


def test_dump_writes_the_whole_result_when_it_fits(tmp_path):
    g = torch.Generator().manual_seed(0)
    D = torch.randn(50, 7, generator=g)
    I = torch.randint(0, 10_000_000, (50, 7), generator=g)
    assert bench.dump_outputs(tmp_path, D, I) == 50
    d, i = np.load(tmp_path / "D.npy"), np.load(tmp_path / "I.npy")
    assert d.dtype == np.float32 and i.dtype == np.float64
    assert np.array_equal(d, D.numpy()) and np.array_equal(i, I.numpy().astype(np.float64))


def test_dump_samples_the_same_rows_of_both_arrays_under_the_cap(tmp_path):
    nq, k, limit = 5000, 100, 1_000_000
    D = torch.arange(nq * k, dtype=torch.float32).view(nq, k)
    I = torch.arange(nq * k).view(nq, k) + 2**40  # ids above the float32 range stay exact in float64
    n = bench.dump_outputs(tmp_path / "a", D, I, limit=limit)
    assert 0 < n < nq
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= limit
    d, i = np.load(tmp_path / "a" / "D.npy"), np.load(tmp_path / "a" / "I.npy")
    rows = (d[:, 0] // k).astype(np.int64)
    assert d.shape == i.shape == (n, k) and np.all(np.diff(rows) > 0)
    assert np.array_equal(d, D.numpy()[rows]) and np.array_equal(i, I.numpy()[rows].astype(np.float64))
    bench.dump_outputs(tmp_path / "b", D.clone(), I.clone(), limit=limit)
    for name in ("D.npy", "I.npy"):
        assert (tmp_path / "a" / name).read_bytes() == (tmp_path / "b" / name).read_bytes()


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_arguments_it_cannot_honour(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit) as e:
        bench.parse()
    assert e.value.code == 2
