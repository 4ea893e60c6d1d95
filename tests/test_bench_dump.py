"""bench.py --dump-outputs (no GPU: the result tensors live on the CPU here): the same seeded sample of rows on every run,
float32 / float64 files only, the rows of the result exactly, at most 64 MB at the size of the default workload."""
import importlib.util
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
bench = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(bench)


@pytest.mark.parametrize("nq,k,dtype", [(1_000_000, 10, torch.float32), (10_000, 10, torch.float64), (7, 3, torch.float32)])
def test_dump_outputs_sample(tmp_path, nq, k, dtype):
    idx = torch.arange(nq * k, dtype=torch.int64).reshape(nq, k) * 3
    dist = torch.arange(nq * k, dtype=dtype).reshape(nq, k) / 7
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), idx, dist)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["distances.npy", "indices.npy", "query_rows.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 64 << 20
    got = {f: np.load(tmp_path / "a" / f) for f in names}
    for f in names:
        assert got[f].dtype in (np.float32, np.float64)
        assert np.array_equal(got[f], np.load(tmp_path / "b" / f))
    rows = got["query_rows.npy"].astype(np.int64)
    assert np.all(np.diff(rows) > 0) and rows[-1] < nq
    assert rows.size == nq or rows.size >= nq // 10
    assert np.array_equal(got["indices.npy"], idx.numpy()[rows].astype(np.float64))
    assert got["distances.npy"].dtype == dist.numpy().dtype and np.array_equal(got["distances.npy"], dist.numpy()[rows])
