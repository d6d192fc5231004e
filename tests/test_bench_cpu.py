"""CPU: bench.py's --dump-outputs files (a stand-in sample on host tensors) and its argument checks."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench
from quasimodo_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class FakeSample:
    def __init__(self, n):
        self.t = torch.arange(_lib.NCH * n, dtype=torch.int32).view(_lib.NCH, n)

    def counts_tensor(self):
        return self.t


@pytest.mark.parametrize("n_cols,n_calls", [(1000, 0), (bench.DUMP_COUNT_COLS + 5000, 7)])
def test_dump_outputs_are_exact_float64(tmp_path, n_cols, n_calls):
    calls = np.zeros(n_calls, _lib.CALL_DTYPE)
    calls["pos"], calls["alt"], calls["dp"], calls["qual"], calls["af"] = np.arange(n_calls) * 7, 2, 40, 12.5, 0.1
    d_calls = torch.zeros(4096, dtype=torch.uint8)
    d_calls[:n_calls * 40] = torch.from_numpy(calls.view(np.uint8))
    s = FakeSample(n_cols)
    bench.dump_outputs(str(tmp_path), s, (n_calls, 1, 2, 3), (100, 12345), d_calls)
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(got) == ["calls", "counts", "counts_pos", "eval", "stats"]
    assert all(a.dtype == np.float64 for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    pos = got["counts_pos"].astype(np.int64)
    assert len(pos) == min(n_cols, bench.DUMP_COUNT_COLS) and np.all(np.diff(pos) > 0)
    assert np.array_equal(got["counts"], s.t.numpy()[:, pos])
    fields = [f for f in _lib.CALL_DTYPE.names if not f.startswith("pad")]
    assert got["calls"].shape == (n_calls, len(fields))
    for k, f in enumerate(fields):
        assert np.array_equal(got["calls"][:, k], calls[f].astype(np.float64))
    assert got["eval"].tolist() == [n_calls, 1, 2, 3] and got["stats"].tolist() == [100, 12345]
    bench.dump_outputs(str(tmp_path / "again"), s, (n_calls, 1, 2, 3), (100, 12345), d_calls)
    assert np.array_equal(np.load(tmp_path / "again" / "counts_pos.npy"), got["counts_pos"])


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "d"]])
def test_bench_rejects_bad_arguments(argv):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True)
    assert p.returncode == 2 and "error:" in p.stderr
