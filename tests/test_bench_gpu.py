"""GPU: bench.py --dump-outputs writes what the last timed step computed."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from quasimodo_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_is_the_last_timed_step(tmp_path):
    """--warmup 1 --steps 2 on config 2 times samples TA-50-1 and TA-10-1 (step i runs sample i % 10, sample 0 is the warm-up):
    the dump must equal TA-10-1's counts, calls and stats, recomputed here through the library on the same simulated reads"""
    from quasimodo_b200 import Context, workloads
    n, L = 100_000, 150
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "2", "--pairs", str(n), "--warmup", "1",
                        "--steps", "2", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-3000:]
    ctx = Context(0)
    W = workloads.config2(2, n)
    opt = _lib.default_opt()
    opt.w = 100
    idx = ctx.index(W.ref, 31)
    s = ctx.sample(idx, opt)
    dev = torch.device("cuda:0")
    c = torch.empty((2 * n, L), dtype=torch.uint8, device=dev)
    q = torch.empty((2 * n, L), dtype=torch.uint8, device=dev)
    ctx.simulate_pairs(W, 0, n, torch.from_numpy(W.src_codes).to(dev), c, q, 0)
    s.add_pairs(c, q, torch.full((2 * n,), L, dtype=torch.int32, device=dev), pair_id0=0)
    counts = s.counts_tensor().cpu().numpy()
    calls = s.call_snps(max_calls=1 << 18)
    stats = s.stats()
    fields = [f for f in _lib.CALL_DTYPE.names if not f.startswith("pad")]
    assert len(calls) > 0
    assert np.array_equal(np.load(tmp_path / "counts_pos.npy"), np.arange(counts.shape[1]))
    assert np.array_equal(np.load(tmp_path / "counts.npy"), counts)
    assert np.array_equal(np.load(tmp_path / "calls.npy"), np.column_stack([calls[f] for f in fields]).astype(np.float64))
    assert np.load(tmp_path / "eval.npy")[0] == len(calls)
    assert np.load(tmp_path / "stats.npy").tolist() == list(stats)
    s.close()
    idx.close()
    ctx.close()
