"""Mate rescue on the device (qm_mate_rescue: rescue_scan_kernel, rescue_align_kernel, rescue_apply_kernel over local_pass_warp)
against the CPU oracle's mate_rescue on the hand-built pairs of tests/reggen.py: every region list afterwards (every field), the
number of local alignments and their cells, for mates in each query-column template (strides 150 / 256 / 512) and three sets of
insert-size models.  tests/test_cigar_oracle.py holds the same cases against oracle/rescue_py.py."""
import numpy as np
import pytest

from tests import reggen
from tests.test_cigar_oracle import RESCUE_PES

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from quasimodo_b200 import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def genome():
    return reggen.genome()


@pytest.fixture(scope="module")
def ref(genome):
    from oracle import qmo_py
    return qmo_py.Ref(genome.codes, genome.lens, k=31)


@pytest.fixture(scope="module")
def idx(ctx, genome):
    i = ctx.index(genome, 31)
    yield i
    i.close()


@pytest.mark.parametrize("name", list(RESCUE_PES))
@pytest.mark.parametrize("max_len", [150, 256, 512])
def test_mate_rescue_cases(ctx, idx, genome, ref, name, max_len):
    import torch
    from oracle import qmo_py
    from quasimodo_b200 import _lib
    cs, pes = reggen.rescue_cases(genome, max_len, pes=reggen.rescue_pes(**RESCUE_PES[name]))
    codes, lens, regs, n_regs = reggen.region_arrays(cs)
    want, n_want = regs.copy(), n_regs.copy()
    want_stats = qmo_py.mate_rescue(ref, codes, lens, want, n_want, pes, opt=qmo_py.default_opt())
    dev = torch.device("cuda:0")
    d_regs = torch.from_numpy(regs.view(np.uint8).reshape(-1).copy()).to(dev)
    d_n = torch.from_numpy(n_regs.copy()).to(dev)
    d_stats = torch.zeros(2, dtype=torch.int64, device=dev)
    ctx.mate_rescue(idx, torch.from_numpy(codes).to(dev), torch.from_numpy(lens).to(dev), d_regs, d_n, pes, d_stats=d_stats,
                    opt=_lib.default_opt())
    torch.cuda.synchronize()
    got = d_regs.cpu().numpy().view(_lib.REG_DTYPE).reshape(-1, _lib.MAX_REGS)
    n_got = d_n.cpu().numpy()
    bad = [r for r in range(len(lens)) if n_got[r] != n_want[r] or not np.array_equal(got[r, :n_want[r]], want[r, :n_want[r]])]
    assert not bad, f"{len(bad)} reads with different regions, first {bad[0]} ({cs.tags[bad[0]]!r}): " \
                    f"{got[bad[0], :n_got[bad[0]]]} vs {want[bad[0], :n_want[bad[0]]]}"
    assert tuple(int(x) for x in d_stats.cpu()) == want_stats
    assert want_stats[0] > 0 and (n_want != n_regs).sum() > 10


def test_mate_rescue_inline_path_is_bit_exact():
    """QM_RESCUE_INLINE=1: the apply pass runs every local alignment itself instead of looking up the up-front results"""
    import os
    import subprocess
    import sys
    if os.environ.get("QM_RESCUE_INLINE"):
        pytest.skip("already inside the QM_RESCUE_INLINE run")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    p = subprocess.run([sys.executable, "-m", "pytest", "tests/test_rescue_gpu.py", "-q", "-x", "-k", "test_mate_rescue_cases"],
                       cwd=root, env=dict(os.environ, QM_RESCUE_INLINE="1"), capture_output=True, text=True)
    assert p.returncode == 0 and " passed" in p.stdout, p.stdout[-2000:] + p.stderr[-2000:]
