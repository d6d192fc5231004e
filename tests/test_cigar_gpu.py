"""The CIGAR stage on the device (qm_pair_finish: pair_decide_kernel, cig_score_kernel, cig_trace_kernel, cigar_kernel) against
the CPU oracle's pair_and_finish on the hand-built cases of tests/reggen.py (tests/test_cigar_oracle.py shows which task list
each family reaches).  Mate rescue is off and every insert-size model failed, so every record is the single-end finish of the
read's one region.  Every field of every record must be identical."""
import numpy as np
import pytest

from tests import reggen
from tests.test_cigar_oracle import CONFIGS, CONFIG_IDS

pytestmark = pytest.mark.gpu

FIELDS = ("rid", "pos", "flag", "mapq", "n_cigar", "score", "sub", "nm", "mate_rid", "mate_pos", "tlen", "qb", "qe")


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


def opts(scheme, w):
    from oracle import qmo_py
    from quasimodo_b200 import _lib
    return reggen.set_opt(qmo_py.default_opt(), scheme, w), reggen.set_opt(_lib.default_opt(), scheme, w)


def device_records(ctx, idx, arrays, og):
    import torch
    from quasimodo_b200 import _lib
    codes, lens, regs, n_regs = arrays
    dev = torch.device("cuda:0")
    d_alns = ctx.pair_finish(idx, torch.from_numpy(codes).to(dev), torch.from_numpy(lens).to(dev),
                             torch.from_numpy(regs.view(np.uint8).reshape(-1).copy()).to(dev), torch.from_numpy(n_regs.copy()).to(dev),
                             reggen.failed_pes(), opt=og)
    torch.cuda.synchronize()
    return d_alns.cpu().numpy().view(_lib.ALN_DTYPE)


def compare(g, o, cs, got, want, rows=None):
    """field by field; the message names the first differing read's family and the list its task went to"""
    rows = np.arange(len(want)) if rows is None else rows
    dbl = reggen.doubled(g)

    def where(r):
        k = int(rows[r])
        reg = cs.regs[k]
        rt = reggen.route(o, dbl, g.l_pac, cs.reads[k], reg) if reg is not None else {}
        return f"read {r} (case {k}, {cs.tags[k]!r}, list {rt.get('list')}, first {rt.get('first')}, band {rt.get('band')})"

    for f in FIELDS:
        d = np.nonzero(got[f] != want[f])[0]
        assert d.size == 0, f"field {f}: {d.size} records differ, first {where(d[0])}: {got[d[0]]} vs {want[d[0]]}"
    nc = np.where(want["n_cigar"] == 255, 0, want["n_cigar"])
    mask = np.arange(got["cigar"].shape[1])[None, :] < nc[:, None]
    d = np.nonzero((np.where(mask, got["cigar"], 0) != np.where(mask, want["cigar"], 0)).any(1))[0]
    assert d.size == 0, f"cigar: {d.size} records differ, first {where(d[0])}: {got[d[0]]} vs {want[d[0]]}"


def oracle_records(ref, arrays, oo):
    from oracle import qmo_py
    codes, lens, regs, n_regs = arrays
    return qmo_py.pair_and_finish(ref, codes, lens, regs.copy(), n_regs.copy(), reggen.failed_pes(), opt=oo)


@pytest.mark.parametrize("scheme,w", CONFIGS, ids=CONFIG_IDS)
def test_cigar_cases(ctx, idx, genome, ref, scheme, w):
    oo, og = opts(scheme, w)
    cs = reggen.cigar_cases(genome, scheme, w, long_refs=scheme == "default" and w == 100)
    arrays = cs.arrays()
    compare(genome, oo, cs, device_records(ctx, idx, arrays, og), oracle_records(ref, arrays, oo))


def test_every_list_empty_and_one_task_per_list(ctx, idx, genome, ref):
    """a batch that only takes the no-DP path (every task list empty), then one with exactly one task in each list"""
    oo, og = opts("default", 100)
    cs = reggen.cigar_cases(genome, "default", long_refs=False)
    dbl = reggen.doubled(genome)
    lists = [reggen.route(oo, dbl, genome.l_pac, r, h)["list"] if h is not None else None for r, h in zip(cs.reads, cs.regs)]
    for pick in ([k for k, c in enumerate(lists) if c is None],
                 [next(k for k, c in enumerate(lists) if c == x) for x in range(9)]):
        sub = reggen.Cases(genome, reggen.SCHEMES["default"], 5)
        for k in pick:
            sub.reads.append(cs.reads[k]); sub.regs.append(cs.regs[k]); sub.tags.append(cs.tags[k])
        arrays = sub.arrays()
        compare(genome, oo, sub, device_records(ctx, idx, arrays, og), oracle_records(ref, arrays, oo))


def test_replicated_cases(ctx, idx, genome, ref):
    """each task list's reads repeated until the list holds more tasks than its kernel has threads (or, for the warp kernel,
    more than one round of its cursor loop): the grid-stride loops and the reuse of a thread's slab region run, and every copy
    equals the oracle's record of its original.  Each read is paired with a read without a region, so that its record does not
    depend on where its copies sit."""
    oo, og = opts("default", 100)
    cs = reggen.cigar_cases(genome, "default", long_refs=False)
    dbl = reggen.doubled(genome)
    sms = ctx.sm_count
    # threads of cig_score_kernel<32 / 48 / 72> (blocks_for in qm_pair_finish), cig_trace_kernel<32 / 64 / 128> (tr_blocks) and
    # the warps of cigar_kernel, times 1.25
    threads = [sms * min(16, (227 * 1024) // (b * 128 * 6 + 1024)) * 128 for b in (32, 48, 72)] + \
              [sms * 8 * 128, sms * 4 * 128, sms * 2 * 128] + [sms * 3 * 4] * 3
    base = reggen.Cases(genome, reggen.SCHEMES["default"], 5)
    per_list = [[] for _ in range(9)]
    for read, reg, tag in zip(cs.reads, cs.regs, cs.tags):
        if reg is None:
            continue
        c = reggen.route(oo, dbl, genome.l_pac, read, reg)["list"]
        if c is None:
            continue
        per_list[c].append(len(base.reads))
        base.reads += [read, np.zeros(5, np.uint8)]
        base.regs += [reg, None]
        base.tags += [tag, "no region"]
    codes, lens, regs, n_regs = arrays = base.arrays()
    want = oracle_records(ref, arrays, oo)
    pairs = []
    for c, rows in enumerate(per_list):
        assert rows, f"no task in list {c}"
        reps = int(1.25 * threads[c]) // len(rows) + 1
        pairs.append(np.tile(np.array(rows) // 2, reps))
    pairs = np.concatenate(pairs)
    rows = np.stack([2 * pairs, 2 * pairs + 1], 1).reshape(-1)
    got = device_records(ctx, idx, (codes[rows], lens[rows], regs[rows], n_regs[rows]), og)
    compare(genome, oo, base, got, want[rows], rows)


def test_hard_limits_fail_the_call(ctx, idx, genome):
    """the warp kernel holds queries of up to 512 bases and direction matrices of up to 1 MiB: beyond either the call fails with
    QM_ELIMIT instead of returning records"""
    from quasimodo_b200 import QmError
    from tests.reggen import M, D
    oo, og = opts("default", 100)
    for ops, rev in (([(M, 260), (D, 3), (M, 260)], False),        # a 520-base query with a length difference
                     ([(M, 256), (D, 1540), (M, 256)], True)):     # 512 columns x 2,052 rows
        cs = reggen.Cases(genome, reggen.SCHEMES["default"], 9)
        cs.add(0, 3000, ops, rev)
        cs.add(0, 100, [(M, 50), (D, 2), (M, 50)])
        with pytest.raises(QmError, match="traceback scratch exhausted"):
            device_records(ctx, idx, cs.arrays(), og)
    # and the context still works afterwards
    cs = reggen.Cases(genome, reggen.SCHEMES["default"], 9)
    cs.add(0, 100, [(M, 50), (D, 2), (M, 50)])
    cs.add(0, 300, [(M, 50), (D, 2), (M, 50)], True)
    assert (device_records(ctx, idx, cs.arrays(), og)["n_cigar"] == 3).all()
