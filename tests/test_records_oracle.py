"""The two pileup oracles (oracle/qmo_pileup.c through qmo_py, and oracle/pileup_py.py) on hand-built records
(tests/recgen.py) rather than aligner output: count tensor, indel alleles and text pileup must agree exactly on the
adversarial list and on seeded random M/I/D/S records over a four-contig reference with a 1-base contig."""
import ctypes as C

import numpy as np
import pytest

from tests import recgen
from tests.recgen import D, I, M, S

OPTS = [dict(), dict(min_bq=0), dict(min_bq=30, min_mapq=20), dict(count_orphans=1, ignore_overlaps=1)]


@pytest.fixture(scope="module")
def genome():
    return recgen.Genome()


@pytest.fixture(scope="module")
def ref(genome):
    from oracle import qmo_py
    return qmo_py.Ref(genome.codes, genome.lens, k=31)


@pytest.fixture(scope="module", params=["adversarial", "random"])
def batch(request, genome):
    b = recgen.adversarial(genome) if request.param == "adversarial" else recgen.random_batch(genome, 1500, 5)
    return b.arrays(150)


def popt_of(d):
    from oracle import qmo_py
    po = qmo_py.PileupOpt()
    qmo_py.lib().qmo_pileup_opt_default(C.byref(po))
    for k, v in d.items():
        setattr(po, k, v)
    return po


def py_args(po):
    return po.min_mapq, po.min_bq, bool(po.count_orphans), bool(po.ignore_overlaps)


def test_records_are_consistent(genome, batch):
    alns, codes, quals, lens = batch
    for a, L in zip(alns, lens):
        if int(a["n_cigar"]) in (0, 255):
            continue
        ops = [(int(c) & 15, int(c) >> 4) for c in a["cigar"][:int(a["n_cigar"])]]
        assert sum(ln for op, ln in ops if op in (0, 1, 4)) == L
        assert 0 <= a["pos"] and a["pos"] + recgen.span(ops) <= genome.lens[a["rid"]]


@pytest.mark.parametrize("opt", OPTS, ids=lambda d: ",".join(f"{k}={v}" for k, v in d.items()) or "default")
def test_count_tensor(genome, ref, batch, opt):
    from oracle import qmo_py, pileup_py
    alns, codes, quals, lens = batch
    po = popt_of(opt)
    a = qmo_py.pileup(ref, alns, codes, quals, lens, popt=po)
    b = pileup_py.count_tensor(genome.offs, genome.l_pac, alns, codes, quals, lens, *py_args(po))
    assert a[:, 14].sum() > 0
    assert np.array_equal(a, b), np.argwhere(a != b)[:10]


def test_indel_table(genome, ref, batch):
    from oracle import qmo_py, pileup_py
    alns, codes, quals, lens = batch
    a = qmo_py.indels(ref, alns, codes, lens)
    b = pileup_py.indel_alleles(genome.offs, alns, codes, lens)
    got = {(int(r[0]), int(r[1]), int(r[3]), int(r[2]), int(r[5]), int(r[4])): [int(r[6]), int(r[7])] for r in a}
    assert len(got) == len(a) > 100
    assert got == b
    # the key carries the same fields: global anchor | type | clamped length | has_n | bases
    key = a[:, 8].astype(np.uint32).astype(np.uint64) | (a[:, 9].astype(np.uint32).astype(np.uint64) << np.uint64(32))
    want = ((genome.offs[a[:, 0]] + a[:, 1]).astype(np.uint64) << np.uint64(32) | a[:, 3].astype(np.uint64) << np.uint64(31)
            | a[:, 2].astype(np.uint64) << np.uint64(23) | a[:, 4].astype(np.uint64) << np.uint64(22) | a[:, 5].astype(np.uint64))
    assert np.array_equal(key, want) and (np.diff(key.astype(np.float64)) > 0).all()


@pytest.mark.parametrize("opt", OPTS, ids=lambda d: ",".join(f"{k}={v}" for k, v in d.items()) or "default")
def test_text_pileup(genome, ref, batch, opt):
    from oracle import qmo_py, pileup_py
    alns, codes, quals, lens = batch
    po = popt_of(opt)
    a = qmo_py.mpileup_text(ref, alns, codes, quals, lens, genome.names, popt=po)
    b = pileup_py.mpileup_text(genome.codes, genome.offs, genome.lens, genome.names, alns, codes, quals, lens, *py_args(po))
    assert len(a) > 10000
    if a != b:
        la, lb = a.split(b"\n"), b.split(b"\n")
        bad = [i for i in range(min(len(la), len(lb))) if la[i] != lb[i]]
        assert not bad and len(la) == len(lb), (len(la), len(lb), len(bad), la[bad[0]][:200] if bad else b"", lb[bad[0]][:200] if bad else b"")
    assert a == b


def test_overlap_cap_is_visible_above_200(ref, batch):
    """the records reach the cap: a base quality summed to 200 passes -Q 200 and fails -Q 201"""
    from oracle import qmo_py
    alns, codes, quals, lens = batch
    raw = (quals.astype(np.int64) >= 201).sum()
    n200 = qmo_py.pileup(ref, alns, codes, quals, lens, popt=popt_of(dict(min_bq=200)))
    n201 = qmo_py.pileup(ref, alns, codes, quals, lens, popt=popt_of(dict(min_bq=201)))
    assert raw > 0 and n200[:, :12].sum() > n201[:, :12].sum() > 0


def test_deleted_base_takes_the_query_cursor(genome, ref):
    """a deleted base's quality is the one at htslib's qpos = the query cursor at the D (the first base behind the deletion
    in read order, here an inserted base or a soft-clipped one), and an insertion right after a deletion prints the bases
    at qpos + 1 .. qpos + n, 'N' past the read's end"""
    from oracle import qmo_py, pileup_py
    rng = np.random.default_rng(1)
    b = recgen.Batch(genome, rng, sub=0.0, n_rate=0.0)
    ql = np.array([40] * 5 + [7, 50, 8, 9, 40, 40, 40], np.uint8)        # qualities in SEQ order
    seq = np.array(list(genome.codes[genome.offs[2] + 100:genome.offs[2] + 105]) + [0, 1, 2, 3, 0, 1, 2], np.uint8)
    # 5M 2D 2I 5M: the deleted bases carry the quality of query base 5 (7 < 13, filtered); 2I prints bases 6 and 7 (C, G)
    r0 = b.read(2, 100, [(M, 5), (D, 2), (I, 2), (M, 5)], 0, seq=seq, quals=ql)
    # 5M 2D 7S: the quality of the first soft-clipped base
    r1 = b.read(2, 100, [(M, 5), (D, 2), (S, 7)], 0, seq=seq, quals=np.array([40] * 5 + [33] + [0] * 6, np.uint8))
    b.add(r0, r1)
    alns, codes, quals, lens = b.arrays()
    a = qmo_py.mpileup_text(ref, alns, codes, quals, lens, genome.names)
    p = pileup_py.mpileup_text(genome.codes, genome.offs, genome.lens, genome.names, alns, codes, quals, lens)
    assert a == p
    lines = {int(f[1]): f for f in (l.split(b"\t") for l in a.split(b"\n") if l)}
    deleted = "".join("ACGT"[c] for c in genome.codes[genome.offs[2] + 105:genome.offs[2] + 107]).encode()
    assert lines[105][3:] == [b"2", b".-2" + deleted + b".-2" + deleted, b"II"]
    assert lines[106][3:] == [b"1", b"*", b"B"]                     # read 0 filtered (Q7), read 1 prints Q33
    del1 = recgen.Batch(genome, rng, sub=0.0, n_rate=0.0)
    s2 = np.array(list(genome.codes[genome.offs[2] + 200:genome.offs[2] + 204]) + [3, 2], np.uint8)
    q2 = np.array([40, 40, 40, 40, 20, 40], np.uint8)
    # 4M 1D 2I: the deletion takes base 4's quality (20 -> '5') and, as htslib prints it, the insertion base 5 then 'N'
    del1.add(del1.read(2, 200, [(M, 4), (D, 1), (I, 2)], 0, seq=s2, quals=q2), del1.read(0, 0, [(M, 1), (S, 5)], 0, seq=s2, quals=q2))
    alns, codes, quals, lens = del1.arrays()
    a = qmo_py.mpileup_text(ref, alns, codes, quals, lens, genome.names)
    assert a == pileup_py.mpileup_text(genome.codes, genome.offs, genome.lens, genome.names, alns, codes, quals, lens)
    line = [f for f in (l.split(b"\t") for l in a.split(b"\n") if l) if f[0] == b"chrC" and f[1] == b"205"][0]
    assert line[3:] == [b"1", b"*+2GN$", b"5"]
