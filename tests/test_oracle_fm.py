"""The FM-index side of the oracle (oracle/qmo_fm.c), and the one part of the alignment oracle the reference can PIN:
bwa's own index files ship in the reference (ref/*.bwt, ref/*.sa; digests in tests/golden/fm_digests.json, made by
tests/golden/make_fm_digests.py).  The index the restatement builds from the packed genome must equal them byte for byte --
BWT words, the interleaved occurrence checkpoints, primary, cumulative counts and every suffix-array sample.  The SMEM search
on top of it is checked against a brute-force enumeration of super-maximal exact matches."""
import hashlib
import json
import os

import numpy as np
import pytest

from oracle import qmo_py
from quasimodo_b200 import genomes

GOLD = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fm_digests.json")))


@pytest.mark.parametrize("stem", ["Phix", "Merlin", "TB40E", "AD169"])
def test_index_equals_bwas_own_files(stem):
    G = genomes.load(stem)
    fm = qmo_py.FmIndex(codes=G.codes)
    b, s = fm.bwt_bytes(), fm.sa_bytes()
    assert len(b) == GOLD[stem]["bwt"]["bytes"] and hashlib.sha256(b).hexdigest() == GOLD[stem]["bwt"]["sha256"]
    assert len(s) == GOLD[stem]["sa"]["bytes"] and hashlib.sha256(s).hexdigest() == GOLD[stem]["sa"]["sha256"]
    # and loading the serialised files gives the same index back
    again = qmo_py.FmIndex(bwt=b, sa=s)
    assert again.bwt_bytes() == b and again.sa_bytes() == s


def test_ecoli_suffix_array_samples_equal_bwas_file():
    G = genomes.load("Ecoli")
    s = qmo_py.FmIndex(codes=G.codes).sa_bytes()
    assert len(s) == GOLD["Ecoli"]["sa"]["bytes"] and hashlib.sha256(s).hexdigest() == GOLD["Ecoli"]["sa"]["sha256"]


def brute_smems(T, q, min_len):
    """super-maximal exact matches of q against text T (bytes), as (start, end, occurrences)"""
    n = len(q)
    qs = bytes(np.asarray(q, np.uint8) + 65)

    def occ(sub):
        c, s = 0, 0
        while True:
            k = T.find(sub, s)
            if k < 0:
                return c
            c += 1
            s = k + 1
    mems = set()
    for i in range(n):
        if q[i] > 3:
            continue
        j = i
        while j < n and q[j] <= 3 and occ(qs[i:j + 1]) > 0:
            j += 1
        if j > i:
            mems.add((i, j))
    out = [(i, j, occ(qs[i:j])) for (i, j) in sorted(mems) if not any(a <= i and b >= j and (a, b) != (i, j) for (a, b) in mems)]
    return [m for m in out if m[1] - m[0] >= min_len]


def test_smem_seeds_against_brute_force():
    G = genomes.load("Phix")
    codes = np.ascontiguousarray(G.codes, np.uint8)
    n = len(codes)
    fm = qmo_py.FmIndex(codes=codes)
    ref = qmo_py.Ref(G.codes, G.lens, k=19)
    opt = qmo_py.default_opt()
    opt.min_seed_len = 19
    T = np.concatenate([codes, 3 - codes[::-1]]).astype(np.uint8)
    Ts = bytes(T + 65)
    rng = np.random.default_rng(3)
    for t in range(150):
        L = int(rng.integers(30, 120))
        p = int(rng.integers(0, n - L))
        q = codes[p:p + L].copy()
        if rng.random() < 0.5:
            q = (3 - q[::-1]).astype(np.uint8)
        for _ in range(int(rng.integers(0, 4))):
            q[rng.integers(0, L)] = rng.integers(0, 4)
        if rng.random() < 0.2:
            q[rng.integers(0, L)] = 4
        seeds = fm.seeds(ref, q, opt, max_mem_intv=0)              # rounds one and two
        got = set()
        for r, qb, ln in seeds:
            assert bytes(T[r:r + ln]) == bytes(q[qb:qb + ln]), (t, r, qb, ln)       # an exact match where the suffix array says
            got.add((int(qb), int(qb + ln)))
        want = brute_smems(Ts, list(q), 19)
        assert {(a, b) for a, b, _ in want} <= got, (t, want, sorted(got))
        for c, (a, b, occ_n) in enumerate(want):                   # every occurrence of an SMEM is reported
            assert sum(1 for r, qb, ln in seeds if (qb, qb + ln) == (a, b)) == min(occ_n, opt.max_occ)
        for (a, b) in got - {(a, b) for a, b, _ in want}:          # anything else comes from re-seeding a long, rare SMEM
            assert any(A <= a and b <= B and B - A >= 28 and c <= 10 for A, B, c in want), (t, (a, b), want)
        # third round on: only more seeds, all exact
        more = fm.seeds(ref, q, opt, max_mem_intv=20)
        assert len(more) >= len(seeds)
        for r, qb, ln in more:
            assert ln >= 19 and bytes(T[r:r + ln]) == bytes(q[qb:qb + ln])


def test_seeds_of_error_free_reads_are_the_read():
    G = genomes.load("Merlin")
    fm = qmo_py.FmIndex(codes=G.codes)
    ref = qmo_py.Ref(G.codes, G.lens, k=31)
    rng = np.random.default_rng(5)
    l_pac = len(G.codes)
    hits = 0
    for _ in range(200):
        p = int(rng.integers(0, l_pac - 150))
        q = np.ascontiguousarray(G.codes[p:p + 150], np.uint8)
        rev = rng.random() < 0.5
        if rev:
            q = (3 - q[::-1]).astype(np.uint8)
        s = fm.seeds(ref, q, max_mem_intv=0)
        full = [x for x in s if x[1] == 0 and x[2] == 150]
        want = 2 * l_pac - (p + 150) if rev else p
        assert any(x[0] == want for x in full), (p, rev, s)
        hits += len(full)
    assert hits >= 200


def test_reseeding_finds_the_second_copy_of_a_repeat():
    """round two of mem_collect_intv: a long SMEM with few occurrences is searched again from its middle for matches with MORE
    occurrences -- on a genome with a diverged repeat that is how the seeds in the other copy appear"""
    rng = np.random.default_rng(11)
    g = rng.integers(0, 4, 4000).astype(np.uint8)
    copy = g[500:740].copy()
    copy[60] = (copy[60] + 1) & 3
    copy[180] = (copy[180] + 2) & 3
    g[2500:2740] = copy                                            # second copy of g[500:740] with two substitutions
    fm = qmo_py.FmIndex(codes=g)
    ref = qmo_py.Ref(g, [len(g)], k=19)
    opt = qmo_py.default_opt()
    opt.min_seed_len = 19
    q = np.ascontiguousarray(g[520:670])                            # read from the first copy, spanning the first difference
    one = fm.seeds(ref, q, opt, max_mem_intv=0)
    T = np.concatenate([g, 3 - g[::-1]]).astype(np.uint8)
    for r, qb, ln in one:
        assert bytes(T[r:r + ln]) == bytes(q[qb:qb + ln])
    # the whole read matches copy one; re-seeding must also report the two-occurrence match on either side of the difference
    assert any(qb == 0 and ln == 150 and r == 520 for r, qb, ln in one)
    second = [(r, qb, ln) for r, qb, ln in one if 2500 <= r < 2740]
    assert second, one
    assert all(ln < 150 for _, _, ln in second)
