"""The hash seeder's contract (DESIGN.md 5.1) on hand-built repetitive genomes (tests/seedgen.py), CPU only: the oracle's seeds equal a
brute force of the contract, seed for seed, on every family, at k = 31, 20 and 16 and across the occurrence cap; and every family
reaches what it is there for (64 seeds, 16 regions, copy counts 2..5 in mixed strands, per-strand counts 32 and 33, palindromic
k-mers, seeds at position 0, at l_pac and at contig ends), so that a family cannot silently stop testing anything."""
import numpy as np
import pytest

from oracle import qmo_py
from tests import seedgen as sg

N_READS = 64


def occs_of(g):
    """max_occ values a family is run at: all of them where the cap matters, the default and a tight one elsewhere"""
    return sg.MAX_OCCS if g.name.startswith(("occ", "tan")) else (500, 2)


@pytest.fixture(scope="module", params=[31, 20, 16])
def runs(request):
    k = request.param
    out = []
    for g in sg.families(k):
        ix = sg.KmerIndex(g, k)
        ref = qmo_py.Ref(g.codes, g.lens, k=k)
        codes, lens = sg.reads(g, k, N_READS, 150, seed=1000 + k)
        for mo in occs_of(g):
            opt = qmo_py.default_opt()
            opt.min_seed_len, opt.max_occ = k, mo
            o = qmo_py.align_se(ref, codes, lens, opt=opt)
            stats = {}
            want = sg.brute_batch(ix, codes, lens, mo, stats)
            out.append(dict(g=g, k=k, max_occ=mo, codes=codes, lens=lens, o=o, want=want, stats=stats))
    return k, out


def test_oracle_seeds_equal_brute_force(runs):
    k, rs = runs
    for x in rs:
        got = sg.seed_lists(x["o"]["seeds"], x["o"]["n_seeds"])
        bad = [r for r in range(len(got)) if got[r] != x["want"][r]]
        assert not bad, (x["g"].name, k, x["max_occ"], bad[:5], got[bad[0]][:8], x["want"][bad[0]][:8])


def test_families_reach_the_caps(runs):
    """reads at exactly 64 seeds and at 16 regions, both through the tandem and the occurrence families"""
    k, rs = runs
    at64 = {x["g"].name for x in rs if (x["o"]["n_seeds"] == sg.MAX_SEEDS).any()}
    at16 = {x["g"].name for x in rs if (x["o"]["n_regs"] == qmo_py.MAX_REGS).any()}
    assert {"tan30d", "tan45d", "tan45x"} <= at64, sorted(at64)
    assert {"tan30d", "tan45d"} <= at16, sorted(at16)
    assert sum(int((x["o"]["n_seeds"] == sg.MAX_SEEDS).sum()) for x in rs) > 100
    assert sum(int((x["o"]["n_regs"] == qmo_py.MAX_REGS).sum()) for x in rs) > 100


def test_families_reach_copy_counts_and_strand_splits(runs):
    """k-mers with 2, 3, 4 and 5 occurrences in total, with hits on both strands, were looked up by reads (the tracked path and one
    past it); per-strand counts of 32 (kept) and 33 (ignored) occurred; at even k, palindromic k-mers were looked up"""
    k, rs = runs
    counts = set().union(*(x["stats"].get("strand_counts", set()) for x in rs))
    for tot in (2, 3, 4, 5):
        assert any(a + b == tot and a and b for a, b in counts), tot
        assert any(a + b == tot and not (a and b) for a, b in counts), tot
    assert (1, 1) in counts
    per_strand = {a for a, b in counts} | {b for a, b in counts}
    assert {31, 32, 33} <= per_strand
    assert any(a == 20 and b == 20 for a, b in counts) and any(a == 33 and b == 1 for a, b in counts)
    pal = set().union(*(x["stats"].get("palindromes", set()) for x in rs))
    assert bool(pal) == (k % 2 == 0), pal


def test_families_reach_contig_ends(runs):
    """seeds that start at position 0, end at l_pac (the doubled coordinates' midpoint) and touch inner contig boundaries"""
    k, rs = runs
    x = next(x for x in rs if x["g"].name == "ctg" and x["max_occ"] == 500)
    g = x["g"]
    spans = {sg.fwd_span(g.l_pac, s) for ss in x["want"] for s in ss}
    assert any(b == 0 for b, e in spans) and any(e == g.l_pac for b, e in spans)
    starts, ends = {b for b, e in spans}, {e for b, e in spans}
    inner = [int(o) for o in g.offs[1:-1]]
    assert sum(o in starts for o in inner) >= 4 and sum(o in ends for o in inner) >= 4
    # contig 1 is k - 1 bases long: nothing may be seeded inside it
    assert not any(g.offs[1] <= b < g.offs[2] for b, e in spans)
    # a seed of exactly k bases over the whole of contig 2 (k bases long)
    assert (int(g.offs[2]), int(g.offs[3])) in spans


def test_max_occ_cap_is_per_strand_pass():
    """20 + 20 copies: each pass sees 20 hits, so at max_occ = 20 a read inside the array gets hits on both strands; at 19 none"""
    g = sg.occurrences(20, 20)
    k = 31
    ix = sg.KmerIndex(g, k)
    ref = qmo_py.Ref(g.codes, g.lens, k=k)
    b = g.hot[0][0]
    read = np.ascontiguousarray(g.codes[b:b + 40][None, :])
    for mo, want in ((20, 40), (19, 0)):
        opt = qmo_py.default_opt()
        opt.max_occ = mo
        o = qmo_py.align_se(ref, read, np.array([40], np.int32), opt=opt)
        assert int(o["n_seeds"][0]) == want == len(sg.brute_seeds(ix, read[0], mo))
