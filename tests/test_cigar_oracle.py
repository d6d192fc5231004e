"""The CIGAR stage of the CPU oracle (oracle/qmo_mem.c reg_to_aln through qmo_py.pair_and_finish) against the independent
restatement oracle/cigar_py.py on hand-built reads and regions (tests/reggen.py): every family of cases, four scoring schemes
and a narrow band, position / strand / CIGAR / NM of every record.  The router restatement shows which of pair.cu's task
lists each family reaches, so that tests/test_cigar_gpu.py, which runs the same cases on the device, is known to exercise
every kernel."""
import collections

import numpy as np
import pytest

from oracle import cigar_py, qmo_py
from tests import reggen

# (scheme, -w); the mate rescue cases at the end of this file
CONFIGS = [("default", 100), ("a2", 100), ("harsh", 100), ("extreme", 100), ("default", 8)]
CONFIG_IDS = [f"{s}-w{w}" for s, w in CONFIGS]
MAX_DP_OPS = qmo_py.MAX_CIGAR - 2


@pytest.fixture(scope="module")
def genome():
    return reggen.genome()


@pytest.fixture(scope="module")
def ref(genome):
    return qmo_py.Ref(genome.codes, genome.lens, k=31)


def oracle_records(ref, cs, o):
    codes, lens, regs, n_regs = cs.arrays()
    return qmo_py.pair_and_finish(ref, codes, lens, regs, n_regs, reggen.failed_pes(), opt=o)


def coverage(g, cs, o):
    """route() of every read with a region -> Counter of what the stage does with them"""
    dbl, seen = reggen.doubled(g), collections.Counter()
    for read, reg in zip(cs.reads, cs.regs):
        if reg is None:
            continue
        rt = reggen.route(o, dbl, g.l_pac, read, reg)
        seen["none" if rt["list"] is None else rt["list"]] += 1
        if rt["list"] is not None and not rt["fits16"]:
            seen["16-bit guard"] += 1
            q, t = reggen.task_seqs(dbl, g.l_pac, read, reg)
            seen["below -20000"] += qmo_py.ksw_global2(q, t, reggen.cig_band(o, 1, len(q), len(t)), o, max_cigar=4096)[0] < -20000
        if rt["list"] is not None and rt["list"] >= 6:
            lq = rt["lq"]
            seen["template " + ("5" if lq <= 160 else "8" if lq <= 256 else "16")] += 1
            need = max(n for _, n in rt["tries"])
            seen["global direction matrix" if need > reggen.DIR_SMEM else "shared direction matrix"] += 1
    return seen


@pytest.mark.parametrize("scheme,w", CONFIGS, ids=CONFIG_IDS)
def test_cigar_stage_equals_an_independent_restatement(genome, ref, scheme, w):
    g = genome
    cs = reggen.cigar_cases(g, scheme, w, long_refs=scheme == "default" and w == 100)
    o = reggen.set_opt(qmo_py.default_opt(), scheme, w)
    alns = oracle_records(ref, cs, o)
    dbl = reggen.doubled(g)
    offs = [int(x) for x in g.offs]
    seen = collections.Counter()
    for r, (read, reg) in enumerate(zip(cs.reads, cs.regs)):
        a = alns[r]
        if reg is None:
            assert a["flag"] & 4
            continue
        hit = {f: int(reg[f]) for f in ("rb", "re", "qb", "qe", "truesc", "w")}
        want = cigar_py.hit_to_record(dbl, g.l_pac, offs, read, hit, w=w, **reggen.SCHEMES[scheme])
        start = 2 * g.l_pac - hit["re"] if want["rev"] else hit["rb"]
        dp = [c for c in want["cigar"] if c[0] != 4]
        lead = offs[want["rid"]] + want["pos"] - start
        tail = (hit["re"] - hit["rb"]) - lead - sum(ln for op, ln in dp if op != 1)
        n_dp = len(dp) + (lead > 0) + (tail > 0)
        if n_dp > MAX_DP_OPS:                 # more operations than a record holds: unmapped, n_cigar 255
            assert a["n_cigar"] == 255 and a["flag"] & 4, (r, cs.tags[r], want, a)
            seen["overflow"] += 1
            continue
        got = [(int(c) & 15, int(c) >> 4) for c in a["cigar"][:int(a["n_cigar"])]]
        assert (int(a["rid"]), int(a["pos"]), bool(a["flag"] & 0x10), got, int(a["nm"])) == \
            (want["rid"], want["pos"], want["rev"], want["cigar"], want["nm"]), (r, cs.tags[r], a, want)
        seen[f"{n_dp} operations"] += n_dp == MAX_DP_OPS
        seen["gapped"] += any(op in (1, 2) for op, _ in got)
        if lead or tail:
            seen[("leading" if lead else "trailing") + (" reverse" if want["rev"] else " forward")] += 1
        seen["clipped both ends"] += got[0][0] == 4 and got[-1][0] == 4
    seen.update(coverage(g, cs, o))
    # what every configuration reaches
    need = ["none", 0, 3, 7, 8, "gapped", "overflow", f"{MAX_DP_OPS} operations", "clipped both ends",
            "leading forward", "leading reverse", "trailing forward", "trailing reverse"]
    if scheme == "extreme":                  # every task longer than ~70 bases goes to the warp kernel (cig_fits16)
        need = ["none", 0, 6, 7, "16-bit guard", "below -20000", "gapped", "overflow", "template 16"]
    elif scheme == "harsh":                  # its gap costs keep every equal-length band below 16, and its tasks of more than
        need = [k for k in need if k != 8] + [6, "16-bit guard"]          # ~150 bases go to the warp kernel (cig_fits16)
    elif w == 100:
        need += [1, 2, 4, 5, 6, "template 5", "template 8", "template 16", "global direction matrix", "shared direction matrix"]
    missing = [k for k in need if seen[k] == 0]
    assert not missing, (missing, seen)



# ---------------------------------------------------------------------------------------------------------------------
# mate rescue: oracle/rescue_py.py against oracle/qmo_mem.c on the hand-built pairs of reggen.rescue_cases
RESCUE_PES = {"wide": dict(), "window 4096 / 4097": dict(low=100, high=100 + 4096 - 150),
              "one orientation": dict(failed=(1, 0, 1, 1)), "narrow": dict(low=10, high=25)}


def rescue_both(g, ref, max_len, pes_kw):
    cs, pes = reggen.rescue_cases(g, max_len, pes=reggen.rescue_pes(**pes_kw))
    codes, lens, regs, n_regs = reggen.region_arrays(cs)
    o = qmo_py.default_opt()
    after, n_after = regs.copy(), n_regs.copy()
    stats = qmo_py.mate_rescue(ref, codes, lens, after, n_after, pes, opt=o)
    return cs, pes, (codes, lens, regs, n_regs), (after, n_after, stats)


@pytest.mark.parametrize("name", list(RESCUE_PES))
@pytest.mark.parametrize("max_len", [150, 256, 512])
def test_mate_rescue_cases_equal_an_independent_restatement(genome, ref, name, max_len):
    from oracle import rescue_py
    g = genome
    cs, pes, (codes, lens, regs, n_regs), (after, n_after, stats) = rescue_both(g, ref, max_len, RESCUE_PES[name])
    o = qmo_py.default_opt()
    dbl = reggen.doubled(g)
    offs = [int(x) for x in g.offs]
    fields = ("rid", "score", "csub", "qb", "qe", "rb", "re")
    counters = dict(sw=0, cells=0)
    n_new = n_csub = 0
    for p in range(len(lens) // 2):
        hits = [[{f: int(r[f]) for f in fields} for r in regs[2 * p + m][:int(n_regs[2 * p + m])]] for m in (0, 1)]
        got = rescue_py.rescue_pair(dbl, g.l_pac, offs, g.lens, pes, hits, [codes[2 * p, :lens[2 * p]], codes[2 * p + 1, :lens[2 * p + 1]]],
                                    o, counters)
        for m in (0, 1):
            want = [{f: int(r[f]) for f in fields} for r in after[2 * p + m][:int(n_after[2 * p + m])]]
            assert got[m] == want, (p, m, cs.tags[2 * p], got[m], want)
            n_new += len(want) > len(hits[m])
            n_csub += any(h["csub"] > 0 for h in want)
    assert (counters["sw"], counters["cells"]) == stats and n_new > 10, (counters, stats, n_new)
    # what the cases reach: second hits, best scores around min_seed_len * a, windows of 4,096 / 4,097 bases (151-base mates) and
    # windows shorter than min_seed_len (neither of the last two is searched)
    sc, win = collections.Counter(counters["scores"]), collections.Counter(counters["windows"])
    minsc = o.min_seed_len * o.a
    if name != "narrow":
        assert n_csub > 0
    if name == "wide":
        assert all(sc[minsc + d] for d in (-1, 0, 1)), sc
    if name == "window 4096 / 4097" and max_len > 150:
        assert win[4096] and win[4097], win
    if name == "narrow":
        assert any(0 <= x < o.min_seed_len for x in win), win
