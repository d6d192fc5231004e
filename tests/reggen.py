"""Hand-built reads and regions for the parity tests of the CIGAR stage (mem_reg2aln -> bwa_gen_cigar2 -> ksw_global2) and of
mate rescue (mem_matesw -> ksw_align2): a genome of three contigs (recgen.Genome), reads cut from it with planned edits, one
qm_reg per read whose fields follow the edit, and a Python restatement of how pair.cu routes a read to its kernel, used to
show which kernel each family reaches.

A read is cut from the forward strand along `ops` (M / I / D), gets substitutions and N's at planned query positions and random
soft-clipped bases at both ends; a reverse read is the reverse complement of all that.  Its region spans exactly the cut:
rb / re in bwa's doubled coordinates, qb / qe inside the clips, truesc the score of the planned path unless given."""
import numpy as np

from oracle import qmo_py
from oracle.qmo_py import REG_DTYPE, MAX_REGS
from tests import recgen

M, I, D = 0, 1, 2
# contig 0: room for 4,096-base rescue windows; contig 1: short, windows clipped at both of its ends; contig 2: a planted tandem
# copy (TANDEM: bases [src, src + n) again at dst) and a short-period repeat (PERIODIC: [beg, end) with period p)
CONTIG_LENS = (9000, 160, 3000)
TANDEM = (600, 1100, 300)
PERIODIC = (2000, 2400, 70)
HOMOPOLYMER = (8600, 8750)                  # contig 0: A's; a mate of A's logs a run of consecutive rows of equal maxima
SCHEMES = {
    "default": dict(a=1, b=4, o_del=6, e_del=1, o_ins=6, e_ins=1),
    "a2": dict(a=2, b=5, o_del=5, e_del=2, o_ins=7, e_ins=1),
    # large penalties: a two-base mismatch pair already outweighs a one-base deletion plus insertion (cig_gain_cap 1)
    "harsh": dict(a=1, b=60, o_del=40, e_del=12, o_ins=40, e_ins=12),
    # larger still: the DP values of a 400 - 512-base read with mismatch clusters fall below -20,000, out of 16-bit reach
    "extreme": dict(a=1, b=100, o_del=100, e_del=60, o_ins=100, e_ins=60),
}
_COMP = np.array([3, 2, 1, 0, 4], np.uint8)


def genome(seed=23):
    g = recgen.Genome(seed, CONTIG_LENS)
    o2 = int(g.offs[2])
    s, d, n = TANDEM
    g.codes[o2 + d:o2 + d + n] = g.codes[o2 + s:o2 + s + n]
    b, e, p = PERIODIC
    for x in range(b + p, e):
        g.codes[o2 + x] = g.codes[o2 + x - p]
    g.codes[HOMOPOLYMER[0]:HOMOPOLYMER[1]] = 0
    return g


def doubled(g):
    fwd = np.asarray(g.codes, np.uint8)
    return np.concatenate([fwd, _COMP[fwd[::-1]]])


def set_opt(o, scheme, w=100, flags=qmo_py.F_NO_RESCUE):
    """o (the oracle's or the library's Opt) with the scheme's scores, band w and flags -> o"""
    for k, v in dict(SCHEMES[scheme], w=w, flags=flags).items():
        setattr(o, k, v)
    return o


def path_score(sc, q, t, ops):
    """score of the alignment `ops` of q against t (both in the same orientation)"""
    s, i, k = 0, 0, 0
    for op, ln in ops:
        if op == M:
            s += sum(-1 if (x > 3 or y > 3) else sc["a"] if x == y else -sc["b"] for x, y in zip(q[k:k + ln], t[i:i + ln]))
            i += ln
            k += ln
        elif op == I:
            s -= sc["o_ins"] + sc["e_ins"] * ln
            k += ln
        else:
            s -= sc["o_del"] + sc["e_del"] * ln
            i += ln
    return s


class Cases:
    """reads with one region each (or none); read 2i and 2i + 1 are a pair"""

    def __init__(self, g, sc, seed=0, w=100):
        self.g, self.sc, self.w = g, sc, w
        self.rng = np.random.default_rng(seed)
        self.reads, self.regs, self.tags = [], [], []

    def add(self, rid, pos, ops, rev=False, subs=(), ns=(), clip=(0, 0), truesc=None, dsc=0, w=None, tag=""):
        """one read cut at forward position `pos` of contig `rid` along ops; subs / ns: positions in the aligned part of the
        forward-strand read; clip: random bases before / after it on the forward strand.  -> index of the read"""
        g, rng = self.g, self.rng
        f0 = int(g.offs[rid]) + pos
        span = sum(ln for op, ln in ops if op != I)
        assert pos >= 0 and pos + span <= int(g.lens[rid]), (rid, pos, span)
        t = g.codes[f0:f0 + span]
        q, i = [], 0
        for op, ln in ops:
            if op == M:
                q.extend(t[i:i + ln])
                i += ln
            elif op == I:
                q.extend(rng.integers(0, 4, ln))
            else:
                i += ln
        q = np.array(q, np.uint8)
        for p in subs:
            q[p] = (q[p] + rng.integers(1, 4)) % 4
        for p in ns:
            q[p] = 4
        if truesc is None:
            truesc = path_score(self.sc, q, t, ops) + dsc
        full = np.concatenate([rng.integers(0, 4, clip[0]), q, rng.integers(0, 4, clip[1])]).astype(np.uint8)
        l_pac = g.l_pac
        if rev:
            full = _COMP[full[::-1]]
            qb, qe, rb, re = clip[1], clip[1] + len(q), 2 * l_pac - (f0 + span), 2 * l_pac - f0
        else:
            qb, qe, rb, re = clip[0], clip[0] + len(q), f0, f0 + span
        r = np.zeros((), REG_DTYPE)
        r["rb"], r["re"], r["qb"], r["qe"], r["rid"] = rb, re, qb, qe, rid
        r["score"] = max(int(truesc), 30 * self.sc["a"], 1)
        r["truesc"], r["w"] = truesc, self.w if w is None else w
        r["secondary"], r["sub"], r["csub"], r["sub_n"] = -1, 0, 0, 0
        r["seedcov"], r["seedlen0"] = min(len(q), span) >> 1, min(len(q), 31)
        self.reads.append(full)
        self.regs.append(r)
        self.tags.append(tag)
        return len(self.reads) - 1

    def add_unmapped(self, L, tag="no region"):
        self.reads.append(self.rng.integers(0, 4, L).astype(np.uint8))
        self.regs.append(None)
        self.tags.append(tag)
        return len(self.reads) - 1

    def tune(self, r, o, dbl, pred, lo=-3000, hi=None, pre=None):
        """the highest truesc (from hi down) at which route() of read r (the last one) satisfies pred; the read keeps it.  A read
        no truesc steers there (a band the scheme cannot reach) is dropped -> None.  pre: a quick filter on route(full=False)"""
        reg = self.regs[r]
        hi = int(reg["qe"] - reg["qb"]) * o.a + 50 if hi is None else hi
        for ts in range(hi, lo, -1):
            reg["truesc"] = ts
            if pre is not None and not pre(route(o, dbl, self.g.l_pac, self.reads[r], reg, full=False)):
                continue
            if pred(route(o, dbl, self.g.l_pac, self.reads[r], reg)):
                reg["score"] = max(ts, 30 * o.a, 1)
                return r
        self.drop()

    def drop(self):
        self.reads.pop(); self.regs.pop(); self.tags.pop()

    def arrays(self, stride=None, seed=0):
        """-> codes [n, stride], lens, regs [n, MAX_REGS], n_regs; an odd read count gets a read without a region.  Bytes past a
        read's length are junk (N's included)."""
        if len(self.reads) % 2:
            self.add_unmapped(5)
        lens = np.array([len(s) for s in self.reads], np.int32)
        stride = stride or int(lens.max())
        rng = np.random.default_rng(seed)
        codes = rng.integers(0, 5, (len(lens), stride)).astype(np.uint8)
        for r, s in enumerate(self.reads):
            codes[r, :len(s)] = s
        regs = np.zeros((len(lens), MAX_REGS), REG_DTYPE)
        n_regs = np.zeros(len(lens), np.int32)
        for r, h in enumerate(self.regs):
            if h is not None:
                regs[r, 0] = h
                n_regs[r] = 1
        return codes, lens, regs, n_regs


def failed_pes():
    pes = np.zeros(4, qmo_py.PESTAT_DTYPE)
    pes["failed"] = 1
    return pes


# ---------------------------------------------------------------------------------------------------------------------
# pair.cu's router, restated: which list a read's CIGAR task lands in.  Used only to show coverage.
WMAX = {3: 15, 4: 31, 5: 63}
SLAB_WORDS, DIR_SMEM, CIG16_BOUND = 4096, 14 * 1024, 12000


def infer_bw(l1, l2, score, a, q, r):
    if l1 == l2 and l1 * a - score < (q + r - a) << 1:
        return 0
    return max(int((min(l1, l2) * a - score - q) / r + 2.), abs(l1 - l2))


def cig_gain_cap(o, n_low):
    x = (o.a + max(o.b, 1)) * n_low - o.a - o.o_ins - o.o_del
    es = o.e_ins + o.e_del
    return 0 if x <= es else (x - 1) // es


def cig_band(o, w2, lq, rlen):
    w2 = min(w2, o.w << 2)
    max_gap = max(int((((lq + 1) >> 1) * o.a - o.o_ins) / o.e_ins + 1.), int((((lq + 1) >> 1) * o.a - o.o_del) / o.e_del + 1.), 1)
    return max(min((max_gap + abs(rlen - lq) + 1) >> 1, w2), abs(rlen - lq) + 3)


def cig_fits16(o, lq, rlen):
    return max(o.b, 1) * min(lq, rlen) + max(o.o_del + o.e_del * rlen, o.o_ins + o.e_ins * lq) + \
        max(o.o_del + o.e_del, o.o_ins + o.e_ins) <= CIG16_BOUND


def cig_class(o, lq, rlen, w2, wcap):
    if not cig_fits16(o, lq, rlen):
        return 6
    w = cig_band(o, w2, lq, rlen)
    if lq != rlen:
        return 3 if w <= 15 else 4 if w <= 31 else 5 if w <= 63 else 6
    w = min(w, wcap)
    return 0 if w <= 15 else 1 if w <= 23 else 2 if w <= 35 else 6


def task_seqs(dbl, l_pac, read, reg):
    q, t = read[reg["qb"]:reg["qe"]], dbl[reg["rb"]:reg["re"]]
    return (q[::-1], t[::-1]) if reg["rb"] >= l_pac else (q, t)


def route(o, dbl, l_pac, read, reg, full=True):
    """-> dict(list = None (no DP) or 0..8, first = the list of pair_decide_kernel, band = its band, tries = [(w, dir bytes of the
    warp kernel)], n_low)"""
    q, t = task_seqs(dbl, l_pac, read, reg)
    lq, rlen = len(q), len(t)
    w2 = max(infer_bw(lq, rlen, int(reg["truesc"]), o.a, o.o_del, o.e_del), infer_bw(lq, rlen, int(reg["truesc"]), o.a, o.o_ins, o.e_ins))
    if w2 > o.w:
        w2 = min(w2, int(reg["w"]))
    out = dict(list=None, first=None, band=None, tries=[], n_low=None, lq=lq, rlen=rlen, fits16=cig_fits16(o, lq, rlen))
    wcap = 1 << 20
    if lq == rlen:
        n_low = int(((q != t) | (q > 3)).sum())
        out["n_low"] = n_low
        wcap = cig_gain_cap(o, n_low)
        if w2 == 0 or wcap == 0:
            return out
    c = out["first"] = out["list"] = cig_class(o, lq, rlen, w2, wcap)
    out["band"] = min(cig_band(o, w2, lq, rlen), wcap)
    out["w0"] = cig_band(o, w2, lq, rlen)          # the band of the warp kernel's first try
    if not full:
        return out
    if c <= 2:
        us = sum(-1 if (x > 3 or y > 3) else o.a if x == y else -o.b for x, y in zip(q, t))
        if qmo_py.ksw_global2(q, t, out["band"], o, max_cigar=4096)[0] != us:
            out["list"] = 7
    elif c <= 5:
        out["trace"] = _tries(o, q, t, w2, reg["truesc"])
        if lq > 500 or rlen > 1000 or any(w > WMAX[c] or ((min(lq, 2 * w + 1) + 7) >> 3) * rlen > SLAB_WORDS for w in out["trace"]):
            out["list"] = 8
    if out["list"] >= 6:
        out["tries"] = [(w, min(lq, 2 * w + 1) * rlen) for w in _tries(o, q, t, w2, reg["truesc"])]
    return out


def _tries(o, q, t, w2, truesc):
    """the bands of mem_reg2aln's tries (up to three, w2 doubled while the score stays below truesc - a and changes)"""
    out, last = [], None
    while True:
        w2 = min(w2, o.w << 2)
        w = cig_band(o, w2, len(q), len(t))
        out.append(w)
        s = qmo_py.ksw_global2(q, t, w, o, max_cigar=4096)[0]
        if s == last or w2 == o.w << 2 or len(out) == 3 or s >= int(truesc) - o.a:
            return out
        last, w2 = s, w2 << 1


# ---------------------------------------------------------------------------------------------------------------------
# CIGAR case families
def _scatter(rng, L, n, lo=0):
    return sorted(rng.choice(np.arange(lo, L), size=min(n, L - lo), replace=False).tolist())


def cigar_cases(g, scheme, w=100, seed=1, long_refs=True):
    """every family of CIGAR cases for one scheme and band; tags name the family"""
    sc = SCHEMES[scheme]
    o = set_opt(qmo_py.default_opt(), scheme, w)
    dbl = doubled(g)
    cs = Cases(g, sc, seed, w)
    rng = cs.rng
    cl = [int(x) for x in g.lens]

    def band_is(b):
        return lambda r: r["band"] == b

    # class boundaries, equal lengths (a compensating deletion / insertion and scattered mismatches: cig_gain_cap stays wide)
    for b in (15, 16, 23, 24, 35, 36):
        for rev in (False, True):
            L = 160 if sc["a"] == 1 else 150
            for ops in ([(M, 50), (D, 2), (M, 40), (I, 2), (M, L - 92)], [(M, L)]):
                r = cs.add(0, 100 + 37 * b, ops, rev, subs=_scatter(rng, L, 14 + 3 * len(ops)), tag=f"equal-length band {b}")
                cs.tune(r, o, dbl, band_is(b), pre=lambda x: x["band"] == b)
    # a deletion of k bases: the band is at least k + 3 in every scheme
    for k in (12, 13, 28, 29, 60, 61):
        for rev in (False, True):
            cs.add(0, 4000 + 50 * k, [(M, 100), (D, k), (M, 100)], rev, subs=_scatter(rng, 200, 6), tag=f"deletion of {k}")
    # class boundaries, length difference
    for b in (15, 16, 31, 32, 63, 64):
        for rev in (False, True):
            ops = [(M, 130), (D, 4), (M, 126)]
            r = cs.add(0, 2000 + 41 * b, ops, rev, subs=_scatter(rng, 256, 10), tag=f"length-difference band {b}")
            cs.tune(r, o, dbl, band_is(b), pre=lambda x: x["band"] == b)
    # query lengths at the warp kernel's templates and the thread kernels' lq <= 500
    for L in (160, 161, 256, 257, 500, 501, 511):
        for rev in (False, True):
            h = L // 2
            cs.add(0, 3000 + 3 * L, [(M, h), (D, 3), (M, L - h)], rev, subs=_scatter(rng, L, L // 25), tag=f"lq {L} deletion")
            r = cs.add(2, 100 + L, [(M, h - 20), (D, 2), (M, 40), (I, 2), (M, L - h - 22)], rev, subs=_scatter(rng, L, L // 10),
                       tag=f"lq {L} equal length")
            cs.tune(r, o, dbl, lambda x: x["list"] == 6 or x["list"] == 7, pre=lambda x: x["first"] in (0, 1, 2, 6))
    # reference spans around 1,000 (the thread kernels' rlen <= 1000) and direction matrices around the warp kernel's 14 KB of
    # shared memory
    if long_refs:
        for k in (550, 551):
            cs.add(0, 5000, [(M, 225), (D, k), (M, 225)], k % 2 == 1, tag=f"rlen {450 + k}")
    if sc["a"] == 1 and sc["o_ins"] + sc["e_ins"] < 20:
        for wb in (39, 40):
            for rev in (False, True):
                r = cs.add(0, 6000 + wb, [(M, 60), (D, 2), (M, 60), (I, 2), (M, 58)], rev, subs=_scatter(rng, 180, 30),
                           tag=f"direction matrix {'under' if wb == 39 else 'over'} 14 KB")
                cs.tune(r, o, dbl, lambda x: x["list"] == 6 and x["tries"][0][0] == wb, pre=lambda x: x.get("w0") == wb)
    # retries: truesc above anything a band reaches (all three tries), tries that do not change the score, second traceback try
    # beyond the thread kernel's band
    for rev in (False, True):
        cs.add(2, 200, [(M, 60), (D, 5), (M, 60)], rev, subs=_scatter(rng, 120, 6), dsc=80 * sc["a"], tag="retry: truesc unreachable")
        cs.add(2, 400, [(M, 60), (D, 1), (M, 60)], rev, subs=_scatter(rng, 120, 2), dsc=5 * sc["a"], tag="retry: score unchanged")
        for c in (3, 4, 5):
            L = {3: 90, 4: 200, 5: 300}[c]
            r = cs.add(0, 7000 + 100 * c, [(M, L // 2), (D, 3), (M, L // 2)], rev, subs=_scatter(rng, L, L // 8),
                       tag=f"retry: trace kernel {c} passes on")
            cs.tune(r, o, dbl, lambda x: x["first"] == c and x["list"] == 8, hi=3 * L * sc["a"], pre=lambda x: x["first"] == c)
    # ... with a second try exactly one above the kernel's band (its ring of slots would not hold it), on a path that runs along
    # that band's outermost diagonal: a deletion (insertion) of wmax + 1 and an insertion (deletion) of 4 leave a length
    # difference of wmax - 3, so the first band is wmax; the query length makes the second exactly wmax + 1
    for c in (3, 4, 5) if w >= 64 else ():        # (a narrow -w caps the second band below these)
        wm = WMAX[c]
        for first_del in (True, False):
            for rev in (False, True):
                big, small = (D, I) if first_del else (I, D)
                n_kept = 0
                for lq in range(20, 400):
                    m = lq - (4 if first_del else wm + 1)
                    if m < 30 or cig_band(o, 1 << 20, lq, lq + (wm - 3 if first_del else 3 - wm)) != wm + 1:
                        continue
                    ops = [(M, m // 3), (big, wm + 1), (M, m // 3), (small, 4), (M, m - 2 * (m // 3))]
                    r = cs.add(0, 7500 + 20 * c, ops, rev, subs=_scatter(rng, lq, lq // 12),
                               tag=f"retry: trace kernel {c}, second band {wm + 1} on its edge")
                    if cs.tune(r, o, dbl, lambda x: x["first"] == c and wm + 1 in x.get("trace", ()), hi=3 * lq * sc["a"],
                               pre=lambda x: x["first"] == c) is not None:
                        n_kept += 1
                        if n_kept == 2:
                            break
    # the no-DP path: every alignment mod 4 of query and reference start, lengths 1 - 7 and not multiples of 4, N's, both strands,
    # the genome's first and last base
    for L in (1, 2, 3, 4, 5, 6, 7, 9, 13, 31, 33, 150):
        for qm in range(4):
            for rm in range(4):
                rev = (qm + rm + L) % 2 == 1
                subs = _scatter(rng, L, 1) if L > 8 and rm == 1 else ()
                ns = [L // 2] if L > 4 and qm == 2 else ()
                cs.add(0, 8 + rm + 8 * L, [(M, L)], rev, subs=subs, ns=ns, clip=(qm, 3 - qm), tag=f"no DP: {L} bases")
    for rev in (False, True):
        cs.add(0, 0, [(M, 37)], rev, clip=(2, 1), tag="no DP: genome start")
        cs.add(2, cl[2] - 41, [(M, 41)], rev, subs=[3], clip=(1, 0), tag="no DP: genome end")
        cs.add(1, 0, [(M, 30), (D, 2), (M, 40)], rev, subs=[50], tag="contig start")
        cs.add(1, cl[1] - 75, [(M, 30), (I, 2), (M, 43)], rev, subs=[10], clip=(3, 4), tag="contig end")
    # records: soft clips, leading / trailing deletions to squeeze out, 19 and 20 operations
    for rev in (False, True):
        cs.add(0, 300, [(M, 40), (D, 2), (M, 60)], rev, subs=[5], clip=(7, 12), tag="clips both ends")
        for ops in ([(D, 3), (M, 80)], [(M, 80), (D, 3)], [(D, 2), (M, 40), (I, 1), (M, 40)], [(M, 40), (D, 1), (M, 40), (D, 4)]):
            cs.add(0, 500, ops, rev, clip=(4, 2), tag="squeeze")
        for n_gap, tail in ((8, 0), (9, 0), (9, 3), (10, 0)):
            ops = [(M, 18)]
            for k in range(n_gap):
                ops += [(D if k % 2 == 0 else I, 2), (M, 18)]
            if tail:
                ops.append((D, tail))
            cs.add(2, 2500 if rev else 0, ops, rev, clip=(2, 3), tag=f"{len(ops)} operations")
    # cig_gain_cap edges: equal lengths, a deletion and an insertion d apart, mismatches placed so that n_low sits where the cap
    # changes; the planned gapped path beats, ties or loses to the ungapped one by 0 or 1
    want = {(nl, dd): 2 for nl in range(2, 7) for dd in (-1, 0, 1)}
    for _ in range(4000):
        if not any(want.values()):
            break
        L, k, d = int(rng.integers(24, 90)), int(rng.integers(1, 4)), int(rng.integers(0, 5))
        x = int(rng.integers(5, L - d - 2 * k - 4))
        ops = [(M, x), (D, k), (M, d), (I, k), (M, L - x - d - k)] if rng.random() < 0.5 else \
              [(M, x), (I, k), (M, d), (D, k), (M, L - x - d - k)]
        subs = _scatter(rng, L, int(rng.integers(0, 3)))
        pos = int(rng.integers(0, cl[0] - L - 10))
        rev = bool(rng.random() < 0.5)
        r = cs.add(0, pos, ops, rev, subs=subs, truesc=L * sc["a"] - 30 * sc["a"], tag="gain cap")
        q, t = task_seqs(dbl, g.l_pac, cs.reads[r], cs.regs[r])
        nl = int(((q != t) | (q > 3)).sum())
        us = sum(sc["a"] if x_ == y_ else -sc["b"] for x_, y_ in zip(q, t))
        planned = path_score(sc, cs.reads[r][cs.regs[r]["qb"]:cs.regs[r]["qe"]] if not rev else _COMP[cs.reads[r][::-1]],
                             g.codes[g.offs[0] + pos:g.offs[0] + pos + L], ops)
        key = (nl, planned - us)
        if want.get(key, 0) > 0:
            want[key] -= 1
        else:
            cs.drop()
    # ... and the tightest cap: a one-base deletion and a one-base insertion next to each other (under "harsh" n_low = 2 gives
    # cap 1, and the gapped path wins)
    for d in (0, 1, 2):
        for j in range(8):
            L = 60 + 7 * j
            x = 20 + j
            cs.add(0, 6500 + 50 * j + 10 * d, [(M, x), (D, 1), (M, d), (I, 1), (M, L - x - d - 1)], j % 2 == 1, dsc=-150 * sc["a"],
                   tag="gain cap: 1-base gaps")
    # the 16-bit cells: 400 - 512-base reads with four in five bases substituted (under "extreme" their DP values fall below
    # -20,000, where 16-bit cells with -20000 as minus infinity go wrong)
    if scheme == "extreme":
        for L in (400, 450, 500, 512):
            for rev in (False, True):
                subs = _scatter(rng, L, 4 * L // 5)
                cs.add(2, 150, [(M, L // 2), (D, 3), (M, L - L // 2)], rev, subs=subs, tag=f"16-bit: {L} bases, length difference")
                cs.add(0, 1500 + L, [(M, L // 2 - 30), (D, 3), (M, 60), (I, 3), (M, L - L // 2 - 33)], rev, subs=subs,
                       tag=f"16-bit: {L} bases, equal length")
    # random gapped reads of every length up to 150
    for _ in range(60):
        L = int(rng.integers(20, 151))
        ops, q_ = [], 0
        while q_ < L:
            m = min(int(rng.integers(5, 40)), L - q_)
            ops.append((M, m)); q_ += m
            if q_ < L - 5 and rng.random() < 0.5:
                k = int(rng.integers(1, 6))
                if rng.random() < 0.5:
                    ops.append((D, k))
                else:
                    k = min(k, L - q_ - 1); ops.append((I, k)); q_ += k
        span = sum(ln for op, ln in ops if op != I)
        cs.add(0, int(rng.integers(0, cl[0] - span)), ops, bool(rng.random() < 0.5), subs=_scatter(rng, L, int(rng.integers(0, L // 10 + 1))),
               clip=(int(rng.integers(0, 6)), int(rng.integers(0, 6))), dsc=int(rng.integers(-10, 10)), tag="random")
    # the longest read last: it ends at the batch's last byte (stride == length)
    cs.add(0, 8000, [(M, 256), (D, 1), (M, 256)], False, subs=_scatter(rng, 512, 12), tag="last read, 512 bases")
    return cs


# ---------------------------------------------------------------------------------------------------------------------
# mate rescue cases: pairs in which end 0 has its regions (the anchors) and end 1 a few or none
def rescue_pes(low=150, high=650, failed=(0, 0, 0, 0)):
    pes = np.zeros(4, qmo_py.PESTAT_DTYPE)
    pes["low"], pes["high"], pes["failed"] = low, high, failed
    pes["avg"], pes["std"] = (low + high) / 2, (high - low) / 8
    return pes


def _mate(cs, rid, pos, L, rev, subs=(), ns=(), tag=""):
    """a read cut at (rid, pos) whose region is thrown away again: its sequence is the mate"""
    r = cs.add(rid, pos, [(M, L)], rev, subs=subs, ns=ns, tag=tag)
    cs.regs[r] = None
    return r


def rescue_cases(g, max_len, seed=3, pes=None):
    """pairs for one stride class (mates of at most max_len bases); pes: the models the windows come from"""
    pes = rescue_pes() if pes is None else pes
    sc = SCHEMES["default"]
    cs = Cases(g, sc, seed)
    rng = cs.rng
    cl = [int(x) for x in g.lens]
    lens = sorted({1, 2, 19, 31, 33, 64, 100, 150, 151, 160, max_len - 1, max_len} | set(int(x) for x in rng.integers(20, max_len + 1, 6)))
    lens = [L for L in lens if L <= max_len]
    # every orientation: anchor on either strand, mate on either strand at a distance in or out of the model, one or two of its
    # bases off, N's in some mates
    for L in lens:
        for _ in range(6):
            A = min(max(L, 40), 150)
            p0 = int(rng.integers(700, cl[0] - 1500))
            ra, rm = bool(rng.random() < 0.5), bool(rng.random() < 0.5)
            d = int(rng.integers(int(pes["low"].min()) - 100, int(pes["high"].max()) + 100))
            cs.add(0, p0, [(M, A)], ra, tag=f"anchor for a {L}-base mate")
            pm = min(max(p0 + (d if rng.random() < 0.5 else -d), 0), cl[0] - L)
            ns = [int(rng.integers(0, L))] if L > 5 and rng.random() < 0.3 else ()
            _mate(cs, 0, pm, L, rm, subs=_scatter(rng, L, int(rng.integers(0, 3))) if L > 10 else (), ns=ns, tag=f"mate of {L}")
    # windows clipped at contig ends (the short contig: both ends) and at the strand boundary (end of the last contig)
    for rid, pos in ((1, 0), (1, cl[1] - 40), (0, 0), (0, cl[0] - 40), (2, cl[2] - 40), (2, 0)):
        for ra in (False, True):
            cs.add(rid, pos, [(M, 40)], ra, tag="anchor at a contig end")
            L = min(max_len, 30)
            _mate(cs, rid, min(max(pos + (60 if pos == 0 else -60), 0), cl[rid] - L), L, not ra, tag="mate near a contig end")
    # the tandem copy and the short-period repeat: a second hit of the mate in the same window (score2 / te2 -> csub), further
    # than and closer than `score` rows from the best one
    s, dcopy, n = TANDEM
    b, e, p = PERIODIC
    for L in (40, 100, min(max_len, 130)):
        for ra in (False, True):
            cs.add(2, s - 250, [(M, 50)], ra, tag="anchor before a tandem copy")
            _mate(cs, 2, s + 20, L, not ra, tag="mate with a tandem copy")
            cs.add(2, b - 300, [(M, 50)], ra, tag="anchor before a periodic repeat")
            _mate(cs, 2, b + 10, min(L, e - b - 20), not ra, tag="mate in a periodic repeat")
    # best score around min_seed_len * a (31): a random mate holding 29 - 33 bases of the window
    for k in (29, 30, 31, 32, 33):
        for ra in (False, True):
            L = min(max_len, 60)
            p0 = int(rng.integers(1000, cl[0] - 2000))
            cs.add(0, p0, [(M, 60)], ra, tag="anchor for a barely found mate")
            m = _mate(cs, 0, p0 + 300, L, not ra, tag=f"mate with {k} bases of the window")
            keep = cs.reads[m][10:10 + k].copy()
            cs.reads[m] = rng.integers(0, 4, L).astype(np.uint8)
            cs.reads[m][10:10 + k] = keep
    # a mate of A's against the homopolymer run: the rows after the best one keep its maximum, then fall.  Consecutive logged rows
    # merge into one entry that moves on only when the maximum rises, so a new entry opens every other row; at these lengths the
    # best entry outside the exclusion zone (score2 -> csub) depends on that rule
    for L in (75, 79, 92, 96):
        cs.add(0, HOMOPOLYMER[0] - 300, [(M, 50)], False, tag="anchor before a homopolymer")
        m = _mate(cs, 0, HOMOPOLYMER[0], L, True, tag="mate of A's")
        cs.reads[m][:] = 3                         # T's as sequenced: searched as the reverse complement
    # several anchors within pen_unpaired, and an anchor whose mate already has a region at a proper distance
    for ra in (False, True):
        p0 = int(rng.integers(1000, cl[0] - 2000))
        a = cs.add(0, p0, [(M, 80)], ra, tag="anchors within pen_unpaired")
        extra = [cs.regs[a].copy() for _ in range(2)]
        for j, x in enumerate(extra):
            x["rb"] += 700 * (j + 1) * (1 if not ra else -1)
            x["re"] += 700 * (j + 1) * (1 if not ra else -1)
            x["score"] -= 5 + 8 * j
        cs.regs[a] = [cs.regs[a]] + extra
        _mate(cs, 0, p0 + 400, 70, not ra, tag="mate of several anchors")
        cs.add(0, p0, [(M, 80)], ra, tag="anchor with a served mate")
        cs.add(0, p0 + 300 if not ra else p0 - 300, [(M, 70)], not ra, tag="mate already served")
    return cs, pes


def region_arrays(cs, stride=None):
    """Cases.arrays for reads that may carry a list of regions"""
    multi = {k: h for k, h in enumerate(cs.regs) if isinstance(h, list)}
    for k in multi:
        cs.regs[k] = None
    codes, lens, regs, n_regs = cs.arrays(stride)
    for k, hs in multi.items():
        hs = sorted(hs, key=lambda h: -int(h["score"]))
        for j, h in enumerate(hs):
            regs[k, j] = h
        n_regs[k] = len(hs)
        cs.regs[k] = hs
    return codes, lens, regs, n_regs
