"""Hand-built repetitive genomes and reads for the parity tests of the read-level front end (seeding, chaining, the extension
state machine), and a brute force of the hash seeder's contract (DESIGN.md 5.1) to hold both the oracle and the kernels against.

Every genome is a `Genome` (codes 0..3 of the concatenated contigs, contig lengths), which Context.index and qmo_py.Ref both take,
plus the forward intervals reads are preferably cut from (`hot`).  Everything is deterministic from the seed.  The families:

  unique      random background only: the lone-hit path, filter misses behind every mismatch
  disp*       a 200-base unit in 2..5 copies in a given strand mix ('+' as is, '-' reverse-complemented), exact or diverged by one
              substitution per ~40 bases per copy: the 2..4-hit tracked path, and 5 copies, one past it
  inv*        a unit, a spacer of 0, 1 or 5 bases, the unit's reverse complement: one hit per strand; palindromic k-mers at even k
  occ*        a 40-base unit in a+b copies (a as is, b reverse-complemented): per-strand counts of 31, 32 and 33 around the cap
  tan*        tandem arrays of period 1 .. 45, exact or 1 % diverged: runs of hits that break and restart, 64 seeds, 16 regions
  ctg         16 contigs, some of length k - 1, k, k + 1 and 32 m +- 1, repeat copies at position 0 and at l_pac, a copy across a
              contig boundary

Reads come from both strands, are cut across contig boundaries as they fall, and carry one of the edit plans of EDITS; the row
padding past a read's length holds random bases (never N), so a kernel that reads past the length is seen."""
import numpy as np

MAX_SEEDS, OCC_CAP = 64, 32
_COMP = np.array([3, 2, 1, 0, 4], np.uint8)
READ_LENS = (0, 1, 31, 33, 63, 65, 127, 129, 150, 250, 400, 512)        # with k - 1, k, k + 1 added per k
EDITS = ("clean", "errors", "planned_subs", "n_edges", "n_run", "all_n", "chimera", "errors_n")
DISP_MIXES = ("++", "+-", "+++", "+-+", "++++", "+--+", "+++++", "++-+-")
OCC_SPLITS = ((31, 0), (32, 0), (33, 0), (16, 16), (20, 20), (33, 1))
TAN_PERIODS = (1, 2, 3, 7, 30, 31, 32, 33, 45)
MAX_OCCS = (1, 2, 3, 4, 5, 32, 33, 500)


def rc(a):
    return _COMP[np.asarray(a, np.uint8)[::-1]]


class Genome:
    def __init__(self, name, contigs, hot=()):
        self.name = name
        self.lens = np.array([len(c) for c in contigs], np.int64)
        self.offs = np.concatenate([[0], np.cumsum(self.lens)]).astype(np.int64)
        self.codes = np.concatenate(contigs).astype(np.uint8)
        self.l_pac = int(self.lens.sum())
        self.hot = list(hot)                     # forward intervals [b, e) that reads favour

    def doubled(self):
        return np.concatenate([self.codes, rc(self.codes)])


def _mutate(rng, a, rate):
    a = np.array(a, np.uint8)
    for j in np.flatnonzero(rng.random(len(a)) < rate):
        a[j] = (a[j] + 1 + rng.integers(0, 3)) % 4
    return a


def _build(name, parts, seed):
    """parts: list of arrays; a tuple ('hot', array) marks an interval reads favour"""
    seq, hot, at = [], [], 0
    for p in parts:
        if isinstance(p, tuple):
            p = p[1]
            hot.append((at, at + len(p)))
        seq.append(np.asarray(p, np.uint8))
        at += len(p)
    return Genome(name, [np.concatenate(seq)], hot)


def unique(seed=1):
    rng = np.random.default_rng(seed)
    return Genome("unique", [rng.integers(0, 4, 2500), rng.integers(0, 4, 1200)], [(0, 3700)])


def dispersed(mix, diverged, seed=2):
    rng = np.random.default_rng(seed + 97 * len(mix))
    unit = rng.integers(0, 4, 200).astype(np.uint8)
    parts = [rng.integers(0, 4, 300)]
    for s in mix:
        u = unit if s == "+" else rc(unit)
        parts += [("hot", _mutate(rng, u, 1 / 40) if diverged else u), rng.integers(0, 4, 300)]
    return _build(f"disp{mix}{'d' if diverged else 'x'}", parts, seed)


def inverted(spacer, seed=3):
    rng = np.random.default_rng(seed + spacer)
    unit = rng.integers(0, 4, 150).astype(np.uint8)
    arm = np.concatenate([unit, rng.integers(0, 4, spacer), rc(unit)]).astype(np.uint8)
    return _build(f"inv{spacer}", [rng.integers(0, 4, 400), ("hot", arm), rng.integers(0, 4, 400)], seed)


def occurrences(n_fwd, n_rev, seed=4):
    rng = np.random.default_rng(seed + n_fwd * 64 + n_rev)
    unit = rng.integers(0, 4, 40).astype(np.uint8)
    arr = []
    for j in range(n_fwd + n_rev):
        arr += [unit if j < n_fwd else rc(unit), rng.integers(0, 4, 5)]
    return _build(f"occ{n_fwd}+{n_rev}", [rng.integers(0, 4, 300), ("hot", np.concatenate(arr)), rng.integers(0, 4, 300)], seed)


def tandem(period, diverged, seed=5):
    rng = np.random.default_rng(seed + 7 * period)
    unit = np.zeros(1, np.uint8) if period == 1 else rng.integers(0, 4, period).astype(np.uint8)
    copies = 30 if period >= 30 else max(2, 300 // period)
    arr = np.tile(unit, copies)
    if diverged:
        arr = _mutate(rng, arr, 0.01)
    return _build(f"tan{period}{'d' if diverged else 'x'}", [rng.integers(0, 4, 250), ("hot", arr), rng.integers(0, 4, 250)], seed)


def contigs(k, seed=6):
    """16 contigs (the most an index holds): lengths k - 1, k, k + 1 and 32 m +- 1 among them; a 60-base unit at the very start of
    contig 0, at the very end of the last contig, inside contig 9, and across the boundary of contigs 12 and 13"""
    rng = np.random.default_rng(seed + k)
    lens = [400, k - 1, k, k + 1, 31, 33, 63, 65, 95, 300, 97, 129, 250, 220, 127, 400]
    cs = [rng.integers(0, 4, n).astype(np.uint8) for n in lens]
    unit = rng.integers(0, 4, 60).astype(np.uint8)
    cs[0][:60] = unit
    cs[15][-60:] = rc(unit)
    cs[9][100:160] = unit
    cs[12][-30:] = unit[:30]
    cs[13][:30] = unit[30:]
    g = Genome("ctg", cs)
    o = g.offs
    g.hot = [(0, 120), (int(o[15]) + 300, int(o[16])), (int(o[9]) + 60, int(o[9]) + 200), (int(o[12]) + 150, int(o[13]) + 80),
             (int(o[1]), int(o[9]))]
    return g


def mixed(seed=7):
    """paired-end ground: 24 kb of background holding an exact 300-base unit in four copies (+ + - +), a 45 x 30 tandem array with
    1 % divergence, an inverted repeat and a 40-base unit in 20 + 20 copies, in two contigs"""
    rng = np.random.default_rng(seed)
    bg = lambda n: rng.integers(0, 4, n).astype(np.uint8)
    u300, u45, u40, u150 = bg(300), bg(45), bg(40), bg(150)
    tan = _mutate(rng, np.tile(u45, 30), 0.01)
    occ = np.concatenate([np.concatenate([u40 if j < 20 else rc(u40), bg(5)]) for j in range(40)])
    c0 = [bg(1500), u300, bg(2500), u300, bg(2000), tan, bg(2500), rc(u300), bg(2000), np.concatenate([u150, bg(1), rc(u150)]), bg(1500)]
    c1 = [bg(1800), u300, bg(2000), occ, bg(2200)]
    return Genome("mixed", [np.concatenate(c0), np.concatenate(c1)])


def families(k):
    """every genome family at seed length k (only `ctg` depends on k)"""
    out = [unique()]
    out += [dispersed(m, d) for m in DISP_MIXES for d in (False, True)]
    out += [inverted(s) for s in (0, 1, 5)]
    out += [occurrences(a, b) for a, b in OCC_SPLITS]
    out += [tandem(p, d) for p in TAN_PERIODS for d in (False, True)]
    out.append(contigs(k))
    return out


def by_name(k, name):
    return next(g for g in families(k) if g.name == name)


# ---------------------------------------------------------------------------------------------------------------------------
# reads
def _cut(rng, g, D, L):
    """L bases of the doubled genome: from a hot interval (either strand) two times in three, else anywhere"""
    n2 = len(D)
    if L > n2:
        return rng.integers(0, 4, L).astype(np.uint8)
    if g.hot and L <= g.l_pac and rng.random() < 0.67:
        b, e = g.hot[rng.integers(0, len(g.hot))]
        x = int(rng.integers(b - L // 2, max(b - L // 2 + 1, e - L // 2)))
        x = min(max(x, 0), g.l_pac - L)
        if rng.random() < 0.5:
            x = n2 - x - L                        # the same bases read from the other strand
    else:
        x = int(rng.integers(0, n2 - L + 1))
    return D[x:x + L].copy()


def edit(rng, g, D, rd, kind, k):
    L = len(rd)
    if kind == "errors":
        rd = _mutate(rng, rd, 0.02)
    elif kind == "planned_subs":
        for j in (0, k - 1, k, 31, 32, 63, 64, L - 1):
            if 0 <= j < L:
                rd[j] = (rd[j] + 1 + rng.integers(0, 3)) % 4
    elif kind == "n_edges":
        for j in (31, 32, 63, 64, 127, 128):
            if j < L and rng.random() < 0.6:
                rd[j] = 4
    elif kind == "n_run" and L > 0:
        n = int(rng.integers(k + 1, 2 * k + 2))
        b = int(rng.integers(0, max(1, L - n // 2)))
        rd[b:b + n] = 4
    elif kind == "all_n":
        rd[:] = 4
    elif kind == "chimera" and L >= 2:
        h = L // 2
        rd[h:] = rc(_cut(rng, g, D, L - h))
    elif kind == "errors_n" and L > 0:
        rd = _mutate(rng, rd, 0.01)
        rd[int(rng.integers(0, L))] = 4
    return rd


def reads(g, k, n, stride, seed, lens=None):
    """n reads in rows of `stride` -> (codes [n, stride] uint8, lens [n] int32).  Lengths cycle through READ_LENS and k - 1, k, k + 1
    (those that fit the row), two reads in three are full rows; edits cycle through EDITS."""
    rng = np.random.default_rng(seed)
    D = g.doubled()
    choices = [x for x in READ_LENS + (k - 1, k, k + 1) if x <= stride]
    codes = rng.integers(0, 4, (n, stride)).astype(np.uint8)
    out_lens = np.zeros(n, np.int32)
    for r in range(n):
        L = int(lens[r]) if lens is not None else (stride if r % 3 else choices[(r // 3) % len(choices)])
        rd = edit(rng, g, D, _cut(rng, g, D, L), EDITS[r % len(EDITS)], k)
        codes[r, :L] = rd
        out_lens[r] = L
    return codes, out_lens


def pairs(g, n_pairs, seed, read_len=150, ins_mean=400, ins_sd=30, err=0.01):
    """n_pairs FR pairs from either strand of the doubled genome -> (codes [2 n, read_len], lens); no fragment leaves its contig"""
    rng = np.random.default_rng(seed)
    D = g.doubled()
    ends = np.concatenate([g.offs[1:], g.l_pac + np.cumsum(g.lens[::-1])])
    starts = np.concatenate([g.offs[:-1], g.l_pac + np.concatenate([[0], np.cumsum(g.lens[::-1])[:-1]])])
    codes = np.zeros((2 * n_pairs, read_len), np.uint8)
    for p in range(n_pairs):
        while True:
            f = int(np.clip(rng.normal(ins_mean, ins_sd), read_len, 3 * ins_mean))
            x = int(rng.integers(0, len(D) - f + 1))
            c = np.searchsorted(ends, x, side="right")
            if x + f <= ends[c] and x >= starts[c]:
                break
        frag = D[x:x + f]
        codes[2 * p] = _mutate(rng, frag[:read_len], err)
        codes[2 * p + 1] = _mutate(rng, rc(frag[-read_len:]), err)
    return codes, np.full(2 * n_pairs, read_len, np.int32)


# ---------------------------------------------------------------------------------------------------------------------------
# the brute force of DESIGN.md 5.1
class KmerIndex:
    """forward positions of every k-mer inside one contig, ascending"""

    def __init__(self, g, k):
        self.g, self.k = g, k
        self.pos = {}
        for c in range(len(g.lens)):
            b, e = int(g.offs[c]), int(g.offs[c + 1])
            for p in range(b, e - k + 1):
                self.pos.setdefault(g.codes[p:p + k].tobytes(), []).append(p)

    def count(self, km):
        return len(self.pos.get(np.asarray(km, np.uint8).tobytes(), ()))


def brute_seeds(ix, read, max_occ, stats=None):
    """the seeds of one read, in creation order, as (qbeg, rbeg, len); `stats` (a dict of sets) collects what the read looked up:
    'strand_counts' (pass-0 count, pass-1 count) of every N-free k-mer found at all, 'palindromes' the count of palindromic ones"""
    k, l_pac = ix.k, ix.g.l_pac
    cap = min(max_occ, OCC_CAP)
    read = np.asarray(read, np.uint8)
    seeds, tail = [], {}                         # tail: diagonal -> index of its latest seed
    for q in range(len(read) - k + 1):
        km = read[q:q + k]
        if (km > 3).any():
            continue
        kr = rc(km)
        occ = [ix.pos.get(km.tobytes(), ()), ix.pos.get(kr.tobytes(), ())]
        if stats is not None and (occ[0] or occ[1]):
            stats.setdefault("strand_counts", set()).add((len(occ[0]), len(occ[1])))
            if np.array_equal(km, kr):
                stats.setdefault("palindromes", set()).add(len(occ[0]))
        for pss in (0, 1):
            if not occ[pss] or len(occ[pss]) > cap:
                continue
            for p in occ[pss]:
                rpos = p if pss == 0 else 2 * l_pac - p - k
                d = rpos - q
                m = tail.get(d)
                if m is not None and seeds[m][0] + seeds[m][2] - k == q - 1:
                    seeds[m][2] += 1
                elif len(seeds) < MAX_SEEDS:
                    tail[d] = len(seeds)
                    seeds.append([q, rpos, k])
    return [tuple(s) for s in seeds]


def brute_batch(ix, codes, lens, max_occ, stats=None):
    """sorted (qbeg, rbeg, len) lists of every read of a batch"""
    return [sorted(brute_seeds(ix, codes[r, :lens[r]], max_occ, stats)) for r in range(len(lens))]


def seed_lists(seeds, n_seeds):
    """a batch's seed array ([n, 64] of SEED_DTYPE, either side's) -> sorted (qbeg, rbeg, len) lists"""
    return [sorted((int(s["qbeg"]), int(s["rbeg"]), int(s["len"])) for s in seeds[r, :n_seeds[r]]) for r in range(len(n_seeds))]


def fwd_span(l_pac, qrbeg_len):
    """forward interval [b, e) of a seed given as (qbeg, rbeg, len)"""
    _, rb, ln = qrbeg_len
    return (rb, rb + ln) if rb < l_pac else (2 * l_pac - rb - ln, 2 * l_pac - rb)
