"""Strain pairs with planted differences for the genome diff (DESIGN.md 5c), built from the bundled genomes with a seeded
numpy RNG.  Each pair comes with the rows the contract says it must give: the planted substitutions and indel bases, indels at
their leftmost equivalent placement, minus the differences in both copies of a duplication (-C).

The reference is a 60 kb slice of Merlin's unique long region.  The query is the slice with, in this order along the reference:
  - isolated SNPs, clusters of SNPs closer than max_gap, 1-8-base insertions and deletions, some inside homopolymers;
  - 150 bases replaced by unrelated sequence, too divergent to bridge: the alignment ends on both sides of it;
  - a 3 kb deletion;
  - a 5 kb inversion carrying SNPs (rows with FRM -1);
  - a 2 kb block moved 3 kb downstream (transposition), with a SNP in each moved piece;
  - a 2 kb tandem duplication with a SNP in both copies (dropped by -C);
  - a break into two query contigs;
  - more small differences on the second contig;
  - SNPs 10 and 9 bases from the contig ends, which only the extension of the alignment ends reaches."""
import numpy as np

from quasimodo_b200 import genomes
from quasimodo_b200.genomes import Genome

ACGT = "ACGT"
SLICE = (60000, 120000)
DIVERGENT = (20300, 20450)          # replaced by unrelated bases in the planted pair's query: the alignment must end there


def base_ref(stem="Merlin", span=SLICE):
    g = genomes.load(stem)
    return Genome([f"{stem}_{span[0]}_{span[1]}"], [span[1] - span[0]], g.codes[span[0]:span[1]].copy())


def _left_del(ref, x, n):
    while x > 0 and ref[x - 1] == ref[x + n - 1]:
        x -= 1
    return x


def _left_ins(ref, x, s):
    """insertion of s in front of reference base x -> leftmost (x, s)"""
    s = list(s)
    while x > 0 and ref[x - 1] == s[-1]:
        s = [int(ref[x - 1])] + s[:-1]
        x -= 1
    return x, s


def _small_events(rng, ref, lo, hi, step):
    """(kind, x, data) every `step` bases in [lo, hi): kind 'snp' (data = new base), 'del' (length), 'ins' (bases)"""
    ev = []
    x = lo
    kinds = ["snp", "cluster", "del", "ins", "hdel", "hins"]
    while x < hi:
        kind = kinds[(x - lo) // step % len(kinds)]
        if kind == "snp":
            ev.append(("snp", x, int((ref[x] + rng.integers(1, 4)) % 4)))
        elif kind == "cluster":
            for d in (0, 7, 19, 33):
                ev.append(("snp", x + d, int((ref[x + d] + rng.integers(1, 4)) % 4)))
        elif kind in ("del", "ins"):
            n = int(rng.integers(1, 9))
            if kind == "del":
                ev.append(("del", x, n))
            else:
                ev.append(("ins", x, [int(b) for b in rng.integers(0, 4, n)]))
        else:                                             # in a homopolymer run of at least 3 bases
            y = x
            while y < x + step - 60 and not (ref[y] == ref[y + 1] == ref[y + 2]):
                y += 1
            if y < x + step - 60:
                n = int(rng.integers(1, 3))
                ev.append(("del", y + 1, n) if kind == "hdel" else ("ins", y + 1, [int(ref[y])] * n))
        x += step
    return ev


def planted_pair(seed=1):
    """-> (ref Genome, qry Genome, expected rows as a list of dicts in show-snps -r order, -C applied)"""
    rng = np.random.default_rng(seed)
    R = base_ref()
    ref = R.codes
    L = len(ref)
    ev = _small_events(rng, ref, 300, 20000, 310)
    inv = (26000, 31000)
    ev += [("snp", x, int((ref[x] + rng.integers(1, 4)) % 4)) for x in range(inv[0] + 300, inv[1] - 200, 600)]
    ev += [("snp", 34000, int((ref[34000] + 1) % 4)), ("snp", 36500, int((ref[36500] + 2) % 4))]
    dup = (41000, 43000)
    ev += [("snp", 42000, int((ref[42000] + 1) % 4))]
    ev += _small_events(rng, ref, 45200, 58000, 330)
    ev += [("snp", 10, int((ref[10] + 1) % 4)), ("snp", L - 9, int((ref[L - 9] + 1) % 4))]
    # one base per query position: (code, reference position or -1, strand)
    Q = [(int(b), x, 1) for x, b in enumerate(ref)]
    norm = []
    for kind, x, data in sorted(ev, key=lambda e: -e[1]):
        if kind == "snp":
            Q[x] = (data, x, 1)
            norm.append((kind, x, data))
        elif kind == "del":
            x = _left_del(ref, x, data)
            del Q[x:x + data]
            norm.append((kind, x, data))
        else:
            x, s = _left_ins(ref, x, data)
            Q[x:x] = [(b, -1, 0) for b in s]
            norm.append((kind, x, s))

    def where(x):
        for i, q in enumerate(Q):
            if q[1] == x:
                return i
        raise KeyError(x)

    # structural changes, located by reference position
    a, b = where(DIVERGENT[0]), where(DIVERGENT[1])
    Q[a:b] = [(int(c), -1, 0) for c in rng.integers(0, 4, b - a)]
    a, b = where(21000), where(24000)
    del Q[a:b]
    a, b = where(inv[0]), where(inv[1])
    Q[a:b] = [(3 - c, x, -s) for c, x, s in reversed(Q[a:b])]
    a, b, c = where(33000), where(35000), where(38000)
    Q[a:c] = Q[b:c] + Q[a:b]
    a, b = where(dup[0]), where(dup[1])
    Q[b:b] = Q[a:b]
    cut = where(44000)
    contigs = [Q[:cut], Q[cut:]]
    qry = Genome(["qry_a", "qry_b"], [len(c) for c in contigs], np.array([q[0] for q in Q], np.uint8))

    copies = {}
    for ci, c in enumerate(contigs):
        for i, q in enumerate(c):
            copies.setdefault(q[1], []).append((ci, i + 1, q[2]))

    def locate(x):
        """query contig, 1-based forward position and strand of reference base x (its only copy)"""
        assert len(copies[x]) == 1, (x, copies[x])
        return copies[x][0]

    rows = []
    for kind, x, data in norm:
        if dup[0] <= x < dup[1]:
            continue                                      # in both copies of the duplication
        if kind == "snp":
            ci, p2, s = locate(x)
            sub_q = ACGT[data]
            rows.append(dict(p1=x + 1, p2=p2, sub_r=ACGT[ref[x]], sub_q=sub_q, frm_q=s, qid=ci))
        elif kind == "del":
            ci, p2, s = locate(x - 1)
            for t in range(data):
                rows.append(dict(p1=x + 1 + t, p2=p2, sub_r=ACGT[ref[x + t]], sub_q=".", frm_q=s, qid=ci))
        else:
            ci, p2, s = locate(x - 1)
            for t, bq in enumerate(data):
                rows.append(dict(p1=x, p2=p2 + 1 + t, sub_r=".", sub_q=ACGT[bq], frm_q=s, qid=ci))
    rows.sort(key=lambda w: (w["p1"], w["p2"]))
    return R, qry, rows


def mutated_copy(genome, seed=7, n_snp=3000, n_indel=600, k=20):
    """a one-contig genome with spread-out SNPs and 1-8-base indels -> (query Genome, expected rows).  Events are at least 100
    bases apart and only where every reference k-mer within 150 bases is unique: a difference inside a repeat has no anchor
    next to it and is not reported (DESIGN.md 5c)"""
    from tests.gdiff_oracle import unique_kmers
    rng = np.random.default_rng(seed)
    ref = genome.codes
    L = len(ref)
    uniq = np.zeros(L + 1, np.int64)
    uniq[unique_kmers(genome, k)[1] + 1] = 1
    cum = np.cumsum(uniq)                                 # cum[x] = unique k-mers starting before x
    cand = np.arange(2, (L - 400) // 100) * 100
    ok = cum[cand + 150 - k] - cum[cand - 150] == 300 - k
    slots = np.sort(rng.choice(cand[ok], n_snp + n_indel, replace=False))
    kinds = rng.permutation(np.array(["snp"] * n_snp + ["del"] * (n_indel // 2) + ["ins"] * (n_indel - n_indel // 2)))
    parts, rows, last = [], [], 0
    shift = 0
    for x, kind in zip(slots.tolist(), kinds.tolist()):
        if kind == "snp":
            nb = int((ref[x] + rng.integers(1, 4)) % 4)
            parts += [ref[last:x], np.array([nb], np.uint8)]
            rows.append(dict(p1=x + 1, p2=x + shift + 1, sub_r=ACGT[ref[x]], sub_q=ACGT[nb], frm_q=1, qid=0))
            last = x + 1
        elif kind == "del":
            n = int(rng.integers(1, 9))
            x = _left_del(ref, x, n)
            parts.append(ref[last:x])
            rows += [dict(p1=x + 1 + t, p2=x + shift, sub_r=ACGT[ref[x + t]], sub_q=".", frm_q=1, qid=0) for t in range(n)]
            last = x + n
            shift -= n
        else:
            s = [int(b) for b in rng.integers(0, 4, int(rng.integers(1, 9)))]
            x, s = _left_ins(ref, x, s)
            parts += [ref[last:x], np.array(s, np.uint8)]
            rows += [dict(p1=x, p2=x + shift + 1 + t, sub_r=".", sub_q=ACGT[b], frm_q=1, qid=0) for t, b in enumerate(s)]
            last = x
            shift += len(s)
    parts.append(ref[last:])
    codes = np.concatenate(parts).astype(np.uint8)
    return Genome([genome.names[0] + "_mut"], [len(codes)], codes), rows


def key(rows):
    """the comparable part of a row: (P1, SUB_R, SUB_Q, P2, FRM_Q, query contig)"""
    out = []
    for w in rows:
        sr, sq = w["sub_r"], w["sub_q"]
        sr = sr.decode() if isinstance(sr, bytes) else sr
        sq = sq.decode() if isinstance(sq, bytes) else sq
        out.append((int(w["p1"]), sr, sq, int(w["p2"]), int(w["frm_q"]), int(w["qid"])))
    return out
