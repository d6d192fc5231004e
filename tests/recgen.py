"""Hand-built alignment records for the parity tests of the record consumers (pileup counts, indel table, text pileup,
BAQ): a small four-contig reference, a seeded generator of self-consistent records and an adversarial list aimed at the
code paths that aligner output rarely reaches (gap-free fast path, mate-overlap rewrite, operation-level channels,
contig ends, indel keys, admission flags).

Records are qm_aln (ALN_DTYPE); bases and qualities are stored as sequenced (a reverse read reverse-complemented against
its CIGAR), one row of `stride` bytes per read, reads 2i and 2i + 1 mates.  Every record with a CIGAR is consistent:
its query length is lens[r] and its reference span lies inside its contig."""
import numpy as np

from oracle.qmo_py import ALN_DTYPE, MAX_CIGAR

M, I, D, S = 0, 1, 2, 4
CONTIG_LENS = (300, 1, 517, 64)             # a 1-base contig, and a last contig whose end a read can reach
NAMES = ["chrA", "chrB", "chrC", "chrD"]
_COMP = np.array([3, 2, 1, 0, 4], np.uint8)


class Genome:
    """what qmo_py.Ref and Context.index take: base codes 0..3 of the concatenated contigs and their lengths"""

    def __init__(self, seed=11, lens=CONTIG_LENS):
        self.lens = np.array(lens, np.int64)
        self.offs = np.concatenate([[0], np.cumsum(self.lens)]).astype(np.int64)
        self.codes = np.random.default_rng(seed).integers(0, 4, int(self.lens.sum())).astype(np.uint8)
        self.names = NAMES[:len(lens)]
        self.l_pac = int(self.lens.sum())


class Batch:
    """records, bases, qualities and lengths of a batch of pairs; add() appends one pair"""

    def __init__(self, genome, rng, sub=0.05, n_rate=0.02):
        self.g, self.rng, self.sub, self.n_rate = genome, rng, sub, n_rate
        self.recs, self.seqs, self.qls = [], [], []

    def read(self, rid, pos, ops, flag=0x1 | 0x2, mapq=60, quals=None, seq=None):
        """one read: bases in BAM SEQ orientation follow the reference on M (sub / n_rate errors), random elsewhere"""
        rng = self.rng
        L = sum(ln for op, ln in ops if op in (M, I, S))
        if seq is None:
            seq = rng.integers(0, 4, L).astype(np.uint8)
            q, p = 0, pos
            for op, ln in ops:
                if op == M:
                    seq[q:q + ln] = self.g.codes[self.g.offs[rid] + p:self.g.offs[rid] + p + ln]
                    q += ln; p += ln
                elif op in (I, S):
                    q += ln
                elif op == D:
                    p += ln
            flip = rng.random(L) < self.sub
            seq[flip] = (seq[flip] + rng.integers(1, 4, int(flip.sum()))) % 4
            seq[rng.random(L) < self.n_rate] = 4
        if quals is None:
            quals = rng.integers(0, 60, L)
            hi = rng.random(L) < 0.1                 # some qualities above 59: overlap sums then reach the cap at 200
            quals[hi] = rng.integers(60, 256, int(hi.sum()))
        return dict(rid=rid, pos=pos, ops=list(ops), flag=flag, mapq=mapq, seq=np.asarray(seq, np.uint8),
                    quals=np.broadcast_to(np.asarray(quals, np.uint8), (L,)).copy())

    def unmapped(self, L, flag=0x1 | 0x4, n_cigar=0):
        rng = self.rng
        return dict(rid=-1, pos=-1, ops=[], flag=flag, mapq=0, n_cigar=n_cigar, seq=rng.integers(0, 5, L).astype(np.uint8),
                    quals=rng.integers(0, 60, L).astype(np.uint8))

    def add(self, r0, r1, tlen=None):
        """a pair; tlen None: the template length the two placements imply (0 across contigs)"""
        if tlen is None:
            tlen = 0
            if r0["rid"] == r1["rid"] and r0["rid"] >= 0:
                e0, e1 = r0["pos"] + span(r0["ops"]), r1["pos"] + span(r1["ops"])
                t = max(e0, e1) - min(r0["pos"], r1["pos"])
                tlen = t if r0["pos"] <= r1["pos"] else -t
        for e, (r, m) in enumerate(((r0, r1), (r1, r0))):
            a = np.zeros((), ALN_DTYPE)
            flag = r["flag"]
            if flag & 0x1:
                flag |= 0x40 if e == 0 else 0x80
                if m["flag"] & 0x10:
                    flag |= 0x20
            a["rid"], a["pos"], a["flag"], a["mapq"] = r["rid"], r["pos"], flag, r["mapq"]
            a["n_cigar"] = r.get("n_cigar", len(r["ops"]))
            a["cigar"][:len(r["ops"])] = [(ln << 4) | op for op, ln in r["ops"]]
            a["mate_rid"], a["mate_pos"] = m["rid"], m["pos"]
            a["tlen"] = tlen if e == 0 else -tlen
            self.recs.append(a)
            seq, ql = r["seq"], r["quals"]
            if flag & 0x10:                          # stored as sequenced
                seq, ql = _COMP[seq[::-1]], ql[::-1]
            self.seqs.append(seq)
            self.qls.append(ql)

    def arrays(self, stride=None, seed=0):
        """-> alns, codes [n, stride], quals [n, stride], lens; the bytes past a read's length are junk"""
        lens = np.array([len(s) for s in self.seqs], np.int32)
        stride = stride or int(lens.max())
        return (np.array(self.recs, ALN_DTYPE),) + lay_out(self.seqs, self.qls, lens, stride, seed=seed) + (lens,)


def span(ops):
    return sum(ln for op, ln in ops if op in (M, D))


def lay_out(seqs, quals, lens, stride, offset=0, seed=0):
    """the reads at `stride` bytes per row behind `offset` leading bytes -> (codes, quals): [n, stride] arrays when offset is
    0, flat arrays of offset + n * stride bytes otherwise (read r at offset + r * stride).  Junk everywhere else: a consumer
    that reads past a read's length sees it."""
    n = len(lens)
    assert int(np.max(lens, initial=0)) <= stride
    rng = np.random.default_rng(seed)
    c = rng.integers(0, 256, offset + n * stride).astype(np.uint8)
    q = rng.integers(0, 256, offset + n * stride).astype(np.uint8)
    for r in range(n):
        L = int(lens[r])
        c[offset + r * stride:offset + r * stride + L] = seqs[r][:L]
        q[offset + r * stride:offset + r * stride + L] = quals[r][:L]
    if offset == 0:
        return c.reshape(n, stride), q.reshape(n, stride)
    return c, q


def relayout(codes, quals, lens, stride, offset=0, seed=0):
    """lay_out for rows of an existing [n, old stride] batch"""
    return lay_out(list(codes), list(quals), lens, stride, offset, seed)


def random_ops(rng, L, max_span):
    """an M/I/D/S CIGAR of query length L and reference span 1..max_span with at most QM_MAX_CIGAR operations, or None"""
    for _ in range(200):
        ops, q = [], 0
        if rng.random() < 0.3:
            s = int(rng.integers(1, max(2, L // 3)))
            ops.append((S, min(s, L)))
            q += ops[-1][1]
        while q < L and len(ops) < MAX_CIGAR:
            u, ln = rng.random(), int(rng.integers(1, 12))
            if u < 0.55 or q == 0 and u < 0.7:
                ln = min(ln if rng.random() < 0.5 else int(rng.integers(1, 80)), L - q)
                ops.append((M, ln)); q += ln
            elif u < 0.75:
                ln = min(ln, L - q); ops.append((I, ln)); q += ln
            elif u < 0.95:
                ops.append((D, ln))
            else:
                ops.append((S, L - q)); q = L
        if q == L and rng.random() < 0.05 and len(ops) < MAX_CIGAR:
            ops.append((D, int(rng.integers(1, 4))))          # a read that ends in a deletion
        sp = span(ops)
        if q == L and len(ops) <= MAX_CIGAR and 0 < sp <= max_span and any(op == M for op, _ in ops):
            return ops
    return None


def random_batch(genome, n_pairs, seed, max_len=150, batch=None):
    """n_pairs seeded random pairs: read lengths 1..max_len, M/I/D/S CIGARs, mates that mostly overlap on one contig,
    admission flags and MAPQs spread over their ranges"""
    rng = np.random.default_rng(seed)
    b = batch or Batch(genome, rng)
    clens = genome.lens
    for _ in range(n_pairs):
        reads = []
        for e in range(2):
            L = int(rng.integers(1, max_len + 1))
            rid = int(rng.integers(0, len(clens)))
            ops = random_ops(rng, L, int(clens[rid]))
            if ops is None:
                reads.append(b.unmapped(L))
                continue
            flag = 0x1 | 0x2 | (0x10 if rng.random() < 0.5 else 0)
            u = rng.random()
            if u < 0.04:
                flag &= ~0x2                                   # orphan
            elif u < 0.06:
                flag |= int(rng.choice([0x100, 0x200, 0x400]))
            reads.append(dict(rid=rid, L=L, ops=ops, flag=flag, mapq=int(rng.integers(0, 61))))
        x, y = reads
        if "L" in x and "L" in y and rng.random() < 0.75 and span(y["ops"]) <= clens[x["rid"]]:
            y["rid"] = x["rid"]                                 # the mates overlap (or nearly)
            lim = int(clens[x["rid"]]) - span(y["ops"])
            x_pos = int(rng.integers(0, int(clens[x["rid"]]) - span(x["ops"]) + 1))
            x["pos"] = x_pos
            y["pos"] = int(min(max(0, x_pos + int(rng.integers(-30, 31))), lim))
            if rng.random() < 0.1:
                y["pos"] = min(x_pos, lim)                      # equal positions: the strand decides which mate is `a`
        for r in (x, y):
            if "L" in r and "pos" not in r:
                r["pos"] = int(rng.integers(0, int(clens[r["rid"]]) - span(r["ops"]) + 1))
        rr = [b.read(r["rid"], r["pos"], r["ops"], r["flag"], r["mapq"]) if "L" in r else r for r in (x, y)]
        if rng.random() < 0.03:
            rr[int(rng.integers(0, 2))]["flag"] |= 0x8         # mate unmapped on one record only
        tlen = None
        if "L" in x and rng.random() < 0.1:
            tlen = int(rng.choice([2 * x["L"], 2 * x["L"] - 1, -2 * x["L"]]))
        b.add(rr[0], rr[1], tlen)
    return b


def adversarial(genome, seed=3):
    """the hand-written cases, one or a few pairs each (see the comments); lengths <= 150"""
    rng = np.random.default_rng(seed)
    b = Batch(genome, rng)
    r = b.read
    P = 0x1 | 0x2
    R = 0x10
    last = len(genome.lens) - 1
    cl = [int(x) for x in genome.lens]

    def q(v, L):
        return np.full(L, v, np.uint8)

    # gap-free fast path: [S] M [S] at every length class around the 4-base groups, both strands, leading clips of 0..3
    # (unaligned group starts), starting at 0 and ending at the contig's last base
    for L in (1, 2, 3, 4, 5, 7, 8, 9, 31, 32, 33, 127, 128, 129, 150):
        for clip in (0, 1, 2, 3):
            for tail in (0, 2):
                m = L - clip - tail
                if m < 1:
                    continue
                ops = ([(S, clip)] if clip else []) + [(M, m)] + ([(S, tail)] if tail else [])
                rid = 2 if m <= cl[2] else 0
                b.add(r(rid, 0, ops, P), r(rid, cl[rid] - m, ops, P | R))
                b.add(r(0, 7, ops, P | R), r(last, cl[last] - m, ops, P) if m <= cl[last] else r(0, 0, ops, P))
    # the same with reads equal to the reference and high qualities: whole groups take the no-mismatch branch
    for L in (4, 64, 150):
        ex = Batch(genome, rng, sub=0.0, n_rate=0.0)
        b.add(ex.read(2, 11, [(M, L)], P, quals=q(40, L)), ex.read(2, 13, [(M, L)], P | R, quals=q(40, L)), tlen=10 * L)
        b.add(ex.read(2, 200, [(S, 3), (M, L - 3)], P | R, quals=q(40, L)), ex.read(0, 1, [(M, L - 1), (S, 1)], P, quals=q(40, L)))
    # mate overlap: equal positions (strand tie-break both ways), mismatching bases with equal qualities (qa >= qb picks `a`),
    # sums above 200, |tlen| at and just under 2 L, flag 0x8 on one mate only, proper-pair flag on one mate only
    for r0, r1 in ((R, 0), (0, R), (0, 0), (R, R)):
        L = 40
        s = rng.integers(0, 4, L).astype(np.uint8)
        b.add(r(2, 50, [(M, L)], P | r0, seq=s, quals=q(30, L)), r(2, 50, [(M, L)], P | r1, seq=(s + 1) % 4, quals=q(30, L)))
        b.add(r(2, 50, [(M, L)], P | r0, seq=s, quals=q(110, L)), r(2, 50, [(M, L)], P | r1, seq=s, quals=q(120, L)))
        b.add(r(2, 60, [(M, L)], P | r0, seq=s, quals=q(25, L)), r(2, 60, [(M, L)], P | r1, seq=(s + 2) % 4, quals=q(31, L)))
    for t in (80, 79, -80, -79, 81):
        b.add(r(0, 100, [(M, 40)], P), r(0, 110, [(M, 40)], P | R), tlen=t)
    b.add(r(0, 100, [(M, 40)], P | 0x8), r(0, 110, [(M, 40)], P | R))
    b.add(r(0, 100, [(M, 40)], P), r(0, 110, [(M, 40)], P | R | 0x8))
    b.add(r(0, 100, [(M, 40)], 0x1), r(0, 110, [(M, 40)], P | R))
    b.add(r(0, 100, [(M, 40)], P), r(0, 110, [(M, 40)], 0x1 | R))
    b.add(r(0, 100, [(M, 40)], P), r(1, 0, [(M, 1)], P | R))                               # mates on different contigs
    # overlap through gaps: the mates' CIGARs disagree about where the query bases sit
    b.add(r(2, 30, [(M, 10), (I, 3), (M, 10), (D, 4), (M, 20)], P), r(2, 35, [(S, 2), (M, 8), (D, 2), (M, 30)], P | R))
    b.add(r(2, 30, [(M, 10), (D, 5), (M, 10)], P | R), r(2, 30, [(M, 5), (I, 5), (M, 15)], P))
    # operation-level channels: I / D right after a soft clip or first (no anchor), D / I last, adjacent gaps, 1-base M blocks
    for ops in ([(S, 3), (I, 2), (M, 20)], [(S, 3), (D, 2), (M, 20)], [(I, 2), (M, 20)], [(D, 3), (M, 20)],
                [(M, 20), (D, 3)], [(M, 20), (I, 3)], [(M, 20), (I, 2), (S, 3)], [(M, 10), (D, 2), (I, 3), (M, 10)],
                [(M, 10), (I, 3), (D, 2), (M, 10)], [(M, 10), (D, 2), (D, 3), (M, 10)], [(M, 10), (I, 2), (I, 1), (M, 10)],
                [(M, 10), (D, 2), (S, 4)], [(S, 2), (D, 1), (I, 1), (M, 5), (D, 1)], [(M, 1), (D, 1)] * 10 + [(M, 1)],
                [(M, 1), (I, 1)] * 10 + [(M, 1)], [(S, 1)] + [(M, 1), (I, 1), (M, 1), (D, 1)] * 5,
                [(M, 1)], [(S, 5), (M, 1), (S, 5)], [(I, 1), (D, 1), (M, 1), (S, 1)]):
        for flag in (P, P | R):
            b.add(r(2, 300, ops, flag), r(2, 305, ops, flag ^ R))
            b.add(r(0, 0, ops, flag), r(last, cl[last] - span(ops), ops, flag))
    # the 1-base contig: every read there covers its only base
    for ops in ([(M, 1)], [(S, 2), (M, 1), (S, 3)], [(M, 1), (I, 4)], [(I, 2), (M, 1)], [(S, 1), (M, 1)]):
        b.add(r(1, 0, ops, P), r(1, 0, ops, P | R))
    # indel keys: deletions longer than 255 (clamped), N among the first 11 inserted bases, N only after the 11th
    b.add(r(2, 10, [(M, 20), (D, 300), (M, 20)], P), r(2, 12, [(M, 20), (D, 256), (M, 30)], P | R))
    b.add(r(2, 10, [(M, 20), (D, 255), (M, 20)], P | R), r(0, 5, [(M, 30), (D, 255), (M, 5)], P))
    for npos in (0, 5, 10, 11, 13):
        s = np.concatenate([b.g.codes[b.g.offs[2] + 40:b.g.offs[2] + 60], rng.integers(0, 4, 14), b.g.codes[b.g.offs[2] + 60:b.g.offs[2] + 80]])
        s = s.astype(np.uint8)
        s[20 + npos] = 4
        for flag in (P, P | R):
            b.add(r(2, 40, [(M, 20), (I, 14), (M, 20)], flag, seq=s.copy()), r(2, 41, [(M, 19), (I, 14), (M, 21)], flag ^ R, seq=s.copy()))
    # admission: every flag that drops a read, unpaired reads, n_cigar 0 and 255, MAPQ around 20, MAPQ above 93
    for f in (0x4, 0x100, 0x200, 0x400):
        b.add(r(0, 50, [(M, 30)], P | f), r(0, 55, [(M, 30)], P | R | f))
    b.add(r(0, 50, [(M, 30)], 0), r(0, 55, [(M, 30)], R))
    b.add(r(0, 50, [(M, 30)], 0x1), r(0, 55, [(M, 30)], 0x1 | R))
    b.add(b.unmapped(30, 0x1 | 0x2, 0), r(0, 55, [(M, 30)], P | R))
    b.add(r(0, 60, [(M, 30)], P), b.unmapped(30, 0x1 | 0x4, 255))
    for mq in (19, 20, 21, 93, 94, 255):
        b.add(r(2, 400, [(M, 30)], P, mapq=mq), r(2, 410, [(S, 5), (M, 25)], P | R, mapq=mq))
    return b


def tiled(arrays, n_pairs, seed):
    """a batch of n_pairs pairs from the pairs of `arrays` (alns, codes, quals, lens) repeated in turn, every repeat with
    qualities drawn afresh (a large batch at the cost of a small one)"""
    alns, codes, quals, lens = arrays
    pick = np.arange(n_pairs) % (len(lens) // 2)
    rows = np.stack([2 * pick, 2 * pick + 1], 1).reshape(-1)
    q = np.random.default_rng(seed).integers(0, 60, (2 * n_pairs, quals.shape[1])).astype(np.uint8)
    q[:len(lens)] = quals
    return alns[rows].copy(), codes[rows].copy(), q, lens[rows].copy()


def long_batch(genome, n_pairs, seed):
    """reads up to 512 bases (insertions longer than 255: the clamped length key) next to random ones"""
    rng = np.random.default_rng(seed)
    b = Batch(genome, rng)
    P, R = 0x1 | 0x2, 0x10
    b.add(b.read(2, 5, [(M, 10), (I, 300), (M, 10)], P), b.read(2, 6, [(M, 9), (I, 256), (M, 11)], P | R))
    b.add(b.read(2, 5, [(M, 10), (I, 255), (M, 10)], P | R), b.read(2, 0, [(S, 12), (M, 500)], P))
    b.add(b.read(2, 0, [(M, 512)], P | R), b.read(2, 5, [(M, 400), (D, 100), (M, 12)], P))
    return random_batch(genome, n_pairs, seed + 1, max_len=512, batch=b)
