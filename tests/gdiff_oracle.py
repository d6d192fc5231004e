"""CPU restatement of the genome diff (qm_genome_diff_host, DESIGN.md 5c): rows of `show-snps -CTHlr` after
`nucmer; delta-filter -r -q` as this project defines them.  Written from the contract, not from gdiff.cu:

- anchors by brute force: the reference's k-mers of both strands in a table, every query k-mer looked up, every unique hit
  extended base by base to its maximal exact match;
- the same clustering, merging, filter and row rules;
- every gap filled by the affine DP over the WHOLE rectangle (no band), with the same tie rules and the same divergence test;
- the alignment ends extended by the project's C restatement of ksw_extend2 (oracle/qmo_ksw.c), in the same windows.

Fast enough for HCMV-size pairs (a quarter of a megabase) on one CPU core."""
import numpy as np

from quasimodo_b200 import _lib

NEG = -(1 << 29)
OP_M, OP_D, OP_I = 0, 1, 2
ACGT = "ACGT"


def default_opt():
    return dict(min_match=20, min_cluster=65, max_gap=90, break_len=200, diag_factor=0.12, max_diag=5, match=1, mismatch=4,
                gap_open=6, gap_extend=1, flags=0)


def opt_from_struct(o):
    return {f: getattr(o, f) for f in default_opt()}


def _keys(codes, k):
    """2-bit keys (first base most significant) of every k-mer of one contig"""
    n = len(codes) - k + 1
    if n <= 0:
        return np.zeros(0, np.uint64)
    key = np.zeros(n, np.uint64)
    c = codes.astype(np.uint64)
    for j in range(k):
        key = (key << np.uint64(2)) | c[j:j + n]
    return key


def _contigs(genome):
    off = np.concatenate([[0], np.cumsum(genome.lens)]).astype(np.int64)
    return [(int(off[i]), int(genome.lens[i])) for i in range(len(genome.lens))]


def unique_kmers(ref, k):
    """sorted keys and forward positions of the reference k-mers that occur once and whose reverse complement never does"""
    fk, fp, rk = [], [], []
    for o, ln in _contigs(ref):
        c = ref.codes[o:o + ln]
        key = _keys(c, k)
        fk.append(key)
        fp.append(np.arange(len(key), dtype=np.int64) + o)
        rk.append(_keys((3 - c[::-1]).astype(np.uint8), k))
    fk, fp, rk = np.concatenate(fk), np.concatenate(fp), np.concatenate(rk)
    u, first, cnt = np.unique(fk, return_index=True, return_counts=True)
    keep = (cnt == 1) & ~np.isin(u, rk)
    return u[keep], fp[first[keep]]


def _match_right(a, i, b, j, limit):
    """length of the common run of a[i:] and b[j:], at most limit"""
    n = 0
    while n < limit:
        step = min(256, limit - n)
        ne = np.nonzero(a[i + n:i + n + step] != b[j + n:j + n + step])[0]
        if len(ne):
            return n + int(ne[0])
        n += step
    return n


def anchors(ref, qry, k):
    """(s, qc, rc, qs, rs, len) of every maximal exact match containing a unique reference k-mer, sorted"""
    ukeys, upos = unique_kmers(ref, k)
    rcon = _contigs(ref)
    roff = np.array([o for o, _ in rcon], np.int64)
    out = set()
    for qc, (o, ln) in enumerate(_contigs(qry)):
        fwd = qry.codes[o:o + ln]
        for s, Q in ((0, fwd), (1, (3 - fwd[::-1]).astype(np.uint8))):
            key = _keys(Q, k)
            ix = np.searchsorted(ukeys, key)
            ix[ix >= len(ukeys)] = 0
            hit = np.nonzero(ukeys[ix] == key)[0] if len(ukeys) else np.zeros(0, np.int64)
            hits = sorted((int(upos[ix[x]]) - int(x), int(x)) for x in hit)       # (diagonal, query position)
            cur_diag, cur_end = None, -1
            for diag, x in hits:
                if diag == cur_diag and x < cur_end:
                    continue
                p = diag + x
                rc = int(np.searchsorted(roff, p, side="right") - 1)
                rb, rl = rcon[rc]
                R = ref.codes[rb:rb + rl]
                pr = p - rb
                a = 0
                while a < min(x, pr) and Q[x - a - 1] == R[pr - a - 1]:
                    a += 1
                b = k + _match_right(Q, x + k, R, pr + k, min(ln - x - k, rl - pr - k))
                out.add((s, qc, rc, x - a, pr - a, a + b))
                cur_diag, cur_end = diag, x + b
    return sorted(out, key=lambda t: (t[1], t[0], t[2], t[4], t[3]))


def _trim_after(a, b):
    ov = max(0, a[4] + a[5] - b[4], a[3] + a[5] - b[3])
    if ov >= b[5]:
        return None
    return (b[0], b[1], b[2], b[3] + ov, b[4] + ov, b[5] - ov)


def clusters(group, o):
    """one (qc, s, rc) group's anchors, sorted by (rs, qs) -> clusters of at least min_cluster anchored bases"""
    n = len(group)
    maxlen = max(a[5] for a in group)
    score = [a[5] for a in group]
    pred = [-1] * n
    for j in range(n):
        b = group[j]
        best, bp = b[5], -1
        for i in range(j):
            a = group[i]
            if b[4] - a[4] > o["max_gap"] + maxlen:
                continue
            if not (a[4] < b[4] and a[3] < b[3] and a[4] + a[5] < b[4] + b[5] and a[3] + a[5] < b[3] + b[5]):
                continue
            gr, gq = b[4] - (a[4] + a[5]), b[3] - (a[3] + a[5])
            sep = max(gr, gq)
            if sep > o["max_gap"]:
                continue
            if abs(gr - gq) > max(float(o["max_diag"]), float(np.float32(o["diag_factor"])) * max(sep, 0)):
                continue
            if score[i] + b[5] > best:
                best, bp = score[i] + b[5], i
        score[j], pred[j] = best, bp
    order = sorted(range(n), key=lambda j: -score[j])
    used = [False] * n
    out = []
    for e in order:
        if used[e]:
            continue
        path = []
        i = e
        while i >= 0 and not used[i]:
            used[i] = True
            path.append(group[i])
            i = pred[i]
        kept = []
        for b in reversed(path):
            if kept:
                b = _trim_after(kept[-1], b)
                if b is None:
                    continue
            kept.append(b)
        if sum(a[5] for a in kept) >= o["min_cluster"]:
            out.append(kept)
    return out


def gap_dp(R, Q, o):
    """global affine alignment of R against Q over the whole matrix -> ops, first column first"""
    n, m = len(R), len(Q)
    ma, mi, go, ge = o["match"], o["mismatch"], o["gap_open"], o["gap_extend"]
    H = np.full((n + 1, m + 1), NEG, np.int64)
    E = np.full((n + 1, m + 1), NEG, np.int64)
    F = np.full((n + 1, m + 1), NEG, np.int64)
    TB = np.zeros((n + 1, m + 1), np.uint8)
    H[0, 0] = 0
    for i in range(1, n + 1):
        E[i, 0] = H[i, 0] = -(go + i * ge)
        TB[i, 0] = 1 | (4 if i > 1 else 0)
    for j in range(1, m + 1):
        F[0, j] = H[0, j] = -(go + j * ge)
        TB[0, j] = 2 | (8 if j > 1 else 0)
    Ra, Qa = np.asarray(R, np.int64), np.asarray(Q, np.int64)
    for d in range(2, n + m + 1):
        i = np.arange(max(1, d - m), min(n, d - 1) + 1)
        if not len(i):
            continue
        j = d - i
        eo, ex = H[i - 1, j] - (go + ge), E[i - 1, j] - ge
        fo, fx = H[i, j - 1] - (go + ge), F[i, j - 1] - ge
        e, f = np.maximum(eo, ex), np.maximum(fo, fx)
        h = H[i - 1, j - 1] + np.where(Ra[i - 1] == Qa[j - 1], ma, -mi)
        src = np.zeros(len(i), np.uint8)
        src[e > h] = 1
        h = np.maximum(h, e)
        src[f > h] = 2
        h = np.maximum(h, f)
        H[i, j], E[i, j], F[i, j] = h, e, f
        TB[i, j] = src | np.where(ex > eo, 4, 0).astype(np.uint8) | np.where(fx > fo, 8, 0).astype(np.uint8)
    ops, i, j, state = [], n, m, 0
    while i > 0 or j > 0:
        b = int(TB[i, j])
        if state == 0:
            if b & 3 == 0:
                ops.append(OP_M)
                i, j = i - 1, j - 1
            else:
                state = b & 3
        elif state == 1:
            ops.append(OP_D)
            state = 1 if b & 4 else 0
            i -= 1
        else:
            ops.append(OP_I)
            state = 2 if b & 8 else 0
            j -= 1
    return ops[::-1]


def left_align(ops, R, Q, rs, qs):
    ops = list(ops)
    ri, qj, c = rs, qs, 0
    while c < len(ops):
        op = ops[c]
        if op == OP_M:
            ri, qj, c = ri + 1, qj + 1, c + 1
            continue
        e = c
        while e < len(ops) and ops[e] == op:
            e += 1
        ln = e - c
        while c > 1 and ops[c - 1] == OP_M and R[ri - 1] == Q[qj - 1] and \
                (R[ri - 1] == R[ri + ln - 1] if op == OP_D else Q[qj - 1] == Q[qj + ln - 1]):
            ops[e - 1], ops[c - 1] = OP_M, op
            c, e, ri, qj = c - 1, e - 1, ri - 1, qj - 1
        if op == OP_D:
            ri += ln
        else:
            qj += ln
        c = e
    return ops, ri, qj


def split_divergent(anc, R, Q, o):
    """the alignment's gaps filled by gap_dp; a gap ends the alignment when its poor-scoring stretch is longer than break_len: the
    columns after the one where the score along the gap was best, plus the matching bases it takes to win the loss back
    -> [(anchors, gap columns)] pieces"""
    pieces, cur, gaps = [], [anc[0]], []
    for x, y in zip(anc, anc[1:]):
        ops = gap_dp(R[x[4] + x[5]:y[4]], Q[x[3] + x[5]:y[3]], o)
        sc = best = at = 0
        ri, qj = x[4] + x[5], x[3] + x[5]
        for c, op in enumerate(ops):
            if op == OP_M:
                sc += o["match"] if R[ri] == Q[qj] else -o["mismatch"]
                ri, qj = ri + 1, qj + 1
            else:
                sc -= (o["gap_open"] if c == 0 or ops[c - 1] != op else 0) + o["gap_extend"]
                ri, qj = (ri + 1, qj) if op == OP_D else (ri, qj + 1)
            if sc > best:
                best, at = sc, c + 1
        if len(ops) - at + (best - sc + o["match"] - 1) // o["match"] > o["break_len"]:
            pieces.append((cur, gaps))
            cur, gaps = [y], []
        else:
            cur.append(y)
            gaps.append(ops)
    pieces.append((cur, gaps))
    return pieces


def extend_end(R, Q, r, q, side, h0, o, lim=None):
    """ksw_extend2 (the project's C restatement, oracle/qmo_ksw.c) from reference position r / query position q, leftwards
    (side 0: over the reversed sequences) or rightwards, zdrop and band break_len, in windows of at most 511 query bases, again
    while an extension reaches the end of its window with sequence left -> [(r, q)] from the start point, one per window"""
    from oracle import qmo_py
    kopt = qmo_py.default_opt()
    kopt.a, kopt.b, kopt.o_del, kopt.o_ins = o["match"], o["mismatch"], o["gap_open"], o["gap_open"]
    kopt.e_del, kopt.e_ins, kopt.zdrop = o["gap_extend"], o["gap_extend"], o["break_len"]
    pts = [(r, q)]
    while True:
        lr, lq = lim if lim else ((len(R), len(Q)) if side else (0, 0))
        rem_q, rem_r = (lq - q, lr - r) if side else (q - lq, r - lr)
        qw = min(511, rem_q)
        tw = min(rem_r, qw + o["break_len"])
        if qw == 0 or tw == 0:
            return pts
        qs = Q[q:q + qw] if side else Q[q - qw:q][::-1]
        ts = R[r:r + tw] if side else R[r - tw:r][::-1]
        (score, qle, tle, _, _, _), _ = qmo_py.ksw_extend2(qs, ts, h0, o["break_len"], 0, kopt)
        if qle == 0 and tle == 0:
            return pts
        q, r = (q + qle, r + tle) if side else (q - qle, r - tle)
        pts.append((r, q))
        h0 = score
        if not ((qle == qw and qw < rem_q) or (tle == tw and tw < rem_r)):
            return pts


def assemble(anc, gaps, lim0, lim1, s, qc, rc, R, Q, ql, o):
    """one alignment: extended ends, columns, left-aligned indels, counts"""
    f, l = anc[0], anc[-1]
    left = extend_end(R, Q, f[4], f[3], 0, max(1, f[5] * o["match"]), o, lim0)
    right = extend_end(R, Q, l[4] + l[5], l[3] + l[5], 1, max(1, l[5] * o["match"]), o, lim1)
    r0, q0 = left[-1]
    head, tail = [], []
    for (ra, qa), (rb_, qb) in zip(left, left[1:]):             # each window's stretch aligned globally, outermost first
        head = gap_dp(R[rb_:ra], Q[qb:qa], o) + head
    for (ra, qa), (rb_, qb) in zip(right, right[1:]):
        tail = tail + gap_dp(R[ra:rb_], Q[qa:qb], o)
    c = 0
    while c < len(head) and head[c] != OP_M:                      # indel columns at the outer ends are dropped
        r0, q0 = (r0 + 1, q0) if head[c] == OP_D else (r0, q0 + 1)
        c += 1
    head = head[c:]
    while tail and tail[-1] != OP_M:
        tail.pop()
    ops = list(head)
    for g, x in enumerate(anc):
        ops += [OP_M] * x[5]
        if g + 1 < len(anc):
            ops += gaps[g]
    ops += tail
    ops, re, qe = left_align(ops, R, Q, r0, q0)
    ri, qj, matches, edits = r0, q0, 0, 0
    for op in ops:
        if op == OP_M:
            if R[ri] == Q[qj]:
                matches += 1
            else:
                edits += 1
            ri, qj = ri + 1, qj + 1
        else:
            edits += 1
            ri, qj = (ri + 1, qj) if op == OP_D else (ri, qj + 1)
    return dict(s=s, qc=qc, rc=rc, rs=r0, re=re, qs=q0, qe=qe, ops=ops, matches=matches, edits=edits,
                fqs=ql - qe if s else q0, fqe=ql - q0 if s else qe)


def _chain_filter(al, by):
    key = (lambda a: a["qc"]) if by else (lambda a: a["rc"])
    beg = (lambda a: a["fqs"]) if by else (lambda a: a["rs"])
    end = (lambda a: a["fqe"]) if by else (lambda a: a["re"])
    idx = sorted(range(len(al)), key=lambda x: (key(al[x]), beg(al[x]), end(al[x])))
    keep = set()
    g0 = 0
    while g0 < len(idx):
        g1 = g0
        while g1 < len(idx) and key(al[idx[g1]]) == key(al[idx[g0]]):
            g1 += 1
        grp = [al[x] for x in idx[g0:g1]]
        best = [a["matches"] for a in grp]
        pred = [-1] * len(grp)
        for j, b in enumerate(grp):
            for i in range(j):
                a = grp[i]
                if beg(a) < beg(b) and end(a) < end(b) and best[i] + b["matches"] > best[j]:
                    best[j], pred[j] = best[i] + b["matches"], i
        e = max(range(len(grp)), key=lambda j: (best[j], -j))
        while e >= 0:
            keep.add(idx[g0 + e])
            e = pred[e]
        g0 = g1
    return [a for x, a in enumerate(al) if x in keep]


def genome_diff(ref, qry, opt=None):
    """-> (rows, alignments): lists of dicts with the fields of GDIFF_ROW_DTYPE / GDIFF_ALN_DTYPE"""
    o = dict(default_opt(), **(opt or {}))
    k = o["min_match"]
    A = anchors(ref, qry, k)
    rcon, qcon = _contigs(ref), _contigs(qry)
    qstr = {}
    for qc, (qo, ql) in enumerate(qcon):
        f = qry.codes[qo:qo + ql]
        qstr[qc, 0], qstr[qc, 1] = f, (3 - f[::-1]).astype(np.uint8)
    al = []
    g0 = 0
    while g0 < len(A):
        g1 = g0
        while g1 < len(A) and A[g1][:3] == A[g0][:3]:
            g1 += 1
        grp = A[g0:g1]
        cl = sorted(clusters(grp, o), key=lambda c: (c[0][4], c[0][3]))
        nxt, has_prev = [-1] * len(cl), [False] * len(cl)
        for i in range(len(cl)):
            t = cl[i][-1]
            for j in range(i + 1, len(cl)):
                if has_prev[j]:
                    continue
                h = _trim_after(t, cl[j][0])
                if h is None:
                    continue
                if h[4] - (t[4] + t[5]) <= o["break_len"] and h[3] - (t[3] + t[5]) <= o["break_len"]:
                    nxt[i], has_prev[j] = j, True
                    cl[j][0] = h
                    break
        pieces = []
        s, qc, rc = grp[0][0], grp[0][1], grp[0][2]
        rb, rl = rcon[rc]
        R = ref.codes[rb:rb + rl]
        Q = qstr[qc, s]
        for i in range(len(cl)):
            if has_prev[i]:
                continue
            anc, c = [], i
            while c >= 0:
                anc += cl[c]
                c = nxt[c]
            pieces += split_divergent(anc, R, Q, o)
        # ends extend no further than the nearest piece of the group ahead of them on both sequences
        for anc, gaps in pieces:
            f, l = anc[0], anc[-1]
            ahead = [(b[0][4], b[0][3]) for b, _ in pieces if b is not anc and b[0][4] >= l[4] + l[5] and b[0][3] >= l[3] + l[5]]
            behind = [(b[-1][4] + b[-1][5], b[-1][3] + b[-1][5]) for b, _ in pieces
                      if b is not anc and b[-1][4] + b[-1][5] <= f[4] and b[-1][3] + b[-1][5] <= f[3]]
            al.append(assemble(anc, gaps, max(behind) if behind else None, min(ahead) if ahead else None, s, qc, rc, R, Q,
                               qcon[qc][1], o))
        g0 = g1
    al = _chain_filter(al, 0)
    al = _chain_filter(al, 1)
    al.sort(key=lambda a: (a["rc"], a["rs"], a["re"], a["qc"], a["s"], a["qs"]))
    rows = []
    for a in al:
        rb, rl = rcon[a["rc"]]
        R = ref.codes[rb:rb + rl]
        Q = qstr[a["qc"], a["s"]]
        ql = qcon[a["qc"]][1]
        fwd = (lambda y: ql - y + 1) if a["s"] else (lambda y: y)
        mine = []
        ri, qj = a["rs"], a["qs"]
        for op in a["ops"]:
            if op == OP_M:
                if R[ri] != Q[qj]:
                    mine.append((ri + 1, ACGT[R[ri]], ACGT[Q[qj]], fwd(qj + 1)))
                ri, qj = ri + 1, qj + 1
            elif op == OP_D:
                mine.append((ri + 1, ACGT[R[ri]], ".", fwd(qj)))
                ri += 1
            else:
                mine.append((ri, ".", ACGT[Q[qj]], fwd(qj + 1)))
                qj += 1
        for x, (p1, sr, sq, p2) in enumerate(mine):
            b = min(p1 - (a["rs"] + 1), a["re"] - p1)
            if x > 0:
                b = min(b, p1 - mine[x - 1][0])
            if x + 1 < len(mine):
                b = min(b, mine[x + 1][0] - p1)
            rows.append(dict(p1=p1, p2=p2, buff=b, dist=min(p1 - 1, rl - p1, p2 - 1, ql - p2), sub_r=sr, sub_q=sq, frm_r=1,
                             frm_q=-1 if a["s"] else 1, rid=a["rc"], qid=a["qc"]))
    kept = []
    for w in rows:
        if o["flags"] & _lib.GDIFF_NO_INDELS and "." in (w["sub_r"], w["sub_q"]):
            continue
        if not o["flags"] & _lib.GDIFF_KEEP_AMBIGUOUS:
            cr = sum(1 for a in al if a["rc"] == w["rid"] and a["rs"] < w["p1"] <= a["re"])
            cq = sum(1 for a in al if a["qc"] == w["qid"] and a["fqs"] < w["p2"] <= a["fqe"])
            if cr > 1 or cq > 1:
                continue
        kept.append(w)
    kept.sort(key=lambda w: (w["rid"], w["p1"]))
    alns = [dict(rid=a["rc"], qid=a["qc"], rs=a["rs"] + 1, re=a["re"], qs=a["fqe"] if a["s"] else a["fqs"] + 1,
                 qe=a["fqs"] + 1 if a["s"] else a["fqe"], strand=-1 if a["s"] else 1, edits=a["edits"], matches=a["matches"])
            for a in al]
    return kept, alns


def rows_array(rows):
    """oracle rows as a GDIFF_ROW_DTYPE array (comparable with Context.genome_diff)"""
    out = np.zeros(len(rows), _lib.GDIFF_ROW_DTYPE)
    for i, w in enumerate(rows):
        for f in ("p1", "p2", "buff", "dist", "frm_r", "frm_q", "rid", "qid"):
            out[i][f] = w[f]
        out[i]["sub_r"], out[i]["sub_q"] = w["sub_r"].encode(), w["sub_q"].encode()
    return out


def alns_array(alns):
    out = np.zeros(len(alns), _lib.GDIFF_ALN_DTYPE)
    for i, a in enumerate(alns):
        for f, v in a.items():
            out[i][f] = v
    return out


def snps_lines(rows, ref, qry):
    """the 12 tab-separated columns of show-snps -CTHlr: P1 SUB SUB P2 BUFF DIST LEN_R LEN_Q FRM FRM TAG_R TAG_Q"""
    return ["\t".join(map(str, (w["p1"], w["sub_r"], w["sub_q"], w["p2"], w["buff"], w["dist"], ref.lens[w["rid"]], qry.lens[w["qid"]],
                                w["frm_r"], w["frm_q"], ref.names[w["rid"]], qry.names[w["qid"]]))) for w in rows]


def vcf_records(rows, ref, qry):
    """mummer2vcf.py -n: SNP rows collapsed per position (ALTs joined by ','), runs of indel rows merged with the anchor base
    first.  Returns the data lines."""
    off = np.concatenate([[0], np.cumsum(ref.lens)]).astype(np.int64)
    base = lambda rid, p1: ACGT[ref.codes[off[rid] + p1 - 1]]
    out, i = [], 0
    while i < len(rows):
        w = rows[i]
        rname, qname = ref.names[w["rid"]], qry.names[w["qid"]]
        j = i + 1
        if w["sub_r"] != "." and w["sub_q"] != ".":
            alts = [w["sub_q"]]
            while j < len(rows) and rows[j]["rid"] == w["rid"] and rows[j]["p1"] == w["p1"] and "." not in (rows[j]["sub_r"], rows[j]["sub_q"]):
                if rows[j]["sub_q"] not in alts:
                    alts.append(rows[j]["sub_q"])
                j += 1
            pos, r, a, typ = w["p1"], w["sub_r"], ",".join(alts), "SNV"
        elif w["sub_q"] == ".":                           # deletion: consecutive reference bases, one query position
            while j < len(rows) and rows[j]["rid"] == w["rid"] and rows[j]["sub_q"] == "." and rows[j]["p2"] == w["p2"] and \
                    rows[j]["p1"] == rows[j - 1]["p1"] + 1:
                j += 1
            pos = w["p1"] - 1
            r = base(w["rid"], pos) + "".join(x["sub_r"] for x in rows[i:j])
            a, typ = base(w["rid"], pos), "INDEL"
        else:                                             # insertion: one reference position, consecutive query bases
            while j < len(rows) and rows[j]["rid"] == w["rid"] and rows[j]["sub_r"] == "." and rows[j]["p1"] == w["p1"] and \
                    abs(rows[j]["p2"] - rows[j - 1]["p2"]) == 1:
                j += 1
            pos = w["p1"]
            r = base(w["rid"], pos)
            a, typ = r + "".join(x["sub_q"] for x in rows[i:j]), "INDEL"
        out.append(f"{rname}\t{pos}\t.\t{r}\t{a}\t30\tPASS\tDP=30;REF1={rname};REF2={qname};ORIG={qname}:{w['p2']};TYPE={typ}")
        i = j
    return out
