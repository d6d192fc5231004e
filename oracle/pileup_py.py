"""ORACLE (test infrastructure) -- a SECOND, independently formulated restatement of the per-column counting of
`bcftools mpileup -B` (reference call site rules/vcfcall.smk:115; spec SURVEY.md A.8-A.9), written to be diffed against
oracle/qmo_pileup.c (SURVEY.md Appendix A: "write two independent restatements and diff them" -- neither can be pinned to
bcftools, which is absent from the image).

Where qmo_pileup.c walks a pair's two CIGARs side by side with two cursors, this one goes the way htslib does: every read
becomes a list of pileup entries (reference position -> query position / deleted), the mate-overlap rewrite looks the second
mate's positions up in a hash of the first's (htslib overlap_push / tweak_overlap_quality), and the tensor is tallied from the
entries at the end.  Pure Python: for a few thousand pairs."""
import numpy as np

NCH = 16
M, I, D, N_, S = 0, 1, 2, 3, 4


def _entries(aln, L):
    """-> (cols, ins_after, del_after, first_col): cols = [(ref_pos, query_pos or None when the base is deleted)] in SEQ
    orientation; ins_after / del_after = reference positions of the aligned base in front of an insertion / a deletion"""
    cols, ins_after, del_after = [], [], []
    q, r, last = 0, int(aln["pos"]), None
    for c in aln["cigar"][:int(aln["n_cigar"])]:
        op, ln = int(c) & 15, int(c) >> 4
        if op == M:
            cols.extend((r + j, q + j) for j in range(ln))
            q += ln
            r += ln
            last = r - 1
        elif op == I:
            if last is not None:
                ins_after.append(last)
            q += ln
        elif op == S:
            q += ln
        elif op == D:
            if last is not None:
                del_after.append(last)
            cols.extend((r + j, None) for j in range(ln))
            r += ln
        elif op == N_:
            r += ln
    assert q == L, (q, L)
    aligned = [p for p, x in cols if x is not None]
    return cols, ins_after, del_after, (aligned[0] if aligned else None)


def _admitted(aln, min_mapq, count_orphans):
    f = int(aln["flag"])
    if f & (0x4 | 0x100 | 0x200 | 0x400):
        return False
    if int(aln["n_cigar"]) in (0, 255):                    # no alignment stored / CIGAR beyond the record's room
        return False
    if int(aln["mapq"]) < min_mapq:
        return False
    if (f & 0x1) and not (f & 0x2) and not count_orphans:
        return False
    return True


def count_tensor(ref_offs, l_pac, alns, codes, quals, lens, min_mapq=0, min_bq=13, count_orphans=False, ignore_overlaps=False):
    """-> int32 [l_pac, 16], channels as include/quasimodo_b200.h documents them"""
    counts = np.zeros((l_pac, NCH), dtype=np.int64)
    comp = np.array([3, 2, 1, 0, 4], dtype=np.uint8)
    for pi in range(len(alns) // 2):
        reads = []
        for e in (0, 1):
            a, L = alns[2 * pi + e], int(lens[2 * pi + e])
            if not _admitted(a, min_mapq, count_orphans):
                reads.append(None)
                continue
            seq, ql = np.minimum(codes[2 * pi + e, :L], 4), quals[2 * pi + e, :L].astype(np.int64)
            if int(a["flag"]) & 0x10:                      # BAM stores the reverse strand's read reverse-complemented
                seq, ql = comp[seq[::-1]], ql[::-1]
            cols, ia, da, first = _entries(a, L)
            reads.append(dict(a=a, L=L, seq=seq, q=ql.copy(), cols=cols, ia=ia, da=da, first=first, rev=bool(int(a["flag"]) & 0x10)))
        x, y = reads
        if (not ignore_overlaps and x is not None and y is not None and int(x["a"]["rid"]) == int(y["a"]["rid"])
                and (int(x["a"]["flag"]) & 0x2) and not (int(x["a"]["flag"]) & 0x8)
                and abs(int(x["a"]["tlen"])) < 2 * x["L"] and abs(int(y["a"]["tlen"])) < 2 * y["L"]):
            # the mate the sorted BAM delivers first is hashed, the other one is matched against it
            kx, ky = (int(x["a"]["pos"]), x["rev"]), (int(y["a"]["pos"]), y["rev"])
            first, second = (x, y) if kx <= ky else (y, x)
            where = {p: qp for p, qp in first["cols"] if qp is not None}
            for p, qb in second["cols"]:
                if qb is None or p not in where:
                    continue
                qa = where[p]
                if first["seq"][qa] == second["seq"][qb]:
                    first["q"][qa] = min(200, first["q"][qa] + second["q"][qb])
                    second["q"][qb] = 0
                elif first["q"][qa] >= second["q"][qb]:
                    first["q"][qa] = int(0.8 * first["q"][qa])
                    second["q"][qb] = 0
                else:
                    second["q"][qb] = int(0.8 * second["q"][qb])
                    first["q"][qa] = 0
        for rd in reads:
            if rd is None:
                continue
            base = int(ref_offs[int(rd["a"]["rid"])])
            strand = 6 if rd["rev"] else 0
            if rd["first"] is not None:
                counts[base + rd["first"], 15] += 1
            for p, qp in rd["cols"]:
                if qp is None:
                    counts[base + p, 11 if rd["rev"] else 5] += 1
                    continue
                counts[base + p, 14] += 1
                if rd["q"][qp] >= min_bq:
                    counts[base + p, strand + int(rd["seq"][qp])] += 1
            for p in rd["ia"]:
                counts[base + p, 12] += 1
            for p in rd["da"]:
                counts[base + p, 13] += 1
    return counts.astype(np.int32)


def indel_alleles(ref_offs, alns, codes, lens, min_mapq=0, count_orphans=False, seq_bases=11):
    """The indel allele tally (include/quasimodo_b200.h: anchor = the aligned base in front of the event; an insertion is told
    apart by its first `seq_bases` bases on the forward strand of the reference, an N among them flagged and stored as A; lengths
    above 255 clamped) from the BAM view of every admitted read.
    -> {(rid, anchor pos, type 0 ins / 1 del, length, bases packed 2 bits each, has_n): [forward reads, reverse reads]}"""
    comp = np.array([3, 2, 1, 0, 4], dtype=np.uint8)
    table = {}
    for r in range(len(alns)):
        a, L = alns[r], int(lens[r])
        if not _admitted(a, min_mapq, count_orphans):
            continue
        rev = bool(int(a["flag"]) & 0x10)
        seq = np.minimum(codes[r, :L], 4)
        if rev:
            seq = comp[seq[::-1]]
        q, ref_pos, anchor = 0, int(a["pos"]), None
        for c in a["cigar"][:int(a["n_cigar"])]:
            op, ln = int(c) & 15, int(c) >> 4
            if op == M:
                q += ln
                ref_pos += ln
                anchor = ref_pos - 1
            elif op == S:
                q += ln
            elif op in (I, D):
                if anchor is not None:
                    ins = [int(b) for b in seq[q:q + min(ln, seq_bases)]] if op == I else []
                    packed = sum((b if b < 4 else 0) << (2 * j) for j, b in enumerate(ins))
                    key = (int(a["rid"]), anchor, int(op == D), min(ln, 255), packed, int(any(b > 3 for b in ins)))
                    table.setdefault(key, [0, 0])[1 if rev else 0] += 1
                if op == I:
                    q += ln
                else:
                    ref_pos += ln
    return table


def mpileup_text(ref_codes, ref_offs, ref_lens, contig_names, alns, codes, quals, lens, min_mapq=0, min_bq=13, count_orphans=False,
                 ignore_overlaps=False):
    """The text pileup of `samtools mpileup` (rules/vcfcall.smk:39; SURVEY.md A.10) with -B semantics, assembled column by column
    from per-read pileup entries -- a second formulation next to oracle/qmo_pileup.c qmo_mpileup_text.  -> bytes"""
    comp = np.array([3, 2, 1, 0, 4], dtype=np.uint8)
    n = len(alns)
    view = [None] * n
    for r in range(n):
        a, L = alns[r], int(lens[r])
        if not _admitted(a, min_mapq, count_orphans):
            continue
        rev = bool(int(a["flag"]) & 0x10)
        seq, ql = np.minimum(codes[r, :L], 4), quals[r, :L].astype(np.int64)
        if rev:
            seq, ql = comp[seq[::-1]], ql[::-1]
        cols, _, _, _ = _entries(a, L)
        view[r] = dict(a=a, L=L, rev=rev, seq=seq, q=ql.copy(), cols=cols)
    if not ignore_overlaps:
        for p in range(n // 2):
            x, y = view[2 * p], view[2 * p + 1]
            if x is None or y is None or int(x["a"]["rid"]) != int(y["a"]["rid"]):
                continue
            if not (int(x["a"]["flag"]) & 0x2) or (int(x["a"]["flag"]) & 0x8):
                continue
            if abs(int(x["a"]["tlen"])) >= 2 * x["L"] or abs(int(y["a"]["tlen"])) >= 2 * y["L"]:
                continue
            first, second = (x, y) if (int(x["a"]["pos"]), x["rev"]) <= (int(y["a"]["pos"]), y["rev"]) else (y, x)
            at = {pos: qp for pos, qp in first["cols"] if qp is not None}
            for pos, qb in second["cols"]:
                if qb is None or pos not in at:
                    continue
                qa = at[pos]
                if first["seq"][qa] == second["seq"][qb]:
                    first["q"][qa], second["q"][qb] = min(200, first["q"][qa] + second["q"][qb]), 0
                elif first["q"][qa] >= second["q"][qb]:
                    first["q"][qa], second["q"][qb] = int(0.8 * first["q"][qa]), 0
                else:
                    first["q"][qa], second["q"][qb] = 0, int(0.8 * second["q"][qb])
    # reads reach a column in the order of the sorted BAM: (contig, position, strand), input order on ties
    order = sorted((r for r in range(n) if view[r] is not None),
                   key=lambda r: (int(view[r]["a"]["rid"]), int(view[r]["a"]["pos"]), view[r]["rev"], r))
    columns = {}                                           # (rid, pos) -> [bases string parts, quality chars]; every covered column has an entry
    for r in order:
        v = view[r]
        a, L, rid = v["a"], v["L"], int(v["a"]["rid"])
        ops = [(int(c) & 15, int(c) >> 4) for c in a["cigar"][:int(a["n_cigar"])]]
        # htslib resolve_cigar2 gives a deleted base the query cursor at its D operation (p->qpos = s->y): the first query
        # base behind the deletion in read order, whatever operation holds it (M, I or S), or l_qseq when the read ends there.
        # samtools takes that base's quality (0 past the end) and prints an insertion as the bases at qpos + 1 .. qpos + n.
        follows = {}                                       # reference position of the last base of an M / D run -> (indel after it, its qpos)
        del_q = {}                                         # reference position of a deleted base -> its qpos
        q, pos = 0, int(a["pos"])
        for i, (op, ln) in enumerate(ops):
            if op == D:
                del_q.update((pos + j, q) for j in range(ln))
            if op in (M, D):
                pos += ln
                if i + 1 < len(ops) and ops[i + 1][0] in (I, D):
                    follows[pos - 1] = (ops[i + 1][0], ops[i + 1][1], q + ln - 1 if op == M else q)
            if op in (M, I, S):
                q += ln
        last = pos - 1
        letters = "acgtn" if v["rev"] else "ACGTN"
        for cpos, qp in v["cols"]:
            col = columns.setdefault((rid, cpos), [[], []])
            qq = qp if qp is not None else del_q[cpos]
            qual = int(v["q"][qq]) if qq < L else 0
            if qual < min_bq:
                continue
            s = ""
            if cpos == int(a["pos"]):
                s += "^" + chr(126 if int(a["mapq"]) > 93 else int(a["mapq"]) + 33)
            if qp is None:
                s += "*"
            else:
                b = int(v["seq"][qp])
                s += ("," if v["rev"] else ".") if b < 4 and b == int(ref_codes[int(ref_offs[rid]) + cpos]) else letters[b]
            if cpos in follows:
                kind, ln, qpos = follows[cpos]
                if kind == I:
                    s += "+%d" % ln + "".join(letters[int(v["seq"][qpos + j])] if qpos + j < L else letters[4] for j in range(1, ln + 1))
                else:
                    s += "-%d" % ln + "".join(letters[int(ref_codes[int(ref_offs[rid]) + cpos + 1 + j])] if cpos + 1 + j < int(ref_lens[rid]) else letters[4]
                                              for j in range(ln))
            if cpos == last:
                s += "$"
            col[0].append(s)
            col[1].append(chr(min(qual + 33, 126)))
    out = []
    for (rid, cpos) in sorted(columns):
        bases, qs = columns[(rid, cpos)]
        out.append("%s\t%d\t%s\t%d\t%s\t%s\n" % (contig_names[rid], cpos + 1, "ACGT"[int(ref_codes[int(ref_offs[rid]) + cpos])], len(qs),
                                               "".join(bases) or "*", "".join(qs) or "*"))
    return "".join(out).encode()
