"""ORACLE (test infrastructure) -- a second restatement of how bwa-mem turns a hit into a record (bwamem.c mem_reg2aln, bwa.c
bwa_gen_cigar2; SURVEY.md A.4): the band guessed from the score, up to three global alignments with a doubling band, the ungapped
fast path, reverse-strand hits aligned on the forward strand so that indels sit leftmost there, NM, leading / trailing deletions
squeezed out, soft clips, the forward-strand position.  The global alignment itself is oracle/ksw_py.py's whole-matrix one.
To be diffed against oracle/qmo_mem.c reg_to_aln."""
from oracle import ksw_py


def _band_from_score(l1, l2, score, a, gap_open, gap_ext):
    if l1 == l2 and l1 * a - score < 2 * (gap_open + gap_ext - a):
        return 0
    w = int((min(l1, l2) * a - score - gap_open) / gap_ext + 2.)
    return max(w, abs(l1 - l2))


def hit_to_record(doubled, l_pac, offs, read, hit, a=1, b=4, o_del=6, e_del=1, o_ins=6, e_ins=1, w=100):
    """doubled = forward strand + its reverse complement (base codes); read = the read as sequenced; hit = dict(rb, re, qb, qe,
    truesc, w).  -> dict(rid, pos, rev, cigar [(op, len)] with 0 M 1 I 2 D 4 S, nm)"""
    qb, qe, rb, re = hit["qb"], hit["qe"], hit["rb"], hit["re"]
    lq, lr = qe - qb, re - rb
    band = max(_band_from_score(lq, lr, hit["truesc"], a, o_del, e_del), _band_from_score(lq, lr, hit["truesc"], a, o_ins, e_ins))
    if band > w:
        band = min(band, hit["w"])
    rev = rb >= l_pac
    q, t = [int(x) for x in read[qb:qe]], [int(x) for x in doubled[rb:re]]
    if rev:
        q, t = q[::-1], t[::-1]
    last, tries = None, 0
    while True:
        band = min(band, 4 * w)
        if lq == lr and band == 0:
            score, ops = sum(ksw_py.score(a, b, x, y) for x, y in zip(t, q)), [(0, lq)]
        else:
            half = (lq + 1) >> 1
            reach = max(1, int((half * a - o_ins) / e_ins + 1.), int((half * a - o_del) / e_del + 1.))
            eff = max(min((reach + abs(lr - lq) + 1) >> 1, band), abs(lr - lq) + 3)
            score, ops = ksw_py.ksw_global2(q, t, eff, a, b, o_del, e_del, o_ins, e_ins)
        if score == last or band == 4 * w:
            break
        last = score
        band <<= 1
        tries += 1
        if not (tries < 3 and score < hit["truesc"] - a):
            break
    # edit distance over the whole path, before anything is trimmed; a leading or trailing deletion is not counted (bwa_gen_cigar2
    # leaves it out of NM and MD, and mem_reg2aln then squeezes it out of the CIGAR)
    nm, i, k = 0, 0, 0
    for x, (op, ln) in enumerate(ops):
        if op == 0:
            nm += sum(1 for j in range(ln) if q[k + j] != t[i + j] or q[k + j] > 3 or t[i + j] > 3)
            i += ln
            k += ln
        elif op == 1:
            nm += ln
            k += ln
        else:
            nm += ln if 0 < x < len(ops) - 1 else 0
            i += ln
    # (both sequences were turned round for a reverse-strand hit, so the path already reads along the forward strand, as a BAM
    # record wants it: bwa turns only the query back afterwards.  SURVEY.md A.4's "reverse the CIGAR after" is not what happens --
    # tests/drvutil.check_bam_records rebuilds the reference from SEQ + CIGAR + MD and would not do so with a reversed CIGAR.)
    pos = (2 * l_pac - re) if rev else rb
    if ops and ops[0][0] == 2:
        pos += ops[0][1]
        ops = ops[1:]
    elif ops and ops[-1][0] == 2:
        ops = ops[:-1]
    head, tail = (len(read) - qe, qb) if rev else (qb, len(read) - qe)
    cigar = ([(4, head)] if head else []) + list(ops) + ([(4, tail)] if tail else [])
    rid = max(c for c in range(len(offs) - 1) if pos >= offs[c])
    return dict(rid=rid, pos=pos - int(offs[rid]), rev=rev, cigar=cigar, nm=nm)
