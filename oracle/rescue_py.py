"""ORACLE (test infrastructure) -- a second restatement of bwa-mem's mate rescue (bwamem_pair.c mem_matesw and its loop in
mem_sam_pe; SURVEY.md A.6) and of the redundancy filter it ends with (bwamem.c mem_sort_dedup_patch without the patch step), to be
diffed against oracle/qmo_mem.c.  The local alignment itself is the C ksw_align2 (already diffed against oracle/ksw_py.py); what is
restated here is which windows are searched, in what order, what a hit becomes and how the mate's hit list changes.
Limits shared with oracle and product: a window longer than 4,096 bases is not searched, a list holds 16 hits."""
from oracle import qmo_py

MAX_REGS, MAX_WINDOW, MAX_MATESW = 16, 4096, 50


def remove_redundant(hits, max_chain_gap=10000, redun=0.95):
    """hits that overlap a better hit by more than 95 % on read and reference go; then (score desc, rb, qb) and exact twins go"""
    hits = sorted(hits, key=lambda h: h["re"])             # stable: ties keep their order
    for i in range(1, len(hits)):
        p = hits[i]
        for j in range(i - 1, -1, -1):
            q = hits[j]
            if not (p["rid"] == q["rid"] and p["rb"] < q["re"] + max_chain_gap):
                break
            if q["qe"] == q["qb"]:
                continue
            on_ref = q["re"] - p["rb"]
            on_read = q["qe"] - p["qb"] if q["qb"] < p["qb"] else p["qe"] - q["qb"]
            if on_ref > redun * min(q["re"] - q["rb"], p["re"] - p["rb"]) and on_read > redun * min(q["qe"] - q["qb"], p["qe"] - p["qb"]):
                if p["score"] < q["score"]:
                    p["qe"] = p["qb"]
                    break
                q["qe"] = q["qb"]
    hits = sorted((h for h in hits if h["qe"] > h["qb"]), key=lambda h: (-h["score"], h["rb"], h["qb"]))
    out = []
    for h in hits:
        if out and (h["score"], h["rb"], h["qb"]) == (out[-1]["score"], out[-1]["rb"], out[-1]["qb"]):
            continue
        out.append(h)
    return out


def _orientation(l_pac, b1, b2):
    r1, r2 = b1 >= l_pac, b2 >= l_pac
    p2 = b2 if r1 == r2 else 2 * l_pac - 1 - b2
    return (0 if r1 == r2 else 1) ^ (0 if p2 > b1 else 3), abs(p2 - b1)


def rescue_from(doubled, l_pac, offs, clens, pes, anchor, mate_seq, mate_hits, opt, counters):
    """one anchoring hit: every orientation with a model in which the mate has no hit at a proper distance is searched"""
    done = [bool(pes[r]["failed"]) for r in range(4)]
    for h in mate_hits:
        r, dist = _orientation(l_pac, anchor["rb"], h["rb"])
        if int(pes[r]["low"]) <= dist <= int(pes[r]["high"]):
            done[r] = True
    if all(done):
        return mate_hits
    L = len(mate_seq)
    searched = 0
    for r in range(4):
        if done[r]:
            continue
        opposite, after = (r >> 1) != (r & 1), not (r >> 1)
        lo, hi = (anchor["rb"] + int(pes[r]["low"]), anchor["rb"] + int(pes[r]["high"])) if after else \
                 (anchor["rb"] - int(pes[r]["high"]), anchor["rb"] - int(pes[r]["low"]))
        rb, re = (lo - L, hi) if opposite else (lo, hi + L)
        rb, re = max(rb, 0), min(re, 2 * l_pac)
        rid = -1
        if rb < re:                                        # the contig (and strand) of the window's middle bounds the window
            mid = (rb + re) >> 1
            rev = mid >= l_pac
            f = 2 * l_pac - 1 - mid if rev else mid
            rid = max(c for c in range(len(clens)) if f >= offs[c])
            cb, ce = int(offs[rid]), int(offs[rid]) + int(clens[rid])
            if rev:
                cb, ce = 2 * l_pac - ce, 2 * l_pac - cb
            rb, re = max(rb, cb), min(re, ce)
        counters.setdefault("windows", []).append(re - rb if anchor["rid"] == rid else -1)     # (what the tests show they reach)
        if anchor["rid"] == rid and opt.min_seed_len <= re - rb <= MAX_WINDOW:
            seq = [(3 - int(c) if int(c) < 4 else 4) for c in mate_seq[::-1]] if opposite else [int(c) for c in mate_seq]
            (score, te, qe, score2, _, tb, qb), cells = qmo_py.ksw_align2(seq, doubled[rb:re], opt.min_seed_len * opt.a, opt)
            counters["cells"] += cells
            counters.setdefault("scores", []).append(score)
            if score >= opt.min_seed_len and qb >= 0:
                new = dict(rid=anchor["rid"], score=score, csub=score2,
                           qb=L - (qe + 1) if opposite else qb, qe=L - qb if opposite else qe + 1,
                           rb=2 * l_pac - (rb + te + 1) if opposite else rb + tb, re=2 * l_pac - (rb + tb) if opposite else rb + te + 1)
                at = next((i for i, h in enumerate(mate_hits) if h["score"] < score), len(mate_hits))
                mate_hits = (mate_hits[:at] + [new] + mate_hits[at:])[:MAX_REGS]
            searched += 1
        if searched:
            mate_hits = remove_redundant(mate_hits, opt.max_chain_gap, opt.mask_level_redun)
    counters["sw"] += searched
    return mate_hits


def rescue_pair(doubled, l_pac, offs, clens, pes, hits, seqs, opt, counters):
    """hits = [hits of mate 0, hits of mate 1] -> the two lists after rescue"""
    anchors = [[dict(h) for h in hs if h["score"] >= hs[0]["score"] - opt.pen_unpaired][:MAX_MATESW] for hs in hits]
    hits = [list(hits[0]), list(hits[1])]
    for m in (0, 1):
        for anchor in anchors[m]:
            hits[1 - m] = rescue_from(doubled, l_pac, offs, clens, pes, anchor, seqs[1 - m], hits[1 - m], opt, counters)
    return hits
