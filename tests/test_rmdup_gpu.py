"""GPU tests of duplicate marking of a BAM (`qm_driver rmdup`, qm_bam_mark_duplicates):

1. round trip: simulated pairs of BASELINE configs 1, 3 and 5 with duplicates added on purpose (pairs copied 1-4 times, with
   perturbed or with identical qualities) go through `sample --rmdup 1`; `rmdup` on its BAM (stale 0x400 flags) and on the BAM of
   a `sample` run without --rmdup gives identical records and `sample`'s metrics byte for byte; the records equal `sample`'s
   .rmdup.bam except in groups tied at the top score, and everywhere equal the rule restated below; the .bai finds every record;
2. hand-built records (clips, N / = / X, secondary and supplementary records, unmapped mates, missing mates, three primaries of
   a name, 0x200, reads over 512 bases, QUAL '*'): the verdict of every record equals oracle/dedup_py.py fed the units in id order;
3. with the name hash cut to 1, 2 and 7 bits the verdicts are the 64-bit ones;
4. chain: `pileup` on the output of `rmdup` gives the counts and VCF of `pileup` on `sample`'s .rmdup.bam (no score ties)."""
import ctypes as C
import struct
from collections import defaultdict

import numpy as np
import pytest

from tests import bamio, drvutil
from tests.test_bam_input_gpu import encode

pytestmark = pytest.mark.gpu

CLIP, SPAN = (4, 5), (0, 2, 3, 7, 8)


# ---- the rule for a file, restated over parsed records (dicts: name flag rid pos cigar [(op, len)] qual) ---------------------
def placed(r):
    return not (r["flag"] & 0x4) and r["rid"] >= 0 and len(r["cigar"]) > 0


def oracle_cigar(cig):
    """the CIGAR in the terms oracle/dedup_py.py reads (S at the ends, M / D inside): clips before the first and after the last
    aligned operation merge into one S each, the reference span becomes one M -- the same end"""
    body = [i for i, (op, _) in enumerate(cig) if op not in CLIP]
    first, last = (body[0], body[-1]) if body else (len(cig), -1)
    lead = sum(ln for i, (_, ln) in enumerate(cig) if i < first)
    trail = sum(ln for i, (_, ln) in enumerate(cig) if i > last >= 0)
    span = sum(ln for op, ln in cig if op in SPAN)
    return [(4, lead)] * (lead > 0) + [(0, span)] + [(4, trail)] * (trail > 0)


def end_of(r):
    cig = oracle_cigar(r["cigar"])
    lead = cig[0][1] if cig[0][0] == 4 else 0
    trail = cig[-1][1] if cig[-1][0] == 4 and len(cig) > 1 else 0
    rev = bool(r["flag"] & 0x10)
    span = sum(ln for op, ln in cig if op == 0)
    return r["rid"], (r["pos"] + span - 1 + trail if rev else r["pos"] - lead), int(rev)


def units(recs):
    """-> [(id, [record indices])] for every unit: the pairing rule of qm_bam_to_pairs, ids of rule 4 (None: no placed end)"""
    by_name = defaultdict(list)
    for f, r in enumerate(recs):
        if (r["flag"] & 0xc0) in (0x40, 0x80) and not (r["flag"] & 0x900):
            by_name[r["name"]].append(f)
    partner = {}
    for fs in by_name.values():
        if len(fs) == 2 and (recs[fs[0]]["flag"] & 0xc0) != (recs[fs[1]]["flag"] & 0xc0):
            partner[fs[0]], partner[fs[1]] = fs[1], fs[0]
    out = []
    for f, r in enumerate(recs):
        if r["flag"] & 0x900 or partner.get(f, f + 1) < f:
            continue
        mem = [f] + ([partner[f]] if f in partner else [])
        pl = [g for g in mem if placed(recs[g])]
        if len(pl) == 2:
            ea, eb = end_of(recs[pl[0]])[:2], end_of(recs[pl[1]])[:2]
            uid = pl[0] if ea <= eb else pl[1]
        else:
            uid = pl[0] if pl else None
        out.append((uid, mem))
    return out


def score(r):
    q = r["qual"]
    return 0 if len(q) == 0 or q[0] == 0xff else int(q[q >= 15].sum())


def rule(recs):
    """-> (verdict per record, units, duplicate units, names of the units in groups tied at the top score) through
    oracle/dedup_py.py, fed the candidate units in id order (its ties go to the first)"""
    from oracle import dedup_py
    from oracle.qmo_py import ALN_DTYPE
    us = units(recs)
    cand = sorted((u for u in us if u[0] is not None), key=lambda u: u[0])
    stride = max([1] + [len(r["qual"]) for r in recs])
    alns = np.zeros(2 * len(cand), ALN_DTYPE)
    quals = np.zeros((2 * len(cand), stride), np.uint8)
    lens = np.zeros(2 * len(cand), np.int32)
    alns["flag"], alns["rid"] = 0x4, -1
    for k, (uid, mem) in enumerate(cand):
        for e, g in enumerate(mem):
            r = recs[g]
            if not placed(r):
                continue
            cig = oracle_cigar(r["cigar"])
            a = alns[2 * k + e]
            a["rid"], a["pos"], a["flag"], a["n_cigar"] = r["rid"], r["pos"], r["flag"], len(cig)
            a["cigar"][:len(cig)] = [(ln << 4) | op for op, ln in cig]
            if score(r):
                quals[2 * k + e, :len(r["qual"])] = r["qual"]
            lens[2 * k + e] = len(r["qual"])
    dup = dedup_py.mark_duplicates(alns, quals, lens) if cand else np.zeros(0, bool)
    verdict = np.zeros(len(recs), np.uint8)
    groups = defaultdict(list)
    for k, (uid, mem) in enumerate(cand):
        pl = [recs[g] for g in mem if placed(recs[g])]
        ends = tuple(sorted(end_of(r) for r in pl))
        groups[ends if len(pl) == 2 else ("frag",) + ends].append((sum(score(r) for r in pl), mem))
        if dup[k]:
            for g in mem:
                verdict[g] = placed(recs[g])
    tied = set()
    for members in groups.values():
        top = max(s for s, _ in members)
        if sum(s == top for s, _ in members) > 1:
            tied |= {recs[g]["name"] for s, mem in members for g in mem}
    return verdict, len(us), int(dup.sum()), tied


# ---- 1. round trip through the driver ------------------------------------------------------------------------------------
def add_copies(codes, quals, rng, n_src):
    """copy n_src random pairs 1-4 times; a copy keeps its source's qualities (an exact tie) or gets some changed"""
    src = rng.choice(len(codes) // 2, n_src, replace=False)
    c2, q2 = [codes], [quals]
    for i in src:
        for _ in range(int(rng.integers(1, 5))):
            c, q = codes[2 * i:2 * i + 2].copy(), quals[2 * i:2 * i + 2].copy()
            if rng.random() < 0.5:
                q[:, rng.integers(0, q.shape[1], 6)] = rng.integers(2, 41, 6)
            c2.append(c)
            q2.append(q)
    codes, quals = np.concatenate(c2), np.concatenate(q2)
    order = rng.permutation(len(codes) // 2)                      # copies spread over the FASTQ, not after their source
    rows = np.stack([2 * order, 2 * order + 1], 1).ravel()
    return codes[rows], quals[rows]


def unique_scores(quals, L):
    """qualities that give read r the score L x 15 + r (every base counts, 78 is the most a base can add): no two reads tie, so
    neither fragments nor pairs (pair i scores 2 L x 15 + 4 i + 1) tie, duplicates or not"""
    r = np.arange(len(quals))
    assert len(quals) <= 78 * L
    q = (15 + np.clip(r[:, None] - 78 * np.arange(L)[None, :], 0, 78)).astype(np.uint8)
    quals = quals.copy()
    quals[:, :L] = q
    return quals


def simulate(d, cfg, ties, seed, n_pairs=None):
    from quasimodo_b200 import workloads
    W = {"cfg1": lambda: workloads.config1(n_pairs or 20_000), "cfg3": lambda: workloads.config3(n_pairs or 20_000),
         "cfg5": lambda: workloads.config5(n_pairs or 8_000)}[cfg]()
    codes, quals, _, _ = W.simulate_host(0, W.n_pairs)
    codes, quals = add_copies(codes, quals, np.random.default_rng(seed), 300)
    if not ties:
        quals = unique_scores(quals, W.params.read_len)
    n = len(codes) // 2
    lens = np.full(2 * n, W.params.read_len, np.int32)
    fa, r1, r2 = d / "ref.fa", d / "r1.fq", d / "r2.fq"
    drvutil.write_fasta(W.ref, fa)
    drvutil.write_fastq(codes, quals, lens, drvutil.pair_names("rd", n), r1, r2)
    return dict(d=d, fa=fa, r1=r1, r2=r2, n=n)


def records(path):
    b = bamio.Bam(path)
    for r in b.records:
        r["cigar"] = [(x & 15, x >> 4) for x in r["cigar"]]
        r["raw"] = b.data[r["ustart"]:r["uend"]]
    return b


def cleared(raw):
    """the record bytes with 0x400 cleared"""
    flag = struct.unpack_from("<H", raw, 18)[0] & ~0x400
    return raw[:18] + struct.pack("<H", flag) + raw[20:]


def no_pg(text):
    return [ln for ln in text.split("\n") if not ln.startswith("@PG")]


def check_bai(path):
    from oracle.sort_py import reg2bin
    b = bamio.Bam(path)
    refs, n_no_coor = bamio.read_bai(path + ".bai")
    assert len(refs) == len(b.refs) and n_no_coor == sum(r["rid"] < 0 for r in b.records)
    for r in b.records:
        if r["rid"] < 0:
            continue
        span = sum(x >> 4 for x in r["cigar"] if (x & 15) in SPAN) if not r["flag"] & 4 else 0
        bins = refs[r["rid"]][0]
        chunks = bins[reg2bin(r["pos"], r["pos"] + max(span, 1))]
        assert any(b.voffset_to_u(v0) <= r["ustart"] < b.voffset_to_u(v1) for v0, v1 in chunks), r["name"]


@pytest.mark.parametrize("cfg", ["cfg1", "cfg3", "cfg5"])
def test_round_trip(tmp_path, cfg):
    s = simulate(tmp_path, cfg, ties=True, seed=7)
    d = s["d"]
    common = ["--ref", s["fa"], "--r1", s["r1"], "--r2", s["r2"], "--sample", "LIB", "-t", 4]
    drvutil.run_driver(["sample", "--rmdup", 1, "--bam", d / "s.bam", "--rmdup-bam", d / "s.rmdup.bam", "--metrics", d / "s.m"] + common)
    drvutil.run_driver(["sample", "--bam", d / "n.bam"] + common)
    outs = {}
    for src in ("s", "n"):
        p = drvutil.run_driver(["rmdup", "--bam", d / f"{src}.bam", "--rmdup-bam", d / f"{src}.out.bam", "--metrics", d / f"{src}.out.m",
                                "--sample", "LIB", "-t", 4])
        assert "phases (s):" in p.stderr
        outs[src] = records(d / f"{src}.out.bam")
        check_bai(str(d / f"{src}.out.bam"))
    a, b = outs["s"], outs["n"]
    assert [r["raw"] for r in a.records] == [r["raw"] for r in b.records]
    assert no_pg(a.text) == no_pg(b.text) and a.refs == b.refs
    pg = [ln for ln in a.text.split("\n") if ln.startswith("@PG")]
    assert len(pg) == 2 and "ID:quasimodo_b200.rmdup\t" in pg[1] and "PP:quasimodo_b200\t" in pg[1]
    metrics = (d / "s.m").read_bytes()
    assert (d / "s.out.m").read_bytes() == metrics and (d / "n.out.m").read_bytes() == metrics
    # the rule on the input: every kept record, byte for byte with 0x400 cleared
    sb = records(d / "s.bam")
    assert sum((r["flag"] & 0x400) != 0 for r in sb.records) > 300            # stale flags in the input
    verdict, n_units, n_dup, tied = rule(sb.records)
    assert n_units == s["n"] and f"LIB\t{n_units}\t{n_dup}\t".encode() in metrics
    assert [r["raw"] for r in a.records] == [cleared(r["raw"]) for r, v in zip(sb.records, verdict) if not v]
    # sample's .rmdup.bam: the same records outside the groups tied at the top score (sample gives a tie to the lowest FASTQ pair)
    sr = records(d / "s.rmdup.bam")
    assert tied
    assert [r["raw"] for r in a.records if r["name"] not in tied] == [r["raw"] for r in sr.records if r["name"] not in tied]
    assert len(a.records) == len(sr.records)


# ---- 2. hand-built records -----------------------------------------------------------------------------------------------
def hand_built(seed, n_templates=500):
    """records of a sorted BAM on contigs of 3000, 500 and 3000 bases, unclipped coordinates drawn from a small pool so that keys
    collide, copies with equal and with different scores; every oddity of the module docstring"""
    rng = np.random.default_rng(seed)
    pool = [(int(rng.integers(0, 3)), int(rng.integers(60, 400))) for _ in range(30)]
    recs = []

    def cigar(L, hard):
        lead = [] if rng.random() < 0.4 else [(int(rng.choice([4, 5] if hard else [4])), int(rng.integers(1, 6)))]
        if lead and rng.random() < 0.3:
            lead = [(5, int(rng.integers(1, 4))), (4, int(rng.integers(1, 4)))]
        trail = [] if rng.random() < 0.4 else [(int(rng.choice([4, 5] if hard else [4])), int(rng.integers(1, 6)))]
        if trail and rng.random() < 0.3:
            trail = [(4, int(rng.integers(1, 4))), (5, int(rng.integers(1, 4)))]
        q = sum(ln for op, ln in lead + trail if op == 4)
        body, left = [], L - q
        while left > 0:
            op = int(rng.choice([0, 0, 0, 7, 8, 1, 2, 3, 6]))
            ln = int(rng.integers(1, 30))
            if op in (0, 7, 8, 1):
                ln = min(ln, left)
                left -= ln
            body.append((op, ln))
        if body[0][0] not in SPAN:
            body.insert(0, (0, 1))
        return lead + body + trail, q + sum(ln for op, ln in body if op in (0, 7, 8, 1))

    def read(name, flag, u=None, L=None, hard=False):
        rid, c = pool[int(rng.integers(0, len(pool)))] if u is None else u
        L = L or int(rng.integers(30, 120))
        cig, ql = cigar(L, hard)
        rev = bool(flag & 0x10)
        body = [i for i, (op, _) in enumerate(cig) if op not in CLIP]
        lead = sum(ln for i, (_, ln) in enumerate(cig) if i < body[0])
        trail = sum(ln for i, (_, ln) in enumerate(cig) if i > body[-1])
        span = sum(ln for op, ln in cig if op in SPAN)
        pos = c - span + 1 - trail if rev else c + lead
        return dict(name=name, flag=flag, rid=rid, pos=max(pos, 0), cigar=cig, seq=rng.integers(0, 5, ql).astype(np.uint8),
                    qual=rng.integers(2, 42, ql).astype(np.uint8))

    def unmapped(name, flag, at=None, L=50):
        rid, pos = (at["rid"], at["pos"]) if at else (-1, -1)
        return dict(name=name, flag=flag | 0x4, rid=rid, pos=pos, cigar=[], seq=rng.integers(0, 5, L).astype(np.uint8),
                    qual=rng.integers(2, 42, L).astype(np.uint8))

    P1, P2 = 0x1 | 0x40, 0x1 | 0x80
    for t in range(n_templates):
        kind = rng.choice(["pair", "pair", "pair", "frag", "unmapped", "lonely", "three", "single", "long"])
        nm = f"t{t}"
        s1, s2 = 0x10 * int(rng.integers(0, 2)), 0x10 * int(rng.integers(0, 2))
        extra = (0x200 if rng.random() < 0.05 else 0) | (0x400 if rng.random() < 0.1 else 0)
        if kind in ("pair", "long"):
            L = 600 if kind == "long" else None
            grp = [read(nm, P1 | s1 | extra, L=L), read(nm, P2 | s2, L=L)]
            if rng.random() < 0.2:
                grp.append(read(nm, P1 | s1 | 0x800, hard=True))
            if rng.random() < 0.1:
                grp.append(read(nm, P2 | s2 | 0x100))
        elif kind == "frag":
            x = read(nm, P1 | s1 | extra)
            grp = [x, unmapped(nm, P2 | s1, at=x)]
        elif kind == "unmapped":
            grp = [unmapped(nm, P1), unmapped(nm, P2)]
        elif kind == "lonely":
            grp = [read(nm, P1 | s1 | extra)]
        elif kind == "three":
            grp = [read(nm, P1 | s1), read(nm, P2 | s2), read(nm, P2)]
        else:
            grp = [read(nm, s1 | extra)]
            if rng.random() < 0.3:                                 # QUAL '*'
                grp[0]["qual"] = np.full(len(grp[0]["seq"]), 0xff, np.uint8)
        recs += grp
        # copies: same ends, other CIGARs allowed (the unclipped coordinate is what counts), scores equal or not
        for k in range(int(rng.integers(0, 3)) if kind in ("pair", "long", "frag", "lonely", "single") else 0):
            for r in grp:
                if r["flag"] & 0x900:
                    continue
                c = dict(r, name=f"{nm}.c{k}", qual=r["qual"].copy())
                if rng.random() < 0.5 and c["qual"][0] != 0xff:
                    c["qual"][rng.integers(0, len(c["qual"]))] = rng.integers(2, 42)
                recs.append(c)
    order = rng.permutation(len(recs))
    recs = [recs[i] for i in order]
    recs.sort(key=lambda r: (r["rid"] if r["rid"] >= 0 else 1 << 20, r["pos"]))
    return recs


def device_verdicts(ctx, recs, hash_bits=64):
    import torch
    from quasimodo_b200 import _lib
    L = _lib.lib()
    blobs = [encode(r) for r in recs]
    offs = np.concatenate([[0], np.cumsum([len(b) for b in blobs])[:-1]]).astype(np.int64)
    data = np.frombuffer(b"".join(blobs), np.uint8)
    nu, nd = C.c_int64(), C.c_int64()
    if hash_bits == 64:
        out = np.zeros(len(recs), np.uint8)
        rc = L.qm_bam_mark_duplicates_host(ctx._h, data.ctypes.data, len(data), offs.ctypes.data, len(recs), out.ctypes.data, C.byref(nu), C.byref(nd))
        assert rc == 0, L.qm_last_error(ctx._h)
        return out, nu.value, nd.value
    dev = torch.device("cuda:0")
    d_data, d_offs = torch.from_numpy(data.copy()).to(dev), torch.from_numpy(offs).to(dev)
    d_out = torch.zeros(len(recs), dtype=torch.uint8, device=dev)
    fn = L.qm_bam_mark_duplicates_hashbits
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_void_p]
    rc = fn(ctx._h, d_data.data_ptr(), d_offs.data_ptr(), len(recs), hash_bits, d_out.data_ptr(), C.byref(nu), C.byref(nd), None)
    assert rc == 0, L.qm_last_error(ctx._h)
    torch.cuda.synchronize()
    return d_out.cpu().numpy(), nu.value, nd.value


@pytest.fixture(scope="module")
def ctx():
    from quasimodo_b200 import Context
    c = Context(0)
    yield c
    c.close()


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_hand_built_records(ctx, seed):
    recs = hand_built(seed)
    got, n_units, n_dup = device_verdicts(ctx, recs)
    want, w_units, w_dup, tied = rule(recs)
    assert n_units == w_units and n_dup == w_dup
    bad = np.flatnonzero(got != want)
    assert not len(bad), [(recs[i]["name"], recs[i]["flag"], int(got[i]), int(want[i])) for i in bad[:8]]
    # what the rule promises, and that the input reaches it
    assert n_dup > 20 and tied
    fl = np.array([r["flag"] for r in recs])
    assert not got[(fl & 0x900) != 0].any() and not got[(fl & 0x4) != 0].any()
    assert got[(fl & 0x900) == 0].any() and got[(fl & 0x200) != 0].any() and got[(fl & 0x400) == 0].any()
    assert any(got[i] for i, r in enumerate(recs) if len(r["seq"]) > 512)
    assert any(got[i] for i, r in enumerate(recs) if r["qual"][0] == 0xff)


def test_fragment_on_a_pair_end_and_hand_picked_cases(ctx):
    """a fragment whose end is a pair's end is a duplicate whatever its score; the supplementary record and the unplaced mate of
    a duplicate stay; a tie goes to the unit whose leftmost end comes first in the file"""
    q = lambda v, L=40: np.full(L, v, np.uint8)       # noqa: E731
    s = lambda L=40: np.zeros(L, np.uint8)            # noqa: E731
    P1, P2, R = 0x1 | 0x40, 0x1 | 0x80, 0x10
    rec = lambda name, flag, rid, pos, cig, qual: dict(name=name, flag=flag, rid=rid, pos=pos, cigar=cig, seq=s(len(qual)), qual=qual)  # noqa: E731
    recs = [
        rec("pa", P1, 0, 100, [(0, 40)], q(20)), rec("pb", P1, 0, 102, [(5, 2), (0, 40)], q(20)),      # pb: same end through H clips
        rec("fr", P1 | 0x20, 0, 100, [(0, 40)], q(40)), rec("fr", P2 | 0x4 | R, 0, 100, [], q(40)),   # fragment on pa's end
        rec("pb", P1 | 0x800, 0, 150, [(5, 10), (0, 30)], q(40, 30)),
        # reverse ends at 247 through N / = / X and an S, and through a D and S + H; both pairs score 1500
        rec("pa", P2 | R, 0, 200, [(0, 30), (3, 5), (7, 5), (8, 5), (4, 3)], np.r_[q(20, 35), q(10, 8)]),
        rec("pb", P2 | R, 0, 202, [(0, 30), (2, 3), (4, 5), (5, 8)], q(20, 35)),
    ]
    recs.sort(key=lambda r: (r["rid"], r["pos"]))
    got, n_units, n_dup = device_verdicts(ctx, recs)
    want, *_ = rule(recs)
    assert np.array_equal(got, want)
    v = {(r["name"], r["flag"]): int(x) for r, x in zip(recs, got)}
    assert v[("pa", P1)] == 0 and v[("pa", P2 | R)] == 0                      # pa and pb tie (same ends, same score): pa is first
    assert v[("pb", P1)] == 1 and v[("pb", P2 | R)] == 1 and v[("pb", P1 | 0x800)] == 0
    assert v[("fr", P1 | 0x20)] == 1 and v[("fr", P2 | 0x4 | R)] == 0
    assert n_units == 3 and n_dup == 2


# ---- 3. name collisions --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hash_bits", [1, 2, 7])
def test_hash_collisions_change_nothing(ctx, hash_bits):
    recs = hand_built(5, n_templates=250)
    want = device_verdicts(ctx, recs)
    got = device_verdicts(ctx, recs, hash_bits)
    assert np.array_equal(got[0], want[0]) and got[1:] == want[1:]


# ---- 4. chain into pileup ------------------------------------------------------------------------------------------------
def test_rmdup_then_pileup(tmp_path):
    s = simulate(tmp_path, "cfg1", ties=False, seed=3, n_pairs=4_000)          # with the copies, fewer reads than unique scores
    d = s["d"]
    drvutil.run_driver(["sample", "--ref", s["fa"], "--r1", s["r1"], "--r2", s["r2"], "--rmdup", 1, "--bam", d / "s.bam", "--rmdup-bam",
                        d / "s.rmdup.bam", "-t", 4])
    drvutil.run_driver(["rmdup", "--bam", d / "s.bam", "--rmdup-bam", d / "g.rmdup.bam", "-t", 4])
    _, _, n_dup, tied = rule(records(d / "s.bam").records)
    assert n_dup > 300 and not tied
    got = {}
    for src in ("s", "g"):
        drvutil.run_driver(["pileup", "--ref", s["fa"], "--bam", d / f"{src}.rmdup.bam", "--counts", d / f"{src}.tsv", "--vcf", d / f"{src}.vcf",
                            "-t", 4])
        got[src] = [(d / f"{src}.{e}").read_bytes() for e in ("tsv", "vcf")]
    assert got["s"] == got["g"] and got["s"][1].count(b"\n") > 20
