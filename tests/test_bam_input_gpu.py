"""GPU tests of BAM input (`qm_driver pileup`, qm_bam_to_pairs):

1. the round trip: `sample` writes a BAM, `pileup` reads it back, and the count TSV, VCF, inflated .vcf.gz and text pileup are
   `sample`'s bytes, under the defaults, --rmdup 1 (.rmdup.bam and the full BAM), --max-depth 50, --baq 1 and the admission
   options, on simulated pairs of BASELINE configs 1, 3 (several contigs) and 5 (2x250, indels);
2. hand-built records (tests/recgen.py) as BAM records: the count planes, indel table and text pileup of the pair layout equal
   the C oracle's on the layout the pairing rule defines, and the depth cap replays htslib over FILE order;
3. records the driver never writes: supplementary records with H clips, left-out flags, = / X operations, a missing mate,
   three records of one name, mates that tie on position and strand in either file order;
4. name collisions: with the hash cut to 2 bits the pairs are still the exact-name join."""
import ctypes as C
import gzip
import struct
from collections import defaultdict

import numpy as np
import pytest

from tests import drvutil, recgen

pytestmark = pytest.mark.gpu

_COMP = np.array([3, 2, 1, 0, 4], np.uint8)
_NT16 = np.array([1, 2, 4, 8, 15], np.uint8)                    # codes 0..4 -> SAM's 4-bit codes


# ---- 1. round trip through the driver ------------------------------------------------------------------------------------
OPTION_SETS = {
    "default": [],
    "rmdup": ["--rmdup", 1],
    "max-depth-50": ["--max-depth", 50],
    "baq": ["--baq", 1],
    "admission": ["-q", 20, "-Q", 20, "--count-orphans", 1, "--ignore-overlaps", 1],
}


@pytest.fixture(scope="module", params=["cfg1", "cfg3", "cfg5"])
def sim(request, tmp_path_factory):
    from quasimodo_b200 import workloads
    W = {"cfg1": lambda: workloads.config1(40_000), "cfg3": lambda: workloads.config3(40_000),
         "cfg5": lambda: workloads.config5(16_000)}[request.param]()
    d = tmp_path_factory.mktemp(request.param)
    codes, quals, _, _ = W.simulate_host(0, W.n_pairs)
    lens = np.full(2 * W.n_pairs, W.params.read_len, np.int32)
    fa, r1, r2 = d / "ref.fa", d / "r1.fq", d / "r2.fq"
    drvutil.write_fasta(W.ref, fa)
    drvutil.write_fastq(codes, quals, lens, drvutil.pair_names("rt", W.n_pairs), r1, r2)
    return dict(d=d, fa=fa, r1=r1, r2=r2)


def _outputs(prefix):
    return dict(counts=f"{prefix}.tsv", vcf=f"{prefix}.vcf", mpileup=f"{prefix}.mpileup")


def _read_outputs(o):
    got = {k: open(v, "rb").read() for k, v in o.items()}
    got["vcf.gz"] = gzip.open(o["vcf"] + ".gz", "rb").read()
    return got


@pytest.mark.parametrize("opts", list(OPTION_SETS), ids=list(OPTION_SETS))
def test_round_trip_is_byte_identical(sim, opts):
    d, extra = sim["d"], OPTION_SETS[opts]
    so = _outputs(d / f"s.{opts}")
    bam, rbam = d / f"s.{opts}.bam", d / f"s.{opts}.rmdup.bam"
    args = ["sample", "--ref", sim["fa"], "--r1", sim["r1"], "--r2", sim["r2"], "--bam", bam, "--counts", so["counts"], "--vcf", so["vcf"],
            "--mpileup", so["mpileup"], "-t", 4] + extra
    if opts == "rmdup":
        args += ["--rmdup-bam", rbam]
    drvutil.run_driver(args)
    want = _read_outputs(so)
    assert want["mpileup"].count(b"\n") > 1000 and want["vcf"].count(b"\n") > 20
    pile_extra = [] if opts == "rmdup" else extra             # the BAMs hold the duplicate marking already
    inputs = [bam, rbam] if opts == "rmdup" else [bam]
    for src in inputs:
        po = _outputs(d / f"p.{opts}.{src.name}")
        p = drvutil.run_driver(["pileup", "--ref", sim["fa"], "--bam", src, "--counts", po["counts"], "--vcf", po["vcf"], "--mpileup", po["mpileup"],
                                "-t", 4] + pile_extra)
        if opts == "max-depth-50":
            assert "depth cap 50:" in p.stderr and " 0 reads dropped" not in p.stderr, p.stderr
        got = _read_outputs(po)
        for k in want:
            if got[k] != want[k]:
                gl, wl = got[k].split(b"\n"), want[k].split(b"\n")
                bad = [i for i in range(min(len(gl), len(wl))) if gl[i] != wl[i]][:1]
                raise AssertionError(f"{src.name} {k}: lines {len(gl)} vs {len(wl)}; first difference {bad}: "
                                     f"{gl[bad[0]][:200] if bad else b''} / {wl[bad[0]][:200] if bad else b''}")


# ---- record helpers ------------------------------------------------------------------------------------------------------
def encode(rec):
    """a record dict (file form: SEQ / QUAL in BAM orientation, codes 0..4) -> BAM record bytes"""
    seq, qual = np.asarray(rec["seq"], np.uint8), np.asarray(rec["qual"], np.uint8)
    L = len(seq)
    nib = _NT16[seq]
    if L & 1:
        nib = np.append(nib, 0)
    packed = ((nib[0::2] << 4) | nib[1::2]).astype(np.uint8).tobytes()
    nm = rec["name"].encode() + b"\0"
    cig = [(ln << 4) | op for op, ln in rec["cigar"]]
    tags = rec.get("tags", b"")
    body = struct.pack("<iiBBHHHiiii", rec["rid"], rec["pos"], len(nm), rec.get("mapq", 60), 0, len(cig), rec["flag"], L,
                       rec.get("mrid", -1), rec.get("mpos", -1), rec.get("tlen", 0))
    body += nm + struct.pack(f"<{len(cig)}I", *cig) + packed + qual.tobytes() + tags
    return struct.pack("<i", len(body)) + body


def kept(rec):
    return not (rec["flag"] & 0x704) and rec["rid"] >= 0 and len(rec["cigar"]) > 0


def pairing_primary(rec):
    return (rec["flag"] & 0xc0) in (0x40, 0x80) and not (rec["flag"] & 0x900)


def pair_rows(recs):
    """the pairing rule as a dictionary join over the records handed in (file order): -> row -> record index, -1 = placeholder"""
    by_name = defaultdict(list)
    for f, r in enumerate(recs):
        if pairing_primary(r):
            by_name[r["name"]].append(f)
    partner = [-1] * len(recs)
    for fs in by_name.values():
        if len(fs) == 2 and (recs[fs[0]]["flag"] & 0xc0) != (recs[fs[1]]["flag"] & 0xc0):
            partner[fs[0]], partner[fs[1]] = fs[1], fs[0]
    rows = []
    for f in range(len(recs)):
        if partner[f] < 0:
            rows += [f, -1]
        elif f < partner[f]:
            rows += [f, partner[f]]
    return rows


def decode(rec, stride):
    """what the device decode makes of a record: qm_aln, codes and qualities as sequenced, length"""
    from oracle.qmo_py import ALN_DTYPE
    a = np.zeros((), ALN_DTYPE)
    ops = []
    for op, ln in rec["cigar"]:
        if op == 5 or ln == 0:
            continue
        op = 0 if op in (7, 8) else op
        if ops and ops[-1][0] == op:
            ops[-1] = (op, ops[-1][1] + ln)
        else:
            ops.append((op, ln))
    a["rid"], a["pos"], a["flag"], a["mapq"] = rec["rid"], rec["pos"], rec["flag"], rec.get("mapq", 60)
    a["mate_rid"], a["mate_pos"], a["tlen"] = rec.get("mrid", -1), rec.get("mpos", -1), rec.get("tlen", 0)
    a["n_cigar"] = len(ops)
    a["cigar"][:len(ops)] = [(ln << 4) | op for op, ln in ops]
    seq, qual = np.asarray(rec["seq"], np.uint8), np.asarray(rec["qual"], np.uint8)
    if rec["flag"] & 0x10:
        seq, qual = _COMP[seq[::-1]], qual[::-1]
    c, q = np.full(stride, 4, np.uint8), np.zeros(stride, np.uint8)
    c[:len(seq)], q[:len(seq)] = seq, qual
    return a, c, q, len(seq)


def layout(recs, rows, stride):
    from oracle.qmo_py import ALN_DTYPE
    n = len(rows)
    alns, codes, quals, lens = np.zeros(n, ALN_DTYPE), np.full((n, stride), 4, np.uint8), np.zeros((n, stride), np.uint8), np.zeros(n, np.int32)
    for i, f in enumerate(rows):
        if f < 0:
            alns[i]["rid"], alns[i]["pos"], alns[i]["flag"], alns[i]["mate_rid"], alns[i]["mate_pos"] = -1, -1, 0x4, -1, -1
        else:
            alns[i], codes[i], quals[i], lens[i] = decode(recs[f], stride)
    return alns, codes, quals, lens


def sort_key(rec):
    return (rec["rid"] if rec["rid"] >= 0 else 1 << 20, rec["pos"], (rec["flag"] >> 4) & 1)


def batch_records(alns, codes, quals, lens):
    """recgen's pairs (reads 2i / 2i + 1, name p<i>) as the records of a coordinate-sorted BAM.  Ties of position and strand
    are written in the order of the pair layout the reader will build, so that the oracle -- which breaks such ties by read
    index -- sees reads in file order too: the pairs are laid out by their first record's key, and the file is sorted by
    (key, row)."""
    recs = []
    for r in range(len(alns)):
        a = alns[r]
        L, nc = int(lens[r]), int(a["n_cigar"])
        seq, q = codes[r, :L].copy(), np.minimum(quals[r, :L], 254)
        if a["flag"] & 0x10:
            seq, q = _COMP[seq[::-1]], q[::-1]
        recs.append(dict(name=f"p{r // 2}", flag=int(a["flag"]), rid=int(a["rid"]), pos=int(a["pos"]), mapq=int(a["mapq"]),
                         cigar=[(int(w) & 15, int(w) >> 4) for w in a["cigar"][:nc]] if nc != 255 else [], seq=seq, qual=q,
                         mrid=int(a["mate_rid"]), mpos=int(a["mate_pos"]), tlen=int(a["tlen"])))
    units = []
    for i in range(len(recs) // 2):
        r0, r1 = recs[2 * i], recs[2 * i + 1]
        if kept(r0) and kept(r1) and pairing_primary(r0) and pairing_primary(r1) and (r0["flag"] & 0xc0) != (r1["flag"] & 0xc0):
            units.append((r0, r1) if sort_key(r0) <= sort_key(r1) else (r1, r0))
        else:
            units += [(r, None) for r in (r0, r1) if kept(r)]
    units.sort(key=lambda u: sort_key(u[0]))
    row = {}
    for i, (x, y) in enumerate(units):
        row[id(x)] = 2 * i
        if y is not None:
            row[id(y)] = 2 * i + 1
    return sorted(recs, key=lambda r: sort_key(r) + (row.get(id(r), 1 << 40),))


# ---- device entry --------------------------------------------------------------------------------------------------------
def _d2h(ptr, nbytes):
    out = np.empty(nbytes, np.uint8)
    if nbytes:
        rt = C.CDLL("libcudart.so.12")
        rt.cudaMemcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
        assert rt.cudaMemcpy(out.ctypes.data, ptr, nbytes, 2) == 0
    return out


def run_bam_input(ctx, idx, recs, names, pg, max_depth=0, hash_bits=64, want_text=True):
    """the records of the file (file order) through qm_bam_to_pairs: -> row_file, drop, planes, indel rows, text"""
    import torch
    from quasimodo_b200 import _lib
    from tests.test_indels_gpu import as_rows
    L = _lib.lib()
    ks = [r for r in recs if kept(r)]
    blobs = [encode(r) for r in ks]
    offs = np.concatenate([[0], np.cumsum([len(b) for b in blobs])[:-1]]).astype(np.int64) if blobs else np.zeros(0, np.int64)
    data = np.frombuffer(b"".join(blobs) or b"\0", np.uint8)
    stride = max([16] + [(len(r["seq"]) + 15) & ~15 for r in ks])
    bp = _lib.BamPairs()
    if hash_bits == 64:
        rc = L.qm_bam_to_pairs_host(ctx._h, idx._h, data.ctypes.data, len(data), offs.ctypes.data, len(ks), stride, C.byref(pg), 0, max_depth,
                                    C.byref(bp))
    else:
        dev = torch.device("cuda:0")
        d_data, d_offs = torch.from_numpy(data.copy()).to(dev), torch.from_numpy(offs).to(dev)
        fn = L.qm_bam_to_pairs_hashbits
        fn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int, C.c_int, C.c_int,
                       C.POINTER(_lib.BamPairs), C.c_void_p]
        rc = fn(ctx._h, idx._h, d_data.data_ptr(), d_offs.data_ptr(), len(ks), stride, C.byref(pg), 0, max_depth, hash_bits, C.byref(bp), None)
    assert rc == 0, L.qm_last_error(ctx._h)
    n = 2 * bp.n_pairs
    row_file = _d2h(bp.d_row_file, 8 * n).view(np.int64)
    drop = _d2h(bp.d_drop, n) if bp.d_drop else None
    dev = torch.device("cuda:0")
    counts = torch.zeros(16 * idx.l_pac, dtype=torch.int32, device=dev)
    tab = C.c_void_p()
    assert L.qm_indel_table_create(ctx._h, 16, C.byref(tab)) == 0
    try:
        rc = L.qm_pileup_accumulate_masked(ctx._h, idx._h, C.byref(pg), bp.d_alns, bp.d_codes, bp.d_quals, bp.stride, bp.d_lens, bp.n_pairs,
                                           C.c_void_p(counts.data_ptr()), tab, bp.d_drop, None)
        assert rc == 0, L.qm_last_error(ctx._h)
        torch.cuda.synchronize()
        out = np.zeros(1 << 16, _lib.INDEL_DTYPE)
        m = C.c_int64()
        assert L.qm_indel_table_fetch_host(tab, idx._h, out.ctypes.data, len(out), C.byref(m)) == 0
    finally:
        L.qm_indel_table_destroy(tab)
    text = None
    if want_text:
        arr = (C.c_char_p * len(names))(*[s.encode() for s in names])
        d_text, nbytes = C.c_char_p(), C.c_int64()
        rc = L.qm_mpileup_text_ranked(ctx._h, idx._h, C.byref(pg), bp.d_alns, bp.d_codes, bp.d_quals, bp.stride, bp.d_lens, bp.n_pairs, arr,
                                      bp.d_row_file, C.byref(d_text), C.byref(nbytes), None)
        assert rc == 0, L.qm_last_error(ctx._h)
        buf = C.create_string_buffer(max(1, nbytes.value))
        assert L.qm_mpileup_text_fetch(ctx._h, buf, nbytes.value) == 0
        text = buf.raw[:nbytes.value]
    return dict(ks=ks, stride=stride, row_file=row_file, drop=drop, n_capped=bp.n_capped, planes=counts.view(16, idx.l_pac).cpu().numpy(),
                indels=as_rows(out[:m.value]), text=text)


@pytest.fixture(scope="module")
def ctx():
    from quasimodo_b200 import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def genome():
    return recgen.Genome()


@pytest.fixture(scope="module")
def ref(genome):
    from oracle import qmo_py
    return qmo_py.Ref(genome.codes, genome.lens, k=31)


@pytest.fixture(scope="module")
def idx(ctx, genome):
    i = ctx.index(genome, 31)
    yield i
    i.close()


def expected(ref, genome, ks, stride, po, max_depth=0, text=True):
    """the oracle on the layout the pairing rule gives the kept records (file order); the cap replayed over file order"""
    from oracle import qmo_py
    rows = pair_rows(ks)
    alns, codes, quals, lens = layout(ks, rows, stride)
    drop_rows = np.zeros(len(rows), np.uint8)
    if max_depth:
        from oracle.qmo_py import ALN_DTYPE
        fa = np.array([decode(r, stride)[0] for r in ks], dtype=ALN_DTYPE)
        keep = qmo_py.depth_cap(ref, fa, max_depth, po)
        adm = qmo_py.depth_cap(ref, fa, 1 << 30, po)
        for i, f in enumerate(rows):
            if f >= 0 and adm[f] and not keep[f]:
                drop_rows[i] = 1
        alns = alns.copy()
        alns["flag"][drop_rows == 1] |= 0x200
    out = dict(rows=np.array(rows, np.int64), drop=drop_rows, planes=qmo_py.pileup(ref, alns, codes, quals, lens, popt=po),
               indels=qmo_py.indels(ref, alns, codes, lens, popt=po))
    if text:
        a0, c0, q0, l0 = layout(ks, rows, stride)
        out["text"] = qmo_py.mpileup_text(ref, a0, c0, q0, l0, genome.names, popt=po)
    return out


def check(got, want, max_depth=0):
    assert np.array_equal(got["row_file"], want["rows"]), (got["row_file"][:20], want["rows"][:20])
    if max_depth:
        assert np.array_equal(got["drop"], want["drop"]) and got["n_capped"] == int(want["drop"].sum())
    assert np.array_equal(got["planes"].T, want["planes"]), np.argwhere(got["planes"].T != want["planes"])[:8]
    assert np.array_equal(got["indels"], want["indels"])
    if "text" in want and got["text"] is not None:
        assert got["text"] == want["text"]


# ---- 2. hand-built records -----------------------------------------------------------------------------------------------
from tests.test_records_gpu import OPT_IDS, OPTS, popts   # noqa: E402  (the option sets of the record tests)


@pytest.fixture(scope="module")
def batches(genome):
    return {"random+adversarial": batch_records(*recgen.random_batch(genome, 1500, 5, batch=recgen.adversarial(genome)).arrays(150)),
            "long": batch_records(*recgen.long_batch(genome, 300, 23).arrays(512))}


@pytest.mark.parametrize("opt", OPTS, ids=OPT_IDS)
@pytest.mark.parametrize("which", ["random+adversarial", "long"])
def test_hand_built_records(ctx, idx, ref, genome, batches, which, opt):
    recs = batches[which]
    po, pg = popts(opt)
    got = run_bam_input(ctx, idx, recs, genome.names, pg)
    want = expected(ref, genome, got["ks"], got["stride"], po)
    assert want["planes"][:, 14].sum() > 0
    check(got, want)


@pytest.mark.parametrize("max_depth", [2, 5, 8])
def test_depth_cap_follows_file_order(ctx, idx, ref, genome, max_depth):
    """reads of different pairs tie on (position, strand), and the file order of the tied reads is not the order of their
    pairs: p1's second read comes before p0's second read in the file, although p0 opens the layout"""
    rng = np.random.default_rng(max_depth)
    b = recgen.Batch(genome, rng)
    recs = []
    P = 0x1 | 0x2
    for i in range(12):                  # pair i: first read at 10 + i, second read at 100 for every pair (reverse strand)
        x = b.read(0, 10 + i, [(recgen.M, 30)], P)
        y = b.read(0, 100, [(recgen.M, 30)], P | 0x10)
        for r, fl in ((x, 0x40 | 0x20), (y, 0x80)):
            recs.append(dict(name=f"t{i}", flag=r["flag"] | fl, rid=0, pos=r["pos"], cigar=r["ops"], seq=r["seq"], qual=np.minimum(r["quals"], 60)))
    # the second reads all start at 100: written in the reverse order of their pairs
    firsts, seconds = recs[0::2], recs[1::2][::-1]
    recs = firsts + seconds
    po, pg = popts({})
    got = run_bam_input(ctx, idx, recs, genome.names, pg, max_depth=max_depth, want_text=False)
    want = expected(ref, genome, got["ks"], got["stride"], po, max_depth=max_depth, text=False)
    assert want["drop"].sum() > 0
    check(got, want, max_depth)
    # the replay over pair order would drop other reads
    rows = want["rows"]
    alns, _, _, _ = layout(got["ks"], list(rows), got["stride"])
    from oracle import qmo_py
    assert not np.array_equal(~qmo_py.depth_cap(ref, alns, max_depth, po) & qmo_py.depth_cap(ref, alns, 1 << 30, po), want["drop"] == 1)


# ---- 3. what the driver never writes -------------------------------------------------------------------------------------
def test_records_the_driver_never_writes(ctx, idx, ref, genome):
    rng = np.random.default_rng(9)
    b = recgen.Batch(genome, rng)
    M, I, D, S = recgen.M, recgen.I, recgen.D, recgen.S

    def rec(name, flag, rid, pos, ops, clip_h=(0, 0), eqx=False):
        r = b.read(rid, pos, ops, flag)
        cig = list(r["ops"])
        if eqx:                          # M blocks written as = / X runs
            cig = [x for op, ln in cig for x in (([(7, ln // 2), (8, 1), (7, ln - ln // 2 - 1)] if ln > 2 else [(7, ln)]) if op == M else [(op, ln)])]
        cig = ([(5, clip_h[0])] if clip_h[0] else []) + cig + ([(5, clip_h[1])] if clip_h[1] else [])
        return dict(name=name, flag=flag, rid=rid, pos=pos, cigar=cig, seq=r["seq"], qual=np.minimum(r["quals"], 60))

    P1, P2, R, MR = 0x1 | 0x2 | 0x40, 0x1 | 0x2 | 0x80, 0x10, 0x20
    recs = [
        rec("pair", P1 | MR, 0, 10, [(M, 40)]), rec("pair", P2 | R, 0, 30, [(M, 20), (I, 2), (M, 18)]),
        # supplementary with hard clips next to its proper pair: a pair of its own
        rec("supp", P1 | MR, 0, 50, [(M, 30)]), rec("supp", P1 | 0x800, 0, 52, [(M, 20)], clip_h=(10, 0)),
        rec("supp", P2 | R, 0, 60, [(M, 30)]),
        # secondary, QC-failed, duplicate: left out; their mates stay alone
        rec("sec", P1, 0, 70, [(M, 30)]), rec("sec", P2 | 0x100 | R, 0, 75, [(M, 30)]),
        rec("qcf", P1, 0, 80, [(M, 30)]), rec("qcf", P2 | 0x200 | R, 0, 90, [(M, 30)]),
        rec("dup", P1 | 0x400, 0, 95, [(M, 30)]), rec("dup", P2 | R, 0, 99, [(M, 30)]),
        # = / X operations
        rec("eqx", P1 | MR, 2, 5, [(S, 3), (M, 40)], eqx=True), rec("eqx", P2 | R, 2, 20, [(M, 10), (D, 3), (M, 30)], eqx=True),
        # a mate missing from the file
        rec("lonely", P1, 2, 40, [(M, 35)]),
        # three primary records of one name: nobody pairs
        rec("three", P1, 2, 60, [(M, 30)]), rec("three", P2 | R, 2, 70, [(M, 30)]), rec("three", P2, 2, 80, [(M, 30)]),
        # mates tied on position and strand, the second segment first in the file, and the first segment first
        rec("tieA", P2 | MR | R, 2, 100, [(M, 40)]), rec("tieA", P1 | MR | R, 2, 100, [(M, 40)]),
        rec("tieB", P1, 2, 150, [(M, 40)]), rec("tieB", P2, 2, 150, [(M, 40)]),
        # single-end
        rec("se", 0, 2, 200, [(M, 30)]),
    ]
    recs.sort(key=sort_key)
    for opt in ({}, {"ignore_overlaps": 1}, {"count_orphans": 1}):
        po, pg = popts(opt)
        got = run_bam_input(ctx, idx, recs, genome.names, pg)
        want = expected(ref, genome, got["ks"], got["stride"], po)
        check(got, want)
    names = [got["ks"][f]["name"] if f >= 0 else None for f in got["row_file"]]
    pairs = {(names[i], names[i + 1]) for i in range(0, len(names), 2)}
    assert ("pair", "pair") in pairs and ("supp", "supp") in pairs and ("supp", None) in pairs and ("tieA", "tieA") in pairs
    assert ("lonely", None) in pairs and ("three", "three") not in pairs and ("sec", None) in pairs and ("se", None) in pairs
    # the tie rule: row 2i is the record that comes first in the file
    for i in range(0, len(names), 2):
        if names[i + 1] is not None:
            assert got["row_file"][i] < got["row_file"][i + 1]


# ---- 4. name collisions --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hash_bits", [1, 2, 7])
def test_pairs_are_the_exact_name_join(ctx, idx, ref, genome, batches, hash_bits):
    recs = batches["random+adversarial"]
    po, pg = popts({})
    got = run_bam_input(ctx, idx, recs, genome.names, pg, hash_bits=hash_bits, want_text=False)
    want = expected(ref, genome, got["ks"], got["stride"], po, text=False)
    check(got, want)
