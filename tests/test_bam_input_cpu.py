"""CPU tests of `qm_driver pileup`'s BAM reader: everything the host checks before a CUDA context exists.  The BGZF layer is
damaged in a BAM written by `qm_driver bam-from-records --perm` (no GPU touched); header and record failures come from the
small BAM writer below.  Each must exit 2 with a message naming the problem; an unknown option is a usage error (1); a valid
BAM gets as far as the context, which without a GPU is exit 3."""
import ctypes
import struct
import zlib

import numpy as np
import pytest

from tests import drvutil, recgen

CIGAR_OPS = "MIDNSHP=X"
_NT16 = {c: i for i, c in enumerate("=ACMGRSVTWYHKDBN")}
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf(data, block=0xff00):
    """BGZF members of at most `block` uncompressed bytes each, then the end-of-file block"""
    out = bytearray()
    for i in range(0, len(data), block):
        chunk = data[i:i + block]
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        comp = co.compress(chunk) + co.flush()
        out += b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", 18 + len(comp) + 8 - 1)
        out += comp + struct.pack("<II", zlib.crc32(chunk), len(chunk))
    return bytes(out) + EOF_BLOCK


def record(name, rid, pos, cigar, seq, qual=None, flag=0x1 | 0x2 | 0x40, mapq=60, mrid=-1, mpos=-1, tlen=0, tags=b""):
    """one BAM record; cigar: "10M2I5S" style, seq: SAM letters or "" for '*', qual: phred list or None for '*'"""
    ops = []
    num = ""
    for ch in cigar:
        if ch.isdigit():
            num += ch
        else:
            ops.append((int(num) << 4) | CIGAR_OPS.index(ch))
            num = ""
    l_seq = len(seq)
    nb = bytearray((l_seq + 1) // 2)
    for i, ch in enumerate(seq):
        nb[i >> 1] |= _NT16[ch] << (0 if i & 1 else 4)
    q = bytes([0xff] * l_seq) if qual is None else bytes(qual)
    nm = name.encode() + b"\0"
    body = struct.pack("<iiBBHHHiiii", rid, pos, len(nm), mapq, 4680, len(ops), flag, l_seq, mrid, mpos, tlen)
    body += nm + struct.pack(f"<{len(ops)}I", *ops) + bytes(nb) + q + tags
    return struct.pack("<i", len(body)) + body


def bam(refs, records, magic=b"BAM\x01"):
    text = b"@HD\tVN:1.6\tSO:coordinate\n"
    hdr = magic + struct.pack("<i", len(text)) + text + struct.pack("<i", len(refs))
    for name, ln in refs:
        hdr += struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + struct.pack("<i", ln)
    return bgzf(hdr + b"".join(records))


def has_gpu():
    try:
        cu = ctypes.CDLL("libcuda.so.1")
        n = ctypes.c_int(0)
        return cu.cuInit(0) == 0 and cu.cuDeviceGetCount(ctypes.byref(n)) == 0 and n.value > 0
    except OSError:
        return False


@pytest.fixture(scope="module")
def case(tmp_path_factory):
    d = tmp_path_factory.mktemp("bamin")
    g = recgen.Genome()
    ref = d / "ref.fa"
    drvutil.write_fasta(g, ref)
    b = recgen.random_batch(g, 60, 7)
    alns, codes, quals, lens = b.arrays()
    quals = np.minimum(quals, 60)
    names = drvutil.pair_names("bamin", len(alns) // 2)
    drvutil.write_fastq(codes, quals, lens, names, d / "r1.fq", d / "r2.fq")
    alns.tofile(d / "alns.bin")
    n_c = len(g.lens)
    keys = [((n_c if a["rid"] < 0 else int(a["rid"])) << 33) | ((int(a["pos"]) + 1) << 1) | ((int(a["flag"]) >> 4) & 1) for a in alns]
    np.argsort(np.array(keys, np.uint64), kind="stable").astype(np.uint32).tofile(d / "perm.bin")
    drvutil.run_driver(["bam-from-records", "--ref", ref, "--r1", d / "r1.fq", "--r2", d / "r2.fq", "--alns", d / "alns.bin",
                        "--perm", d / "perm.bin", "--bam", d / "ok.bam"])
    refs = list(zip(g.names, [int(x) for x in g.lens]))
    return dict(d=d, g=g, ref=ref, ok=(d / "ok.bam").read_bytes(), refs=refs)


def run_pileup(case, data, name="in.bam", extra=()):
    p = case["d"] / name
    p.write_bytes(data)
    return drvutil.run_driver(["pileup", "--ref", case["ref"], "--bam", p, "--counts", case["d"] / "out.tsv"] + list(extra), check=False)


def expect_2(res, words):
    assert res.returncode == 2, res.stderr
    for w in words:
        assert w in res.stderr, res.stderr


def test_valid_bam_needs_a_gpu(case):
    res = run_pileup(case, case["ok"])
    if has_gpu():
        assert res.returncode == 0, res.stderr
    else:
        assert res.returncode == 3, res.stderr
        assert "no usable B200" in res.stderr


def test_unknown_option_is_a_usage_error(case):
    res = run_pileup(case, case["ok"], extra=["--min-qual", "20"])
    assert res.returncode == 1 and "unknown option '--min-qual'" in res.stderr
    res = drvutil.run_driver(["pileup", "--ref", case["ref"]], check=False)
    assert res.returncode == 1


def test_bgzf_damage(case):
    ok = case["ok"]
    expect_2(run_pileup(case, ok[:len(ok) // 2]), ["truncated BGZF block"])
    expect_2(run_pileup(case, ok[:-28]), ["no BGZF end-of-file block"])
    bsize = struct.unpack_from("<H", ok, 16)[0] + 1
    bad = bytearray(ok)
    bad[bsize - 8] ^= 0xff                                   # the first block's CRC32
    expect_2(run_pileup(case, bytes(bad)), ["CRC32 mismatch", "byte 0"])
    bad = bytearray(ok)
    bad[0] = 0x1e
    expect_2(run_pileup(case, bytes(bad)), ["bad BGZF magic"])
    expect_2(run_pileup(case, bam(case["refs"], [], magic=b"BAX\x01")), ["bad BAM magic"])


def test_header_must_match_the_reference(case):
    refs = case["refs"]
    renamed = [("chrZ", refs[0][1])] + refs[1:]
    expect_2(run_pileup(case, bam(renamed, [])), ["@SQ 1 is chrZ", "not aligned to this reference"])
    longer = refs[:2] + [(refs[2][0], refs[2][1] + 1)] + refs[3:]
    expect_2(run_pileup(case, bam(longer, [])), ["@SQ 3 is chrC of 518 bp"])
    swapped = [refs[1], refs[0]] + refs[2:]
    expect_2(run_pileup(case, bam(swapped, [])), ["@SQ 1 is chrB"])
    expect_2(run_pileup(case, bam(refs[:3], [])), ["3 contigs"])
    # the header alone (no records) is a valid, empty input
    res = run_pileup(case, bam(refs, []))
    assert res.returncode == (0 if has_gpu() else 3), res.stderr


def _r(name, pos, cigar="10M", seq="ACGTACGTAC", rid=0, **kw):
    return record(name, rid, pos, cigar, seq, kw.pop("qual", [30] * len(seq)), **kw)


@pytest.mark.parametrize("recs,words", [
    ([_r("a", 20), _r("b", 10)], ["not coordinate-sorted", "read b", "chrA:11"]),
    ([_r("a", 5, rid=2), _r("b", 10, rid=0)], ["not coordinate-sorted", "read b"]),
    ([_r("n_op", 5, cigar="4M3N6M")], ["read n_op", "CIGAR operation N"]),
    ([_r("p_op", 5, cigar="4M3P6M")], ["read p_op", "CIGAR operation P"]),
    ([_r("ops22", 5, cigar="1M1I" * 10 + "1M1S", seq="A" * 22)], ["read ops22", "22 CIGAR operations"]),
    ([_r("long", 0, rid=2, cigar="513M", seq="A" * 513)], ["read long", "513 bases"]),
    ([_r("noseq", 5, seq="", cigar="10M", qual=[])], ["read noseq", "no stored SEQ"]),
    ([_r("noqual", 5, qual=None)], ["read noqual", "no stored QUAL"]),
    ([_r("qlen", 5, cigar="9M")], ["read qlen", "CIGAR query length 9"]),
    ([_r("past", 295)], ["read past", "outside contig chrA"]),
], ids=["unsorted", "unsorted-contigs", "N-op", "P-op", "22-ops", "513-bases", "no-SEQ", "no-QUAL", "query-length", "past-end"])
def test_bad_records(case, recs, words):
    expect_2(run_pileup(case, bam(case["refs"], recs)), words)


def test_records_never_admitted_are_not_checked(case):
    # unmapped, secondary, QC-failed and duplicate records are left out before any check: their CIGARs do not matter, nor does
    # the position of an unmapped record
    recs = [_r("dup", 5, cigar="4M3N6M", flag=0x1 | 0x400), _r("sec", 6, cigar="22M", seq="A" * 22, flag=0x100),
            _r("qc", 7, seq="", qual=[], flag=0x200), _r("ok", 8), _r("unm", 3, flag=0x1 | 0x4), _r("hclip", 9, cigar="5H10M5H")]
    res = run_pileup(case, bam(case["refs"], recs))
    assert res.returncode == (0 if has_gpu() else 3), res.stderr
    assert "6 records, 4 left out" in res.stderr
