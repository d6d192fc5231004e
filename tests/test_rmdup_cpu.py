"""CPU tests of `qm_driver rmdup`: everything the host checks before a CUDA context exists.  Each failure of the header or of a
record must exit 2 with a message naming the read or the limit; usage errors exit 1; a valid BAM -- including the records the
pileup's reader refuses but duplicate marking accepts (N and P operations, reads over 512 bases, more than 21 operations, QUAL
'*') -- gets as far as the context, which without a GPU is exit 3.  And rules.rmdup_command names the rule's paths."""
import struct

import pytest

from quasimodo_b200 import rules
from tests import drvutil, recgen
from tests.test_bam_input_cpu import bgzf, has_gpu, record

REFS = list(zip(recgen.Genome().names, [int(x) for x in recgen.Genome().lens]))       # chrA 300, chrB 1, chrC 517, chrD 64


def bam(records, refs=REFS, text="@HD\tVN:1.6\tSO:coordinate\n", magic=b"BAM\x01"):
    t = text.encode()
    hdr = magic + struct.pack("<i", len(t)) + t + struct.pack("<i", len(refs))
    for name, ln in refs:
        hdr += struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + struct.pack("<i", ln)
    return bgzf(hdr + b"".join(records))


def _r(name, pos, cigar="10M", seq="ACGTACGTAC", rid=0, **kw):
    return record(name, rid, pos, cigar, seq, kw.pop("qual", [30] * len(seq)), **kw)


def run_rmdup(tmp_path, data, extra=()):
    p = tmp_path / "in.bam"
    p.write_bytes(data)
    return drvutil.run_driver(["rmdup", "--bam", p, "--rmdup-bam", tmp_path / "out.bam", "--metrics", tmp_path / "m.txt"] + list(extra),
                              check=False)


def expect_2(res, words):
    assert res.returncode == 2, res.stderr
    for w in words:
        assert w in res.stderr, res.stderr


def expect_valid(res):
    assert res.returncode == (0 if has_gpu() else 3), res.stderr
    if not has_gpu():
        assert "no usable B200" in res.stderr


def test_valid_bam_needs_a_gpu(tmp_path):
    expect_valid(run_rmdup(tmp_path, bam([_r("a", 5), _r("b", 5, flag=0x1 | 0x80 | 0x10), _r("u", -1, rid=-1, cigar="", flag=0x1 | 0x4)])))
    expect_valid(run_rmdup(tmp_path, bam([])))                       # the header alone


def test_usage_errors(tmp_path):
    res = run_rmdup(tmp_path, bam([]), extra=["--ref", "x.fa"])
    assert res.returncode == 1 and "unknown option '--ref'" in res.stderr
    res = drvutil.run_driver(["rmdup", "--bam", tmp_path / "in.bam"], check=False)
    assert res.returncode == 1 and "--rmdup-bam" in res.stderr
    res = drvutil.run_driver(["rmdup", "--rmdup-bam", tmp_path / "o.bam"], check=False)
    assert res.returncode == 1
    res = drvutil.run_driver([], check=False)
    assert res.returncode == 1 and "rmdup" in res.stderr


def test_bad_bam_and_header(tmp_path):
    expect_2(run_rmdup(tmp_path, bam([], magic=b"BAX\x01")), ["bad BAM magic"])
    expect_2(run_rmdup(tmp_path, bgzf(b"BAM\x01" + struct.pack("<i", 100) + b"@HD\tVN:1.6\n")), ["truncated BAM header"])
    expect_2(run_rmdup(tmp_path, bam([], refs=[(f"c{i}", 100) for i in range(17)])), ["17 contigs", "at most 16"])
    expect_2(run_rmdup(tmp_path, bam([], refs=REFS[:1] + [("big", (1 << 26) - 4096)])), ["@SQ big", "under 2^26 - 4096"])
    rg = "@HD\tVN:1.6\tSO:coordinate\n@RG\tID:a\tLB:lib1\tSM:s\n@RG\tID:b\tLB:lib2\tSM:s\n"
    expect_2(run_rmdup(tmp_path, bam([], text=rg)), ["2 libraries (LB)"])
    # two read groups of one library are fine
    expect_valid(run_rmdup(tmp_path, bam([], text=rg.replace("lib2", "lib1"))))


def _malformed():
    r = bytearray(_r("short", 5))
    struct.pack_into("<i", r, 20, 400)                    # l_seq of 400 bases in a record that stores 10
    return bytes(r)


def _op9():
    r = bytearray(_r("op9", 5, cigar="5M5M"))
    struct.pack_into("<I", r, 36 + 4 + 4, (5 << 4) | 9)   # the second CIGAR word (after the fixed fields and "op9\0"): operation 9
    return bytes(r)


@pytest.mark.parametrize("recs,words", [
    ([_r("ok", 3), _malformed()], ["read short", "malformed record"]),
    ([_r("far", 5, rid=4)], ["read far", "contig id 4 is not in the header"]),
    ([_r("neg", 5, rid=-2)], ["read neg", "contig id -2"]),
    ([_op9()], ["read op9", "invalid CIGAR operation 9"]),
    ([_r("a", 20), _r("b", 10)], ["not coordinate-sorted", "read b", "chrA:11"]),
    ([_r("a", 5, rid=2), _r("b", 10, rid=0)], ["not coordinate-sorted", "read b"]),
    ([_r("u", -1, rid=-1, cigar="", flag=0x1 | 0x4), _r("late", 10)], ["read late", "after records without a contig"]),
    ([_r("hclip", 10, cigar="5000H10M")], ["read hclip", "unclipped 5' coordinate -4989"]),
    ([_r("rclip", 60, rid=3, cigar="4M67108860H", seq="ACGT", flag=0x1 | 0x40 | 0x10)], ["read rclip", "unclipped 5' coordinate"]),
], ids=["malformed", "contig-id", "negative-contig-id", "cigar-op-9", "unsorted", "unsorted-contigs", "contig-after-unplaced",
        "clip-before-contig", "clip-past-end-code"])
def test_bad_records(tmp_path, recs, words):
    expect_2(run_rmdup(tmp_path, bam(recs)), words)


def test_accepted_oddities(tmp_path):
    """what the pileup's reader refuses is fine here: N and P, 600 bases, 30 operations, QUAL '*', SEQ '*', an unmapped pair at
    the end, a 0x400 flag and a supplementary record with hard clips"""
    recs = [_r("n_op", 5, cigar="4M3N6M"), _r("p_op", 6, cigar="4M3P6M"), _r("long", 0, rid=2, cigar="600M", seq="A" * 600),
            _r("ops30", 1, rid=2, cigar="1M1I" * 14 + "1M1S", seq="A" * 30), _r("noqual", 2, rid=2, qual=None),
            _r("noseq", 3, rid=2, seq="", cigar="10M", qual=[]), _r("dup", 4, rid=2, flag=0x1 | 0x40 | 0x400),
            _r("supp", 5, rid=2, cigar="20H10M", flag=0x1 | 0x40 | 0x800),
            _r("u", -1, rid=-1, cigar="", flag=0x1 | 0x4 | 0x40), _r("u", -1, rid=-1, cigar="", flag=0x1 | 0x4 | 0x80)]
    expect_valid(run_rmdup(tmp_path, bam(recs)))


def test_rmdup_command_names_the_rules_paths(tmp_path):
    dirs = {k: str(tmp_path / k) for k in ("seq_dir", "report_dir", "snpcall_dir")}
    argv, paths = rules.rmdup_command("qm_driver", dirs, "TM-1-1", "Merlin", threads=8)
    bam = str(tmp_path / "seq_dir" / "bam" / "TM-1-1.Merlin.bam")
    rbam = str(tmp_path / "seq_dir" / "bam" / "TM-1-1.Merlin.rmdup.bam")
    log = str(tmp_path / "report_dir" / "picard" / "TM-1-1.Merlin.rmdup.metrics.txt")
    assert paths == [rbam, rbam + ".bai", log]
    assert argv[:2] == ["qm_driver", "rmdup"] and "--ref" not in argv
    for opt, val in (("--bam", bam), ("--rmdup-bam", rbam), ("--metrics", log), ("--sample", "TM-1-1"), ("-t", "8")):
        assert argv[argv.index(opt) + 1] == val
    assert rules.expand(dirs, "rmdup", "rmdupbam", "TM-1-1", "Merlin") == rbam
