"""CPU tests of `qm_driver index`: everything the host checks before a CUDA context exists.  Each FASTA that `bwa index` or
`samtools faidx` would not index as this command does must exit 2 with a message naming the contig, the line or the limit; usage
errors exit 1; a valid FASTA gets as far as the context, which without a GPU is exit 3.  And rules.index_command names the
files the two tools write."""
import os

from quasimodo_b200 import rules
from tests import drvutil
from tests.test_bam_input_cpu import has_gpu


def run_index(tmp_path, text, extra=()):
    fa = tmp_path / "g.fa"
    fa.write_bytes(text.encode() if isinstance(text, str) else text)
    return drvutil.run_driver(["index", "--ref", fa, "--prefix", tmp_path / "idx"] + list(extra), check=False)


def expect_2(res, words):
    assert res.returncode == 2, res.stderr
    for w in words:
        assert w in res.stderr, res.stderr


def expect_valid(res):
    assert res.returncode == (0 if has_gpu() else 3), res.stderr
    if not has_gpu():
        assert "no usable B200" in res.stderr


def test_valid_fasta_needs_a_gpu(tmp_path):
    expect_valid(run_index(tmp_path, ">c1 first contig\nACGTACGT\nACGTAC\n>c2\nGGGG\n"))
    expect_valid(run_index(tmp_path, ">c1\r\nACGT\r\nAC\r\n"))                      # CRLF lines
    expect_valid(run_index(tmp_path, ">c1\nACGTACGT\nACG\n\n\n>c2\nT"))           # blank lines behind a contig, no final newline
    expect_valid(run_index(tmp_path, "".join(f">c{i}\nacgt\n" for i in range(16))))   # 16 contigs, lower case


def test_no_contig_or_an_empty_one(tmp_path):
    expect_2(run_index(tmp_path, ""), ["no contigs"])
    expect_2(run_index(tmp_path, "\n\n"), ["no contigs"])
    expect_2(run_index(tmp_path, ">c1\nACGT\n>c2\n>c3\nAC\n"), ["contig c2 has no bases"])
    expect_2(run_index(tmp_path, ">c1\nACGT\n>c2\n"), ["contig c2 has no bases"])
    expect_2(run_index(tmp_path, "ACGT\n>c1\nACGT\n"), ["line 1", "before the first '>'"])
    expect_2(run_index(tmp_path, "> anno only\nACGT\n"), ["line 1", "without a name"])


def test_duplicate_names(tmp_path):
    expect_2(run_index(tmp_path, ">c1 one\nACGT\n>c2\nAC\n>c1 two\nGG\n"), ["line 5", "c1 occurs twice"])


def test_too_many_contigs(tmp_path):
    expect_2(run_index(tmp_path, "".join(f">c{i}\nACGT\n" for i in range(17))), ["line 33", "more than 16 contigs"])


def test_bases_outside_acgt(tmp_path):
    expect_2(run_index(tmp_path, ">c1\nACGT\n>c2\nACGT\nACNT\n"), ["line 5", "base 'N'", "contig c2", "A/C/G/T"])
    expect_2(run_index(tmp_path, ">c1\nAC-T\n"), ["line 2", "base '-'", "contig c1"])
    expect_2(run_index(tmp_path, ">c1\nACRT\n"), ["base 'R'"])


def test_line_lengths_faidx_refuses(tmp_path):
    # a line longer than the contig's first
    expect_2(run_index(tmp_path, ">c1\nACGT\nACGTA\nAC\n"), ["contig c1", "line 3", "samtools faidx"])
    # a short line with more sequence behind it
    expect_2(run_index(tmp_path, ">c1\nACGT\nAC\nACGT\n"), ["contig c1", "line 3", "samtools faidx"])
    # a blank line inside a contig
    expect_2(run_index(tmp_path, ">c0\nAAAA\n>c1\nACGT\n\nACGT\n"), ["contig c1", "line 5", "samtools faidx"])
    # a change of line terminator inside a contig
    expect_2(run_index(tmp_path, ">c1\nACGT\r\nACGT\nAC\n"), ["contig c1", "line 3", "samtools faidx"])


def test_compressed_fasta(tmp_path):
    import gzip
    expect_2(run_index(tmp_path, gzip.compress(b">c1\nACGT\n")), ["compressed"])


def test_missing_file(tmp_path):
    res = drvutil.run_driver(["index", "--ref", tmp_path / "absent.fa"], check=False)
    assert res.returncode == 2 and "cannot open" in res.stderr


def test_usage_errors(tmp_path):
    res = run_index(tmp_path, ">c1\nACGT\n", extra=["--bam", "x.bam"])
    assert res.returncode == 1 and "unknown option '--bam'" in res.stderr
    res = run_index(tmp_path, ">c1\nACGT\n", extra=["-a", "bwtsw"])
    assert res.returncode == 1 and "unknown option '-a'" in res.stderr
    res = drvutil.run_driver(["index", "--prefix", tmp_path / "p"], check=False)
    assert res.returncode == 1 and "--ref" in res.stderr
    res = drvutil.run_driver(["index", "--ref"], check=False)
    assert res.returncode == 1
    res = drvutil.run_driver([], check=False)
    assert res.returncode == 1 and "index" in res.stderr


def test_nothing_written_on_refusal(tmp_path):
    run_index(tmp_path, ">c1\nACNT\n")
    assert sorted(os.listdir(tmp_path)) == ["g.fa"]


def test_index_command_paths(tmp_path):
    fa = str(tmp_path / "ref" / "Merlin.BAC.fa")
    argv, paths = rules.index_command("qm_driver", fa, threads=8)
    assert argv == ["qm_driver", "index", "--ref", fa, "-t", "8"]
    # `bwa index X.fa` (prefix = the FASTA path) and `samtools faidx X.fa`
    assert paths == [fa + ".amb", fa + ".ann", fa + ".bwt", fa + ".pac", fa + ".sa", fa + ".fai"]
    b = str(tmp_path / "bench" / "Merlin.index.benchmark.txt")
    argv, paths2 = rules.index_command("qm_driver", fa, benchmark=b, extra=["--gpu", "1"])
    assert argv[-4:] == ["--benchmark", b, "--gpu", "1"] and paths2 == paths
    assert os.path.isdir(os.path.dirname(b))
    # the sample commands take the same prefix: --bwa-index X.fa reads X.fa.bwt and X.fa.sa
    assert {p[len(fa):] for p in paths} >= {".bwt", ".sa"}
