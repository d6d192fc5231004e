"""bwa mem's -K (input chunks of K bases, one insert-size model per chunk) and -I (a given model) on the driver's host side:
option parsing, --print-options, and the cut of the input into chunks (`fastq-check -K`) against a restatement of bwa's
bseq_read (bwa.c, bwa 0.7.17 as recalled)."""
import numpy as np
import pytest

from tests import drvutil


def bseq_read_chunks(lens1, lens2, K):
    """bwa.c bseq_read: pairs in order, both mates' lengths into a running sum, a chunk ends after the first pair at which the sum
    is >= K; the last chunk is whatever remains"""
    out, s, n = [], 0, 0
    for a, b in zip(lens1, lens2):
        s += int(a) + int(b)
        n += 1
        if s >= K:
            out.append(n)
            s, n = 0, 0
    if n:
        out.append(n)
    return out


def resolved(*args):
    p = drvutil.run_driver(["sample", "--print-options", "1", *args])
    return dict(kv.split("=") for kv in p.stdout.split())


def test_print_options_without_k_and_i_is_unchanged():
    r = resolved()
    assert "K" not in r and "I" not in r


@pytest.mark.parametrize("spec,want", [
    ("500", (500.0, 50.0, 700, 300)),                  # std = mean / 10, high / low = mean +- 4 std
    ("500,30", (500.0, 30.0, 620, 380)),
    ("500,30,900", (500.0, 30.0, 900, 380)),
    ("500,30,900,100", (500.0, 30.0, 900, 100)),
    ("250.5;20.25", (250.5, 20.25, 331, 169)),         # any punctuation before a digit separates; (int)(169.5 + .499) = 169
    ("10,5", (10.0, 5.0, 30, 1)),                      # low clamped to 1
    ("300.2,0.1", (300.2, 0.1, 301, 300)),             # (int)(x + .499)
])
def test_dash_i_resolves_as_bwa(spec, want):
    r = resolved("-I", spec)
    avg, std, hi, lo = r["I"].split(",")
    assert (float(avg), float(std), int(hi), int(lo)) == want


def test_dash_k_is_shown():
    assert resolved("-K", "80000000")["K"] == "80000000"
    r = resolved("-K", "1000", "-I", "400")
    assert r["K"] == "1000" and r["I"].startswith("400,40,")


@pytest.mark.parametrize("bad", [["-K", "0"], ["-K", "-5"], ["-K", "1e7"], ["-K", ""], ["-K", "12x"],
                                 ["-I", "abc"], ["-I", "0"], ["-I", "-300"], ["-I", "500,"], ["-I", "500,30x"],
                                 ["-I", "500,30,100,200"], ["-I", ""]])
def test_bad_values_exit_1(bad):
    p = drvutil.run_driver(["sample", "--print-options", "1", *bad], check=False)
    assert p.returncode == 1 and "option -" in p.stderr, (bad, p.stderr)


def test_k_with_decontam_chain_runs_on_one_gpu(tmp_path):
    for f in ("x.fa", "y.fa"):
        (tmp_path / f).write_text(">c\n" + "ACGTTGCA" * 20 + "\n")
    r1, r2 = _fastq(tmp_path, [50] * 10, [50] * 10, "one")
    p = drvutil.run_driver(["sample", "--ref", tmp_path / "x.fa", "--r1", r1, "--r2", r2, "--decontam", tmp_path / "y.fa", "-K", "1000",
                            "--gpus", "0,1"], check=False)
    assert p.returncode == 1 and "one GPU" in p.stderr, p.stderr


def test_chunk_past_the_pair_limit_is_refused_while_reading(tmp_path):
    """K above a sample of more than 2^21 pairs: the read-on stops at the limit and names it, before the sample is held in memory"""
    n = (1 << 21) + 10
    for m, path in ((1, tmp_path / "a.fq"), (2, tmp_path / "b.fq")):
        path.write_text("".join(f"@p{i}/{m}\nA\n+\nI\n" for i in range(n)))
    p = drvutil.run_driver(["fastq-check", "--r1", tmp_path / "a.fq", "--r2", tmp_path / "b.fq", "-K", 10 ** 12, "--batch-pairs", 100000],
                           check=False)
    assert p.returncode == 1 and "QM_CHUNK_MAX_PAIRS" in p.stderr and "2097152" in p.stderr, p.stderr


def _fastq(tmp_path, lens1, lens2, tag):
    rng = np.random.default_rng(len(lens1))
    n = len(lens1)
    L = int(max(max(lens1), max(lens2)))
    codes = rng.integers(0, 4, (2 * n, L)).astype(np.uint8)
    quals = np.full((2 * n, L), 30, np.uint8)
    lens = np.empty(2 * n, np.int64)
    lens[0::2], lens[1::2] = lens1, lens2
    r1, r2 = tmp_path / f"{tag}_1.fq", tmp_path / f"{tag}_2.fq"
    drvutil.write_fastq(codes, quals, lens, drvutil.pair_names("p", n), r1, r2)
    return r1, r2


def _check_cut(tmp_path, lens1, lens2, K, tag, batch=None):
    r1, r2 = _fastq(tmp_path, lens1, lens2, tag)
    args = ["fastq-check", "--r1", r1, "--r2", r2, "-K", K] + (["--batch-pairs", batch] if batch else [])
    p = drvutil.run_driver(args)
    line = [ln for ln in p.stdout.splitlines() if ln.startswith("chunks:")]
    assert len(line) == 1, p.stdout
    got = [int(x) for x in line[0].split()[1:]]
    assert got == bseq_read_chunks(lens1, lens2, K)
    assert sum(got) == len(lens1)
    return got


def test_fastq_check_cut_variable_lengths(tmp_path):
    rng = np.random.default_rng(3)
    lens1 = rng.integers(20, 151, 5000)
    lens2 = rng.integers(1, 151, 5000)
    for K, batch in ((1000, None), (7919, None), (40000, "1000"), (1000, "7"), (10 ** 9, None)):
        got = _check_cut(tmp_path, lens1, lens2, K, f"v{K}_{batch}", batch)
        if K == 10 ** 9:
            assert got == [5000]                       # K above the sample: one chunk of everything


def test_fastq_check_cut_exact_multiple(tmp_path):
    """every pair has 2 x 100 bases and K = 2000: each chunk closes exactly on its 10th pair, and nothing remains"""
    lens = np.full(300, 100)
    got = _check_cut(tmp_path, lens, lens, 2000, "exact")
    assert got == [10] * 30
    got = _check_cut(tmp_path, lens, lens, 2000, "exact_b", batch="25")      # batches end inside chunks: read on to the chunk's end
    assert got == [10] * 30


def test_fastq_check_without_k_prints_no_chunks(tmp_path):
    r1, r2 = _fastq(tmp_path, [50] * 10, [50] * 10, "nok")
    p = drvutil.run_driver(["fastq-check", "--r1", r1, "--r2", r2])
    assert "chunks:" not in p.stdout


def test_rules_builder_takes_chunk_bases(tmp_path):
    from quasimodo_b200 import rules
    dirs = {k: str(tmp_path / k) for k in ("seq_dir", "snpcall_dir", "report_dir")}
    args = dict(driver="qm_driver", dirs=dirs, sample="S", ref_name="R", ref_fa="r.fa", r1="a.fq", r2="b.fq")
    argv, paths = rules.sample_command(**args)
    assert "-K" not in argv
    argv2, paths2 = rules.sample_command(**args, chunk_bases=80000000)
    assert argv2[argv2.index("-K") + 1] == "80000000" and paths2 == paths
    assert [x for x in argv2 if x not in ("-K", "80000000")] == argv
    argv3, _ = rules.decontam_sample_command(**args, phix_fa="phix.fa", chunk_bases=3000000)
    assert argv3[argv3.index("-K") + 1] == "3000000" and "--decontam" in argv3
