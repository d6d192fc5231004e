"""`qm_driver genome-diff` without a GPU: usage errors exit 1, FASTA refusals exit 2 and write nothing, both before a CUDA context
is asked for; and the paths of rules.genome_diff_command (rule `nucmer`, rules/genome_diff.smk:10-11)."""
import os

import numpy as np
import pytest

from quasimodo_b200 import rules
from quasimodo_b200.genomes import Genome
from tests import drvutil


@pytest.fixture(scope="module")
def fastas(tmp_path_factory):
    d = tmp_path_factory.mktemp("gd")
    rng = np.random.default_rng(3)
    g = Genome(["r"], [3000], rng.integers(0, 4, 3000).astype(np.uint8))
    ref, qry = str(d / "r.fa"), str(d / "q.fa")
    drvutil.write_fasta(g, ref)
    drvutil.write_fasta(g, qry)
    return d, ref, qry


@pytest.mark.parametrize("extra, msg", [
    (["--bogus", "1"], "unknown option"),
    (["-l", "40"], "option -l"),
    (["-l", "7"], "option -l"),
    (["-l", "x"], "option -l"),
    (["-d", "abc"], "option -d"),
    (["-d", "-1"], "option -d"),
    (["-b", "5000"], "-b"),
    (["--indels", "2"], "--indels"),
    (["--indels", "-1"], "indels"),
    (["-c", "-1"], "option -c"),
    (["-g", "-5"], "option -g"),
    (["-b", "x"], "option -b"),
])
def test_usage_errors_exit_1(fastas, extra, msg):
    d, ref, qry = fastas
    p = drvutil.run_driver(["genome-diff", "--ref", ref, "--qry", qry, "--snps", str(d / "o.snps")] + extra, check=False)
    assert p.returncode == 1 and msg in p.stderr, p.stderr
    assert not os.path.exists(d / "o.snps")


def test_required_options(fastas):
    d, ref, qry = fastas
    for argv in (["--qry", qry, "--snps", "x"], ["--ref", ref, "--snps", "x"], ["--ref", ref, "--qry", qry]):
        p = drvutil.run_driver(["genome-diff"] + argv, check=False)
        assert p.returncode == 1, p.stderr


def _bad_fastas(d):
    rng = np.random.default_rng(4)
    seq = "".join("ACGT"[c] for c in rng.integers(0, 4, 300))
    lines = lambda s: "\n".join(s[i:i + 60] for i in range(0, len(s), 60)) + "\n"
    return {
        "n_base": ">a\n" + lines(seq[:100] + "N" + seq[101:]),
        "many_contigs": "".join(f">c{i}\n" + lines(seq) for i in range(17)),
        "ragged_lines": ">a\n" + seq[:60] + "\n" + seq[60:100] + "\n" + seq[100:160] + "\n",
        "empty_contig": ">a\n>b\n" + lines(seq),
        "no_contigs": "\n",
        "twice": ">a\n" + lines(seq) + ">a\n" + lines(seq),
    }


@pytest.mark.parametrize("side", ["ref", "qry"])
@pytest.mark.parametrize("case", ["n_base", "many_contigs", "ragged_lines", "empty_contig", "no_contigs", "twice"])
def test_fasta_refusals_exit_2_and_write_nothing(fastas, tmp_path, side, case):
    d, ref, qry = fastas
    bad = tmp_path / f"{case}.fa"
    bad.write_text(_bad_fastas(tmp_path)[case])
    files = {"ref": ref, "qry": qry, side: str(bad)}
    out = tmp_path / "out"
    out.mkdir()
    p = drvutil.run_driver(["genome-diff", "--ref", files["ref"], "--qry", files["qry"], "--snps", str(out / "x.snps"),
                            "--vcf", str(out / "x.vcf")], check=False)
    assert p.returncode == 2, (p.returncode, p.stderr)
    assert os.listdir(out) == []


def test_genome_diff_command_paths(tmp_path):
    dirs = {"snp_dir": str(tmp_path / "snp")}
    argv, paths = rules.genome_diff_command("/bin/qm_driver", dirs, "TM", "Merlin.fa", "TB40E.fa", threads=3, snps="TM.snps",
                                            benchmark=str(tmp_path / "b" / "nucmer.TM.txt"))
    vcf = str(tmp_path / "snp" / "nucmer" / "TM.maskrepeat.variants.vcf")
    assert paths == [vcf, vcf + ".gz", vcf + ".gz.tbi"]
    assert argv == ["/bin/qm_driver", "genome-diff", "--ref", "Merlin.fa", "--qry", "TB40E.fa", "--vcf", vcf, "-t", "3",
                    "--snps", "TM.snps", "--benchmark", str(tmp_path / "b" / "nucmer.TM.txt")]
    assert os.path.isdir(os.path.dirname(vcf)) and os.path.isdir(tmp_path / "b")
    argv, paths = rules.genome_diff_command("qm", dirs, "TA", "AD169.fa", "TB40E.fa")
    assert argv == ["qm", "genome-diff", "--ref", "AD169.fa", "--qry", "TB40E.fa", "--vcf", paths[0], "-t", "2"]
    assert paths[0].endswith("/nucmer/TA.maskrepeat.variants.vcf")
    assert rules.NUCMER_REF == {"TM": "Merlin", "TA": "AD169"} and rules.NUCMER_QUERY == "TB40E"
