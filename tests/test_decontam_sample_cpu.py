"""CPU checks of `qm_driver sample --decontam`: the usage errors of the new options, a contaminant FASTA refused before any CUDA
context, a valid command reaching the context (exit 3 without a GPU), and the paths of rules.decontam_sample_command."""
import pytest

from quasimodo_b200 import rules
from tests import drvutil


@pytest.fixture()
def files(tmp_path):
    fa = tmp_path / "t.fa"
    fa.write_text(">t\n" + "ACGT" * 50 + "\n")
    (tmp_path / "p.fa").write_text(">phix\n" + "GATTACA" * 20 + "\n")
    (tmp_path / "r1.fq").write_text("@a/1\nACGTACGT\n+\nIIIIIIII\n")
    (tmp_path / "r2.fq").write_text("@a/2\nACGTACGT\n+\nIIIIIIII\n")
    return tmp_path


def run(d, *extra, cmd="sample"):
    base = [cmd, "--ref", d / "t.fa", "--r1", d / "r1.fq", "--r2", d / "r2.fq"]
    if cmd == "decontam":
        base += ["--out-r1", d / "o1.fq", "--out-r2", d / "o2.fq"]
    return drvutil.run_driver(base + list(extra), check=False)


@pytest.mark.parametrize("extra,name", [
    (["--decontam2", "p.fa"], "--decontam2"),
    (["--decontam", "p.fa", "--clean-r1", "c1.fq"], "--clean-r2"),
    (["--decontam", "p.fa", "--clean-r2", "c2.fq"], "--clean-r1"),
    (["--clean-r1", "c1.fq", "--clean-r2", "c2.fq"], "--clean-r1"),
    (["--decontam", "p.fa", "--keep-contigs", "1"], "--keep-contigs"),
])
def test_usage_errors_name_the_option(files, extra, name):
    extra = [str(files / x) if x.endswith((".fa", ".fq")) else x for x in extra]
    p = run(files, *extra)
    assert p.returncode == 1 and name in p.stderr, p.stderr


@pytest.mark.parametrize("opt", ["decontam", "decontam2", "clean-r1", "clean-r2"])
def test_decontam_command_does_not_take_the_new_options(files, opt):
    p = run(files, f"--{opt}", files / "p.fa", cmd="decontam")
    assert p.returncode == 1 and f"unknown option '--{opt}'" in p.stderr, p.stderr


@pytest.mark.parametrize("opt", ["decontam", "decontam2"])
@pytest.mark.parametrize("text,msg", [(">p\nACGTNACGT\n", "base 'N'"), (">p\nACGT\n>q\n\n>r\nAC\n", "contig q is empty")])
def test_bad_pass_fasta_exits_2_before_the_context(files, opt, text, msg):
    bad = files / "bad.fa"
    bad.write_text(text)
    extra = ["--decontam", files / "p.fa"] if opt == "decontam2" else []
    p = run(files, *extra, f"--{opt}", bad, "--gpu", 99)
    assert p.returncode == 2 and msg in p.stderr and str(bad) in p.stderr, p.stderr


def test_valid_command_reaches_the_context(files):
    (files / "e.fa").write_text(">ecoli\n" + "CCGGA" * 30 + "\n>human\nTTGCA\n")
    p = run(files, "--decontam", files / "p.fa", "--decontam2", f"{files / 'e.fa'},{files / 't.fa'}", "--clean-r1", files / "c1.fq",
            "--clean-r2", files / "c2.fq", "--gpus", "0,1", "--gpu", 99)
    assert p.returncode == 3 and "no usable B200" in p.stderr, p.stderr


def test_decontam_sample_command_names_every_path(tmp_path):
    dirs = {k: str(tmp_path / k) for k in ("seq_dir", "snpcall_dir", "report_dir")}
    _, plain = rules.sample_command("qm_driver", dirs, "TM-1-1", "Merlin", "ref.fa", "a.fq", "b.fq")
    argv, paths = rules.decontam_sample_command("qm_driver", dirs, "TM-1-1", "Merlin", "ref.fa", "a.fq", "b.fq", "phix.fa",
                                                ["human.fa", "ecoli.fa"], benchmark=True)
    cl = [str(tmp_path / "seq_dir" / "cl_fq" / f"TM-1-1.qc.cl.r{m}.fq") for m in (1, 2)]
    assert paths == plain + cl and len(set(paths)) == len(paths)
    assert argv[argv.index("--decontam") + 1] == "phix.fa" and argv[argv.index("--decontam2") + 1] == "human.fa,ecoli.fa"
    assert argv[argv.index("--clean-r1") + 1] == cl[0] and argv[argv.index("--clean-r2") + 1] == cl[1]
    assert argv[argv.index("--r1") + 1] == "a.fq" and "--benchmark" in argv
    for opt in ("--bam", "--rmdup-bam", "--mpileup", "--vcf", "--metrics"):
        assert argv[argv.index(opt) + 1] in paths
    argv1, paths1 = rules.decontam_sample_command("qm_driver", dirs, "TM-1-1", "Merlin", "ref.fa", "a.fq", "b.fq", "phix.fa")
    assert "--decontam2" not in argv1
    assert paths1[-2:] == [str(tmp_path / "seq_dir" / "cl_fq" / f"TM-1-1.qc.nophix.r{m}.fq") for m in (1, 2)]
