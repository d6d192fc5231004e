"""CPU checks of the per-rule replacements of `mpileup` and `bcftools` (rules.pileup_commands): each reads the rule's input BAM
and writes the paths the rule declares, with its own benchmark file."""
from quasimodo_b200 import rules


def test_pileup_commands_name_each_rules_paths(tmp_path):
    dirs = {k: str(tmp_path / k) for k in ("seq_dir", "snpcall_dir", "report_dir")}
    cmds = rules.pileup_commands("qm_driver", dirs, "TM-1-1", "Merlin", "ref.fa", benchmark=True)
    assert sorted(cmds) == ["bcftools", "mpileup"]
    bam = str(tmp_path / "seq_dir" / "bam" / "TM-1-1.Merlin.rmdup.bam")
    for rule, (argv, paths) in cmds.items():
        assert argv[1] == "pileup" and argv[argv.index("--bam") + 1] == bam
        for name in rules.RULE_OUTPUTS[rule]:
            assert rules.expand(dirs, rule, name, "TM-1-1", "Merlin") in paths
        assert argv[-2:] == ["--benchmark", rules.benchmark_path(dirs, rule, "TM-1-1", "Merlin")]
        assert "--r1" not in argv and "--rmdup" not in argv
    m_argv, m_paths = cmds["mpileup"]
    assert m_paths == [str(tmp_path / "seq_dir" / "pileup" / "TM-1-1.Merlin.mpileup")] and "--vcf" not in m_argv
    b_argv, b_paths = cmds["bcftools"]
    vcf = str(tmp_path / "snpcall_dir" / "bcftools" / "TM-1-1.Merlin.bcftools.vcf")
    assert b_argv[b_argv.index("--vcf") + 1] == vcf and "--mpileup" not in b_argv
    assert b_paths == [vcf, vcf + ".gz", vcf + ".gz.tbi"]
