"""Static check of the drop-in boundary (SURVEY.md 8b): every `output:` / `log:` / `benchmark:` path the reference's rules `bwa`,
`rmdup`, `mpileup` and `bcftools` declare is one quasimodo_b200.rules knows and the driver command writes.  What the reference's
own rule files declare is stored in tests/golden/rule_contract.json (made by tests/golden/make_rules_golden.py from a Quasimodo
checkout)."""
import json
import os

from quasimodo_b200 import rules

GOLD = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rule_contract.json")))


def test_declared_outputs_of_the_replaced_rules_are_all_produced():
    assert sorted(GOLD["rules"]) == sorted(rules.RULE_OUTPUTS)
    for rule, want in GOLD["rules"].items():
        outs = {k: tuple(v) for k, v in want["output"].items()}
        assert outs == rules.RULE_OUTPUTS[rule], (rule, outs)
        assert (tuple(want["log"]) if want["log"] else None) == rules.RULE_LOGS.get(rule), (rule, want["log"])
        assert (tuple(want["benchmark"]) if want["benchmark"] else None) == rules.RULE_BENCHMARKS.get(rule), (rule, want["benchmark"])
        for name in outs:
            assert (rule, name) in rules.DRIVER_OPTION, f"output {name!r} of rule {rule} has no driver option"
    # the shell lines' side files: `samtools index` after bwa and rmdup, `tabix -p vcf` after bcftools
    side = {}
    for f, lines in GOLD["shell"].items():
        rule_of = {o: r for r, w in GOLD["rules"].items() if w["file"] == f for o in w["output"]}
        for ln in lines:
            out = ln.rsplit("{output.", 1)[1].rstrip("}")
            side[(rule_of[out], out)] = ".bai" if ln.startswith("samtools index ") else ".tbi"
    assert side == rules.SIDE_FILES


def test_sample_command_names_every_path(tmp_path):
    dirs = {k: str(tmp_path / k) for k in ("seq_dir", "snpcall_dir", "report_dir")}
    argv, paths = rules.sample_command("qm_driver", dirs, "TM-1-1", "Merlin", "ref.fa", "a.fq", "b.fq")
    assert len(paths) == 6 + 3 and len(set(paths)) == len(paths)
    for opt in ("--bam", "--rmdup-bam", "--mpileup", "--vcf", "--metrics"):
        assert argv[argv.index(opt) + 1] in paths
    assert str(tmp_path / "seq_dir" / "bam" / "TM-1-1.Merlin.bam") in paths
    assert str(tmp_path / "snpcall_dir" / "bcftools" / "TM-1-1.Merlin.bcftools.vcf.gz.tbi") in paths
    argv_b, paths_b = rules.sample_command("qm_driver", dirs, "TM-1-1", "Merlin", "ref.fa", "a.fq", "b.fq", benchmark=True)
    assert paths_b == paths and argv_b[:len(argv)] == argv
    assert argv_b[-2:] == ["--benchmark", str(tmp_path / "report_dir" / "benchmarks" / "TM-1-1.Merlin.bcftools.benchmark.txt")]
