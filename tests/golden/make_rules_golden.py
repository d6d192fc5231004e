#!/usr/bin/env python3
"""Golden file contract of the reference rules this implementation replaces, parsed from hzi-bifo/Quasimodo's own rule files:
the `output:`, `log:` and `benchmark:` entries of rules `bwa` (rules/bwa.smk:1-19), `rmdup` (rules/rmdup.smk:1-18), `mpileup`
(rules/vcfcall.smk:26-40) and `bcftools` (rules/vcfcall.smk:101-120), and the shell lines that leave side files next to a
declared output (`samtools index`, `tabix -p vcf`).  Writes tests/golden/rule_contract.json, which tests/test_rules_cpu.py
holds quasimodo_b200/rules.py against.

The committed file holds what this parser returned on the rule files when the comparison last ran against them (commit
fc104e4, where rules.py gained the `benchmark:` paths); rules.py's tables have not changed since.
Usage: python tests/golden/make_rules_golden.py QUASIMODO_CHECKOUT"""
import json
import os
import re
import sys

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "rule_contract.json")
WHERE = {"bwa": "bwa.smk", "rmdup": "rmdup.smk", "mpileup": "vcfcall.smk", "bcftools": "vcfcall.smk"}
SHELL = {"bwa.smk": ["samtools index {output.sortedbam}"], "rmdup.smk": ["samtools index {output.rmdupbam}"],
         "vcfcall.smk": ["tabix -p vcf {output.vcf_bgz}"]}


def parse_rule(path, rule):
    """-> (outputs {name: (dir variable, pattern)}, log (dir variable, pattern) or None, benchmark likewise) of `rule` in a .smk file"""
    text = open(path).read()
    m = re.search(rf"^rule {rule}:\n(.*?)(?=^rule |\Z)", text, re.S | re.M)
    assert m, f"rule {rule} not found in {path}"
    body = m.group(1)

    def section(key):
        s = re.search(rf"^    {key}:\s*\n((?:^        .*\n|^\s*\n)*)", body, re.M)
        return s.group(1) if s else ""

    def entries(sec):
        out = {}
        for ln in sec.splitlines():
            ln = ln.split("#")[0].strip().rstrip(",")
            if not ln:
                continue
            e = re.match(r'(?:(\w+)\s*=\s*)?(\w+)\s*\+\s*"([^"]+)"$', ln)
            assert e, f"unparsed line in rule {rule}: {ln!r}"
            out[e.group(1) or ""] = (e.group(2), e.group(3))
        return out

    outs = entries(section("output"))
    log = entries(section("log"))
    bench = entries(section("benchmark"))
    return outs, (log.get("") if log else None), (bench.get("") if bench else None)


def main(root):
    rules = {}
    for rule, f in WHERE.items():
        outs, log, bench = parse_rule(os.path.join(root, "rules", f), rule)
        rules[rule] = {"file": f, "output": {k: list(v) for k, v in outs.items()},
                       "log": list(log) if log else None, "benchmark": list(bench) if bench else None}
    for f, lines in SHELL.items():
        text = open(os.path.join(root, "rules", f)).read()
        for ln in lines:
            assert ln in text, f"{ln!r} not in rules/{f}"
    with open(OUT, "w") as fh:
        fh.write(json.dumps({"rules": rules, "shell": SHELL}, indent=1) + "\n")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__.rsplit("\n", 1)[-1])
    main(sys.argv[1])
