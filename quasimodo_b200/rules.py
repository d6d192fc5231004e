"""The file contract of the reference rules this implementation replaces (SURVEY.md 8b): the declared `output:` / `log:`
paths of rules `bwa` (rules/bwa.smk:1-19), `rmdup` (rules/rmdup.smk:1-18), `mpileup` (rules/vcfcall.smk:26-40) and `bcftools`
(rules/vcfcall.smk:101-120), and the ONE `qm_driver sample` invocation that produces all of them.  Snakemake deletes a job
whose declared output is missing, so tests/test_rules_cpu.py checks these tables against the reference's rule files and
tests/test_driver_gpu.py checks that the command really writes every path.  pileup_commands gives rules `mpileup` and
`bcftools` one `qm_driver pileup` job each, on the .rmdup.bam a separate alignment step left."""
import os

# rule -> {output name ("" = the rule's single unnamed output): (directory variable, path pattern)}
RULE_OUTPUTS = {
    "bwa": {"sortedbam": ("seq_dir", "/bam/{sample}.{ref_name}.bam")},
    "rmdup": {"rmdupbam": ("seq_dir", "/bam/{sample}.{ref_name}.rmdup.bam")},
    "mpileup": {"": ("seq_dir", "/pileup/{sample}.{ref_name}.mpileup")},
    "bcftools": {"vcf": ("snpcall_dir", "/bcftools/{sample}.{ref_name}.bcftools.vcf"),
                 "vcf_bgz": ("snpcall_dir", "/bcftools/{sample}.{ref_name}.bcftools.vcf.gz")},
}
RULE_LOGS = {
    "bwa": ("report_dir", "/bwa/{sample}.{ref_name}.log"),
    "rmdup": ("report_dir", "/picard/{sample}.{ref_name}.rmdup.metrics.txt"),
}
# `benchmark:` files of the replaced rules (rules/vcfcall.smk:32-33,108-109; `bwa` and `rmdup` declare none): one driver job stands
# for all four rules, its `--benchmark` file goes to the last rule's path; the per-rule `qm_driver pileup` jobs
# (pileup_commands) write one each
RULE_BENCHMARKS = {
    "mpileup": ("report_dir", "/benchmarks/{sample}.{ref_name}.mpileup.benchmark.txt"),
    "bcftools": ("report_dir", "/benchmarks/{sample}.{ref_name}.bcftools.benchmark.txt"),
}
# files the rules' shell lines leave next to a declared output (`samtools index`, `tabix -p vcf`)
SIDE_FILES = {("bwa", "sortedbam"): ".bai", ("rmdup", "rmdupbam"): ".bai", ("bcftools", "vcf_bgz"): ".tbi"}
# which driver option writes which declared path
DRIVER_OPTION = {("bwa", "sortedbam"): "--bam", ("rmdup", "rmdupbam"): "--rmdup-bam", ("mpileup", ""): "--mpileup",
                 ("bcftools", "vcf"): "--vcf", ("bcftools", "vcf_bgz"): None,      # written next to --vcf (bgzip -c + tabix)
                 ("rmdup", "log"): "--metrics"}


def expand(dirs, rule, name, sample, ref_name):
    var, pat = RULE_LOGS[rule] if name == "log" else RULE_OUTPUTS[rule][name]
    return dirs[var] + pat.format(sample=sample, ref_name=ref_name)


def benchmark_path(dirs, rule, sample, ref_name):
    var, pat = RULE_BENCHMARKS[rule]
    return dirs[var] + pat.format(sample=sample, ref_name=ref_name)


def sample_command(driver, dirs, sample, ref_name, ref_fa, r1, r2, threads=4, extra=(), benchmark=False):
    """-> (argv, [every path the four reference rules declare or leave behind]) for one {sample}.{ref_name};
    benchmark=True adds `--benchmark` at rule bcftools' benchmark path (not part of the returned list: Snakemake does not
    fail a job over it)"""
    argv = [driver, "sample", "--ref", ref_fa, "--r1", r1, "--r2", r2, "--sample", sample, "-t", str(threads), "--rmdup", "1"]
    paths = []
    for key, opt in DRIVER_OPTION.items():
        p = expand(dirs, key[0], key[1], sample, ref_name)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        paths.append(p)
        if opt:
            argv += [opt, p]
        if key in SIDE_FILES:
            paths.append(p + SIDE_FILES[key])
    os.makedirs(os.path.dirname(expand(dirs, "bwa", "log", sample, ref_name)), exist_ok=True)
    if benchmark:
        b = benchmark_path(dirs, "bcftools", sample, ref_name)
        os.makedirs(os.path.dirname(b), exist_ok=True)
        argv += ["--benchmark", b]
    return argv + list(extra), paths


def pileup_commands(driver, dirs, sample, ref_name, ref_fa, threads=4, extra=(), benchmark=False):
    """-> {rule: (argv, [every path the rule declares or leaves behind])} for the per-rule replacements of `mpileup` and
    `bcftools`: each runs `qm_driver pileup` on the rule's own input, {sample}.{ref_name}.rmdup.bam (rules/vcfcall.smk:29,104),
    writes only the rule's declared outputs and, with benchmark=True, its own `benchmark:` file (so that Snakemake can rerun
    one of them without the alignment)."""
    bam = expand(dirs, "rmdup", "rmdupbam", sample, ref_name)
    out = {}
    for rule in ("mpileup", "bcftools"):
        argv = [driver, "pileup", "--ref", ref_fa, "--bam", bam, "--sample", sample, "-t", str(threads)]
        paths = []
        for name in RULE_OUTPUTS[rule]:
            p = expand(dirs, rule, name, sample, ref_name)
            os.makedirs(os.path.dirname(p), exist_ok=True)
            paths.append(p)
            opt = DRIVER_OPTION[(rule, name)]
            if opt:
                argv += [opt, p]
            if (rule, name) in SIDE_FILES:
                paths.append(p + SIDE_FILES[(rule, name)])
        if benchmark:
            b = benchmark_path(dirs, rule, sample, ref_name)
            os.makedirs(os.path.dirname(b), exist_ok=True)
            argv += ["--benchmark", b]
        out[rule] = (argv + list(extra), paths)
    return out
