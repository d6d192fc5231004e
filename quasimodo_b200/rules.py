"""The file contract of the reference rules this implementation replaces (SURVEY.md 8b): the declared `output:` / `log:`
paths of rules `bwa` (rules/bwa.smk:1-19), `rmdup` (rules/rmdup.smk:1-18), `mpileup` (rules/vcfcall.smk:26-40) and `bcftools`
(rules/vcfcall.smk:101-120), and the ONE `qm_driver sample` invocation that produces all of them.  Snakemake deletes a job
whose declared output is missing, so tests/test_rules_cpu.py checks these tables against the reference's rule files and
tests/test_driver_gpu.py checks that the command really writes every path.  pileup_commands gives rules `mpileup` and
`bcftools` one `qm_driver pileup` job each, on the .rmdup.bam a separate alignment step left; rmdup_command gives rule `rmdup`
one `qm_driver rmdup` job on the sorted BAM of any aligner; index_command gives rule `build_idx` (rules/index.smk:12-14) one
`qm_driver index` job in place of `bwa index` + `samtools faidx`; decontam_sample_command puts the decontamination rules
`rm_phix` and `rm_human_ecoli` (rules/decontamination.smk) in front of the four in the same job."""
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


def sample_command(driver, dirs, sample, ref_name, ref_fa, r1, r2, threads=4, extra=(), benchmark=False, chunk_bases=None):
    """-> (argv, [every path the four reference rules declare or leave behind]) for one {sample}.{ref_name};
    benchmark=True adds `--benchmark` at rule bcftools' benchmark path (not part of the returned list: Snakemake does not
    fail a job over it); chunk_bases=K adds bwa mem's `-K K` (one insert-size model per input chunk of K bases, as bwa pairs;
    `bwa mem -t T` itself is `-K 10000000*T`)"""
    argv = [driver, "sample", "--ref", ref_fa, "--r1", r1, "--r2", r2, "--sample", sample, "-t", str(threads), "--rmdup", "1"]
    if chunk_bases is not None:
        argv += ["-K", str(int(chunk_bases))]
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


def rmdup_command(driver, dirs, sample, ref_name, threads=4, extra=()):
    """-> (argv, [the .rmdup.bam, its .bai, the metrics log]) of the per-rule replacement of `rmdup`: `qm_driver rmdup` on the
    rule's input, the {sample}.{ref_name}.bam of rule `bwa` (rules/rmdup.smk:8), with picard's library name --sample"""
    argv = [driver, "rmdup", "--bam", expand(dirs, "bwa", "sortedbam", sample, ref_name), "--sample", sample, "-t", str(threads)]
    paths = []
    for name in ("rmdupbam", "log"):
        p = expand(dirs, "rmdup", name, sample, ref_name)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        argv += [DRIVER_OPTION[("rmdup", name)], p]
        paths.append(p)
        if ("rmdup", name) in SIDE_FILES:
            paths.append(p + SIDE_FILES[("rmdup", name)])
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


# the cleaned FASTQ of the decontamination rules (rules/decontamination.smk:8-9,36-37): rm_phix writes the reads without PhiX,
# rm_human_ecoli those without human and E. coli either; rule `bwa` reads the last
CLEAN_FASTQ = {"rm_phix": ("seq_dir", "/cl_fq/{sample}.qc.nophix.r{mate}.fq"), "rm_human_ecoli": ("seq_dir", "/cl_fq/{sample}.qc.cl.r{mate}.fq")}


def decontam_sample_command(driver, dirs, sample, ref_name, ref_fa, r1, r2, phix_fa, human_ecoli_fa=(), threads=4, extra=(), benchmark=False,
                            chunk_bases=None):
    """-> (argv, [every path the job writes]) of rules rm_phix [+ rm_human_ecoli] + bwa + rmdup + mpileup + bcftools as ONE
    `qm_driver sample --decontam` job on the raw reads r1 / r2: sample_command's outputs plus the last pass's cleaned FASTQ (rule
    rm_human_ecoli's when human_ecoli_fa names its genomes, else rule rm_phix's), the FASTQ the assemblers read.  With both passes
    rule rm_phix's intermediate FASTQ is not written."""
    argv, paths = sample_command(driver, dirs, sample, ref_name, ref_fa, r1, r2, threads, benchmark=benchmark, chunk_bases=chunk_bases)
    argv += ["--decontam", phix_fa]
    last = "rm_phix"
    if human_ecoli_fa:
        argv += ["--decontam2", ",".join(human_ecoli_fa)]
        last = "rm_human_ecoli"
    var, pat = CLEAN_FASTQ[last]
    for mate in (1, 2):
        p = dirs[var] + pat.format(sample=sample, mate=mate)
        os.makedirs(os.path.dirname(p), exist_ok=True)
        argv += [f"--clean-r{mate}", p]
        paths.append(p)
    return argv + list(extra), paths


# the files rule `build_idx` (rules/index.smk:12-14) leaves next to a genome X.fa: `bwa index X.fa` writes X.fa.{amb,ann,bwt,pac,sa}
# (its prefix defaults to the FASTA path), `samtools faidx X.fa` writes X.fa.fai
BWA_INDEX_SUFFIXES = (".amb", ".ann", ".bwt", ".pac", ".sa")
FAIDX_SUFFIX = ".fai"


def index_command(driver, ref_fa, threads=4, extra=(), benchmark=None):
    """-> (argv, [the five bwa index files and the .fai]) of the per-rule replacement of `build_idx`: `qm_driver index` on one
    genome, writing what `bwa index` and `samtools faidx` write, under the names they use (the sample commands' --bwa-index
    takes ref_fa as its prefix); benchmark=PATH adds `--benchmark PATH`"""
    argv = [driver, "index", "--ref", ref_fa, "-t", str(threads)]
    if benchmark:
        os.makedirs(os.path.dirname(os.path.abspath(benchmark)), exist_ok=True)
        argv += ["--benchmark", benchmark]
    return argv + list(extra), [ref_fa + s for s in BWA_INDEX_SUFFIXES] + [ref_fa + FAIDX_SUFFIX]
