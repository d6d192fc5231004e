"""Wall clock of the decontamination chain against the one-job form: rules rm_phix + rm_human_ecoli + bwa + rmdup + mpileup +
bcftools as three driver jobs (`decontam` PhiX | `decontam` E. coli | `sample` on the cleaned FASTQ) and as one
`sample --decontam PhiX --decontam2 E. coli` job, on a simulated sample of Merlin reads with 1 % PhiX and 2 % E. coli reads.

For every GPU list: one run of each form, one JSON line with each job's wall clock and phase clock, the two totals and whether the
outputs (count TSV, VCF, text pileup, metrics, cleaned FASTQ) are byte-identical.  The card's name and power limit are read in the
same run.  Work files go to a temporary directory.

    python tools/decontam_bench.py [--pairs 2000000] [--gpus 0,0-7] [-t 16] [--out DIR]
"""
import argparse
import filecmp
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from quasimodo_b200 import genomes, workloads  # noqa: E402
from tests import drvutil  # noqa: E402
from tools.bam_pileup_bench import phases, write_fastq_fast  # noqa: E402


def job(argv):
    t0 = time.time()
    p = subprocess.run(argv, capture_output=True, text=True)
    if p.returncode:
        sys.exit(f"{' '.join(argv[:2])} failed:\n{p.stderr}")
    return dict(wall_s=round(time.time() - t0, 3), phases_s=phases(p.stderr))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=2_000_000)
    ap.add_argument("--gpus", default="0,0-7", help="GPU lists separated by ';' or ',' (one list each: 0 or 0-7)")
    ap.add_argument("-t", type=int, default=16)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()
    drv = drvutil.driver_path()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    n = args.pairs
    me = genomes.load("Merlin").total
    W = workloads.Workload("Merlin+1%PhiX+2%Ecoli", [("Merlin", 1), ("Phix", 1), ("Ecoli", 1)], ["Merlin"], n, 7001,
                           extra_weights=[97 * me, 1 * me, 2 * me])
    lines = []
    with tempfile.TemporaryDirectory() as d:
        fa, pfa, efa, r1, r2 = (os.path.join(d, x) for x in ("ref.fa", "phix.fa", "ecoli.fa", "r1.fq", "r2.fq"))
        drvutil.write_fasta(W.ref, fa)
        drvutil.write_fasta(genomes.load("Phix"), pfa)
        drvutil.write_fasta(genomes.load("Ecoli"), efa)
        write_fastq_fast(W, n, r1, r2)
        for gl in args.gpus.replace(";", ",").split(","):
            gp = ["--gpus", gl] if "-" in gl else ["--gpu", gl]
            common = ["-t", str(args.t)]

            def outs(tag):
                o = os.path.join(d, tag)
                os.makedirs(o, exist_ok=True)
                return o, ["--rmdup", "1", "--bam", f"{o}/s.bam", "--rmdup-bam", f"{o}/s.rmdup.bam", "--metrics", f"{o}/s.metrics",
                           "--counts", f"{o}/s.tsv", "--vcf", f"{o}/s.vcf", "--mpileup", f"{o}/s.txt"]
            oc, chain_out = outs("chain")
            c1 = job([drv, "decontam", "--ref", pfa, "--r1", r1, "--r2", r2, "--out-r1", f"{oc}/c1.r1.fq", "--out-r2", f"{oc}/c1.r2.fq"] + common)
            c2 = job([drv, "decontam", "--ref", efa, "--r1", f"{oc}/c1.r1.fq", "--r2", f"{oc}/c1.r2.fq", "--out-r1", f"{oc}/c2.r1.fq",
                      "--out-r2", f"{oc}/c2.r2.fq"] + common)
            c3 = job([drv, "sample", "--ref", fa, "--r1", f"{oc}/c2.r1.fq", "--r2", f"{oc}/c2.r2.fq"] + chain_out + common + gp)
            of, fused_out = outs("fused")
            f = job([drv, "sample", "--ref", fa, "--r1", r1, "--r2", r2, "--decontam", pfa, "--decontam2", efa, "--clean-r1", f"{of}/cl.r1.fq",
                     "--clean-r2", f"{of}/cl.r2.fq"] + fused_out + common + gp)
            same = all(filecmp.cmp(os.path.join(oc, a), os.path.join(of, b), shallow=False) for a, b in
                       (("s.tsv", "s.tsv"), ("s.vcf", "s.vcf"), ("s.txt", "s.txt"), ("s.metrics", "s.metrics"),
                        ("c2.r1.fq", "cl.r1.fq"), ("c2.r2.fq", "cl.r2.fq")))
            chain_s = c1["wall_s"] + c2["wall_s"] + c3["wall_s"]
            rec = dict(pairs=n, gpus=gl, card=card, chain=dict(decontam_phix=c1, decontam_ecoli=c2, sample=c3, total_s=round(chain_s, 3)),
                       fused=f, fused_total_s=f["wall_s"], outputs_identical=same)
            lines.append(json.dumps(rec))
            print(lines[-1], flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "decontam_bench.jsonl"), "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
