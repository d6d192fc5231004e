"""Pairs per second of `qm_driver sample` on a simulated config-2 sample (TM-6-1: Merlin reads, 6 % of them TB40E) with bwa mem's
per-chunk insert-size model (`-K 80000000`, about 266 k pairs of 2 x 150 per chunk: bwa mem -t 8) against the default path (one
model per sample), in the same run and alternating, with `--rmdup 1` and every output of the `sample` rule.

One JSON line per repetition: each form's wall clock, its "FASTQ -> records + counts" phase, pairs/s over that phase, and the card's
name and power limit (read in the same run).  Work files go to a temporary directory.

    python tools/chunk_bench.py [--pairs 4000000] [-K 80000000] [--reps 2] [-t 16] [--gpu 0] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from quasimodo_b200 import workloads  # noqa: E402
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
    ap.add_argument("--pairs", type=int, default=4_000_000)
    ap.add_argument("-K", type=int, default=80_000_000)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("-t", type=int, default=16)
    ap.add_argument("--gpu", default="0")
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()
    drv = drvutil.driver_path()
    card = subprocess.run(["nvidia-smi", "-i", args.gpu, "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    n = args.pairs
    W = workloads.config2(6, n)
    lines = []
    with tempfile.TemporaryDirectory() as d:
        fa, r1, r2 = (os.path.join(d, x) for x in ("ref.fa", "r1.fq", "r2.fq"))
        drvutil.write_fasta(W.ref, fa)
        write_fastq_fast(W, n, r1, r2)

        def run(tag, extra):
            o = os.path.join(d, tag)
            os.makedirs(o, exist_ok=True)
            r = job([drv, "sample", "--ref", fa, "--r1", r1, "--r2", r2, "--gpu", args.gpu, "-t", str(args.t), "--rmdup", "1",
                     "--bam", f"{o}/s.bam", "--rmdup-bam", f"{o}/s.rmdup.bam", "--metrics", f"{o}/s.metrics", "--counts", f"{o}/s.tsv",
                     "--vcf", f"{o}/s.vcf", "--mpileup", f"{o}/s.txt"] + extra)
            loop = r["phases_s"].get("FASTQ -> records + counts")
            r["pairs_per_s"] = round(n / loop) if loop else None
            return r
        for rep in range(args.reps):
            default = run("default", [])
            chunked = run("chunked", ["-K", str(args.K)])
            rec = dict(pairs=n, K=args.K, rep=rep, card=card, default=default, chunked=chunked)
            lines.append(json.dumps(rec))
            print(lines[-1], flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "chunk_bench.jsonl"), "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
