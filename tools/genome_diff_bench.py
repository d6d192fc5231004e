"""Phase times of the genome diff (qm_genome_diff_host, rule `nucmer`'s replacement; DESIGN.md 5c) on the three bundled HCMV
pairs (Merlin/TB40E and AD169/TB40E, the pairs of rules/genome_diff.smk, and Merlin/AD169, config 3's truth set) and on E. coli
against a copy with 3,000 SNPs and 600 indels planted (tests/gdiffgen.py, 4.6 Mb).

One warm-up call per pair, then --reps timed calls.  One JSON line per pair: the card's name and power limit (read in the same
run), the index build, and each phase's milliseconds per call (anchors: upload + anchor kernel + read-back; clusters: host;
gaps: the gap DP kernel with its copies; ends: the extension rounds and the gap kernel over the extended stretches; rows: host),
plus the wall clock of each call, rows and alignments.

    python tools/genome_diff_bench.py [--reps 3] [--gpu 0] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from quasimodo_b200 import Context, genomes  # noqa: E402
from tests import gdiffgen  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--gpu", type=int, default=0)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "-i", str(args.gpu), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    g = {s: genomes.load(s) for s in ("Merlin", "TB40E", "AD169", "Ecoli")}
    ecoli_mut, _ = gdiffgen.mutated_copy(g["Ecoli"])
    pairs = [("Merlin", "TB40E", g["TB40E"]), ("AD169", "TB40E", g["TB40E"]), ("Merlin", "AD169", g["AD169"]),
             ("Ecoli", "Ecoli_mut", ecoli_mut)]
    ctx = Context(args.gpu)
    lines = []
    for ref, qname, qry in pairs:
        t0 = time.perf_counter()
        idx = ctx.index(g[ref], 20)
        index_ms = (time.perf_counter() - t0) * 1e3
        rows, alns = ctx.genome_diff(idx, qry)
        tot = {}
        walls = []
        for _ in range(args.reps):
            ph = {}
            t0 = time.perf_counter()
            ctx.genome_diff(idx, qry, phases=ph)
            walls.append((time.perf_counter() - t0) * 1e3)
            for k, v in ph.items():
                tot[k] = tot.get(k, 0.0) + v
        idx.close()
        rec = dict(ref=ref, qry=qname, ref_bases=g[ref].total, qry_bases=int(sum(qry.lens)), card=card, reps=args.reps,
                   index_ms=round(index_ms, 1), phase_ms={k: round(v / args.reps, 2) for k, v in tot.items()},
                   call_ms=[round(w, 1) for w in walls], rows=len(rows), alignments=len(alns))
        lines.append(json.dumps(rec))
        print(lines[-1], flush=True)
    ctx.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "genome_diff_bench.jsonl"), "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
