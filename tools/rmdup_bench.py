"""Phase clock of `qm_driver rmdup` (coordinate-sorted BAM in -> BAM without duplicates + BAI + metrics) on the BAM that
`qm_driver sample` writes for a simulated sample.

For every size: simulate BASELINE config 1 pairs, run `sample --bam` (FASTQ -> sorted BAM), then `rmdup` on that BAM, and print
one JSON line per size with `rmdup`'s phase clock (BGZF inflate, validation walk, context, H2D + decision, BAM + BAI), its
device stages, the input's size and the duplicate counts.  The card's name and power limit are read in the same run.  Work files
go to a temporary directory.

    python tools/rmdup_bench.py [--pairs 2000000,20000000] [-t 16] [--out DIR]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from quasimodo_b200 import workloads  # noqa: E402
from tests import drvutil  # noqa: E402
from tools.bam_pileup_bench import phases, write_fastq_fast  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", default="2000000,20000000")
    ap.add_argument("-t", type=int, default=16)
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()
    drv = drvutil.driver_path()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    lines = []
    for n in [int(x) for x in args.pairs.split(",")]:
        W = workloads.config1(n)
        with tempfile.TemporaryDirectory() as d:
            fa, r1, r2, bam, out = (os.path.join(d, x) for x in ("ref.fa", "r1.fq", "r2.fq", "s.bam", "s.rmdup.bam"))
            drvutil.write_fasta(W.ref, fa)
            write_fastq_fast(W, n, r1, r2)
            s = subprocess.run([drv, "sample", "--ref", fa, "--r1", r1, "--r2", r2, "--bam", bam, "-t", str(args.t)], capture_output=True, text=True)
            if s.returncode:
                sys.exit(f"sample failed:\n{s.stderr}")
            r = subprocess.run([drv, "rmdup", "--bam", bam, "--rmdup-bam", out, "--metrics", os.path.join(d, "m.txt"), "-t", str(args.t),
                                "--stage-ms", "1"], capture_output=True, text=True)
            if r.returncode:
                sys.exit(f"rmdup failed:\n{r.stderr}")
            st = re.search(r"stages \(ms of device time\): (.*)", r.stderr)
            dup = re.search(r"rmdup: (.*)", r.stderr)
            rec = dict(cmd="rmdup", pairs=n, card=card, bam_bytes=os.path.getsize(bam), rmdup_bam_bytes=os.path.getsize(out),
                       phases_s=phases(r.stderr), device_stages_ms=st.group(1) if st else None, duplicates=dup.group(1) if dup else None)
            lines.append(json.dumps(rec))
            print(lines[-1], flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "rmdup_bench.jsonl"), "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
