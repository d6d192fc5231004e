"""Phase clock of `qm_driver pileup` (BAM in -> count TSV, VCF, text pileup) next to the counting phases of `qm_driver sample` on
the same simulated sample.

For every size: simulate BASELINE config 1 pairs, run `sample` (FASTQ -> BAM + the same outputs), then `pileup` on that BAM,
and print one JSON line per run with the driver's phase clock: for `pileup` BGZF inflate, the validation walk, device decode +
pairing, counting and the outputs; for `sample` its phases (FASTQ -> records + counts is where its counting happens).  The
card's name and power limit are read in the same run.  Work files go to a temporary directory.

    python tools/bam_pileup_bench.py [--pairs 2000000,20000000] [-t 16] [--text 0] [--out DIR]

--text 0 leaves the text pileup out of both runs: at 20 M pairs of config 1 (about 25,000x) it is some 12 GB.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from quasimodo_b200 import workloads  # noqa: E402
from tests import drvutil  # noqa: E402


def write_fastq_fast(W, n_pairs, p1, p2, chunk=500_000):
    """fixed-width names (r<11 digits>/1, /2): whole chunks of records formatted with numpy"""
    L = W.params.read_len
    lut = np.frombuffer(b"ACGTN", np.uint8)
    with open(p1, "wb") as f1, open(p2, "wb") as f2:
        for p0 in range(0, n_pairs, chunk):
            n = min(chunk, n_pairs - p0)
            codes, quals, _, _ = W.simulate_host(p0, n)
            for m, fh in ((0, f1), (1, f2)):
                names = np.array([f"@r{p0 + i:011d}/{m + 1}\n".encode() for i in range(n)])
                hdr = np.frombuffer(names.tobytes(), np.uint8).reshape(n, -1)
                rec = np.concatenate([hdr, lut[codes[m::2, :L]], np.tile(np.frombuffer(b"\n+\n", np.uint8), (n, 1)),
                                      quals[m::2, :L] + 33, np.full((n, 1), 10, np.uint8)], 1)
                fh.write(rec.tobytes())


def phases(stderr):
    m = re.search(r"phases \(s\): (.*); total ([0-9.]+)", stderr)
    out = {k.strip(): float(v) for k, v in (x.rsplit(" ", 1) for x in m.group(1).split(", "))}
    out["total"] = float(m.group(2))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", default="2000000,20000000")
    ap.add_argument("-t", type=int, default=16)
    ap.add_argument("--text", type=int, default=1, help="0: no text pileup (--mpileup) in either run")
    ap.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap.parse_args()
    drv = drvutil.driver_path()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    lines = []
    for n in [int(x) for x in args.pairs.split(",")]:
        W = workloads.config1(n)
        with tempfile.TemporaryDirectory() as d:
            fa, r1, r2, bam = (os.path.join(d, x) for x in ("ref.fa", "r1.fq", "r2.fq", "s.bam"))
            drvutil.write_fasta(W.ref, fa)
            t0 = time.time()
            write_fastq_fast(W, n, r1, r2)
            sim_s = time.time() - t0
            exts = (".tsv", ".vcf", ".mpileup") if args.text else (".tsv", ".vcf")
            outs = lambda p: [x for o, e in zip(("--counts", "--vcf", "--mpileup"), exts) for x in (o, p + e)]        # noqa: E731
            s = subprocess.run([drv, "sample", "--ref", fa, "--r1", r1, "--r2", r2, "--bam", bam, "-t", str(args.t)] + outs(os.path.join(d, "s")),
                               capture_output=True, text=True)
            if s.returncode:
                sys.exit(f"sample failed:\n{s.stderr}")
            p = subprocess.run([drv, "pileup", "--ref", fa, "--bam", bam, "-t", str(args.t), "--stage-ms", "1"] + outs(os.path.join(d, "p")),
                               capture_output=True, text=True)
            if p.returncode:
                sys.exit(f"pileup failed:\n{p.stderr}")
            same = all(open(os.path.join(d, "s" + e), "rb").read() == open(os.path.join(d, "p" + e), "rb").read() for e in exts)
            for cmd, r in (("sample", s), ("pileup", p)):
                rec = dict(cmd=cmd, pairs=n, card=card, bam_bytes=os.path.getsize(bam), phases_s=phases(r.stderr), outputs_equal=same, text=bool(args.text),
                           fastq_simulation_s=round(sim_s, 2))
                if cmd == "pileup":
                    st = re.search(r"stages \(ms of device time\): (.*)", r.stderr)
                    rec["device_stages_ms"] = st.group(1) if st else None
                lines.append(json.dumps(rec))
                print(lines[-1], flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bam_pileup_bench.jsonl"), "w") as fh:
            fh.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
