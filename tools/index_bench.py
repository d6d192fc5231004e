#!/usr/bin/env python3
"""Time qm_index_build_fm -- bwa's FM-index (suffix array of both strands, BWT, occurrence checkpoints, suffix-array samples)
built from the genome -- on the five bundled genomes and on a simulated 50 M-base genome.

One line of JSON per genome: l_pac, suffixes, the build's wall time (host clock around the call, which ends in a device
synchronise; min and median of --reps builds after one warm-up build) and the SHA-256 of the two files it exports, so that
two libraries timed on the same inputs can be checked to build the same bytes.  The first line names the card and its
power limit.  --lib times another build of the library (same C ABI), e.g. one of an earlier commit.

    python tools/index_bench.py [--reps 3] [--only Phix,Sim50M] [--lib path/to/libquasimodo_b200.so] [--out FILE]"""
import argparse
import ctypes as C
import hashlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))

from quasimodo_b200 import genomes  # noqa: E402

STEMS = ["Phix", "AD169", "TB40E", "Merlin", "Ecoli"]


def simulated(l_pac=50_000_000, seed=50):
    """uniform random bases with a few kinds of repeats, so that the doubling runs many rounds: 40 copies of a 6 kb element
    (some reverse-complemented), a 20 kb tandem array of a 171-base unit and a 3 kb homopolymer"""
    rng = np.random.default_rng(seed)
    g = rng.integers(0, 4, l_pac).astype(np.uint8)
    elem = rng.integers(0, 4, 6000).astype(np.uint8)
    for k, p in enumerate(rng.integers(0, l_pac - 6000, 40)):
        g[p:p + 6000] = elem if k % 3 else 3 - elem[::-1]
    unit = rng.integers(0, 4, 171).astype(np.uint8)
    p = l_pac // 3
    g[p:p + 171 * 117] = np.tile(unit, 117)
    g[2 * l_pac // 3:2 * l_pac // 3 + 3000] = 0
    return genomes.Genome(["sim50M"], [l_pac], g)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        return q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default="")
    ap.add_argument("--lib", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "quasimodo_b200", "libquasimodo_b200.so"))
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    L = C.CDLL(os.path.abspath(a.lib))
    P = C.c_void_p
    L.qm_ctx_create.argtypes = [C.c_int, C.POINTER(P)]
    L.qm_index_build.argtypes = [P, P, C.c_int, P, C.c_int, C.POINTER(P)]
    L.qm_index_build_fm.argtypes = [P, P, P]
    L.qm_index_fm_export.argtypes = [P, P, C.POINTER(C.c_int64), P, C.POINTER(C.c_int64)]
    L.qm_index_destroy.argtypes = [P, P]
    L.qm_ctx_destroy.argtypes = [P]
    L.qm_last_error.argtypes = [P]
    L.qm_last_error.restype = C.c_char_p
    ctx = P()
    rc = L.qm_ctx_create(0, C.byref(ctx))
    if rc != 0:
        raise SystemExit(f"qm_ctx_create failed ({rc}): no usable GPU")

    def check(rc, what):
        if rc != 0:
            raise SystemExit(f"{what} failed ({rc}): {L.qm_last_error(ctx).decode()}")

    out = open(a.out, "a") if a.out else None

    def emit(d):
        line = json.dumps(d)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    emit({"card": card(), "lib": os.path.abspath(a.lib)})
    names = [s for s in (a.only.split(",") if a.only else STEMS + ["Sim50M"])]
    for name in names:
        G = simulated() if name == "Sim50M" else genomes.load(name)
        codes = np.ascontiguousarray(G.codes, np.uint8)
        lens = np.ascontiguousarray(G.lens, np.int64)
        idx = P()
        check(L.qm_index_build(ctx, codes.ctypes.data, len(lens), lens.ctypes.data, 31, C.byref(idx)), "qm_index_build")
        times = []
        for r in range(a.reps + 1):                         # build 0 is the warm-up (module load, first allocations)
            t0 = time.perf_counter()
            check(L.qm_index_build_fm(ctx, idx, codes.ctypes.data), "qm_index_build_fm")
            dt = time.perf_counter() - t0
            if r:
                times.append(dt)
        nb, ns = C.c_int64(), C.c_int64()
        check(L.qm_index_fm_export(idx, None, C.byref(nb), None, C.byref(ns)), "qm_index_fm_export")
        b, s = np.zeros(nb.value, np.uint8), np.zeros(ns.value, np.uint8)
        check(L.qm_index_fm_export(idx, b.ctypes.data, C.byref(nb), s.ctypes.data, C.byref(ns)), "qm_index_fm_export")
        L.qm_index_destroy(ctx, idx)
        emit({"genome": name, "l_pac": int(len(codes)), "suffixes": 2 * int(len(codes)), "reps": a.reps,
              "build_s_min": round(min(times), 4), "build_s_median": round(statistics.median(times), 4),
              "bwt_sha256": hashlib.sha256(b.tobytes()).hexdigest(), "sa_sha256": hashlib.sha256(s.tobytes()).hexdigest()})
    L.qm_ctx_destroy(ctx)


if __name__ == "__main__":
    main()
