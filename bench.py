#!/usr/bin/env python
"""bench.py -- read pairs/s aligned + piled up (+ called + classified) on B200, BASELINE.json's metric.

A STEP is one pass of the whole read-level hot path over one sample's batch of synthetic read pairs:
seeding/chaining -> ksw_extend2 rounds -> mate rescue -> pairing + CIGAR -> pileup counts -> (N>1: all-reduce of the
int32 count tensor) -> SNP calls -> TP/FP/FN match against the strain-difference truth set.

Workloads (--config, BASELINE.json `configs`; the default is configs[1], the one the metric is quoted on):
  1  TM-1-1, 100,000 2x150 bp pairs vs Merlin (the reference's own CPU-runnable case); steps rotate over 16 windows
  2  10-sample TA-* abundance-ratio series, 2,000,000 2x150 bp pairs each; step i runs sample i % 10        [default]
  3  AD169:Merlin 1:10 + 5 % PhiX + 5 % E. coli, 1,000,000 pairs vs the concatenated Merlin|PhiX|E. coli index
  4  TM-1-50, 50,000,000 pairs (about 61,000x), STRONG scaling: the sample is split over the N GPUs
  5  Merlin:TB40E:AD169 10:3:1, 2,000,000 2x250 bp pairs with simulated indels, band w = 200
With N GPUs each rank takes a contiguous range of the sample's pairs (configs 1, 2, 3, 5: N x the pairs, weak scaling;
config 4: the same 50 M pairs, strong scaling); the insert-size model comes from the sample's first 65,536 pairs on
every rank, the counts are merged with one all-reduce.

  value : whole-job pairs/s with the reads already resident in HBM (timed with CUDA events, max over ranks)
  e2e   : the same through the host-buffer C-ABI call (qm_sample_add_pairs_host): pinned host reads -> H2D ->
          pipeline -> calls D2H, all inside the timed region
  roofline / stages : per-stage CUDA-event times measured live by the library's stage timers (same run)
  cpu_baseline : the oracle port (oracle/, CPU restatement of bwa-mem extension + bcftools counting, OpenMP on
          all host cores, built -O3 -march=native on the host it runs on) on a bounded sample of the same workload
          -- a reported baseline, not the target
  --impl reference : that CPU path as its own arm (the upstream binaries are not in the image: kind "port")
  --dump-outputs DIR : after the timed steps, what the last timed step computed as DIR/<name>.npy (float64), so that two
          builds can be compared output for output on the same seeded inputs (see dump_outputs)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

_json_out = sys.stdout                     # replaced in __main__ by the saved original stdout
METRIC = "read_pairs_per_s_aligned_piledup"
UNIT = "pairs/s"
CHUNK = 2_000_000                          # pairs handed to the library per call (bounds its per-chunk scratch)
CPU_NOTE = ("bwa/samtools/bcftools are not in the image and not vendored: the CPU arm is the repo's C restatement "
            "(oracle/, scalar C, OpenMP over reads), not the upstream binaries")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5], help="BASELINE.json configs[N-1]")
    ap.add_argument("--pairs", type=int, default=0, help="pairs per step per GPU (config 4: in the whole sample); 0 = the config's own size")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return a


class Plan:
    """what one step of a config is: which workload window, how many pairs per rank, read length, band, truth set"""

    def __init__(self, args, world):
        from quasimodo_b200 import workloads
        c = args.config
        self.cfg, self.world = c, world
        self.strong = c == 4
        own = {1: 100_000, 2: 2_000_000, 3: 1_000_000, 4: 50_000_000, 5: 2_000_000}[c]
        size = args.pairs or own
        self.total = size if self.strong else size * world          # pairs of one sample (all ranks together)
        self.L = 250 if c == 5 else 150
        self.w = 200 if c == 5 else 100
        self.truth = {1: "TM", 2: "TA", 4: "TM"}.get(c)
        self.n_inputs = {1: 16, 2: 10}.get(c, 1)                    # distinct step inputs the steps rotate over
        mk = {1: lambda i: workloads.config1(self.total * 16), 2: lambda i: workloads.config2(i, self.total),
              3: lambda i: workloads.config3(self.total), 4: lambda i: workloads.config4(self.total),
              5: lambda i: workloads.config5(self.total)}[c]
        self.make = mk
        self.names = {1: "cfg1: TM-1-1 (TB40E:Merlin 1:1) vs Merlin, 2x150 bp; steps rotate over 16 windows of the pair stream",
                      2: "cfg2: 10-sample TA-* abundance-ratio series (TB40E:AD169 1:0 ... 0:1), synthetic 2x150 bp pairs, "
                         "step i = sample i%10, reference AD169 (TB40E for TA-1-0)",
                      3: "cfg3: AD169:Merlin 1:10 + 5% PhiX + 5% E. coli pairs vs the concatenated Merlin|PhiX|E. coli index (4.89 Mb), 2x150 bp",
                      4: "cfg4: TM-1-50 deep sample (TB40E:Merlin 1:50) vs Merlin, 2x150 bp, the sample split over the GPUs",
                      5: "cfg5: Merlin:TB40E:AD169 10:3:1 vs Merlin, 2x250 bp with simulated indels, band w=200"}

    def window(self, i):
        """first pair (in the simulator's index space) of step input i"""
        return (i % 16) * self.total if self.cfg == 1 else 0

    def config_dict(self, n_gpus, per_rank):
        return {"workload": self.names[self.cfg], "baseline_config": self.cfg,
                "pairs_per_step_per_gpu": per_rank, "read_len": self.L, "band_w": self.w, "global_pairs_per_step": self.total,
                "parallelism": (f"reads sharded over {n_gpus} GPU(s), int32 count tensor all-reduced" if n_gpus > 1 else "1 GPU"),
                "l2_policy": f"inputs larger than L2: the steps rotate over {self.n_inputs} input(s) of "
                             f"{per_rank * 4 * self.L / 1e6:.0f} MB (bases + qualities) each vs 126 MB of L2"}


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
def cpu_setup():
    """the CPU arms use every host core (torchrun exports OMP_NUM_THREADS=1) and a build tuned for this host"""
    from oracle import qmo_py
    qmo_py.build()
    qmo_py.use_native_build()
    qmo_py.set_threads(os.cpu_count() or 1)
    return qmo_py


def cpu_arm(plan, steps, warmup, sample_pairs):
    """the oracle port on host cores; each step = the first `sample_pairs` pairs of step input i.  -> (pairs/s, ms/step)"""
    import numpy as np
    from oracle import qmo_py
    refs, times = {}, []
    opt = qmo_py.default_opt()
    opt.w = plan.w
    for i in range(warmup + steps):
        W = plan.make(i % plan.n_inputs)
        key = "|".join(W.ref_stems)
        if key not in refs:
            refs[key] = qmo_py.Ref(W.ref.codes, W.ref.lens, k=31)
        codes, quals = qmo_py.simulate_pairs(W, plan.window(i % plan.n_inputs), sample_pairs)
        lens = np.full(2 * sample_pairs, plan.L, np.int32)
        t0 = time.perf_counter()
        qmo_py.run_sample(refs[key], codes, quals, lens, opt=opt)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    tot = sum(times)
    return sample_pairs * len(times) / tot, tot / len(times) * 1e3


def upstream_tools():
    """SURVEY.md 8d: the reference's own CPU path is `bwa mem | samtools view | samtools sort` + `bcftools mpileup | call`; the image
    has none of them (checked at run time: if they ever appear, the CPU arms run them instead of the port).  -> {name: path or None}"""
    import shutil
    return {t: shutil.which(t) for t in ("bwa", "samtools", "bcftools")}


def upstream_arm(plan, steps, warmup, sample_pairs, threads):
    """the reference's own command lines (rules/bwa.smk:15-18, rules/vcfcall.smk:115-117) on FASTQ files of the same simulated
    pairs; `bwa index` and the FASTQ / FASTA writing are outside the timed region (the index is a one-off rule, rules/index.smk:13).
    Only reachable when bwa, samtools and bcftools are on PATH.  -> (pairs/s, ms/step)"""
    import subprocess
    import tempfile
    import numpy as np
    from oracle import qmo_py
    lut = np.frombuffer(b"ACGTN", np.uint8)
    times = []
    with tempfile.TemporaryDirectory(prefix="qm_upstream_") as d:
        indexed = {}
        for i in range(warmup + steps):
            W = plan.make(i % plan.n_inputs)
            key = "|".join(W.ref_stems)
            if key not in indexed:
                fa = os.path.join(d, f"ref{len(indexed)}.fa")
                with open(fa, "wb") as fh:
                    off = 0
                    for name, ln in zip(W.ref.names, W.ref.lens):
                        fh.write(b">" + str(name).encode() + b"\n")
                        seq = lut[W.ref.codes[off:off + ln]].tobytes()
                        fh.write(b"\n".join(seq[j:j + 70] for j in range(0, ln, 70)) + b"\n")
                        off += ln
                subprocess.run(["bwa", "index", fa], check=True, capture_output=True)
                indexed[key] = fa
            fa = indexed[key]
            codes, quals = qmo_py.simulate_pairs(W, plan.window(i % plan.n_inputs), sample_pairs)
            fq = [os.path.join(d, f"r{m + 1}.fq") for m in (0, 1)]
            for m in (0, 1):
                seq, q = lut[np.minimum(codes[m::2, :plan.L], 4)], (quals[m::2, :plan.L] + 33).astype(np.uint8)
                with open(fq[m], "wb") as fh:
                    for r in range(sample_pairs):
                        fh.write(b"@sim.%d/%d\n" % (r, m + 1) + seq[r].tobytes() + b"\n+\n" + q[r].tobytes() + b"\n")
            bam, vcf = os.path.join(d, "s.bam"), os.path.join(d, "s.vcf")
            cmd = (f"set -e -o pipefail; bwa mem -k 31 -w {plan.w} -t {threads} {fa} {fq[0]} {fq[1]} 2>/dev/null | samtools view -Shb - | "
                   f"samtools sort -@ {threads} - -o {bam}; samtools index {bam}; "
                   f"bcftools mpileup --threads {threads} -Ou -f {fa} {bam} 2>/dev/null | bcftools call --threads {threads} -p 0.01 --ploidy 1 -mv -Ob | "
                   f"bcftools view -i 'INFO/DP>=10' - > {vcf}")
            t0 = time.perf_counter()
            subprocess.run(["bash", "-c", cmd], check=True, capture_output=True)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    tot = sum(times)
    return sample_pairs * len(times) / tot, tot / len(times) * 1e3


def calibrated_cpu_sample(plan, seconds, cap):
    """pick a sample size that costs about `seconds` of CPU wall time"""
    rate, _ = cpu_arm(plan, 1, 0, 20_000)
    n = int(max(20_000, min(cap, rate * seconds)))
    return n - n % 1000


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    qmo_py = cpu_setup()
    plan = Plan(args, args.gpus)
    per_rank = plan.total // args.gpus
    cores = qmo_py.n_threads()
    per_step = max(20_000, int(calibrated_cpu_sample(plan, args.cpu_seconds, per_rank) / max(1, args.steps + args.warmup) * 4))
    per_step = min(per_step - per_step % 1000, plan.total)
    tools, kind, note = upstream_tools(), "port", CPU_NOTE
    value = None
    if all(tools.values()):                           # the reference's own binaries, if the image ever has them (SURVEY.md 8d)
        try:
            value, ms = upstream_arm(plan, args.steps, args.warmup, per_step, cores)
            kind, note = "reference", "upstream bwa + samtools + bcftools found on PATH: the reference's own command lines (rules/bwa.smk:15-18, rules/vcfcall.smk:115-117)"
            sample = f"{per_step} pairs per step (prefix of each step's sample) as FASTQ through bwa mem | samtools view | sort | index + bcftools mpileup | call | view"
        except Exception as e:                         # a broken install must not take the arm down: fall back to the port and say so
            value, note = None, CPU_NOTE + f" (upstream binaries on PATH failed: {type(e).__name__}: {str(e)[:200]})"
    if value is None:
        value, ms = cpu_arm(plan, args.steps, args.warmup, per_step)
        sample = (f"{per_step} pairs per step (prefix of each step's sample), oracle port: seeding+extension+mate rescue+pairing+CIGAR+pileup; "
                  f"build {qmo_py.BUILD_KIND}")
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if plan.strong else "weak",
           "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": plan.config_dict(args.gpus, per_rank),
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0, "note": note, "upstream_tools": tools}
    print(json.dumps(out), file=_json_out, flush=True)


# ---------------------------------------------------------------------------------------------
def load_truth_keys(name):
    import gzip
    import numpy as np
    from quasimodo_b200 import evaluate
    tk = []
    with gzip.open(os.path.join(ROOT, "quasimodo_b200", "data", "truth", f"{name}.maskrepeat.variants.vcf.gz"), "rt") as fh:
        for ln in fh:
            f = ln.rstrip("\n").split("\t")
            if len(f) >= 5 and f[3] in "ACGT" and f[4] in "ACGT" and len(f[3]) == 1 and len(f[4]) == 1 and f[1].isdigit():
                tk.append(int(evaluate.snp_key(f[1], f[3], f[4])))
    return np.array(tk, dtype=np.uint64)


DUMP_COUNT_COLS = 1 << 18                  # count-tensor columns dumped at most: 16 channels x 8 B x 262,144 = 32 MB


def dump_outputs(dirname, s, r, stats, d_calls):
    """what one resident step hands its caller, as float64 .npy files (every value is an int32 or a float32: exact)
      counts.npy      [16, n]  the sample's count tensor (channel planes, include/quasimodo_b200.h) at the columns of
                               counts_pos.npy: all of them, or a fixed seeded sample of 262,144 on a longer reference
      counts_pos.npy  [n]      those columns (positions in the concatenated reference)
      calls.npy       [c, 11]  the SNP calls: rid, pos, ref, alt, dp, ad_ref_f, ad_ref_r, ad_alt_f, ad_alt_r, qual, af
      eval.npy        [4]      calls, TP, FP, FN against the truth set (the finish_sample tuple)
      stats.npy       [2]      pairs added, executed ksw_extend2 cells
    At most 32 MB of counts + 23 MB of calls (2^18 calls)."""
    import numpy as np
    import torch
    from quasimodo_b200 import _lib
    os.makedirs(dirname, exist_ok=True)
    counts = s.counts_tensor()
    n = counts.shape[1]
    if n <= DUMP_COUNT_COLS:
        pos = np.arange(n)
        cols = counts.cpu().numpy()
    else:
        pos = np.sort(np.random.default_rng(0).choice(n, DUMP_COUNT_COLS, replace=False))
        cols = counts[:, torch.from_numpy(pos).to(counts.device)].cpu().numpy()
    calls = d_calls[:r[0] * _lib.CALL_DTYPE.itemsize].cpu().numpy().view(_lib.CALL_DTYPE)
    fields = [f for f in _lib.CALL_DTYPE.names if not f.startswith("pad")]
    out = {"counts": cols, "counts_pos": pos, "calls": np.column_stack([calls[f] for f in fields]).reshape(-1, len(fields)),
           "eval": np.array(r), "stats": np.array(stats)}
    for name, a in out.items():
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def run_ours(args):
    import ctypes as C
    import numpy as np
    import torch
    import torch.distributed as dist
    from quasimodo_b200 import Context, _lib, sharding
    from quasimodo_b200.api import Comm

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    K, Wm = args.steps, args.warmup
    plan = Plan(args, world)
    L = plan.L
    lo, hi = sharding.shard_range(plan.total, rank, world)
    P = hi - lo                                       # this rank's pairs per step
    ctx = Context(local)                              # raises without the CUDA library / a B200: no CPU fallback
    lib = _lib.lib()
    comm = None
    if world > 1:                                     # the library's own NCCL communicator: torch only carries the 128-byte id
        box = [Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        comm = Comm(ctx, world, rank, box[0])
    st = torch.cuda.current_stream().cuda_stream
    opt = _lib.default_opt()
    opt.w = plan.w
    n_used = min(plan.n_inputs, K + Wm)

    # ---- per-input state: workload, index + qm_sample per reference, resident reads ----
    wl = [plan.make(i) for i in range(n_used)]
    idx, smp = {}, {}
    for W in wl:
        key = "|".join(W.ref_stems)
        if key not in idx:
            idx[key] = ctx.index(W.ref, 31)
            smp[key] = ctx.sample(idx[key], opt)
            if comm is not None:
                smp[key].set_comm(comm)
    tkeys = load_truth_keys(plan.truth) if plan.truth else np.zeros(0, np.uint64)
    d_tkeys = torch.from_numpy(tkeys.view(np.int64)).to(dev)
    d_lens = torch.full((2 * min(P, CHUNK),), L, dtype=torch.int32, device=dev)
    npre = min(_lib.PESTAT_PAIRS, plan.total)
    # The insert-size model is the one of the sample's first 65,536 pairs on every rank.  When rank 0's first batch holds them
    # (always at BASELINE sizes) it is rank 0's, broadcast by the library (qm_sample_set_comm); a shard too small for that
    # aligns the designated prefix itself -- every rank alike, rank 0 included.
    r0_lo, r0_hi = sharding.shard_range(plan.total, 0, world)
    need_pre = world > 1 and min(r0_hi - r0_lo, CHUNK) < npre
    d_lens_pre = torch.full((2 * npre,), L, dtype=torch.int32, device=dev)
    d_reads, d_prefix = [], []
    for i, W in enumerate(wl):
        g = torch.from_numpy(W.src_codes).to(dev)
        c = torch.empty((2 * P, L), dtype=torch.uint8, device=dev)
        q = torch.empty((2 * P, L), dtype=torch.uint8, device=dev)
        for o in range(0, P, 8 * CHUNK):
            n = min(8 * CHUNK, P - o)
            ctx.simulate_pairs(W, plan.window(i) + lo + o, n, g, c[2 * o:2 * (o + n)], q[2 * o:2 * (o + n)], st)
        d_reads.append((c, q))
        if need_pre:                                   # the sample's designated insert-size prefix (its first 65,536 pairs)
            pc = torch.empty((2 * npre, L), dtype=torch.uint8, device=dev)
            pq = torch.empty((2 * npre, L), dtype=torch.uint8, device=dev)
            ctx.simulate_pairs(W, plan.window(i), npre, g, pc, pq, st)
            d_prefix.append(pc)
            del pq
        else:
            d_prefix.append(None)
    torch.cuda.synchronize()
    max_calls = 1 << 18
    d_calls = torch.empty(max_calls * 40, dtype=torch.uint8, device=dev)
    copt = _lib.default_call_opt()
    results = {}
    last_step = []                                    # (sample, finish_sample's result, stats) of the latest step

    def finish_sample(i, s, key):
        """all-reduce (N>1), call SNPs, classify against the truth set; returns (n_calls, tp, fp, fn)"""
        if world > 1:
            s.allreduce_counts(st)                     # qm_counts_allreduce: one in-place ncclAllReduce(int32, sum) over NVLink
        if rank != 0:
            return None
        n = C.c_int64()
        rc = lib.qm_call_snps(ctx._h, idx[key]._h, C.byref(copt), C.c_void_p(s.counts_ptr()), C.c_void_p(d_calls.data_ptr()),
                              max_calls, C.byref(n), C.c_void_p(st))
        if rc:
            raise RuntimeError(lib.qm_last_error(ctx._h).decode())
        nc = n.value
        pure = wl[i].name.endswith(("-1-0", "-0-1"))
        if pure or nc == 0 or not plan.truth:
            return nc, 0, nc, 0
        tpfpfn = (C.c_int64 * 3)()
        rc = lib.qm_eval_calls(ctx._h, C.c_void_p(d_calls.data_ptr()), nc, C.c_void_p(d_tkeys.data_ptr()), len(tkeys), None,
                               tpfpfn, C.c_void_p(st))
        if rc:
            raise RuntimeError(lib.qm_last_error(ctx._h).decode())
        return nc, int(tpfpfn[0]), int(tpfpfn[1]), int(tpfpfn[2])

    def step_resident(i):
        j = i % n_used
        W = wl[j]
        key = "|".join(W.ref_stems)
        s = smp[key]
        s.reset(st)
        c, q = d_reads[j]
        if need_pre:
            s.estimate_pestat(d_prefix[j], d_lens_pre, st)
        for o in range(0, P, CHUNK):
            n = min(CHUNK, P - o)
            s.add_pairs(c[2 * o:2 * (o + n)], q[2 * o:2 * (o + n)], d_lens[:2 * n], pair_id0=lo + o, stream=st)
        r = finish_sample(j, s, key)
        if r is not None:
            results[W.name + (f"@{plan.window(j)}" if plan.cfg == 1 else "")] = r
        stats = s.stats(st)                            # (pairs, executed ksw_extend2 cells) of this step (8-byte read-back)
        last_step[:] = [s, r, stats]
        return stats[1]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- warm-up, then EXACTLY K timed steps between barriers ----
    for i in range(Wm):
        step_resident(i)
    barrier()
    ctx.profile_collect()
    ctx.profile_enable(True)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cells_total = 0
    barrier()
    e0.record()
    marks = []
    for i in range(K):
        cells_total += step_resident(Wm + i)
        marks.append(torch.cuda.Event(enable_timing=True))
        marks[-1].record()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    step_ms = [a.elapsed_time(b) for a, b in zip([e0] + marks[:-1], marks)]
    stage_ms, stage_launch = ctx.profile_collect()
    ctx.profile_enable(False)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:               # before the e2e steps reuse the samples
        dump_outputs(args.dump_outputs, *last_step, d_calls)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = plan.total * K / ms * 1e3

    # ---- e2e: host buffers through the C-ABI, copies inside the timed region ----
    e2e = None
    if not args.no_e2e:
        # the public host entry with PACKED bases: 2 bits per base + an N bit per base cross the link (qm_sample_add_pairs_host_packed)
        Lp = (L + 7) // 8 * 8
        h_b2 = torch.empty((2 * P, (L + 3) // 4), dtype=torch.uint8).pin_memory()
        h_nm = torch.empty((2 * P, (L + 7) // 8), dtype=torch.uint8).pin_memory()
        h_quals = torch.empty((2 * P, L), dtype=torch.uint8).pin_memory()
        h_lens = torch.full((2 * P,), L, dtype=torch.int32).pin_memory()
        h_calls = torch.empty(max_calls * 40, dtype=torch.uint8).pin_memory()
        w4 = torch.tensor([1, 4, 16, 64], dtype=torch.uint8, device=dev)
        w8 = torch.tensor([1, 2, 4, 8, 16, 32, 64, 128], dtype=torch.uint8, device=dev)

        def pack_to_host(c):
            """what a FASTQ parser does as it goes (outside the timed region): codes -> packed bases + N mask, in pinned memory"""
            for o in range(0, 2 * P, 1 << 20):
                cp = torch.nn.functional.pad(c[o:o + (1 << 20)], (0, Lp - L), value=4)
                isn = cp > 3
                b = torch.where(isn, torch.zeros_like(cp), cp).view(cp.shape[0], Lp // 4, 4)
                h_b2[o:o + cp.shape[0]].copy_((b * w4).sum(-1, dtype=torch.uint8)[:, :h_b2.shape[1]])
                h_nm[o:o + cp.shape[0]].copy_((isn.view(cp.shape[0], Lp // 8, 8).to(torch.uint8) * w8).sum(-1, dtype=torch.uint8))
        e2e_times, d2h = [], 0

        h_alns = [None]                                 # set for the e2e_records pass: the 128-byte records come back too

        def step_host(i):
            j = i % n_used
            W = wl[j]
            key = "|".join(W.ref_stems)
            s = smp[key]
            s.reset(st)
            if need_pre:
                s.estimate_pestat(d_prefix[j], d_lens_pre, st)
            torch.cuda.synchronize()
            for o in range(0, P, 4 * CHUNK):            # the library chunks and double-buffers its copies itself
                n = min(4 * CHUNK, P - o)
                s.add_pairs_host_packed(h_b2[2 * o:2 * (o + n)], h_nm[2 * o:2 * (o + n)], h_quals[2 * o:2 * (o + n)], h_lens[2 * o:2 * (o + n)],
                                        pair_id0=lo + o, h_alns=None if h_alns[0] is None else h_alns[0][2 * o * 128:2 * (o + n) * 128])
            r = finish_sample(j, s, key)
            nb = 0
            if r is not None:
                nb = r[0] * 40
                h_calls[:nb].copy_(d_calls[:nb], non_blocking=True)
            torch.cuda.synchronize()
            return nb + 8

        last = -1
        for i in range(Wm + K):
            if i % n_used != last:                      # outside the timed region: this step's reads into the pinned buffers
                c, q = d_reads[i % n_used]
                pack_to_host(c)
                h_quals.copy_(q)
                last = i % n_used
            barrier()
            t0 = time.perf_counter()
            nb = step_host(i)
            barrier()
            dt = time.perf_counter() - t0
            if i >= Wm:
                e2e_times.append(dt)
                d2h = max(d2h, nb)
        # where the host-entry step spends its time (2 extra untimed steps with the stage events on)
        ctx.profile_collect()
        ctx.profile_enable(True)
        for i in range(Wm + K - 2, Wm + K):
            step_host(i if i % n_used == last else last)
        e2e_stage_ms, _ = ctx.profile_collect()
        ctx.profile_enable(False)
        # the same step with the alignment records (128 B per read: what the BAM writer needs) returned to pinned host memory inside the
        # timed region; 3 steps on the buffers the last step left in place
        rec_times = []
        try:
            if P > 8_000_000:
                raise RuntimeError("records pass skipped: more than 2 GB of records per step")
            h_alns[0] = torch.empty(2 * P * 128, dtype=torch.uint8).pin_memory()
            for i in range(4):
                barrier()
                t0 = time.perf_counter()
                step_host(last)
                barrier()
                if i:
                    rec_times.append(time.perf_counter() - t0)
        except RuntimeError:
            rec_times = []
        h_alns[0] = None
        te = torch.tensor([sum(e2e_times), sum(rec_times)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        t_rec = float(te[1].item())
        te = te[:1]
        e2e = {"value": plan.total * K / float(te.item()), "unit": UNIT,
               "h2d_bytes_per_step": int(2 * P * (h_b2.shape[1] + h_nm.shape[1] + L) + 4 * 2 * P), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": float(te.item()) / K * 1e3, "step_ms": [round(x * 1e3, 3) for x in e2e_times],
               "stages_ms_per_step": {k: v / 2 for k, v in e2e_stage_ms.items()},
               "api": "qm_sample_add_pairs_host_packed (2-bit bases + N mask + 1 B/base qualities; + qm_call_snps, qm_eval_calls), pinned host buffers",
               "with_records": None if not rec_times else {
                   "value": plan.total * len(rec_times) / t_rec, "unit": UNIT, "ms_per_step": t_rec / len(rec_times) * 1e3,
                   "d2h_bytes_per_step": int(d2h + 2 * P * 128),
                   "what": "the same call with h_alns: every read's 128-byte alignment record (position, flag, MAPQ, CIGAR, mate fields) copied back to "
                           "pinned host memory inside the timed region, as the BAM writer of qm_driver needs them"}}

    if rank != 0:
        for x in smp.values():
            x.close()
        comm.close()
        dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel + every stage ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except OSError:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    dpx_gops, _ = ctx.dpx_peak(1, 4096)                 # measured now: G lane-instr/s of __viaddmax_s16x2_relu
    gcups_peak = dpx_gops * 2.0 / 9.0                   # 2 packed cells per lane-instr, 9 DPX-class instr per cell
    traffic = None
    try:                                                   # per-launch DRAM bytes of the extension kernel from the committed ncu capture
        traffic = json.load(open(os.path.join(ROOT, "profiles", "ext3_traffic.json")))["dram_bytes_per_launch"]
    except (OSError, KeyError, ValueError):
        pass
    ext_ms = stage_ms["extend"]
    dom = max(("seed_chain", "advance", "extend", "pair_cigar", "pileup", "rescue"), key=lambda k: stage_ms[k])
    gcups = cells_total / ext_ms / 1e6 if ext_ms > 0 else 0.0
    Pk = P * K
    roofline = {"kernel": "ksw_extend2 kernels (thread-per-task-pair ext3_kernel / ext2_kernel, warp-per-task ext_kernel, tail_kernel)",
                "bound": "int-issue (DPX), not hbm/tensor",
                "achieved": gcups, "peak": gcups_peak, "unit": "GCUPS", "frac": gcups / gcups_peak if gcups_peak else None,
                "traffic": traffic, "traffic_how": "ncu --set full dram__bytes_read.sum + dram__bytes_write.sum per extension-kernel launch "
                                               "(profiles/ext3_traffic.json: the class 65-80 launch of a sample's first round); the kernel is issue-bound, not DRAM-bound",
                "avg_launch_ms": ext_ms / max(1, stage_launch["extend"]),
                "work": f"{cells_total} executed ksw_extend2 cells in {K} steps ({cells_total / max(1, Pk):.0f} cells/pair)",
                "cells_per_pair": cells_total / max(1, Pk),
                "peak_how": f"measured in this run: {dpx_gops:.0f} G lane-instr/s of viaddmax_s16x2_relu x 2 cells / 9 instr",
                "dominant_stage": dom}
    pile_ms = stage_ms["pileup"]
    pile_b = 2 * ((L + 3) // 4 + L + 16 + 8)            # SURVEY.md 8d: packed bases + qualities + header + 2 CIGAR ops, per read
    pile_gbs = pile_b * Pk / pile_ms / 1e6 if pile_ms > 0 else 0.0
    pile_traffic = None
    try:
        pile_traffic = json.load(open(os.path.join(ROOT, "profiles", "pileup_traffic.json")))["dram_bytes_per_launch"]
    except (OSError, KeyError, ValueError):
        pass
    roofline_pileup = {"kernel": "pileup_kernel", "bound": "hbm", "achieved": pile_gbs, "peak": hbm_peak, "unit": "GB/s",
                       "frac": pile_gbs / hbm_peak, "traffic": pile_traffic, "peak_how": hbm_src,
                       "work": f"{pile_b} B/pair algorithmic x {Pk} pairs"}
    seed_ms = stage_ms["seed_chain"]
    seed_b = 2 * ((L + 3) // 4)                         # SURVEY.md 8d: packed read bytes read once (seed records are reported apart)
    seed_gbs = seed_b * Pk / seed_ms / 1e6 if seed_ms > 0 else 0.0
    seed_traffic = None
    try:
        seed_traffic = json.load(open(os.path.join(ROOT, "profiles", "seed_traffic.json")))["dram_bytes_per_launch"]
    except (OSError, KeyError, ValueError):
        pass
    roofline_seed = {"kernel": "pack_reads_kernel + seed_walk_kernel + plan_kernel", "bound": "hbm (algorithmic); in practice the latency of dependent L2 look-ups at ~11 of 32 lanes",
                     "achieved": seed_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": seed_gbs / hbm_peak, "traffic": seed_traffic,
                     "work": f"{seed_b} B/pair of 2-bit packed read bases x {Pk} pairs; the reads arrive 1 B/base ({2 * L} B/pair), are packed once by "
                             f"pack_reads_kernel and walked from the packed copy"}
    launches = int(sum(stage_launch.values()))
    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
           "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong" if plan.strong else "weak", "vs_baseline": None,
           "dtype": "int32", "data": "synthetic", "config": plan.config_dict(world, P), "clocks": clk, "e2e": e2e,
           "gpu_launches": launches, "roofline": roofline, "roofline_pileup": roofline_pileup, "roofline_seed": roofline_seed,
           "step_ms": [round(x, 3) for x in step_ms],
           "stages_ms_per_step": {k: v / K for k, v in stage_ms.items()},
           "stage_launches": stage_launch,
           "results": {k: {"calls": v[0], "TP": v[1], "FP": v[2], "FN": v[3]} for k, v in results.items()}}

    if not args.no_cpu_baseline and world == 1:
        qmo_py = cpu_setup()
        n = calibrated_cpu_sample(plan, args.cpu_seconds, P)
        v, cms = cpu_arm(plan, 1, 0, n)
        out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": qmo_py.n_threads(), "kind": "port",
                               "sample": f"first {n} pairs of the first step's sample ({cms / 1e3:.1f} s): oracle port of bwa-mem "
                                         f"extension + mate rescue + pairing + CIGAR + bcftools-style counting, OpenMP over reads; "
                                         f"build {qmo_py.BUILD_KIND}", "note": CPU_NOTE}
    print(json.dumps(out), file=_json_out, flush=True)
    if world > 1:
        for x in smp.values():
            x.close()
        comm.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    # stdout carries exactly one JSON line: whatever else a library prints there (NCCL's version banner, for one) goes to
    # stderr -- file descriptor 1 is pointed at stderr for the whole run and the line is written to the saved original
    sys.dont_write_bytecode = True          # the tree may be read-only: nothing is written into it
    sys.stdout.flush()
    _json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
