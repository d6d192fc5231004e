"""Duplicate marking and the depth cap over a sample sharded across ranks: each rank exports small tuples (qm_dup_keys, qm_cap_keys),
the union of every rank's tuples decides, each rank applies the verdict to its own records (qm_mark_duplicates_keys,
qm_depth_cap_keys; qm_sample_finish_comm wraps the whole sequence).  The result must be the one of one device holding the whole
sample.  The first tests emulate the ranks on one GPU (a concatenation in shuffled rank order stands in for the all-gather); the last
two run real ranks and skip on a machine with one GPU."""
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CHUNKS = [0, 3001, 7000, 11999, 16000, 20500, 26003, 30000]       # uneven chunks of the 30,000-pair sample


@pytest.fixture(scope="module")
def ctx():
    from quasimodo_b200 import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def deep():
    """the deep PhiX sample of tests/test_dedup_gpu.py: 30,000 pairs at ~1700x, 600 of them with the second mate blanked to N"""
    from oracle import dedup_py, qmo_py
    from quasimodo_b200 import workloads
    n = 30_000
    W = workloads.Workload("phix-deep", [("Phix", 1)], ["Phix"], n, 901)
    codes, quals, _, _ = W.simulate_host(0, n)
    lens = np.full(2 * n, 150, np.int32)
    codes[1:1200:2] = 4
    ref = qmo_py.Ref(W.ref.codes, W.ref.lens, k=31)
    alns, _, _, _ = qmo_py.run_sample(ref, codes, quals, lens)
    dup = dedup_py.mark_duplicates(alns, quals, lens)
    marked = alns.copy()
    for e in (0, 1):
        sel = dup & ((marked["flag"][e::2] & 4) == 0)
        marked["flag"][e::2][sel] |= 0x400
    return dict(W=W, n=n, ref=ref, codes=codes, quals=quals, lens=lens, alns=alns, dup=dup, marked=marked)


def _splits(n, k):
    """(name, ranks): each rank a list of (lo, hi) pair ranges -- whole chunks dealt round-robin, or one ragged contiguous range per
    rank (with k = 5 one rank holds nothing)"""
    rr = [[(CHUNKS[c], CHUNKS[c + 1]) for c in range(len(CHUNKS) - 1) if c % k == r] for r in range(k)]
    rng = np.random.default_rng(k)
    cuts = sorted(rng.choice(np.arange(1, n), k - 1, replace=False).tolist())
    if k == 5:
        cuts[2] = cuts[1]
    b = [0] + cuts + [n]
    cont = [[(b[r], b[r + 1])] if b[r + 1] > b[r] else [] for r in range(k)]
    return [("round-robin", rr), ("contiguous", cont)]


def _dev(deep, alns):
    import torch
    return (torch.from_numpy(np.ascontiguousarray(alns).view(np.uint8).reshape(-1, 128).copy()).cuda(),
            torch.from_numpy(deep["quals"]).cuda(), torch.from_numpy(deep["lens"]).cuda())


def _flags(d_alns):
    from quasimodo_b200 import _lib
    return d_alns.cpu().numpy().reshape(-1).view(_lib.ALN_DTYPE)["flag"]


def _union(parts, seed):
    """the all-gather's stand-in: every rank's tuples concatenated in a shuffled rank order"""
    import torch
    order = np.random.default_rng(seed).permutation(len(parts))
    return torch.cat([parts[r] for r in order])


@pytest.mark.parametrize("k", [2, 3, 5])
def test_duplicates_over_emulated_ranks(ctx, deep, k):
    import torch
    from quasimodo_b200 import QmError, _lib
    n = deep["n"]
    d_a0, d_q, d_l = _dev(deep, deep["alns"])
    whole = d_a0.clone()
    n_whole = ctx.mark_duplicates([whole], [d_q], [d_l])
    assert n_whole == int(deep["dup"].sum()) > 0
    assert np.array_equal(_flags(whole), deep["marked"]["flag"])
    for name, ranks in _splits(n, k):
        d_a = d_a0.clone()
        view = [dict(a=[d_a[2 * lo:2 * hi] for lo, hi in rk], q=[d_q[2 * lo:2 * hi] for lo, hi in rk], l=[d_l[2 * lo:2 * hi] for lo, hi in rk],
                     ids=[lo for lo, _ in rk]) for rk in ranks]
        parts = [ctx.dup_keys(v["a"], v["q"], v["l"], v["ids"]) for v in view]
        union = _union(parts, k)
        ids = union.cpu().numpy().reshape(-1).view(_lib.DUP_KEY_DTYPE)["pair_id"]
        assert len(np.unique(ids)) == len(ids) and 0 < len(ids) <= n, name
        # a repeated pair id: every rank gets the same refusal and nothing is flagged
        bad = torch.cat([union, union[:1]])
        with pytest.raises(QmError, match="code -1"):
            ctx.mark_duplicates_keys(bad, view[0]["a"], view[0]["ids"])
        assert np.array_equal(_flags(d_a), deep["alns"]["flag"]), name
        totals = [ctx.mark_duplicates_keys(union, v["a"], v["ids"]) for v in view]
        assert totals == [n_whole] * k, name
        assert np.array_equal(_flags(d_a), deep["marked"]["flag"]), name


@pytest.mark.parametrize("max_depth", [250, 1000, 8000])
def test_depth_cap_over_emulated_ranks(ctx, deep, max_depth):
    import torch
    from oracle import qmo_py
    from quasimodo_b200 import QmError
    n = deep["n"]
    keep = qmo_py.depth_cap(deep["ref"], deep["marked"], max_depth)            # the keep mask of qmo_py.pileup_capped
    admitted = qmo_py.depth_cap(deep["ref"], deep["marked"], 1 << 30)
    want = (admitted & ~keep).astype(np.uint8)
    d_a, _, _ = _dev(deep, deep["marked"])
    drops, n_whole = ctx.depth_cap([d_a], max_depth)
    assert np.array_equal(drops[0].cpu().numpy(), want) and n_whole == int(want.sum())
    if max_depth < 8000:
        assert 0 < n_whole < admitted.sum()
    else:
        assert n_whole == 0
    for k in (2, 3, 5):
        for name, ranks in _splits(n, k):
            view = [dict(a=[d_a[2 * lo:2 * hi] for lo, hi in rk], n=[hi - lo for lo, hi in rk], ids=[lo for lo, _ in rk]) for rk in ranks]
            parts = [ctx.cap_keys(v["a"], v["ids"]) for v in view]
            union = _union(parts, 10 * k + 1)
            assert union.shape[0] == int(admitted.sum()), (k, name)
            with pytest.raises(QmError, match="code -1"):
                ctx.depth_cap_keys(torch.cat([union[:3], union]), max_depth, view[0]["n"], view[0]["ids"])
            got = np.zeros(2 * n, np.uint8)
            totals = []
            for v in view:
                dr, t = ctx.depth_cap_keys(union, max_depth, v["n"], v["ids"])
                totals.append(t)
                for d, lo in zip(dr, v["ids"]):
                    got[2 * lo:2 * lo + d.numel()] = d.cpu().numpy()
            assert totals == [n_whole] * k, (k, name)
            assert np.array_equal(got, want), (k, name)


def _sample_run(ctx, idx, deep, rmdup, max_depth, comm=None):
    s = ctx.sample(idx)
    if rmdup:
        s.set_rmdup(True)
    if max_depth:
        s.set_max_depth(max_depth)
    h = deep["n"] // 3 * 2
    s.add_pairs_host(deep["codes"][:h], deep["quals"][:h], deep["lens"][:h])
    s.add_pairs_host(deep["codes"][h:], deep["quals"][h:], deep["lens"][h:], pair_id0=h // 2)
    totals = s.finish_comm(comm) if comm is not None else s.finish()
    out = dict(totals=totals, counts=s.counts_host(), flags=s.kept_alns(deep["n"])["flag"], indels=s.indels())
    s.close()
    return out


@pytest.mark.parametrize("rmdup,max_depth", [(True, 0), (False, 500), (True, 500)], ids=["rmdup", "cap", "both"])
def test_one_rank_communicator_equals_finish(ctx, deep, rmdup, max_depth):
    from quasimodo_b200.api import Comm
    if not Comm.available():
        pytest.skip("NCCL is not loadable")
    idx = ctx.index(deep["W"].ref, 31)
    (comm,) = Comm.init_all([ctx])
    want = _sample_run(ctx, idx, deep, rmdup, max_depth)
    got = _sample_run(ctx, idx, deep, rmdup, max_depth, comm)
    comm.close()
    idx.close()
    assert got["totals"] == want["totals"]
    assert (want["totals"][0] > 0) == rmdup and (want["totals"][1] > 0) == (max_depth > 0)
    assert np.array_equal(got["counts"], want["counts"]) and want["counts"].any()
    assert np.array_equal(got["flags"], want["flags"])
    assert got["indels"].tobytes() == want["indels"].tobytes()


def _rank_worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from quasimodo_b200 import Context, sharding
        from quasimodo_b200.api import Comm
        d = np.load(os.path.join(out_dir, "reads.npz"))
        codes, quals, lens = d["codes"], d["quals"], d["lens"]
        n = len(lens) // 2
        torch.cuda.set_device(rank)
        ctx = Context(rank)
        box = [Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        comm = Comm(ctx, world, rank, box[0])
        from quasimodo_b200 import workloads
        W = workloads.Workload("phix-deep", [("Phix", 1)], ["Phix"], n, 901)
        idx = ctx.index(W.ref, 31)
        s = ctx.sample(idx)
        s.set_comm(comm)
        s.set_rmdup(True)
        s.set_max_depth(500)
        # the sample is smaller than the insert-size prefix: every rank takes the model from the whole sample's first pairs
        s.estimate_pestat(torch.from_numpy(codes).cuda(), torch.from_numpy(lens).cuda())
        lo, hi = sharding.shard_range(n, rank, world)
        s.add_pairs_host(codes[2 * lo:2 * hi], quals[2 * lo:2 * hi], lens[2 * lo:2 * hi], pair_id0=lo)
        nd, nc = s.finish_comm(comm)
        s.allreduce_counts()
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), totals=np.array([nd, nc]), counts=s.counts_host(),
                 flags=s.kept_alns(hi - lo)["flag"], lo=lo, hi=hi, indels=s.indels().view(np.uint8))
        s.close()
        idx.close()
        comm.close()
        ctx.close()
    finally:
        dist.barrier()
        dist.destroy_process_group()


def test_two_processes_equal_one_gpu(ctx, deep, tmp_path):
    import torch
    import torch.multiprocessing as mp
    from quasimodo_b200.api import Comm
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    if not Comm.available():
        pytest.skip("NCCL is not loadable")
    idx = ctx.index(deep["W"].ref, 31)
    s = ctx.sample(idx)
    s.set_rmdup(True)
    s.set_max_depth(500)
    s.add_pairs_host(deep["codes"], deep["quals"], deep["lens"])
    want_totals = s.finish()
    want = dict(counts=s.counts_host(), flags=s.kept_alns(deep["n"])["flag"], indels=s.indels())
    s.close()
    idx.close()
    assert want_totals[0] > 0 and want_totals[1] > 0
    np.savez(tmp_path / "reads.npz", codes=deep["codes"], quals=deep["quals"], lens=deep["lens"])
    with socket.socket() as so:
        so.bind(("127.0.0.1", 0))
        port = so.getsockname()[1]
    mp.spawn(_rank_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        got = np.load(tmp_path / f"rank{r}.npz")
        assert tuple(got["totals"]) == want_totals, r
        assert np.array_equal(got["counts"], want["counts"]), r
        lo, hi = int(got["lo"]), int(got["hi"])
        assert np.array_equal(got["flags"], want["flags"][2 * lo:2 * hi]), r
        assert got["indels"].tobytes() == want["indels"].tobytes(), r


def test_driver_on_two_gpus_with_rmdup_and_cap_writes_the_same_files(tmp_path):
    """--gpus 0,1 --rmdup 1 --max-depth 250 writes what --gpu 0 writes.  The driver raises --batch-pairs to the 65,536 pairs of the
    insert-size prefix, so 280,000 pairs make five batches: three on GPU 0, two on GPU 1"""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import re
    from quasimodo_b200 import workloads
    from tests import bamio, drvutil
    n = 280_000
    W = workloads.config1(n)
    codes, quals, _, _ = W.simulate_host(0, n)
    lens = np.full(2 * n, 150, np.int32)
    fa, r1, r2 = str(tmp_path / "ref.fa"), str(tmp_path / "r1.fq"), str(tmp_path / "r2.fq")
    drvutil.write_fasta(W.ref, fa)
    drvutil.write_fastq(codes, quals, lens, drvutil.pair_names("p", n), r1, r2)

    def records(path):
        data = b"".join(d for _, d in bamio.bgzf_blocks(path))
        return data[8 + int.from_bytes(data[4:8], "little"):]

    outs = []
    for tag, gp in (("one", ["--gpu", 0]), ("two", ["--gpus", "0,1"])):
        f = {x: str(tmp_path / f"{tag}.{x}") for x in ("bam", "rmdup.bam", "tsv", "vcf", "metrics", "mpileup")}
        p = drvutil.run_driver(["sample", "--ref", fa, "--r1", r1, "--r2", r2, "--sample", "s", "--rmdup", 1, "--max-depth", 250,
                                "--batch-pairs", 4096, "--bam", f["bam"], "--rmdup-bam", f["rmdup.bam"], "--metrics", f["metrics"],
                                "--counts", f["tsv"], "--vcf", f["vcf"], "--mpileup", f["mpileup"]] + gp)
        n_dup = int(re.search(r"rmdup: (\d+) of", p.stderr).group(1))
        n_cap = int(re.search(r"depth cap 250: (\d+) reads", p.stderr).group(1))
        outs.append(dict(bam=records(f["bam"]), rbam=records(f["rmdup.bam"]), tsv=open(f["tsv"], "rb").read(),
                         vcf=[ln for ln in open(f["vcf"]) if not ln.startswith("##reference")], met=open(f["metrics"]).read(),
                         txt=open(f["mpileup"], "rb").read(), n_dup=n_dup, n_cap=n_cap, log=p.stderr))
    one, two = outs
    assert "5 batch(es)" in one["log"] and "count tensors of 2 GPUs merged" in two["log"]
    assert one["n_dup"] > 0 and one["n_cap"] > 0
    for key in ("n_dup", "n_cap", "bam", "rbam", "tsv", "vcf", "met", "txt"):
        assert one[key] == two[key], key
