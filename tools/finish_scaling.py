"""Cost of qm_sample_finish_comm: duplicate marking and the depth cap over a sample sharded across ranks.

    torchrun --nproc-per-node N tools/finish_scaling.py [--pairs 1000000] [--max-depth 250]

Each rank simulates its contiguous shard of a deep Merlin sample on its GPU, adds it to a qm_sample with rmdup on and the cap at
--max-depth, and times qm_sample_finish_comm (host clock around the synchronous call, all ranks started together).  Rank 0 then
runs qm_sample_finish on the whole sample on its own GPU for comparison and prints one JSON line: ranks, pairs, duplicate pairs,
capped reads, bytes of tuples in the two unions every rank gathers, and the milliseconds of both calls."""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from quasimodo_b200 import Context, _lib, sharding, workloads  # noqa: E402
from quasimodo_b200.api import Comm  # noqa: E402


def sample(ctx, idx, W, g, lo, hi, max_depth, pre, stream):
    """a deferred sample of pairs [lo, hi) on ctx's GPU -> (sample, codes, quals, lens)"""
    dev = torch.device(f"cuda:{ctx.device}")
    n = hi - lo
    c = torch.empty((2 * n, 150), dtype=torch.uint8, device=dev)
    q = torch.empty_like(c)
    ctx.simulate_pairs(W, lo, n, g, c, q, stream)
    lens = torch.full((2 * n,), 150, dtype=torch.int32, device=dev)
    s = ctx.sample(idx)
    s.set_rmdup(True)
    s.set_max_depth(max_depth)
    s.estimate_pestat(pre[0], pre[1], stream)            # every rank: the model of the sample's first pairs
    s.add_pairs(c, q, lens, pair_id0=lo, stream=stream)
    torch.cuda.synchronize(dev)
    return s, c, q, lens


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=1_000_000)
    ap.add_argument("--max-depth", type=int, default=250)
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(local)
    ctx = Context(local)
    box = [Comm.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    comm = Comm(ctx, world, rank, box[0])
    st = torch.cuda.current_stream().cuda_stream
    W = workloads.Workload("merlin-deep", [("Merlin", 1)], ["Merlin"], args.pairs, 4242)
    idx = ctx.index(W.ref, 31)
    g = torch.from_numpy(W.src_codes).cuda()
    npre = min(_lib.PESTAT_PAIRS, args.pairs)
    pc = torch.empty((2 * npre, 150), dtype=torch.uint8, device="cuda")
    ctx.simulate_pairs(W, 0, npre, g, pc, torch.empty_like(pc), st)
    pre = (pc, torch.full((2 * npre,), 150, dtype=torch.int32, device="cuda"))
    lo, hi = sharding.shard_range(args.pairs, rank, world)
    s, c, q, lens = sample(ctx, idx, W, g, lo, hi, args.max_depth, pre, st)
    dist.barrier()
    t0 = time.perf_counter()
    n_dup, n_cap = s.finish_comm(comm, st)
    ms_comm = 1e3 * (time.perf_counter() - t0)
    # tuples this rank put into the two unions: pairs with a placed end, admitted reads after marking
    kept = torch.from_numpy(s.kept_alns(hi - lo).view(np.uint8).reshape(-1, 128)).cuda()
    n_tuples = (ctx.dup_keys([kept], [q], [lens], [lo]).shape[0], ctx.cap_keys([kept], [lo]).shape[0])
    s.close()
    del c, q, lens, kept
    stats = [None] * world
    dist.all_gather_object(stats, (ms_comm, n_dup, n_cap, n_tuples))
    if rank == 0:
        s1, c, q, lens = sample(ctx, idx, W, g, 0, args.pairs, args.max_depth, pre, st)
        t0 = time.perf_counter()
        n_dup1, n_cap1 = s1.finish(st)
        ms_one = 1e3 * (time.perf_counter() - t0)
        s1.close()
        assert all(x[1] == n_dup1 and x[2] == n_cap1 for x in stats), (stats, n_dup1, n_cap1)
        print(json.dumps(dict(gpu=torch.cuda.get_device_name(0), ranks=world, pairs=args.pairs, max_depth=args.max_depth,
                              dup_pairs=n_dup1, capped_reads=n_cap1,
                              union_bytes=sum(32 * x[3][0] + 16 * x[3][1] for x in stats),
                              finish_comm_ms=[round(x[0], 2) for x in stats], finish_one_gpu_ms=round(ms_one, 2))))
    dist.barrier()
    idx.close()
    comm.close()
    ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
