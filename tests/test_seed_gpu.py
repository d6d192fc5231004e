"""The read-level front end on the GPU -- seeding (pack_reads_kernel, seed_walk_kernel, seed_chain_kernel), chaining (plan_kernel) and
the extension state machine (advance_kernel, tail_kernel, the speculative finish) -- on hand-built repetitive genomes
(tests/seedgen.py), where reads reach the tracked 2..5-copy paths, inverted repeats, the occurrence cap, 64 seeds and 16 regions:
  * seeds equal the brute force of DESIGN.md 5.1, seed for seed, at k = 31, 20, 16, rows of 150, 400 and 512 bases (512: too wide
    for the staged pack, the per-thread loads run), every max_occ where the cap matters, and batches of 1 .. 3,000 reads;
  * regions and executed cells equal the oracle's, with the default scores and another scheme;
  * pairs from repeats: insert-size model, mate rescue and records equal the oracle's (equal-score hits, MAPQ 0);
  * with QM_F_FM_SEEDS the seeds equal the oracle's FM seeds in bwa's order;
  * the seed and region tests again under every kernel variant switch (read once per process: a subprocess each)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests import seedgen as sg

pytestmark = pytest.mark.gpu

VARIANT_ENV = ("QM_SEED_PERSIST", "QM_SEED_STAGE", "QM_BLOOM_BATCH", "QM_SEED_THREADS", "QM_SEED_REFILL", "QM_TAIL_MIN", "QM_SPEC",
               "QM_SPEC_DEPTH", "QM_EXT3")
SCHEMES = {"default": {}, "a2": dict(a=2, b=5, o_del=5, e_del=2, o_ins=7, e_ins=1, T=50)}


@pytest.fixture(scope="module")
def ctx():
    from quasimodo_b200 import Context
    c = Context(0)
    yield c
    c.close()


def _opts(k, max_occ=500, flags=0, scheme=None):
    from oracle import qmo_py
    from quasimodo_b200 import _lib
    oo, og = qmo_py.default_opt(), _lib.default_opt()
    for o in (oo, og):
        o.min_seed_len, o.max_occ, o.flags = k, max_occ, flags
        for name, v in (scheme or {}).items():
            setattr(o, name, v)
    return oo, og


def _dev(*arrays):
    import torch
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


def gpu_seeds(ctx, idx, codes, lens, opt):
    import torch
    from quasimodo_b200 import _lib
    d_codes, d_lens = _dev(codes, lens)
    seeds, n_seeds = ctx.collect_seeds(idx, d_codes, d_lens, opt=opt)
    torch.cuda.synchronize()
    return seeds.cpu().numpy().view(_lib.SEED_DTYPE).reshape(len(lens), _lib.MAX_SEEDS), n_seeds.cpu().numpy()


def occs_of(g):
    return sg.MAX_OCCS if g.name.startswith(("occ", "tan")) else (500, 2)


@pytest.mark.parametrize("stride", [150, 400, 512])
@pytest.mark.parametrize("k", [31, 20, 16])
def test_seeds_equal_brute_force(ctx, k, stride):
    n64 = 0
    for g in sg.families(k):
        ix = sg.KmerIndex(g, k)
        idx = ctx.index(g, k)
        codes, lens = sg.reads(g, k, 32, stride, seed=2000 + k + stride)
        for mo in occs_of(g):
            _, og = _opts(k, mo)
            seeds, n_seeds = gpu_seeds(ctx, idx, codes, lens, og)
            got = sg.seed_lists(seeds, n_seeds)
            want = sg.brute_batch(ix, codes, lens, mo)
            bad = [r for r in range(len(got)) if got[r] != want[r]]
            assert not bad, (g.name, k, stride, mo, bad[:5], got[bad[0]][:6], want[bad[0]][:6])
            n64 += int((n_seeds == sg.MAX_SEEDS).sum())
        idx.close()
    assert n64 > 20


@pytest.mark.parametrize("n", [1, 31, 33, 65, 3000])
def test_seed_batch_sizes(ctx, n):
    """the persistent walk takes reads in ranges of 64 off a global cursor and refills lanes in bursts: batches of one read, under
    and over a warp, one past a range, and a few thousand"""
    k = 31
    g = sg.tandem(45, True)
    codes, lens = sg.reads(g, k, n, 150, seed=77)
    idx = ctx.index(g, k)
    _, og = _opts(k)
    seeds, n_seeds = gpu_seeds(ctx, idx, codes, lens, og)
    idx.close()
    want = sg.brute_batch(sg.KmerIndex(g, k), codes, lens, 500)
    got = sg.seed_lists(seeds, n_seeds)
    assert [r for r in range(n) if got[r] != want[r]] == []


@pytest.mark.parametrize("scheme", ["default", "a2"])
@pytest.mark.parametrize("k", [31, 20, 16])
def test_regions_equal_oracle(ctx, k, scheme):
    """regions (build_plan at 64 seeds, mem_chain_flt over many chains on both strands and several contigs, the 16-region cap) and the
    executed-cell count of every family"""
    import torch
    from oracle import qmo_py
    from quasimodo_b200 import _lib
    n16 = n64 = 0
    for g in sg.families(k):
        codes, lens = sg.reads(g, k, 64, 150, seed=3000 + k)
        ref = qmo_py.Ref(g.codes, g.lens, k=k)
        oo, og = _opts(k, scheme=SCHEMES[scheme])
        o = qmo_py.align_se(ref, codes, lens, opt=oo)
        idx = ctx.index(g, k)
        d_codes, d_lens = _dev(codes, lens)
        d_cells = torch.zeros(1, dtype=torch.int64, device="cuda")
        d_regs, d_nr = ctx.align_se(idx, d_codes, d_lens, d_cells=d_cells, opt=og)
        torch.cuda.synchronize()
        idx.close()
        regs = d_regs.cpu().numpy().view(_lib.REG_DTYPE).reshape(-1, _lib.MAX_REGS)
        nr = d_nr.cpu().numpy()
        assert np.array_equal(nr, o["n_regs"]), (g.name, np.flatnonzero(nr != o["n_regs"])[:5])
        bad = [r for r in range(len(nr)) if regs[r, :nr[r]].tobytes() != o["regs"][r, :nr[r]].tobytes()]
        assert not bad, (g.name, bad[:5])
        assert int(d_cells.item()) == o["cells"], g.name
        n16 += int((nr == qmo_py.MAX_REGS).sum())
        n64 += int((o["n_seeds"] == qmo_py.MAX_SEEDS).sum())
    assert n16 > 20 and n64 > 20


def test_records_equal_oracle(ctx):
    """pairs from a genome of dispersed, tandem, inverted and capped repeats: insert-size model, mate rescue, pairing and every record
    field as the oracle has them; reads in exact repeats give equal-score hits (bwa's hash tie-break, sub / sub_n, MAPQ 0)"""
    import torch
    from oracle import qmo_py
    from quasimodo_b200 import _lib
    g = sg.mixed()
    n = 3000
    codes, lens = sg.pairs(g, n, seed=91)
    k = 31
    ref = qmo_py.Ref(g.codes, g.lens, k=k)
    oo, og = _opts(k)
    o = qmo_py.align_se(ref, codes, lens, opt=oo)
    o_pes = qmo_py.pestat(ref, o["regs"], o["n_regs"], opt=oo)
    o_alns = qmo_py.pair_and_finish(ref, codes, lens, o["regs"], o["n_regs"], o_pes, opt=oo)
    idx = ctx.index(g, k)
    d_codes, d_lens = _dev(codes, lens)
    d_regs, d_nr = ctx.align_se(idx, d_codes, d_lens, opt=og)
    g_pes = ctx.pestat(idx, d_regs, d_nr, n, opt=og)
    d_alns = ctx.pair_finish(idx, d_codes, d_lens, d_regs, d_nr, g_pes, opt=og)
    torch.cuda.synchronize()
    alns = d_alns.cpu().numpy().view(_lib.ALN_DTYPE)
    idx.close()
    assert g_pes.tobytes() == o_pes.tobytes() and not o_pes[1]["failed"]
    for f in ("rid", "pos", "flag", "mapq", "n_cigar", "score", "sub", "nm", "mate_rid", "mate_pos", "tlen", "qb", "qe"):
        d = np.flatnonzero(alns[f] != o_alns[f])
        assert d.size == 0, (f, d[:5], alns[f][d[:5]], o_alns[f][d[:5]])
    nc = np.where(o_alns["n_cigar"] == 255, 0, o_alns["n_cigar"])
    mask = np.arange(alns["cigar"].shape[1])[None, :] < nc[:, None]
    assert np.array_equal(np.where(mask, alns["cigar"], 0), np.where(mask, o_alns["cigar"], 0))
    mapped = (o_alns["flag"] & 4) == 0
    assert mapped.mean() > 0.9 and int((mapped & (o_alns["mapq"] == 0)).sum()) > 30 and int((o_alns["sub"] > 0).sum()) > 100


@pytest.mark.parametrize("k", [31, 16])
def test_fm_seeds_equal_oracle(ctx, k):
    """QM_F_FM_SEEDS: the FM-index kernel's seeds on every family, in bwa's order, as the oracle's restatement finds them"""
    from oracle import qmo_py
    for g in sg.families(k):
        codes, lens = sg.reads(g, k, 48, 150, seed=4000 + k)
        ref = qmo_py.Ref(g.codes, g.lens, k=k)
        ref.set_fm(qmo_py.FmIndex(codes=g.codes))
        oo, og = _opts(k, flags=qmo_py.F_FM_SEEDS)
        o = qmo_py.align_se(ref, codes, lens, opt=oo)
        idx = ctx.index(g, k)
        idx.build_fm()
        seeds, n_seeds = gpu_seeds(ctx, idx, codes, lens, og)
        idx.close()
        assert np.array_equal(n_seeds, o["n_seeds"]), g.name
        bad = [r for r in range(len(lens)) if seeds[r, :n_seeds[r]].tobytes() != o["seeds"][r, :n_seeds[r]].tobytes()]
        assert not bad, (g.name, bad[:5])


def test_rows_longer_than_512_are_refused(ctx):
    """the read-level entries take rows of at most 512 bases (QM_ELIMIT above), as the paired and sample entries do"""
    from quasimodo_b200 import QmError
    g = sg.unique()
    idx = ctx.index(g, 31)
    _, og = _opts(31)
    codes, lens = sg.reads(g, 31, 4, 513, seed=5)
    d_codes, d_lens = _dev(codes, lens)
    for call in (ctx.collect_seeds, ctx.align_se):
        with pytest.raises(QmError, match="code -5"):
            call(idx, d_codes, d_lens, opt=og)
    idx.close()


@pytest.mark.parametrize("env", [
    {"QM_SEED_PERSIST": "0"}, {"QM_SEED_STAGE": "0"}, {"QM_BLOOM_BATCH": "1"}, {"QM_SEED_THREADS": "32"}, {"QM_SEED_REFILL": "1"},
    {"QM_TAIL_MIN": "0"}, {"QM_TAIL_MIN": "0", "QM_SPEC_DEPTH": "2"}, {"QM_TAIL_MIN": "0", "QM_SPEC": "0"}, {"QM_EXT3": "0"},
], ids=["one-kernel-seeding", "unstaged-pack", "one-filter-lookup", "32-thread-pack", "refill-one-lane", "speculative-finish",
        "two-seeds-per-pass", "bulk-rounds", "scalar-extension"])
def test_kernel_variants(env):
    """a test-sized batch never reaches the bulk rounds (fewer than max(2048, n / 64) tasks go to the tail kernel, fewer than
    max(8192, n / 8) to the speculative finish): QM_TAIL_MIN=0 and QM_SPEC=0 send it there; the seeding switches select the
    one-kernel seeder, the per-thread pack, one filter look-up at a time, 32-thread pack blocks and one-lane refills"""
    if any(os.environ.get(v) for v in VARIANT_ENV):
        pytest.skip("already inside a variant run")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    here = "tests/test_seed_gpu.py::"
    ids = [here + "test_seeds_equal_brute_force[" + p + "]" for p in ("31-150", "20-400", "16-512")] + \
          [here + "test_regions_equal_oracle[" + p + "]" for p in ("31-default", "20-default", "16-a2")] + [here + "test_seed_batch_sizes[3000]"]
    p = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-p", "no:cacheprovider"] + ids,
                       cwd=root, env=dict(os.environ, **env), capture_output=True, text=True)
    assert p.returncode == 0 and " passed" in p.stdout, p.stdout[-3000:] + p.stderr[-2000:]
