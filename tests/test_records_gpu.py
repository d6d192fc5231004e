"""The record consumers on the device against the C oracle, on hand-built records (tests/recgen.py) instead of aligner
output: the count planes, counts_to_rows and the indel table of qm_pileup_accumulate_indels at every staging path of the
kernel (strides 150 / 151 / 256 / 300 / 512, bases and qualities one byte off their alignment), the persistent loop of a
batch larger than the grid, the text pileup byte for byte, BAQ at contig ends, and the stride limit."""
import ctypes as C

import numpy as np
import pytest

from tests import recgen
from tests.recgen import M, S

pytestmark = pytest.mark.gpu

OPTS = [dict(), dict(min_bq=0), dict(min_bq=30, min_mapq=20), dict(count_orphans=1, ignore_overlaps=1),
        dict(min_bq=-1), dict(min_bq=201), dict(min_bq=256)]
OPT_IDS = [",".join(f"{k}={v}" for k, v in d.items()) or "default" for d in OPTS]
# (stride, byte offset): every kPre launch of the kernel with the wide copy, and the byte-wise copy (odd stride, or
# bases / qualities not 4-byte aligned)
LAYOUTS = [(150, 0), (151, 0), (256, 0), (300, 0), (512, 0), (150, 1), (512, 1)]


@pytest.fixture(scope="module")
def ctx():
    from quasimodo_b200 import Context
    c = Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def genome():
    return recgen.Genome()


@pytest.fixture(scope="module")
def ref(genome):
    from oracle import qmo_py
    return qmo_py.Ref(genome.codes, genome.lens, k=31)


@pytest.fixture(scope="module")
def idx(ctx, genome):
    i = ctx.index(genome, 31)
    yield i
    i.close()


@pytest.fixture(scope="module")
def batch(genome):
    b = recgen.random_batch(genome, 1500, 5, batch=recgen.adversarial(genome))
    return b.arrays(150)


def popts(d):
    from oracle import qmo_py
    from quasimodo_b200 import _lib
    po, pg = qmo_py.PileupOpt(), _lib.default_pileup_opt()
    qmo_py.lib().qmo_pileup_opt_default(C.byref(po))
    for k, v in d.items():
        setattr(po, k, v)
        setattr(pg, k, v)
    return po, pg


def gpu_pileup(ctx, idx, alns, codes, quals, lens, stride, offset, pg):
    """-> (planes [16, l_pac], rows [l_pac, 16], indel records) of one qm_pileup_accumulate_indels call on the records
    laid out at `stride`, bases and qualities starting `offset` bytes into their buffers"""
    import torch
    from quasimodo_b200 import _lib
    L = _lib.lib()
    dev = torch.device("cuda:0")
    c, q = recgen.relayout(codes, quals, lens, stride, offset, seed=stride + offset)
    d_c, d_q = torch.from_numpy(c.reshape(-1)).to(dev)[offset:], torch.from_numpy(q.reshape(-1)).to(dev)[offset:]
    d_a = torch.from_numpy(alns.view(np.uint8).reshape(-1)).to(dev)
    d_l = torch.from_numpy(np.ascontiguousarray(lens, np.int32)).to(dev)
    counts = torch.zeros(16 * idx.l_pac, dtype=torch.int32, device=dev)
    tab = C.c_void_p()
    assert L.qm_indel_table_create(ctx._h, 16, C.byref(tab)) == 0
    try:
        rc = L.qm_pileup_accumulate_indels(ctx._h, idx._h, C.byref(pg), C.c_void_p(d_a.data_ptr()), C.c_void_p(d_c.data_ptr()),
                                           C.c_void_p(d_q.data_ptr()), stride, C.c_void_p(d_l.data_ptr()), len(lens) // 2,
                                           C.c_void_p(counts.data_ptr()), tab, None)
        assert rc == 0, L.qm_last_error(ctx._h)
        rows = ctx.counts_to_rows(idx, counts).cpu().numpy()
        out = np.zeros(1 << 16, _lib.INDEL_DTYPE)
        n = C.c_int64()
        assert L.qm_indel_table_fetch_host(tab, idx._h, out.ctypes.data, len(out), C.byref(n)) == 0
    finally:
        L.qm_indel_table_destroy(tab)
    return counts.view(16, idx.l_pac).cpu().numpy(), rows, out[:n.value]


@pytest.mark.parametrize("opt", OPTS, ids=OPT_IDS)
def test_counts_and_indels_at_every_layout(ctx, idx, ref, batch, opt):
    from oracle import qmo_py
    from tests.test_indels_gpu import as_rows
    alns, codes, quals, lens = batch
    po, pg = popts(opt)
    want = qmo_py.pileup(ref, alns, codes, quals, lens, popt=po)
    want_ind = qmo_py.indels(ref, alns, codes, lens, popt=po)
    assert want[:, 14].sum() > 0 and len(want_ind) > 100
    for stride, offset in LAYOUTS:
        planes, rows, ind = gpu_pileup(ctx, idx, alns, codes, quals, lens, stride, offset, pg)
        where = (stride, offset)
        assert np.array_equal(planes.T, want), (where, np.argwhere(planes.T != want)[:8])
        assert np.array_equal(rows, want), where
        assert np.array_equal(as_rows(ind), want_ind), where


def test_persistent_loop_of_a_large_batch(ctx, idx, ref, batch):
    """more pairs than warps in the persistent grid (sm_count * 16 blocks of 4 warps): every warp takes several pairs and
    prefetches the next one's words"""
    from oracle import qmo_py
    from tests.test_indels_gpu import as_rows
    n = ctx.sm_count * 64 * 2 + 77
    alns, codes, quals, lens = recgen.tiled(batch, n, 17)
    for opt in (dict(), dict(min_bq=-1, ignore_overlaps=1)):
        po, pg = popts(opt)
        want = qmo_py.pileup(ref, alns, codes, quals, lens, popt=po)
        for stride, offset in ((150, 0), (151, 0)):
            planes, _, ind = gpu_pileup(ctx, idx, alns, codes, quals, lens, stride, offset, pg)
            assert np.array_equal(planes.T, want), (opt, stride)
            assert np.array_equal(as_rows(ind), qmo_py.indels(ref, alns, codes, lens, popt=po)), (opt, stride)


def test_long_reads(ctx, idx, ref, genome):
    """reads up to 512 bases (insertions longer than 255) at stride 512, wide and byte-wise"""
    from oracle import qmo_py
    from tests.test_indels_gpu import as_rows
    alns, codes, quals, lens = recgen.long_batch(genome, 400, 23).arrays(512)
    po, pg = popts({})
    want, want_ind = qmo_py.pileup(ref, alns, codes, quals, lens, popt=po), qmo_py.indels(ref, alns, codes, lens, popt=po)
    assert (want_ind[:, 2] == 255).any()
    for offset in (0, 1):
        planes, _, ind = gpu_pileup(ctx, idx, alns, codes, quals, lens, 512, offset, pg)
        assert np.array_equal(planes.T, want), offset
        assert np.array_equal(as_rows(ind), want_ind), offset


@pytest.mark.parametrize("opt", OPTS, ids=OPT_IDS)
def test_text_pileup(ctx, idx, ref, genome, batch, opt):
    import torch
    from oracle import qmo_py
    alns, codes, quals, lens = batch
    po, pg = popts(opt)
    want = qmo_py.mpileup_text(ref, alns, codes, quals, lens, genome.names, popt=po)
    dev = torch.device("cuda:0")
    got = ctx.mpileup_text(idx, torch.from_numpy(alns.view(np.uint8).reshape(-1)).to(dev), torch.from_numpy(codes).to(dev),
                           torch.from_numpy(quals).to(dev), torch.from_numpy(lens).to(dev), genome.names, popt=pg)
    assert len(want) > 10000
    if got != want:
        gl, wl = got.split(b"\n"), want.split(b"\n")
        bad = [i for i in range(min(len(gl), len(wl))) if gl[i] != wl[i]]
        assert not bad and len(gl) == len(wl), (len(gl), len(wl), gl[bad[0]][:200] if bad else b"", wl[bad[0]][:200] if bad else b"")
    assert got == want


@pytest.mark.parametrize("flag", [3, 1])
def test_baq_at_contig_ends(ctx, idx, ref, genome, batch, flag):
    from oracle import qmo_py
    alns, codes, quals, lens = batch
    placed = (alns["n_cigar"] > 0) & (alns["n_cigar"] < 255) & (alns["rid"] >= 0)
    ends = np.array([recgen.span([(int(c) & 15, int(c) >> 4) for c in a["cigar"][:int(a["n_cigar"])]]) for a in alns]) + alns["pos"]
    assert (placed & (alns["pos"] == 0)).any() and (placed & (ends == genome.lens[np.maximum(alns["rid"], 0)])).any()
    assert (placed & (alns["rid"] == 1)).any() and (placed & (alns["rid"] == len(genome.lens) - 1)).any()
    want = qmo_py.baq(ref, alns, codes, quals, lens, flag=flag)
    got = ctx.baq_apply_host(idx, alns, codes, quals, lens, flag=flag)
    assert (want != quals).any()
    for r in range(len(lens)):
        assert np.array_equal(got[r, :lens[r]], want[r, :lens[r]]), r


def test_stride_above_512_is_refused(ctx, idx, genome):
    """a stride above the kernel's 512-base staging is an error (QM_ELIMIT), not a batch whose long reads vanish"""
    import torch
    from quasimodo_b200 import _lib
    rng = np.random.default_rng(2)
    b = recgen.Batch(genome, rng)
    b.add(b.read(2, 0, [(S, 100), (M, 500)]), b.read(2, 10, [(M, 300)], 0x1 | 0x2 | 0x10))
    alns, codes, quals, lens = b.arrays(600)
    dev = torch.device("cuda:0")
    counts = torch.zeros(16 * idx.l_pac, dtype=torch.int32, device=dev)
    L = _lib.lib()
    args = [torch.from_numpy(x).to(dev) for x in (alns.view(np.uint8).reshape(-1), codes, quals, lens)]
    rc = L.qm_pileup_accumulate(ctx._h, idx._h, C.byref(_lib.default_pileup_opt()), *[C.c_void_p(t.data_ptr()) for t in args[:3]], 600,
                                C.c_void_p(args[3].data_ptr()), 1, C.c_void_p(counts.data_ptr()), None)
    assert rc == -5 and b"512" in L.qm_last_error(ctx._h)
    assert int(counts.abs().sum()) == 0
