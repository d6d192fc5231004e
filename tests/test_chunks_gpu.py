"""Per-chunk insert-size models (qm_sample_set_chunks, `sample -K`): bwa mem pairs each input chunk against mem_pestat over all of that
chunk's pairs.  The device's models and records are held against the CPU oracle run chunk by chunk over slices of the batch
(oracle.qmo_py.pestat + pair_and_finish per slice); the records must not depend on how the chunks are spread over add calls,
entries or GPUs; a given model (-I) replaces every chunk's."""
import numpy as np
import pytest

from tests import drvutil

pytestmark = pytest.mark.gpu

FIELDS = ("rid", "pos", "flag", "mapq", "n_cigar", "score", "sub", "nm", "mate_rid", "mate_pos", "tlen", "qb", "qe")


@pytest.fixture(scope="module")
def ctx():
    from quasimodo_b200 import Context
    c = Context(0)
    yield c
    c.close()


def _workload(name, n):
    from quasimodo_b200 import workloads
    return {"cfg1": lambda: workloads.config1(n), "cfg2": lambda: workloads.config2(6, n),
            "cfg2-rescue-heavy": lambda: workloads.config2(1, n), "cfg5": lambda: workloads.config5(n)}[name]()


def oracle_by_chunk(W, codes, lens, chunks):
    """the oracle over each chunk's slice: -> (models [n_chunks, 4], records, rescue ran somewhere)"""
    from oracle import qmo_py
    opt = qmo_py.default_opt()
    opt.w = W.w
    ref = qmo_py.Ref(W.ref.codes, W.ref.lens, k=31)
    o = qmo_py.align_se(ref, codes, lens, opt=opt)
    regs = o["regs"].reshape(-1, qmo_py.MAX_REGS)
    models, alns = [], []
    p0 = 0
    for c in chunks:
        sl = slice(2 * p0, 2 * (p0 + c))
        r, nr = np.ascontiguousarray(regs[sl]).copy(), np.ascontiguousarray(o["n_regs"][sl]).copy()
        pes = qmo_py.pestat(ref, r, nr, opt=opt)
        models.append(pes)
        alns.append(qmo_py.pair_and_finish(ref, np.ascontiguousarray(codes[sl]), np.ascontiguousarray(lens[sl]), r, nr, pes, pair_id0=p0, opt=opt))
        p0 += c
    return np.stack(models), np.concatenate(alns)


def device_run(ctx, W, codes, quals, lens, calls, pes=None, entry="device"):
    """one sample; calls = [[chunk sizes of add call 0], [.. of call 1], ..] (None: the default path, one call); -> (records,
    models of every call's chunks, counts)"""
    import torch
    from quasimodo_b200 import _lib
    opt = _lib.default_opt()
    opt.w = W.w
    idx = ctx.index(W.ref, 31)
    s = ctx.sample(idx, opt=opt)
    if pes is not None:
        s.set_pestat(pes)
    n = codes.shape[0] // 2
    out = np.zeros(2 * n, dtype=_lib.ALN_DTYPE)
    models = []
    p0 = 0
    for sizes in (calls or [[n]]):
        m = int(sum(sizes))
        rows = slice(2 * p0, 2 * (p0 + m))
        if calls is not None:
            s.set_chunks(sizes)
        if entry == "device":
            dev = torch.device("cuda:0")
            d_alns = torch.zeros(2 * m * _lib.ALN_DTYPE.itemsize, dtype=torch.uint8, device=dev)
            s.add_pairs(torch.from_numpy(np.ascontiguousarray(codes[rows])).to(dev), torch.from_numpy(np.ascontiguousarray(quals[rows])).to(dev),
                        torch.from_numpy(np.ascontiguousarray(lens[rows])).to(dev), pair_id0=p0, d_alns=d_alns)
            torch.cuda.synchronize()
            out[rows] = d_alns.cpu().numpy().view(_lib.ALN_DTYPE)
        else:
            h = np.zeros(2 * m, dtype=_lib.ALN_DTYPE)
            s.add_pairs_host(np.ascontiguousarray(codes[rows]), np.ascontiguousarray(quals[rows]), np.ascontiguousarray(lens[rows]), pair_id0=p0, h_alns=h)
            out[rows] = h
        if calls is not None:
            models.append(s.chunk_pestat())
        p0 += m
    counts = s.counts_host()
    s.close()
    idx.close()
    return out, (np.concatenate(models) if models else None), counts


def same_records(g, o):
    for f in FIELDS:
        d = np.nonzero(g[f] != o[f])[0]
        assert d.size == 0, f"field {f}: {d.size} records differ, first {d[:5]}: {g[f][d[:5]]} vs {o[f][d[:5]]}"
    nc = np.where(o["n_cigar"] == 255, 0, o["n_cigar"])
    mask = np.arange(g["cigar"].shape[1])[None, :] < nc[:, None]
    assert np.array_equal(np.where(mask, g["cigar"], 0), np.where(mask, o["cigar"], 0))


def plan(n, rng):
    """chunk sizes over n pairs: a 4-pair chunk (too small for any orientation: every one fails, nothing is paired), one of 40
    (some orientations only), the rest random"""
    sizes = [4, 40]
    while sum(sizes) < n:
        sizes.append(int(min(n - sum(sizes), rng.integers(150, 900))))
    return sizes


@pytest.mark.parametrize("name,n", [("cfg1", 3000), ("cfg2", 3000), ("cfg5", 2000), ("cfg2-rescue-heavy", 6000)])
def test_chunks_equal_oracle_chunk_by_chunk(ctx, name, n):
    W = _workload(name, n)
    codes, quals, _, _ = W.simulate_host(0, n)
    lens = np.full(2 * n, W.params.read_len, np.int32)
    sizes = plan(n, np.random.default_rng(n))
    o_models, o_alns = oracle_by_chunk(W, codes, lens, sizes)
    # several chunks per add call, and a call boundary between chunks
    calls = [sizes[:5], sizes[5:]]
    g_alns, g_models, _ = device_run(ctx, W, codes, quals, lens, calls)
    assert g_models.shape == o_models.shape
    assert g_models.tobytes() == o_models.tobytes(), (g_models[:3], o_models[:3])
    assert o_models[0]["failed"].all()                              # the 4-pair chunk: every orientation failed
    assert not o_models[2:]["failed"][:, 1].any()                   # the others have an FR model
    same_records(g_alns, o_alns)
    small = g_alns[:8]
    assert not (small["flag"] & 2).any()                            # no proper pair in a chunk without a model
    # the models really differ from chunk to chunk, and the records from the one-model default path
    assert len({m.tobytes() for m in o_models[2:]}) > 1
    d_alns, _, _ = device_run(ctx, W, codes, quals, lens, None)
    assert any((d_alns[f] != g_alns[f]).any() for f in ("flag", "mapq", "pos"))


def test_rescue_fires_with_chunk_models(ctx):
    """mate rescue runs against each chunk's windows: a rescue-heavy sample in chunks places reads only rescue can place"""
    from oracle import qmo_py
    from quasimodo_b200 import _lib
    W = _workload("cfg2-rescue-heavy", 3000)
    codes, quals, _, _ = W.simulate_host(0, 3000)
    lens = np.full(6000, 150, np.int32)
    sizes = [1000, 1000, 1000]
    on, _, _ = device_run(ctx, W, codes, quals, lens, [sizes])
    o_models, o_alns = oracle_by_chunk(W, codes, lens, sizes)
    same_records(on, o_alns)
    oo = qmo_py.default_opt()
    oo.flags = _lib.F_NO_RESCUE
    oo.w = W.w
    ref = qmo_py.Ref(W.ref.codes, W.ref.lens, k=31)
    o = qmo_py.align_se(ref, codes, lens, opt=oo)
    regs = o["regs"].reshape(-1, qmo_py.MAX_REGS)
    no = []
    for c, p0 in zip(sizes, (0, 1000, 2000)):
        sl = slice(2 * p0, 2 * (p0 + c))
        r, nr = np.ascontiguousarray(regs[sl]).copy(), np.ascontiguousarray(o["n_regs"][sl]).copy()
        no.append(qmo_py.pair_and_finish(ref, np.ascontiguousarray(codes[sl]), np.ascontiguousarray(lens[sl]), r, nr, o_models[len(no)], pair_id0=p0, opt=oo))
    no = np.concatenate(no)
    assert int(((on["flag"] & 4) == 0).sum()) > int(((no["flag"] & 4) == 0).sum())


def test_records_do_not_depend_on_batching(ctx):
    W = _workload("cfg1", 5000)
    codes, quals, _, _ = W.simulate_host(0, 5000)
    lens = np.full(10000, W.params.read_len, np.int32)
    sizes = plan(5000, np.random.default_rng(9))
    a, ma, ca = device_run(ctx, W, codes, quals, lens, [sizes])                                   # many chunks in one call
    b, mb, cb = device_run(ctx, W, codes, quals, lens, [[c] for c in sizes])                      # one chunk per call
    c, mc, cc = device_run(ctx, W, codes, quals, lens, [sizes[:3], sizes[3:9], sizes[9:]], entry="host")   # the host entry
    for x, m, cn in ((b, mb, cb), (c, mc, cc)):
        assert x.tobytes() == a.tobytes() and m.tobytes() == ma.tobytes() and np.array_equal(cn, ca)


def test_chunk_sizes_must_match_the_call(ctx):
    from quasimodo_b200.api import QmError
    W = _workload("cfg1", 100)
    idx = ctx.index(W.ref, 31)
    s = ctx.sample(idx)
    codes, quals, _, _ = W.simulate_host(0, 100)
    lens = np.full(200, W.params.read_len, np.int32)
    s.set_chunks([60, 30])
    with pytest.raises(QmError, match="add up to 90"):
        s.add_pairs_host(codes, quals, lens)
    with pytest.raises(QmError) as e:
        s.set_chunks([(1 << 21) + 1])
    assert "2097152" in str(e.value)
    s.set_chunks([100])
    s.add_pairs_host(codes, quals, lens)
    assert s.chunk_pestat().shape == (1, 4)
    s.close()
    idx.close()


def test_single_chunk_model_comes_from_every_pair(ctx):
    """K above the sample: one chunk, whose model is mem_pestat over all of its pairs -- not the default path's first
    QM_PESTAT_PAIRS pairs"""
    import torch
    from quasimodo_b200 import _lib
    n = 70000
    W = _workload("cfg1", n)
    codes, quals, _, _ = W.simulate_host(0, n)
    lens = np.full(2 * n, W.params.read_len, np.int32)
    _, models, _ = device_run(ctx, W, codes, quals, lens, [[n]], entry="host")
    opt = _lib.default_opt()
    opt.w = W.w
    idx = ctx.index(W.ref, 31)
    dev = torch.device("cuda:0")
    d_regs, d_nr = ctx.align_se(idx, torch.from_numpy(codes).to(dev), torch.from_numpy(lens).to(dev), opt=opt)
    whole = ctx.pestat(idx, d_regs, d_nr, n, opt=opt)
    prefix = ctx.pestat(idx, d_regs, d_nr, _lib.PESTAT_PAIRS, opt=opt)
    idx.close()
    assert models.shape == (1, 4) and models[0].tobytes() == whole.tobytes()
    assert whole.tobytes() != prefix.tobytes()


@pytest.mark.parametrize("chunked", [False, True])
def test_given_model_replaces_chunk_models(ctx, chunked):
    """-I: qm_sample_set_pestat with bwa's FR-only model gives the same records with and without chunks, and they are the oracle's
    pair_and_finish with that model"""
    from oracle import qmo_py
    from quasimodo_b200 import _lib
    W = _workload("cfg1", 2000)
    codes, quals, _, _ = W.simulate_host(0, 2000)
    lens = np.full(4000, W.params.read_len, np.int32)
    pes = np.zeros(4, dtype=_lib.PESTAT_DTYPE)
    pes["failed"] = 1
    pes[1] = (250, 420, 0, 0, 330.0, 20.0)       # low, high, failed, pad, avg, std: -I 330,20,420,250
    g, models, _ = device_run(ctx, W, codes, quals, lens, [[700, 800, 500]] if chunked else None, pes=pes)
    if chunked:
        assert models.size == 0
    opt = qmo_py.default_opt()
    opt.w = W.w
    ref = qmo_py.Ref(W.ref.codes, W.ref.lens, k=31)
    o = qmo_py.align_se(ref, codes, lens, opt=opt)
    o_alns = qmo_py.pair_and_finish(ref, codes, lens, o["regs"], o["n_regs"], pes.view(qmo_py.PESTAT_DTYPE), opt=opt)
    same_records(g, o_alns)


# ---- the driver ----

def _fastq(d, name, n, seed=5):
    from quasimodo_b200 import workloads
    W = workloads.config1(n) if name == "cfg1" else workloads.config2(6, n)
    codes, quals, _, _ = W.simulate_host(0, n)
    lens = np.full(2 * n, W.params.read_len, np.int32)
    r1, r2 = d / f"{name}.r1.fq", d / f"{name}.r2.fq"
    drvutil.write_fastq(codes, quals, lens, drvutil.pair_names("p", n), r1, r2)
    fa = d / f"{name}.fa"
    drvutil.write_fasta(W.ref, fa)
    return fa, r1, r2


def _outputs(d):
    return ["--bam", d / "s.bam", "--counts", d / "s.tsv", "--vcf", d / "s.vcf", "--vcf-gz", 0, "--mpileup", d / "s.txt",
            "--rmdup", 1, "--rmdup-bam", d / "s.rmdup.bam", "--metrics", d / "s.metrics"]


def _records(path):
    from tests import bamio
    return [(r["rid"], r["pos"], r["mapq"], r["flag"], tuple(r["cigar"]), r["mrid"], r["mpos"], r["tlen"], r["name"])
            for r in bamio.Bam(str(path)).records]


def _same_outputs(a, b):
    for f in ("s.tsv", "s.vcf", "s.txt", "s.metrics"):
        assert (a / f).read_bytes() == (b / f).read_bytes(), f
    for f in ("s.bam", "s.rmdup.bam"):
        assert _records(a / f) == _records(b / f), f


def _gpu_count():
    import torch
    return torch.cuda.device_count()


def test_driver_k_independent_of_batch_size_and_gpus(tmp_path):
    fa, r1, r2 = _fastq(tmp_path, "cfg2", 90000)
    runs = {}
    for tag, extra in (("b", ["--batch-pairs", 70000]), ("c", ["--batch-pairs", 200000])) + ((("g2", ["--gpus", "0,1"]),) if _gpu_count() >= 2 else ()):
        d = tmp_path / tag
        d.mkdir()
        drvutil.run_driver(["sample", "--ref", fa, "--r1", r1, "--r2", r2, "-K", 3000000] + _outputs(d) + extra)
        runs[tag] = d
    for tag in runs:
        _same_outputs(runs["b"], runs[tag])


def test_driver_dash_i_same_with_and_without_k(tmp_path):
    fa, r1, r2 = _fastq(tmp_path, "cfg1", 20000)
    runs = []
    for tag, extra in (("i", []), ("ik", ["-K", 500000])):
        d = tmp_path / tag
        d.mkdir()
        drvutil.run_driver(["sample", "--ref", fa, "--r1", r1, "--r2", r2, "-I", "330,25"] + _outputs(d) + extra)
        runs.append(d)
    _same_outputs(runs[0], runs[1])


@pytest.mark.skipif("not __import__('torch').cuda.device_count() >= 2")
def test_driver_k_two_gpus_small_batches(tmp_path):
    """whole chunks dealt to two GPUs, each GPU many chunks per batch: the one-GPU outputs"""
    fa, r1, r2 = _fastq(tmp_path, "cfg1", 150000)
    runs = []
    for tag, extra in (("one", ["--gpu", 0]), ("two", ["--gpus", "0,1", "--batch-pairs", 65536])):
        d = tmp_path / tag
        d.mkdir()
        drvutil.run_driver(["sample", "--ref", fa, "--r1", r1, "--r2", r2, "-K", 1000000] + _outputs(d) + extra)
        runs.append(d)
    _same_outputs(runs[0], runs[1])


def test_many_chunks_histogram_groups(ctx):
    """2,000 chunks of 10 pairs in one add call at max_ins = 2^20: 16 MB of histogram per chunk, so the models are estimated 16
    chunks at a time (125 groups); every model and record still equals the oracle chunk by chunk"""
    from oracle import qmo_py
    from quasimodo_b200 import _lib
    n = 20000
    W = _workload("cfg1", n)
    codes, quals, _, _ = W.simulate_host(0, n)
    lens = np.full(2 * n, W.params.read_len, np.int32)
    sizes = [10] * (n // 10)
    opt_o = qmo_py.default_opt()
    opt_o.w, opt_o.max_ins = W.w, 1 << 20
    ref = qmo_py.Ref(W.ref.codes, W.ref.lens, k=31)
    o = qmo_py.align_se(ref, codes, lens, opt=opt_o)
    regs = o["regs"].reshape(-1, qmo_py.MAX_REGS)
    o_models, o_alns = [], []
    for c in range(len(sizes)):
        sl = slice(20 * c, 20 * (c + 1))
        r, nr = np.ascontiguousarray(regs[sl]).copy(), np.ascontiguousarray(o["n_regs"][sl]).copy()
        pes = qmo_py.pestat(ref, r, nr, opt=opt_o)
        o_models.append(pes)
        o_alns.append(qmo_py.pair_and_finish(ref, np.ascontiguousarray(codes[sl]), np.ascontiguousarray(lens[sl]), r, nr, pes, pair_id0=10 * c, opt=opt_o))
    o_models, o_alns = np.stack(o_models), np.concatenate(o_alns)
    opt = _lib.default_opt()
    opt.w, opt.max_ins = W.w, 1 << 20
    idx = ctx.index(W.ref, 31)
    s = ctx.sample(idx, opt=opt)
    s.set_chunks(sizes)
    h = np.zeros(2 * n, dtype=_lib.ALN_DTYPE)
    s.add_pairs_host(codes, quals, lens, h_alns=h)
    models = s.chunk_pestat()
    s.close()
    idx.close()
    assert models.shape == (len(sizes), 4) and models.tobytes() == o_models.tobytes()
    assert (~o_models["failed"].astype(bool)).any()                 # some 10-pair chunks do have a model
    same_records(h, o_alns)


def test_call_larger_than_one_internal_chunk(ctx):
    """22 chunks of 100,000 pairs in one call: the call is cut into internal chunks of at most 2^21 pairs at a chunk end (20 + 2
    chunks); the records equal those of one chunk per call"""
    n, c = 2_200_000, 100_000
    W = _workload("cfg1", n)
    codes, quals, _, _ = W.simulate_host(0, n)
    lens = np.full(2 * n, W.params.read_len, np.int32)
    sizes = [c] * (n // c)
    a, ma, ca = device_run(ctx, W, codes, quals, lens, [sizes], entry="host")
    b, mb, cb = device_run(ctx, W, codes, quals, lens, [[x] for x in sizes], entry="host")
    assert a.tobytes() == b.tobytes() and ma.tobytes() == mb.tobytes() and np.array_equal(ca, cb)


def test_decontam_sample_k_equals_the_chain(tmp_path):
    """`sample --decontam A --decontam2 B -K` = `decontam -K` | `decontam -K` | `sample -K`: each stage cuts chunks over its own
    input (pass 2 over pass 1's survivors, the target over pass 2's), across raw batches that end elsewhere"""
    from quasimodo_b200 import genomes
    from tests.test_decontam_sample_gpu import run_chain, run_fused, same_fastq, same_outputs, simulate
    refs = {}
    for stem in ("Merlin", "Phix", "Ecoli"):
        refs[stem] = str(tmp_path / f"{stem}.fa")
        drvutil.write_fasta(genomes.load(stem), refs[stem])
    r1, r2 = simulate(tmp_path, 150_000, {"AD169": 10, "Merlin": 70, "Phix": 8, "Ecoli": 12}, 21)
    passes = [refs["Phix"], refs["Ecoli"]]
    common = ["-K", 3_000_000, "--batch-pairs", 65536, "-t", 4]
    c = run_chain(tmp_path / "chain", refs, passes, r1, r2, [], rmdup=True, common=common)
    *f, log = run_fused(tmp_path / "fused", refs, passes, r1, r2, [], rmdup=True, common=common)
    same_fastq(c, f)
    assert same_outputs(tmp_path / "chain", tmp_path / "fused", rmdup=True) > 100_000
    n2 = sum(1 for _ in open(f[0])) // 4
    assert f"pass 2: {n2} of" in log and n2 < 150_000
