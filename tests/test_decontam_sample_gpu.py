"""GPU tests of `qm_driver sample --decontam` (rules rm_phix + rm_human_ecoli + bwa + rmdup + mpileup + bcftools in one job): every
output equals the three-job chain `decontam` | `decontam` | `sample` on the cleaned FASTQ -- BAM records and header (the @PG command
line aside), what the .bai finds, count TSV, VCF (+ .gz), text pileup, metrics and the cleaned FASTQ -- and the library's filter mode
gives the keep rule of the records `qm_sample_add_pairs_host` returns."""
import gzip

import numpy as np
import pytest

from tests import bamio, drvutil

pytestmark = pytest.mark.gpu

def out_opts(d, rmdup=False):
    o = ["--bam", d / "s.bam", "--counts", d / "s.tsv", "--vcf", d / "s.vcf", "--mpileup", d / "s.txt"]
    if rmdup:
        o += ["--rmdup", 1, "--rmdup-bam", d / "s.rmdup.bam", "--metrics", d / "s.metrics"]
    return o


@pytest.fixture(scope="module")
def refs(tmp_path_factory):
    from quasimodo_b200 import genomes
    d = tmp_path_factory.mktemp("dcref")
    out = {}
    for stem in ("Merlin", "Phix", "Ecoli"):
        out[stem] = str(d / f"{stem}.fa")
        drvutil.write_fasta(genomes.load(stem), out[stem])
    return out


def simulate(d, n, weights, seed, tag="raw"):
    """n pairs of Merlin / AD169 / PhiX / E. coli reads in the given read shares, as FASTQ"""
    from quasimodo_b200 import workloads
    stems = [s for s in ("AD169", "Merlin", "Phix", "Ecoli") if weights.get(s)]
    W = workloads.Workload("dc", [(s, 1) for s in stems], ["Merlin"], n, seed, extra_weights=[weights[s] for s in stems])
    codes, quals, _, _ = W.simulate_host(0, n)
    lens = np.full(2 * n, 150, np.int32)
    r1, r2 = str(d / f"{tag}.r1.fq"), str(d / f"{tag}.r2.fq")
    drvutil.write_fastq(codes, quals, lens, drvutil.pair_names(f"{tag}.p", n), r1, r2)
    return r1, r2


def run_chain(d, refs, passes, r1, r2, opts, rmdup=False, common=()):
    """decontam per pass (with the options every job takes: `common`), then sample on the last cleaned FASTQ; outputs under d"""
    d.mkdir()
    for k, fa in enumerate(passes):
        o1, o2 = d / f"c{k + 1}.r1.fq", d / f"c{k + 1}.r2.fq"
        drvutil.run_driver(["decontam", "--ref", fa, "--r1", r1, "--r2", r2, "--out-r1", o1, "--out-r2", o2] + list(common))
        r1, r2 = o1, o2
    drvutil.run_driver(["sample", "--ref", refs["Merlin"], "--r1", r1, "--r2", r2] + out_opts(d, rmdup) + opts + list(common))
    return r1, r2


def run_fused(d, refs, passes, r1, r2, opts, rmdup=False, common=()):
    d.mkdir()
    pa = ["--decontam", passes[0]] + (["--decontam2", passes[1]] if len(passes) > 1 else [])
    p = drvutil.run_driver(["sample", "--ref", refs["Merlin"], "--r1", r1, "--r2", r2] + pa + ["--clean-r1", d / "cl.r1.fq", "--clean-r2", d / "cl.r2.fq"]
                           + out_opts(d, rmdup) + opts + list(common))
    return d / "cl.r1.fq", d / "cl.r2.fq", p.stderr


def rec_key(r):
    return (r["rid"], r["pos"], r["mapq"], r["bin"], r["flag"], tuple(r["cigar"]), r["mrid"], r["mpos"], r["tlen"], r["name"], r["seq"],
            r["qual"].tobytes(), tuple(sorted(r["tags"].items())))


def bai_query(bam, bai, rid, beg, end):
    """records overlapping [beg, end) of contig rid, found the way samtools finds them: bins, linear index, coordinates"""
    bins, lin = bai[0][rid]
    min_off = lin[min(beg >> 14, len(lin) - 1)] if lin else 0
    by_start = {r["ustart"]: r for r in bam.records}
    starts = sorted(by_start)
    got = set()
    for b in bamio.reg2bins(beg, end):
        for v0, v1 in bins.get(b, []):
            if v1 <= min_off:
                continue
            u0, u1 = bam.voffset_to_u(max(v0, min_off)), bam.voffset_to_u(v1)
            for u in starts[np.searchsorted(starts, u0):np.searchsorted(starts, u1)]:
                r = by_start[u]
                span = sum(x >> 4 for x in r["cigar"] if (x & 15) in (0, 2, 3, 7, 8)) if not r["flag"] & 4 else 0
                if r["rid"] == rid and r["pos"] < end and r["pos"] + max(span, 1) > beg:
                    got.add(u)
    return [rec_key(by_start[u]) for u in sorted(got)]


def no_pg(text):
    return [ln for ln in text.split("\n") if not ln.startswith("@PG")]


def same_bam(a, b):
    A, B = bamio.Bam(str(a)), bamio.Bam(str(b))
    assert no_pg(A.text) == no_pg(B.text) and A.refs == B.refs
    assert [rec_key(r) for r in A.records] == [rec_key(r) for r in B.records]
    ia, ib = bamio.read_bai(str(a) + ".bai"), bamio.read_bai(str(b) + ".bai")
    assert ia[1] == ib[1]
    rng = np.random.default_rng(3)
    for rid, (_, ln) in enumerate(A.refs):
        wins = [(0, ln)] + [(int(x), int(x) + int(w)) for x, w in zip(rng.integers(0, ln, 6), rng.integers(1, 40000, 6))]
        for beg, end in wins:
            assert bai_query(A, ia, rid, beg, end) == bai_query(B, ib, rid, beg, end), (rid, beg, end)
    return len(A.records)


def same_outputs(a, b, rmdup=False):
    n = same_bam(a / "s.bam", b / "s.bam")
    for f in ("s.tsv", "s.vcf", "s.txt") + (("s.metrics",) if rmdup else ()):
        assert (a / f).read_bytes() == (b / f).read_bytes(), f
    assert gzip.open(a / "s.vcf.gz").read() == gzip.open(b / "s.vcf.gz").read()
    if rmdup:
        same_bam(a / "s.rmdup.bam", b / "s.rmdup.bam")
    return n


def same_fastq(a, b):
    for x, y in zip(a, b):
        assert open(x, "rb").read() == open(y, "rb").read()


@pytest.fixture(scope="module")
def mixture(tmp_path_factory, refs):
    d = tmp_path_factory.mktemp("dcmix")
    r1, r2 = simulate(d, 20_000, {"AD169": 10, "Merlin": 70, "Phix": 8, "Ecoli": 12}, 11)
    return d, r1, r2


def test_one_pass_with_rmdup_and_depth_cap(mixture, refs):
    d, r1, r2 = mixture
    opts, common = ["--max-depth", 50, "--min-dp", 3, "--min-alt", 2], ["-t", 4]
    c = run_chain(d / "chain1", refs, [refs["Phix"]], r1, r2, opts, rmdup=True, common=common)
    *f, log = run_fused(d / "fused1", refs, [refs["Phix"]], r1, r2, opts, rmdup=True, common=common)
    same_fastq(c, f)
    assert same_outputs(d / "chain1", d / "fused1", rmdup=True) > 20_000
    kept = sum(1 for _ in open(f[0])) // 4
    assert f"decontam pass 1: {kept} of 20000 pairs kept" in log and 15_000 < kept < 20_000


def test_two_passes(mixture, refs):
    d, r1, r2 = mixture
    passes = [refs["Phix"], refs["Ecoli"]]
    c = run_chain(d / "chain2", refs, passes, r1, r2, [], common=["-t", 4, "-B", 5])
    *f, log = run_fused(d / "fused2", refs, passes, r1, r2, [], common=["-t", 4, "-B", 5])
    same_fastq(c, f)
    same_outputs(d / "chain2", d / "fused2")
    n1 = sum(1 for _ in open(d / "chain2" / "c1.r1.fq")) // 4
    n2 = sum(1 for _ in open(f[0])) // 4
    assert f"decontam pass 1: {n1} of 20000 pairs kept" in log and f"decontam pass 2: {n2} of {n1} pairs kept" in log
    assert n2 < n1 < 20_000


def test_first_batches_carry_over(tmp_path, refs):
    """--batch-pairs 65536 with contaminants: the first raw batch keeps fewer than 65,536 pairs, so pass 2 fixes its insert-size model
    only from the survivors of two raw batches, as from its first FASTQ batch in the chain (fixed too early, the records differ)"""
    r1, r2 = simulate(tmp_path, 150_000, {"Merlin": 80, "Phix": 10, "Ecoli": 10}, 12)
    passes = [refs["Phix"], refs["Ecoli"]]
    common = ["--batch-pairs", 65536, "-t", 4]
    c = run_chain(tmp_path / "chain", refs, passes, r1, r2, ["--max-depth", 100], common=common)
    *f, log = run_fused(tmp_path / "fused", refs, passes, r1, r2, ["--max-depth", 100], common=common)
    assert "the first batch of pass 2" in log and "carries over the pairs of 2 raw batches" in log
    same_fastq(c, f)
    same_outputs(tmp_path / "chain", tmp_path / "fused")


def test_clean_sample_equals_plain_sample(tmp_path, refs):
    r1, r2 = simulate(tmp_path, 8000, {"AD169": 20, "Merlin": 80}, 13)
    (tmp_path / "plain").mkdir()
    drvutil.run_driver(["sample", "--ref", refs["Merlin"], "--r1", r1, "--r2", r2] + out_opts(tmp_path / "plain"))
    *f, log = run_fused(tmp_path / "fused", refs, [refs["Phix"]], r1, r2, [])
    assert "decontam pass 1: 8000 of 8000 pairs kept" in log
    same_outputs(tmp_path / "plain", tmp_path / "fused")


def test_fully_contaminated_sample(tmp_path, refs):
    r1, r2 = simulate(tmp_path, 3000, {"Phix": 1}, 14)
    e1, e2 = tmp_path / "e1.fq", tmp_path / "e2.fq"
    e1.write_text("")
    e2.write_text("")
    (tmp_path / "empty").mkdir()
    drvutil.run_driver(["sample", "--ref", refs["Merlin"], "--r1", e1, "--r2", e2] + out_opts(tmp_path / "empty"))
    *f, log = run_fused(tmp_path / "fused", refs, [refs["Phix"]], r1, r2, [])
    assert "decontam pass 1: 0 of 3000 pairs kept" in log
    assert open(f[0]).read() == "" and open(f[1]).read() == ""
    assert same_outputs(tmp_path / "empty", tmp_path / "fused") == 0


def test_two_gpus_equal_one(tmp_path, refs):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    r1, r2 = simulate(tmp_path, 300_000, {"AD169": 10, "Merlin": 80, "Phix": 4, "Ecoli": 6}, 15)
    passes = [refs["Phix"], refs["Ecoli"]]
    opts = ["--batch-pairs", 65536, "--max-depth", 200]
    f1 = run_fused(tmp_path / "one", refs, passes, r1, r2, opts + ["--gpu", 0], rmdup=True)
    f2 = run_fused(tmp_path / "two", refs, passes, r1, r2, opts + ["--gpus", "0,1"], rmdup=True)
    assert "count tensors of 2 GPUs merged" in f2[2]
    same_fastq(f1[:2], f2[:2])
    same_outputs(tmp_path / "one", tmp_path / "two", rmdup=True)


def test_filter_mode_keep_bytes_equal_the_rule_on_the_records():
    from quasimodo_b200 import Context, QmError, _lib, genomes, workloads
    ctx = Context(0)
    W = workloads.Workload("f", [("Merlin", 1), ("Phix", 1)], ["Merlin"], 6000, 16, extra_weights=[80, 20])
    codes, quals, _, _ = W.simulate_host(0, 6000)
    lens = np.full(2 * 6000, 150, np.int32)
    lens[7], lens[100] = 20, 0
    idx = ctx.index(genomes.load("Phix"), 31)
    f, ref = ctx.sample(idx), ctx.sample(idx)
    f.set_filter(True)
    with pytest.raises(QmError):
        ref.keep(0)                                          # not in filter mode
    for p0, p1 in ((0, 4000), (4000, 6000)):               # the second batch runs with the first batch's model
        a = np.zeros(2 * (p1 - p0), dtype=_lib.ALN_DTYPE)
        ref.add_pairs_host(codes[2 * p0:2 * p1], quals[2 * p0:2 * p1], lens[2 * p0:2 * p1], pair_id0=p0, h_alns=a)
        f.add_pairs_host(codes[2 * p0:2 * p1], quals[2 * p0:2 * p1], lens[2 * p0:2 * p1], pair_id0=p0)
        fl = a["flag"].reshape(-1, 2)
        want = (((fl & 12) == 12) & ((fl & 256) == 0)).all(1).astype(np.uint8)
        assert 0 < want.sum() < p1 - p0
        assert np.array_equal(f.keep(p1 - p0), want)
        with pytest.raises(QmError):
            f.keep(p1 - p0 + 1)                              # not the last batch's size
    assert not f.counts_host().any() and ref.counts_host().any()
    f.close()
    ref.close()
    idx.close()
    ctx.close()
