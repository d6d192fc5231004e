"""The genome diff on the B200 (qm_genome_diff_host, `qm_driver genome-diff`; DESIGN.md 5c): rows and alignments equal the CPU
restatement (tests/gdiff_oracle.py) row for row on the planted pairs and on the three bundled HCMV pairs; E. coli against a
mutated copy gives exactly the planted differences; the driver's files equal what the oracle's rows give; and the agreement with
the committed truth VCFs is the one DESIGN.md 5c records."""
import gzip
import os

import numpy as np
import pytest

from quasimodo_b200 import _lib, evaluate, genomes
from tests import gdiff_oracle as G
from tests import gdiffgen as GG

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from quasimodo_b200 import Context
    c = Context(0)
    yield c
    c.close()


def gpu_diff(ctx, ref, qry, opt=None):
    o = _lib.default_gdiff_opt()
    for f, v in (opt or {}).items():
        setattr(o, f, v)
    idx = ctx.index(ref, o.min_match)
    try:
        return ctx.genome_diff(idx, qry, o)
    finally:
        idx.close()


def assert_same(ctx, ref, qry, opt=None):
    rows, alns = gpu_diff(ctx, ref, qry, opt)
    o_rows, o_alns = G.genome_diff(ref, qry, opt)
    assert len(alns) == len(o_alns) and np.array_equal(alns, G.alns_array(o_alns))
    assert len(rows) == len(o_rows)
    want = G.rows_array(o_rows)
    bad = np.nonzero(rows != want)[0]
    assert len(bad) == 0, (rows[bad[:5]], want[bad[:5]])
    return rows, alns


@pytest.mark.parametrize("opt", [None, {"flags": _lib.GDIFF_NO_INDELS}, {"flags": _lib.GDIFF_KEEP_AMBIGUOUS},
                                 {"min_match": 16, "max_gap": 60, "break_len": 400, "diag_factor": 0.2, "min_cluster": 40},
                                 {"min_match": 31, "mismatch": 3, "gap_open": 5, "gap_extend": 2}])
def test_planted_pair_equals_oracle(ctx, opt):
    R, Q, want = GG.planted_pair()
    rows, _ = assert_same(ctx, R, Q, opt)
    if opt is None:
        assert GG.key(rows) == GG.key(want)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_more_planted_pairs_equal_oracle(ctx, seed):
    R, Q, want = GG.planted_pair(seed)
    rows, _ = assert_same(ctx, R, Q)
    assert GG.key(rows) == GG.key(want)
    Q2, want2 = GG.mutated_copy(R, seed=seed, n_snp=150, n_indel=80)
    rows, _ = assert_same(ctx, R, Q2)
    assert GG.key(rows) == GG.key(want2)


@pytest.mark.parametrize("ref, qry", [("Merlin", "TB40E"), ("AD169", "TB40E"), ("Merlin", "AD169")])
def test_hcmv_pairs_equal_oracle(ctx, ref, qry):
    assert_same(ctx, genomes.load(ref), genomes.load(qry))


def test_ecoli_against_mutated_copy_gives_the_planted_differences(ctx):
    e = genomes.load("Ecoli")
    Q, want = GG.mutated_copy(e)
    rows, alns = gpu_diff(ctx, e, Q)
    assert GG.key(rows) == GG.key(want)
    assert len(alns) >= 1 and (alns["strand"] == 1).all()


def _truth_snp_keys(mix):
    keys = set()
    for ln in gzip.open(os.path.join(os.path.dirname(genomes.DATA), "truth", f"{mix}.maskrepeat.variants.vcf.gz"), "rt"):
        if ln.startswith("#") or not ln.strip():
            continue
        f = ln.split("\t")
        if len(f[3]) == 1 and len(f[4]) == 1:
            keys.add((int(f[1]), f[3], f[4]))
    return keys


# single-base SNP keys (POS, REF, ALT) against the committed truth VCFs (projected from the reference's MAFFT alignment):
# (ours, committed, in both) -- measured with tests/gdiff_oracle.py, DESIGN.md 5c
TRUTH_AGREEMENT = {"TM": ("Merlin", 3166, 2551, 2384), "TA": ("AD169", 2931, 2612, 2225)}


@pytest.mark.parametrize("mix", ["TM", "TA"])
def test_agreement_with_committed_truth(ctx, mix):
    ref, n_ours, n_truth, n_both = TRUTH_AGREEMENT[mix]
    rows, _ = gpu_diff(ctx, genomes.load(ref), genomes.load("TB40E"))
    ours = {(int(w["p1"]), w["sub_r"].decode(), w["sub_q"].decode()) for w in rows if b"." not in (w["sub_r"], w["sub_q"])}
    truth = _truth_snp_keys(mix)
    assert (len(ours), len(truth), len(ours & truth)) == (n_ours, n_truth, n_both)


def test_driver_files_equal_the_oracle_rows(tmp_path):
    from quasimodo_b200 import rules
    from tests import bamio, drvutil
    R, Q, _ = GG.planted_pair()
    ref_fa, qry_fa = str(tmp_path / "ref.fa"), str(tmp_path / "qry.fa")
    drvutil.write_fasta(R, ref_fa)
    drvutil.write_fasta(Q, qry_fa, width=61)
    dirs = {"snp_dir": str(tmp_path / "snp")}
    snps = str(tmp_path / "pair.snps")
    argv, paths = rules.genome_diff_command(drvutil.driver_path(), dirs, "TM", ref_fa, qry_fa, snps=snps)
    drvutil.run_driver(argv[1:])
    for p in paths:
        assert os.path.getsize(p) > 0, p
    rows, _ = G.genome_diff(R, Q)
    assert open(snps).read() == "".join(ln + "\n" for ln in G.snps_lines(rows, R, Q))
    vcf = paths[0]
    text = open(vcf).read()
    body = [ln for ln in text.split("\n") if ln and not ln.startswith("#")]
    assert body == G.vcf_records(rows, R, Q)
    header = [ln for ln in text.split("\n") if ln.startswith("##")]
    assert header[:3] == ["##fileformat=VCFv4.2", "##source=mummer2vcf.py", f"##reference={ref_fa}"]
    assert header[3] == f"##contig=<ID={R.names[0]},length={R.lens[0]}>"
    assert gzip.open(vcf + ".gz", "rb").read() == open(vcf, "rb").read()
    tbi = bamio.read_tbi(vcf + ".gz.tbi")
    bg = bamio.BgzfText(vcf + ".gz")
    recs = [ln.encode() for ln in body]
    assert tbi["names"] == [R.names[0]]
    assert bamio.tabix_query(tbi, bg, R.names[0], 0, 1 << 29) == recs
    lo, hi = int(recs[5].split(b"\t")[1]) - 1, int(recs[9].split(b"\t")[1])
    assert bamio.tabix_query(tbi, bg, R.names[0], lo, hi) == recs[5:10]
    # --indels 0: the rows of show-snps -CTHIlr, which the custom evaluator reads
    drvutil.run_driver(["genome-diff", "--ref", ref_fa, "--qry", qry_fa, "--snps", str(tmp_path / "i.snps"), "--indels", "0"])
    o = G.default_opt()
    o["flags"] = _lib.GDIFF_NO_INDELS
    rows_i, _ = G.genome_diff(R, Q, o)
    assert open(tmp_path / "i.snps").read() == "".join(ln + "\n" for ln in G.snps_lines(rows_i, R, Q))


def test_custom_evaluator_scores_calls_against_rows_without_indels(ctx, tmp_path):
    R, Q, _ = GG.planted_pair()
    rows, _ = gpu_diff(ctx, R, Q, {"flags": _lib.GDIFF_NO_INDELS})
    rows = [dict(zip(rows.dtype.names, (v.decode() if isinstance(v, bytes) else int(v) for v in w))) for w in rows]
    snps = tmp_path / "truth.snps"
    snps.write_text("".join(ln + "\n" for ln in G.snps_lines(rows, R, Q)))
    head = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS\n"
    calls = [f"{R.names[0]}\t{w['p1']}\t.\t{w['sub_r']}\t{w['sub_q']}\t50\tPASS\tDP=40\tGT\t1" for w in rows[:30]]
    calls.append(f"{R.names[0]}\t5\t.\tA\tC\t50\tPASS\tDP=40\tGT\t1")
    vcf = tmp_path / "TM-1-1.caller.vcf"
    vcf.write_text(head + "".join(c + "\n" for c in calls))
    n, tp, fp = evaluate.extract_tp_fp_custom_snp(ctx, str(vcf), str(snps), str(tmp_path / "out"), "caller")
    assert (n, tp, fp) == (31, 30, 1)
