"""CPU checks of the genome diff's restatement (tests/gdiff_oracle.py, DESIGN.md 5c) on pairs with planted differences
(tests/gdiffgen.py): the rows are exactly the planted differences after left-alignment, BUFF and DIST follow from the planted
list, the options -I and -C act as documented, and the custom evaluator reads the -I rows."""
import numpy as np
import pytest

from quasimodo_b200 import _lib, evaluate
from tests import gdiff_oracle as G
from tests import gdiffgen as GG


@pytest.fixture(scope="module")
def planted():
    R, Q, want = GG.planted_pair()
    rows, alns = G.genome_diff(R, Q)
    return R, Q, want, rows, alns


def test_planted_pair_rows_are_the_planted_differences(planted):
    R, Q, want, rows, alns = planted
    assert GG.key(rows) == GG.key(want)
    kinds = {("snp" if "." not in (w["sub_r"], w["sub_q"]) else "del" if w["sub_q"] == "." else "ins") for w in want}
    assert kinds == {"snp", "del", "ins"}
    assert any(w["frm_q"] == -1 for w in want) and {w["qid"] for w in want} == {0, 1}
    # the divergent block, the 3 kb deletion, the inversion, the transposition and the duplication each break the alignment
    assert len(alns) == 10 and sum(a["strand"] == -1 for a in alns) == 1
    assert any(GG.DIVERGENT[0] - 20 < a["re"] <= GG.DIVERGENT[0] + 5 for a in alns)
    assert any(GG.DIVERGENT[1] - 5 < a["rs"] <= GG.DIVERGENT[1] + 20 for a in alns)
    assert not any(GG.DIVERGENT[0] + 5 < w["p1"] <= GG.DIVERGENT[1] - 5 for w in rows)
    # the ends are extended past the outermost anchors: the SNPs 10 and 9 bases from the contig ends are reported
    assert rows[0]["p1"] == 11 and rows[-1]["p1"] == R.lens[0] - 8
    assert alns[0]["rs"] == 1 and max(a["re"] for a in alns) == R.lens[0]


def test_planted_pair_buff_and_dist_follow_from_the_planted_list(planted):
    R, Q, want, rows, alns = planted
    for w in rows:
        dist = min(w["p1"] - 1, R.lens[0] - w["p1"], w["p2"] - 1, Q.lens[w["qid"]] - w["p2"])
        assert w["dist"] == dist
        a, = [a for a in alns if a["rs"] <= w["p1"] <= a["re"] and a["qid"] == w["qid"] and a["strand"] == w["frm_q"]]
        others = [v["p1"] for v in want if v is not w and v["qid"] == w["qid"] and v["frm_q"] == w["frm_q"] and a["rs"] <= v["p1"] <= a["re"]
                  and (v["p1"], v["p2"]) != (w["p1"], w["p2"])]
        buff = min([w["p1"] - a["rs"], a["re"] - w["p1"]] + [abs(w["p1"] - p) for p in others])
        assert w["buff"] == buff, w


def test_mutated_copy_rows_are_the_planted_differences():
    R = GG.base_ref()
    Q, want = GG.mutated_copy(R, n_snp=200, n_indel=60)
    rows, alns = G.genome_diff(R, Q)
    assert GG.key(rows) == GG.key(want) and len(alns) == 1


def test_no_indels_and_ambiguous_positions(planted):
    R, Q, want, rows, _ = planted
    o = G.default_opt()
    o["flags"] = _lib.GDIFF_NO_INDELS
    snp_rows, _ = G.genome_diff(R, Q, o)
    assert GG.key(snp_rows) == [k for k in GG.key(want) if "." not in k[1:3]]
    o["flags"] = _lib.GDIFF_KEEP_AMBIGUOUS
    amb, _ = G.genome_diff(R, Q, o)
    dup = [w for w in amb if 41000 < w["p1"] <= 43000]
    assert [w["p1"] for w in dup] == [42001, 42001]           # the SNP in both copies of the duplication, once per copy
    assert len(amb) == len(rows) + 2


def test_custom_evaluator_reads_rows_without_indels(planted, tmp_path):
    R, Q, want, _, _ = planted
    o = G.default_opt()
    o["flags"] = _lib.GDIFF_NO_INDELS
    rows, _ = G.genome_diff(R, Q, o)
    path = tmp_path / "pair.snps"
    path.write_text("".join(ln + "\n" for ln in G.snps_lines(rows, R, Q)))
    keys = evaluate.custom_truth_keys(str(path))
    assert len(keys) == len(rows)
    assert sorted(keys.tolist()) == sorted(evaluate.snp_key(str(w["p1"]), w["sub_r"], w["sub_q"]) for w in rows)


def test_vcf_records_merge_indel_runs_and_collapse_snps():
    from quasimodo_b200.genomes import Genome
    ref = Genome(["r"], [12], np.array([0, 1, 2, 3, 0, 1, 2, 3, 0, 1, 2, 3], np.uint8))
    qry = Genome(["q"], [12], np.zeros(12, np.uint8))
    row = lambda p1, sr, sq, p2: dict(p1=p1, sub_r=sr, sub_q=sq, p2=p2, rid=0, qid=0)
    rows = [row(2, "C", "A", 2), row(2, "C", "G", 5), row(4, "T", ".", 3), row(5, "A", ".", 3), row(8, ".", "G", 6), row(8, ".", "T", 7)]
    recs = [ln.split("\t")[:5] + [ln.split("ORIG=")[1]] for ln in G.vcf_records(rows, ref, qry)]
    assert recs == [["r", "2", ".", "C", "A,G", "q:2;TYPE=SNV"], ["r", "3", ".", "GTA", "G", "q:3;TYPE=INDEL"],
                    ["r", "8", ".", "T", "TGT", "q:6;TYPE=INDEL"]]


@pytest.mark.parametrize("ins, pieces", [(8, 1), (60, 1), (150, 2)])
def test_unrelated_insertion_between_anchors_ends_the_alignment_when_long(ins, pieces):
    """the divergence rule on one gap: an unrelated insertion of 150 bases between two anchors ends the alignment (poor-scoring
    stretch 150 columns + 156 to win back > -b 200); 8 and 60 bases are bridged"""
    rng = np.random.default_rng(ins)
    R = rng.integers(0, 4, 1000).astype(np.uint8)
    Q = np.concatenate([R[:400], rng.integers(0, 4, ins).astype(np.uint8), R[400:]])
    anc = [(0, 0, 0, 0, 0, 400), (0, 0, 0, 400 + ins, 400, 600)]
    got = G.split_divergent(anc, R, Q, G.default_opt())
    assert len(got) == pieces
    if pieces == 1:
        assert got[0][1] == [[G.OP_I] * ins]
