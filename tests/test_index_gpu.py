"""GPU tests of the device-built FM-index and of `qm_driver index` (rule build_idx: `bwa index` + `samtools faidx`):
- the .bwt / .sa the command writes equal bwa's own files of the bundled genomes (tests/golden/fm_digests.json; E. coli: .sa);
- the .pac unpacks to the genome bwa packed (tests/golden/pac_digests.json), the .ann / .amb / .fai agree with a Python
  restatement of bwa's and samtools' formats;
- qm_index_build_fm equals the oracle's bytes (oracle/qmo_fm.c) on genomes that keep the prefix doubling busy for many rounds
  or end a suffix inside a tie;
- `sample --bwa-index` on the written files gives the records, count TSV and VCF of `sample --fm-seeds 1`."""
import hashlib
import json
import os

import numpy as np
import pytest

from quasimodo_b200 import genomes
from tests import bamio, drvutil

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
FM = json.load(open(os.path.join(HERE, "golden", "fm_digests.json")))
PAC = json.load(open(os.path.join(HERE, "golden", "pac_digests.json")))


@pytest.fixture(scope="module")
def ctx():
    from quasimodo_b200 import Context
    c = Context(0)
    yield c
    c.close()


def unpack_pac(pac):
    """bwa's .pac: base i in byte i >> 2 at shift ((~i) & 3) << 1; the last byte is l_pac % 4, with a zero byte before it when
    l_pac % 4 == 0"""
    pac = np.frombuffer(pac, np.uint8)
    rem = int(pac[-1])
    body = pac[:-1] if rem else pac[:-2]
    if not rem:
        assert pac[-2] == 0
    l_pac = 4 * len(body) - ((4 - rem) % 4 if rem else 0)
    i = np.arange(l_pac, dtype=np.int64)
    return ((body[i >> 2] >> (((~i) & 3) << 1)) & 3).astype(np.uint8)


def ann_amb_restated(G, annos):
    ann = f"{G.total} {len(G.names)} 11\n"
    off = 0
    for name, anno, ln in zip(G.names, annos, G.lens):
        ann += f"0 {name} {anno or '(null)'}\n{off} {ln} 0\n"
        off += ln
    return ann, f"{G.total} {len(G.names)} 0\n"


def fai_restated(text):
    """samtools faidx's columns from the FASTA text: name, length, offset of the first base, bases and bytes per line"""
    rows, pos = [], 0
    for line in text.splitlines(keepends=True):
        body = line.rstrip("\r\n")
        if body.startswith(">"):
            rows.append([body[1:].split()[0], 0, pos + len(line), 0, 0])
        elif body:
            r = rows[-1]
            if r[3] == 0:
                r[3], r[4] = len(body), len(line) if line.endswith("\n") else len(body) + 1
            r[1] += len(body)
        pos += len(line)
    return "".join("\t".join(map(str, r)) + "\n" for r in rows)


def digest(b):
    return hashlib.sha256(b).hexdigest()


@pytest.mark.parametrize("stem", ["Merlin", "TB40E", "AD169", "Phix", "Ecoli"])
def test_driver_writes_bwas_index_files(tmp_path, stem):
    G = genomes.load(stem)
    fa = str(tmp_path / f"{stem}.fa")
    drvutil.write_fasta(G, fa)                              # headers ">name test contig", 70 bases a line
    drvutil.run_driver(["index", "--ref", fa])
    rd = lambda ext: open(fa + ext, "rb").read()          # noqa: E731
    for kind in ("bwt", "sa"):
        if kind in FM[stem]:
            b = rd("." + kind)
            assert len(b) == FM[stem][kind]["bytes"] and digest(b) == FM[stem][kind]["sha256"], kind
    codes = unpack_pac(rd(".pac"))
    assert len(codes) == PAC[stem]["l_pac"] and digest(codes.tobytes()) == PAC[stem]["sha256_codes"]
    ann = rd(".ann").decode()
    lines = ann.split("\n")
    assert [lines[1 + 2 * c].split()[1] for c in range(len(G.names))] == PAC[stem]["names"]
    assert [int(lines[2 + 2 * c].split()[1]) for c in range(len(G.names))] == PAC[stem]["lens"]
    want_ann, want_amb = ann_amb_restated(G, ["test contig"] * len(G.names))
    assert ann == want_ann and rd(".amb").decode() == want_amb
    assert rd(".fai").decode() == fai_restated(open(fa).read())


def test_prefix_annotations_and_line_layouts(tmp_path):
    """--prefix, a header without annotation ((null)), CRLF lines, a short last line, a contig on one line without a newline"""
    rng = np.random.default_rng(4)
    seqs = ["".join("ACGT"[x] for x in rng.integers(0, 4, n)) for n in (130, 61, 1, 45)]
    text = (">a\r\n" + seqs[0][:60] + "\r\n" + seqs[0][60:120] + "\r\n" + seqs[0][120:] + "\r\n"
            + ">b  two  words\n" + "\n".join(seqs[1][i:i + 20] for i in range(0, 61, 20)) + "\n\n"
            + ">c\tx\n" + seqs[2] + "\n" + ">d\n" + seqs[3])
    fa = tmp_path / "g.fa"
    fa.write_bytes(text.encode())
    drvutil.run_driver(["index", "--ref", fa, "--prefix", tmp_path / "sub_idx"])
    G = genomes.Genome(["a", "b", "c", "d"], [130, 61, 1, 45], np.array(["ACGT".index(ch) for ch in "".join(seqs)], np.uint8))
    ann, amb = ann_amb_restated(G, ["", " two  words", "x", ""])
    assert (tmp_path / "sub_idx.ann").read_text() == ann and (tmp_path / "sub_idx.amb").read_text() == amb
    assert np.array_equal(unpack_pac((tmp_path / "sub_idx.pac").read_bytes()), G.codes)
    assert (tmp_path / "g.fa.fai").read_text() == fai_restated(text)
    assert not os.path.exists(str(fa) + ".bwt")
    from oracle import qmo_py
    fm = qmo_py.FmIndex(codes=G.codes)
    assert (tmp_path / "sub_idx.bwt").read_bytes() == fm.bwt_bytes() and (tmp_path / "sub_idx.sa").read_bytes() == fm.sa_bytes()


def _stress_genomes():
    rng = np.random.default_rng(17)
    x = rng.integers(0, 4, 1500).astype(np.uint8)
    out = {
        "homopolymer": [np.zeros(5000, np.uint8)],
        "period2": [np.tile(np.array([0, 1], np.uint8), 2500)],
        "period3": [np.tile(np.array([2, 0, 3], np.uint8), 1700)],
        "period7": [np.tile(np.array([0, 3, 1, 1, 2, 0, 3], np.uint8), 700)],
        "revcomp_palindrome": [np.concatenate([x, 3 - x[::-1]]).astype(np.uint8)],   # equals its own reverse complement
        "one_base": [np.array([2], np.uint8)],
        "one_base_among_others": [rng.integers(0, 4, 300).astype(np.uint8), np.array([1], np.uint8), np.zeros(40, np.uint8)],
        "sixteen_short": [rng.integers(0, 4, int(n)).astype(np.uint8) for n in rng.integers(1, 90, 16)],
        "random_2M": [rng.integers(0, 4, 2_000_000).astype(np.uint8)],
    }
    rep = rng.integers(0, 4, 700).astype(np.uint8)           # a long repeat in three copies, one of them reverse-complemented
    out["repeats"] = [np.concatenate([rng.integers(0, 4, 900), rep, rng.integers(0, 4, 50), 3 - rep[::-1], rep]).astype(np.uint8)]
    return out


STRESS = _stress_genomes()


@pytest.mark.parametrize("name", list(STRESS))
def test_build_fm_equals_oracle(ctx, name):
    from oracle import qmo_py
    parts = STRESS[name]
    codes = np.concatenate(parts).astype(np.uint8)
    G = genomes.Genome([f"c{i}" for i in range(len(parts))], [len(p) for p in parts], codes)
    idx = ctx.index(G, 31)
    idx.build_fm()
    b, s = idx.fm_export()
    fm = qmo_py.FmIndex(codes=codes)
    assert b == fm.bwt_bytes()
    assert s == fm.sa_bytes()
    idx.build_fm()                                          # a second build replaces the first
    assert idx.fm_export() == (b, s)
    idx.close()


def _records(path):
    bam = bamio.Bam(path)
    return bam.data[bam.records[0]["ustart"]:] if bam.records else b""


def test_sample_on_written_index_equals_fm_seeds(tmp_path):
    from quasimodo_b200 import workloads
    n = 3000
    W = workloads.config1(n)
    codes, quals, _, _ = W.simulate_host(0, n)
    lens = np.full(2 * n, 150, np.int32)
    fa, r1, r2 = str(tmp_path / "Merlin.fa"), str(tmp_path / "r1.fq"), str(tmp_path / "r2.fq")
    drvutil.write_fasta(W.ref, fa)
    drvutil.write_fastq(codes, quals, lens, drvutil.pair_names("i", n), r1, r2)
    drvutil.run_driver(["index", "--ref", fa])
    out = {}
    for how, extra in (("files", ["--bwa-index", fa]), ("rebuilt", ["--fm-seeds", "1"])):
        d = tmp_path / how
        d.mkdir()
        drvutil.run_driver(["sample", "--ref", fa, "--r1", r1, "--r2", r2, "--bam", d / "s.bam", "--counts", d / "s.tsv",
                            "--vcf", d / "s.vcf", "--vcf-gz", "0"] + extra)
        out[how] = (_records(str(d / "s.bam")), (d / "s.tsv").read_bytes(), (d / "s.vcf").read_bytes())
    assert len(out["files"][0]) > 0 and out["files"][1]
    assert out["files"][0] == out["rebuilt"][0]
    assert out["files"][1] == out["rebuilt"][1]
    assert out["files"][2] == out["rebuilt"][2]
