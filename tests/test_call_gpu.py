"""qm_call_snps (csrc/evalcall.cu) on hand-made channel-major count tensors against a float64 restatement of its rule:
every field of every call, on an index of four contigs whose l_pac (882) is not a multiple of the kernel's 128-column
blocks, at the columns where a threshold caller goes wrong (no counted base, f == 1, f around the error rate 0.002, AD
exactly min_af * total, QUAL around the 999 cap, several alts), and the max_calls overflow path."""
import ctypes as C
import math

import numpy as np
import pytest

from tests import recgen

pytestmark = pytest.mark.gpu

E = 0.002
QM_ELIMIT = -5


def expected(planes, ref_codes, offs, copt):
    """the caller's rule restated in float64: -> list of dict, in (position, alt) order"""
    min_af = float(np.float32(copt.min_af))
    out = []
    for p in range(planes.shape[1]):
        adf = planes[0:4, p].astype(np.int64)
        ad = adf + planes[6:10, p]
        tot, dp, r = int(ad.sum()), int(planes[14, p]), int(ref_codes[p])
        for b in range(4):
            if b == r or not (dp >= copt.min_dp and ad[b] >= copt.min_alt and tot > 0 and float(ad[b]) >= min_af * tot):
                continue
            f = float(ad[b]) / tot
            q = 0.0
            if f > E:
                kl = f * math.log(f / E) + ((1 - f) * math.log((1 - f) / (1 - E)) if f < 1 else 0.0)
                q = 10 / math.log(10) * tot * kl
            rid = int(np.searchsorted(offs, p, side="right") - 1)
            out.append(dict(rid=rid, pos=p - int(offs[rid]), ref=r, alt=b, dp=dp, ad_ref_f=int(adf[r]), ad_ref_r=int(ad[r] - adf[r]),
                            ad_alt_f=int(adf[b]), ad_alt_r=int(ad[b] - adf[b]), qual=np.float32(min(999.0, q)), af=np.float32(f)))
    return out


def qual_near(tot, below):
    """(ad, tot') with QUAL closest to 999 from below / above, searched over totals around `tot`"""
    best = None
    for t in range(tot - 20, tot + 20):
        for a in range(2, t + 1):
            f = a / t
            kl = f * math.log(f / E) + ((1 - f) * math.log((1 - f) / (1 - E)) if f < 1 else 0.0)
            q = 10 / math.log(10) * t * kl
            d = 999 - q if below else q - 999
            if d > 0 and (best is None or d < best[0]):
                best = (d, a, t)
    return best[1], best[2]


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
def idx(ctx, genome):
    i = ctx.index(genome, 31)
    yield i
    i.close()


@pytest.fixture(scope="module")
def planes(genome):
    """[16, l_pac] int32; column p gets one of the cases below, the rest random counts"""
    assert genome.l_pac % 128 != 0
    rng = np.random.default_rng(4)
    P = np.zeros((16, genome.l_pac), np.int32)
    ref = genome.codes
    cols = iter(range(genome.l_pac))

    def put(fwd, rev=(0, 0, 0, 0), dp=None, extra=True):
        """counts per base code relative to the column's reference base: index 0 = reference, 1..3 = the other bases"""
        p = next(cols)
        order = [int(ref[p])] + [b for b in range(4) if b != ref[p]]
        for k in range(4):
            P[order[k], p], P[6 + order[k], p] = fwd[k], rev[k]
        if extra:                                  # N and deleted bases are not part of the total
            P[4, p], P[10, p], P[5, p], P[11, p] = rng.integers(0, 3, 4)
        P[14, p] = dp if dp is not None else P[[0, 1, 2, 3, 4, 6, 7, 8, 9, 10], p].sum()
        return p

    put((0, 0, 0, 0), dp=50)                       # dp >= 10, nothing counted: tot == 0
    put((0, 0, 0, 0), dp=50, extra=False)
    put((0, 20, 0, 0), (0, 10, 0, 0))              # f == 1
    put((0, 3, 0, 0), (0, 0, 0, 0))                # f == 1 below min_dp
    for tot in (999, 1000, 1001, 500, 501, 499):   # f = 2 / tot around e = 0.002 (equal at 1000) and 1 / 500
        put((tot - 2, 1, 0, 0), (0, 1, 0, 0))
        put((tot - 1, 1, 0, 0), (0, 0, 0, 0))
    for a, t in ((5, 20), (5, 21), (4, 20), (2, 200), (2, 201), (3, 300), (3, 301), (1, 100)):  # AD == min_af * tot (0.25, 0.01f)
        put((t - a, a - a // 2, 0, 0), (0, a // 2, 0, 0))
    for below in (True, False):                    # QUAL just under / over the cap
        for t0 in (40, 120, 300):
            a, t = qual_near(t0, below)
            put((t - a, 0, a, 0), (0, 0, 0, 0))
    put((10, 5, 7, 9), (3, 5, 0, 2))               # three alts
    put((0, 5, 7, 0), (0, 5, 0, 0))                # two alts, no reference base
    put((1, 2, 2, 0), (0, 0, 0, 2))
    for p in cols:                                 # the rest: random columns, many with a call or two
        k = rng.integers(0, 4)
        sc = [1, 5, 40, 400][k]
        fwd, rev = rng.integers(0, sc + 1, 4), rng.integers(0, sc + 1, 4)
        P[0:4, p], P[6:10, p] = fwd, rev
        P[[0, 6], p] += 0 if rng.random() < 0.3 else 3 * sc
        P[14, p] = P[0:4, p].sum() + P[6:10, p].sum() + rng.integers(0, 5)
    # the last column of the last contig and the 1-base contig carry calls
    for p in (genome.l_pac - 1, int(genome.offs[1])):
        r = int(ref[p])
        P[:, p] = 0
        P[(r + 1) % 4, p], P[6 + (r + 2) % 4, p], P[r, p], P[14, p] = 12, 6, 20, 40
    return P


def call_opts():
    from quasimodo_b200 import _lib
    out = []
    for kw in (dict(), dict(min_af=0.25), dict(min_af=0.001), dict(min_dp=0, min_alt=0, min_af=0.0), dict(min_dp=11, min_alt=5)):
        o = _lib.default_call_opt()
        for k, v in kw.items():
            setattr(o, k, v)
        out.append(pytest.param(o, id=",".join(f"{k}={v}" for k, v in kw.items()) or "default"))
    return out


def run(ctx, idx, planes, copt, max_calls):
    import torch
    from quasimodo_b200 import _lib
    dev = torch.device("cuda:0")
    d = torch.from_numpy(np.ascontiguousarray(planes).reshape(-1)).to(dev)
    out = torch.full((max(max_calls, 1) * 40,), 0xAB, dtype=torch.uint8, device=dev)
    n = C.c_int64(-1)
    rc = _lib.lib().qm_call_snps(ctx._h, idx._h, C.byref(copt), C.c_void_p(d.data_ptr()), C.c_void_p(out.data_ptr()) if max_calls else None,
                                 max_calls, C.byref(n), None)
    torch.cuda.synchronize()
    return rc, n.value, out.cpu().numpy().view(_lib.CALL_DTYPE)


def check(got, want):
    assert len(got) == len(want)
    for i, (g, w) in enumerate(zip(got, want)):
        for k in ("rid", "pos", "ref", "alt", "dp", "ad_ref_f", "ad_ref_r", "ad_alt_f", "ad_alt_r"):
            assert int(g[k]) == w[k], (i, k, int(g[k]), w)
        assert np.float32(g["af"]) == w["af"], (i, g, w)
        q = np.float32(g["qual"])
        assert np.isfinite(q) and abs(float(q) - float(w["qual"])) <= float(np.spacing(w["qual"])), (i, float(q), float(w["qual"]), w)


@pytest.mark.parametrize("copt", call_opts())
def test_calls_equal_the_rule(ctx, idx, genome, planes, copt):
    want = expected(planes, genome.codes, genome.offs, copt)
    assert len(want) > 50
    rc, n, got = run(ctx, idx, planes, copt, 4096)
    assert rc == 0 and n == len(want)
    check(got[:n], want)


def test_the_edge_columns_are_there(genome, planes):
    from quasimodo_b200 import _lib
    o = _lib.default_call_opt()
    o.min_af = 0.001
    want = expected(planes, genome.codes, genome.offs, o)
    quals = np.array([w["qual"] for w in want])
    assert (quals == 999).sum() >= 3 and ((quals > 990) & (quals < 999)).sum() >= 3
    assert ((quals > 0) & (quals < 0.01)).any() and (quals == 0).any()       # f just above e, and f == e
    assert any(w["af"] == 1 for w in want)
    assert {w["rid"] for w in want} == set(range(len(genome.lens)))
    assert any(w["rid"] == 3 and w["pos"] == genome.lens[3] - 1 for w in want)
    assert max(np.unique([(w["rid"], w["pos"]) for w in want], axis=0, return_counts=True)[1]) == 3


def test_max_calls_overflow(ctx, idx, genome, planes):
    from quasimodo_b200 import _lib
    copt = _lib.default_call_opt()
    want = expected(planes, genome.codes, genome.offs, copt)
    n_all = len(want)
    rc, n, got = run(ctx, idx, planes, copt, n_all)
    assert rc == 0 and n == n_all
    check(got, want)
    rc, n, got = run(ctx, idx, planes, copt, n_all - 1)
    assert rc == QM_ELIMIT and n == n_all
    check(got, want[:n_all - 1])                   # what fits is written, in order
    rc, n, _ = run(ctx, idx, planes, copt, 0)
    assert rc == QM_ELIMIT and n == n_all
