"""ctypes binding of the CPU oracle (oracle/libqmo.so).  TEST INFRASTRUCTURE ONLY: importable from
tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs; never from the
product package."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class Opt(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("a", "b", "o_del", "e_del", "o_ins", "e_ins", "w", "zdrop", "pen_clip5", "pen_clip3",
                 "min_seed_len", "max_occ", "T", "pen_unpaired", "max_ins", "max_chain_gap", "mapq_coef_len")] + \
               [("mask_level", C.c_float), ("drop_ratio", C.c_float), ("mask_level_redun", C.c_float),
                ("min_chain_weight", C.c_int32), ("flags", C.c_int32), ("reserved", C.c_int32 * 2)]


EXT_DTYPE = np.dtype([("score", "<i4"), ("qle", "<i4"), ("tle", "<i4"), ("gtle", "<i4"),
                      ("gscore", "<i4"), ("max_off", "<i4")])


def build(force=False):
    so = os.path.join(_HERE, "libqmo.so")
    srcs = [os.path.join(_HERE, f) for f in os.listdir(_HERE) if f.endswith((".c", ".h", ".cpp"))] + [os.path.join(_HERE, "Makefile")]
    outs = [so, os.path.join(_HERE, "libqmsim.so")]
    if force or any(not os.path.exists(o) or any(os.path.getmtime(s) > os.path.getmtime(o) for s in srcs) for o in outs):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "all"])
    return so


BUILD_KIND = "-O3, portable x86-64"


def use_native_build():
    """bench.py's CPU arms: rebuild the restatement with -O3 -march=native ON THIS HOST (never shipped) and use it from now on.
    The library goes to a temporary directory, removed at exit: the tree may be read-only.  Falls back to the portable build
    when the compile fails."""
    global _LIB, BUILD_KIND
    d = tempfile.mkdtemp(prefix="qmo_native_")
    atexit.register(shutil.rmtree, d, True)
    so = os.path.join(d, "libqmo_native.so")
    try:
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "native"], env=dict(os.environ, NATIVE_OUT=so))
    except (subprocess.CalledProcessError, OSError):
        return False
    _LIB = None
    lib(so)
    BUILD_KIND = "-O3 -march=native (built on this host)"
    return True


def lib(path=None):
    global _LIB
    if _LIB is None:
        _LIB = C.CDLL(path or build())
        _LIB.qmo_ksw_extend2.restype = C.c_int64
        _LIB.qmo_ksw_global2.restype = C.c_int
        _LIB.qmo_ksw_align2.restype = C.c_int64
    return _LIB


def default_opt():
    o = Opt()
    lib().qmo_opt_default(C.byref(o))
    return o


def _u8(a):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    return a, a.ctypes.data_as(C.c_void_p)


def ksw_extend2(query, target, h0, w, end_bonus, opt=None):
    """-> ((score,qle,tle,gtle,gscore,max_off), executed_cells)"""
    opt = opt or default_opt()
    q, qp = _u8(query)
    t, tp = _u8(target)
    out = np.zeros(1, dtype=EXT_DTYPE)
    cells = lib().qmo_ksw_extend2(len(q), qp, len(t), tp, C.byref(opt), int(w), int(end_bonus), int(h0),
                                  out.ctypes.data_as(C.c_void_p))
    return tuple(int(x) for x in out[0]), int(cells)


def ksw_global2(query, target, w, opt=None, max_cigar=64):
    """-> (score, [(op,len)...]) with op 0=M 1=I 2=D"""
    opt = opt or default_opt()
    q, qp = _u8(query)
    t, tp = _u8(target)
    cig = np.zeros(max_cigar, dtype=np.uint32)
    n = C.c_int(0)
    s = lib().qmo_ksw_global2(len(q), qp, len(t), tp, C.byref(opt), int(w), C.byref(n),
                              cig.ctypes.data_as(C.c_void_p), max_cigar)
    if n.value < 0:
        raise OverflowError("cigar overflow")
    return int(s), [(int(c & 0xf), int(c >> 4)) for c in cig[:n.value]]


SW_DTYPE = np.dtype([("score", "<i4"), ("te", "<i4"), ("qe", "<i4"), ("score2", "<i4"), ("te2", "<i4"),
                     ("tb", "<i4"), ("qb", "<i4"), ("pad", "<i4")])


def ksw_align2(query, target, minsc, opt=None):
    """-> ((score, te, qe, score2, te2, tb, qb), executed_cells)"""
    opt = opt or default_opt()
    q, qp = _u8(query)
    t, tp = _u8(target)
    out = np.zeros(1, dtype=SW_DTYPE)
    cells = lib().qmo_ksw_align2(len(q), qp, len(t), tp, C.byref(opt), int(minsc), out.ctypes.data_as(C.c_void_p))
    return tuple(int(x) for x in out[0])[:7], int(cells)


# ---------------------------------------------------------------------------------------------
# pipeline stages
MAX_SEEDS, MAX_REGS, MAX_CIGAR = 64, 16, 21
SEED_DTYPE = np.dtype([("rbeg", "<i8"), ("qbeg", "<i4"), ("len", "<i4")])
REG_DTYPE = np.dtype([("rb", "<i8"), ("re", "<i8"), ("qb", "<i4"), ("qe", "<i4"), ("rid", "<i4"), ("score", "<i4"),
                      ("truesc", "<i4"), ("sub", "<i4"), ("csub", "<i4"), ("sub_n", "<i4"), ("w", "<i4"),
                      ("seedcov", "<i4"), ("secondary", "<i4"), ("seedlen0", "<i4")])
ALN_DTYPE = np.dtype([("rid", "<i4"), ("pos", "<i4"), ("flag", "<u2"), ("mapq", "u1"), ("n_cigar", "u1"),
                      ("score", "<i4"), ("sub", "<i4"), ("nm", "<i4"), ("mate_rid", "<i4"), ("mate_pos", "<i4"),
                      ("tlen", "<i4"), ("qb", "<i4"), ("qe", "<i4"), ("cigar", "<u4", (MAX_CIGAR,))])
PESTAT_DTYPE = np.dtype([("low", "<i4"), ("high", "<i4"), ("failed", "<i4"), ("pad", "<i4"), ("avg", "<f8"), ("std", "<f8")])
EXT_TASK_DTYPE = np.dtype([("q_off", "<u4"), ("t_off", "<u4"), ("qlen", "<i4"), ("tlen", "<i4"),
                           ("h0", "<i4"), ("w", "<i4"), ("end_bonus", "<i4"), ("flags", "<u4")])
assert REG_DTYPE.itemsize == 64 and ALN_DTYPE.itemsize == 128 and SEED_DTYPE.itemsize == 16


class ExtLog(C.Structure):
    _fields_ = [("seq", C.c_void_p), ("seq_len", C.c_int64), ("seq_cap", C.c_int64),
                ("tasks", C.c_void_p), ("results", C.c_void_p), ("w_used", C.c_void_p), ("cells", C.c_void_p),
                ("n", C.c_int64), ("cap", C.c_int64)]


class Ref:
    def __init__(self, codes, lens, k=31):
        L = lib()
        L.qmo_ref_create.restype = C.c_void_p
        L.qmo_ref_create.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        L.qmo_ref_destroy.argtypes = [C.c_void_p]
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        lens = np.ascontiguousarray(lens, dtype=np.int64)
        self.l_pac = int(lens.sum())
        self.lens = lens
        self.k = k
        self._h = L.qmo_ref_create(codes.ctypes.data, len(lens), lens.ctypes.data, k)

    def set_fm(self, fm, max_mem_intv=20):
        """attach bwa's FM-index of the same genome (FmIndex, kept alive here): opt.flags |= F_FM_SEEDS then seeds through it"""
        L = lib()
        L.qmo_ref_set_fm.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        self._fm = fm
        L.qmo_ref_set_fm(self._h, fm._h if fm is not None else None, max_mem_intv)

    def __del__(self):
        if getattr(self, "_h", None):
            lib().qmo_ref_destroy(self._h)
            self._h = None


F_NO_RESCUE, F_FM_SEEDS = 1, 2


def _libc_free(ptr):
    C.CDLL(None).free(C.c_void_p(ptr))


def align_se(ref, reads, lens, opt=None, want_log=False):
    """-> dict(seeds, n_seeds, regs, n_regs, cells[, log])"""
    opt = opt or default_opt()
    L = lib()
    L.qmo_align_se.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    n, stride = reads.shape
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    seeds = np.zeros((n, MAX_SEEDS), dtype=SEED_DTYPE)
    n_seeds = np.zeros(n, dtype=np.int32)
    regs = np.zeros((n, MAX_REGS), dtype=REG_DTYPE)
    n_regs = np.zeros(n, dtype=np.int32)
    cells = C.c_int64(0)
    log = ExtLog()
    L.qmo_align_se(ref._h, C.byref(opt), n, reads.ctypes.data, stride, lens.ctypes.data, seeds.ctypes.data,
                   n_seeds.ctypes.data, regs.ctypes.data, n_regs.ctypes.data, C.byref(log) if want_log else None,
                   C.byref(cells))
    out = dict(seeds=seeds, n_seeds=n_seeds, regs=regs, n_regs=n_regs, cells=cells.value)
    if want_log:
        m = log.n
        if m:
            out["log"] = dict(
                seq=np.ctypeslib.as_array(C.cast(log.seq, C.POINTER(C.c_uint8)), (log.seq_len,)).copy(),
                tasks=np.frombuffer(C.string_at(log.tasks, m * 32), dtype=EXT_TASK_DTYPE).copy(),
                results=np.frombuffer(C.string_at(log.results, m * 24), dtype=EXT_DTYPE).copy(),
                w_used=np.frombuffer(C.string_at(log.w_used, m * 4), dtype="<i4").copy(),
                cells=np.frombuffer(C.string_at(log.cells, m * 8), dtype="<i8").copy())
            for p in (log.seq, log.tasks, log.results, log.w_used, log.cells):
                _libc_free(p)
        else:
            out["log"] = dict(seq=np.zeros(1, np.uint8), tasks=np.zeros(0, EXT_TASK_DTYPE), results=np.zeros(0, EXT_DTYPE),
                              w_used=np.zeros(0, "<i4"), cells=np.zeros(0, "<i8"))
    return out


def pestat(ref, regs, n_regs, opt=None):
    opt = opt or default_opt()
    L = lib()
    L.qmo_pestat.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    pes = np.zeros(4, dtype=PESTAT_DTYPE)
    L.qmo_pestat(ref._h, C.byref(opt), len(n_regs) // 2, regs.ctypes.data, n_regs.ctypes.data, pes.ctypes.data)
    return pes


F_NO_RESCUE = 1


def mate_rescue(ref, reads, lens, regs, n_regs, pes, opt=None):
    """regs / n_regs updated in place -> (local alignments run, cells)"""
    opt = opt or default_opt()
    L = lib()
    L.qmo_mate_rescue.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_void_p]
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    n, stride = reads.shape
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    n_sw, cells = C.c_int64(0), C.c_int64(0)
    L.qmo_mate_rescue(ref._h, C.byref(opt), n // 2, reads.ctypes.data, stride, lens.ctypes.data, regs.ctypes.data,
                      n_regs.ctypes.data, pes.ctypes.data, C.byref(n_sw), C.byref(cells))
    return n_sw.value, cells.value


def pair_and_finish(ref, reads, lens, regs, n_regs, pes, pair_id0=0, opt=None):
    """regs / n_regs are modified in place (primary marking re-sorts them)"""
    opt = opt or default_opt()
    L = lib()
    L.qmo_pair_and_finish.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    n, stride = reads.shape
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    alns = np.zeros(n, dtype=ALN_DTYPE)
    L.qmo_pair_and_finish(ref._h, C.byref(opt), n // 2, int(pair_id0), reads.ctypes.data, stride, lens.ctypes.data,
                          regs.ctypes.data, n_regs.ctypes.data, pes.ctypes.data, alns.ctypes.data)
    return alns


NCH = 16


class PileupOpt(C.Structure):
    _fields_ = [("min_mapq", C.c_int32), ("min_bq", C.c_int32), ("count_orphans", C.c_int32),
                ("ignore_overlaps", C.c_int32)]


def pileup(ref, alns, reads, quals, lens, popt=None):
    """-> int32 counts [l_pac, 16] (rows = forward reference positions, contigs concatenated)"""
    L = lib()
    L.qmo_pileup.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                             C.c_void_p, C.c_void_p]
    if popt is None:
        popt = PileupOpt()
        L.qmo_pileup_opt_default(C.byref(popt))
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    quals = np.ascontiguousarray(quals, dtype=np.uint8)
    n, stride = reads.shape
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    alns = np.ascontiguousarray(alns, dtype=ALN_DTYPE)
    counts = np.zeros((ref.l_pac, NCH), dtype=np.int32)
    L.qmo_pileup(ref._h, C.byref(popt), n // 2, alns.ctypes.data, reads.ctypes.data, quals.ctypes.data, stride,
                 lens.ctypes.data, counts.ctypes.data)
    return counts


def depth_cap(ref, alns, max_depth, popt=None):
    """htslib's per-file depth cap (bcftools mpileup -d): -> bool mask of the reads the pileup iterator keeps (False for dropped
    and for not admitted reads)"""
    L = lib()
    L.qmo_depth_cap.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_void_p]
    if popt is None:
        popt = PileupOpt()
        L.qmo_pileup_opt_default(C.byref(popt))
    alns = np.ascontiguousarray(alns, dtype=ALN_DTYPE)
    keep = np.zeros(len(alns), np.uint8)
    L.qmo_depth_cap(ref._h, C.byref(popt), len(alns), alns.ctypes.data, int(max_depth), keep.ctypes.data)
    return keep.astype(bool)


def pileup_capped(ref, alns, reads, quals, lens, max_depth, popt=None):
    """counts with the depth cap on: the dropped reads never reach the pileup (flag QCFAIL on a copy of the records)"""
    keep = depth_cap(ref, alns, max_depth, popt)
    a = np.array(alns, dtype=ALN_DTYPE, copy=True)
    adm = depth_cap(ref, alns, 1 << 30, popt)
    a["flag"][adm & ~keep] |= 0x200
    return pileup(ref, a, reads, quals, lens, popt), keep


def indels(ref, alns, reads, lens, popt=None, max_out=1 << 20):
    """-> int32 [n, 10]: rid, pos, len, type (0 ins, 1 del), has_n, seq, n_fwd, n_rev, key_lo, key_hi; sorted by key"""
    L = lib()
    L.qmo_indels.restype = C.c_int64
    L.qmo_indels.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int64]
    if popt is None:
        popt = PileupOpt()
        L.qmo_pileup_opt_default(C.byref(popt))
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    n, stride = reads.shape
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    alns = np.ascontiguousarray(alns, dtype=ALN_DTYPE)
    out = np.zeros((max_out, 10), dtype=np.int32)
    m = L.qmo_indels(ref._h, C.byref(popt), n // 2, alns.ctypes.data, reads.ctypes.data, stride, lens.ctypes.data, out.ctypes.data, max_out)
    assert m <= max_out
    return out[:m].copy()


def mpileup_text(ref, alns, reads, quals, lens, names, popt=None):
    """-> bytes: samtools-mpileup text of the batch"""
    L = lib()
    L.qmo_mpileup_text.restype = C.c_int64
    L.qmo_mpileup_text.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                   C.c_void_p, C.c_void_p]
    L.qmo_free.argtypes = [C.c_void_p]
    if popt is None:
        popt = PileupOpt()
        L.qmo_pileup_opt_default(C.byref(popt))
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    quals = np.ascontiguousarray(quals, dtype=np.uint8)
    n, stride = reads.shape
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    alns = np.ascontiguousarray(alns, dtype=ALN_DTYPE)
    arr = (C.c_char_p * len(names))(*[s.encode() for s in names])
    out = C.c_void_p()
    size = L.qmo_mpileup_text(ref._h, C.byref(popt), n // 2, alns.ctypes.data, reads.ctypes.data, quals.ctypes.data, stride,
                              lens.ctypes.data, arr, C.byref(out))
    text = C.string_at(out, size)
    L.qmo_free(out)
    return text


def baq(ref, alns, reads, quals, lens, popt=None, flag=3):
    """-> quals with every admitted read's base qualities capped by its base alignment quality (htslib sam_prob_realn, flag 3 =
    extended BAQ as both mpileups run it)"""
    L = lib()
    L.qmo_baq.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]
    L.qmo_baq.restype = None
    if popt is None:
        popt = PileupOpt()
        L.qmo_pileup_opt_default(C.byref(popt))
    reads = np.ascontiguousarray(reads, dtype=np.uint8)
    quals = np.ascontiguousarray(quals, dtype=np.uint8)
    n, stride = reads.shape
    lens = np.ascontiguousarray(lens, dtype=np.int32)
    alns = np.ascontiguousarray(alns, dtype=ALN_DTYPE)
    out = np.empty_like(quals)
    L.qmo_baq(ref._h, C.byref(popt), n, alns.ctypes.data, reads.ctypes.data, quals.ctypes.data, stride, lens.ctypes.data, int(flag),
              out.ctypes.data)
    return out


def kpa_glocal(ref_codes, query_codes, quals, d=0.001, e=0.1, bw=7):
    """the banded profile HMM of BAQ -> (state[int32], q[uint8], phred likelihood)"""
    L = lib()
    L.qmo_kpa_glocal.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_void_p]
    L.qmo_kpa_glocal.restype = C.c_int
    r = np.ascontiguousarray(ref_codes, dtype=np.uint8); qy = np.ascontiguousarray(query_codes, dtype=np.uint8)
    ql = np.ascontiguousarray(quals, dtype=np.uint8)
    state = np.zeros(len(qy), np.int32); q = np.zeros(len(qy), np.uint8)
    pr = L.qmo_kpa_glocal(r.ctypes.data, len(r), qy.ctypes.data, len(qy), ql.ctypes.data, d, e, bw, state.ctypes.data, q.ctypes.data)
    return state, q, pr


PESTAT_PAIRS = 65536


def run_sample(ref, codes, quals, lens, pair_id0=0, opt=None, popt=None, prefix=None):
    """The whole read-level path for one batch of a sample, as the product's qm_sample does it: single-end
    alignment, insert-size model from the sample's first min(n, PESTAT_PAIRS) pairs (`prefix` = (codes, lens) of
    those pairs when this batch is a later shard), pairing + CIGAR, pileup.  -> (alns, counts, cells, pes)"""
    opt = opt or default_opt()
    o = align_se(ref, codes, lens, opt=opt)
    n_pairs = len(lens) // 2
    if prefix is None:
        m = min(n_pairs, PESTAT_PAIRS)
        pes = pestat(ref, o["regs"][:2 * m], o["n_regs"][:2 * m], opt=opt)
    else:
        pc, pl = prefix
        m = min(len(pl) // 2, PESTAT_PAIRS)
        po = align_se(ref, pc[:2 * m], pl[:2 * m], opt=opt)
        pes = pestat(ref, po["regs"], po["n_regs"], opt=opt)
    alns = pair_and_finish(ref, codes, lens, o["regs"], o["n_regs"], pes, pair_id0=pair_id0, opt=opt)
    counts = pileup(ref, alns, codes, quals, lens, popt)
    return alns, counts, o["cells"], pes


class FmIndex:
    """bwa's FM-index (oracle/qmo_fm.c): built from the packed genome as `bwa index` builds it, or loaded from bwa's own
    .bwt / .sa files; bwt_bytes() / sa_bytes() serialise it exactly as bwa writes those files"""

    def __init__(self, codes=None, bwt=None, sa=None, sa_intv=32):
        L = lib()
        L.qmo_fm_build.restype = C.c_void_p
        L.qmo_fm_build.argtypes = [C.c_void_p, C.c_int64, C.c_int]
        L.qmo_fm_load.restype = C.c_void_p
        L.qmo_fm_load.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]
        L.qmo_fm_free.argtypes = [C.c_void_p]
        for f in ("qmo_fm_bwt_bytes", "qmo_fm_sa_bytes"):
            getattr(L, f).restype = C.c_int64
            getattr(L, f).argtypes = [C.c_void_p, C.c_void_p]
        L.qmo_fm_seeds.restype = C.c_int
        L.qmo_fm_seeds.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
        if codes is not None:
            codes = np.ascontiguousarray(codes, dtype=np.uint8)
            self._h = L.qmo_fm_build(codes.ctypes.data, len(codes), sa_intv)
        else:
            b, s = np.frombuffer(bwt, np.uint8), np.frombuffer(sa, np.uint8)
            self._h = L.qmo_fm_load(b.ctypes.data, len(b), s.ctypes.data, len(s))
        if not self._h:
            raise ValueError("FM-index: inconsistent .bwt / .sa contents")

    def __del__(self):
        try:
            if self._h:
                lib().qmo_fm_free(self._h)
        except Exception:
            pass

    def _bytes(self, fn):
        n = fn(self._h, None)
        out = np.zeros(n, np.uint8)
        fn(self._h, out.ctypes.data)
        return out.tobytes()

    def bwt_bytes(self):
        return self._bytes(lib().qmo_fm_bwt_bytes)

    def sa_bytes(self):
        return self._bytes(lib().qmo_fm_sa_bytes)

    def seeds(self, ref, read, opt=None, max_mem_intv=20, max_seeds=4096):
        """bwa-mem's seeds of one read (codes 0..4), in the order mem_chain visits them -> int64 [n, 3]: rbeg, qbeg, len"""
        opt = opt or default_opt()
        q = np.ascontiguousarray(read, dtype=np.uint8)
        out = np.zeros((max_seeds, 3), np.int64)
        n = lib().qmo_fm_seeds(self._h, ref._h, C.byref(opt), len(q), q.ctypes.data, max_mem_intv, out.ctypes.data, max_seeds)
        return out[:min(n, max_seeds)].copy()


_SIM = None


def simulate_pairs(W, pair0, n_pairs, stride=None):
    """host half of the input simulator (oracle/libqmsim.so): the same bytes as the product's qm_simulate_pairs*"""
    global _SIM
    if _SIM is None:
        build()
        _SIM = C.CDLL(os.path.join(_HERE, "libqmsim.so"))
    stride = stride or W.params.read_len
    codes = np.empty((2 * n_pairs, stride), dtype=np.uint8)
    quals = np.empty((2 * n_pairs, stride), dtype=np.uint8)
    rc = _SIM.qmsim_pairs_host(C.byref(W.params), C.c_void_p(W.src_codes.ctypes.data), C.c_void_p(W.src_off.ctypes.data),
                               C.c_void_p(W.src_len.ctypes.data), C.c_void_p(W.src_cum.ctypes.data), C.c_int64(pair0),
                               C.c_int64(n_pairs), C.c_int32(stride), C.c_void_p(codes.ctypes.data), C.c_void_p(quals.ctypes.data),
                               None, None)
    if rc:
        raise RuntimeError("qmsim_pairs_host failed")
    return codes, quals


def set_threads(n):
    """OpenMP threads of the restatement (torchrun exports OMP_NUM_THREADS=1: the CPU arm must undo that itself)"""
    try:
        C.CDLL("libgomp.so.1").omp_set_num_threads(int(n))
    except OSError:
        pass


def n_threads():
    L = lib()
    try:
        omp = C.CDLL("libgomp.so.1")
        return int(omp.omp_get_max_threads())
    except OSError:
        return 1
