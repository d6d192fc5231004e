"""Host-side (Python) face of the C-ABI: a thin object wrapper used by tests and bench.py.  Device
memory comes from torch (plumbing only); every computation goes through libquasimodo_b200.so."""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import QmError


def _check(ctx, rc, what):
    if rc != 0:
        msg = _lib.lib().qm_last_error(ctx).decode() if ctx else ""
        raise QmError(f"{what} failed with code {rc}: {msg}")


def _ptr(t):
    """device pointer of a torch tensor (or None)"""
    return C.c_void_p(0 if t is None else t.data_ptr())


def _ptrs(ts):
    """array of device pointers of a list of torch tensors"""
    return (C.c_void_p * max(1, len(ts)))(*[t.data_ptr() for t in ts])


def _i64(v):
    """ctypes int64 array of a list of ints (passed as the object itself, so it lives through the call)"""
    return (C.c_int64 * max(1, len(v)))(*[int(x) for x in v])


def _n_pairs(d_alns):
    """pairs in a device tensor of alignment records (2 records of 128 bytes per pair)"""
    return d_alns.numel() * d_alns.element_size() // 256


class Index:
    """Device-resident k-mer hash index + reference bases (qm_index)."""

    def __init__(self, ctx, genome, k=31):
        self.ctx, self.genome, self.k = ctx, genome, k
        codes = np.ascontiguousarray(genome.codes, dtype=np.uint8)
        lens = np.ascontiguousarray(genome.lens, dtype=np.int64)
        self._h = C.c_void_p()
        rc = _lib.lib().qm_index_build(ctx._h, codes.ctypes.data, len(lens), lens.ctypes.data, k, C.byref(self._h))
        _check(ctx._h, rc, "qm_index_build")
        self.l_pac = int(_lib.lib().qm_index_lpac(self._h))
        self.offsets = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)

    def build_fm(self):
        """bwa's FM-index of this genome, rebuilt here (enables opt.flags |= F_FM_SEEDS)"""
        codes = np.ascontiguousarray(self.genome.codes, dtype=np.uint8)
        _check(self.ctx._h, _lib.lib().qm_index_build_fm(self.ctx._h, self._h, codes.ctypes.data), "qm_index_build_fm")

    def attach_bwa(self, bwt_bytes, sa_bytes):
        """bwa's own index files (the bytes of X.bwt and X.sa) as this index's FM-index"""
        b, s = np.frombuffer(bwt_bytes, np.uint8), np.frombuffer(sa_bytes, np.uint8)
        _check(self.ctx._h, _lib.lib().qm_index_attach_bwa(self.ctx._h, self._h, b.ctypes.data, len(b), s.ctypes.data, len(s)), "qm_index_attach_bwa")

    def fm_export(self):
        nb, ns = C.c_int64(), C.c_int64()
        _check(self.ctx._h, _lib.lib().qm_index_fm_export(self._h, None, C.byref(nb), None, C.byref(ns)), "qm_index_fm_export")
        b, s = np.zeros(nb.value, np.uint8), np.zeros(ns.value, np.uint8)
        _check(self.ctx._h, _lib.lib().qm_index_fm_export(self._h, b.ctypes.data, C.byref(nb), s.ctypes.data, C.byref(ns)), "qm_index_fm_export")
        return b.tobytes(), s.tobytes()

    def close(self):
        if getattr(self, "_h", None) and self.ctx._h:
            _lib.lib().qm_index_destroy(self.ctx._h, self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Comm:
    """NCCL communicator of the library (one process per GPU): rank 0 makes the id with Comm.unique_id(), the host carries the
    128 bytes to the other ranks (e.g. torch.distributed.broadcast), every rank constructs Comm(ctx, n_ranks, rank, id)."""

    @staticmethod
    def available():
        return bool(_lib.lib().qm_comm_available())

    @staticmethod
    def unique_id():
        buf = (C.c_uint8 * 128)()
        rc = _lib.lib().qm_comm_unique_id(buf)
        if rc:
            raise QmError(f"qm_comm_unique_id failed with code {rc} (is libnccl.so.2 loadable?)")
        return bytes(buf)

    def __init__(self, ctx, n_ranks, rank, uid):
        self.ctx = ctx
        self._h = C.c_void_p()
        buf = (C.c_uint8 * 128).from_buffer_copy(bytes(uid))
        _check(ctx._h, _lib.lib().qm_comm_init_rank(ctx._h, int(n_ranks), int(rank), buf, C.byref(self._h)), "qm_comm_init_rank")
        self.rank, self.size = int(rank), int(n_ranks)

    @classmethod
    def init_all(cls, ctxs):
        """one communicator per context, all in this process (qm_comm_init_all): comms[i] belongs to ctxs[i]; call the collectives
        from one host thread per GPU"""
        n = len(ctxs)
        hs = (C.c_void_p * n)(*[c._h for c in ctxs])
        out = (C.c_void_p * n)()
        _check(ctxs[0]._h, _lib.lib().qm_comm_init_all(n, hs, out), "qm_comm_init_all")
        comms = []
        for r, c in enumerate(ctxs):
            cm = cls.__new__(cls)
            cm.ctx, cm._h, cm.rank, cm.size = c, C.c_void_p(out[r]), r, n
            comms.append(cm)
        return comms

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().qm_comm_destroy(self._h)
        self._h = None

    def bcast_pestat(self, pes, root=0, stream=0):
        pes = np.ascontiguousarray(pes, dtype=_lib.PESTAT_DTYPE)
        _check(self.ctx._h, _lib.lib().qm_pestat_bcast(self.ctx._h, self._h, pes.ctypes.data, int(root), C.c_void_p(stream)), "qm_pestat_bcast")
        return pes

    def allreduce_counts(self, d_counts, stream=0):
        """in-place integer sum of a torch int32 tensor over the ranks"""
        _check(self.ctx._h, _lib.lib().qm_counts_allreduce(self.ctx._h, self._h, _ptr(d_counts), d_counts.numel(), C.c_void_p(stream)),
               "qm_counts_allreduce")
        return d_counts


class Sample:
    """One {sample}.{ref_name}: owns the count tensor; pairs are added batch by batch (qm_sample_*)."""

    def __init__(self, ctx, idx, opt=None, popt=None):
        self.ctx, self.idx = ctx, idx
        self.opt = opt or ctx.opt
        self.popt = popt or ctx.pileup_opt
        self._h = C.c_void_p()
        rc = _lib.lib().qm_sample_begin(ctx._h, idx._h, C.byref(self.opt), C.byref(self.popt), C.byref(self._h))
        _check(ctx._h, rc, "qm_sample_begin")

    def close(self):
        if getattr(self, "_h", None) and self.ctx._h:
            _lib.lib().qm_sample_destroy(self._h)
        self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self, stream=0):
        _check(self.ctx._h, _lib.lib().qm_sample_reset(self._h, C.c_void_p(stream)), "qm_sample_reset")

    def set_comm(self, comm):
        """spread the sample over the communicator's ranks (see qm_sample_set_comm); None clears"""
        _check(self.ctx._h, _lib.lib().qm_sample_set_comm(self._h, comm._h if comm is not None else None), "qm_sample_set_comm")

    def allreduce_counts(self, stream=0):
        _check(self.ctx._h, _lib.lib().qm_sample_allreduce_counts(self._h, C.c_void_p(stream)), "qm_sample_allreduce_counts")

    def set_pestat(self, pes):
        pes = np.ascontiguousarray(pes, dtype=_lib.PESTAT_DTYPE)
        _check(self.ctx._h, _lib.lib().qm_sample_set_pestat(self._h, pes.ctypes.data), "qm_sample_set_pestat")

    def get_pestat(self):
        pes = np.zeros(4, dtype=_lib.PESTAT_DTYPE)
        _check(self.ctx._h, _lib.lib().qm_sample_get_pestat(self._h, pes.ctypes.data), "qm_sample_get_pestat")
        return pes

    def estimate_pestat(self, d_codes, d_lens, stream=0):
        """insert-size model from the sample's first pairs (device tensors); see qm_sample_estimate_pestat"""
        n, stride = d_codes.shape
        rc = _lib.lib().qm_sample_estimate_pestat(self._h, _ptr(d_codes), stride, _ptr(d_lens), n // 2, C.c_void_p(stream))
        _check(self.ctx._h, rc, "qm_sample_estimate_pestat")

    def set_chunks(self, chunk_pairs):
        """per-chunk mode (bwa mem's model per input chunk): the sizes in pairs of the next add call's chunks, which must add up
        to its pairs; see qm_sample_set_chunks"""
        c = np.ascontiguousarray(chunk_pairs, dtype=np.int64)
        _check(self.ctx._h, _lib.lib().qm_sample_set_chunks(self._h, c.ctypes.data if len(c) else None, len(c)), "qm_sample_set_chunks")

    def chunk_pestat(self):
        """per-chunk mode: the models of the last add call's chunks, [n_chunks, 4] of PESTAT_DTYPE"""
        n = C.c_int64()
        _check(self.ctx._h, _lib.lib().qm_sample_chunk_pestat(self._h, None, 0, C.byref(n)), "qm_sample_chunk_pestat")
        buf = np.zeros(4 * max(n.value, 1), dtype=_lib.PESTAT_DTYPE)
        _check(self.ctx._h, _lib.lib().qm_sample_chunk_pestat(self._h, buf.ctypes.data, n.value, C.byref(n)), "qm_sample_chunk_pestat")
        return buf[:4 * n.value].reshape(-1, 4)

    def add_pairs(self, d_codes, d_quals, d_lens, pair_id0=0, d_alns=None, stream=0):
        """device-resident batch: torch uint8 [2n, stride] codes / quals, int32 [2n] lens"""
        n, stride = d_codes.shape
        rc = _lib.lib().qm_sample_add_pairs(self._h, _ptr(d_codes), _ptr(d_quals), stride, _ptr(d_lens), n // 2,
                                            int(pair_id0), _ptr(d_alns), C.c_void_p(stream))
        _check(self.ctx._h, rc, "qm_sample_add_pairs")

    def add_pairs_host(self, h_codes, h_quals, h_lens, pair_id0=0, h_alns=None):
        """host batch (numpy arrays or pinned torch CPU tensors); copies happen inside"""
        def hp(a):
            return C.c_void_p(0) if a is None else C.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)
        n, stride = h_codes.shape
        rc = _lib.lib().qm_sample_add_pairs_host(self._h, hp(h_codes), hp(h_quals), int(stride), hp(h_lens), n // 2,
                                                 int(pair_id0), hp(h_alns))
        _check(self.ctx._h, rc, "qm_sample_add_pairs_host")

    def add_pairs_host_packed(self, h_bases2, h_nmask, h_quals, h_lens, pair_id0=0, h_alns=None):
        """host batch with the bases packed (pack_reads): 2 bits per base + an N bit per base cross the link instead of a byte"""
        def hp(a):
            return C.c_void_p(0) if a is None else C.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)
        n, stride = h_quals.shape
        rc = _lib.lib().qm_sample_add_pairs_host_packed(self._h, hp(h_bases2), hp(h_nmask), hp(h_quals), int(stride), hp(h_lens), n // 2,
                                                        int(pair_id0), hp(h_alns))
        _check(self.ctx._h, rc, "qm_sample_add_pairs_host_packed")

    def set_rmdup(self, on=True):
        """duplicate removal (picard MarkDuplicates REMOVE_DUPLICATES=true): keep reads + records, count at rmdup_finish()"""
        _check(self.ctx._h, _lib.lib().qm_sample_set_rmdup(self._h, 1 if on else 0), "qm_sample_set_rmdup")

    def set_max_depth(self, max_depth):
        """bcftools mpileup -d: htslib's depth cap (0 = off); counting is deferred to finish()"""
        _check(self.ctx._h, _lib.lib().qm_sample_set_max_depth(self._h, int(max_depth)), "qm_sample_set_max_depth")

    def set_filter(self, on=True):
        """filter mode (a contaminant pass): align and finish pairs, count nothing, leave one keep byte per pair of each batch"""
        _check(self.ctx._h, _lib.lib().qm_sample_set_filter(self._h, 1 if on else 0), "qm_sample_set_filter")

    def keep(self, n_pairs):
        """filter mode: -> uint8 [n_pairs], 1 for each pair of the last batch whose records both pass `samtools view -f 12 -F 256`"""
        k = np.zeros(n_pairs, dtype=np.uint8)
        n = C.c_int64()
        _check(self.ctx._h, _lib.lib().qm_sample_keep_host(self._h, k.ctypes.data, int(n_pairs), C.byref(n)), "qm_sample_keep_host")
        assert n.value == int(k.sum())
        return k

    def set_baq(self, flag=3):
        """base alignment quality for the pileup: 0 off (-B, default), 3 extended BAQ (what both mpileups run), 1 plain"""
        _check(self.ctx._h, _lib.lib().qm_sample_set_baq(self._h, int(flag)), "qm_sample_set_baq")

    def finish(self, stream=0):
        """deferred counting (rmdup and / or depth cap) -> (duplicate pairs, reads the cap dropped)"""
        nd, nc = C.c_int64(), C.c_int64()
        _check(self.ctx._h, _lib.lib().qm_sample_finish(self._h, C.byref(nd), C.byref(nc), C.c_void_p(stream)), "qm_sample_finish")
        return nd.value, nc.value

    def finish_comm(self, comm, stream=0):
        """deferred counting of a sample sharded over the ranks of `comm` (collective: every rank calls it) -> sample-wide (duplicate
        pairs, reads the cap dropped); this rank's count tensor then holds its survivors' counts: all-reduce them next"""
        nd, nc = C.c_int64(), C.c_int64()
        _check(self.ctx._h, _lib.lib().qm_sample_finish_comm(self._h, comm._h, C.byref(nd), C.byref(nc), C.c_void_p(stream)),
               "qm_sample_finish_comm")
        return nd.value, nc.value

    def rmdup_finish(self, stream=0):
        """-> number of duplicate pairs; the count tensor then holds the survivors' counts"""
        n = C.c_int64()
        _check(self.ctx._h, _lib.lib().qm_sample_rmdup_finish(self._h, C.byref(n), C.c_void_p(stream)), "qm_sample_rmdup_finish")
        return n.value

    def kept_alns(self, n_pairs):
        a = np.zeros(2 * n_pairs, dtype=_lib.ALN_DTYPE)
        _check(self.ctx._h, _lib.lib().qm_sample_kept_alns_host(self._h, a.ctypes.data, len(a)), "qm_sample_kept_alns_host")
        return a

    def counts_ptr(self):
        return _lib.lib().qm_sample_counts(self._h)

    def counts_tensor(self):
        """torch int32 view [NCH, l_pac] of the device count tensor (no copy)"""
        import torch
        n = _lib.NCH * self.idx.l_pac

        class _Holder:
            pass
        h = _Holder()
        h.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (self.counts_ptr(), False), "version": 3}
        return torch.as_tensor(h, device=f"cuda:{self.ctx.device}").view(_lib.NCH, self.idx.l_pac)

    def stats(self, stream=0):
        n, c = C.c_int64(), C.c_int64()
        rc = _lib.lib().qm_sample_stats_sync(self._h, C.byref(n), C.byref(c), C.c_void_p(stream))
        _check(self.ctx._h, rc, "qm_sample_stats_sync")
        return n.value, c.value

    def indels(self, max_out=1 << 18):
        """the sample's indel alleles -> structured array INDEL_DTYPE, sorted by (position, type, length, bases)"""
        out = np.zeros(max_out, dtype=_lib.INDEL_DTYPE)
        n = C.c_int64()
        tab = _lib.lib().qm_sample_indel_table(self._h)
        rc = _lib.lib().qm_indel_table_fetch_host(tab, self.idx._h, out.ctypes.data, max_out, C.byref(n))
        _check(self.ctx._h, rc, "qm_indel_table_fetch_host")
        return out[:n.value].copy()

    def counts_host(self):
        rows = np.empty((self.idx.l_pac, _lib.NCH), dtype=np.int32)
        _check(self.ctx._h, _lib.lib().qm_sample_counts_host(self._h, rows.ctypes.data), "qm_sample_counts_host")
        return rows

    def call_snps(self, copt=None, max_calls=1 << 20, stream=0):
        """-> structured array CALL_DTYPE, sorted by (position, alt)"""
        import torch
        copt = copt or _lib.default_call_opt()
        d_calls = torch.empty(max_calls * 40, dtype=torch.uint8, device=f"cuda:{self.ctx.device}")
        n = C.c_int64()
        rc = _lib.lib().qm_call_snps(self.ctx._h, self.idx._h, C.byref(copt), C.c_void_p(self.counts_ptr()), _ptr(d_calls),
                                     max_calls, C.byref(n), C.c_void_p(stream))
        _check(self.ctx._h, rc, "qm_call_snps")
        return d_calls[:n.value * 40].cpu().numpy().view(_lib.CALL_DTYPE)


class Context:
    """One per (process, device).  Raises if no B200-class device is usable (no CPU fallback)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        rc = _lib.lib().qm_ctx_create(int(device), C.byref(self._h))
        if rc != 0:
            self._h = None
            raise QmError(f"qm_ctx_create(device={device}) failed with code {rc}: a CUDA device of compute "
                          "capability 10.x is required; this library has no CPU fallback")
        self.device = device
        self.opt = _lib.default_opt()
        self.pileup_opt = _lib.default_pileup_opt()

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().qm_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def sm_count(self):
        return _lib.lib().qm_device_sm_count(self._h)

    # ---- extension (ksw_extend2) ----
    def extend_batch_host(self, seq, tasks, opt=None):
        """seq: uint8 arena of base codes; tasks: structured array EXT_TASK_DTYPE -> EXT_RESULT_DTYPE array"""
        opt = opt or self.opt
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        tasks = np.ascontiguousarray(tasks, dtype=_lib.EXT_TASK_DTYPE)
        out = np.zeros(len(tasks), dtype=_lib.EXT_RESULT_DTYPE)
        rc = _lib.lib().qm_extend_batch_host(self._h, C.byref(opt), seq.ctypes.data, seq.nbytes,
                                             tasks.ctypes.data, len(tasks), out.ctypes.data)
        _check(self._h, rc, "qm_extend_batch_host")
        return out

    def extend_batch(self, d_seq, d_tasks, n_tasks, d_out, stream=0, opt=None):
        """device pointers (ints), asynchronous on `stream` (a cudaStream_t handle as int)"""
        opt = opt or self.opt
        rc = _lib.lib().qm_extend_batch(self._h, C.byref(opt), C.c_void_p(d_seq), C.c_void_p(d_tasks),
                                        int(n_tasks), C.c_void_p(d_out), C.c_void_p(stream))
        _check(self._h, rc, "qm_extend_batch")

    def dpx_peak(self, kind=1, iters=4096):
        g, ms = C.c_double(), C.c_double()
        rc = _lib.lib().qm_dpx_peak_sync(self._h, kind, iters, C.byref(g), C.byref(ms))
        _check(self._h, rc, "qm_dpx_peak_sync")
        return g.value, ms.value

    def sample(self, idx, opt=None, popt=None):
        return Sample(self, idx, opt, popt)

    # ---- genome diff (rule `nucmer`: nucmer; delta-filter -r -q; show-snps -CTHlr) ----
    def genome_diff(self, ref_idx, qry_genome, opt=None, phases=None):
        """rows (GDIFF_ROW_DTYPE, show-snps -CTHlr) and kept alignments (GDIFF_ALN_DTYPE) of qry_genome against the reference of
        ref_idx, whose k must be opt.min_match (default opt: nucmer's, min_match 20).  phases: a dict that receives the
        milliseconds of each phase (_lib.GDIFF_PHASES)."""
        opt = opt or _lib.default_gdiff_opt()
        codes = np.ascontiguousarray(qry_genome.codes, dtype=np.uint8)
        lens = np.ascontiguousarray(qry_genome.lens, dtype=np.int64)
        n_rows, n_alns = C.c_int64(), C.c_int64()
        ms = (C.c_double * len(_lib.GDIFF_PHASES))()
        max_rows, max_alns = 1 << 16, 1 << 10
        L = _lib.lib()
        while True:
            rows = np.zeros(max_rows, _lib.GDIFF_ROW_DTYPE)
            alns = np.zeros(max_alns, _lib.GDIFF_ALN_DTYPE)
            rc = L.qm_genome_diff_host(self._h, ref_idx._h, codes.ctypes.data, len(lens), lens.ctypes.data, C.byref(opt),
                                       rows.ctypes.data, max_rows, C.byref(n_rows), alns.ctypes.data, max_alns, C.byref(n_alns), ms)
            if rc == -5 and (n_rows.value > max_rows or n_alns.value > max_alns):      # QM_ELIMIT: room for what it reported
                max_rows, max_alns = max(max_rows, n_rows.value), max(max_alns, n_alns.value)
                continue
            _check(self._h, rc, "qm_genome_diff_host")
            break
        if phases is not None:
            phases.update(zip(_lib.GDIFF_PHASES, list(ms)))
        return rows[:n_rows.value].copy(), alns[:n_alns.value].copy()

    def profile_enable(self, on=True):
        _check(self._h, _lib.lib().qm_profile_enable(self._h, 1 if on else 0), "qm_profile_enable")

    def profile_collect(self):
        """-> ({stage: ms}, {stage: launches}); synchronises the device and clears the totals"""
        ms = (C.c_double * _lib.N_STAGES)()
        ln = (C.c_int64 * _lib.N_STAGES)()
        _check(self._h, _lib.lib().qm_profile_collect(self._h, ms, ln), "qm_profile_collect")
        return dict(zip(_lib.STAGES, list(ms))), dict(zip(_lib.STAGES, list(ln)))

    # ---- alignment pipeline on a device-resident read batch (torch uint8 tensors [2*n_pairs, stride]) ----
    def index(self, genome, k=None):
        return Index(self, genome, k or self.opt.min_seed_len)

    def collect_seeds(self, idx, d_codes, d_lens, stream=0, opt=None):
        import torch
        opt = opt or self.opt
        n, stride = d_codes.shape
        seeds = torch.zeros(n * _lib.MAX_SEEDS * 16, dtype=torch.uint8, device=d_codes.device)
        n_seeds = torch.zeros(n, dtype=torch.int32, device=d_codes.device)
        rc = _lib.lib().qm_collect_seeds(self._h, idx._h, C.byref(opt), _ptr(d_codes), stride, _ptr(d_lens), n,
                                         _ptr(seeds), _ptr(n_seeds), C.c_void_p(stream))
        _check(self._h, rc, "qm_collect_seeds")
        return seeds, n_seeds

    def align_se(self, idx, d_codes, d_lens, d_regs=None, d_n_regs=None, d_cells=None, stream=0, opt=None):
        import torch
        opt = opt or self.opt
        n, stride = d_codes.shape
        if d_regs is None:
            d_regs = torch.zeros(n * _lib.MAX_REGS * 64, dtype=torch.uint8, device=d_codes.device)
        if d_n_regs is None:
            d_n_regs = torch.zeros(n, dtype=torch.int32, device=d_codes.device)
        rc = _lib.lib().qm_align_se(self._h, idx._h, C.byref(opt), _ptr(d_codes), stride, _ptr(d_lens), n,
                                    _ptr(d_regs), _ptr(d_n_regs), _ptr(d_cells), C.c_void_p(stream))
        _check(self._h, rc, "qm_align_se")
        return d_regs, d_n_regs

    def pestat(self, idx, d_regs, d_n_regs, n_pairs, stream=0, opt=None):
        opt = opt or self.opt
        pes = np.zeros(4, dtype=_lib.PESTAT_DTYPE)
        rc = _lib.lib().qm_pestat_sync(self._h, idx._h, C.byref(opt), _ptr(d_regs), _ptr(d_n_regs), int(n_pairs),
                                       pes.ctypes.data, C.c_void_p(stream))
        _check(self._h, rc, "qm_pestat_sync")
        return pes

    def mate_rescue(self, idx, d_codes, d_lens, d_regs, d_n_regs, pes, d_stats=None, stream=0, opt=None):
        """mem_matesw for every pair: d_regs / d_n_regs updated in place; d_stats: int64[2] += (alignments run, cells)"""
        opt = opt or self.opt
        n, stride = d_codes.shape
        pes = np.ascontiguousarray(pes, dtype=_lib.PESTAT_DTYPE)
        rc = _lib.lib().qm_mate_rescue(self._h, idx._h, C.byref(opt), _ptr(d_codes), stride, _ptr(d_lens), n // 2, _ptr(d_regs),
                                       _ptr(d_n_regs), pes.ctypes.data, _ptr(d_stats) if d_stats is not None else None,
                                       C.c_void_p(stream))
        _check(self._h, rc, "qm_mate_rescue")

    def pair_finish(self, idx, d_codes, d_lens, d_regs, d_n_regs, pes, pair_id0=0, d_alns=None, stream=0, opt=None):
        import torch
        opt = opt or self.opt
        n, stride = d_codes.shape
        if d_alns is None:
            d_alns = torch.zeros(n * 128, dtype=torch.uint8, device=d_codes.device)
        pes = np.ascontiguousarray(pes, dtype=_lib.PESTAT_DTYPE)
        rc = _lib.lib().qm_pair_finish(self._h, idx._h, C.byref(opt), _ptr(d_codes), stride, _ptr(d_lens), n // 2,
                                       int(pair_id0), _ptr(d_regs), _ptr(d_n_regs), pes.ctypes.data, _ptr(d_alns),
                                       C.c_void_p(stream))
        _check(self._h, rc, "qm_pair_finish")
        return d_alns

    def pileup_accumulate(self, idx, d_alns, d_codes, d_quals, d_lens, d_counts, stream=0, popt=None):
        popt = popt or self.pileup_opt
        n, stride = d_codes.shape
        rc = _lib.lib().qm_pileup_accumulate(self._h, idx._h, C.byref(popt), _ptr(d_alns), _ptr(d_codes), _ptr(d_quals),
                                             stride, _ptr(d_lens), n // 2, _ptr(d_counts), C.c_void_p(stream))
        _check(self._h, rc, "qm_pileup_accumulate")
        return d_counts

    def baq_apply(self, idx, d_alns, d_codes, d_quals, d_lens, flag=3, stream=0, popt=None):
        """-> device tensor like d_quals: the qualities capped by base alignment quality (htslib sam_prob_realn)"""
        import torch
        popt = popt or self.pileup_opt
        n, stride = d_codes.shape
        out = torch.empty_like(d_quals)
        rc = _lib.lib().qm_baq_apply(self._h, idx._h, C.byref(popt), _ptr(d_alns), _ptr(d_codes), _ptr(d_quals), stride, _ptr(d_lens), n,
                                     int(flag), _ptr(out), C.c_void_p(stream))
        _check(self._h, rc, "qm_baq_apply")
        return out

    def baq_apply_host(self, idx, alns, codes, quals, lens, flag=3, popt=None):
        """host arrays in, host array out (numpy)"""
        popt = popt or self.pileup_opt
        codes = np.ascontiguousarray(codes, dtype=np.uint8); quals = np.ascontiguousarray(quals, dtype=np.uint8)
        lens = np.ascontiguousarray(lens, dtype=np.int32); alns = np.ascontiguousarray(alns, dtype=_lib.ALN_DTYPE)
        n, stride = codes.shape
        out = np.empty_like(quals)
        rc = _lib.lib().qm_baq_apply_host(self._h, idx._h, C.byref(popt), alns.ctypes.data, codes.ctypes.data, quals.ctypes.data, stride,
                                          lens.ctypes.data, n, int(flag), out.ctypes.data)
        _check(self._h, rc, "qm_baq_apply_host")
        return out

    def mpileup_text(self, idx, d_alns, d_codes, d_quals, d_lens, names, stream=0, popt=None):
        """samtools-mpileup text of the device-resident records -> bytes (copied to the host)"""
        popt = popt or self.pileup_opt
        n, stride = d_codes.shape
        arr = (C.c_char_p * len(names))(*[s.encode() for s in names])
        d_text, nbytes = C.c_void_p(), C.c_int64(0)
        rc = _lib.lib().qm_mpileup_text(self._h, idx._h, C.byref(popt), _ptr(d_alns), _ptr(d_codes), _ptr(d_quals), stride, _ptr(d_lens),
                                        n // 2, arr, C.byref(d_text), C.byref(nbytes), C.c_void_p(stream))
        _check(self._h, rc, "qm_mpileup_text")
        buf = C.create_string_buffer(max(1, nbytes.value))
        _check(self._h, _lib.lib().qm_mpileup_text_fetch(self._h, buf, nbytes.value), "qm_mpileup_text_fetch")
        return buf.raw[:nbytes.value]

    # ---- duplicate marking and depth cap on device-resident records.  A chunk list gives one rank's records: d_alns[c] holds the
    # records (2 per pair) of pairs pair_id0[c] .. pair_id0[c] + n - 1 (any torch tensor, n = its bytes / 256) ----
    def mark_duplicates(self, d_alns, d_quals, d_lens, stream=0):
        """qm_mark_duplicates over the chunks (input order, pair ids = running offsets): flags 0x400 in place -> duplicate pairs"""
        n = [_n_pairs(a) for a in d_alns]
        strides = (C.c_int32 * max(1, len(n)))(*[q.shape[1] for q in d_quals])
        nd = C.c_int64()
        rc = _lib.lib().qm_mark_duplicates(self._h, len(n), _ptrs(d_alns), _ptrs(d_quals), strides, _ptrs(d_lens),
                                           _i64(n), C.byref(nd), C.c_void_p(stream))
        _check(self._h, rc, "qm_mark_duplicates")
        return nd.value

    def dup_keys(self, d_alns, d_quals, d_lens, pair_id0, stream=0):
        """one rank's duplicate tuples (qm_dup_keys) -> torch uint8 tensor [n, 32] on the device (rows of DUP_KEY_DTYPE)"""
        import torch
        n = [_n_pairs(a) for a in d_alns]
        strides = (C.c_int32 * max(1, len(n)))(*[q.shape[1] for q in d_quals])
        out = torch.empty((max(1, sum(n)), 32), dtype=torch.uint8, device=f"cuda:{self.device}")
        n_out = C.c_int64()
        rc = _lib.lib().qm_dup_keys(self._h, len(n), _ptrs(d_alns), _ptrs(d_quals), strides, _ptrs(d_lens), _i64(n),
                                    _i64(pair_id0), _ptr(out), C.byref(n_out), C.c_void_p(stream))
        _check(self._h, rc, "qm_dup_keys")
        return out[:n_out.value]

    def mark_duplicates_keys(self, d_all, d_alns, pair_id0, stream=0):
        """decide over the union d_all (uint8 [n, 32]) and flag this rank's chunks (qm_mark_duplicates_keys) -> duplicate pairs of the union"""
        n = [_n_pairs(a) for a in d_alns]
        nd = C.c_int64()
        rc = _lib.lib().qm_mark_duplicates_keys(self._h, _ptr(d_all), d_all.shape[0], len(n), _ptrs(d_alns), _i64(n),
                                                _i64(pair_id0), C.byref(nd), C.c_void_p(stream))
        _check(self._h, rc, "qm_mark_duplicates_keys")
        return nd.value

    def depth_cap(self, d_alns, max_depth, stream=0, popt=None):
        """qm_depth_cap over the chunks (input order) -> ([uint8 drop mask [2n] per chunk on the device], reads dropped)"""
        import torch
        popt = popt or self.pileup_opt
        n = [_n_pairs(a) for a in d_alns]
        drops = [torch.zeros(max(1, 2 * k), dtype=torch.uint8, device=f"cuda:{self.device}") for k in n]
        nd = C.c_int64()
        rc = _lib.lib().qm_depth_cap(self._h, C.byref(popt), len(n), _ptrs(d_alns), _i64(n), int(max_depth), _ptrs(drops),
                                     C.byref(nd), C.c_void_p(stream))
        _check(self._h, rc, "qm_depth_cap")
        return [d[:2 * k] for d, k in zip(drops, n)], nd.value

    def cap_keys(self, d_alns, pair_id0, stream=0, popt=None):
        """one rank's depth-cap tuples (qm_cap_keys) -> torch uint8 tensor [n, 16] on the device (rows of CAP_KEY_DTYPE)"""
        import torch
        popt = popt or self.pileup_opt
        n = [_n_pairs(a) for a in d_alns]
        out = torch.empty((max(1, 2 * sum(n)), 16), dtype=torch.uint8, device=f"cuda:{self.device}")
        n_out = C.c_int64()
        rc = _lib.lib().qm_cap_keys(self._h, C.byref(popt), len(n), _ptrs(d_alns), _i64(n), _i64(pair_id0),
                                    _ptr(out), C.byref(n_out), C.c_void_p(stream))
        _check(self._h, rc, "qm_cap_keys")
        return out[:n_out.value]

    def depth_cap_keys(self, d_all, max_depth, n_pairs, pair_id0, stream=0):
        """replay over the union d_all (uint8 [n, 16]) for this rank's chunks of n_pairs[c] pairs (qm_depth_cap_keys)
        -> ([uint8 drop mask [2 n_pairs[c]] per chunk on the device], reads dropped in the union)"""
        import torch
        drops = [torch.zeros(max(1, 2 * int(k)), dtype=torch.uint8, device=f"cuda:{self.device}") for k in n_pairs]
        nd = C.c_int64()
        rc = _lib.lib().qm_depth_cap_keys(self._h, _ptr(d_all), d_all.shape[0], int(max_depth), len(n_pairs), _i64(n_pairs),
                                          _i64(pair_id0), _ptrs(drops), C.byref(nd), C.c_void_p(stream))
        _check(self._h, rc, "qm_depth_cap_keys")
        return [d[:2 * int(k)] for d, k in zip(drops, n_pairs)], nd.value

    def counts_to_rows(self, idx, d_planes, stream=0):
        import torch
        rows = torch.empty(idx.l_pac * _lib.NCH, dtype=torch.int32, device=d_planes.device)
        rc = _lib.lib().qm_counts_to_rows(self._h, idx._h, _ptr(d_planes), _ptr(rows), C.c_void_p(stream))
        _check(self._h, rc, "qm_counts_to_rows")
        return rows.view(idx.l_pac, _lib.NCH)

    def simulate_pairs(self, workload, pair0, n_pairs, d_genome, d_codes, d_quals, stream=0):
        n, stride = d_codes.shape
        rc = _lib.lib().qm_simulate_pairs(self._h, C.byref(workload.params), _ptr(d_genome), workload.src_off.ctypes.data,
                                          workload.src_len.ctypes.data, workload.src_cum.ctypes.data, int(pair0),
                                          int(n_pairs), int(stride), _ptr(d_codes), _ptr(d_quals), C.c_void_p(stream))
        _check(self._h, rc, "qm_simulate_pairs")


def pack_reads(codes, out_bases2=None, out_nmask=None):
    """codes [n, stride] (0..3, else N) -> (bases2 [n, (stride+3)//4], nmask [n, (stride+7)//8]) for add_pairs_host_packed;
    numpy arrays or (pinned) torch CPU tensors, optionally into given buffers"""
    def hp(a):
        return C.c_void_p(a.data_ptr() if hasattr(a, "data_ptr") else a.ctypes.data)
    n, stride = codes.shape
    if out_bases2 is None:
        out_bases2 = np.empty((n, (stride + 3) // 4), np.uint8)
        out_nmask = np.empty((n, (stride + 7) // 8), np.uint8)
    rc = _lib.lib().qm_pack_reads_host(hp(codes), int(stride), int(n), hp(out_bases2), hp(out_nmask))
    if rc:
        raise QmError(f"qm_pack_reads_host failed with code {rc}")
    return out_bases2, out_nmask


def pack_ext_tasks(pairs, h0s, ws, end_bonus, flags=0):
    """Helper: build (seq arena, task array) from a list of (query, target) code arrays."""
    n = len(pairs)
    tasks = np.zeros(n, dtype=_lib.EXT_TASK_DTYPE)
    chunks, off = [], 0
    for i, (q, t) in enumerate(pairs):
        q = np.asarray(q, dtype=np.uint8)
        t = np.asarray(t, dtype=np.uint8)
        tasks[i]["q_off"] = off
        chunks.append(q)
        off += len(q)
        tasks[i]["t_off"] = off
        chunks.append(t)
        off += len(t)
        tasks[i]["qlen"] = len(q)
        tasks[i]["tlen"] = len(t)
    tasks["h0"] = h0s
    tasks["w"] = ws
    tasks["end_bonus"] = end_bonus
    tasks["flags"] = flags
    seq = np.concatenate(chunks) if chunks else np.zeros(0, dtype=np.uint8)
    if len(seq) == 0:
        seq = np.zeros(1, dtype=np.uint8)
    return seq, tasks
