"""ctypes loader of the C-ABI library (quasimodo_b200/libquasimodo_b200.so).

There is no CPU fallback: if the library is missing this raises, and creating a context without a
B200 raises.  The struct layouts mirror include/quasimodo_b200.h."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libquasimodo_b200.so")

_LIB = None


class QmError(RuntimeError):
    pass


class Opt(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("a", "b", "o_del", "e_del", "o_ins", "e_ins", "w", "zdrop", "pen_clip5", "pen_clip3",
                 "min_seed_len", "max_occ", "T", "pen_unpaired", "max_ins", "max_chain_gap", "mapq_coef_len")] + \
               [("mask_level", C.c_float), ("drop_ratio", C.c_float), ("mask_level_redun", C.c_float),
                ("min_chain_weight", C.c_int32), ("flags", C.c_int32), ("reserved", C.c_int32 * 2)]


class SimParams(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("read_len", C.c_int32), ("ins_mean", C.c_int32), ("ins_sd", C.c_int32),
                ("ins_max", C.c_int32), ("n_sources", C.c_int32), ("indel_ppm", C.c_int32), ("n_ppm", C.c_int32),
                ("lowq_ppm", C.c_int32), ("reserved", C.c_int32 * 3)]


class PileupOpt(C.Structure):
    _fields_ = [("min_mapq", C.c_int32), ("min_bq", C.c_int32), ("count_orphans", C.c_int32),
                ("ignore_overlaps", C.c_int32)]


class BamPairs(C.Structure):
    """qm_bam_pairs: the pair layout qm_bam_to_pairs leaves in library scratch (device pointers)"""
    _fields_ = [("n_pairs", C.c_int64), ("stride", C.c_int32), ("pad", C.c_int32), ("d_alns", C.c_void_p), ("d_codes", C.c_void_p),
                ("d_quals", C.c_void_p), ("d_lens", C.c_void_p), ("d_row_file", C.c_void_p), ("d_drop", C.c_void_p),
                ("n_capped", C.c_int64)]


class CallOpt(C.Structure):
    _fields_ = [("min_dp", C.c_int32), ("min_alt", C.c_int32), ("min_af", C.c_float), ("reserved", C.c_int32)]


MAX_SEEDS, MAX_REGS, MAX_CIGAR, NCH, N_STAGES, PESTAT_PAIRS = 64, 16, 21, 16, 9, 65536
F_NO_RESCUE = 1          # qm_opt.flags: bwa mem -S
F_FM_SEEDS, F_FM_NO_ROUND3 = 2, 4   # seeds through bwa's FM-index; without its third seeding round
STAGES = ("seed_chain", "advance", "extend", "pair_cigar", "pileup", "h2d", "d2h", "other", "rescue")
CALL_DTYPE = np.dtype([("rid", "<i4"), ("pos", "<i4"), ("ref", "u1"), ("alt", "u1"), ("pad", "u1", (2,)), ("dp", "<i4"),
                       ("ad_ref_f", "<i4"), ("ad_ref_r", "<i4"), ("ad_alt_f", "<i4"), ("ad_alt_r", "<i4"),
                       ("qual", "<f4"), ("af", "<f4")])
assert CALL_DTYPE.itemsize == 40
INDEL_DTYPE = np.dtype([("rid", "<i4"), ("pos", "<i4"), ("len", "<i4"), ("type", "u1"), ("has_n", "u1"), ("pad", "u1", (2,)),
                        ("seq", "<u4"), ("n_fwd", "<i4"), ("n_rev", "<i4"), ("pad2", "<u4"), ("key", "<u8")])
assert INDEL_DTYPE.itemsize == 40
EXT_TASK_DTYPE = np.dtype([("q_off", "<u4"), ("t_off", "<u4"), ("qlen", "<i4"), ("tlen", "<i4"),
                           ("h0", "<i4"), ("w", "<i4"), ("end_bonus", "<i4"), ("flags", "<u4")])
EXT_RESULT_DTYPE = np.dtype([("score", "<i4"), ("qle", "<i4"), ("tle", "<i4"), ("gtle", "<i4"),
                             ("gscore", "<i4"), ("max_off", "<i4"), ("w_used", "<i4"), ("cells", "<i4")])
SEED_DTYPE = np.dtype([("rbeg", "<i8"), ("qbeg", "<i4"), ("len", "<i4")])
REG_DTYPE = np.dtype([("rb", "<i8"), ("re", "<i8"), ("qb", "<i4"), ("qe", "<i4"), ("rid", "<i4"), ("score", "<i4"),
                      ("truesc", "<i4"), ("sub", "<i4"), ("csub", "<i4"), ("sub_n", "<i4"), ("w", "<i4"),
                      ("seedcov", "<i4"), ("secondary", "<i4"), ("seedlen0", "<i4")])
ALN_DTYPE = np.dtype([("rid", "<i4"), ("pos", "<i4"), ("flag", "<u2"), ("mapq", "u1"), ("n_cigar", "u1"),
                      ("score", "<i4"), ("sub", "<i4"), ("nm", "<i4"), ("mate_rid", "<i4"), ("mate_pos", "<i4"),
                      ("tlen", "<i4"), ("qb", "<i4"), ("qe", "<i4"), ("cigar", "<u4", (MAX_CIGAR,))])
DUP_KEY_DTYPE = np.dtype([("pair_id", "<i8"), ("key", "<u8"), ("end0", "<u4"), ("end1", "<u4"), ("score", "<i4"), ("pad", "<i4")])
CAP_KEY_DTYPE = np.dtype([("key", "<u8"), ("read_id", "<i4"), ("end", "<i4")])
assert DUP_KEY_DTYPE.itemsize == 32 and CAP_KEY_DTYPE.itemsize == 16
PESTAT_DTYPE = np.dtype([("low", "<i4"), ("high", "<i4"), ("failed", "<i4"), ("pad", "<i4"), ("avg", "<f8"), ("std", "<f8")])
assert REG_DTYPE.itemsize == 64 and ALN_DTYPE.itemsize == 128 and SEED_DTYPE.itemsize == 16 and PESTAT_DTYPE.itemsize == 32
QM_EXT_BAND_RETRY = 1
QM_EXT_PREV_H0 = 2

_P, _I, _L = C.c_void_p, C.c_int32, C.c_int64

# every symbol include/quasimodo_b200.h declares (checked by tests/test_cabi.py): name -> (restype, argtypes)
SIGNATURES = {
    "qm_opt_default": (None, [_P]),
    "qm_ctx_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "qm_ctx_destroy": (None, [_P]),
    "qm_last_error": (C.c_char_p, [_P]),
    "qm_version": (C.c_char_p, []),
    "qm_device_sm_count": (C.c_int, [_P]),
    "qm_extend_batch": (C.c_int, [_P, _P, _P, _P, _L, _P, _P]),
    "qm_extend_batch_host": (C.c_int, [_P, _P, _P, C.c_size_t, _P, _L, _P]),
    "qm_index_build": (C.c_int, [_P, _P, C.c_int, _P, C.c_int, C.POINTER(C.c_void_p)]),
    "qm_index_destroy": (None, [_P, _P]),
    "qm_index_lpac": (_L, [_P]),
    "qm_index_attach_bwa": (C.c_int, [_P, _P, _P, _L, _P, _L]),
    "qm_index_build_fm": (C.c_int, [_P, _P, _P]),
    "qm_index_fm_export": (C.c_int, [_P, _P, C.POINTER(C.c_int64), _P, C.POINTER(C.c_int64)]),
    "qm_collect_seeds": (C.c_int, [_P, _P, _P, _P, _I, _P, _L, _P, _P, _P]),
    "qm_align_se": (C.c_int, [_P, _P, _P, _P, _I, _P, _L, _P, _P, _P, _P]),
    "qm_pestat_sync": (C.c_int, [_P, _P, _P, _P, _P, _L, _P, _P]),
    "qm_mate_rescue": (C.c_int, [_P, _P, _P, _P, _I, _P, _L, _P, _P, _P, _P, _P]),
    "qm_pair_finish": (C.c_int, [_P, _P, _P, _P, _I, _P, _L, _L, _P, _P, _P, _P, _P]),
    "qm_pileup_opt_default": (None, [_P]),
    "qm_pileup_accumulate": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _L, _P, _P]),
    "qm_counts_to_rows": (C.c_int, [_P, _P, _P, _P, _P]),
    "qm_sample_begin": (C.c_int, [_P, _P, _P, _P, C.POINTER(C.c_void_p)]),
    "qm_sample_destroy": (None, [_P]),
    "qm_sample_reset": (C.c_int, [_P, _P]),
    "qm_sample_set_pestat": (C.c_int, [_P, _P]),
    "qm_sample_get_pestat": (C.c_int, [_P, _P]),
    "qm_sample_estimate_pestat": (C.c_int, [_P, _P, _I, _P, _L, _P]),
    "qm_sample_set_chunks": (C.c_int, [_P, _P, _L]),
    "qm_sample_chunk_pestat": (C.c_int, [_P, _P, _L, C.POINTER(C.c_int64)]),
    "qm_sample_add_pairs": (C.c_int, [_P, _P, _P, _I, _P, _L, _L, _P, _P]),
    "qm_sample_add_pairs_host": (C.c_int, [_P, _P, _P, _I, _P, _L, _L, _P]),
    "qm_sample_add_pairs_host_packed": (C.c_int, [_P, _P, _P, _P, _I, _P, _L, _L, _P]),
    "qm_pack_reads_host": (C.c_int, [_P, _I, _L, _P, _P]),
    "qm_sample_set_filter": (C.c_int, [_P, C.c_int]),
    "qm_sample_keep_host": (C.c_int, [_P, _P, _L, C.POINTER(C.c_int64)]),
    "qm_sample_counts": (_P, [_P]),
    "qm_sample_stats_sync": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), _P]),
    "qm_sample_counts_host": (C.c_int, [_P, _P]),
    "qm_call_opt_default": (None, [_P]),
    "qm_call_snps": (C.c_int, [_P, _P, _P, _P, _P, _L, C.POINTER(C.c_int64), _P]),
    "qm_eval_match": (C.c_int, [_P, _P, _L, _P, _L, _P, _P, _P]),
    "qm_eval_match_host": (C.c_int, [_P, _P, _L, _P, _L, _P, _P]),
    "qm_eval_calls": (C.c_int, [_P, _P, _L, _P, _L, _P, _P, _P]),
    "qm_sample_call_snps_host": (C.c_int, [_P, _P, _P, _L, C.POINTER(C.c_int64)]),
    "qm_aln_sort_keys": (C.c_int, [_P, _P, _P, _L, _P, C.POINTER(C.c_int), _P]),
    "qm_sort_pairs": (C.c_int, [_P, _P, _P, _L, C.c_int, _P]),
    "qm_sort_keys_host": (C.c_int, [_P, _P, _L, C.c_int, _P]),
    "qm_host_alloc": (C.c_int, [_P, C.c_size_t, C.POINTER(C.c_void_p)]),
    "qm_host_free": (None, [_P, _P]),
    "qm_mark_duplicates": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, C.POINTER(C.c_int64), _P]),
    "qm_sample_set_rmdup": (C.c_int, [_P, C.c_int]),
    "qm_sample_rmdup_finish": (C.c_int, [_P, C.POINTER(C.c_int64), _P]),
    "qm_sample_kept_alns_host": (C.c_int, [_P, _P, _L]),
    "qm_depth_cap": (C.c_int, [_P, _P, C.c_int, _P, _P, C.c_int, _P, C.POINTER(C.c_int64), _P]),
    "qm_sample_set_max_depth": (C.c_int, [_P, C.c_int]),
    "qm_dup_keys": (C.c_int, [_P, C.c_int, _P, _P, _P, _P, _P, _P, _P, C.POINTER(C.c_int64), _P]),
    "qm_mark_duplicates_keys": (C.c_int, [_P, _P, _L, C.c_int, _P, _P, _P, C.POINTER(C.c_int64), _P]),
    "qm_cap_keys": (C.c_int, [_P, _P, C.c_int, _P, _P, _P, _P, C.POINTER(C.c_int64), _P]),
    "qm_depth_cap_keys": (C.c_int, [_P, _P, _L, C.c_int, C.c_int, _P, _P, _P, C.POINTER(C.c_int64), _P]),
    "qm_sample_finish_comm": (C.c_int, [_P, _P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), _P]),
    "qm_sample_finish": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), _P]),
    "qm_sample_set_baq": (C.c_int, [_P, C.c_int]),
    "qm_baq_apply": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _L, _I, _P, _P]),
    "qm_baq_apply_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _L, _I, _P]),
    "qm_mpileup_text": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _L, _P, _P, _P, _P]),
    "qm_mpileup_text_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _L, _P, _P]),
    "qm_mpileup_text_fetch": (C.c_int, [_P, _P, _L]),
    "qm_mpileup_text_ranked": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _L, _P, _P, _P, _P, _P]),
    "qm_bam_to_pairs": (C.c_int, [_P, _P, _P, _P, _L, _I, _P, C.c_int, C.c_int, C.POINTER(BamPairs), _P]),
    "qm_bam_to_pairs_host": (C.c_int, [_P, _P, _P, _L, _P, _L, _I, _P, C.c_int, C.c_int, C.POINTER(BamPairs)]),
    "qm_bam_mark_duplicates": (C.c_int, [_P, _P, _P, _L, _P, C.POINTER(C.c_int64), C.POINTER(C.c_int64), _P]),
    "qm_bam_mark_duplicates_host": (C.c_int, [_P, _P, _L, _P, _L, _P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "qm_pileup_accumulate_masked": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _L, _P, _P, _P, _P]),
    "qm_profile_enable": (C.c_int, [_P, C.c_int]),
    "qm_profile_collect": (C.c_int, [_P, _P, _P]),
    "qm_simulate_pairs_host": (C.c_int, [_P, _P, _P, _P, _P, _L, _L, _I, _P, _P, _P, _P]),
    "qm_simulate_pairs": (C.c_int, [_P, _P, _P, _P, _P, _P, _L, _L, _I, _P, _P, _P]),
    "qm_comm_available": (C.c_int, []),
    "qm_comm_unique_id": (C.c_int, [_P]),
    "qm_comm_init_rank": (C.c_int, [_P, C.c_int, C.c_int, _P, C.POINTER(C.c_void_p)]),
    "qm_comm_init_all": (C.c_int, [C.c_int, _P, _P]),
    "qm_comm_destroy": (None, [_P]),
    "qm_comm_rank": (C.c_int, [_P]),
    "qm_comm_size": (C.c_int, [_P]),
    "qm_counts_allreduce": (C.c_int, [_P, _P, _P, _L, _P]),
    "qm_counts_allreduce_nccl": (C.c_int, [_P, _P, _P, _L, _P]),
    "qm_pestat_bcast": (C.c_int, [_P, _P, _P, C.c_int, _P]),
    "qm_comm_allgather": (C.c_int, [_P, _P, _P, _P, C.c_size_t, _P]),
    "qm_indel_table_create": (C.c_int, [_P, C.c_int, C.POINTER(C.c_void_p)]),
    "qm_indel_table_destroy": (None, [_P]),
    "qm_indel_table_reset": (C.c_int, [_P, _P]),
    "qm_indel_table_fetch_host": (C.c_int, [_P, _P, _P, _L, C.POINTER(C.c_int64)]),
    "qm_indel_table_merge": (C.c_int, [_P, _P, _L, _P]),
    "qm_pileup_accumulate_indels": (C.c_int, [_P, _P, _P, _P, _P, _P, _I, _P, _L, _P, _P, _P]),
    "qm_sample_indel_table": (_P, [_P]),
    "qm_sample_set_comm": (C.c_int, [_P, _P]),
    "qm_sample_allreduce_counts": (C.c_int, [_P, _P]),
    "qm_dpx_peak_sync": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}
EXPORTS = sorted(SIGNATURES)


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise QmError(f"{SO_PATH} is missing: build it with `python -m quasimodo_b200.build` "
                          "(there is no CPU fallback)")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def default_opt():
    o = Opt()
    lib().qm_opt_default(C.byref(o))
    return o


def default_call_opt():
    o = CallOpt()
    lib().qm_call_opt_default(C.byref(o))
    return o


def default_pileup_opt():
    o = PileupOpt()
    lib().qm_pileup_opt_default(C.byref(o))
    return o
