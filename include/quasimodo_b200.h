/*
 * quasimodo_b200.h -- C-ABI of the B200-native QuasiModo read-level hot path.
 *
 * The reference (hzi-bifo/Quasimodo) has NO in-process plugin/FFI interface: its hot path is a chain of
 * Snakemake `shell:` lines calling external binaries (SURVEY.md section 8b).  Each entry point below
 * therefore cites the rule line / upstream function whose work it replaces.  Conventions:
 *   - extern "C", plain pointers and sizes, no C++/torch types;
 *   - every function returns 0 on success or a negative QM_E* code; qm_last_error(ctx) explains;
 *   - pointers named d_* are DEVICE pointers owned by the caller, h_* are HOST pointers owned by the
 *     caller; the library never frees caller memory and never returns memory the caller must free;
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous w.r.t. the host unless their
 *     name ends in _host or _sync;
 *   - a qm_ctx is bound to one CUDA device and is not thread-safe; distinct ctxs are independent;
 *   - there is NO CPU fallback: without a CUDA device qm_ctx_create fails with QM_ENODEV.
 */
#ifndef QUASIMODO_B200_H
#define QUASIMODO_B200_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QM_OK        0
#define QM_EINVAL   -1   /* bad argument                                   */
#define QM_ENODEV   -2   /* no usable CUDA device / extension not usable   */
#define QM_ECUDA    -3   /* CUDA runtime error (see qm_last_error)         */
#define QM_ENOMEM   -4
#define QM_ELIMIT   -5   /* input exceeds a documented hard limit          */
#define QM_EIO      -6

typedef struct qm_ctx qm_ctx;

/* ---- scoring and bwa-mem options in effect for `bwa mem -k 31` (rules/bwa.smk:15; SURVEY.md A.1) ---- */
typedef struct {
    int32_t a, b;                 /* match score, mismatch penalty (N vs anything = -1)  */
    int32_t o_del, e_del, o_ins, e_ins;
    int32_t w;                    /* band width (-w)                                     */
    int32_t zdrop;                /* -d                                                  */
    int32_t pen_clip5, pen_clip3; /* -L                                                  */
    int32_t min_seed_len;         /* -k                                                  */
    int32_t max_occ;              /* -c                                                  */
    int32_t T;                    /* -T                                                  */
    int32_t pen_unpaired;         /* -U                                                  */
    int32_t max_ins;
    int32_t max_chain_gap;
    int32_t mapq_coef_len;
    float   mask_level, drop_ratio, mask_level_redun;
    int32_t min_chain_weight;
    int32_t flags;                /* QM_F_*                                              */
    int32_t reserved[2];
} qm_opt;
#define QM_F_NO_RESCUE 1          /* bwa mem -S: skip mate rescue                        */
#define QM_F_FM_SEEDS  2          /* seeds through bwa's FM-index (qm_index_attach_bwa / _build_fm) instead of the k-mer hash */
#define QM_F_FM_NO_ROUND3 4       /* with QM_F_FM_SEEDS: skip the third seeding round (bwa's max_mem_intv = 0)       */

void qm_opt_default(qm_opt *opt);

/* ---- context ---- */
int         qm_ctx_create(int device, qm_ctx **out);
void        qm_ctx_destroy(qm_ctx *ctx);
const char *qm_last_error(const qm_ctx *ctx);          /* owned by ctx */
const char *qm_version(void);
int         qm_device_sm_count(const qm_ctx *ctx);

/* ---- alignment: batched banded affine-gap extension ----
 * Replaces bwa ksw.c:ksw_extend2 as called from bwamem.c:mem_chain2aln (reference call site
 * rules/bwa.smk:15 `bwa mem -k 31`); semantics in SURVEY.md Appendix A.3.  This is the parity entry
 * point: one task = one ksw_extend2 call.  Sequences are base codes 0..4 (A C G T N), one byte each,
 * in one device arena `d_seq`; a task addresses its query/target by byte offset.
 * If (flags & QM_EXT_BAND_RETRY) the task is run as mem_chain2aln runs it: with w, then with 2w when
 * the first try's score moved and max_off >= 3/4 w (MAX_BAND_TRY = 2); w_used reports the last band.
 */
#define QM_EXT_BAND_RETRY 1u
#define QM_EXT_PREV_H0    2u       /* retry loop starts with prev = h0 (right extension: prev = sc0),
                                      otherwise prev = -1 (left extension)                            */
#define QM_EXT_MAX_QLEN   511      /* hard limit of the kernel's column striping */

typedef struct {
    uint32_t q_off, t_off;        /* byte offsets into d_seq                         */
    int32_t  qlen, tlen;
    int32_t  h0;                  /* score of the seed (+ left extension)            */
    int32_t  w;                   /* band width for this call                        */
    int32_t  end_bonus;           /* pen_clip5 / pen_clip3                           */
    uint32_t flags;
} qm_ext_task;                    /* 32 bytes */

typedef struct {
    int32_t score, qle, tle, gtle, gscore, max_off;   /* ksw_extend2's return value and out-params */
    int32_t w_used;               /* band of the last try                            */
    int32_t cells;                /* inner-loop cells the reference loop executes (sum of end-beg
                                     over rows, over all tries) -- the GCUPS work unit */
} qm_ext_result;                  /* 32 bytes */

int qm_extend_batch(qm_ctx *ctx, const qm_opt *opt, const uint8_t *d_seq, const qm_ext_task *d_tasks,
                    int64_t n_tasks, qm_ext_result *d_out, void *stream);

/* same, host buffers: copies seq + tasks in, results out, synchronises.  seq_bytes = arena size. */
int qm_extend_batch_host(qm_ctx *ctx, const qm_opt *opt, const uint8_t *h_seq, size_t seq_bytes,
                         const qm_ext_task *h_tasks, int64_t n_tasks, qm_ext_result *h_out);

/* ---- reference index (replaces `bwa index`, rules/index.smk:13; SURVEY.md 8a1) ----
 * k-mer hash index (k = opt->min_seed_len, 8 <= k <= 31) over the forward strands of the concatenated contigs
 * plus the 2-bit packed reference; both live in device memory owned by the index object. */
typedef struct qm_index qm_index;
#define QM_MAX_CONTIGS 16
int     qm_index_build(qm_ctx *ctx, const uint8_t *h_codes /* 0..3 */, int n_contigs, const int64_t *h_lens,
                       int k, qm_index **out);
void    qm_index_destroy(qm_ctx *ctx, qm_index *idx);
int64_t qm_index_lpac(const qm_index *idx);
/* bwa's own FM-index of the same genome as an alternative seeder (SURVEY.md 8f-4): with qm_opt.flags & QM_F_FM_SEEDS the seeds
 * are bwa-mem's -- the three rounds of mem_collect_intv (SMEMs, re-seeding, the LAST-like round) and the suffix-array walk of
 * mem_chain, at most QM_MAX_SEEDS per read in bwa's order -- instead of all exact matches of the k-mer hash index.
 * qm_index_attach_bwa takes the bytes of the index files `bwa index` wrote (rules/index.smk:13: X.bwt and X.sa; the reference
 * ships them as ref/X.bwt, ref/X.sa); qm_index_build_fm rebuilds the same bytes from the genome given to qm_index_build, on the
 * device (suffix array of forward + reverse complement by prefix doubling, BWT, checkpoints and samples; about 58 bytes of
 * device memory per suffix while it runs, QM_ELIMIT past 2^31 - 1 suffixes); qm_index_fm_export copies them back as the two
 * files (pass NULL buffers for the sizes).  Once per genome; the index stays in device memory. */
int qm_index_attach_bwa(qm_ctx *ctx, qm_index *idx, const uint8_t *h_bwt, int64_t bwt_bytes, const uint8_t *h_sa, int64_t sa_bytes);
int qm_index_build_fm(qm_ctx *ctx, qm_index *idx, const uint8_t *h_codes);
int qm_index_fm_export(const qm_index *idx, uint8_t *h_bwt, int64_t *bwt_bytes, uint8_t *h_sa, int64_t *sa_bytes);

/* ---- alignment of read pairs (replaces `bwa mem -k 31 ref r1 r2`, rules/bwa.smk:15) ----
 * Read batch layout: see the simulator below (codes/quals, reads 2i and 2i+1 are mates).
 * Stage 1  qm_align_se      : seeding (all MEMs >= k via the hash index), chaining (bwamem.c mem_chain,
 *                             mem_chain_flt), extension (mem_chain2aln -> the batched ksw_extend2 kernel),
 *                             redundancy removal (mem_sort_dedup_patch) -> per-read region lists.
 * Stage 2  qm_pestat_sync   : insert-size model of the batch (bwamem_pair.c mem_pestat).
 * Stage 3  qm_pair_finish   : mate rescue (qm_mate_rescue), primary marking, pairing, MAPQ (mem_sam_pe), CIGAR/NM
 *                             (mem_reg2aln -> bwa_gen_cigar2 -> ksw_global2), SAM flags -> qm_aln records.
 * Hard limits (shared with the oracle): QM_MAX_SEEDS seeds and QM_MAX_REGS regions per read, k-mers with
 * more than min(max_occ, QM_OCC_CAP) occurrences are ignored, QM_MAX_CIGAR operations per alignment. */
#define QM_MAX_SEEDS 64
#define QM_MAX_REGS  16
#define QM_MAX_CIGAR 21
#define QM_OCC_CAP   32

typedef struct { int64_t rbeg; int32_t qbeg, len; } qm_seed;                 /* 16 B */
typedef struct {
    int64_t rb, re;               /* [rb,re) in bwa's doubled coordinates (>= l_pac: reverse strand) */
    int32_t qb, qe;
    int32_t rid, score, truesc, sub, csub, sub_n, w, seedcov, secondary, seedlen0;
} qm_reg;                                                                     /* 64 B */
typedef struct {
    int32_t  rid, pos;            /* 0-based leftmost position on contig rid; -1 when unplaced        */
    uint16_t flag; uint8_t mapq; uint8_t n_cigar;   /* n_cigar = 255: CIGAR overflow (read unmapped)  */
    int32_t  score, sub, nm;
    int32_t  mate_rid, mate_pos, tlen;
    int32_t  qb, qe;              /* aligned interval of the read as sequenced                        */
    uint32_t cigar[QM_MAX_CIGAR]; /* BAM encoding len<<4|op, ops M=0 I=1 D=2 S=4                       */
} qm_aln;                                                                     /* 128 B */
typedef struct { int32_t low, high, failed, pad; double avg, std; } qm_pestat;  /* x4: FF FR RF RR */

/* Read arrays of the two entries below: read r occupies row r of `stride` bytes, lens[r] in [0, stride], stride <= 512
 * (QM_ELIMIT otherwise).  qm_align_se fails with QM_ECUDA should reads be left unfinished after its last round. */
/* diagnostic / parity entry: seeds of every read, sorted by (qbeg, rbeg) (SURVEY.md 8a2) */
int qm_collect_seeds(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride,
                     const int32_t *d_lens, int64_t n_reads, qm_seed *d_seeds /* [n][QM_MAX_SEEDS] */,
                     int32_t *d_n_seeds, void *stream);
/* d_cells (may be NULL): one int64, += executed extension cells (GCUPS work unit) */
int qm_align_se(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride,
                const int32_t *d_lens, int64_t n_reads, qm_reg *d_regs /* [n][QM_MAX_REGS] */, int32_t *d_n_regs,
                int64_t *d_cells, void *stream);
int qm_pestat_sync(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const qm_reg *d_regs, const int32_t *d_n_regs,
                   int64_t n_pairs, qm_pestat h_pes[4], void *stream);
/* mate rescue (bwamem_pair.c mem_matesw as driven by mem_sam_pe; ksw.c ksw_align2): for every region of an end that
 * scores within pen_unpaired of the end's best and has no properly placed region of the mate, the mate is aligned
 * locally inside the window the insert-size model implies; hits of at least min_seed_len join the mate's list.
 * d_regs / d_n_regs are updated in place.  d_stats (may be NULL): two int64, += local alignments run, += their cells.
 * qm_pair_finish runs it first unless opt->flags & QM_F_NO_RESCUE.  Windows longer than 4096 bases are not searched. */
int qm_mate_rescue(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride,
                   const int32_t *d_lens, int64_t n_pairs, qm_reg *d_regs, int32_t *d_n_regs, const qm_pestat pes[4],
                   int64_t *d_stats, void *stream);
int qm_pair_finish(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride,
                   const int32_t *d_lens, int64_t n_pairs, int64_t pair_id0, qm_reg *d_regs, int32_t *d_n_regs,
                   const qm_pestat h_pes[4], qm_aln *d_alns, void *stream);

/* ---- pileup counting (replaces the counting of `bcftools mpileup`, rules/vcfcall.smk:115, and of
 * `samtools mpileup`, rules/vcfcall.smk:39; upstream mplp_func / bam_plp_push / overlap_push /
 * bcf_call_glfgen; SURVEY.md A.8-A.9, 8a9) ----
 * Count tensor: int32 [QM_NCH][l_pac], CHANNEL-MAJOR planes (plane c at d_counts + c*l_pac), position =
 * forward coordinate on the concatenated contigs.  Channels:
 *   0-3 A,C,G,T forward strand, BQ >= min_bq      4 N forward        5 deleted base, forward read
 *   6-9 A,C,G,T reverse strand                   10 N reverse       11 deleted base, reverse read
 *  12 an insertion follows this base             13 a deletion follows this base
 *  14 raw depth (every aligned base of every admitted read, before the BQ filter = bcftools ori_depth)
 *  15 admitted reads whose leftmost aligned base is here
 * Admission as bcftools mpileup: skip UNMAP|SECONDARY|QCFAIL|DUP, MAPQ < min_mapq, and paired reads that
 * are not proper pairs unless count_orphans; mate-overlap quality rewrite unless ignore_overlaps; BAQ off
 * (-B) and no depth cap (deliberate, SURVEY.md A.8).  Accumulates (+=) into d_counts.
 * Reads as in the read batch layout, lens[r] <= stride; stride <= 512 (QM_ELIMIT otherwise, nothing counted). */
#define QM_NCH 16
typedef struct {
    int32_t min_mapq;        /* -q (0)   */
    int32_t min_bq;          /* -Q (13)  */
    int32_t count_orphans;   /* -A       */
    int32_t ignore_overlaps; /* -x       */
} qm_pileup_opt;
void qm_pileup_opt_default(qm_pileup_opt *p);
int qm_pileup_accumulate(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns,
                         const uint8_t *d_codes, const uint8_t *d_quals, int32_t stride, const int32_t *d_lens,
                         int64_t n_pairs, int32_t *d_counts, void *stream);
/* Indel alleles (SURVEY.md 8a9, 8e): every insertion / deletion operation of an admitted read's CIGAR is tallied per
 * (anchor position = the reference base in front of the event, type, length, inserted bases) in a device hash table, forward and
 * reverse reads apart.  Insertions are told apart by their first QM_INDEL_SEQ_BASES bases (plus a flag when one of them is N);
 * lengths above 255 are clamped.  The table is sparse (a few alleles per kb at the simulated error rates); it is what crosses GPUs
 * next to the dense count tensor: qm_indel_table_merge adds gathered records of other ranks into the local table. */
#define QM_INDEL_SEQ_BASES 11
typedef struct {
    int32_t  rid, pos;            /* anchor: 0-based position on contig rid of the base in front of the event      */
    int32_t  len;                 /* inserted / deleted bases                                                       */
    uint8_t  type;                /* 0 insertion, 1 deletion                                                        */
    uint8_t  has_n, pad[2];       /* an N among the first QM_INDEL_SEQ_BASES inserted bases (stored as A)           */
    uint32_t seq;                 /* insertion: base k (forward strand of the reference) at bits 2k, k < 11        */
    int32_t  n_fwd, n_rev;        /* supporting forward / reverse reads                                             */
    uint64_t key;                 /* the table key: sorts by (global position, type, length, bases)                 */
} qm_indel;                       /* 40 B */
typedef struct qm_indel_table qm_indel_table;
int  qm_indel_table_create(qm_ctx *ctx, int log2_slots, qm_indel_table **out);
void qm_indel_table_destroy(qm_indel_table *t);
int  qm_indel_table_reset(qm_indel_table *t, void *stream);
int  qm_indel_table_fetch_host(qm_indel_table *t, const qm_index *idx, qm_indel *h_out, int64_t max_out, int64_t *n_out);
int  qm_indel_table_merge(qm_indel_table *t, const qm_indel *d_records, int64_t n, void *stream);
/* qm_pileup_accumulate plus the indel alleles of the batch into `tab` (may be NULL) */
int  qm_pileup_accumulate_indels(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns,
                                 const uint8_t *d_codes, const uint8_t *d_quals, int32_t stride, const int32_t *d_lens,
                                 int64_t n_pairs, int32_t *d_counts, qm_indel_table *tab, void *stream);
/* the same with a per-read drop mask: d_drop[r] != 0 (2 * n_pairs bytes, may be NULL) leaves read r out, as the depth cap's
 * verdict (qm_depth_cap, qm_bam_pairs.d_drop) asks */
int  qm_pileup_accumulate_masked(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns,
                                 const uint8_t *d_codes, const uint8_t *d_quals, int32_t stride, const int32_t *d_lens,
                                 int64_t n_pairs, int32_t *d_counts, qm_indel_table *tab, const uint8_t *d_drop, void *stream);
/* ---- base alignment quality (SURVEY.md 8f-2; htslib 1.9 realn.c sam_prob_realn over probaln.c kpa_glocal) ----
 * Both mpileups of the reference flow run WITHOUT -B (rules/vcfcall.smk:39 and :115), i.e. with BAQ on: every read is re-aligned
 * to its reference window by a banded profile HMM in double precision and each aligned base's quality is capped by the phred-scaled
 * posterior of its placement (flag 3: "extended" BAQ, the running-maximum form both tools pass; flag 1: plain BAQ).
 * d_quals_out (same layout as d_quals, may not alias it) receives the capped qualities of every read the pileup admits under
 * `po`; other reads keep theirs.  The pileup entries then take d_quals_out in place of d_quals.  Off by default everywhere:
 * the north-star parity configuration is `-B`.  Bit-exact against oracle/qmo_baq.c (tests/test_baq_gpu.py). */
int qm_baq_apply(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns, const uint8_t *d_codes,
                 const uint8_t *d_quals, int32_t stride, const int32_t *d_lens, int64_t n_reads, int32_t flag, uint8_t *d_quals_out,
                 void *stream);
int qm_baq_apply_host(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *h_alns, const uint8_t *h_codes,
                      const uint8_t *h_quals, int32_t stride, const int32_t *h_lens, int64_t n_reads, int32_t flag, uint8_t *h_quals_out);

/* planes [QM_NCH][l_pac] -> rows [l_pac][QM_NCH] (row order of the count TSV, SURVEY.md B.3) */
int qm_counts_to_rows(qm_ctx *ctx, const qm_index *idx, const int32_t *d_planes, int32_t *d_rows, void *stream);

/* ---- one sample end to end: the rule-level entry (replaces the compute of rule `bwa`, rules/bwa.smk:15-18,
 * and the counting of rules `mpileup` / `bcftools`, rules/vcfcall.smk:39,115, for one {sample}.{ref_name}) ----
 * A qm_sample owns the sample's count tensor (device, planes [QM_NCH][l_pac]).  Read pairs are handed in
 * batch by batch, from device memory (qm_sample_add_pairs, asynchronous on `stream` except for the small
 * per-round read-backs) or from host memory (qm_sample_add_pairs_host: chunked, the next chunk's copy overlaps
 * the current chunk's kernels when the host buffers are page-locked; synchronous).
 * bwa estimates its insert-size model per input chunk (mem_pestat); by default it is fixed ONCE per sample, from
 * the first min(n, QM_PESTAT_PAIRS) pairs handed in, or from that prefix of the sample given explicitly
 * (qm_sample_estimate_pestat: a shard that does not start at pair 0 passes the sample's first pairs; every
 * GPU derives the same model, no collective), or set directly, so that the records do not depend on batching
 * or sharding.
 * Per-chunk mode reproduces bwa instead: qm_sample_set_chunks(s, h_chunk_pairs, n_chunks) gives the sizes in pairs of the
 * chunks of the NEXT add call (in order; they must add up to its n_pairs, QM_EINVAL there otherwise, so no chunk straddles two
 * calls) and puts the sample in that mode for good (before its first pairs: QM_EINVAL after them; a reset keeps the mode).
 * Each chunk's pairs are paired against mem_pestat over ALL of that chunk's pairs, estimated on the device; a chunk with too few
 * pairs for an orientation fails it, as in bwa.  A chunk holds 1 .. QM_CHUNK_MAX_PAIRS pairs (QM_ELIMIT above).  Where chunks
 * end is the caller's rule (bwa mem: bseq_read's running base count, -K); the records then depend neither on the batching nor on
 * the GPUs, and no model crosses between GPUs.  qm_sample_set_pestat (bwa mem -I) still replaces every chunk's model.
 * qm_sample_chunk_pestat: the models of the last add call's chunks, 4 per chunk, in order (*n_chunks of them; none when a model
 * was set); with h_pes NULL and max_chunks 0 only *n_chunks.
 * Contract of the read arrays (every entry below): read r occupies row r of `stride` bytes, its length lens[r] lies in
 * [0, stride], stride <= 512 (QM_ELIMIT otherwise); the lengths are the caller's word -- the device entry cannot check them
 * without a pass over the data, the driver checks them while it parses FASTQ. */
#define QM_PESTAT_PAIRS 65536
#define QM_CHUNK_MAX_PAIRS (1 << 21)
typedef struct qm_sample qm_sample;
int  qm_sample_begin(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const qm_pileup_opt *popt, qm_sample **out);
void qm_sample_destroy(qm_sample *s);
int  qm_sample_reset(qm_sample *s, void *stream);                 /* zero counts, forget the insert-size model */
int  qm_sample_set_pestat(qm_sample *s, const qm_pestat pes[4]);
int  qm_sample_get_pestat(const qm_sample *s, qm_pestat pes[4]);
int  qm_sample_estimate_pestat(qm_sample *s, const uint8_t *d_codes, int32_t stride, const int32_t *d_lens, int64_t n_pairs,
                               void *stream);
int  qm_sample_set_chunks(qm_sample *s, const int64_t *h_chunk_pairs, int64_t n_chunks);
int  qm_sample_chunk_pestat(const qm_sample *s, qm_pestat *h_pes, int64_t max_chunks, int64_t *n_chunks);
int  qm_sample_add_pairs(qm_sample *s, const uint8_t *d_codes, const uint8_t *d_quals, int32_t stride,
                         const int32_t *d_lens, int64_t n_pairs, int64_t pair_id0, qm_aln *d_alns /* may be NULL */,
                         void *stream);
int  qm_sample_add_pairs_host(qm_sample *s, const uint8_t *h_codes, const uint8_t *h_quals, int32_t stride,
                              const int32_t *h_lens, int64_t n_pairs, int64_t pair_id0, qm_aln *h_alns /* may be NULL */);
/* The same with the bases PACKED on the host side of the link (north_star: 2-bit-packed read input): h_bases2[r][(stride+3)/4]
 * holds base j of read r at bits 2 (j & 3) of byte j >> 2, h_nmask[r][(stride+7)/8] one "this base is N" bit per base (bit j & 7
 * of byte j >> 3).  0.375 instead of 1 byte per base crosses PCIe (the bases are what the first kernel waits for; the qualities
 * travel behind them); a kernel on the copy stream expands each piece as it lands.  qm_pack_reads_host packs a 1-byte-per-base
 * batch (the driver packs while it parses FASTQ). */
int  qm_sample_add_pairs_host_packed(qm_sample *s, const uint8_t *h_bases2, const uint8_t *h_nmask, const uint8_t *h_quals, int32_t stride,
                                     const int32_t *h_lens, int64_t n_pairs, int64_t pair_id0, qm_aln *h_alns /* may be NULL */);
int  qm_pack_reads_host(const uint8_t *h_codes, int32_t stride, int64_t n_reads, uint8_t *h_bases2, uint8_t *h_nmask);
/* ---- contaminant passes (replaces rules `rm_phix` / `rm_human_ecoli`, rules/decontamination.smk:15-17,43-48: `bwa mem` against
 * the contaminants | `samtools view -f 12 -F 256` | `sort -n` | `bedtools bamtofastq`) ----
 * qm_sample_set_filter(on) before the first pairs (QM_EINVAL after them, or on a sample in rmdup / depth-cap mode, which in turn
 * refuse a filter-mode sample): the sample aligns and finishes its pairs as usual, the CIGAR stage included (a CIGAR overflow
 * unmaps a read), and its insert-size model is fixed as above; it runs no pileup, fills neither the count tensor (which stays
 * zero) nor the indel table, ignores qm_sample_set_baq and keeps no records across batches.  A kernel applies the rule's keep
 * test to each pair of every batch on the device: keep = (flag & 12) == 12 && !(flag & 256) on both records.
 * qm_sample_keep_host: h_keep[p] = 1 for each kept pair p of the LAST batch handed in (any entry above; n_pairs must be that
 * batch's pair count, QM_EINVAL otherwise), *h_n_kept (may be NULL) = their number.  n_pairs bytes come back, not the records.
 * Synchronous.  QM_EINVAL when the sample is not in filter mode. */
int  qm_sample_set_filter(qm_sample *s, int on);
int  qm_sample_keep_host(qm_sample *s, uint8_t *h_keep, int64_t n_pairs, int64_t *h_n_kept);
int32_t *qm_sample_counts(qm_sample *s);                          /* device pointer, planes [QM_NCH][l_pac] */
int  qm_sample_stats_sync(qm_sample *s, int64_t *n_pairs, int64_t *cells, void *stream);
int  qm_sample_counts_host(qm_sample *s, int32_t *h_rows /* [l_pac][QM_NCH] */);
/* the sample's indel alleles (see qm_indel below), sorted by (position, type, length, bases); synchronous */
struct qm_indel_table *qm_sample_indel_table(qm_sample *s);

/* ---- SNP calls from the count tensor (stands in for `bcftools call -p 0.01 --ploidy 1 -mv | bcftools view
 * -i 'INFO/DP>=10'`, rules/vcfcall.smk:116-117).  A threshold caller: a non-reference base b is called at a
 * position when raw depth (channel 14) >= min_dp, AD[b] >= min_alt and AD[b] >= min_af * sum(AD).  bcftools'
 * likelihood model and QUAL are outside the parity contract (SURVEY.md 8a10); QUAL here is a phred-scaled
 * Chernoff bound of the binomial error tail.  Output sorted by (position, alt).  Synchronous. */
typedef struct { int32_t min_dp, min_alt; float min_af; int32_t reserved; } qm_call_opt;
typedef struct {
    int32_t rid, pos;             /* 0-based position on contig rid */
    uint8_t ref, alt, pad[2];     /* base codes 0..3 */
    int32_t dp, ad_ref_f, ad_ref_r, ad_alt_f, ad_alt_r;
    float   qual, af;
} qm_call;                        /* 40 B */
void qm_call_opt_default(qm_call_opt *o);
int  qm_call_snps(qm_ctx *ctx, const qm_index *idx, const qm_call_opt *copt, const int32_t *d_counts, qm_call *d_calls,
                  int64_t max_calls, int64_t *h_n_calls, void *stream);
int  qm_sample_call_snps_host(qm_sample *s, const qm_call_opt *copt, qm_call *h_calls, int64_t max_calls, int64_t *n_calls);

/* ---- TP/FP/FN matcher (replaces the `fgrep -wf` / `fgrep -wvf` pipelines of
 * program/extract_TP_FP_SNPs.py:47-57 and the set arithmetic of scripts/caller_performance_compare.R:93-99) ----
 * key = pos << 8 | ref << 4 | alt (1-based VCF POS, base codes 0..3); CHROM is not part of the key, exactly
 * like the script's pattern "POS\t.\tREF\tALT".  call_flags[i] = 1 iff call key i occurs among the truth keys
 * (TP, else FP); truth_flags[j] = 1 iff truth key j occurs among the call keys (else FN).  d_truth_flags may be
 * NULL.  Asynchronous on `stream`. */
int qm_eval_match(qm_ctx *ctx, const uint64_t *d_call_keys, int64_t n_call, const uint64_t *d_truth_keys, int64_t n_truth,
                  uint8_t *d_call_flags, uint8_t *d_truth_flags, void *stream);
/* one sample's device-resident calls against the truth keys in one call: keys from the qm_call records, both membership
 * passes and the totals h_tp_fp_fn = {TP, FP, FN} (scripts/caller_performance_compare.R:93-99).  d_call_flags may be NULL.
 * Synchronous (24 bytes come back). */
int qm_eval_calls(qm_ctx *ctx, const qm_call *d_calls, int64_t n_call, const uint64_t *d_truth_keys, int64_t n_truth,
                  uint8_t *d_call_flags, int64_t h_tp_fp_fn[3], void *stream);
int qm_eval_match_host(qm_ctx *ctx, const uint64_t *h_call_keys, int64_t n_call, const uint64_t *h_truth_keys, int64_t n_truth,
                       uint8_t *h_call_flags, uint8_t *h_truth_flags /* may be NULL */);

/* ---- coordinate sort (replaces the ordering of `samtools sort`, rules/bwa.smk:17; comparator bam1_lt of samtools
 * bam_sort.c: (uint64)tid << 32 | (pos+1) << 1 | is_rev, unplaced (tid = -1) last, ties in input order; SURVEY.md A.7) ----
 * The key below orders records exactly like that comparator in as few bits as the reference needs: contig (unplaced
 * = n_contigs) above pos+1 above the strand bit.  The sort is a stable LSD radix sort of (key, record index) pairs;
 * records are not moved: the caller gathers through the permutation. */
#ifdef __CUDACC__
#define QM_INLINE_HD __host__ __device__
#else
#define QM_INLINE_HD
#endif
static inline QM_INLINE_HD int qm_sort_pos_bits(int64_t max_contig_len)
{
    int b = 1;
    while (((int64_t)1 << b) <= max_contig_len + 1) ++b;         /* pos + 1 <= max_contig_len */
    return b;
}
static inline QM_INLINE_HD int qm_sort_key_bits(int n_contigs, int pos_bits)
{
    int b = 1;
    while ((1 << b) <= n_contigs) ++b;                            /* contig codes 0..n_contigs */
    return b + pos_bits + 1;
}
static inline QM_INLINE_HD uint64_t qm_sort_key(int32_t rid, int32_t pos, int is_rev, int n_contigs, int pos_bits)
{
    return ((uint64_t)(uint32_t)(rid < 0 ? n_contigs : rid) << (pos_bits + 1)) | ((uint64_t)(uint32_t)(pos + 1) << 1) | (uint64_t)(is_rev != 0);
}
/* keys of device-resident records; *key_bits (may be NULL) receives the number of key bits in use */
int qm_aln_sort_keys(qm_ctx *ctx, const qm_index *idx, const qm_aln *d_alns, int64_t n, uint64_t *d_keys, int *key_bits, void *stream);
/* in place: d_keys sorted ascending (stable), d_vals[i] = input index of the record at sorted position i */
int qm_sort_pairs(qm_ctx *ctx, uint64_t *d_keys, uint32_t *d_vals, int64_t n, int key_bits, void *stream);
/* host keys in, permutation out; synchronous */
int qm_sort_keys_host(qm_ctx *ctx, const uint64_t *h_keys, int64_t n, int key_bits, uint32_t *h_perm);

/* page-locked host buffers for the driver (host<->device copies of qm_sample_add_pairs_host overlap the kernels) */
int  qm_host_alloc(qm_ctx *ctx, size_t bytes, void **out);
void qm_host_free(qm_ctx *ctx, void *p);

/* ---- duplicate removal (replaces `picard MarkDuplicates REMOVE_DUPLICATES=true`, rules/rmdup.smk:13-16, the step between
 * rule `bwa` and every caller; semantics SURVEY.md B.9) ----
 * Fully placed pairs are keyed by {contig, unclipped 5' coordinate, strand} of both ends; the pair with the highest sum of
 * base qualities >= 15 stays, ties go to the earliest pair of the input.  A read with an unplaced mate is a duplicate
 * whenever an end of a fully placed pair shares its {contig, unclipped 5' coordinate, strand}, otherwise the best such read
 * stays.  Duplicates get flag 0x400 (the pileup's read admission skips them).
 * qm_mark_duplicates: the records of one sample in n_chunks device chunks, input order.  Synchronous.
 * qm_sample_set_rmdup(on) before the first pairs: the sample keeps reads and records on the device and does not count;
 * qm_sample_rmdup_finish marks the duplicates over everything added and then counts the survivors;
 * qm_sample_kept_alns_host returns all records (input order) with their final flags. */
int qm_mark_duplicates(qm_ctx *ctx, int n_chunks, qm_aln *const *d_alns, const uint8_t *const *d_quals, const int32_t *strides,
                       const int32_t *const *d_lens, const int64_t *n_pairs, int64_t *h_n_dup_pairs, void *stream);
int qm_sample_set_rmdup(qm_sample *s, int on);
int qm_sample_rmdup_finish(qm_sample *s, int64_t *n_dup_pairs, void *stream);
int qm_sample_kept_alns_host(qm_sample *s, qm_aln *h_alns, int64_t max_records);

/* ---- depth cap (`bcftools mpileup -d N`, rules/vcfcall.smk:115 runs with bcftools' default; SURVEY.md A.8, 8f-2) ----
 * htslib's pileup iterator refuses a read whose start equals the position it is assembling while more than N reads are
 * buffered: an order-dependent rule, replayed here read by read over the records in BAM order (qm_depth_cap; d_drop[c][r] = 1
 * for a refused read).  OFF by default: at BASELINE depths the cap discards most of the sample (DESIGN.md 5).
 * qm_sample_set_max_depth(N > 0) before the first pairs: like rmdup mode the sample keeps reads and records on the device and
 * counts in qm_sample_finish, which marks duplicates (when rmdup is on), applies the cap to what is left and counts the rest;
 * qm_sample_rmdup_finish is qm_sample_finish for a sample in rmdup mode. */
int qm_depth_cap(qm_ctx *ctx, const qm_pileup_opt *po, int n_chunks, const qm_aln *const *d_alns, const int64_t *n_pairs, int max_depth,
                 uint8_t *const *d_drop, int64_t *h_n_dropped, void *stream);
int qm_sample_set_max_depth(qm_sample *s, int max_depth);
/* qm_sample_finish decides over this object's pairs only, even with a communicator set: a sample sharded over ranks finishes with
 * qm_sample_finish_comm (below). */
int qm_sample_finish(qm_sample *s, int64_t *n_dup_pairs, int64_t *n_capped_reads, void *stream);
/* base alignment quality for the sample's pileup (qm_baq_apply above): 0 = off (default, `-B`), 3 = extended BAQ as both mpileups of
 * the reference flow run it, 1 = plain BAQ; before the first pairs.  Works with the immediate and the deferred (rmdup / depth cap)
 * counting; duplicate marking keeps the reads' own qualities. */
int qm_sample_set_baq(qm_sample *s, int flag);

/* ---- duplicate marking and depth cap over a sample sharded across ranks ----
 * Both decisions split into an export and a decide step.  Every rank exports one small tuple per pair (duplicates) or per
 * admitted read (cap), tagged with a sample-wide id; the ranks all-gather the tuples; every rank runs the decision over the union
 * and applies it to its own records.  The decision sees identical data on every rank, so the result is the one of a single
 * device holding the whole sample, and every rank reaches the same verdict on an invalid union.
 * Pair ids must be unique across ranks (a pair's id is what its position in the sample is on one device: the running pair
 * offset; gaps are allowed).  Chunk c holds pairs pair_id0[c] .. pair_id0[c] + n_pairs[c] - 1.  Read ids are 2 * pair id + mate
 * and must fit in an int32 (pair ids below 2^30).
 * qm_dup_keys: one qm_dup_key per pair with a placed end (pairs without one are never duplicates and are left out), in no
 * particular order; d_out holds up to sum(n_pairs) records, *h_n_out receives the number written.  end0 / end1: the 31-bit codes of
 * the two ends of a fully placed pair, 0xffffffff for none.  Synchronous; QM_ELIMIT when an end code does not fit (as
 * qm_mark_duplicates).
 * qm_mark_duplicates_keys: d_all is the union of every rank's tuples (any order).  Orders it by pair id (a repeated id: QM_EINVAL,
 * nothing flagged), decides as qm_mark_duplicates with ties to the lowest pair id, and sets 0x400 on the records of the local
 * chunks only.  *h_n_dup_all: duplicate pairs of the whole union.  Synchronous.
 * qm_cap_keys: one qm_cap_key per read the pileup admits (po: min_mapq, count_orphans; reads flagged 0x400 are out), any order;
 * d_out holds up to 2 * sum(n_pairs) records.  Synchronous.
 * qm_depth_cap_keys: d_all is the union of every rank's cap tuples.  Orders it by read id (a repeated id: QM_EINVAL, nothing
 * written), then stably by key (BAM order, ties in read order), replays htslib's iterator on the host as qm_depth_cap and writes
 * the drop bytes of the local reads (d_drop[c]: 2 * n_pairs[c] bytes).  *h_n_dropped_all: reads dropped in the whole union.
 * Synchronous.
 * Memory per rank: the whole union of tuples plus its sort scratch on the device (about 150 bytes per pair of the sample for
 * duplicates, 70 per admitted read for the cap, the all-gather's buffers included) and 17 bytes per admitted read of the sample on the host for the replay. */
typedef struct {
    int64_t  pair_id;
    uint64_t key;                         /* the duplicate key: both ends of a fully placed pair, or the one placed end (bit 63) */
    uint32_t end0, end1;                  /* end codes of a fully placed pair; 0xffffffff = none */
    int32_t  score, pad;                  /* sum of base qualities >= 15 over the placed ends */
} qm_dup_key;
typedef struct {
    uint64_t key;                         /* contig << 33 | start << 1 | reverse */
    int32_t  read_id;                     /* 2 * pair id + mate */
    int32_t  end;                         /* end of the read's reference span (exclusive) */
} qm_cap_key;
int qm_dup_keys(qm_ctx *ctx, int n_chunks, const qm_aln *const *d_alns, const uint8_t *const *d_quals, const int32_t *strides,
                const int32_t *const *d_lens, const int64_t *n_pairs, const int64_t *pair_id0, qm_dup_key *d_out, int64_t *h_n_out,
                void *stream);
int qm_mark_duplicates_keys(qm_ctx *ctx, const qm_dup_key *d_all, int64_t n_all, int n_chunks, qm_aln *const *d_alns,
                            const int64_t *n_pairs, const int64_t *pair_id0, int64_t *h_n_dup_all, void *stream);
int qm_cap_keys(qm_ctx *ctx, const qm_pileup_opt *po, int n_chunks, const qm_aln *const *d_alns, const int64_t *n_pairs,
                const int64_t *pair_id0, qm_cap_key *d_out, int64_t *h_n_out, void *stream);
int qm_depth_cap_keys(qm_ctx *ctx, const qm_cap_key *d_all, int64_t n_all, int max_depth, int n_chunks, const int64_t *n_pairs,
                      const int64_t *pair_id0, uint8_t *const *d_drop, int64_t *h_n_dropped_all, void *stream);

/* ---- text pileup (replaces `samtools mpileup -f ref bam`, rules/vcfcall.smk:39; consumer: the VarScan rule) ----
 * One line per column covered by an admitted read: chrom, 1-based position, reference base, number of entries with base
 * quality >= min_bq, base string (. , ACGTN acgtn * ^X $ +nSEQ -nSEQ), quality string; SURVEY.md A.10.  Admission and
 * mate-overlap quality rewrite as qm_pileup_accumulate (BAQ off, no depth cap); reads enter a column in coordinate-sorted
 * order.  names[i] = name of contig i.  The text is left in library scratch on the device: *d_text is valid until the
 * next text-producing call on the context.  The _host form takes the sample's records / reads / qualities from host
 * memory; qm_mpileup_text_fetch copies the text of the last call out.  Synchronous. */
int qm_mpileup_text(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns, const uint8_t *d_codes,
                    const uint8_t *d_quals, int32_t stride, const int32_t *d_lens, int64_t n_pairs, const char *const *names,
                    const char **d_text, int64_t *h_bytes, void *stream);
int qm_mpileup_text_host(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *h_alns, const uint8_t *h_codes,
                         const uint8_t *h_quals, int32_t stride, const int32_t *h_lens, int64_t n_pairs, const char *const *names,
                         int64_t *h_bytes);
int qm_mpileup_text_fetch(qm_ctx *ctx, char *h_out, int64_t bytes);
/* the same with the order given: reads reach a column in the order of d_rank[r] (one int64 per read; a negative rank sorts after
 * every ranked read, and such a read must not be placed).  The ranked order must list the placed reads by contig, then position.
 * qm_bam_pairs.d_row_file is such an order: the reads of a coordinate-sorted BAM reach a column in file order, as in htslib. */
int qm_mpileup_text_ranked(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns, const uint8_t *d_codes,
                           const uint8_t *d_quals, int32_t stride, const int32_t *d_lens, int64_t n_pairs, const char *const *names,
                           const int64_t *d_rank, const char **d_text, int64_t *h_bytes, void *stream);

/* ---- BAM records in (the way in of rules `mpileup` / `bcftools`, rules/vcfcall.smk:39,115, which read {sample}.rmdup.bam) ----
 * d_bytes: the uncompressed record stream of a BAM (BGZF inflated); d_rec_off[i]: byte offset of record i's block_size field.
 * The records are the caller's selection, in file order, and must be valid: the library does not re-check them.  The driver
 * (qm_driver pileup) checks on the host: a CIGAR of at most QM_MAX_CIGAR operations besides H and without N or P, a query length
 * equal to l_seq, l_seq <= 512, SEQ and QUAL stored, contig and span inside the reference, coordinate order; and it leaves out the
 * records neither mpileup admits (flag 0x4, 0x100, 0x200 or 0x400, no CIGAR, no contig).
 * Each record becomes a read in the read-batch layout (qm_aln, codes 0..4 -- '=' and IUPAC codes are N -- and qualities at one
 * `stride`, lengths), a reverse-strand record turned back to the orientation it was sequenced in.  CIGAR '=' and 'X' become M, H
 * is dropped, neighbouring operations of one kind merge.  rid, pos, flag, mapq, mate_rid, mate_pos, tlen come from the record;
 * nm, score, sub from its NM, AS, XS tags (0 without); qb = 0, qe = l_seq.
 * Pairing: the two primary records of a name (one flagged 0x40, the other 0x80, neither 0x100 nor 0x800) are one pair, matched by
 * a 64-bit name hash and then byte for byte; the one that comes first in the file is row 2i.  Every other record (supplementary
 * records, a read whose mate is not among the records, single-end reads, a third primary record of a name) is a pair of its own
 * with an empty placeholder mate (flag 0x4, rid -1, no CIGAR, length 0).  Pair i is the i-th pair in the file order of its row 2i.
 * max_depth > 0: htslib's depth cap (qm_depth_cap) over the reads in FILE order -- the order the cap depends on -- under po;
 * d_drop then holds the verdict per row.  baq 1 / 3: d_quals are the qualities capped by base alignment quality (qm_baq_apply).
 * The layout lives in library scratch, valid until the next qm_bam_to_pairs* call on the context.
 * Limits: stride <= 512 (QM_ELIMIT), n_recs < 2^31 (QM_ELIMIT); QM_EINVAL on NULL pointers, stride < 1, baq not 0 / 1 / 3.
 * Device memory: about 2 * (150 + 2 * stride) bytes per record (file-order rows and pairing state, then the pair layout, a
 * third copy of the qualities with BAQ) plus the sort's scratch; the _host form stages the record stream (its size) and 8 bytes
 * per record.  Synchronous. */
typedef struct {
    int64_t  n_pairs;                   /* rows 2i / 2i + 1 of pair i, i < n_pairs                               */
    int32_t  stride, pad;
    const qm_aln  *d_alns;
    const uint8_t *d_codes, *d_quals;   /* with baq: the capped qualities                                        */
    const int32_t *d_lens;
    const int64_t *d_row_file;          /* index of each row's record among the n_recs handed in, -1 = placeholder */
    const uint8_t *d_drop;              /* max_depth > 0: 1 = the depth cap refuses the read; else NULL          */
    int64_t  n_capped;                  /* reads the cap refuses                                                 */
} qm_bam_pairs;
int qm_bam_to_pairs(qm_ctx *ctx, const qm_index *idx, const uint8_t *d_bytes, const int64_t *d_rec_off, int64_t n_recs, int32_t stride,
                    const qm_pileup_opt *po, int baq, int max_depth, qm_bam_pairs *out, void *stream);
int qm_bam_to_pairs_host(qm_ctx *ctx, const qm_index *idx, const uint8_t *h_bytes, int64_t n_bytes, const int64_t *h_rec_off, int64_t n_recs,
                         int32_t stride, const qm_pileup_opt *po, int baq, int max_depth, qm_bam_pairs *out);

/* ---- duplicate marking of a coordinate-sorted BAM (the rule `rmdup`, rules/rmdup.smk:13-16: picard MarkDuplicates
 * REMOVE_DUPLICATES=true on a sorted file; qm_driver rmdup) ----
 * d_bytes: the uncompressed record stream; d_rec_off[i]: byte offset of record i's block_size field, for EVERY record of the file in
 * file order.  The records must be well-formed (the library does not re-check them); N and P operations, any number of CIGAR
 * operations, any read length and a missing SEQ or QUAL are fine.  d_dup[i] = 1: record i is a duplicate.
 * The rule (dedup.cu's, SURVEY.md B.9, stated for a file):
 *  - units: the two primary records of a name (one 0x40, one 0x80, neither 0x100 nor 0x800, the only two such records of the
 *    name; qm_bam_to_pairs' pairing rule) are a pair unit; every other primary record is a lone unit.  The pairing runs over all
 *    records, 0x4, 0x200 and 0x400 included;
 *  - a record is placed when it lacks 0x4, has a contig id >= 0 and a CIGAR.  Its end is {contig, unclipped 5' coordinate,
 *    strand}: pos - (S and H at the start) forward, pos + reference span - 1 + (S and H at the end) reverse, the span counting
 *    M D N = X;
 *  - a unit with two placed ends gets a pair key, one with a single placed end a fragment key, one without is never a candidate.
 *    The score is the sum of the stored qualities >= 15 of the placed ends (a QUAL of '*' scores 0);
 *  - a unit's id is the file index of its end with the smaller {contig, unclipped 5' coordinate} (the earlier record on a tie), or
 *    of its one placed record; ties of the decision go to the lowest id, which is picard's read1IndexInFile (recalled, not
 *    checked against picard);
 *  - a duplicate unit loses its placed records; unplaced mates, secondary and supplementary records are never duplicates, and a
 *    0x400 flag in the input is ignored (picard's behaviour on sorted input as recalled).
 * *h_n_units: all units (picard's READ_PAIRS_EXAMINED as qm_driver reports it); *h_n_dup_units: duplicate units.
 * Limits: the 30-bit end code (16 contigs, contigs under 2^26 - 4096 bases, QM_ELIMIT when an end does not fit), n_recs < 2^31
 * (QM_ELIMIT).  Device memory: about 90 bytes per record for the records' state and tuples, plus the decision's 70 bytes per unit
 * with a placed end and the sorts' scratch; the _host form stages the record stream (its size) and 9 bytes per record.
 * The _host form reads the records from and writes the verdicts to host memory.  Synchronous. */
int qm_bam_mark_duplicates(qm_ctx *ctx, const uint8_t *d_bytes, const int64_t *d_rec_off, int64_t n_recs, uint8_t *d_dup, int64_t *h_n_units,
                           int64_t *h_n_dup_units, void *stream);
int qm_bam_mark_duplicates_host(qm_ctx *ctx, const uint8_t *h_bytes, int64_t n_bytes, const int64_t *h_rec_off, int64_t n_recs, uint8_t *h_dup,
                                int64_t *h_n_units, int64_t *h_n_dup_units);

/* ---- multi-GPU: the one collective of the path (north_star: "per-GPU int32 count tensors are merged with one NCCL allreduce
 * over NVLink"; SURVEY.md 8b, 8e).  Reads shard by pair index with no data-path exchange; what crosses GPUs is the count
 * tensor (one in-place integer sum per sample: order independent, bit-exact for any number of GPUs) and the 128 bytes of the
 * insert-size model, so that every rank pairs its reads against the same mem_pestat result (bwamem_pair.c).
 * NCCL is bound at run time (dlopen libnccl.so.2; inside a torch process that is torch's own copy): qm_comm_available() says
 * whether it could be.  Communicators: one process per GPU -- rank 0 calls qm_comm_unique_id, the host carries the 128 bytes
 * to the other ranks (torch.distributed, MPI, a file), every rank calls qm_comm_init_rank; or one process driving N GPUs --
 * qm_comm_init_all (what `qm_driver sample --gpus` does; comms[i] belongs to ctxs[i], call the collectives from one host
 * thread per GPU).  qm_counts_allreduce_nccl takes a caller-owned ncclComm_t instead.  The all-reduce is asynchronous on
 * `stream`; qm_pestat_bcast is synchronous. */
typedef struct qm_comm qm_comm;
int  qm_comm_available(void);
int  qm_comm_unique_id(uint8_t id[128]);
int  qm_comm_init_rank(qm_ctx *ctx, int n_ranks, int rank, const uint8_t id[128], qm_comm **out);
int  qm_comm_init_all(int n, qm_ctx *const *ctxs, qm_comm **comms);
void qm_comm_destroy(qm_comm *c);
int  qm_comm_rank(const qm_comm *c);
int  qm_comm_size(const qm_comm *c);
int  qm_counts_allreduce(qm_ctx *ctx, qm_comm *comm, int32_t *d_counts, int64_t n, void *stream);
int  qm_counts_allreduce_nccl(qm_ctx *ctx, void *nccl_comm /* ncclComm_t */, int32_t *d_counts, int64_t n, void *stream);
int  qm_pestat_bcast(qm_ctx *ctx, qm_comm *comm, qm_pestat pes[4], int root, void *stream);
/* every rank's `bytes` bytes at d_send, concatenated in rank order into d_recv on every rank (the sparse indel tables) */
int  qm_comm_allgather(qm_ctx *ctx, qm_comm *comm, const void *d_send, void *d_recv, size_t bytes, void *stream);
/* a sample spread over the communicator's ranks: rank r holds a contiguous range of the sample's pairs, rank 0 the range
 * that starts at pair 0 (its first batch at least min(sample, QM_PESTAT_PAIRS) pairs).  The insert-size model is then rank
 * 0's, broadcast once every rank has aligned its first batch (no rank aligns the prefix twice); qm_sample_allreduce_counts
 * sums the count tensors in place on every rank and merges the indel allele tables (each rank's records all-gathered and added
 * into every rank's table); synchronous.  Set the communicator before the first pairs; NULL clears. */
int  qm_sample_set_comm(qm_sample *s, qm_comm *comm);
int  qm_sample_allreduce_counts(qm_sample *s, void *stream);
/* Deferred counting (rmdup / depth cap) of a sample spread over the ranks of `comm`.  qm_sample_finish decides over this object's
 * pairs only, even when a communicator is set: a duplicate whose original lies on another rank stays unflagged there.
 * qm_sample_finish_comm decides over the whole sample: each rank exports its duplicate tuples (qm_dup_keys, ids = the pair_id0 its
 * pairs were added with), the ranks all-gather them (counts first, then the tuples padded to the largest count), every rank marks
 * its own records (qm_mark_duplicates_keys); the same for the cap tuples (qm_cap_keys, qm_depth_cap_keys); then each rank counts its
 * survivors.  Collective: every rank of `comm` calls it, with one host thread per GPU when one process drives several.  It does not
 * sum the counts: call qm_sample_allreduce_counts or qm_counts_allreduce next.  *n_dup_pairs and *n_capped_reads are sample-wide and
 * equal on every rank.  The communicator is an argument, not the sample's own (a one-process driver sets none on its samples).
 * Pair ids must be unique across ranks; memory per rank as for qm_mark_duplicates_keys / qm_depth_cap_keys.  A rank that fails
 * before the first all-gather (QM_ELIMIT from an export, out of memory) leaves the other ranks waiting in it, as with the other
 * collectives; errors of the decision (a repeated id) are reached by every rank alike.  Synchronous. */
int  qm_sample_finish_comm(qm_sample *s, qm_comm *comm, int64_t *n_dup_pairs, int64_t *n_capped_reads, void *stream);

/* ---- SNP truth set of a strain pair (replaces rule `nucmer`, rules/genome_diff.smk: `nucmer ref qry; show-snps -CTHlr
 * <(delta-filter -r -q delta)`; SURVEY.md 8a row a13; contract DESIGN.md 5c) ----
 * ref_idx: qm_index_build of the reference with k = opt->min_match (QM_EINVAL otherwise).  The query is h_qry_codes (0..3, contigs
 * concatenated, at most QM_MAX_CONTIGS, fewer than 2^30 bases).
 * Anchors are the maximal exact matches of at least min_match bases between either query strand and the reference that contain a
 * k-mer unique in the reference (it occurs once and its reverse complement never): nucmer's default --mumreference, in the form the
 * index answers.  They are chained into collinear clusters per (query contig, strand, reference contig) (max_gap, max_diag,
 * diag_factor), clusters of fewer than min_cluster anchored bases are dropped, clusters within break_len on both sequences are
 * merged, and every gap between consecutive anchors gets a global affine-gap alignment on the device; a gap whose score along its
 * columns falls more than break_len below its best ends the alignment there.  Each alignment is extended past its outermost
 * anchors with ksw_extend2 (qm_extend_batch; zdrop and band = break_len, windows of at most QM_EXT_MAX_QLEN query bases, again
 * while an extension reaches the end of its window), and the extended stretches are aligned globally.  delta-filter -r -q becomes
 * two heaviest chains (weight: matching columns = aligned length x identity), on reference then on query coordinates.
 * Rows (show-snps -CTHlr): one per substitution and per indel base, indels left-aligned, P1 kept on the reference base in front
 * of an insertion; rows at a position covered by more than one kept alignment are dropped (-C) unless QM_GDIFF_KEEP_AMBIGUOUS;
 * QM_GDIFF_NO_INDELS leaves the indel rows out (-I).  Rows come sorted by (reference contig, P1) (-r), alignments by reference
 * start.  QM_ELIMIT when max_rows / max_alns are too small; *n_rows / *n_alns then hold what is needed.  h_phase_ms (may be
 * NULL, else 5 doubles): milliseconds of anchors, clustering, gap alignment, end extension and rows.  Synchronous. */
typedef struct {
    int32_t min_match;            /* nucmer -l (20)                                                        */
    int32_t min_cluster;          /* -c (65): anchored bases a cluster needs                               */
    int32_t max_gap;              /* -g (90): longest gap between neighbouring anchors of a cluster        */
    int32_t break_len;            /* -b (200): longest gap bridged between clusters                        */
    float   diag_factor;          /* -d (0.12): diagonal difference / gap, above max_diag                  */
    int32_t max_diag;             /* -D (5): diagonal difference always allowed                            */
    int32_t match, mismatch;      /* gap DP and end extension: + match (>= 1), - mismatch (1, 4)            */
    int32_t gap_open, gap_extend; /* a gap of l bases costs gap_open + l * gap_extend (6, 1)               */
    int32_t flags;                /* QM_GDIFF_*                                                            */
    int32_t reserved[5];
} qm_gdiff_opt;
#define QM_GDIFF_NO_INDELS      1 /* show-snps -I */
#define QM_GDIFF_KEEP_AMBIGUOUS 2 /* show-snps without -C */
typedef struct {
    int32_t p1, p2;               /* 1-based reference / query position (query forward strand)              */
    int32_t buff, dist;           /* distance to the nearest other difference or alignment end; to the nearest sequence end */
    char    sub_r, sub_q;         /* A C G T, '.' on the gap side; sub_q on the aligned query strand        */
    int8_t  frm_r, frm_q;         /* 1; -1 for a query on the reverse strand                                */
    int32_t rid, qid;             /* reference / query contig                                              */
} qm_gdiff_row;                   /* 28 B */
typedef struct {
    int32_t rid, qid;
    int32_t rs, re;               /* 1-based first / last reference base                                   */
    int32_t qs, qe;               /* 1-based query positions aligned to rs / re (qs > qe on the reverse strand, as in a delta file) */
    int32_t strand;               /* 1 / -1 */
    int32_t edits, matches;       /* mismatching columns + indel bases; matching columns                   */
    int32_t pad;
} qm_gdiff_aln;                   /* 40 B */
void qm_gdiff_opt_default(qm_gdiff_opt *opt);
int  qm_genome_diff_host(qm_ctx *ctx, const qm_index *ref_idx, const uint8_t *h_qry_codes, int n_qry_contigs, const int64_t *h_qry_lens,
                         const qm_gdiff_opt *opt, qm_gdiff_row *h_rows, int64_t max_rows, int64_t *n_rows, qm_gdiff_aln *h_alns,
                         int64_t max_alns, int64_t *n_alns, double *h_phase_ms);

/* ---- stage timers: CUDA events recorded on the launching stream around every kernel group ----
 * stages: 0 seed+chain, 1 advance (extension state machine), 2 extend (ksw_extend2 kernels), 3 pair+CIGAR,
 * 4 pileup, 5 h2d, 6 d2h, 7 other, 8 mate rescue.  qm_profile_collect synchronises the device and returns + clears the totals;
 * launch counts are kept even when timing is disabled. */
#define QM_N_STAGES 9
int qm_profile_enable(qm_ctx *ctx, int on);
int qm_profile_collect(qm_ctx *ctx, double ms_out[QM_N_STAGES], int64_t launches_out[QM_N_STAGES]);

/* ---- synthetic inputs (SURVEY.md 8d): deterministic, index-addressable read-pair simulator ----
 * The reference ships no reads (data/PRJEB32127.txt lists ENA URLs; no network), so benchmark and
 * parity inputs are simulated from the bundled genomes.  Pair i is a pure function of (seed, i):
 * any shard can be generated independently, on the host or on the device, with identical bytes.
 * genome: base codes 0..3 of all source genomes, source s at [src_off[s], src_off[s]+src_len[s]);
 * src_cum[s] = floor(2^32 * cumulative weight share) (last = 2^32-1), weight = copies x length.
 * Output layout ("read batch", used by every later stage): reads 2i / 2i+1 are the mates of pair i,
 * codes[r*stride + j] in 0..4 (4 = N), quals[r*stride + j] = phred, stride >= read_len. */
typedef struct {
    uint64_t seed;
    int32_t  read_len;
    int32_t  ins_mean, ins_sd, ins_max;   /* insert size model N(mean, sd) clipped to [read_len, max] */
    int32_t  n_sources;
    int32_t  indel_ppm;                   /* indel events per 1e6 bases (cfg 5: 200)                  */
    int32_t  n_ppm;                       /* bases forced to N per 1e6 (1000)                         */
    int32_t  lowq_ppm;                    /* bases with Q2..Q12 per 1e6 (20000)                       */
    int32_t  reserved[3];
} qm_sim_params;

int qm_simulate_pairs_host(const qm_sim_params *p, const uint8_t *h_genome, const int64_t *src_off,
                           const int64_t *src_len, const uint32_t *src_cum, int64_t pair0, int64_t n_pairs,
                           int32_t stride, uint8_t *h_codes, uint8_t *h_quals, int32_t *h_src /* may be NULL */,
                           int64_t *h_pos /* may be NULL */);
int qm_simulate_pairs(qm_ctx *ctx, const qm_sim_params *p, const uint8_t *d_genome, const int64_t *h_src_off,
                      const int64_t *h_src_len, const uint32_t *h_src_cum, int64_t pair0, int64_t n_pairs,
                      int32_t stride, uint8_t *d_codes, uint8_t *d_quals, void *stream);

/* ---- measurement helper: whole-GPU issue rate of the DPX instruction the extension kernel leans on
 * (register-resident dependent chains of __viaddmax_s16x2_relu / __viaddmax_s32_relu on every SM).
 * Returns giga warp-lane instructions per second in *out_gops (packed: per 32-bit lane op).
 * kind: 0 = __viaddmax_s32_relu, 1 = __viaddmax_s16x2_relu, 2 = __vimax3_s32.  SURVEY.md 8d / BASELINE.md 2. */
int qm_dpx_peak_sync(qm_ctx *ctx, int kind, int iters, double *out_gops, double *out_ms);

#ifdef __cplusplus
}
#endif
#endif /* QUASIMODO_B200_H */
