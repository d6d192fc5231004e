// pipeline.cuh -- device-side views and internal task formats shared by the alignment kernels.
#pragma once
#include "common.cuh"
#include "fm_core.cuh"

// ---- reference index as kernels see it (passed by value) ----
struct IndexView {
    const uint8_t *refb;      // forward strand, one base code (0..3) per byte, contigs concatenated
    const uint4 *table;       // open addressing: {key lo, key hi, first, count}; empty = key all-ones; first = slot of the k-mer's
                              // occurrences in pos[], or, when count == 1, the position itself
    const uint32_t *pos;      // occurrence lists (ascending forward positions)
    const uint32_t *uniq;     // bit p: the k-mer starting at forward position p occurs exactly once in the reference
                              // and its reverse complement does not occur at all (both look-ups of a read k-mer equal
                              // to it are then known without touching the table)
    const uint64_t *ref2p;    // forward strand, 2 bits per base, base x at bits 2*((x+32)&31) of word (x+32)>>5: 32 pad bases in
                              // front, 64 behind, so that any 32-base window touching the reference can be fetched whole
    const uint32_t *uniqp;    // the uniq bitmap with the same padding: bit x+32 (pad bits are 0)
    const uint32_t *uniq2p;   // same layout: the k-mer starting at x occurs once, and its reverse complement occurs once too
                              // (inverted repeats): a read k-mer equal to it has exactly one hit per strand
    const uint32_t *cnteqp[3];// same layout: the k-mer starting at x and its reverse complement occur 2 / 3 / 4 times in total
                              // (repeats in a few copies): a read k-mer equal to it has exactly that many hits
    const uint32_t *bloom;    // Bloom filter over the canonical (min of k-mer and its reverse complement) reference k-mers,
    uint32_t bloom_bits;      // 3 hash functions; 0 bits = no filter (a reference of more than 128 M distinct k-mers)
    uint64_t mask;            // table size - 1
    int shift;                // 64 - log2(table size)
    int k, n_contigs;
    int64_t l_pac;
    int64_t off[QM_MAX_CONTIGS], len[QM_MAX_CONTIGS];
};

struct qm_index {
    IndexView v;
    void *d_refb = nullptr, *d_table = nullptr, *d_pos = nullptr, *d_uniq = nullptr, *d_bloom = nullptr, *d_ref2p = nullptr,
         *d_uniqp = nullptr, *d_uniq2p = nullptr, *d_cnteqp[3] = {nullptr, nullptr, nullptr};
    int64_t n_kmers = 0, n_unique = 0, table_size = 0;
    // bwa's FM-index of the same genome (fmindex.cu), when attached: the seeds then can be bwa's own (QM_F_FM_SEEDS)
    bool have_fm = false;
    FmView fm = {};
    void *d_fm_bwt = nullptr, *d_fm_sa = nullptr;
    int64_t fm_words = 0;                                 // uint32 words of the .bwt behind its 40-byte header (qm_index_fm_export)
    int fm_device = -1;
};

static __device__ __forceinline__ int qm_ref_base(const IndexView &V, int64_t x)
{   // bwa's doubled coordinates: [l_pac, 2 l_pac) is the reverse complement strand
    return x < V.l_pac ? V.refb[x] : 3 - V.refb[2 * V.l_pac - 1 - x];
}
static __device__ __forceinline__ int qm_pos2rid(const IndexView &V, int64_t fpos)
{
    int r = -1;
    for (int c = 0; c < V.n_contigs; ++c)
        if (fpos >= V.off[c] && fpos < V.off[c] + V.len[c]) r = c;
    return r;
}
// the three bit positions of a canonical k-mer in a filter of `bits` bits (same on host and device)
static __host__ __device__ __forceinline__ void qm_bloom_pos(uint64_t canon, uint32_t bits, uint32_t p[3])
{
    const uint64_t h = canon * 0x9E3779B97F4A7C15ull;
    const uint32_t a = (uint32_t)(h >> 32), b = (uint32_t)h, c = a ^ (b >> 9) ^ (b << 23);
    p[0] = (uint32_t)(((uint64_t)a * bits) >> 32);
    p[1] = (uint32_t)(((uint64_t)b * bits) >> 32);
    p[2] = (uint32_t)(((uint64_t)c * bits) >> 32);
}
constexpr uint32_t kBloomMinBytes = 208 * 1024, kBloomMaxBytes = 256u << 20;      // the seeding filter: 16 bits per k-mer between these
static __device__ __forceinline__ bool qm_idx_lookup(const IndexView &V, uint64_t key, uint32_t &first, uint32_t &cnt)
{
    uint64_t h = (key * 0x9E3779B97F4A7C15ull) >> V.shift;
    for (;;) {
        const uint4 e = __ldg(&V.table[h]);
        const uint64_t kk = (uint64_t)e.x | ((uint64_t)e.y << 32);
        if (kk == key) { first = e.z; cnt = e.w; return true; }
        if (kk == ~0ull) return false;
        h = (h + 1) & V.mask;
    }
}

// the same look-up when the caller has fetched the key's first slot already (slot h, entry e)
static __device__ __forceinline__ bool qm_idx_lookup_from(const IndexView &V, uint64_t key, uint64_t h, uint4 e, uint32_t &first, uint32_t &cnt)
{
    for (;;) {
        const uint64_t kk = (uint64_t)e.x | ((uint64_t)e.y << 32);
        if (kk == key) { first = e.z; cnt = e.w; return true; }
        if (kk == ~0ull) return false;
        h = (h + 1) & V.mask;
        e = __ldg(&V.table[h]);
    }
}

// orientation class (FF FR RF RR) and distance of two hits in doubled coordinates (bwamem_pair.c mem_infer_dir)
static __device__ __forceinline__ int qm_infer_dir(int64_t l_pac, int64_t b1, int64_t b2, int64_t *dist)
{
    const int r1 = (b1 >= l_pac), r2 = (b2 >= l_pac);
    const int64_t p2 = r1 == r2 ? b2 : (l_pac << 1) - 1 - b2;
    *dist = p2 > b1 ? p2 - b1 : b1 - p2;
    return (r1 == r2 ? 0 : 1) ^ (p2 > b1 ? 0 : 3);
}


// ---- mem_sort_dedup_patch without mem_patch_reg (stable sorts) ----
__device__ inline int qm_sort_dedup(const qm_opt &o, int n, qm_reg *a)
{
    if (n <= 1) return n;
    for (int i = 1; i < n; ++i) { const qm_reg x = a[i]; int j = i - 1; while (j >= 0 && a[j].re > x.re) { a[j + 1] = a[j]; --j; } a[j + 1] = x; }
    for (int i = 1; i < n; ++i) {
        qm_reg *p = &a[i];
        if (p->rid != a[i - 1].rid || p->rb >= a[i - 1].re + o.max_chain_gap) continue;
        for (int j = i - 1; j >= 0 && p->rid == a[j].rid && p->rb < a[j].re + o.max_chain_gap; --j) {
            qm_reg *q = &a[j];
            if (q->qe == q->qb) continue;
            const int64_t orr = q->re - p->rb;
            const int64_t oq = q->qb < p->qb ? q->qe - p->qb : p->qe - q->qb;
            const int64_t mr = q->re - q->rb < p->re - p->rb ? q->re - q->rb : p->re - p->rb;
            const int64_t mq = q->qe - q->qb < p->qe - p->qb ? q->qe - q->qb : p->qe - p->qb;
            if (orr > o.mask_level_redun * mr && oq > o.mask_level_redun * mq) {
                if (p->score < q->score) { p->qe = p->qb; break; }
                else q->qe = q->qb;
            }
        }
    }
    int m = 0;
    for (int i = 0; i < n; ++i) if (a[i].qe > a[i].qb) { if (m != i) a[m] = a[i]; ++m; }
    n = m;
    for (int i = 1; i < n; ++i) {
        const qm_reg x = a[i];
        int j = i - 1;
        while (j >= 0 && !(a[j].score > x.score || (a[j].score == x.score && (a[j].rb < x.rb || (a[j].rb == x.rb && a[j].qb <= x.qb))))) { a[j + 1] = a[j]; --j; }
        a[j + 1] = x;
    }
    for (int i = 1; i < n; ++i)
        if (a[i].score == a[i - 1].score && a[i].rb == a[i - 1].rb && a[i].qb == a[i - 1].qb) a[i].qe = a[i].qb;
    m = n ? 1 : 0;
    for (int i = 1; i < n; ++i) if (a[i].qe > a[i].qb) { if (m != i) a[m] = a[i]; ++m; }
    return m;
}


// ---- internal extension task (superset of qm_ext_task) ----
#define QM_EXTI_INDIRECT 0x100u   // target = reference bases at doubled coordinate t0 + i*tstep
struct ExtTaskI {
    const uint8_t *q;             // query base j = q[j*qstep]
    const uint8_t *t;             // direct target bytes (when !INDIRECT)
    int64_t t0;
    int32_t qstep, tstep;
    int32_t qlen, tlen, h0, w, end_bonus;
    uint32_t flags;
    int32_t pad[2];
};                                // 64 B

struct ExtParams {
    int a, b, o_del, e_del, o_ins, e_ins, zdrop;
};
static inline ExtParams qm_ext_params(const qm_opt *o)
{
    ExtParams P = {o->a, o->b, o->o_del, o->e_del, o->o_ins, o->e_ins, o->zdrop};
    return P;
}

constexpr int kExtClasses = 10;   // query-length classes: 16-wide up to 128 (thread-per-task kernel, shared memory sized per
                                  // class), <= 256 (thread-per-task), <= 511 (warp-per-task only)
constexpr int kExtCtr = 16;       // slots per counter array (>= kExtClasses)
static __host__ __device__ __forceinline__ int qm_ext_class(int qlen)
{
    return qlen <= 128 ? (qlen <= 0 ? 0 : (qlen - 1) >> 4) : qlen <= 256 ? 8 : 9;
}

// sort key of a round's extension tasks: query length (9 bits: the classes are ranges of it), rows / 4 (8 bits), seed score / 2
// (7 bits) -- tasks that agree in all three run the same rectangle of cells
constexpr int kExtSortKeyBits = 24;
static __host__ __device__ __forceinline__ uint64_t qm_ext_sort_key(int qlen, int tlen, int h0)
{
    const int q = qlen < 0 ? 0 : qlen > 511 ? 511 : qlen, t = tlen < 0 ? 0 : (tlen >> 2) > 255 ? 255 : tlen >> 2, h = h0 < 0 ? 0 : (h0 >> 1) > 127 ? 127 : h0 >> 1;
    return (uint64_t)q << 15 | (uint64_t)t << 7 | (uint64_t)h;
}

// Launch the per-class extension kernels.  lists: [kExtClasses][list_stride] task indices, or (h_list_off given) ONE array in
// which class c starts at h_list_off[c] (the round's tasks sorted by query length, rows and seed score); h_counts may be
// NULL (unknown on the host: persistent grids sized for the SM count) or the 5 class counts.
// one class (0..8) on the thread-per-task kernel; h_count < 0: unknown on the host
// bytes: the caller guarantees h0 + qlen*a <= 255 for every task of the list (eh[] held in bytes, see extend2.cu)
int qm_ext2_launch_class(qm_ctx *ctx, int cls, const ExtParams &P, const IndexView &V, const ExtTaskI *d_tasks,
                         const int *d_list, const int *d_counts, int *d_cursors, int h_count,
                         qm_ext_result *d_out, cudaStream_t st, bool bytes = false);
// two tasks per thread in the halves of s16x2 words (extend3.cu), classes 0..8; tasks it cannot hold (scores above 255) are
// appended to the class's fallback list d_fb_lists[cls][.] (count d_fb_ctr[cls]) for a scalar kernel
bool qm_ext3_scores_ok(const ExtParams &P);
int qm_ext3_launch_class(qm_ctx *ctx, int cls, const ExtParams &P, const IndexView &V, const ExtTaskI *d_tasks,
                         const int *d_list, const int *d_counts, int *d_cursors, int h_count,
                         qm_ext_result *d_out, int *d_fb_list, int *d_fb_ctr, cudaStream_t st);
// d_fb_lists: [kExtClasses][list_stride] ints, d_fb_ctr: 2 * kExtCtr ints zeroed by the caller (fallback counts,
// then fallback cursors); both NULL: the paired kernel is not used
int qm_ext_launch_classes(qm_ctx *ctx, const ExtParams &P, const IndexView &V, const ExtTaskI *d_tasks,
                          const int *d_lists, int64_t list_stride, const int *d_counts, int *d_cursors,
                          const int *h_counts, qm_ext_result *d_out, int *d_fb_lists, int *d_fb_ctr, cudaStream_t st,
                          bool scores_fit_bytes = false, const int64_t *h_list_off = nullptr);

// internal (sort.cu): the ids of a union of exported tuples sorted stably over the bits in use, d_perm = input positions;
// QM_EINVAL on a negative id.  Synchronous.
int qm_sort_ids(qm_ctx *ctx, uint64_t *d_ids, uint32_t *d_perm, int64_t n, const char *who, cudaStream_t st);

// duplicate marking (dedup.cu, bamdup.cu).  An end is {contig, unclipped 5' coordinate + QM_DUP_COORD_BIAS} as a 30-bit code
// (4 bits of contig, 26 of coordinate; the bias admits clipped bases before the contig's start), times 2, plus 1 for the reverse
// strand; QM_DUP_NO_END = no placed end.  qm_dup_tuple: the tuple of a unit with placed ends e0 (score s0) and / or e1 (score s1)
#define QM_DUP_NO_END 0xffffffffu
#define QM_DUP_COORD_BIAS 4096
__device__ __forceinline__ qm_dup_key qm_dup_tuple(int64_t id, bool p0, uint32_t e0, int s0, bool p1, uint32_t e1, int s1)
{
    qm_dup_key t;
    t.pair_id = id;
    t.end0 = t.end1 = QM_DUP_NO_END;
    t.pad = 0;
    if (p0 && p1) {
        if (e1 < e0) { const uint32_t u = e0; e0 = e1; e1 = u; }
        t.key = ((uint64_t)(e0 >> 1) << 32) | ((uint64_t)(e1 >> 1) << 2) | (uint64_t)((e0 & 1) << 1 | (e1 & 1));
        t.end0 = e0; t.end1 = e1;
        t.score = s0 + s1;
    } else {
        t.key = (1ull << 63) | (uint64_t)(p0 ? e0 : e1);
        t.score = p0 ? s0 : s1;
    }
    return t;
}
// dedup.cu: the decision over a union of tuples.  *d_ids = the ids sorted, (*d_dup)[k] = 1 when the unit of id (*d_ids)[k] is a
// duplicate (scratch 15, valid until the next decision on the context); a repeated id is QM_EINVAL.  Synchronous.
int qm_dup_decide(qm_ctx *ctx, const qm_dup_key *d_all, int64_t n_all, const uint64_t **d_ids, const uint8_t **d_dup, int64_t *h_n_dup,
                  cudaStream_t st);

// bamin.cu: qm_bam_to_pairs with the name hash cut to hash_bits bits (tests: pairing through colliding hashes)
extern "C" int qm_bam_to_pairs_hashbits(qm_ctx *ctx, const qm_index *idx, const uint8_t *d_bytes, const int64_t *d_rec_off, int64_t n_recs,
                                        int32_t stride, const qm_pileup_opt *po, int baq, int max_depth, int hash_bits, qm_bam_pairs *out,
                                        void *stream);

// bamdup.cu: qm_bam_mark_duplicates with the name hash cut to hash_bits bits (tests: pairing through colliding hashes)
extern "C" int qm_bam_mark_duplicates_hashbits(qm_ctx *ctx, const uint8_t *d_bytes, const int64_t *d_rec_off, int64_t n_recs, int hash_bits,
                                               uint8_t *d_dup, int64_t *h_n_units, int64_t *h_n_dup_units, void *stream);

// sample.cu: packed reads (2 bits per base + N flags) -> one code byte per base, rows [0, n_reads)
cudaError_t qm_unpack_reads_launch(const uint8_t *d_bases2, const uint8_t *d_nmask, int stride, int stride_p, int stride_m, int64_t n_reads,
                                   uint8_t *d_codes, cudaStream_t st);

// pair.cu / rescue.cu: the paired stage with one insert-size model per chunk of the batch (qm_sample_set_chunks).  Models are
// 4 qm_pestat each; d_model_of[p] is pair p's model (NULL: model 0 for every pair); d_pes NULL: h_pes is uploaded.
extern "C" int qm_pestat_chunks(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const qm_reg *d_regs, const int32_t *d_n_regs,
                                const int64_t *h_start, int n_chunks, const int32_t **d_model_of, const qm_pestat **d_pes, qm_pestat *h_pes,
                                void *stream);
extern "C" int qm_mate_rescue_models(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride,
                                     const int32_t *d_lens, int64_t n_pairs, qm_reg *d_regs, int32_t *d_n_regs, const qm_pestat *h_pes,
                                     int n_models, const qm_pestat *d_pes, const int32_t *d_model_of, int64_t *d_stats, void *stream);
extern "C" int qm_pair_finish_models(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride,
                                     const int32_t *d_lens, int64_t n_pairs, int64_t pair_id0, qm_reg *d_regs, int32_t *d_n_regs,
                                     const qm_pestat *h_pes, int n_models, const qm_pestat *d_pes, const int32_t *d_model_of, qm_aln *d_alns,
                                     void *stream);
