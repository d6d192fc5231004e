// sample.cu -- one sample end to end on one device: the compute of the reference's `bwa` rule
// (rules/bwa.smk:15 `bwa mem -k 31 ref r1 r2`) followed by the counting of its `bcftools` / `mpileup`
// rules (rules/vcfcall.smk:39,115) for one {sample}.{ref_name}, fed batch by batch.
//
// A qm_sample owns the int32 count tensor [QM_NCH][l_pac] of the sample and chunk-sized scratch (regions,
// alignment records).  Pairs are processed in chunks of kChunkPairs: seeding/chaining -> extension rounds ->
// pairing/CIGAR -> pileup, all on the caller's stream (device entry) or on the context's compute stream with
// the next chunk's host->device copy running on the copy stream (host entry).  By default the insert-size model
// (bwa's per-chunk mem_pestat) is fixed ONCE per sample from the first min(n, QM_PESTAT_PAIRS) pairs handed in -- or
// set by the caller (multi-GPU: rank 0's model is broadcast) -- so that results do not depend on how the
// pair stream is split into batches or across GPUs (SURVEY.md 8e).  In per-chunk mode (qm_sample_set_chunks) the
// caller names bwa's input chunks instead and every chunk is paired against its own model, as bwa mem does; the
// internal chunks are then cut at those chunks' ends, so a model never depends on the batching either.
#include <stdlib.h>
#include <vector>
#include <thread>
#include <algorithm>
#include "pipeline.cuh"

namespace {
constexpr int64_t kChunkPairs = QM_CHUNK_MAX_PAIRS;
constexpr int64_t kPestatPairs = QM_PESTAT_PAIRS;
constexpr int kCopyParts = 8;
}

struct qm_sample {
    qm_ctx *ctx = nullptr;
    const qm_index *idx = nullptr;
    qm_opt opt;
    qm_pileup_opt popt;
    int32_t *d_counts = nullptr;
    qm_indel_table *indels = nullptr;             // sparse indel alleles next to the dense counts
    int64_t *d_cells = nullptr;
    qm_reg *d_regs = nullptr;
    int32_t *d_n_regs = nullptr;
    qm_aln *d_alns = nullptr;
    uint8_t *d_stage[2] = {nullptr, nullptr};     // host-entry staging: codes | quals | lens, double buffered
    size_t stage_cap = 0;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_quals[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
    cudaEvent_t ev_part[2][kCopyParts] = {};      // pieces of a chunk's bases (see qm_ctx::se_part_ev)
    bool have_pes = false;
    qm_pestat pes[4];
    qm_comm *comm = nullptr;                      // multi-GPU: model broadcast from rank 0, counts all-reduced (qm_sample_set_comm)
    int64_t n_pairs = 0;
    // duplicate removal (qm_sample_set_rmdup): every chunk's reads and records stay on the device, counting waits for
    // qm_sample_rmdup_finish
    bool rmdup = false;
    int max_depth = 0;                            // > 0: `bcftools mpileup -d` depth cap (qm_sample_set_max_depth): deferred counting too
    int baq = 0;                                  // 1 / 3: base alignment quality (plain / extended) caps the qualities the pileup sees (qm_sample_set_baq)
    bool rmdup_finished = false;                  // qm_sample_rmdup_finish has run: no more pairs, no second finish until a reset
    // filter mode (qm_sample_set_filter): align and finish pairs, count nothing; the keep rule's byte per pair of the last batch
    // (qm_sample_keep_host) lands in d_keep, the number of kept pairs in d_n_kept
    bool filter = false;
    uint8_t *d_keep = nullptr;
    unsigned long long *d_n_kept = nullptr;
    int64_t keep_cap = 0, last_n = -1;
    struct Kept { uint8_t *codes, *quals; int32_t *lens; qm_aln *alns; int64_t n; int32_t stride; int64_t pair0; };   // pair0: id of the first pair
    std::vector<Kept> kept;
    // per-chunk mode (qm_sample_set_chunks): the next add call's chunk sizes in pairs, and the models of the last call's chunks
    bool chunked = false;
    std::vector<int64_t> next_chunks;
    std::vector<qm_pestat> chunk_pes;
};

namespace {

// Packed read input (qm_sample_add_pairs_host_packed): 2 bits per base (base j of a read at bits 2 (j & 3) of byte j >> 2 of its
// row) + 1 bit per base "this is an N" (bit j & 7 of byte j >> 3).  One thread writes four unpacked base codes as one word.
__global__ void __launch_bounds__(256)
unpack_reads_kernel(const uint8_t *__restrict__ bases2, const uint8_t *__restrict__ nmask, int stride, int stride_p, int stride_m,
                    int64_t n_reads, uint8_t *__restrict__ codes)
{
    const int groups = (stride + 3) >> 2;
    const int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (t >= n_reads * groups) return;
    const int64_t r = t / groups;
    const int g = (int)(t - r * groups);
    const unsigned b = bases2[r * stride_p + g];
    const unsigned m = nmask[r * stride_m + (g >> 1)] >> ((g & 1) << 2);
    uint8_t c[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) c[k] = (m >> k) & 1u ? 4 : (uint8_t)((b >> (2 * k)) & 3u);
    uint8_t *o = codes + r * stride + 4 * g;
    if (4 * g + 3 < stride && (((uintptr_t)o) & 3u) == 0) *(uint32_t *)o = (uint32_t)c[0] | (uint32_t)c[1] << 8 | (uint32_t)c[2] << 16 | (uint32_t)c[3] << 24;
    else for (int k = 0; k < 4 && 4 * g + k < stride; ++k) o[k] = c[k];
}

}  // namespace

cudaError_t qm_unpack_reads_launch(const uint8_t *d_bases2, const uint8_t *d_nmask, int stride, int stride_p, int stride_m, int64_t n_reads,
                                   uint8_t *d_codes, cudaStream_t st)
{
    if (n_reads <= 0) return cudaSuccess;
    const int64_t work = n_reads * ((stride + 3) >> 2);
    unpack_reads_kernel<<<(unsigned)((work + 255) / 256), 256, 0, st>>>(d_bases2, d_nmask, stride, stride_p, stride_m, n_reads, d_codes);
    return cudaGetLastError();
}

namespace {

// rules/decontamination.smk:15-17,43-48 (`samtools view -f 12 -F 256` on the records of a pair, then `bedtools bamtofastq`, which
// re-emits a pair only when both of its records passed): keep[p] = 1 iff both records are unmapped with an unmapped mate and neither
// is secondary.  One thread per pair; the warp's kept pairs go to *n_kept in one atomic.
__global__ void __launch_bounds__(256)
keep_pairs_kernel(const qm_aln *__restrict__ alns, int64_t n_pairs, uint8_t *__restrict__ keep, unsigned long long *__restrict__ n_kept)
{
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    bool k = false;
    if (p < n_pairs) {
        const unsigned f0 = alns[2 * p].flag, f1 = alns[2 * p + 1].flag;
        k = (f0 & 12u) == 12u && !(f0 & 256u) && (f1 & 12u) == 12u && !(f1 & 256u);
        keep[p] = (uint8_t)k;
    }
    const unsigned b = __ballot_sync(0xffffffffu, k);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(n_kept, (unsigned long long)__popc(b));
}

// start of a batch in filter mode: room for its keep bytes, the kept count zeroed on the batch's stream
int filter_begin(qm_sample *s, int64_t n_pairs, cudaStream_t st)
{
    if (!s->filter) return QM_OK;
    qm_ctx *ctx = s->ctx;
    if (n_pairs > s->keep_cap) {
        QM_CUDA(ctx, cudaDeviceSynchronize());      // the last batch may still be writing the old buffer on another stream
        QM_CUDA(ctx, cudaFree(s->d_keep));
        s->d_keep = nullptr; s->keep_cap = 0;
        QM_CUDA(ctx, cudaMalloc(&s->d_keep, (size_t)n_pairs));
        s->keep_cap = n_pairs;
    }
    QM_CUDA(ctx, cudaMemsetAsync(s->d_n_kept, 0, sizeof(unsigned long long), st));
    s->last_n = n_pairs;
    return QM_OK;
}

// The internal chunks of an add call of n_pairs pairs: [starts[k], starts[k] + sizes[k]), at most kChunkPairs each.  In per-chunk
// mode they hold whole bwa chunks (bwa chunks bwa0[k] .. bwa0[k + 1] - 1 of s->next_chunks), which are taken over here.
int plan_chunks(qm_sample *s, int64_t n_pairs, std::vector<int64_t> &starts, std::vector<int64_t> &sizes, std::vector<int64_t> &bwa,
                std::vector<int> &bwa0)
{
    starts.clear(); sizes.clear(); bwa.clear(); bwa0.clear();
    if (!s->chunked) {
        for (int64_t p0 = 0; p0 < n_pairs; p0 += kChunkPairs) { starts.push_back(p0); sizes.push_back(std::min(kChunkPairs, n_pairs - p0)); }
        return QM_OK;
    }
    bwa.swap(s->next_chunks);
    s->next_chunks.clear();
    s->chunk_pes.clear();
    int64_t tot = 0;
    for (int64_t c : bwa) tot += c;
    if (tot != n_pairs)
        return qm_fail(s->ctx, QM_EINVAL, "per-chunk mode: the chunk sizes given (qm_sample_set_chunks) add up to %lld pairs, the call has %lld",
                       (long long)tot, (long long)n_pairs);
    int64_t p0 = 0;
    for (size_t c = 0; c < bwa.size();) {
        bwa0.push_back((int)c);
        int64_t n = 0;
        while (c < bwa.size() && n + bwa[c] <= kChunkPairs) n += bwa[c++];
        starts.push_back(p0); sizes.push_back(n);
        p0 += n;
    }
    bwa0.push_back((int)bwa.size());
    return QM_OK;
}

// the qualities the pileup sees: the reads' own, or (qm_sample_set_baq) capped by their base alignment quality
int sample_pileup_quals(qm_sample *s, const qm_aln *alns, const uint8_t *d_codes, const uint8_t *d_quals, int32_t stride, const int32_t *d_lens,
                        int64_t n_reads, cudaStream_t st, const uint8_t **out)
{
    *out = d_quals;
    if (!s->baq || n_reads == 0) return QM_OK;
    void *p = nullptr;
    int rc = qm_scratch_reserve(s->ctx, 30, (size_t)n_reads * stride, &p);
    if (rc) return rc;
    rc = qm_baq_apply(s->ctx, s->idx, &s->popt, alns, d_codes, d_quals, stride, d_lens, n_reads, s->baq, (uint8_t *)p, st);
    if (rc) return rc;
    *out = (const uint8_t *)p;
    return QM_OK;
}

// quals_ready (may be NULL): event after which d_quals is valid; only the pileup reads the qualities, so their copy
// may still be in flight while the reads are being aligned
// keep_off: the chunk's first pair within its batch (filter mode: where its keep bytes go)
// bwa_sizes (per-chunk mode, NULL otherwise): the sizes of the n_bwa bwa chunks that make up these n pairs
int sample_chunk(qm_sample *s, const uint8_t *d_codes, const uint8_t *d_quals, int32_t stride, const int32_t *d_lens,
                 int64_t n, int64_t pair_id0, int64_t keep_off, qm_aln *d_alns_out, cudaStream_t st, cudaEvent_t quals_ready = nullptr,
                 const int64_t *bwa_sizes = nullptr, int n_bwa = 0)
{
    qm_ctx *ctx = s->ctx;
    // the pileup stages a pair's reads in 512-byte rows and would leave longer reads out of the counts without a word
    if (stride > 512) return qm_fail(ctx, QM_ELIMIT, "rows of %d bases: reads longer than 512 bases are not supported", stride);
    if ((s->rmdup || s->max_depth > 0) && s->rmdup_finished)
        return qm_fail(ctx, QM_EINVAL, "pairs added after qm_sample_rmdup_finish: reset the sample first");
    int rc = qm_align_se(ctx, s->idx, &s->opt, d_codes, stride, d_lens, 2 * n, s->d_regs, s->d_n_regs, s->d_cells, st);
    if (rc) return rc;
    qm_aln *alns = d_alns_out ? d_alns_out : s->d_alns;
    if (bwa_sizes && !s->have_pes) {
        // per-chunk mode without a given model (-I): mem_pestat over every pair of each chunk, each pair against its chunk's model
        std::vector<int64_t> start((size_t)n_bwa + 1, 0);
        for (int c = 0; c < n_bwa; ++c) start[(size_t)c + 1] = start[(size_t)c] + bwa_sizes[c];
        std::vector<qm_pestat> pes((size_t)n_bwa * 4);
        const int32_t *d_model_of = nullptr;
        const qm_pestat *d_pes = nullptr;
        rc = qm_pestat_chunks(ctx, s->idx, &s->opt, s->d_regs, s->d_n_regs, start.data(), n_bwa, &d_model_of, &d_pes, pes.data(), st);
        if (rc) return rc;
        s->chunk_pes.insert(s->chunk_pes.end(), pes.begin(), pes.end());
        rc = qm_pair_finish_models(ctx, s->idx, &s->opt, d_codes, stride, d_lens, n, pair_id0, s->d_regs, s->d_n_regs, pes.data(), n_bwa, d_pes,
                                   d_model_of, alns, st);
        if (rc) return rc;
    } else {
        if (!s->have_pes) {
            // one model per sample.  With a communicator it is rank 0's (the rank that holds the sample's first pairs), broadcast:
            // the other ranks have aligned their own first chunk meanwhile and only wait for 128 bytes.
            const bool root = !s->comm || qm_comm_rank(s->comm) == 0;
            if (root) {
                rc = qm_pestat_sync(ctx, s->idx, &s->opt, s->d_regs, s->d_n_regs, n < kPestatPairs ? n : kPestatPairs, s->pes, st);
                if (rc) return rc;
            }
            if (s->comm && qm_comm_size(s->comm) > 1) {
                rc = qm_pestat_bcast(ctx, s->comm, s->pes, 0, st);
                if (rc) return rc;
            }
            s->have_pes = true;
        }
        rc = qm_pair_finish(ctx, s->idx, &s->opt, d_codes, stride, d_lens, n, pair_id0, s->d_regs, s->d_n_regs, s->pes, alns, st);
        if (rc) return rc;
    }
    if (s->filter) {
        keep_pairs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(alns, n, s->d_keep + keep_off, s->d_n_kept);
        QM_CUDA(ctx, cudaGetLastError());
        s->n_pairs += n;
        return QM_OK;
    }
    if (s->rmdup || s->max_depth > 0) {
        // keep the chunk for qm_sample_rmdup_finish: duplicates are a property of the whole sample
        qm_sample::Kept k = {nullptr, nullptr, nullptr, nullptr, n, stride, pair_id0};
        const size_t sb = (size_t)2 * n * stride;
        cudaError_t e;
        if ((e = cudaMalloc(&k.codes, sb)) != cudaSuccess || (e = cudaMalloc(&k.quals, sb)) != cudaSuccess ||
            (e = cudaMalloc(&k.lens, (size_t)2 * n * 4)) != cudaSuccess || (e = cudaMalloc(&k.alns, (size_t)2 * n * sizeof(qm_aln))) != cudaSuccess) {
            cudaFree(k.codes); cudaFree(k.quals); cudaFree(k.lens); cudaFree(k.alns);
            return qm_fail(ctx, QM_ENOMEM, "rmdup: cannot keep a chunk of %lld pairs on the device: %s", (long long)n, cudaGetErrorString(e));
        }
        if (quals_ready) QM_CUDA(ctx, cudaStreamWaitEvent(st, quals_ready, 0));
        QM_CUDA(ctx, cudaMemcpyAsync(k.codes, d_codes, sb, cudaMemcpyDeviceToDevice, st));
        QM_CUDA(ctx, cudaMemcpyAsync(k.quals, d_quals, sb, cudaMemcpyDeviceToDevice, st));
        QM_CUDA(ctx, cudaMemcpyAsync(k.lens, d_lens, (size_t)2 * n * 4, cudaMemcpyDeviceToDevice, st));
        QM_CUDA(ctx, cudaMemcpyAsync(k.alns, alns, (size_t)2 * n * sizeof(qm_aln), cudaMemcpyDeviceToDevice, st));
        s->kept.push_back(k);
        s->n_pairs += n;
        return QM_OK;
    }
    if (quals_ready) QM_CUDA(ctx, cudaStreamWaitEvent(st, quals_ready, 0));
    const uint8_t *pq = nullptr;
    rc = sample_pileup_quals(s, alns, d_codes, d_quals, stride, d_lens, 2 * n, st, &pq);
    if (rc) return rc;
    rc = qm_pileup_accumulate_indels(ctx, s->idx, &s->popt, alns, d_codes, pq, stride, d_lens, n, s->d_counts, s->indels, st);
    if (rc) return rc;
    s->n_pairs += n;
    return QM_OK;
}

}  // namespace

extern "C" {

int qm_sample_begin(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const qm_pileup_opt *popt, qm_sample **out)
{
    if (!ctx || !idx || !opt || !popt || !out) return QM_EINVAL;
    *out = nullptr;
    if (opt->min_seed_len != idx->v.k) return qm_fail(ctx, QM_EINVAL, "index built with k=%d but min_seed_len=%d", idx->v.k, opt->min_seed_len);
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    qm_sample *s = new qm_sample();
    s->ctx = ctx; s->idx = idx; s->opt = *opt; s->popt = *popt;
    cudaError_t e;
    if ((e = cudaMalloc(&s->d_counts, (size_t)QM_NCH * idx->v.l_pac * sizeof(int32_t))) != cudaSuccess ||
        (e = cudaMalloc(&s->d_cells, 8)) != cudaSuccess ||
        (e = cudaMalloc(&s->d_n_kept, sizeof(unsigned long long))) != cudaSuccess ||
        (e = cudaMalloc(&s->d_regs, (size_t)2 * kChunkPairs * QM_MAX_REGS * sizeof(qm_reg))) != cudaSuccess ||
        (e = cudaMalloc(&s->d_n_regs, (size_t)2 * kChunkPairs * sizeof(int32_t))) != cudaSuccess ||
        (e = cudaMalloc(&s->d_alns, (size_t)2 * kChunkPairs * sizeof(qm_aln))) != cudaSuccess ||
        (e = cudaMemset(s->d_counts, 0, (size_t)QM_NCH * idx->v.l_pac * sizeof(int32_t))) != cudaSuccess ||
        (e = cudaMemset(s->d_cells, 0, 8)) != cudaSuccess) {
        qm_sample_destroy(s);
        return qm_fail(ctx, QM_ENOMEM, "qm_sample_begin: %s", cudaGetErrorString(e));
    }
    if (qm_indel_table_create(ctx, 20, &s->indels) != QM_OK) { qm_sample_destroy(s); return QM_ENOMEM; }
    for (int i = 0; i < 2; ++i) {
        cudaEventCreateWithFlags(&s->ev_copied[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&s->ev_quals[i], cudaEventDisableTiming);
        for (int p = 0; p < kCopyParts; ++p) cudaEventCreateWithFlags(&s->ev_part[i][p], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&s->ev_consumed[i], cudaEventDisableTiming);
    }
    *out = s;
    return QM_OK;
}

static void free_kept(qm_sample *s)
{
    for (auto &k : s->kept) { cudaFree(k.codes); cudaFree(k.quals); cudaFree(k.lens); cudaFree(k.alns); }
    s->kept.clear();
}

void qm_sample_destroy(qm_sample *s)
{
    if (!s) return;
    cudaSetDevice(s->ctx->device);
    cudaDeviceSynchronize();
    free_kept(s);
    qm_indel_table_destroy(s->indels);
    cudaFree(s->d_counts); cudaFree(s->d_cells); cudaFree(s->d_regs); cudaFree(s->d_n_regs); cudaFree(s->d_alns);
    cudaFree(s->d_keep); cudaFree(s->d_n_kept);
    for (int i = 0; i < 2; ++i) {
        cudaFree(s->d_stage[i]);
        if (s->ev_copied[i]) cudaEventDestroy(s->ev_copied[i]);
        if (s->ev_quals[i]) cudaEventDestroy(s->ev_quals[i]);
        for (int p = 0; p < kCopyParts; ++p) if (s->ev_part[i][p]) cudaEventDestroy(s->ev_part[i][p]);
        if (s->ev_consumed[i]) cudaEventDestroy(s->ev_consumed[i]);
    }
    delete s;
}

// zero the counts and forget the insert-size model: the object can be reused for the next sample
int qm_sample_reset(qm_sample *s, void *stream)
{
    if (!s) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    QM_CUDA(ctx, cudaMemsetAsync(s->d_counts, 0, (size_t)QM_NCH * s->idx->v.l_pac * sizeof(int32_t), (cudaStream_t)stream));
    QM_CUDA(ctx, cudaMemsetAsync(s->d_cells, 0, 8, (cudaStream_t)stream));
    { const int rc = qm_indel_table_reset(s->indels, stream); if (rc) return rc; }
    s->have_pes = false; s->n_pairs = 0; s->rmdup_finished = false; s->last_n = -1;
    s->next_chunks.clear(); s->chunk_pes.clear();
    if (!s->kept.empty()) { QM_CUDA(ctx, cudaStreamSynchronize((cudaStream_t)stream)); free_kept(s); }
    return QM_OK;
}

// ---- duplicate removal (the reference's rule `rmdup`: picard MarkDuplicates REMOVE_DUPLICATES=true, rules/rmdup.smk:13-16) ----
int qm_sample_set_rmdup(qm_sample *s, int on)
{
    if (!s) return QM_EINVAL;
    if (s->n_pairs != 0) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_set_rmdup: pairs were already added; reset the sample first");
    if (on && s->filter) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_set_rmdup: the sample is in filter mode");
    s->rmdup = on != 0;
    return QM_OK;
}

// marks the duplicates among everything added since the last reset (flag 0x400 on their records), then counts the rest
int qm_sample_set_max_depth(qm_sample *s, int max_depth)
{
    if (!s || max_depth < 0) return QM_EINVAL;
    if (s->n_pairs != 0) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_set_max_depth: pairs were already added; reset the sample first");
    if (max_depth > 0 && s->filter) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_set_max_depth: the sample is in filter mode");
    s->max_depth = max_depth;
    return QM_OK;
}

// Filter mode (a contaminant pass of `sample --decontam`): pairs are aligned and finished as usual, CIGAR stage included (a CIGAR
// overflow unmaps a read), but nothing is counted and nothing is kept across batches; each batch leaves one keep byte per pair.
int qm_sample_set_filter(qm_sample *s, int on)
{
    if (!s) return QM_EINVAL;
    if (s->n_pairs != 0) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_set_filter: pairs were already added; reset the sample first");
    if (on && (s->rmdup || s->max_depth > 0)) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_set_filter: the sample defers its counting (rmdup / depth cap)");
    s->filter = on != 0;
    return QM_OK;
}

// the keep bytes of the last batch a filter-mode sample was given, and how many pairs they keep; synchronous
int qm_sample_keep_host(qm_sample *s, uint8_t *h_keep, int64_t n_pairs, int64_t *h_n_kept)
{
    if (!s || n_pairs < 0 || (n_pairs > 0 && !h_keep)) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    if (!s->filter) return qm_fail(ctx, QM_EINVAL, "qm_sample_keep_host: the sample is not in filter mode (qm_sample_set_filter)");
    if (n_pairs != s->last_n) return qm_fail(ctx, QM_EINVAL, "qm_sample_keep_host: the last batch had %lld pairs, not %lld", (long long)s->last_n, (long long)n_pairs);
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    QM_CUDA(ctx, cudaDeviceSynchronize());          // the batch may have been added on any stream
    unsigned long long nk = 0;
    if (n_pairs > 0) QM_CUDA(ctx, cudaMemcpy(h_keep, s->d_keep, (size_t)n_pairs, cudaMemcpyDeviceToHost));
    QM_CUDA(ctx, cudaMemcpy(&nk, s->d_n_kept, sizeof nk, cudaMemcpyDeviceToHost));
    if (h_n_kept) *h_n_kept = (int64_t)nk;
    return QM_OK;
}

// Base alignment quality for the sample's pileup: 0 = off (the default: `mpileup -B`, the parity configuration), 3 = extended BAQ as
// `bcftools mpileup` / `samtools mpileup` run it without -B (rules/vcfcall.smk:39,115), 1 = plain BAQ.  Duplicate marking keeps
// using the reads' own qualities (picard runs before the pileup).
int qm_sample_set_baq(qm_sample *s, int flag)
{
    if (!s || (flag != 0 && flag != 1 && flag != 3)) return QM_EINVAL;
    if (s->n_pairs != 0) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_set_baq: pairs were already added; reset the sample first");
    s->baq = flag;
    return QM_OK;
}

// the last step of a deferred sample: count what survived duplicate marking (0x400) and the cap (drop[c], may be NULL), then release
// the kept reads; the records stay for qm_sample_kept_alns_host
static int count_survivors(qm_sample *s, const std::vector<uint8_t *> &drop, void *stream)
{
    qm_ctx *ctx = s->ctx;
    for (size_t c = 0; c < s->kept.size(); ++c) {
        const auto &k = s->kept[c];
        const uint8_t *pq = nullptr;
        int rc = sample_pileup_quals(s, k.alns, k.codes, k.quals, k.stride, k.lens, 2 * k.n, (cudaStream_t)stream, &pq);
        if (!rc) rc = qm_pileup_accumulate_masked(ctx, s->idx, &s->popt, k.alns, k.codes, pq, k.stride, k.lens, k.n, s->d_counts, s->indels, drop[c], stream);
        if (rc) return rc;
    }
    QM_CUDA(ctx, cudaStreamSynchronize((cudaStream_t)stream));
    for (auto &k : s->kept) { cudaFree(k.codes); cudaFree(k.quals); cudaFree(k.lens); k.codes = k.quals = nullptr; k.lens = nullptr; }
    s->rmdup_finished = true;
    return QM_OK;
}

// Deferred counting: marks the duplicates among everything added since the last reset (rmdup mode), replays htslib's depth
// cap over the records that are left (max_depth mode), then counts what survives both.
int qm_sample_finish(qm_sample *s, int64_t *n_dup_pairs, int64_t *n_capped_reads, void *stream)
{
    if (!s) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    if (!s->rmdup && s->max_depth <= 0) return qm_fail(ctx, QM_EINVAL, "qm_sample_finish: the sample counts as it goes (neither rmdup nor a depth cap is set)");
    if (s->rmdup_finished) return qm_fail(ctx, QM_EINVAL, "qm_sample_finish: already finished; reset the sample first");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    QM_CUDA(ctx, cudaDeviceSynchronize());                 // chunks may have been added on any stream
    const int nc = (int)s->kept.size();
    std::vector<qm_aln *> a(nc);
    std::vector<const uint8_t *> q(nc);
    std::vector<const int32_t *> l(nc);
    std::vector<int32_t> st(nc);
    std::vector<int64_t> n(nc);
    for (int c = 0; c < nc; ++c) { a[c] = s->kept[c].alns; q[c] = s->kept[c].quals; l[c] = s->kept[c].lens; st[c] = s->kept[c].stride; n[c] = s->kept[c].n; }
    if (n_dup_pairs) *n_dup_pairs = 0;
    if (n_capped_reads) *n_capped_reads = 0;
    int rc;
    if (s->rmdup) {
        rc = qm_mark_duplicates(ctx, nc, a.data(), q.data(), st.data(), l.data(), n.data(), n_dup_pairs, stream);
        if (rc) return rc;
    }
    std::vector<uint8_t *> drop((size_t)nc, nullptr);
    if (s->max_depth > 0 && nc > 0) {
        for (int c = 0; c < nc; ++c) if (n[c]) QM_CUDA(ctx, cudaMalloc(&drop[c], (size_t)2 * n[c]));
        rc = qm_depth_cap(ctx, &s->popt, nc, a.data(), n.data(), s->max_depth, drop.data(), n_capped_reads, stream);
        if (rc) { for (auto d : drop) cudaFree(d); return rc; }
    }
    rc = count_survivors(s, drop, stream);
    for (auto d : drop) cudaFree(d);
    return rc;
}

// marks the duplicates among everything added since the last reset (flag 0x400 on their records), then counts the rest
int qm_sample_rmdup_finish(qm_sample *s, int64_t *n_dup_pairs, void *stream)
{
    if (!s) return QM_EINVAL;
    if (!s->rmdup) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_rmdup_finish: the sample is not in rmdup mode");
    return qm_sample_finish(s, n_dup_pairs, nullptr, stream);
}

// the records of everything added in rmdup mode, in input order, with their final flags; synchronous
int qm_sample_kept_alns_host(qm_sample *s, qm_aln *h_alns, int64_t max_records)
{
    if (!s || (!h_alns && max_records > 0)) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    int64_t off = 0;
    for (auto &k : s->kept) {
        if (off + 2 * k.n > max_records) return qm_fail(ctx, QM_EINVAL, "qm_sample_kept_alns_host: buffer of %lld records is too small", (long long)max_records);
        QM_CUDA(ctx, cudaMemcpy(h_alns + off, k.alns, (size_t)2 * k.n * sizeof(qm_aln), cudaMemcpyDeviceToHost));
        off += 2 * k.n;
    }
    return QM_OK;
}

// Multi-GPU sample: this rank holds a contiguous range of the sample's pairs, rank 0 the range that starts at pair 0 (with at
// least min(sample, QM_PESTAT_PAIRS) pairs in its first batch).  The insert-size model is then rank 0's, broadcast when the
// first batch of every rank has been aligned; qm_sample_allreduce_counts sums the count tensors in place on every rank.
int qm_sample_set_comm(qm_sample *s, qm_comm *comm)
{
    if (!s) return QM_EINVAL;
    // clearing is always allowed; a communicator has to be there before the first pairs (it decides whose insert-size model is used)
    if (comm && s->n_pairs != 0) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_set_comm: pairs were already added; reset the sample first");
    s->comm = comm;
    return QM_OK;
}

int qm_sample_allreduce_counts(qm_sample *s, void *stream)
{
    if (!s) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    if (!s->comm) return qm_fail(ctx, QM_EINVAL, "qm_sample_allreduce_counts: no communicator set");
    int rc = qm_counts_allreduce(ctx, s->comm, s->d_counts, (int64_t)QM_NCH * s->idx->v.l_pac, stream);
    if (rc) return rc;
    const int size = qm_comm_size(s->comm), rank = qm_comm_rank(s->comm);
    if (size == 1) return QM_OK;
    // the sparse part: every rank's alleles to every rank (counts first, then the records padded to the largest count),
    // the others' records added into the local table
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    constexpr int64_t kMaxRec = 1 << 18;
    std::vector<qm_indel> mine((size_t)kMaxRec);
    int64_t n = 0;
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    rc = qm_indel_table_fetch_host(s->indels, s->idx, mine.data(), kMaxRec, &n);
    if (rc) return rc;
    void *p = nullptr;
    rc = qm_scratch_reserve(ctx, 22, 256 + (size_t)size * 8, &p);
    if (rc) return rc;
    int64_t *d_n = (int64_t *)p, *d_all_n = (int64_t *)((char *)p + 256);
    QM_CUDA(ctx, cudaMemcpyAsync(d_n, &n, 8, cudaMemcpyHostToDevice, st));
    rc = qm_comm_allgather(ctx, s->comm, d_n, d_all_n, 8, st);
    if (rc) return rc;
    std::vector<int64_t> all_n((size_t)size);
    QM_CUDA(ctx, cudaMemcpyAsync(all_n.data(), d_all_n, (size_t)size * 8, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    int64_t mx = 0;
    for (int64_t v : all_n) mx = v > mx ? v : mx;
    if (mx == 0) return QM_OK;
    rc = qm_scratch_reserve(ctx, 23, (size_t)(size + 1) * mx * sizeof(qm_indel), &p);
    if (rc) return rc;
    qm_indel *d_send = (qm_indel *)p, *d_recv = d_send + mx;
    QM_CUDA(ctx, cudaMemsetAsync(d_send, 0, (size_t)mx * sizeof(qm_indel), st));
    if (n) QM_CUDA(ctx, cudaMemcpyAsync(d_send, mine.data(), (size_t)n * sizeof(qm_indel), cudaMemcpyHostToDevice, st));
    rc = qm_comm_allgather(ctx, s->comm, d_send, d_recv, (size_t)mx * sizeof(qm_indel), st);
    if (rc) return rc;
    for (int r = 0; r < size; ++r)
        if (r != rank && all_n[r] > 0) {
            rc = qm_indel_table_merge(s->indels, d_recv + (size_t)r * mx, all_n[r], st);
            if (rc) return rc;
        }
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    return QM_OK;
}

// every rank's n_mine tuples of `rec` bytes at d_mine -> the union of all ranks' tuples (*d_union, *n_union; rank order, no padding).
// The counts cross first (8 bytes per rank), then the tuples padded to the largest count.  Collective, synchronous.
static int allgather_tuples(qm_ctx *ctx, qm_comm *comm, const void *d_mine, int64_t n_mine, size_t rec, void **d_union, int64_t *n_union,
                            cudaStream_t st)
{
    const int size = qm_comm_size(comm);
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 34, 256 + (size_t)size * 8, &p);                 // scratch 34: my count | every rank's count
    if (rc) return rc;
    int64_t *d_n = (int64_t *)p, *d_all_n = (int64_t *)((char *)p + 256);
    QM_CUDA(ctx, cudaMemcpyAsync(d_n, &n_mine, 8, cudaMemcpyHostToDevice, st));
    rc = qm_comm_allgather(ctx, comm, d_n, d_all_n, 8, st);
    if (rc) return rc;
    std::vector<int64_t> all_n((size_t)size);
    QM_CUDA(ctx, cudaMemcpyAsync(all_n.data(), d_all_n, (size_t)size * 8, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    int64_t mx = 0, tot = 0;
    for (int64_t v : all_n) { mx = v > mx ? v : mx; tot += v; }
    *d_union = nullptr; *n_union = tot;
    if (mx == 0) return QM_OK;
    // both buffers before the all-gather: growing one frees device memory, which is not done while a collective is in flight
    void *u = nullptr;
    rc = qm_scratch_reserve(ctx, 35, (size_t)(size + 1) * mx * rec, &p);             // scratch 35: send (mx records) | receive (size x mx)
    if (!rc) rc = qm_scratch_reserve(ctx, 36, (size_t)tot * rec, &u);                 // scratch 36: the union, padding dropped
    if (rc) return rc;
    char *send = (char *)p, *recv = send + (size_t)mx * rec;
    if (n_mine) QM_CUDA(ctx, cudaMemcpyAsync(send, d_mine, (size_t)n_mine * rec, cudaMemcpyDeviceToDevice, st));
    if (n_mine < mx) QM_CUDA(ctx, cudaMemsetAsync(send + (size_t)n_mine * rec, 0, (size_t)(mx - n_mine) * rec, st));
    rc = qm_comm_allgather(ctx, comm, send, recv, (size_t)mx * rec, st);
    if (rc) return rc;
    size_t off = 0;
    for (int r = 0; r < size; ++r) {
        if (all_n[(size_t)r]) QM_CUDA(ctx, cudaMemcpyAsync((char *)u + off, recv + (size_t)r * mx * rec, (size_t)all_n[(size_t)r] * rec,
                                                           cudaMemcpyDeviceToDevice, st));
        off += (size_t)all_n[(size_t)r] * rec;
    }
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    *d_union = u;
    return QM_OK;
}

// Deferred counting of a sample sharded over the ranks of `comm`: duplicates and the cap decided over the union of every rank's
// tuples, this rank's survivors counted (the caller all-reduces the counts next).  Collective.
int qm_sample_finish_comm(qm_sample *s, qm_comm *comm, int64_t *n_dup_pairs, int64_t *n_capped_reads, void *stream)
{
    if (!s || !comm) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    if (!s->rmdup && s->max_depth <= 0) return qm_fail(ctx, QM_EINVAL, "qm_sample_finish_comm: the sample counts as it goes (neither rmdup nor a depth cap is set)");
    if (s->rmdup_finished) return qm_fail(ctx, QM_EINVAL, "qm_sample_finish_comm: already finished; reset the sample first");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    QM_CUDA(ctx, cudaDeviceSynchronize());                 // chunks may have been added on any stream
    cudaStream_t st = (cudaStream_t)stream;
    const int nc = (int)s->kept.size();
    std::vector<qm_aln *> a(nc);
    std::vector<const uint8_t *> q(nc);
    std::vector<const int32_t *> l(nc);
    std::vector<int32_t> sd(nc);
    std::vector<int64_t> n(nc), id0(nc);
    int64_t N = 0;
    for (int c = 0; c < nc; ++c) {
        const auto &k = s->kept[c];
        a[c] = k.alns; q[c] = k.quals; l[c] = k.lens; sd[c] = k.stride; n[c] = k.n; id0[c] = k.pair0;
        N += k.n;
    }
    if (n_dup_pairs) *n_dup_pairs = 0;
    if (n_capped_reads) *n_capped_reads = 0;
    void *p = nullptr, *all = nullptr;
    int64_t n_mine = 0, n_all = 0;
    int rc = qm_scratch_reserve(ctx, 32, (size_t)(N > 0 ? N : 1) * 32, &p);          // scratch 32: this rank's tuples (32 bytes per pair either way)
    if (rc) return rc;
    if (s->rmdup) {
        rc = qm_dup_keys(ctx, nc, a.data(), q.data(), sd.data(), l.data(), n.data(), id0.data(), (qm_dup_key *)p, &n_mine, stream);
        if (!rc) rc = allgather_tuples(ctx, comm, p, n_mine, sizeof(qm_dup_key), &all, &n_all, st);
        if (!rc) rc = qm_mark_duplicates_keys(ctx, (const qm_dup_key *)all, n_all, nc, a.data(), n.data(), id0.data(), n_dup_pairs, stream);
        if (rc) return rc;
    }
    std::vector<uint8_t *> drop((size_t)nc, nullptr);
    if (s->max_depth > 0) {
        for (int c = 0; c < nc; ++c) if (n[c]) QM_CUDA(ctx, cudaMalloc(&drop[c], (size_t)2 * n[c]));
        rc = qm_cap_keys(ctx, &s->popt, nc, a.data(), n.data(), id0.data(), (qm_cap_key *)p, &n_mine, stream);
        if (!rc) rc = allgather_tuples(ctx, comm, p, n_mine, sizeof(qm_cap_key), &all, &n_all, st);
        if (!rc) rc = qm_depth_cap_keys(ctx, (const qm_cap_key *)all, n_all, s->max_depth, nc, n.data(), id0.data(), drop.data(), n_capped_reads, stream);
        if (rc) { for (auto d : drop) cudaFree(d); return rc; }
    }
    rc = count_survivors(s, drop, stream);
    for (auto d : drop) cudaFree(d);
    return rc;
}

qm_indel_table *qm_sample_indel_table(qm_sample *s) { return s ? s->indels : nullptr; }

int qm_sample_set_pestat(qm_sample *s, const qm_pestat pes[4])
{
    if (!s || !pes) return QM_EINVAL;
    for (int d = 0; d < 4; ++d) s->pes[d] = pes[d];
    s->have_pes = true;
    return QM_OK;
}

int qm_sample_get_pestat(const qm_sample *s, qm_pestat pes[4])
{
    if (!s || !pes) return QM_EINVAL;
    if (!s->have_pes) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_get_pestat: no pairs added yet and no model set");
    for (int d = 0; d < 4; ++d) pes[d] = s->pes[d];
    return QM_OK;
}

// Per-chunk mode: bwa mem's insert-size model per input chunk (bwamem.c mem_process_seqs runs mem_pestat over all pairs of
// each chunk).  h_chunk_pairs[0 .. n_chunks) are the sizes in pairs of the chunks of the NEXT add call, in order; they must add up
// to its n_pairs (QM_EINVAL there otherwise), so a chunk never straddles two calls.  Where the chunks end is the caller's rule (bwa:
// bseq_read's running base count); a chunk holds at most QM_CHUNK_MAX_PAIRS pairs.  The prefix model and qm_pestat_bcast are not
// used in this mode; a model given with qm_sample_set_pestat (bwa mem -I) still replaces every chunk's.
int qm_sample_set_chunks(qm_sample *s, const int64_t *h_chunk_pairs, int64_t n_chunks)
{
    if (!s || n_chunks < 0 || (n_chunks > 0 && !h_chunk_pairs)) return QM_EINVAL;
    if (!s->chunked && s->n_pairs != 0) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_set_chunks: pairs were already added; reset the sample first");
    for (int64_t c = 0; c < n_chunks; ++c) {
        if (h_chunk_pairs[c] <= 0) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_set_chunks: chunk %lld has %lld pairs", (long long)c, (long long)h_chunk_pairs[c]);
        if (h_chunk_pairs[c] > kChunkPairs)
            return qm_fail(s->ctx, QM_ELIMIT, "qm_sample_set_chunks: chunk %lld has %lld pairs, at most %lld (QM_CHUNK_MAX_PAIRS) are supported",
                           (long long)c, (long long)h_chunk_pairs[c], (long long)kChunkPairs);
    }
    s->chunked = true;
    s->next_chunks.assign(h_chunk_pairs, h_chunk_pairs + n_chunks);
    return QM_OK;
}

// per-chunk mode: the models of the chunks of the last add call, 4 per chunk (none when a model was given); h_pes NULL with
// max_chunks 0: only their number
int qm_sample_chunk_pestat(const qm_sample *s, qm_pestat *h_pes, int64_t max_chunks, int64_t *n_chunks)
{
    if (!s || !n_chunks || max_chunks < 0 || (max_chunks > 0 && !h_pes)) return QM_EINVAL;
    const int64_t n = (int64_t)s->chunk_pes.size() / 4;
    *n_chunks = n;
    if (!h_pes) return QM_OK;
    if (n > max_chunks) return qm_fail(s->ctx, QM_EINVAL, "qm_sample_chunk_pestat: %lld chunks, room for %lld", (long long)n, (long long)max_chunks);
    std::copy(s->chunk_pes.begin(), s->chunk_pes.end(), h_pes);
    return QM_OK;
}

// insert-size model from a designated prefix of the sample (the first min(n, QM_PESTAT_PAIRS) pairs given):
// single-end alignment of the prefix + mem_pestat, nothing is counted.  A shard that does not start at pair 0
// calls this with the sample's first pairs before adding its own (every rank gets the same model, no collective).
int qm_sample_estimate_pestat(qm_sample *s, const uint8_t *d_codes, int32_t stride, const int32_t *d_lens, int64_t n_pairs,
                              void *stream)
{
    if (!s || n_pairs <= 0 || !d_codes || !d_lens || stride <= 0) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t n = n_pairs < kPestatPairs ? n_pairs : kPestatPairs;
    int rc = qm_align_se(ctx, s->idx, &s->opt, d_codes, stride, d_lens, 2 * n, s->d_regs, s->d_n_regs, nullptr, (cudaStream_t)stream);
    if (rc) return rc;
    rc = qm_pestat_sync(ctx, s->idx, &s->opt, s->d_regs, s->d_n_regs, n, s->pes, (cudaStream_t)stream);
    if (rc) return rc;
    s->have_pes = true;
    return QM_OK;
}

int qm_sample_add_pairs(qm_sample *s, const uint8_t *d_codes, const uint8_t *d_quals, int32_t stride, const int32_t *d_lens,
                        int64_t n_pairs, int64_t pair_id0, qm_aln *d_alns, void *stream)
{
    if (!s || n_pairs < 0 || (n_pairs > 0 && (!d_codes || !d_quals || !d_lens)) || stride <= 0) return QM_EINVAL;
    QM_CUDA(s->ctx, cudaSetDevice(s->ctx->device));
    std::vector<int64_t> starts, sizes, bwa;
    std::vector<int> bwa0;
    { const int rc = plan_chunks(s, n_pairs, starts, sizes, bwa, bwa0); if (rc) return rc; }
    { const int rc = filter_begin(s, n_pairs, (cudaStream_t)stream); if (rc) return rc; }
    for (size_t k = 0; k < starts.size(); ++k) {
        const int64_t p0 = starts[k], n = sizes[k];
        int rc = sample_chunk(s, d_codes + 2 * p0 * stride, d_quals + 2 * p0 * stride, stride, d_lens + 2 * p0, n, pair_id0 + p0, p0,
                              d_alns ? d_alns + 2 * p0 : nullptr, (cudaStream_t)stream, nullptr,
                              s->chunked ? bwa.data() + bwa0[k] : nullptr, s->chunked ? bwa0[k + 1] - bwa0[k] : 0);
        if (rc) return rc;
    }
    return QM_OK;
}

// Host entry: h_* should be page-locked for the copies to overlap the previous chunk's kernels.
// h_alns (may be NULL) receives the alignment records, 2 per pair, in input order.  Synchronous.
// h_codes (1 byte per base) or, when it is NULL, h_bases2 + h_nmask (packed: 0.375 bytes per base over the host link)
static int add_pairs_host_impl(qm_sample *s, const uint8_t *h_codes, const uint8_t *h_bases2, const uint8_t *h_nmask, const uint8_t *h_quals,
                               int32_t stride, const int32_t *h_lens, int64_t n_pairs, int64_t pair_id0, qm_aln *h_alns)
{
    const bool packed = h_codes == nullptr;
    if (!s || n_pairs < 0 || (n_pairs > 0 && ((packed ? (!h_bases2 || !h_nmask) : false) || !h_quals || !h_lens)) || stride <= 0) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    std::vector<int64_t> starts, sizes, bwa;
    std::vector<int> bwa0;
    { const int rc = plan_chunks(s, n_pairs, starts, sizes, bwa, bwa0); if (rc) return rc; }
    { const int rc = filter_begin(s, n_pairs, ctx->own_stream); if (rc) return rc; }
    if (n_pairs == 0) return QM_OK;
    const int stride_p = (stride + 3) >> 2, stride_m = (stride + 7) >> 3;
    const size_t seq_bytes = (size_t)2 * kChunkPairs * stride;
    const size_t seq_al = (seq_bytes + 255) & ~(size_t)255;
    const size_t lens_al = ((size_t)2 * kChunkPairs * sizeof(int32_t) + 255) & ~(size_t)255;
    const size_t pk_al = ((size_t)2 * kChunkPairs * stride_p + 255) & ~(size_t)255, mk_al = ((size_t)2 * kChunkPairs * stride_m + 255) & ~(size_t)255;
    const size_t o_pk = 2 * seq_al + lens_al, o_mk = o_pk + pk_al;
    const size_t need = o_mk + mk_al;
    if (need > s->stage_cap) {
        for (int i = 0; i < 2; ++i) {
            if (s->d_stage[i]) QM_CUDA(ctx, cudaFree(s->d_stage[i]));
            s->d_stage[i] = nullptr;
            QM_CUDA(ctx, cudaMalloc(&s->d_stage[i], need));
        }
        s->stage_cap = need;
    }
    cudaStream_t cs = ctx->copy_stream, ks = ctx->own_stream;
    static const int n_parts = getenv("QM_COPY_PARTS") ? std::max(1, std::min(kCopyParts, atoi(getenv("QM_COPY_PARTS")))) : kCopyParts;   // tuning knob
    // Full-size chunks (large batches: fewer extension rounds, shorter tails).  A chunk's bases are copied in kCopyParts
    // pieces and seeded piece by piece, so only the first piece's copy is exposed; qualities travel behind the bases
    // (only the pileup at the end of a chunk reads them); the next chunk's copies run under this chunk's kernels.
    // (Per-chunk mode: the chunks plan_chunks cut at bwa chunk ends.)
    if (!s->chunked) {
        starts.clear(); sizes.clear();
        int64_t ramp[8] = { kChunkPairs };
        int n_ramp = 1;
        if (const char *e = getenv("QM_HOST_CHUNKS")) {             // measurement knob: comma-separated chunk sizes
            n_ramp = 0;
            for (const char *q = e; *q && n_ramp < 8;) {
                char *end = nullptr;
                const long long v = strtoll(q, &end, 10);
                if (end == q) break;
                if (v > 0) ramp[n_ramp++] = v < kChunkPairs ? v : kChunkPairs;
                q = *end ? end + 1 : end;
            }
            if (n_ramp == 0) { ramp[0] = kChunkPairs; n_ramp = 1; }
        }
        int64_t p0 = 0;
        for (int k = 0; p0 < n_pairs; ++k) {
            int64_t n = k < n_ramp ? ramp[k] : kChunkPairs;
            if (n > n_pairs - p0) n = n_pairs - p0;
            starts.push_back(p0); sizes.push_back(n);
            p0 += n;
        }
    }
    const int64_t n_chunks = (int64_t)starts.size();
    // QM_HOST_TRACE=1 (diagnostics): when each copy piece and the chunk's compute finished, relative to the call's start
    static const bool trace = getenv("QM_HOST_TRACE") != nullptr;
    cudaEvent_t tr0 = nullptr, tr_part[kCopyParts] = {}, tr_quals = nullptr, tr_done = nullptr, tr_chunk[16] = {}, tr_copy[16] = {};
    if (trace) {
        cudaEventCreate(&tr0); cudaEventCreate(&tr_quals); cudaEventCreate(&tr_done);
        for (int i = 0; i < kCopyParts; ++i) cudaEventCreate(&tr_part[i]);
        for (int i = 0; i < 16; ++i) { cudaEventCreate(&tr_chunk[i]); cudaEventCreate(&tr_copy[i]); }
        cudaEventRecord(tr0, ctx->copy_stream);
    }
    auto enqueue_copy = [&](int64_t c) -> cudaError_t {
        const int b = (int)(c & 1);
        const int64_t p0 = starts[c], n = sizes[c];
        cudaError_t e;
        if ((e = cudaStreamWaitEvent(cs, s->ev_consumed[b], 0)) != cudaSuccess) return e;     // buffer b free again
        if ((e = cudaMemcpyAsync(s->d_stage[b] + 2 * seq_al, h_lens + 2 * p0, (size_t)2 * n * sizeof(int32_t), cudaMemcpyHostToDevice, cs)) != cudaSuccess) return e;
        if ((e = cudaEventRecord(s->ev_copied[b], cs)) != cudaSuccess) return e;
        // the bases in kCopyParts pieces, an event behind each: seeding starts on piece 0 while the others are in flight
        for (int pt = 0; pt < n_parts; ++pt) {
            const int64_t r0 = 2 * n * pt / n_parts, r1 = 2 * n * (pt + 1) / n_parts;
            if (r1 > r0 && !packed && (e = cudaMemcpyAsync(s->d_stage[b] + r0 * stride, h_codes + (2 * p0 + r0) * stride, (size_t)(r1 - r0) * stride,
                                                           cudaMemcpyHostToDevice, cs)) != cudaSuccess) return e;
            if (r1 > r0 && packed) {
                // the packed piece.  Its expansion to one byte per base runs on the stream that seeds the piece (qm_align_se through
                // qm_ctx::se_pk), NOT here: a kernel in the copy stream waits for SM slots behind the extension kernels of the
                // chunk in flight, and every copy queued behind it waits with it (+6 ms per chunk of a multi-chunk call)
                uint8_t *d_pk = s->d_stage[b] + o_pk + r0 * stride_p, *d_mk = s->d_stage[b] + o_mk + r0 * stride_m;
                if ((e = cudaMemcpyAsync(d_pk, h_bases2 + (2 * p0 + r0) * stride_p, (size_t)(r1 - r0) * stride_p, cudaMemcpyHostToDevice, cs)) != cudaSuccess) return e;
                if ((e = cudaMemcpyAsync(d_mk, h_nmask + (2 * p0 + r0) * stride_m, (size_t)(r1 - r0) * stride_m, cudaMemcpyHostToDevice, cs)) != cudaSuccess) return e;
            }
            if ((e = cudaEventRecord(s->ev_part[b][pt], cs)) != cudaSuccess) return e;
            if (trace && c == 0) cudaEventRecord(tr_part[pt], cs);
        }
        if ((e = cudaMemcpyAsync(s->d_stage[b] + seq_al, h_quals + 2 * p0 * stride, (size_t)2 * n * stride, cudaMemcpyHostToDevice, cs)) != cudaSuccess) return e;
        if (trace && c == 0) cudaEventRecord(tr_quals, cs);
        if (trace && c < 16) cudaEventRecord(tr_copy[c], cs);
        return cudaEventRecord(s->ev_quals[b], cs);
    };
    // a fresh event counts as completed, so the first two waits on ev_consumed pass immediately
    QM_CUDA(ctx, enqueue_copy(0));
    static const bool no_overlap = getenv("QM_HOST_SEQ") != nullptr;          // diagnostics: copies and kernels one after the other
    if (no_overlap) QM_CUDA(ctx, cudaStreamSynchronize(cs));
    for (int64_t c = 0; c < n_chunks; ++c) {
        const int b = (int)(c & 1);
        const int64_t p0 = starts[c], n = sizes[c];
        if (c + 1 < n_chunks) QM_CUDA(ctx, enqueue_copy(c + 1));
        QM_CUDA(ctx, cudaStreamWaitEvent(ks, s->ev_copied[b], 0));
        ctx->se_n_parts = n_parts;
        if (packed) { ctx->se_pk = s->d_stage[b] + o_pk; ctx->se_mk = s->d_stage[b] + o_mk; ctx->se_sp = stride_p; ctx->se_sm = stride_m; }
        for (int pt = 0; pt < n_parts; ++pt) { ctx->se_part_end[pt] = 2 * n * (pt + 1) / n_parts; ctx->se_part_ev[pt] = s->ev_part[b][pt]; }
        int rc = sample_chunk(s, s->d_stage[b], s->d_stage[b] + seq_al, stride, (const int32_t *)(s->d_stage[b] + 2 * seq_al), n,
                              pair_id0 + p0, p0, nullptr, ks, s->ev_quals[b],
                              s->chunked ? bwa.data() + bwa0[c] : nullptr, s->chunked ? bwa0[c + 1] - bwa0[c] : 0);
        ctx->se_n_parts = 0; ctx->se_pk = ctx->se_mk = nullptr;
        if (rc) return rc;
        if (h_alns) QM_CUDA(ctx, cudaMemcpyAsync(h_alns + 2 * p0, s->d_alns, (size_t)2 * n * sizeof(qm_aln), cudaMemcpyDeviceToHost, ks));
        QM_CUDA(ctx, cudaEventRecord(s->ev_consumed[b], ks));
        if (trace && c == 0) cudaEventRecord(tr_done, ks);
        if (trace && c < 16) cudaEventRecord(tr_chunk[c], ks);
    }
    QM_CUDA(ctx, cudaStreamSynchronize(ks));
    if (trace) {
        float ms = 0;
        fprintf(stderr, "[qm host trace] pairs %lld pieces", (long long)sizes[0]);
        for (int i = 0; i < kCopyParts; ++i) { if (i < n_parts) { cudaEventElapsedTime(&ms, tr0, tr_part[i]); fprintf(stderr, " %.2f", ms); } cudaEventDestroy(tr_part[i]); }
        cudaEventElapsedTime(&ms, tr0, tr_quals); fprintf(stderr, " quals %.2f", ms);
        cudaEventElapsedTime(&ms, tr0, tr_done); fprintf(stderr, " chunk done %.2f ms", ms);
        if (n_chunks > 1) {
            fprintf(stderr, "; chunks (copied / done):");
            for (int64_t c = 0; c < n_chunks && c < 16; ++c) {
                float a = 0, b = 0;
                cudaEventElapsedTime(&a, tr0, tr_copy[c]); cudaEventElapsedTime(&b, tr0, tr_chunk[c]);
                fprintf(stderr, " %.1f/%.1f", a, b);
            }
        }
        fprintf(stderr, "\n");
        for (int i = 0; i < 16; ++i) { cudaEventDestroy(tr_chunk[i]); cudaEventDestroy(tr_copy[i]); }
        cudaEventDestroy(tr0); cudaEventDestroy(tr_quals); cudaEventDestroy(tr_done);
    }
    return QM_OK;
}

int qm_sample_add_pairs_host(qm_sample *s, const uint8_t *h_codes, const uint8_t *h_quals, int32_t stride,
                             const int32_t *h_lens, int64_t n_pairs, int64_t pair_id0, qm_aln *h_alns)
{
    if (n_pairs > 0 && !h_codes) return QM_EINVAL;
    return add_pairs_host_impl(s, h_codes, nullptr, nullptr, h_quals, stride, h_lens, n_pairs, pair_id0, h_alns);
}

// the same with the bases packed on the host side of the link: 2 bits per base + 1 bit per base for N
int qm_sample_add_pairs_host_packed(qm_sample *s, const uint8_t *h_bases2, const uint8_t *h_nmask, const uint8_t *h_quals, int32_t stride,
                                    const int32_t *h_lens, int64_t n_pairs, int64_t pair_id0, qm_aln *h_alns)
{
    if (n_pairs > 0 && (!h_bases2 || !h_nmask)) return QM_EINVAL;
    return add_pairs_host_impl(s, nullptr, h_bases2, h_nmask, h_quals, stride, h_lens, n_pairs, pair_id0, h_alns);
}

// host-side packer for the entry above: codes [n_reads][stride] (0..3, anything else = N) -> bases2 [n_reads][(stride + 3) / 4],
// nmask [n_reads][(stride + 7) / 8]
int qm_pack_reads_host(const uint8_t *h_codes, int32_t stride, int64_t n_reads, uint8_t *h_bases2, uint8_t *h_nmask)
{
    if (stride <= 0 || n_reads < 0 || (n_reads > 0 && (!h_codes || !h_bases2 || !h_nmask))) return QM_EINVAL;
    const int sp = (stride + 3) >> 2, sm = (stride + 7) >> 3;
    auto rows = [=](int64_t r0, int64_t r1) {
        for (int64_t r = r0; r < r1; ++r) {
            const uint8_t *c = h_codes + r * stride;
            uint8_t *b = h_bases2 + r * sp, *m = h_nmask + r * sm;
            memset(b, 0, (size_t)sp); memset(m, 0, (size_t)sm);
            for (int j = 0; j < stride; ++j) {
                if (c[j] > 3) m[j >> 3] |= (uint8_t)(1u << (j & 7));
                else b[j >> 2] |= (uint8_t)(c[j] << (2 * (j & 3)));
            }
        }
    };
    // (the FASTQ side of a host entry: rows are independent, a few threads keep the packing out of the file-level time)
    const unsigned hw = std::thread::hardware_concurrency();
    const int64_t nt = std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(hw ? hw : 4, 16), n_reads / 65536));
    if (nt == 1) rows(0, n_reads);
    else {
        std::vector<std::thread> pool;
        for (int64_t t = 0; t < nt; ++t) pool.emplace_back(rows, n_reads * t / nt, n_reads * (t + 1) / nt);
        for (auto &th : pool) th.join();
    }
    return QM_OK;
}

int32_t *qm_sample_counts(qm_sample *s) { return s ? s->d_counts : nullptr; }

// executed extension cells and pairs so far (synchronises `stream`)
int qm_sample_stats_sync(qm_sample *s, int64_t *n_pairs, int64_t *cells, void *stream)
{
    if (!s) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    int64_t c = 0;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    QM_CUDA(ctx, cudaMemcpyAsync(&c, s->d_cells, 8, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    QM_CUDA(ctx, cudaStreamSynchronize((cudaStream_t)stream));
    if (n_pairs) *n_pairs = s->n_pairs;
    if (cells) *cells = c;
    return QM_OK;
}

// count tensor to the host as rows [l_pac][QM_NCH] (count-TSV order); synchronous
int qm_sample_counts_host(qm_sample *s, int32_t *h_rows)
{
    if (!s || !h_rows) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    QM_CUDA(ctx, cudaDeviceSynchronize());          // counts may have been accumulated on any stream
    void *p = nullptr;
    const size_t bytes = (size_t)QM_NCH * s->idx->v.l_pac * sizeof(int32_t);
    int rc = qm_scratch_reserve(ctx, 6, bytes, &p);
    if (rc) return rc;
    rc = qm_counts_to_rows(ctx, s->idx, s->d_counts, (int32_t *)p, ctx->own_stream);
    if (rc) return rc;
    QM_CUDA(ctx, cudaMemcpyAsync(h_rows, p, bytes, cudaMemcpyDeviceToHost, ctx->own_stream));
    QM_CUDA(ctx, cudaStreamSynchronize(ctx->own_stream));
    return QM_OK;
}

// SNP calls of the sample to host memory (qm_call_snps on the sample's own tensor); synchronous
int qm_sample_call_snps_host(qm_sample *s, const qm_call_opt *copt, qm_call *h_calls, int64_t max_calls, int64_t *n_calls)
{
    if (!s || !copt || !n_calls || max_calls < 0 || (max_calls > 0 && !h_calls)) return QM_EINVAL;
    qm_ctx *ctx = s->ctx;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    QM_CUDA(ctx, cudaDeviceSynchronize());
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 10, (size_t)(max_calls > 0 ? max_calls : 1) * sizeof(qm_call), &p);
    if (rc) return rc;
    rc = qm_call_snps(ctx, s->idx, copt, s->d_counts, (qm_call *)p, max_calls, n_calls, ctx->own_stream);
    if (rc) return rc;
    QM_CUDA(ctx, cudaMemcpyAsync(h_calls, p, (size_t)*n_calls * sizeof(qm_call), cudaMemcpyDeviceToHost, ctx->own_stream));
    QM_CUDA(ctx, cudaStreamSynchronize(ctx->own_stream));
    return QM_OK;
}

}  // extern "C"
