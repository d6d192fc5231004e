// dedup.cu -- duplicate marking with the rule of `picard MarkDuplicates` (the reference's rule `rmdup`,
// rules/rmdup.smk:13-16, which sits between `bwa` and every caller; semantics SURVEY.md B.9).
//
// A pair with both ends placed is keyed by {contig, unclipped 5' coordinate, strand} of both ends (ends in
// coordinate order); among pairs with the same key the one with the highest sum of base qualities >= 15 over both
// mates stays, ties go to the earliest pair of the input (the lowest pair id).  A read whose mate is unplaced ("fragment") is keyed by its
// own {contig, unclipped 5' coordinate, strand}: it is a duplicate whenever an end of some fully placed pair has that
// key, otherwise the best fragment of the key stays.  Pairs with no placed end are never duplicates.
// On the device: one 32-byte tuple per pair with a placed end (key, score, end codes, pair id), the stable radix sort of sort.cu,
// then one pass over the sorted runs.  The tuples are what crosses GPUs when a sample is sharded (qm_sample_finish_comm): every
// rank decides over the union of all ranks' tuples and flags its own records.  Duplicates get SAM flag 0x400, which the pileup's
// read admission already skips.
#include <vector>
#include "pipeline.cuh"

namespace {

constexpr uint64_t kNoKey = ~0ull;
constexpr uint32_t kNoEnd = QM_DUP_NO_END;
constexpr int kCoordBias = QM_DUP_COORD_BIAS;

// {contig, unclipped 5' coordinate} of a placed record as a 30-bit code, and its strand
// (26 bits of coordinate, 4 of contig: a contig of >= 2^26 - 4096 bases or a 17th contig does not fit; *bad is raised then
// and qm_mark_duplicates fails with QM_ELIMIT instead of letting keys collide)
__device__ __forceinline__ uint32_t end_code(const qm_aln &a, int *rev, int *bad)
{
    const bool r = (a.flag & 0x10) != 0;
    int lead = 0, trail = 0, rlen = 0;
    const int nc = a.n_cigar == 255 ? 0 : a.n_cigar;
    for (int k = 0; k < nc; ++k) {
        const int op = a.cigar[k] & 0xf, len = (int)(a.cigar[k] >> 4);
        if (op == 0 || op == 2) rlen += len;
    }
    if (nc > 0 && (a.cigar[0] & 0xf) == 4) lead = (int)(a.cigar[0] >> 4);
    if (nc > 1 && (a.cigar[nc - 1] & 0xf) == 4) trail = (int)(a.cigar[nc - 1] >> 4);
    const int coord = r ? a.pos + rlen - 1 + trail : a.pos - lead;
    *rev = r ? 1 : 0;
    if (coord + kCoordBias < 0 || coord + kCoordBias >= (1 << 26) || a.rid >= 16) *bad = 1;
    return ((uint32_t)a.rid << 26) | (uint32_t)(coord + kCoordBias);
}

__device__ __forceinline__ bool placed(const qm_aln &a) { return !(a.flag & 0x4) && a.rid >= 0 && a.n_cigar != 0 && a.n_cigar != 255; }

// key, score and (for fully placed pairs) the two end codes of every pair with a placed end, appended at an atomic cursor
__global__ void __launch_bounds__(128)
dup_keys_kernel(const qm_aln *__restrict__ alns, const uint8_t *__restrict__ quals, int stride, const int32_t *__restrict__ lens,
                int64_t n_pairs, int64_t pair_id0, qm_dup_key *__restrict__ out, unsigned long long *__restrict__ cnt)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    const qm_aln a = alns[2 * i], b = alns[2 * i + 1];
    const bool pa = placed(a), pb = placed(b);
    if (!pa && !pb) return;                             // never a duplicate, and no end of it can make one
    int sc[2] = {0, 0};
    for (int e = 0; e < 2; ++e) {
        const uint8_t *q = quals + (2 * i + e) * (int64_t)stride;
        const int L = lens[2 * i + e];
        int s = 0;
        for (int j = 0; j < L; ++j) { const int v = q[j]; s += v >= 15 ? v : 0; }
        sc[e] = s;
    }
    int bad = 0, ra = 0, rb = 0;
    const uint32_t ca = pa ? end_code(a, &ra, &bad) : 0, cb = pb ? end_code(b, &rb, &bad) : 0;
    if (bad) atomicAdd(cnt + 1, 1ull);
    out[atomicAdd(cnt, 1ull)] = qm_dup_tuple(pair_id0 + i, pa, ca << 1 | (uint32_t)ra, sc[0], pb, cb << 1 | (uint32_t)rb, sc[1]);
}

// the union in pair-id order: ids[] sorted, perm[] their input positions.  Scatters key, score and end codes into sorted order and
// raises *rep where an id repeats
__global__ void __launch_bounds__(128)
dup_gather_kernel(const qm_dup_key *__restrict__ all, const uint64_t *__restrict__ ids, const uint32_t *__restrict__ perm, int64_t n,
                  uint64_t *__restrict__ keys, int32_t *__restrict__ scores, uint64_t *__restrict__ ends, unsigned long long *__restrict__ rep)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (i > 0 && ids[i - 1] == ids[i]) atomicAdd(rep, 1ull);
    const qm_dup_key t = all[perm[i]];
    keys[i] = t.key;
    scores[i] = t.score;
    ends[2 * i] = t.end0 == kNoEnd ? kNoKey : (uint64_t)t.end0;
    ends[2 * i + 1] = t.end1 == kNoEnd ? kNoKey : (uint64_t)t.end1;
}

// one thread per sorted position: the head of a run of equal keys picks the run's representative (highest score, first in
// pair-id order on ties -- the sort is stable, so that is the first of the run) and flags the others
__global__ void __launch_bounds__(128)
dup_mark_kernel(const uint64_t *__restrict__ skeys, const uint32_t *__restrict__ perm, const int32_t *__restrict__ scores, int64_t n,
                const uint64_t *__restrict__ sorted_ends, int64_t n_ends, uint8_t *__restrict__ dup)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t k = skeys[i];
    if (k == kNoKey) return;
    if (i > 0 && skeys[i - 1] == k) return;             // not the head of its run
    if (k >> 63) {                                      // fragments: any end of a fully placed pair with this key wins
        const uint64_t want = k & ~(1ull << 63);
        int64_t lo = 0, hi = n_ends;
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (sorted_ends[mid] < want) lo = mid + 1; else hi = mid; }
        if (lo < n_ends && sorted_ends[lo] == want) {
            for (int64_t j = i; j < n && skeys[j] == k; ++j) dup[perm[j]] = 1;
            return;
        }
    }
    int64_t best = i;
    int bs = scores[perm[i]];
    for (int64_t j = i + 1; j < n && skeys[j] == k; ++j) { const int s = scores[perm[j]]; if (s > bs) { bs = s; best = j; } }
    for (int64_t j = i; j < n && skeys[j] == k; ++j) if (j != best) dup[perm[j]] = 1;
}

__global__ void __launch_bounds__(128)
dup_count_kernel(const uint8_t *__restrict__ dup, int64_t n, unsigned long long *__restrict__ n_dup)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n && dup[i]) atomicAdd(n_dup, 1ull);
}

// local pair i of a chunk finds its verdict by its id in the sorted ids of the union (absent: no placed end, never a duplicate)
__global__ void __launch_bounds__(128)
dup_apply_kernel(qm_aln *__restrict__ alns, int64_t n_pairs, int64_t pair_id0, const uint64_t *__restrict__ ids, int64_t n_all,
                 const uint8_t *__restrict__ dup)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    const uint64_t want = (uint64_t)(pair_id0 + i);
    int64_t lo = 0, hi = n_all;
    while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (ids[mid] < want) lo = mid + 1; else hi = mid; }
    if (lo == n_all || ids[lo] != want || !dup[lo]) return;
    for (int e = 0; e < 2; ++e)
        if (!(alns[2 * i + e].flag & 0x4)) alns[2 * i + e].flag |= 0x400;      // an unplaced mate is never a duplicate
}

__global__ void __launch_bounds__(256)
dup_ids_kernel(const qm_dup_key *__restrict__ all, int64_t n, uint64_t *__restrict__ ids)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) ids[i] = (uint64_t)all[i].pair_id;
}

}  // namespace

extern "C" {

// one qm_dup_key per pair with a placed end, chunk c = pairs pair_id0[c] .. pair_id0[c] + n_pairs[c] - 1.  Synchronous.
int qm_dup_keys(qm_ctx *ctx, int n_chunks, const qm_aln *const *d_alns, const uint8_t *const *d_quals, const int32_t *strides,
                const int32_t *const *d_lens, const int64_t *n_pairs, const int64_t *pair_id0, qm_dup_key *d_out, int64_t *h_n_out,
                void *stream)
{
    if (!ctx || !h_n_out || n_chunks < 0 || (n_chunks > 0 && (!d_alns || !d_quals || !strides || !d_lens || !n_pairs || !pair_id0)))
        return QM_EINVAL;
    *h_n_out = 0;
    int64_t N = 0;
    for (int c = 0; c < n_chunks; ++c) { if (n_pairs[c] < 0 || pair_id0[c] < 0) return QM_EINVAL; N += n_pairs[c]; }
    if (N == 0) return QM_OK;
    if (!d_out) return QM_EINVAL;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 33, 256, &p);
    if (rc) return rc;
    unsigned long long *cnt = (unsigned long long *)p;           // cnt[0] = tuples written, cnt[1] = pairs whose end code does not fit
    QM_CUDA(ctx, cudaMemsetAsync(cnt, 0, 16, st));
    for (int c = 0; c < n_chunks; ++c)
        if (n_pairs[c]) dup_keys_kernel<<<(unsigned)((n_pairs[c] + 127) / 128), 128, 0, st>>>(d_alns[c], d_quals[c], strides[c], d_lens[c],
                                                                                        n_pairs[c], pair_id0[c], d_out, cnt);
    QM_CUDA(ctx, cudaGetLastError());
    unsigned long long h[2] = {0, 0};
    QM_CUDA(ctx, cudaMemcpyAsync(h, cnt, 16, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    if (h[1]) return qm_fail(ctx, QM_ELIMIT, "qm_mark_duplicates: %llu pairs lie beyond what the 30-bit end code holds (contigs of up to 2^26 - 4096 bases, 16 contigs)", h[1]);
    *h_n_out = (int64_t)h[0];
    return QM_OK;
}

}  // extern "C"

// the decision over a union of tuples: *d_ids = the pair ids sorted, (*d_dup)[k] = 1 when pair (*d_ids)[k] is a duplicate (scratch 15,
// valid until the next decision on the context).  A repeated id is QM_EINVAL.  Synchronous.
int qm_dup_decide(qm_ctx *ctx, const qm_dup_key *d_all, int64_t n_all, const uint64_t **d_ids, const uint8_t **d_dup, int64_t *h_n_dup,
                  cudaStream_t st)
{
    *d_ids = nullptr; *d_dup = nullptr; *h_n_dup = 0;
    if (n_all == 0) return QM_OK;
    if (2 * n_all > 0xffffffffll) return qm_fail(ctx, QM_ELIMIT, "qm_mark_duplicates: more than 2^31 pairs");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t N = n_all;
    // scratch 15: ids | id perm | keys | ends | scores | perm | end perm | dup flags | counters
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t o_ids = 0, o_iperm = o_ids + al((size_t)N * 8), o_keys = o_iperm + al((size_t)N * 4), o_ends = o_keys + al((size_t)N * 8);
    const size_t o_sc = o_ends + al((size_t)2 * N * 8), o_perm = o_sc + al((size_t)N * 4), o_eperm = o_perm + al((size_t)N * 4);
    const size_t o_dup = o_eperm + al((size_t)2 * N * 4), o_cnt = o_dup + al((size_t)N);
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 15, o_cnt + 256, &p);
    if (rc) return rc;
    char *b = (char *)p;
    uint64_t *ids = (uint64_t *)(b + o_ids), *keys = (uint64_t *)(b + o_keys), *ends = (uint64_t *)(b + o_ends);
    int32_t *scores = (int32_t *)(b + o_sc);
    uint32_t *iperm = (uint32_t *)(b + o_iperm), *perm = (uint32_t *)(b + o_perm), *eperm = (uint32_t *)(b + o_eperm);
    uint8_t *dup = (uint8_t *)(b + o_dup);
    unsigned long long *cnt = (unsigned long long *)(b + o_cnt);
    QM_CUDA(ctx, cudaMemsetAsync(dup, 0, (size_t)N, st));
    QM_CUDA(ctx, cudaMemsetAsync(cnt, 0, 16, st));             // cnt[0] = duplicates, cnt[1] = repeated ids
    // the union in pair-id order: the same input on every rank, whatever order the all-gather delivered it in
    dup_ids_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(d_all, N, ids);
    rc = qm_sort_ids(ctx, ids, iperm, N, "qm_mark_duplicates_keys", st);
    if (rc) return rc;
    dup_gather_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(d_all, ids, iperm, N, keys, scores, ends, cnt + 1);
    QM_CUDA(ctx, cudaGetLastError());
    unsigned long long h[2] = {0, 0};
    QM_CUDA(ctx, cudaMemcpyAsync(h + 1, cnt + 1, 8, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    if (h[1]) return qm_fail(ctx, QM_EINVAL, "qm_mark_duplicates_keys: %llu pair ids occur more than once in the union", h[1]);
    rc = qm_sort_pairs(ctx, keys, perm, N, 64, st);
    if (rc) return rc;
    rc = qm_sort_pairs(ctx, ends, eperm, 2 * N, 32, st);          // end keys are 31 bits; kNoKey's low word is all ones: sorts last
    if (rc) return rc;
    dup_mark_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(keys, perm, scores, N, ends, 2 * N, dup);
    dup_count_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(dup, N, cnt);
    QM_CUDA(ctx, cudaGetLastError());
    QM_CUDA(ctx, cudaMemcpyAsync(h, cnt, 8, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    *d_ids = ids; *d_dup = dup; *h_n_dup = (int64_t)h[0];
    return QM_OK;
}

extern "C" {

// the decision over the union of every rank's tuples, applied to this rank's chunks.  Synchronous.
int qm_mark_duplicates_keys(qm_ctx *ctx, const qm_dup_key *d_all, int64_t n_all, int n_chunks, qm_aln *const *d_alns,
                            const int64_t *n_pairs, const int64_t *pair_id0, int64_t *h_n_dup_all, void *stream)
{
    if (!ctx || n_all < 0 || (n_all > 0 && !d_all) || n_chunks < 0 || (n_chunks > 0 && (!d_alns || !n_pairs || !pair_id0))) return QM_EINVAL;
    for (int c = 0; c < n_chunks; ++c) if (n_pairs[c] < 0 || pair_id0[c] < 0) return QM_EINVAL;
    if (h_n_dup_all) *h_n_dup_all = 0;
    cudaStream_t st = (cudaStream_t)stream;
    const uint64_t *ids = nullptr;
    const uint8_t *dup = nullptr;
    int64_t n_dup = 0;
    const int rc = qm_dup_decide(ctx, d_all, n_all, &ids, &dup, &n_dup, st);
    if (rc || n_all == 0) return rc;
    for (int c = 0; c < n_chunks; ++c)
        if (n_pairs[c]) dup_apply_kernel<<<(unsigned)((n_pairs[c] + 127) / 128), 128, 0, st>>>(d_alns[c], n_pairs[c], pair_id0[c], ids, n_all, dup);
    QM_CUDA(ctx, cudaGetLastError());
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    if (h_n_dup_all) *h_n_dup_all = n_dup;
    return QM_OK;
}

// chunks: the sample's records in input order, chunk c = pairs [pair0[c], pair0[c] + n[c]): the export and the decision above on one
// device, pair ids = running pair offsets.  Synchronous.
int qm_mark_duplicates(qm_ctx *ctx, int n_chunks, qm_aln *const *d_alns, const uint8_t *const *d_quals, const int32_t *strides,
                       const int32_t *const *d_lens, const int64_t *n_pairs, int64_t *h_n_dup, void *stream)
{
    if (!ctx || n_chunks < 0 || (n_chunks > 0 && (!d_alns || !d_quals || !strides || !d_lens || !n_pairs))) return QM_EINVAL;
    int64_t N = 0;
    std::vector<int64_t> id0((size_t)n_chunks);
    for (int c = 0; c < n_chunks; ++c) { if (n_pairs[c] < 0) return QM_EINVAL; id0[(size_t)c] = N; N += n_pairs[c]; }
    if (h_n_dup) *h_n_dup = 0;
    if (N == 0) return QM_OK;
    if (2 * N > 0xffffffffll) return qm_fail(ctx, QM_ELIMIT, "qm_mark_duplicates: more than 2^31 pairs");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 32, (size_t)N * sizeof(qm_dup_key), &p);
    if (rc) return rc;
    qm_dup_key *tuples = (qm_dup_key *)p;
    int64_t n_t = 0;
    rc = qm_dup_keys(ctx, n_chunks, d_alns, d_quals, strides, d_lens, n_pairs, id0.data(), tuples, &n_t, stream);
    if (rc) return rc;
    return qm_mark_duplicates_keys(ctx, tuples, n_t, n_chunks, d_alns, n_pairs, id0.data(), h_n_dup, stream);
}

}  // extern "C"
