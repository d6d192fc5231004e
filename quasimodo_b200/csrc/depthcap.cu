// depthcap.cu -- the per-file depth cap of `bcftools mpileup -d N` (rules/vcfcall.smk:115 runs with the default; SURVEY.md
// A.8, 8f-2): which admitted reads htslib's pileup iterator keeps.  htslib 1.9 sam.c: bam_plp_push refuses a read whose start
// equals the position the iterator is assembling while more than `maxcnt` nodes are in use (the buffered reads plus the
// iterator's spare tail node); bam_plp_next releases the reads that end at or before that position, then steps to the next
// position or jumps to the first buffered read; bam_plp_auto feeds one read whenever nothing lies beyond the position.
// The outcome depends on the order of the reads by construction, so this is a replay of the iterator over the records in BAM
// order: one 16-byte tuple per admitted read (key, end, read id) comes from the device and is sorted there (sort.cu); the tuples
// are what crosses GPUs when a sample is sharded (qm_sample_finish_comm).  The replay itself is a host loop of O(reads +
// positions) steps -- a serial dependence from read to read that has no parallel form -- and the drop mask goes back to the
// device for the counting kernel.  Off by default (DESIGN.md 5.4: at BASELINE depths the cap throws away most of the sample).
#include <algorithm>
#include <queue>
#include <vector>
#include "pipeline.cuh"

namespace {

__device__ __forceinline__ bool cap_admitted(const qm_pileup_opt &po, const qm_aln &a)
{
    const int nc = a.n_cigar;
    return !(a.flag & (0x4 | 0x100 | 0x200 | 0x400)) && nc != 0 && nc != 255 && a.mapq >= po.min_mapq &&
           !((a.flag & 0x1) && !(a.flag & 0x2) && !po.count_orphans);
}

// one qm_cap_key per admitted read of a chunk, appended at an atomic cursor
__global__ void __launch_bounds__(256)
cap_keys_kernel(qm_pileup_opt po, const qm_aln *__restrict__ alns, int64_t n, int64_t read_id0, qm_cap_key *__restrict__ out,
                unsigned long long *__restrict__ cnt)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const qm_aln a = alns[i];
    if (!cap_admitted(po, a)) return;
    int rlen = 0;
    for (int k = 0; k < a.n_cigar; ++k) { const int op = a.cigar[k] & 0xf; if (op == 0 || op == 2) rlen += (int)(a.cigar[k] >> 4); }
    qm_cap_key t;
    t.key = (uint64_t)(uint32_t)a.rid << 33 | (uint64_t)(uint32_t)a.pos << 1 | (uint64_t)((a.flag & 0x10) != 0);
    t.read_id = (int32_t)(read_id0 + i);
    t.end = a.pos + (rlen > 0 ? rlen : 1);
    out[atomicAdd(cnt, 1ull)] = t;
}

__global__ void __launch_bounds__(256)
cap_ids_kernel(const qm_cap_key *__restrict__ all, int64_t n, uint64_t *__restrict__ ids)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) ids[i] = (uint64_t)(int64_t)all[i].read_id;
}

// the union in read-id order (ids[] sorted, perm[] their input positions): keys and ends in that order, *rep raised where an id repeats
__global__ void __launch_bounds__(256)
cap_gather_kernel(const qm_cap_key *__restrict__ all, const uint64_t *__restrict__ ids, const uint32_t *__restrict__ perm, int64_t n,
                  uint64_t *__restrict__ keys, int32_t *__restrict__ ends, unsigned long long *__restrict__ rep)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (i > 0 && ids[i - 1] == ids[i]) atomicAdd(rep, 1ull);
    const qm_cap_key t = all[perm[i]];
    keys[i] = t.key;
    ends[i] = t.end;
}

// htslib's pileup iterator over the admitted reads in BAM order: keys[i] / ends[perm[i]] describe the read at sorted position i;
// drop[perm[i]] = 1 for a read the iterator refuses.  Returns the number refused.
int64_t replay_depth_cap(const uint64_t *keys, const uint32_t *perm, const int32_t *ends, int64_t n, int max_depth, uint8_t *drop)
{
    struct Node { int tid; int64_t beg, end; bool gone; };
    std::vector<Node> nodes;                                           // buffered reads in arrival order
    using HeapItem = std::pair<std::pair<int, int64_t>, size_t>;       // ((contig, end), node)
    std::priority_queue<HeapItem, std::vector<HeapItem>, std::greater<HeapItem>> by_end;
    size_t head = 0;
    int cur_tid = 0, last_tid = -1;
    int64_t cur_pos = 0, last_pos = -1, in_use = 1;                    // the spare tail node counts
    int64_t n_dropped = 0;
    for (int64_t i = 0; i < n; ++i) {
        const uint64_t key = keys[i];
        const size_t rec = perm[i];
        const int tid = (int)(key >> 33);
        const int64_t beg = (int64_t)((key >> 1) & 0xffffffffull), end = ends[rec];
        while (last_tid > cur_tid || (last_tid == cur_tid && last_pos > cur_pos)) {
            while (!by_end.empty() && (by_end.top().first.first < cur_tid || (by_end.top().first.first == cur_tid && by_end.top().first.second <= cur_pos))) {
                nodes[by_end.top().second].gone = true;
                --in_use;
                by_end.pop();
            }
            while (head < nodes.size() && nodes[head].gone) ++head;
            if (head < nodes.size() && cur_tid < nodes[head].tid) { cur_tid = nodes[head].tid; cur_pos = nodes[head].beg; }
            else if (head < nodes.size() && cur_pos < nodes[head].beg) cur_pos = nodes[head].beg;
            else ++cur_pos;
        }
        if (cur_tid == tid && cur_pos == beg && in_use > max_depth) { drop[rec] = 1; ++n_dropped; continue; }
        last_tid = tid; last_pos = beg;
        if (end > cur_pos || tid > cur_tid) {
            by_end.push({{tid, end}, nodes.size()});
            nodes.push_back({tid, beg, end, false});
            ++in_use;
        }
    }
    return n_dropped;
}

}  // namespace

extern "C" {

// one qm_cap_key per admitted read, chunk c = pairs pair_id0[c] .. pair_id0[c] + n_pairs[c] - 1.  Synchronous.
int qm_cap_keys(qm_ctx *ctx, const qm_pileup_opt *po, int n_chunks, const qm_aln *const *d_alns, const int64_t *n_pairs,
                const int64_t *pair_id0, qm_cap_key *d_out, int64_t *h_n_out, void *stream)
{
    if (!ctx || !po || !h_n_out || n_chunks < 0 || (n_chunks > 0 && (!d_alns || !n_pairs || !pair_id0))) return QM_EINVAL;
    *h_n_out = 0;
    int64_t N = 0;
    for (int c = 0; c < n_chunks; ++c) {
        if (n_pairs[c] < 0 || pair_id0[c] < 0) return QM_EINVAL;
        if (pair_id0[c] + n_pairs[c] > (1ll << 30)) return qm_fail(ctx, QM_ELIMIT, "qm_depth_cap: pair ids of 2^30 and above do not fit a read id");
        N += 2 * n_pairs[c];
    }
    if (N == 0) return QM_OK;
    if (!d_out) return QM_EINVAL;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 33, 256, &p);
    if (rc) return rc;
    unsigned long long *cnt = (unsigned long long *)p, h = 0;
    QM_CUDA(ctx, cudaMemsetAsync(cnt, 0, 8, st));
    for (int c = 0; c < n_chunks; ++c) {
        const int64_t n = 2 * n_pairs[c];
        if (n) cap_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(*po, d_alns[c], n, 2 * pair_id0[c], d_out, cnt);
    }
    QM_CUDA(ctx, cudaGetLastError());
    QM_CUDA(ctx, cudaMemcpyAsync(&h, cnt, 8, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    *h_n_out = (int64_t)h;
    return QM_OK;
}

// the replay over the union of every rank's cap tuples; the drop bytes of this rank's reads.  Synchronous.
int qm_depth_cap_keys(qm_ctx *ctx, const qm_cap_key *d_all, int64_t n_all, int max_depth, int n_chunks, const int64_t *n_pairs,
                      const int64_t *pair_id0, uint8_t *const *d_drop, int64_t *h_n_dropped_all, void *stream)
{
    if (!ctx || n_all < 0 || (n_all > 0 && !d_all) || max_depth < 1 || n_chunks < 0 || (n_chunks > 0 && (!n_pairs || !pair_id0 || !d_drop)))
        return QM_EINVAL;
    for (int c = 0; c < n_chunks; ++c) if (n_pairs[c] < 0 || pair_id0[c] < 0) return QM_EINVAL;
    if (h_n_dropped_all) *h_n_dropped_all = 0;
    if (n_all > 0x7fffffffll) return qm_fail(ctx, QM_ELIMIT, "qm_depth_cap: more than 2^31 records");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t N = n_all;
    std::vector<uint64_t> h_keys((size_t)N), h_ids((size_t)N);
    std::vector<uint32_t> h_perm((size_t)N);
    std::vector<int32_t> h_ends((size_t)N);
    if (N > 0) {
        // scratch 24: ids | id perm | keys | ends | perm | repeat counter
        auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
        const size_t o_ids = 0, o_iperm = al((size_t)N * 8), o_keys = o_iperm + al((size_t)N * 4), o_ends = o_keys + al((size_t)N * 8);
        const size_t o_perm = o_ends + al((size_t)N * 4), o_cnt = o_perm + al((size_t)N * 4);
        void *p = nullptr;
        int rc = qm_scratch_reserve(ctx, 24, o_cnt + 256, &p);
        if (rc) return rc;
        char *b = (char *)p;
        uint64_t *ids = (uint64_t *)(b + o_ids), *keys = (uint64_t *)(b + o_keys);
        int32_t *ends = (int32_t *)(b + o_ends);
        uint32_t *iperm = (uint32_t *)(b + o_iperm), *perm = (uint32_t *)(b + o_perm);
        unsigned long long *rep = (unsigned long long *)(b + o_cnt), h_rep = 0;
        QM_CUDA(ctx, cudaMemsetAsync(rep, 0, 8, st));
        // read-id order first (the same input on every rank, whatever order the all-gather delivered), then BAM order: the stable sort
        // keeps ties in read order, which is the input order of a single device
        cap_ids_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(d_all, N, ids);
        rc = qm_sort_ids(ctx, ids, iperm, N, "qm_depth_cap_keys", st);
        if (rc) return rc;
        cap_gather_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(d_all, ids, iperm, N, keys, ends, rep);
        QM_CUDA(ctx, cudaGetLastError());
        QM_CUDA(ctx, cudaMemcpyAsync(&h_rep, rep, 8, cudaMemcpyDeviceToHost, st));
        QM_CUDA(ctx, cudaStreamSynchronize(st));
        if (h_rep) return qm_fail(ctx, QM_EINVAL, "qm_depth_cap_keys: %llu read ids occur more than once in the union", h_rep);
        QM_CUDA(ctx, cudaMemcpyAsync(h_ids.data(), ids, (size_t)N * 8, cudaMemcpyDeviceToHost, st));
        QM_CUDA(ctx, cudaMemcpyAsync(h_ends.data(), ends, (size_t)N * 4, cudaMemcpyDeviceToHost, st));
        rc = qm_sort_pairs(ctx, keys, perm, N, 48, st);
        if (rc) return rc;
        QM_CUDA(ctx, cudaMemcpyAsync(h_keys.data(), keys, (size_t)N * 8, cudaMemcpyDeviceToHost, st));
        QM_CUDA(ctx, cudaMemcpyAsync(h_perm.data(), perm, (size_t)N * 4, cudaMemcpyDeviceToHost, st));
        QM_CUDA(ctx, cudaStreamSynchronize(st));
    }
    std::vector<uint8_t> drop((size_t)N, 0);                           // by position in read-id order
    const int64_t n_dropped = replay_depth_cap(h_keys.data(), h_perm.data(), h_ends.data(), N, max_depth, drop.data());
    // the local reads: chunk c holds read ids [2 pair_id0[c], 2 (pair_id0[c] + n_pairs[c])), a contiguous run of the sorted ids
    std::vector<std::vector<uint8_t>> local((size_t)n_chunks);
    for (int c = 0; c < n_chunks; ++c) {
        const int64_t n = 2 * n_pairs[c], r0 = 2 * pair_id0[c];
        if (!n) continue;
        local[(size_t)c].assign((size_t)n, 0);
        for (auto it = std::lower_bound(h_ids.begin(), h_ids.end(), (uint64_t)r0); it != h_ids.end() && (int64_t)*it < r0 + n; ++it)
            local[(size_t)c][(size_t)((int64_t)*it - r0)] = drop[(size_t)(it - h_ids.begin())];
        QM_CUDA(ctx, cudaMemcpyAsync(d_drop[c], local[(size_t)c].data(), (size_t)n, cudaMemcpyHostToDevice, st));
    }
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    if (h_n_dropped_all) *h_n_dropped_all = n_dropped;
    return QM_OK;
}

// chunks: the sample's records in input order.  d_drop[c]: 2 * n_pairs[c] bytes, 1 = the iterator dropped the read.  The export and
// the replay above on one device, pair ids = running pair offsets.  Synchronous.
int qm_depth_cap(qm_ctx *ctx, const qm_pileup_opt *po, int n_chunks, const qm_aln *const *d_alns, const int64_t *n_pairs, int max_depth,
                 uint8_t *const *d_drop, int64_t *h_n_dropped, void *stream)
{
    if (!ctx || !po || n_chunks < 0 || max_depth < 1 || (n_chunks > 0 && (!d_alns || !n_pairs || !d_drop))) return QM_EINVAL;
    int64_t N = 0;
    std::vector<int64_t> id0((size_t)n_chunks);
    for (int c = 0; c < n_chunks; ++c) { if (n_pairs[c] < 0) return QM_EINVAL; id0[(size_t)c] = N / 2; N += 2 * n_pairs[c]; }
    if (h_n_dropped) *h_n_dropped = 0;
    if (N == 0) return QM_OK;
    if (N > 0x7fffffffll) return qm_fail(ctx, QM_ELIMIT, "qm_depth_cap: more than 2^31 records");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 32, (size_t)N * sizeof(qm_cap_key), &p);
    if (rc) return rc;
    qm_cap_key *tuples = (qm_cap_key *)p;
    int64_t n_t = 0;
    rc = qm_cap_keys(ctx, po, n_chunks, d_alns, n_pairs, id0.data(), tuples, &n_t, stream);
    if (rc) return rc;
    return qm_depth_cap_keys(ctx, tuples, n_t, max_depth, n_chunks, n_pairs, id0.data(), d_drop, h_n_dropped, stream);
}

}  // extern "C"
