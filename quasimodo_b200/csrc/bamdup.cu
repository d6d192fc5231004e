// bamdup.cu -- duplicate marking of an existing coordinate-sorted BAM with the rule of dedup.cu (`picard MarkDuplicates`, the
// reference's rule `rmdup`, rules/rmdup.smk:13-16; `qm_driver rmdup` is its one-for-one replacement).
//
// The host has inflated the BGZF blocks and validated every record; what comes here is the uncompressed record stream and the
// byte offset of EVERY record of the file.  On the device:
//   1. one warp per record reads its raw bytes: the flag, the end code {contig, unclipped 5' coordinate, strand} from a
//      lane-parallel CIGAR walk (S and H at both ends count as clipped), the score (sum of the stored qualities >= 15, lane-strided,
//      any length) and the name hash of bamin.cu;
//   2. (hash, file index) pairs are sorted and the two primary records of a name paired by bamin.cu's kernel;
//   3. one thread per record finds its unit and the unit's id: a pair unit is the two paired records, a lone unit any other
//      primary record; the id is the file index of the pair end with the smaller {contig, unclipped 5' coordinate} (the earlier
//      record on a tie) or of the one placed record.  The record that holds its unit's id emits the unit's qm_dup_key;
//   4. the decision of dedup.cu over the tuples (ties to the lowest id = picard's read1IndexInFile);
//   5. one verdict byte per record: 1 for the placed records of a duplicate unit.  Unplaced mates, secondary and supplementary
//      records are never duplicates.  A 0x400 flag in the input plays no part.
#include "bamrec.cuh"

namespace {

// record f: flag, end (QM_DUP_NO_END when the record is not placed: 0x4, no contig or no CIGAR), score, name hash
__global__ void __launch_bounds__(128)
bamdup_decode_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ rec_off, int64_t n, int hash_bits,
                     uint16_t *__restrict__ flags, uint32_t *__restrict__ ends, int32_t *__restrict__ scores, uint64_t *__restrict__ hash,
                     unsigned long long *__restrict__ n_bad)
{
    const int lane = threadIdx.x & 31;
    const int64_t f = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (f >= n) return;
    const uint8_t *r = bytes + rec_off[f];
    const int l_name = r[12], n_cig = (int)qm_ld_u16(r + 16);
    const uint32_t flag = qm_ld_u16(r + 18);
    const int32_t rid = (int32_t)qm_ld_u32(r + 4), pos = (int32_t)qm_ld_u32(r + 8), L = (int32_t)qm_ld_u32(r + 20);
    const uint8_t *cig = r + 36 + l_name, *qual = cig + 4 * n_cig + (L + 1) / 2;
    // score: a QUAL of '*' (first byte 0xff) scores 0
    int s = 0;
    if (L > 0 && qual[0] != 0xff)
        for (int i = lane; i < L; i += 32) { const int v = qual[i]; s += v >= 15 ? v : 0; }
    // CIGAR: reference span (M D N = X) and the first / last operation that is not a clip
    int span = 0, first = n_cig, last = -1;
    for (int k = lane; k < n_cig; k += 32) {
        const uint32_t w = qm_ld_u32(cig + 4 * k), op = w & 0xf;
        if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) span += (int)(w >> 4);
        if (op != 4 && op != 5) { first = min(first, k); last = max(last, k); }
    }
    for (int o = 16; o; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        span += __shfl_xor_sync(0xffffffffu, span, o);
        first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
        last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
    }
    // clipped bases before the first and after the last aligned operation (a CIGAR of clips alone: all of them lead)
    int lead = 0, trail = 0;
    for (int k = lane; k < n_cig; k += 32) {
        const int len = (int)(qm_ld_u32(cig + 4 * k) >> 4);
        if (k < first) lead += len;
        else if (k > last && last >= 0) trail += len;
    }
    for (int o = 16; o; o >>= 1) {
        lead += __shfl_xor_sync(0xffffffffu, lead, o);
        trail += __shfl_xor_sync(0xffffffffu, trail, o);
    }
    if (lane != 0) return;
    flags[f] = (uint16_t)flag;
    scores[f] = s;
    hash[f] = qm_bam_name_hash(r, hash_bits);
    uint32_t e = QM_DUP_NO_END;
    if (!(flag & 0x4) && rid >= 0 && n_cig > 0) {
        const bool rev = (flag & 0x10) != 0;
        const int64_t coord = rev ? (int64_t)pos + span - 1 + trail : (int64_t)pos - lead;
        if (coord + QM_DUP_COORD_BIAS < 0 || coord + QM_DUP_COORD_BIAS >= (1 << 26) || rid >= 16) atomicAdd(n_bad, 1ull);
        else e = ((uint32_t)rid << 26 | (uint32_t)(coord + QM_DUP_COORD_BIAS)) << 1 | (rev ? 1u : 0u);
    }
    ends[f] = e;
}

// the id of record f's unit, -1 for none (a secondary or supplementary record, or a unit without a placed end)
__device__ __forceinline__ int64_t unit_id(const uint16_t *flags, const uint32_t *ends, const int32_t *partner, int64_t f)
{
    if (flags[f] & 0x900) return -1;
    const int64_t g = partner[f];
    const bool pf = ends[f] != QM_DUP_NO_END;
    if (g < 0) return pf ? f : -1;
    const bool pg = ends[g] != QM_DUP_NO_END;
    if (pf && pg) {
        const uint32_t cf = ends[f] >> 1, cg = ends[g] >> 1;       // {contig, coordinate} without the strand
        return cf < cg ? f : cg < cf ? g : min(f, g);
    }
    return pf ? f : pg ? g : -1;
}

// one thread per record: its unit id; the unit's tuple from the record that holds the id (warp-aggregated cursor); units counted
// once, at the record that opens them (a lone record, or the first of a pair in the file)
__global__ void __launch_bounds__(256)
bamdup_units_kernel(const uint16_t *__restrict__ flags, const uint32_t *__restrict__ ends, const int32_t *__restrict__ scores,
                    const int32_t *__restrict__ partner, int64_t n, int32_t *__restrict__ uid, qm_dup_key *__restrict__ out,
                    unsigned long long *__restrict__ cnt)
{
    const int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    bool emit = false, opens = false;
    qm_dup_key t;
    if (f < n) {
        const int64_t id = unit_id(flags, ends, partner, f);
        uid[f] = (int32_t)id;
        const int64_t g = partner[f];
        opens = !(flags[f] & 0x900) && (g < 0 || f < g);
        if (id == f) {
            emit = true;
            const bool pf = ends[f] != QM_DUP_NO_END, pg = g >= 0 && ends[g] != QM_DUP_NO_END;
            t = qm_dup_tuple(id, pf, ends[f], scores[f], pg, pg ? ends[g] : QM_DUP_NO_END, pg ? scores[g] : 0);
        }
    }
    const unsigned me = __ballot_sync(0xffffffffu, emit), mo = __ballot_sync(0xffffffffu, opens);
    unsigned long long base = 0;
    if (lane == 0) {
        if (me) base = atomicAdd(cnt, (unsigned long long)__popc(me));
        if (mo) atomicAdd(cnt + 1, (unsigned long long)__popc(mo));
    }
    base = __shfl_sync(0xffffffffu, base, 0);
    if (emit) out[base + __popc(me & ((1u << lane) - 1))] = t;
}

// record f is a duplicate when it is placed and its unit's id is flagged in the decision (ids sorted: binary search)
__global__ void __launch_bounds__(256)
bamdup_apply_kernel(const uint32_t *__restrict__ ends, const int32_t *__restrict__ uid, int64_t n, const uint64_t *__restrict__ ids,
                    int64_t n_ids, const uint8_t *__restrict__ dup, uint8_t *__restrict__ verdict)
{
    const int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (f >= n) return;
    uint8_t v = 0;
    if (uid[f] >= 0 && ends[f] != QM_DUP_NO_END) {
        const uint64_t want = (uint64_t)uid[f];
        int64_t lo = 0, hi = n_ids;
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (ids[mid] < want) lo = mid + 1; else hi = mid; }
        v = lo < n_ids && ids[lo] == want && dup[lo];
    }
    verdict[f] = v;
}

__global__ void __launch_bounds__(256) bamdup_iota_kernel(uint32_t *v, int64_t n)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) v[i] = (uint32_t)i;
}

inline size_t al256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

extern "C" {

// the body of qm_bam_mark_duplicates with the name hash cut to hash_bits bits (1..64): the tests pair through colliding hashes with it
int qm_bam_mark_duplicates_hashbits(qm_ctx *ctx, const uint8_t *d_bytes, const int64_t *d_rec_off, int64_t n_recs, int hash_bits, uint8_t *d_dup,
                                    int64_t *h_n_units, int64_t *h_n_dup_units, void *stream)
{
    if (!ctx || !h_n_units || !h_n_dup_units || n_recs < 0 || hash_bits < 1 || hash_bits > 64 || (n_recs > 0 && (!d_bytes || !d_rec_off || !d_dup)))
        return QM_EINVAL;
    *h_n_units = *h_n_dup_units = 0;
    if (n_recs > 0x7fffffffll) return qm_fail(ctx, QM_ELIMIT, "qm_bam_mark_duplicates: %lld records: at most 2^31 - 1", (long long)n_recs);
    if (n_recs == 0) return QM_OK;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = n_recs;
    // scratch 41: per record flag | end | score | hash | perm | partner | unit id, then the tuples and two counters
    const size_t o_end = al256((size_t)n * 2), o_sc = o_end + al256((size_t)n * 4), o_hash = o_sc + al256((size_t)n * 4);
    const size_t o_perm = o_hash + al256((size_t)n * 8), o_part = o_perm + al256((size_t)n * 4), o_uid = o_part + al256((size_t)n * 4);
    const size_t o_tup = o_uid + al256((size_t)n * 4), o_cnt = o_tup + al256((size_t)n * sizeof(qm_dup_key));
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 41, o_cnt + 256, &p);
    if (rc) return rc;
    char *b = (char *)p;
    uint16_t *flags = (uint16_t *)b;
    uint32_t *ends = (uint32_t *)(b + o_end), *perm = (uint32_t *)(b + o_perm);
    int32_t *scores = (int32_t *)(b + o_sc), *partner = (int32_t *)(b + o_part), *uid = (int32_t *)(b + o_uid);
    uint64_t *hash = (uint64_t *)(b + o_hash);
    qm_dup_key *tuples = (qm_dup_key *)(b + o_tup);
    unsigned long long *cnt = (unsigned long long *)(b + o_cnt);         // tuples, units, records whose end code does not fit
    const int sp = qm_prof_begin(ctx, QM_ST_OTHER, st);
    QM_CUDA(ctx, cudaMemsetAsync(cnt, 0, 24, st));
    bamdup_decode_kernel<<<(unsigned)((n * 32 + 127) / 128), 128, 0, st>>>(d_bytes, d_rec_off, n, hash_bits, flags, ends, scores, hash, cnt + 2);
    bamdup_iota_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(perm, n);
    QM_CUDA(ctx, cudaGetLastError());
    rc = qm_sort_pairs(ctx, hash, perm, n, hash_bits, st);
    if (rc) return rc;
    QM_CUDA(ctx, qm_bam_pair_launch(d_bytes, d_rec_off, flags, hash, perm, n, partner, st));
    bamdup_units_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(flags, ends, scores, partner, n, uid, tuples, cnt);
    QM_CUDA(ctx, cudaGetLastError());
    unsigned long long h[3] = {0, 0, 0};
    QM_CUDA(ctx, cudaMemcpyAsync(h, cnt, 24, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    if (h[2]) return qm_fail(ctx, QM_ELIMIT, "qm_bam_mark_duplicates: %llu records lie beyond what the 30-bit end code holds (contigs of up to 2^26 - 4096 bases, 16 contigs)", h[2]);
    const uint64_t *ids = nullptr;
    const uint8_t *dup = nullptr;
    int64_t n_dup = 0;
    rc = qm_dup_decide(ctx, tuples, (int64_t)h[0], &ids, &dup, &n_dup, st);
    if (rc) return rc;
    bamdup_apply_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(ends, uid, n, ids, (int64_t)h[0], dup, d_dup);
    QM_CUDA(ctx, cudaGetLastError());
    qm_prof_end(ctx, QM_ST_OTHER, sp, st, 7);
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    *h_n_units = (int64_t)h[1];
    *h_n_dup_units = n_dup;
    return QM_OK;
}

int qm_bam_mark_duplicates(qm_ctx *ctx, const uint8_t *d_bytes, const int64_t *d_rec_off, int64_t n_recs, uint8_t *d_dup, int64_t *h_n_units,
                           int64_t *h_n_dup_units, void *stream)
{
    return qm_bam_mark_duplicates_hashbits(ctx, d_bytes, d_rec_off, n_recs, 64, d_dup, h_n_units, h_n_dup_units, stream);
}

// host bytes in and verdicts out: the record stream, the offsets and the verdicts are staged in scratch 40, then as
// qm_bam_mark_duplicates on the context's stream
int qm_bam_mark_duplicates_host(qm_ctx *ctx, const uint8_t *h_bytes, int64_t n_bytes, const int64_t *h_rec_off, int64_t n_recs, uint8_t *h_dup,
                                int64_t *h_n_units, int64_t *h_n_dup_units)
{
    if (!ctx || !h_n_units || !h_n_dup_units || n_bytes < 0 || n_recs < 0 || (n_bytes > 0 && !h_bytes) || (n_recs > 0 && (!h_rec_off || !h_dup)))
        return QM_EINVAL;
    *h_n_units = *h_n_dup_units = 0;
    if (n_recs == 0) return QM_OK;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t o_off = al256((size_t)n_bytes), o_dup = o_off + al256((size_t)n_recs * 8);
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 40, o_dup + al256((size_t)n_recs), &p);
    if (rc) return rc;
    char *b = (char *)p;
    cudaStream_t st = ctx->own_stream;
    int sp = qm_prof_begin(ctx, QM_ST_H2D, st);
    if (n_bytes) QM_CUDA(ctx, cudaMemcpyAsync(b, h_bytes, (size_t)n_bytes, cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync(b + o_off, h_rec_off, (size_t)n_recs * 8, cudaMemcpyHostToDevice, st));
    qm_prof_end(ctx, QM_ST_H2D, sp, st, 0);
    rc = qm_bam_mark_duplicates(ctx, (const uint8_t *)b, (const int64_t *)(b + o_off), n_recs, (uint8_t *)(b + o_dup), h_n_units, h_n_dup_units, st);
    if (rc) return rc;
    sp = qm_prof_begin(ctx, QM_ST_D2H, st);
    QM_CUDA(ctx, cudaMemcpyAsync(h_dup, b + o_dup, (size_t)n_recs, cudaMemcpyDeviceToHost, st));
    qm_prof_end(ctx, QM_ST_D2H, sp, st, 0);
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    return QM_OK;
}

}  // extern "C"
