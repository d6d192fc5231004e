// pileup.cu -- per-column allele counting with the read admission and mate-overlap rules of
// `bcftools mpileup -B` (reference call site rules/vcfcall.smk:115; upstream htslib sam.c
// bam_plp_push / overlap_push / tweak_overlap_quality and bcftools bam2bcf.c bcf_call_glfgen;
// semantics SURVEY.md A.8-A.9; depth cap disabled, see DESIGN.md "deviations").
//
// One warp per read pair: the mate-overlap quality rewrite is pair-local, so both mates' qualities sit
// in shared memory (BAM SEQ orientation) and the lanes walk the query bases.  Almost every base of a read equals the
// reference and passes the quality threshold, so those are not counted one by one (round 1 did: two
// `red.global.add` per base, 1.2 G reductions per 2 M pairs, the whole kernel time):
//   * coverage is a DIFFERENCE ARRAY per strand: +1 at the first column of an M block, -1 behind its last;
//   * a base that fails the threshold, or differs from the reference, is one reduction into minus[strand][column]
//     (plus its own channel when it counts);
//   * pileup_finish_kernel turns the prefix sum of the difference array into the depth channel and
//     coverage - minus into the reference base's channel.
// Same integers as counting every base; 4 reductions per read + ~0.05 per base instead of 2 per base.
#include <algorithm>
#include <cub/device/device_scan.cuh>
#include "pipeline.cuh"

namespace {

constexpr int kMaxLen = 512;          // read length limit of this kernel (BASELINE reads are 150 / 250)
constexpr int kWarpsPerBlock = 4;

struct AlnS {                         // the fields of a qm_aln the walkers need, in shared memory
    int32_t pos, n_cigar;
    int32_t m0, m1;                   // gap-free alignment ([clip] M [clip], the common case): query bases [m0, m1) are the
                                      // M bases, base i sits at pos + i - m0; m1 = 0: not gap-free, walk the CIGAR
    uint32_t cigar[QM_MAX_CIGAR];
};

// [clip] <len>M [clip] ?  -> the query interval of the M bases
__device__ __forceinline__ void simple_span(const uint32_t *cigar, int nc, int32_t *m0, int32_t *m1)
{
    int k = 0, x = 0;
    *m0 = 0; *m1 = 0;
    if (k < nc && (cigar[k] & 0xf) == 4) { x = (int)(cigar[k] >> 4); ++k; }
    if (k >= nc || (cigar[k] & 0xf) != 0) return;
    const int len = (int)(cigar[k] >> 4);
    ++k;
    if (k < nc && (cigar[k] & 0xf) == 4) ++k;
    if (k != nc) return;
    *m0 = x; *m1 = x + len;
}

// reference position (contig coordinate) of query base i in SEQ order, or -1 when i is not an M-type base
__device__ __forceinline__ int rpos_of(const AlnS &a, int i)
{
    if (a.m1) return i >= a.m0 && i < a.m1 ? a.pos + i - a.m0 : -1;
    int x = 0, p = a.pos;
    for (int k = 0; k < a.n_cigar; ++k) {
        const int op = a.cigar[k] & 0xf, len = (int)(a.cigar[k] >> 4);
        if (op == 0) { if (i < x + len) return p + (i - x); x += len; p += len; }
        else if (op == 1 || op == 4) { if (i < x + len) return -1; x += len; }
        else if (op == 2) p += len;
    }
    return -1;
}
// query index (SEQ order) of the M-type base aligned to contig position p, or -1
__device__ __forceinline__ int qidx_of(const AlnS &a, int p)
{
    if (a.m1) return p >= a.pos && p < a.pos + (a.m1 - a.m0) ? a.m0 + (p - a.pos) : -1;
    int x = 0, pp = a.pos;
    for (int k = 0; k < a.n_cigar; ++k) {
        const int op = a.cigar[k] & 0xf, len = (int)(a.cigar[k] >> 4);
        if (op == 0) { if (p >= pp && p < pp + len) return x + (p - pp); x += len; pp += len; }
        else if (op == 1 || op == 4) x += len;
        else if (op == 2) { if (p < pp + len) return -1; pp += len; }
    }
    return -1;
}

__device__ __forceinline__ void red_add(int32_t *p) { atomicAdd(p, 1); }   // result unused => RED.ADD

// four bytes from any address (shared or global): the two aligned words around it, funnel-shifted; reads up to 4 bytes past
__device__ __forceinline__ uint32_t ld4(const uint8_t *p)
{
    const uint32_t *w = (const uint32_t *)((uintptr_t)p & ~(uintptr_t)3);
    return __funnelshift_r(w[0], w[1], (unsigned)((uintptr_t)p & 3u) * 8u);
}

// ---- indel allele table (SURVEY.md 8a9 "indel alleles into a small hash table", 8e "gather of the sparse indel table") ----
// Open addressing on 64-bit keys: anchor position (forward coordinate on the concatenated contigs, 32 bits) | type (1) |
// length (8, clamped to 255) | "an N among the inserted bases" (1) | the first 11 inserted bases, 2 bits each (22).  Two int32
// counters per slot (forward / reverse reads).  A full table raises the overflow flag; the fetch then fails with QM_ELIMIT.
constexpr unsigned long long kIndelEmpty = ~0ull;
constexpr int kIndelSeqBases = 11;
struct IndelView { unsigned long long *keys; int32_t *cnt; uint32_t mask; int *overflow; };

__device__ __forceinline__ unsigned long long indel_key(int64_t gpos, int type, int len, uint32_t seq, int has_n)
{
    return (unsigned long long)(uint32_t)gpos << 32 | (unsigned long long)(type & 1) << 31 | (unsigned long long)(len > 255 ? 255 : len) << 23 |
           (unsigned long long)(has_n & 1) << 22 | (unsigned long long)(seq & 0x3fffffu);
}
__device__ __forceinline__ void indel_add(const IndelView &T, unsigned long long key, int rev, int n)
{
    uint32_t h = (uint32_t)((key * 0x9E3779B97F4A7C15ull) >> 32) & T.mask;
    for (int probe = 0; probe < 4096; ++probe) {
        const unsigned long long old = atomicCAS(&T.keys[h], kIndelEmpty, key);
        if (old == kIndelEmpty || old == key) { atomicAdd(&T.cnt[2 * h + rev], n); return; }
        h = (h + 1) & T.mask;
    }
    atomicExch(T.overflow, 1);
}

template <int kPre>                  // words per lane of a pair's bases (and of its qualities) held ahead: 64 * kPre >= stride
__global__ void __launch_bounds__(kWarpsPerBlock * 32)
pileup_kernel(IndexView V, qm_pileup_opt po, const qm_aln *__restrict__ alns, const uint8_t *__restrict__ codes,
              const uint8_t *__restrict__ quals, int stride, const int32_t *__restrict__ lens, int64_t n_pairs,
              int32_t *__restrict__ counts, unsigned long long *__restrict__ n_admitted, IndelView T,
              const uint8_t *__restrict__ drop /* may be NULL: reads the depth cap removed */,
              int32_t *__restrict__ cov /* [2][l_pac + 1] difference arrays */, int32_t *__restrict__ minus /* [2][l_pac] */,
              bool wide /* stride even, codes / quals 4-byte aligned, stride <= kMaxLen */)
{
    // The pair's records, bases and qualities come in with a few wide loads per lane, all issued before any is used (round 1
    // walked them byte by byte, one 32-byte sector per warp load and each behind the last: 0.7 TB/s of requests in flight).
    static_assert(sizeof(qm_aln) == 128, "two records = sixteen 16-byte words");
    __shared__ uint4 s_rec[kWarpsPerBlock][16];
    __shared__ __align__(16) uint8_t s_c[kWarpsPerBlock][2 * kMaxLen + 16];      // bases as stored (read orientation); mate e at e * moff
    __shared__ __align__(16) uint8_t s_qr[kWarpsPerBlock][2 * kMaxLen + 16];     // qualities likewise; the mate-overlap rewrite edits them in place
    __shared__ AlnS s_aln[kWarpsPerBlock][2];
    const int lane = qm_lane(), wib = threadIdx.x >> 5;
    const int64_t warp0 = blockIdx.x * (int64_t)kWarpsPerBlock + wib;
    const int64_t n_warps = (int64_t)gridDim.x * kWarpsPerBlock;
    const int64_t L_pac = V.l_pac;
    unsigned long long admitted_local = 0;
    const int moff = wide ? stride : kMaxLen;
    const int n_copy = stride < kMaxLen ? stride : kMaxLen;

    // the NEXT pair's words are fetched into registers before this pair is processed: the loads' latency (~1 us from HBM)
    // runs under ~900 instructions of work instead of in front of them
    uint4 p_rec = {};
    uint32_t p_c[kPre], p_q[kPre];
    int p_len0 = 0, p_len1 = 0;
    auto fetch = [&](int64_t pi) {
        if (lane < 16) p_rec = ((const uint4 *)(alns + 2 * pi))[lane];
        const uint32_t *gc = (const uint32_t *)(codes + 2 * pi * stride), *gq = (const uint32_t *)(quals + 2 * pi * stride);
#pragma unroll
        for (int j = 0; j < kPre; ++j) {
            const int k = lane + 32 * j;
            if (k < (stride >> 1)) { p_c[j] = gc[k]; p_q[j] = gq[k]; }
        }
        p_len0 = lens[2 * pi]; p_len1 = lens[2 * pi + 1];
    };
    if (wide && warp0 < n_pairs) fetch(warp0);

    for (int64_t pi = warp0; pi < n_pairs; pi += n_warps) {
        __syncwarp();
        int len0, len1;
        if (wide) {                                 // 2 * stride bytes of the pair are contiguous and 4-byte aligned
            if (lane < 16) s_rec[wib][lane] = p_rec;
            uint32_t *sc = (uint32_t *)s_c[wib], *sq = (uint32_t *)s_qr[wib];
#pragma unroll
            for (int j = 0; j < kPre; ++j) {
                const int k = lane + 32 * j;
                if (k < (stride >> 1)) { sc[k] = p_c[j]; sq[k] = p_q[j]; }
            }
            len0 = p_len0; len1 = p_len1;
            if (pi + n_warps < n_pairs) fetch(pi + n_warps);
        } else {
            if (lane < 16) s_rec[wib][lane] = ((const uint4 *)(alns + 2 * pi))[lane];
            for (int e = 0; e < 2; ++e)
                for (int k = lane; k < n_copy; k += 32) {
                    s_c[wib][e * moff + k] = codes[(2 * pi + e) * stride + k];
                    s_qr[wib][e * moff + k] = quals[(2 * pi + e) * stride + k];
                }
            len0 = lens[2 * pi]; len1 = lens[2 * pi + 1];
        }
        __syncwarp();
        const qm_aln *g[2] = { (const qm_aln *)&s_rec[wib][0], (const qm_aln *)&s_rec[wib][8] };
        int flag[2], rid[2], tlen[2], L[2];
        bool ok[2], rev[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const uint32_t fm = *(const uint32_t *)&g[e]->flag;           // flag | mapq<<16 | n_cigar<<24
            flag[e] = fm & 0xffff;
            const int mapq = (fm >> 16) & 0xff, nc = fm >> 24;
            rid[e] = g[e]->rid; tlen[e] = g[e]->tlen; L[e] = e ? len1 : len0;
            rev[e] = (flag[e] & 0x10) != 0;
            ok[e] = !(flag[e] & (0x4 | 0x100 | 0x200 | 0x400)) && nc != 0 && nc != 255 && mapq >= po.min_mapq &&
                    !((flag[e] & 0x1) && !(flag[e] & 0x2) && !po.count_orphans) && L[e] <= kMaxLen && !(drop && drop[2 * pi + e]);
            if (ok[e]) {
                if (lane == 0) {
                    s_aln[wib][e].pos = g[e]->pos; s_aln[wib][e].n_cigar = nc;
                    simple_span(g[e]->cigar, nc, &s_aln[wib][e].m0, &s_aln[wib][e].m1);
                }
                if (lane < nc) s_aln[wib][e].cigar[lane] = g[e]->cigar[lane];
            }
        }
        __syncwarp();
        uint8_t *const rd[2] = { s_c[wib], s_c[wib] + moff };
        uint8_t *const qr[2] = { s_qr[wib], s_qr[wib] + moff };
        // base / quality i of mate e in BAM SEQ orientation
        auto seq_base = [&](int e, int i) {
            const int c = rev[e] ? rd[e][L[e] - 1 - i] : rd[e][i];
            return rev[e] ? (c > 3 ? 4 : 3 - c) : c;
        };
        auto qual = [&](int e, int i) -> uint8_t & { return qr[e][rev[e] ? L[e] - 1 - i : i]; };
        // ---- mate overlap: the mate that comes first in coordinate order plays htslib's `a` ----
        if (!po.ignore_overlaps && ok[0] && ok[1] && rid[0] == rid[1] && (flag[0] & 0x2) && !(flag[0] & 0x8) &&
            abs(tlen[0]) < 2 * L[0] && abs(tlen[1]) < 2 * L[1]) {
            const int p0 = s_aln[wib][0].pos, p1 = s_aln[wib][1].pos;
            const int A = (p1 < p0 || (p1 == p0 && (int)rev[1] < (int)rev[0])) ? 1 : 0, B = A ^ 1;
            for (int ia = lane; ia < L[A]; ia += 32) {
                const int p = rpos_of(s_aln[wib][A], ia);
                if (p < 0) continue;
                const int ib = qidx_of(s_aln[wib][B], p);
                if (ib < 0) continue;
                const int qa = qual(A, ia), qb = qual(B, ib);
                if (seq_base(A, ia) == seq_base(B, ib)) {
                    const int q = qa + qb;
                    qual(A, ia) = (uint8_t)(q > 200 ? 200 : q); qual(B, ib) = 0;
                } else if (qa >= qb) { qual(A, ia) = (uint8_t)(0.8 * qa); qual(B, ib) = 0; }
                else { qual(B, ib) = (uint8_t)(0.8 * qb); qual(A, ia) = 0; }
            }
        }
        __syncwarp();
        // ---- counting ----
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            if (!ok[e]) continue;
            ++admitted_local;
            const AlnS &a = s_aln[wib][e];
            const int64_t base = V.off[rid[e]];
            int32_t *const mns = minus + (rev[e] ? L_pac : 0) + base;
            auto count_base = [&](int i, int p) {
                const int c = seq_base(e, i);
                if (qual(e, i) < po.min_bq) red_add(mns + p);                           // covered, not counted
                else if (c != V.refb[base + p]) {                                       // counted in its own channel
                    red_add(mns + p);
                    red_add(counts + (int64_t)((rev[e] ? 6 : 0) + c) * L_pac + base + p);
                }
            };
            if (a.m1 && po.min_bq >= 0 && po.min_bq <= 255) {
                // gap-free alignment: four bases per lane and step; a group whose bases all equal the reference and pass the
                // threshold (most groups) costs three word loads and two SIMD compares
                const int len = a.m1 - a.m0;
                const uint32_t bq4 = (uint32_t)po.min_bq * 0x01010101u;
                for (int t0 = 4 * lane; t0 < len; t0 += 128) {
                    if (t0 + 4 <= len) {
                        const int sidx = rev[e] ? L[e] - 4 - (a.m0 + t0) : a.m0 + t0;     // the group's first byte as stored
                        uint32_t c4 = ld4(rd[e] + sidx), q4 = ld4(qr[e] + sidx);
                        if (rev[e]) { c4 = __byte_perm(c4, 0, 0x0123) ^ 0x03030303u; q4 = __byte_perm(q4, 0, 0x0123); }
                        const uint32_t r4 = ld4(V.refb + base + a.pos + t0);
                        uint32_t att = __vcmpne4(c4, r4) | __vcmpltu4(q4, bq4);
                        for (int k = 0; att; ++k, att >>= 8)
                            if (att & 0xffu) count_base(a.m0 + t0 + k, a.pos + t0 + k);
                    } else {
                        for (int k = 0; t0 + k < len; ++k) count_base(a.m0 + t0 + k, a.pos + t0 + k);
                    }
                }
            } else {
                for (int i = lane; i < L[e]; i += 32) {
                    const int p = rpos_of(a, i);
                    if (p >= 0) count_base(i, p);
                }
            }
            if (lane < a.n_cigar) {          // operation-level channels: lane k owns CIGAR operation k
                int p = a.pos, last_m = -1, x = 0;
                bool started = false;
                for (int k = 0; k < lane; ++k) {
                    const int op = a.cigar[k] & 0xf, len = (int)(a.cigar[k] >> 4);
                    if (op == 0) { p += len; x += len; last_m = p - 1; started = true; }
                    else if (op == 2) p += len;
                    else if (op == 1 || op == 4) x += len;
                }
                const int op = a.cigar[lane] & 0xf, len = (int)(a.cigar[lane] >> 4);
                if (op == 0) {                                                          // coverage of this M block
                    int32_t *const cv = cov + (rev[e] ? L_pac + 1 : 0) + base + p;
                    atomicAdd(cv, 1); atomicAdd(cv + len, -1);
                    if (!started) red_add(counts + 15 * L_pac + base + p);
                } else if (op == 1) {
                    if (last_m >= 0) {
                        red_add(counts + 12 * L_pac + base + last_m);
                        if (T.keys) {                  // the inserted bases as the forward strand of the reference reads them
                            uint32_t seq = 0; int has_n = 0;
                            for (int i = 0; i < len && i < kIndelSeqBases; ++i) { const int c = seq_base(e, x + i); if (c > 3) has_n = 1; else seq |= (uint32_t)c << (2 * i); }
                            indel_add(T, indel_key(base + last_m, 0, len, seq, has_n), rev[e] ? 1 : 0, 1);
                        }
                    }
                } else if (op == 2) {
                    if (last_m >= 0) {
                        red_add(counts + 13 * L_pac + base + last_m);
                        if (T.keys) indel_add(T, indel_key(base + last_m, 1, len, 0, 0), rev[e] ? 1 : 0, 1);
                    }
                    for (int i = 0; i < len; ++i) red_add(counts + (int64_t)(rev[e] ? 11 : 5) * L_pac + base + p + i);
                }
            }
        }
    }
    if (n_admitted && lane == 0 && admitted_local) atomicAdd(n_admitted, admitted_local);
}

// cov holds the inclusive prefix sums of the difference arrays now = reads covering each column, per strand
__global__ void pileup_finish_kernel(IndexView V, const int32_t *__restrict__ cov, const int32_t *__restrict__ minus, int32_t *__restrict__ counts)
{
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t L = V.l_pac;
    if (p >= L) return;
    const int c0 = cov[p], c1 = cov[L + 1 + p];
    if (c0 | c1) {
        counts[14 * L + p] += c0 + c1;
        const int r = V.refb[p];
        if (r < 4) { counts[(int64_t)r * L + p] += c0 - minus[p]; counts[(int64_t)(6 + r) * L + p] += c1 - minus[L + p]; }
    }
}

// [16][l_pac] planes -> [l_pac][16] rows (the count-TSV row order, SURVEY.md B.3)
__global__ void planes_to_rows_kernel(const int32_t *__restrict__ planes, int64_t l_pac, int32_t *__restrict__ rows)
{
    __shared__ int32_t tile[QM_NCH][33];
    const int64_t p0 = blockIdx.x * 32ll;
    for (int c = threadIdx.y; c < QM_NCH; c += blockDim.y) {
        const int64_t p = p0 + threadIdx.x;
        tile[c][threadIdx.x] = p < l_pac ? planes[c * l_pac + p] : 0;
    }
    __syncthreads();
    const int t = threadIdx.y * 32 + threadIdx.x;          // 256 threads: 16 positions x 16 channels per pass
    for (int r = t; r < 32 * QM_NCH; r += 256) {
        const int pos = r / QM_NCH, c = r % QM_NCH;
        if (p0 + pos < l_pac) rows[(p0 + pos) * QM_NCH + c] = tile[c][pos];
    }
}

}  // namespace

extern "C" {

void qm_pileup_opt_default(qm_pileup_opt *p)
{
    p->min_mapq = 0; p->min_bq = 13; p->count_orphans = 0; p->ignore_overlaps = 0;
}

// ---- the indel allele table as an object: device arrays owned by the library ----
struct qm_indel_table {
    qm_ctx *ctx = nullptr;
    unsigned long long *d_keys = nullptr;
    int32_t *d_cnt = nullptr;
    int *d_overflow = nullptr;
    uint32_t cap = 0;
};

int qm_indel_table_create(qm_ctx *ctx, int log2_slots, qm_indel_table **out)
{
    if (!ctx || !out || log2_slots < 8 || log2_slots > 28) return QM_EINVAL;
    *out = nullptr;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    qm_indel_table *t = new qm_indel_table;
    t->ctx = ctx; t->cap = 1u << log2_slots;
    cudaError_t e;
    if ((e = cudaMalloc(&t->d_keys, (size_t)t->cap * 8)) != cudaSuccess || (e = cudaMalloc(&t->d_cnt, (size_t)t->cap * 8)) != cudaSuccess ||
        (e = cudaMalloc(&t->d_overflow, 4)) != cudaSuccess) {
        cudaFree(t->d_keys); cudaFree(t->d_cnt); cudaFree(t->d_overflow); delete t;
        return qm_fail(ctx, QM_ENOMEM, "qm_indel_table_create: %s", cudaGetErrorString(e));
    }
    *out = t;
    return qm_indel_table_reset(t, nullptr);
}

void qm_indel_table_destroy(qm_indel_table *t)
{
    if (!t) return;
    cudaSetDevice(t->ctx->device);
    cudaFree(t->d_keys); cudaFree(t->d_cnt); cudaFree(t->d_overflow);
    delete t;
}

int qm_indel_table_reset(qm_indel_table *t, void *stream)
{
    if (!t) return QM_EINVAL;
    qm_ctx *ctx = t->ctx;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    QM_CUDA(ctx, cudaMemsetAsync(t->d_keys, 0xff, (size_t)t->cap * 8, (cudaStream_t)stream));
    QM_CUDA(ctx, cudaMemsetAsync(t->d_cnt, 0, (size_t)t->cap * 8, (cudaStream_t)stream));
    QM_CUDA(ctx, cudaMemsetAsync(t->d_overflow, 0, 4, (cudaStream_t)stream));
    return QM_OK;
}

namespace {
// slots in use -> records, compacted through a counter (order fixed afterwards by sorting on the key)
__global__ void indel_collect_kernel(IndelView T, uint32_t cap, const IndexView V, qm_indel *__restrict__ out, int64_t max_out,
                                     unsigned long long *__restrict__ n_out)
{
    const uint32_t h = blockIdx.x * blockDim.x + threadIdx.x;
    if (h >= cap) return;
    const unsigned long long k = T.keys[h];
    if (k == kIndelEmpty) return;
    const unsigned long long slot = atomicAdd(n_out, 1ull);
    if ((int64_t)slot >= max_out) return;
    qm_indel r;
    const int64_t g = (int64_t)(k >> 32);
    int rid = 0;
    for (int c = 0; c < V.n_contigs; ++c) if (g >= V.off[c] && g < V.off[c] + V.len[c]) rid = c;
    r.rid = rid; r.pos = (int32_t)(g - V.off[rid]);
    r.type = (uint8_t)((k >> 31) & 1); r.has_n = (uint8_t)((k >> 22) & 1); r.pad[0] = r.pad[1] = 0;
    r.len = (int32_t)((k >> 23) & 0xff);
    r.seq = (uint32_t)(k & 0x3fffffu);
    r.n_fwd = T.cnt[2 * h]; r.n_rev = T.cnt[2 * h + 1];
    r.key = k;
    out[slot] = r;
}
__global__ void indel_merge_kernel(IndelView T, const qm_indel *__restrict__ in, int64_t n)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const qm_indel r = in[i];
    if (r.n_fwd) indel_add(T, r.key, 0, r.n_fwd);
    if (r.n_rev) indel_add(T, r.key, 1, r.n_rev);
    if (!r.n_fwd && !r.n_rev) indel_add(T, r.key, 0, 0);
}
IndelView view_of(qm_indel_table *t)
{
    IndelView T = {nullptr, nullptr, 0, nullptr};
    if (t) { T.keys = t->d_keys; T.cnt = t->d_cnt; T.mask = t->cap - 1; T.overflow = t->d_overflow; }
    return T;
}
}  // namespace

// records of the table, sorted by (position, type, length, bases), on the host.  Synchronous.
int qm_indel_table_fetch_host(qm_indel_table *t, const qm_index *idx, qm_indel *h_out, int64_t max_out, int64_t *n_out)
{
    if (!t || !idx || !n_out || max_out < 0 || (max_out > 0 && !h_out)) return QM_EINVAL;
    qm_ctx *ctx = t->ctx;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->own_stream;
    QM_CUDA(ctx, cudaDeviceSynchronize());
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 21, (size_t)(max_out > 0 ? max_out : 1) * sizeof(qm_indel) + 256, &p);
    if (rc) return rc;
    qm_indel *d_out = (qm_indel *)((char *)p + 256);
    unsigned long long *d_n = (unsigned long long *)p;
    QM_CUDA(ctx, cudaMemsetAsync(d_n, 0, 8, st));
    indel_collect_kernel<<<(t->cap + 255) / 256, 256, 0, st>>>(view_of(t), t->cap, idx->v, d_out, max_out, d_n);
    QM_CUDA(ctx, cudaGetLastError());
    unsigned long long n = 0;
    int ovf = 0;
    QM_CUDA(ctx, cudaMemcpyAsync(&n, d_n, 8, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaMemcpyAsync(&ovf, t->d_overflow, 4, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    *n_out = (int64_t)n;
    if (ovf) return qm_fail(ctx, QM_ELIMIT, "the indel allele table (%u slots) overflowed", t->cap);
    if ((int64_t)n > max_out) return qm_fail(ctx, QM_ELIMIT, "qm_indel_table_fetch_host: %llu alleles exceed max_out=%lld", n, (long long)max_out);
    if (n) QM_CUDA(ctx, cudaMemcpy(h_out, d_out, (size_t)n * sizeof(qm_indel), cudaMemcpyDeviceToHost));
    std::sort(h_out, h_out + n, [](const qm_indel &a, const qm_indel &b) { return a.key < b.key; });
    return QM_OK;
}

// merge records (e.g. another GPU's table, gathered by the caller) into this table: counts add up.  Asynchronous.
int qm_indel_table_merge(qm_indel_table *t, const qm_indel *d_records, int64_t n, void *stream)
{
    if (!t || n < 0 || (n > 0 && !d_records)) return QM_EINVAL;
    if (n == 0) return QM_OK;
    qm_ctx *ctx = t->ctx;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    indel_merge_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(view_of(t), d_records, n);
    QM_CUDA(ctx, cudaGetLastError());
    return QM_OK;
}

int qm_pileup_accumulate_indels(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns,
                                const uint8_t *d_codes, const uint8_t *d_quals, int32_t stride, const int32_t *d_lens,
                                int64_t n_pairs, int32_t *d_counts, qm_indel_table *tab, void *stream)
{
    return qm_pileup_accumulate_masked(ctx, idx, po, d_alns, d_codes, d_quals, stride, d_lens, n_pairs, d_counts, tab, nullptr, stream);
}

// the same with a per-read drop mask (the depth cap's verdict, depthcap.cu): a dropped read is not admitted
int qm_pileup_accumulate_masked(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns,
                                const uint8_t *d_codes, const uint8_t *d_quals, int32_t stride, const int32_t *d_lens,
                                int64_t n_pairs, int32_t *d_counts, qm_indel_table *tab, const uint8_t *d_drop, void *stream)
{
    if (!ctx || !idx || !po || n_pairs < 0 || (n_pairs > 0 && (!d_alns || !d_codes || !d_quals || !d_lens || !d_counts)))
        return QM_EINVAL;
    if (tab && tab->ctx != ctx) return qm_fail(ctx, QM_EINVAL, "the indel table belongs to another context");
    if (n_pairs == 0) return QM_OK;
    // the kernel stages at most kMaxLen bases per read; a longer read would otherwise be dropped without a word
    if (stride > kMaxLen) return qm_fail(ctx, QM_ELIMIT, "qm_pileup_accumulate: reads longer than %d bases (stride %d)", kMaxLen, stride);
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    int64_t blocks = (n_pairs + kWarpsPerBlock - 1) / kWarpsPerBlock;
    const int64_t cap = (int64_t)ctx->sm_count * 16;       // persistent: 16 blocks x 4 warps per SM
    if (blocks > cap) blocks = cap;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t L = idx->v.l_pac;
    if (2 * (L + 1) > 0x7fffffffll) return qm_fail(ctx, QM_ELIMIT, "qm_pileup_accumulate: a reference of %lld bases is beyond the 2^30 the coverage scan indexes", (long long)L);
    // scratch 25: difference arrays [2][L + 1] | minus [2][L] | cub temp
    const size_t cov_bytes = (size_t)2 * (L + 1) * 4, minus_bytes = (size_t)2 * L * 4;
    const size_t o_minus = (cov_bytes + 255) & ~(size_t)255, o_cub = (o_minus + minus_bytes + 255) & ~(size_t)255;
    size_t cub_bytes = 0;
    cub::DeviceScan::InclusiveSum(nullptr, cub_bytes, (int32_t *)nullptr, (int32_t *)nullptr, (int)(2 * (L + 1)), st);
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 25, o_cub + cub_bytes, &p);
    if (rc) return rc;
    int32_t *cov = (int32_t *)p, *minus = (int32_t *)((char *)p + o_minus);
    const int sp = qm_prof_begin(ctx, QM_ST_PILEUP, st);
    QM_CUDA(ctx, cudaMemsetAsync(p, 0, o_minus + minus_bytes, st));
    const bool wide = (stride & 1) == 0 && stride <= kMaxLen && (((uintptr_t)d_codes | (uintptr_t)d_quals) & 3u) == 0;
#define QM_PILEUP_LAUNCH(PRE) pileup_kernel<PRE><<<(unsigned)blocks, kWarpsPerBlock * 32, 0, st>>>( \
        idx->v, *po, d_alns, d_codes, d_quals, stride, d_lens, n_pairs, d_counts, nullptr, view_of(tab), d_drop, cov, minus, wide)
    if (stride <= 192) QM_PILEUP_LAUNCH(3); else if (stride <= 256) QM_PILEUP_LAUNCH(4); else QM_PILEUP_LAUNCH(8);
#undef QM_PILEUP_LAUNCH
    QM_CUDA(ctx, cudaGetLastError());
    // both strands in one scan: a strand's differences sum to zero, so the running sum is back at 0 where the next one starts
    QM_CUDA(ctx, cub::DeviceScan::InclusiveSum((char *)p + o_cub, cub_bytes, cov, cov, (int)(2 * (L + 1)), st));
    pileup_finish_kernel<<<(unsigned)((L + 255) / 256), 256, 0, st>>>(idx->v, cov, minus, d_counts);
    qm_prof_end(ctx, QM_ST_PILEUP, sp, st, 4);
    QM_CUDA(ctx, cudaGetLastError());
    return QM_OK;
}

int qm_pileup_accumulate(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns,
                         const uint8_t *d_codes, const uint8_t *d_quals, int32_t stride, const int32_t *d_lens,
                         int64_t n_pairs, int32_t *d_counts, void *stream)
{
    return qm_pileup_accumulate_indels(ctx, idx, po, d_alns, d_codes, d_quals, stride, d_lens, n_pairs, d_counts, nullptr, stream);
}

int qm_counts_to_rows(qm_ctx *ctx, const qm_index *idx, const int32_t *d_planes, int32_t *d_rows, void *stream)
{
    if (!ctx || !idx || !d_planes || !d_rows) return QM_EINVAL;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t l_pac = idx->v.l_pac;
    planes_to_rows_kernel<<<(unsigned)((l_pac + 31) / 32), dim3(32, 8), 0, (cudaStream_t)stream>>>(d_planes, l_pac, d_rows);
    QM_CUDA(ctx, cudaGetLastError());
    return QM_OK;
}

}  // extern "C"
