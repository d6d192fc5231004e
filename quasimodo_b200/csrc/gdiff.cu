// gdiff.cu -- the SNP truth set of a strain pair from its two genomes (replaces rule `nucmer`, rules/genome_diff.smk:
// `nucmer ref qry; show-snps -CTHlr <(delta-filter -r -q delta)`; SURVEY.md 8a row a13).  The contract is DESIGN.md 5c; the
// CPU restatement that the tests hold this file to is tests/gdiff_oracle.py.
//
//   gdiff_anchor_kernel  one thread per (query strand, query position): the query k-mer (k = min_match) is looked up in the
//                        reference's k-mer index; a hit whose reference k-mer is unique on both strands (IndexView::uniq) that
//                        starts its diagonal run of such hits is extended to a maximal exact match over the packed words, 32
//                        bases at a time (qm_get2_padded, as the seeding walk does).  The thread whose hit is the match's
//                        leftmost unique k-mer writes it, so every anchor is written once.
//   (host)               anchors sorted; collinear clusters chained per (query contig, strand, reference contig) with max_gap /
//                        max_diag / diag_factor, clusters below min_cluster dropped, neighbours within break_len merged.
//   gdiff_gap_kernel     one warp per gap between consecutive anchors of an alignment: global affine-gap DP over the whole
//                        gap rectangle, lanes along each anti-diagonal, one traceback byte per cell in global memory, then
//                        lane 0 walks the traceback.  Tasks run longest first.
//   (host)               indels left-aligned, delta-filter -r -q restated as two weighted chains, rows of show-snps -CTHlr.
#include <algorithm>
#include <chrono>
#include <numeric>
#include <vector>
#include "pipeline.cuh"

namespace {

struct QryView {
    const uint64_t *q2p[2];         // both strands of the concatenated query, padded 2-bit (qm_get2_padded layout); strand 1 is
                                    // the reverse complement of the whole concatenation
    int64_t lq;
    int n;
    int64_t start[2][QM_MAX_CONTIGS], len[QM_MAX_CONTIGS];
};

struct GdAnchor { int32_t s, qc, rc, qs, rs, len; };   // qs: strand coordinate inside query contig qc; rs: inside reference contig rc

__device__ __forceinline__ bool uniq_bit(const IndexView &V, int64_t p) { return (__ldg(&V.uniq[p >> 5]) >> (p & 31)) & 1u; }

__global__ void __launch_bounds__(256)
gdiff_anchor_kernel(IndexView V, QryView Q, GdAnchor *__restrict__ out, int64_t cap, unsigned long long *__restrict__ n_out)
{
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 2 * Q.lq) return;
    const int s = t >= Q.lq;
    const int64_t x = t - (s ? Q.lq : 0);
    const int k = V.k;
    int c = -1;
    for (int i = 0; i < Q.n; ++i) if (x >= Q.start[s][i] && x < Q.start[s][i] + Q.len[i]) c = i;
    const int64_t qb = Q.start[s][c], qe = qb + Q.len[c];
    if (x + k > qe) return;
    const uint64_t *q2 = Q.q2p[s];
    const uint64_t key = qm_grouprev(qm_get2_padded(q2, x)) >> (64 - 2 * k);
    uint32_t first, cnt;
    if (!qm_idx_lookup(V, key, first, cnt) || cnt != 1) return;
    const int64_t p = first;
    if (!uniq_bit(V, p)) return;
    const int rc = qm_pos2rid(V, p);
    const int64_t rb = V.off[rc], re = rb + V.len[rc];
    // the left end of a diagonal run of unique hits only: otherwise the k-mer one base to the left is the same match's
    if (x > qb && p > rb && uniq_bit(V, p - 1) && ((qm_get2_padded(q2, x - 1) ^ qm_get2_padded(V.ref2p, p - 1)) & 3u) == 0) return;
    int64_t a = 0, b = k;
    for (;;) {                      // leftwards, 32 bases per step: the top groups of the words ending at base x - a - 1
        const int64_t avail = min(x - qb - a, p - rb - a);
        if (avail <= 0) break;
        const uint64_t d = qm_get2_padded(q2, x - a - 32) ^ qm_get2_padded(V.ref2p, p - a - 32);
        const int64_t m = min((int64_t)(d ? __clzll(d) >> 1 : 32), avail);
        a += m;
        if (m < 32) break;
    }
    for (;;) {
        const int64_t avail = min(qe - x - b, re - p - b);
        if (avail <= 0) break;
        const uint64_t d = qm_get2_padded(q2, x + b) ^ qm_get2_padded(V.ref2p, p + b);
        const int64_t m = min((int64_t)(d ? (__ffsll((long long)d) - 1) >> 1 : 32), avail);
        b += m;
        if (m < 32) break;
    }
    // another unique k-mer of the same match further left owns it
    for (int64_t y = p - a; y < p;) {
        const uint32_t w = __ldg(&V.uniq[y >> 5]) >> (y & 31);
        const int64_t nb = min((int64_t)(32 - (y & 31)), p - y);
        if (w & (nb == 32 ? 0xffffffffu : ((1u << nb) - 1))) return;
        y += nb;
    }
    const unsigned long long i = atomicAdd(n_out, 1ull);
    if ((int64_t)i < cap) {
        GdAnchor A;
        A.s = s; A.qc = c; A.rc = rc; A.qs = (int32_t)(x - a - qb); A.rs = (int32_t)(p - a - rb); A.len = (int32_t)(a + b);
        out[i] = A;
    }
}

struct GdTask {
    int64_t r0, q0;                 // first reference base (forward, concatenated) / first query base (strand s, concatenated)
    int64_t tb_off, buf_off, op_off;
    int32_t n, m, s, pad;
};

constexpr int kNegInf = -(1 << 29);
enum { OP_M = 0, OP_D = 1, OP_I = 2 };

// Cell (i, j): reference bases [0, i) against query bases [0, j).  E = the column ends in a deletion (reference base i - 1
// against a gap), F = in an insertion.  H takes the diagonal on ties, then E, then F; E and F open from H unless extending
// scores strictly more.  Traceback byte: bits 0-1 H's source (0 diagonal, 1 E, 2 F), bit 2 E extends, bit 3 F extends.
__global__ void __launch_bounds__(128)
gdiff_gap_kernel(const uint8_t *__restrict__ refb, const uint8_t *__restrict__ q0s, const uint8_t *__restrict__ q1s,
                 const GdTask *__restrict__ tasks, int64_t n_tasks, int match, int mismatch, int go, int ge,
                 uint8_t *__restrict__ tb_all, int32_t *__restrict__ buf_all, uint8_t *__restrict__ ops_all, int32_t *__restrict__ n_ops)
{
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_tasks) return;
    const GdTask T = tasks[w];
    const int n = T.n, m = T.m;
    const uint8_t *R = refb + T.r0, *Qy = (T.s ? q1s : q0s) + T.q0;
    uint8_t *tb = tb_all + T.tb_off;
    int32_t *H[3] = {buf_all + T.buf_off, buf_all + T.buf_off + (n + 1), buf_all + T.buf_off + 2 * (n + 1)};
    int32_t *E[2] = {buf_all + T.buf_off + 3 * (n + 1), buf_all + T.buf_off + 4 * (n + 1)};
    int32_t *F[2] = {buf_all + T.buf_off + 5 * (n + 1), buf_all + T.buf_off + 6 * (n + 1)};
    const int oe = go + ge;
    for (int d = 0; d <= n + m; ++d) {
        int32_t *Hc = H[d % 3], *Ec = E[d & 1], *Fc = F[d & 1];
        const int32_t *H1 = H[(d + 2) % 3], *H2 = H[(d + 1) % 3], *E1 = E[(d + 1) & 1], *F1 = F[(d + 1) & 1];
        const int ilo = d - m > 0 ? d - m : 0, ihi = d < n ? d : n;
        for (int i = ilo + lane; i <= ihi; i += 32) {
            const int j = d - i;
            int32_t h, e, f;
            uint8_t b;
            if (i == 0 && j == 0) { h = 0; e = f = kNegInf; b = 0; }
            else if (i == 0) { f = -(go + j * ge); e = kNegInf; h = f; b = 2 | (j > 1 ? 8 : 0); }
            else if (j == 0) { e = -(go + i * ge); f = kNegInf; h = e; b = 1 | (i > 1 ? 4 : 0); }
            else {
                const int32_t eo = H1[i - 1] - oe, ex = E1[i - 1] - ge;
                const int32_t fo = H1[i] - oe, fx = F1[i] - ge;
                e = ex > eo ? ex : eo;
                f = fx > fo ? fx : fo;
                b = (ex > eo ? 4 : 0) | (fx > fo ? 8 : 0);
                h = H2[i - 1] + (R[i - 1] == Qy[j - 1] ? match : -mismatch);
                int src = 0;
                if (e > h) { h = e; src = 1; }
                if (f > h) { h = f; src = 2; }
                b |= (uint8_t)src;
            }
            Hc[i] = h; Ec[i] = e; Fc[i] = f;
            tb[(int64_t)i * (m + 1) + j] = b;
        }
        __syncwarp();
    }
    if (lane) return;
    __threadfence_block();
    uint8_t *ops = ops_all + T.op_off;
    int i = n, j = m, state = 0, k = 0;
    while (i > 0 || j > 0) {
        const uint8_t b = tb[(int64_t)i * (m + 1) + j];
        if (state == 0) {
            const int src = b & 3;
            if (src == 0) { ops[k++] = OP_M; --i; --j; }
            else state = src;
        } else if (state == 1) {
            ops[k++] = OP_D;
            state = (b >> 2) & 1 ? 1 : 0;
            --i;
        } else {
            ops[k++] = OP_I;
            state = (b >> 3) & 1 ? 2 : 0;
            --j;
        }
    }
    n_ops[w] = k;                   // written last column first
}

// an alignment under construction: anchors after overlap trimming, then its columns
struct GdAln {
    int s, qc, rc;
    std::vector<GdAnchor> anc;
    std::vector<std::vector<uint8_t>> gap_ops;   // columns of the gap after anchor g
    std::vector<uint8_t> ops, tail;  // all columns (the left extension's first); the right extension's
    int64_t lim_r0 = -1, lim_q0 = -1, lim_r1 = -1, lim_q1 = -1;   // how far the ends may be extended (-1: to the contig's end)
    int64_t rs, re, qs, qe;         // 0-based half-open; query in strand coordinates
    int64_t matches = 0, edits = 0;
    int64_t fqs, fqe;               // query span on the forward strand, 0-based half-open
};

// trim b's front so that it starts past a on both sequences; false when nothing is left of it
bool trim_after(const GdAnchor &a, GdAnchor &b)
{
    const int64_t ov = std::max<int64_t>({0, (int64_t)a.rs + a.len - b.rs, (int64_t)a.qs + a.len - b.qs});
    if (ov >= b.len) return false;
    b.rs += (int32_t)ov; b.qs += (int32_t)ov; b.len -= (int32_t)ov;
    return true;
}

// one group's anchors (sorted by rs, qs) -> clusters: chained like mgaps, every anchor in at most one cluster
std::vector<std::vector<GdAnchor>> cluster_group(const std::vector<GdAnchor> &A, const qm_gdiff_opt &o)
{
    const int n = (int)A.size();
    std::vector<int64_t> score(n);
    std::vector<int> pred(n, -1);
    int maxlen = 0;
    for (auto &x : A) maxlen = std::max(maxlen, x.len);
    for (int j = 0; j < n; ++j) {
        score[j] = A[j].len;
        for (int i = j - 1; i >= 0 && (int64_t)A[j].rs - A[i].rs <= (int64_t)o.max_gap + maxlen; --i) {
            const GdAnchor &a = A[i], &b = A[j];
            if (!(a.rs < b.rs && a.qs < b.qs && a.rs + a.len < b.rs + b.len && a.qs + a.len < b.qs + b.len)) continue;
            const int64_t gr = (int64_t)b.rs - (a.rs + a.len), gq = (int64_t)b.qs - (a.qs + a.len);
            const int64_t sep = std::max(gr, gq);
            if (sep > o.max_gap) continue;
            const double dd = (double)std::llabs(gr - gq);
            if (dd > std::max((double)o.max_diag, (double)o.diag_factor * (double)std::max<int64_t>(sep, 0))) continue;
            const int64_t sc = score[i] + b.len;
            if (sc > score[j] || (sc == score[j] && pred[j] >= 0 && i < pred[j])) { score[j] = sc; pred[j] = i; }
        }
    }
    std::vector<int> order(n);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return score[x] > score[y]; });
    std::vector<char> used(n, 0);
    std::vector<std::vector<GdAnchor>> out;
    for (int e : order) {
        if (used[e]) continue;
        std::vector<GdAnchor> path;
        for (int i = e; i >= 0 && !used[i]; i = pred[i]) { used[i] = 1; path.push_back(A[i]); }
        std::reverse(path.begin(), path.end());
        std::vector<GdAnchor> kept;
        for (auto b : path) {
            if (!kept.empty() && !trim_after(kept.back(), b)) continue;
            kept.push_back(b);
        }
        int64_t tot = 0;
        for (auto &x : kept) tot += x.len;
        if (tot >= o.min_cluster) out.push_back(kept);
    }
    return out;
}

// delta-filter's -r (by = 0) or -q (by = 1): per contig, the heaviest chain of alignments whose starts and ends both increase
void filter_chain(std::vector<GdAln> &al, int by)
{
    auto key = [&](const GdAln &a) { return by ? a.qc : a.rc; };
    auto beg = [&](const GdAln &a) { return by ? a.fqs : a.rs; };
    auto end = [&](const GdAln &a) { return by ? a.fqe : a.re; };
    std::vector<int> idx(al.size());
    std::iota(idx.begin(), idx.end(), 0);
    std::stable_sort(idx.begin(), idx.end(), [&](int x, int y) {
        const GdAln &a = al[x], &b = al[y];
        if (key(a) != key(b)) return key(a) < key(b);
        if (beg(a) != beg(b)) return beg(a) < beg(b);
        return end(a) < end(b);
    });
    std::vector<char> keep(al.size(), 0);
    for (size_t g0 = 0; g0 < idx.size();) {
        size_t g1 = g0;
        while (g1 < idx.size() && key(al[idx[g1]]) == key(al[idx[g0]])) ++g1;
        const int n = (int)(g1 - g0);
        std::vector<int64_t> best(n);
        std::vector<int> pred(n, -1);
        for (int j = 0; j < n; ++j) {
            const GdAln &b = al[idx[g0 + j]];
            best[j] = b.matches;
            for (int i = 0; i < j; ++i) {
                const GdAln &a = al[idx[g0 + i]];
                if (beg(a) < beg(b) && end(a) < end(b) && best[i] + b.matches > best[j]) { best[j] = best[i] + b.matches; pred[j] = i; }
            }
        }
        int e = 0;
        for (int j = 1; j < n; ++j) if (best[j] > best[e]) e = j;
        for (int i = e; i >= 0; i = pred[i]) keep[idx[g0 + i]] = 1;
        g0 = g1;
    }
    std::vector<GdAln> out;
    for (size_t i = 0; i < al.size(); ++i) if (keep[i]) out.push_back(std::move(al[i]));
    al.swap(out);
}

}  // namespace

extern "C" {

void qm_gdiff_opt_default(qm_gdiff_opt *o)
{
    if (!o) return;
    memset(o, 0, sizeof *o);
    o->min_match = 20; o->min_cluster = 65; o->max_gap = 90; o->break_len = 200; o->diag_factor = 0.12f; o->max_diag = 5;
    o->match = 1; o->mismatch = 4; o->gap_open = 6; o->gap_extend = 1;
}

int qm_genome_diff_host(qm_ctx *ctx, const qm_index *idx, const uint8_t *h_qry, int n_qry, const int64_t *h_qlens, const qm_gdiff_opt *opt,
                        qm_gdiff_row *h_rows, int64_t max_rows, int64_t *n_rows, qm_gdiff_aln *h_alns, int64_t max_alns, int64_t *n_alns,
                        double *h_phase_ms)
{
    using clk = std::chrono::steady_clock;
    if (!ctx) return QM_EINVAL;
    if (!idx || !h_qry || !h_qlens || !opt || !n_rows || !n_alns || (max_rows > 0 && !h_rows) || (max_alns > 0 && !h_alns))
        return qm_fail(ctx, QM_EINVAL, "qm_genome_diff_host: NULL argument");
    const qm_gdiff_opt o = *opt;
    const IndexView &V = idx->v;
    if (o.min_match != V.k) return qm_fail(ctx, QM_EINVAL, "qm_genome_diff_host: min_match %d differs from the index's k %d", o.min_match, V.k);
    if (o.max_gap < 0 || o.break_len < 0 || o.max_gap > 4096 || o.break_len > 4096 || o.min_cluster < 0 || o.max_diag < 0 || !(o.diag_factor >= 0.f) ||
        o.match < 1 || o.mismatch < 0 || o.gap_open < 0 || o.gap_extend < 1 || (o.flags & ~(QM_GDIFF_NO_INDELS | QM_GDIFF_KEEP_AMBIGUOUS)))
        return qm_fail(ctx, QM_EINVAL, "qm_genome_diff_host: option out of range (gaps 0..4096, match >= 1, gap_extend >= 1, penalties >= 0)");
    if (n_qry <= 0 || n_qry > QM_MAX_CONTIGS) return qm_fail(ctx, QM_EINVAL, "qm_genome_diff_host: need 1..%d query contigs", QM_MAX_CONTIGS);
    QryView Q = {};
    Q.n = n_qry;
    int64_t lq = 0;
    for (int c = 0; c < n_qry; ++c) {
        if (h_qlens[c] <= 0) return qm_fail(ctx, QM_EINVAL, "qm_genome_diff_host: query contig %d has no bases", c);
        Q.len[c] = h_qlens[c]; Q.start[0][c] = lq; lq += h_qlens[c];
    }
    if (lq >= (1ll << 30)) return qm_fail(ctx, QM_ELIMIT, "qm_genome_diff_host: query longer than 2^30 - 1 bases");
    for (int c = 0; c < n_qry; ++c) Q.start[1][c] = lq - Q.start[0][c] - Q.len[c];
    Q.lq = lq;
    for (int64_t i = 0; i < lq; ++i)
        if (h_qry[i] > 3) return qm_fail(ctx, QM_EINVAL, "qm_genome_diff_host: query base %lld is not A/C/G/T", (long long)i);
    double ms[5] = {0, 0, 0, 0, 0};
    auto t0 = clk::now();
    auto lap = [&](int ph) { const auto t = clk::now(); ms[ph] += std::chrono::duration<double, std::milli>(t - t0).count(); t0 = t; };
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    const cudaStream_t st = ctx->own_stream;

    // ---- both query strands, as bytes (gap DP) and padded 2-bit words (anchors) ----
    std::vector<uint8_t> qs[2];
    qs[0].assign(h_qry, h_qry + lq);
    qs[1].resize((size_t)lq);
    for (int64_t i = 0; i < lq; ++i) qs[1][(size_t)i] = (uint8_t)(3 - h_qry[lq - 1 - i]);
    const size_t n_words = (size_t)(lq + 32 + 31) / 32 + 2;
    std::vector<uint64_t> q2[2];
    for (int s = 0; s < 2; ++s) {
        q2[s].assign(n_words, 0ull);
        for (int64_t x = 0; x < lq; ++x) q2[s][(size_t)(x + 32) >> 5] |= (uint64_t)qs[s][(size_t)x] << (2 * ((x + 32) & 31));
    }
    std::vector<uint8_t> refb((size_t)V.l_pac);
    const int64_t cap = 2 * lq + 1;
    uint8_t *d_qb = nullptr;
    uint64_t *d_q2 = nullptr;
    GdAnchor *d_anc = nullptr;
    unsigned long long *d_n = nullptr;
    auto free_all = [&]() { cudaFree(d_qb); cudaFree(d_q2); cudaFree(d_anc); cudaFree(d_n); };
    cudaError_t e;
    if ((e = cudaMalloc(&d_qb, 2 * (size_t)lq)) != cudaSuccess || (e = cudaMalloc(&d_q2, 2 * n_words * 8)) != cudaSuccess ||
        (e = cudaMalloc(&d_anc, (size_t)cap * sizeof(GdAnchor))) != cudaSuccess || (e = cudaMalloc(&d_n, 8)) != cudaSuccess ||
        (e = cudaMemcpyAsync(d_qb, qs[0].data(), (size_t)lq, cudaMemcpyHostToDevice, st)) != cudaSuccess ||
        (e = cudaMemcpyAsync(d_qb + lq, qs[1].data(), (size_t)lq, cudaMemcpyHostToDevice, st)) != cudaSuccess ||
        (e = cudaMemcpyAsync(d_q2, q2[0].data(), n_words * 8, cudaMemcpyHostToDevice, st)) != cudaSuccess ||
        (e = cudaMemcpyAsync(d_q2 + n_words, q2[1].data(), n_words * 8, cudaMemcpyHostToDevice, st)) != cudaSuccess ||
        (e = cudaMemsetAsync(d_n, 0, 8, st)) != cudaSuccess) {
        free_all();
        return qm_fail(ctx, QM_ECUDA, "qm_genome_diff_host: %s", cudaGetErrorString(e));
    }
    Q.q2p[0] = d_q2; Q.q2p[1] = d_q2 + n_words;
    gdiff_anchor_kernel<<<(unsigned)((2 * lq + 255) / 256), 256, 0, st>>>(V, Q, d_anc, cap, d_n);
    unsigned long long h_n = 0;
    if ((e = cudaGetLastError()) != cudaSuccess || (e = cudaMemcpyAsync(&h_n, d_n, 8, cudaMemcpyDeviceToHost, st)) != cudaSuccess ||
        (e = cudaStreamSynchronize(st)) != cudaSuccess) {
        free_all();
        return qm_fail(ctx, QM_ECUDA, "gdiff_anchor_kernel: %s", cudaGetErrorString(e));
    }
    std::vector<GdAnchor> anc((size_t)h_n);
    if ((int64_t)h_n > cap) { free_all(); return qm_fail(ctx, QM_ECUDA, "gdiff_anchor_kernel: %llu anchors, room for %lld", h_n, (long long)cap); }
    if ((h_n && (e = cudaMemcpyAsync(anc.data(), d_anc, h_n * sizeof(GdAnchor), cudaMemcpyDeviceToHost, st)) != cudaSuccess) ||
        (e = cudaMemcpyAsync(refb.data(), V.refb, (size_t)V.l_pac, cudaMemcpyDeviceToHost, st)) != cudaSuccess ||
        (e = cudaStreamSynchronize(st)) != cudaSuccess) {
        free_all();
        return qm_fail(ctx, QM_ECUDA, "qm_genome_diff_host: %s", cudaGetErrorString(e));
    }
    cudaFree(d_anc); d_anc = nullptr;
    lap(0);

    // ---- clusters and alignments (host) ----
    std::sort(anc.begin(), anc.end(), [](const GdAnchor &a, const GdAnchor &b) {
        if (a.qc != b.qc) return a.qc < b.qc;
        if (a.s != b.s) return a.s < b.s;
        if (a.rc != b.rc) return a.rc < b.rc;
        if (a.rs != b.rs) return a.rs < b.rs;
        return a.qs < b.qs;
    });
    std::vector<GdAln> al;
    for (size_t g0 = 0; g0 < anc.size();) {
        size_t g1 = g0;
        while (g1 < anc.size() && anc[g1].qc == anc[g0].qc && anc[g1].s == anc[g0].s && anc[g1].rc == anc[g0].rc) ++g1;
        std::vector<GdAnchor> grp(anc.begin() + g0, anc.begin() + g1);
        auto cl = cluster_group(grp, o);
        std::sort(cl.begin(), cl.end(), [](const std::vector<GdAnchor> &a, const std::vector<GdAnchor> &b) {
            return a[0].rs != b[0].rs ? a[0].rs < b[0].rs : a[0].qs < b[0].qs;
        });
        // neighbouring clusters within break_len on both sequences (after the later one's front is trimmed past the earlier one's
        // end) become one alignment
        std::vector<int> next(cl.size(), -1);
        std::vector<char> has_prev(cl.size(), 0);
        for (size_t i = 0; i < cl.size(); ++i) {
            const GdAnchor &t = cl[i].back();
            for (size_t j = i + 1; j < cl.size(); ++j) {
                if (has_prev[j]) continue;
                GdAnchor h = cl[j][0];
                if (!trim_after(t, h)) continue;
                const int64_t gr = (int64_t)h.rs - (t.rs + t.len), gq = (int64_t)h.qs - (t.qs + t.len);
                if (gr <= o.break_len && gq <= o.break_len) { next[i] = (int)j; has_prev[j] = 1; cl[j][0] = h; break; }
            }
        }
        for (size_t i = 0; i < cl.size(); ++i) {
            if (has_prev[i]) continue;
            GdAln A;
            A.s = grp[0].s; A.qc = grp[0].qc; A.rc = grp[0].rc;
            for (int c = (int)i; c >= 0; c = next[c]) A.anc.insert(A.anc.end(), cl[c].begin(), cl[c].end());
            al.push_back(std::move(A));
        }
        g0 = g1;
    }
    lap(1);

    // ---- gap alignment (device): one task per (ref [r0, r0 + n), query strand s [q0, q0 + m)) rectangle; ops first column first ----
    auto run_gaps = [&](const std::vector<GdTask> &in, std::vector<std::vector<uint8_t>> &out) -> int {
        out.assign(in.size(), {});
        std::vector<GdTask> tasks;
        std::vector<int> src;
        int64_t tb_bytes = 0, buf_ints = 0, op_bytes = 0;
        for (size_t i = 0; i < in.size(); ++i) {
            if (in[i].n == 0 && in[i].m == 0) continue;
            GdTask T = in[i];
            T.tb_off = tb_bytes; T.buf_off = buf_ints; T.op_off = op_bytes;
            tb_bytes += (int64_t)(T.n + 1) * (T.m + 1); buf_ints += 7 * (int64_t)(T.n + 1); op_bytes += T.n + T.m;
            tasks.push_back(T);
            src.push_back((int)i);
        }
        if (tasks.empty()) return QM_OK;
        std::stable_sort(tasks.begin(), tasks.end(), [](const GdTask &x, const GdTask &y) {      // longest first
            return (int64_t)(x.n + 1) * (x.m + 1) > (int64_t)(y.n + 1) * (y.m + 1);
        });
        std::vector<uint8_t> ops((size_t)op_bytes);
        const int64_t nt = (int64_t)tasks.size();
        std::vector<int32_t> nops((size_t)nt);
        GdTask *d_t = nullptr;
        uint8_t *d_tb = nullptr, *d_ops = nullptr;
        int32_t *d_buf = nullptr, *d_nops = nullptr;
        auto free_gap = [&]() { cudaFree(d_t); cudaFree(d_tb); cudaFree(d_ops); cudaFree(d_buf); cudaFree(d_nops); };
        if ((e = cudaMalloc(&d_t, nt * sizeof(GdTask))) != cudaSuccess || (e = cudaMalloc(&d_tb, (size_t)tb_bytes)) != cudaSuccess ||
            (e = cudaMalloc(&d_ops, (size_t)op_bytes)) != cudaSuccess ||
            (e = cudaMalloc(&d_buf, (size_t)buf_ints * 4)) != cudaSuccess || (e = cudaMalloc(&d_nops, nt * 4)) != cudaSuccess ||
            (e = cudaMemcpyAsync(d_t, tasks.data(), nt * sizeof(GdTask), cudaMemcpyHostToDevice, st)) != cudaSuccess) {
            free_gap();
            return qm_fail(ctx, QM_ECUDA, "qm_genome_diff_host: %s", cudaGetErrorString(e));
        }
        gdiff_gap_kernel<<<(unsigned)((nt + 3) / 4), 128, 0, st>>>(V.refb, d_qb, d_qb + lq, d_t, nt, o.match, o.mismatch, o.gap_open, o.gap_extend,
                                                                   d_tb, d_buf, d_ops, d_nops);
        if ((e = cudaGetLastError()) != cudaSuccess ||
            (e = cudaMemcpyAsync(ops.data(), d_ops, (size_t)op_bytes, cudaMemcpyDeviceToHost, st)) != cudaSuccess ||
            (e = cudaMemcpyAsync(nops.data(), d_nops, nt * 4, cudaMemcpyDeviceToHost, st)) != cudaSuccess ||
            (e = cudaStreamSynchronize(st)) != cudaSuccess) {
            free_gap();
            return qm_fail(ctx, QM_ECUDA, "gdiff_gap_kernel: %s", cudaGetErrorString(e));
        }
        free_gap();
        // the sort moved the tasks, not their offsets: task k's ops sit at its own op_off, last column first
        std::vector<int> by_off((size_t)nt);
        std::iota(by_off.begin(), by_off.end(), 0);
        std::sort(by_off.begin(), by_off.end(), [&](int x, int y) { return tasks[x].op_off < tasks[y].op_off; });
        for (int64_t k = 0; k < nt; ++k) {
            const GdTask &T = tasks[by_off[k]];
            std::vector<uint8_t> &d = out[src[k]];
            d.assign(ops.begin() + T.op_off, ops.begin() + T.op_off + nops[by_off[k]]);
            std::reverse(d.begin(), d.end());
        }
        return QM_OK;
    };
    auto gap_task = [&](const GdAln &A, int64_t r0, int64_t r1, int64_t q0, int64_t q1) {
        GdTask T = {};
        T.n = (int32_t)(r1 - r0); T.m = (int32_t)(q1 - q0); T.s = A.s;
        T.r0 = V.off[A.rc] + r0; T.q0 = Q.start[A.s][A.qc] + q0;
        return T;
    };
    std::vector<GdTask> gtasks;
    for (const GdAln &A : al)
        for (size_t g = 0; g + 1 < A.anc.size(); ++g) {
            const GdAnchor &x = A.anc[g], &y = A.anc[g + 1];
            gtasks.push_back(gap_task(A, x.rs + x.len, y.rs, x.qs + x.len, y.qs));
        }
    std::vector<std::vector<uint8_t>> gops;
    if (int rc = run_gaps(gtasks, gops)) { free_all(); return rc; }
    lap(2);

    // ---- a gap too divergent to bridge ends the alignment.  Its poor-scoring stretch runs from the column where the score along the
    // gap was best to the gap's end, and then over the bases that matching columns need to win the loss back; longer than break_len
    // columns (nucmer -b: how far an alignment extends through a poor-scoring region) ends the alignment at the gap ----
    {
        std::vector<GdAln> pieces;
        size_t t = 0;
        for (GdAln &A : al) {
            const uint8_t *R = refb.data() + V.off[A.rc];
            const uint8_t *Qy = qs[A.s].data() + Q.start[A.s][A.qc];
            GdAln P;
            P.s = A.s; P.qc = A.qc; P.rc = A.rc;
            for (size_t g = 0; g < A.anc.size(); ++g) {
                P.anc.push_back(A.anc[g]);
                if (g + 1 == A.anc.size()) break;
                std::vector<uint8_t> &go = gops[t++];
                int64_t sc = 0, best = 0, at = 0, ri = A.anc[g].rs + A.anc[g].len, qj = A.anc[g].qs + A.anc[g].len;
                for (size_t c = 0; c < go.size(); ++c) {
                    const uint8_t op = go[c];
                    if (op == OP_M) { sc += R[ri] == Qy[qj] ? o.match : -o.mismatch; ++ri; ++qj; }
                    else {
                        sc -= (c == 0 || go[c - 1] != op ? o.gap_open : 0) + o.gap_extend;
                        if (op == OP_D) ++ri; else ++qj;
                    }
                    if (sc > best) { best = sc; at = (int64_t)c + 1; }
                }
                const bool broken = (int64_t)go.size() - at + (best - sc + o.match - 1) / o.match > o.break_len;
                if (broken) { pieces.push_back(std::move(P)); P = GdAln(); P.s = A.s; P.qc = A.qc; P.rc = A.rc; }
                else P.gap_ops.push_back(std::move(go));
            }
            pieces.push_back(std::move(P));
        }
        al.swap(pieces);
        // an end is extended no further than the nearest alignment of its (query contig, strand, reference contig) ahead of it on
        // both sequences, so that two alignments never extend into each other's anchors
        for (GdAln &A : al)
            for (const GdAln &B : al) {
                if (&A == &B || A.qc != B.qc || A.s != B.s || A.rc != B.rc) continue;
                const GdAnchor &af = A.anc.front(), &al_ = A.anc.back(), &bf = B.anc.front(), &bl = B.anc.back();
                if (bf.rs >= al_.rs + al_.len && bf.qs >= al_.qs + al_.len && (A.lim_r1 < 0 || bf.rs < A.lim_r1 || (bf.rs == A.lim_r1 && bf.qs < A.lim_q1))) {
                    A.lim_r1 = bf.rs; A.lim_q1 = bf.qs;
                }
                const int64_t br = (int64_t)bl.rs + bl.len, bq = (int64_t)bl.qs + bl.len;
                if (br <= af.rs && bq <= af.qs && (br > A.lim_r0 || (br == A.lim_r0 && bq > A.lim_q0))) { A.lim_r0 = br; A.lim_q0 = bq; }
            }
    }

    // ---- alignment ends extended past the outermost anchors: ksw_extend2 (qm_extend_batch), zdrop = break_len, band break_len, in
    // windows of at most QM_EXT_MAX_QLEN query bases, again while an extension reaches the end of its window with sequence left, and no
    // further than the nearest alignment ahead ----
    {
        qm_opt eo;
        qm_opt_default(&eo);
        eo.a = o.match; eo.b = o.mismatch; eo.o_del = eo.o_ins = o.gap_open; eo.e_del = eo.e_ins = o.gap_extend; eo.zdrop = o.break_len;
        struct End { int a, side; int64_t r, q; int h0; bool on; std::vector<std::pair<int64_t, int64_t>> pts; };   // pts: (r, q) after each window
        std::vector<End> ends;
        for (size_t a = 0; a < al.size(); ++a) {
            const GdAnchor &f = al[a].anc.front(), &l = al[a].anc.back();
            ends.push_back({(int)a, 0, f.rs, f.qs, std::max(1, f.len * o.match), true, {{f.rs, f.qs}}});
            ends.push_back({(int)a, 1, (int64_t)l.rs + l.len, (int64_t)l.qs + l.len, std::max(1, l.len * o.match), true,
                            {{(int64_t)l.rs + l.len, (int64_t)l.qs + l.len}}});
        }
        for (;;) {
            std::vector<uint8_t> seq;
            std::vector<qm_ext_task> et;
            std::vector<int> who;
            std::vector<std::pair<int64_t, int64_t>> win;
            for (size_t k = 0; k < ends.size(); ++k) {
                End &E = ends[k];
                if (!E.on) continue;
                const GdAln &A = al[E.a];
                const uint8_t *R = refb.data() + V.off[A.rc];
                const uint8_t *Qy = qs[A.s].data() + Q.start[A.s][A.qc];
                const int64_t lq_ = E.side ? (A.lim_q1 >= 0 ? A.lim_q1 : Q.len[A.qc]) : std::max<int64_t>(A.lim_q0, 0);
                const int64_t lr_ = E.side ? (A.lim_r1 >= 0 ? A.lim_r1 : V.len[A.rc]) : std::max<int64_t>(A.lim_r0, 0);
                const int64_t rem_q = E.side ? lq_ - E.q : E.q - lq_, rem_r = E.side ? lr_ - E.r : E.r - lr_;
                const int64_t qw = std::min<int64_t>(QM_EXT_MAX_QLEN, rem_q), tw = std::min<int64_t>(rem_r, qw + o.break_len);
                if (qw == 0 || tw == 0) { E.on = false; continue; }
                qm_ext_task T = {};
                T.q_off = (uint32_t)seq.size();
                for (int64_t i = 0; i < qw; ++i) seq.push_back(E.side ? Qy[E.q + i] : Qy[E.q - 1 - i]);
                T.t_off = (uint32_t)seq.size();
                for (int64_t i = 0; i < tw; ++i) seq.push_back(E.side ? R[E.r + i] : R[E.r - 1 - i]);
                T.qlen = (int32_t)qw; T.tlen = (int32_t)tw; T.h0 = E.h0; T.w = o.break_len; T.end_bonus = 0; T.flags = 0;
                et.push_back(T);
                who.push_back((int)k);
                win.emplace_back(qw < rem_q ? qw : -1, tw < rem_r ? tw : -1);   // window ends that leave sequence behind them
            }
            if (et.empty()) break;
            std::vector<qm_ext_result> res(et.size());
            if (int rc = qm_extend_batch_host(ctx, &eo, seq.data(), seq.size(), et.data(), (int64_t)et.size(), res.data())) { free_all(); return rc; }
            for (size_t i = 0; i < et.size(); ++i) {
                End &E = ends[who[i]];
                const qm_ext_result &x = res[i];
                if (x.qle == 0 && x.tle == 0) { E.on = false; continue; }
                E.q += E.side ? x.qle : -x.qle;
                E.r += E.side ? x.tle : -x.tle;
                E.h0 = x.score;
                E.pts.emplace_back(E.r, E.q);
                E.on = x.qle == win[i].first || x.tle == win[i].second;
            }
        }
        // each window's stretch gets the gap kernel's global alignment, the stretches in sequence order; indel columns at the outer
        // end are dropped
        std::vector<GdTask> etasks;
        for (const End &E : ends)
            for (size_t w = 0; w + 1 < E.pts.size(); ++w) {
                const auto &a = E.pts[w], &b = E.pts[w + 1];
                etasks.push_back(E.side ? gap_task(al[E.a], a.first, b.first, a.second, b.second) : gap_task(al[E.a], b.first, a.first, b.second, a.second));
            }
        std::vector<std::vector<uint8_t>> eops;
        if (int rc = run_gaps(etasks, eops)) { free_all(); return rc; }
        size_t t0_ = 0;
        for (size_t k = 0; k < ends.size(); ++k) {
            GdAln &A = al[ends[k].a];
            const size_t nw = ends[k].pts.size() - 1;
            std::vector<uint8_t> x;
            for (size_t w = 0; w < nw; ++w) {
                const std::vector<uint8_t> &y = eops[t0_ + (ends[k].side ? w : nw - 1 - w)];
                x.insert(x.end(), y.begin(), y.end());
            }
            t0_ += nw;
            if (ends[k].side == 0) {
                size_t c = 0;
                int64_t r = ends[k].r, q = ends[k].q;
                while (c < x.size() && x[c] != OP_M) { if (x[c] == OP_D) ++r; else ++q; ++c; }
                A.rs = r; A.qs = q;
                A.ops.assign(x.begin() + c, x.end());
            } else {
                while (!x.empty() && x.back() != OP_M) x.pop_back();
                A.tail = std::move(x);
            }
        }
    }
    free_all();
    lap(3);

    // ---- columns, left-aligned indels, filter, rows (host) ----
    for (GdAln &A : al) {
        for (size_t g = 0; g < A.anc.size(); ++g) {
            A.ops.insert(A.ops.end(), (size_t)A.anc[g].len, (uint8_t)OP_M);
            if (g + 1 < A.anc.size()) A.ops.insert(A.ops.end(), A.gap_ops[g].begin(), A.gap_ops[g].end());
        }
        A.ops.insert(A.ops.end(), A.tail.begin(), A.tail.end());
        const uint8_t *R = refb.data() + V.off[A.rc];
        const uint8_t *Qy = qs[A.s].data() + Q.start[A.s][A.qc];
        // left-align every indel run through the matching columns in front of it; the first column stays a match
        int64_t ri = A.rs, qj = A.qs;
        for (size_t c = 0; c < A.ops.size();) {
            const uint8_t op = A.ops[c];
            if (op == OP_M) { ++ri; ++qj; ++c; continue; }
            size_t e2 = c;
            while (e2 < A.ops.size() && A.ops[e2] == op) ++e2;
            const int64_t len = (int64_t)(e2 - c);
            while (c > 1 && A.ops[c - 1] == OP_M && R[ri - 1] == Qy[qj - 1] &&
                   (op == OP_D ? R[ri - 1] == R[ri + len - 1] : Qy[qj - 1] == Qy[qj + len - 1])) {
                A.ops[e2 - 1] = OP_M; A.ops[c - 1] = op; --c; --e2; --ri; --qj;
            }
            if (op == OP_D) ri += len; else qj += len;
            c = e2;
        }
        A.re = ri; A.qe = qj;
        ri = A.rs; qj = A.qs;
        for (uint8_t op : A.ops) {
            if (op == OP_M) { if (R[ri] == Qy[qj]) ++A.matches; else ++A.edits; ++ri; ++qj; }
            else { ++A.edits; if (op == OP_D) ++ri; else ++qj; }
        }
        const int64_t ql = Q.len[A.qc];
        A.fqs = A.s ? ql - A.qe : A.qs;
        A.fqe = A.s ? ql - A.qs : A.qe;
    }
    filter_chain(al, 0);
    filter_chain(al, 1);
    std::stable_sort(al.begin(), al.end(), [](const GdAln &a, const GdAln &b) {
        if (a.rc != b.rc) return a.rc < b.rc;
        if (a.rs != b.rs) return a.rs < b.rs;
        if (a.re != b.re) return a.re < b.re;
        if (a.qc != b.qc) return a.qc < b.qc;
        if (a.s != b.s) return a.s < b.s;
        return a.qs < b.qs;
    });
    std::vector<qm_gdiff_row> rows;
    for (const GdAln &A : al) {
        const uint8_t *R = refb.data() + V.off[A.rc];
        const uint8_t *Qy = qs[A.s].data() + Q.start[A.s][A.qc];
        const int64_t ql = Q.len[A.qc], rl = V.len[A.rc];
        const size_t r0 = rows.size();
        int64_t ri = A.rs, qj = A.qs;
        auto fwd = [&](int64_t y1) { return A.s ? ql - y1 + 1 : y1; };     // 1-based strand position -> forward
        for (uint8_t op : A.ops) {
            qm_gdiff_row w = {};
            w.rid = A.rc; w.qid = A.qc; w.frm_r = 1; w.frm_q = A.s ? -1 : 1;
            if (op == OP_M) {
                if (R[ri] != Qy[qj]) { w.p1 = (int32_t)(ri + 1); w.sub_r = "ACGT"[R[ri]]; w.sub_q = "ACGT"[Qy[qj]]; w.p2 = (int32_t)fwd(qj + 1); rows.push_back(w); }
                ++ri; ++qj;
            } else if (op == OP_D) {
                w.p1 = (int32_t)(ri + 1); w.sub_r = "ACGT"[R[ri]]; w.sub_q = '.'; w.p2 = (int32_t)fwd(qj); rows.push_back(w);
                ++ri;
            } else {
                w.p1 = (int32_t)ri; w.sub_r = '.'; w.sub_q = "ACGT"[Qy[qj]]; w.p2 = (int32_t)fwd(qj + 1); rows.push_back(w);
                ++qj;
            }
        }
        for (size_t i = r0; i < rows.size(); ++i) {
            qm_gdiff_row &w = rows[i];
            int64_t b = std::min<int64_t>(w.p1 - (A.rs + 1), A.re - w.p1);
            if (i > r0) b = std::min<int64_t>(b, (int64_t)w.p1 - rows[i - 1].p1);
            if (i + 1 < rows.size()) b = std::min<int64_t>(b, (int64_t)rows[i + 1].p1 - w.p1);
            w.buff = (int32_t)b;
            w.dist = (int32_t)std::min<int64_t>({(int64_t)w.p1 - 1, rl - w.p1, (int64_t)w.p2 - 1, ql - w.p2});
        }
    }
    std::vector<qm_gdiff_row> kept;
    for (const qm_gdiff_row &w : rows) {
        if ((o.flags & QM_GDIFF_NO_INDELS) && (w.sub_r == '.' || w.sub_q == '.')) continue;
        if (!(o.flags & QM_GDIFF_KEEP_AMBIGUOUS)) {
            int cr = 0, cq = 0;
            for (const GdAln &A : al) {
                cr += A.rc == w.rid && w.p1 > A.rs && w.p1 <= A.re;
                cq += A.qc == w.qid && w.p2 > A.fqs && w.p2 <= A.fqe;
            }
            if (cr > 1 || cq > 1) continue;
        }
        kept.push_back(w);
    }
    std::stable_sort(kept.begin(), kept.end(), [](const qm_gdiff_row &a, const qm_gdiff_row &b) {
        return a.rid != b.rid ? a.rid < b.rid : a.p1 < b.p1;
    });
    lap(4);
    if (h_phase_ms) for (int i = 0; i < 5; ++i) h_phase_ms[i] = ms[i];
    *n_rows = (int64_t)kept.size();
    *n_alns = (int64_t)al.size();
    if (*n_rows > max_rows || *n_alns > max_alns)
        return qm_fail(ctx, QM_ELIMIT, "qm_genome_diff_host: %lld rows and %lld alignments, room for %lld and %lld", (long long)*n_rows,
                       (long long)*n_alns, (long long)max_rows, (long long)max_alns);
    if (!kept.empty()) memcpy(h_rows, kept.data(), kept.size() * sizeof(qm_gdiff_row));
    for (size_t i = 0; i < al.size(); ++i) {
        const GdAln &A = al[i];
        qm_gdiff_aln &x = h_alns[i];
        x.rid = A.rc; x.qid = A.qc;
        x.rs = (int32_t)(A.rs + 1); x.re = (int32_t)A.re;
        x.qs = (int32_t)(A.s ? A.fqe : A.fqs + 1); x.qe = (int32_t)(A.s ? A.fqs + 1 : A.fqe);
        x.strand = A.s ? -1 : 1;
        x.edits = (int32_t)A.edits; x.matches = (int32_t)A.matches; x.pad = 0;
    }
    return QM_OK;
}

}  // extern "C"
