// mplp.cu -- the text pileup of `samtools mpileup -f ref bam` (reference call site rules/vcfcall.smk:39, the
// input of the VarScan rule rules/vcfcall.smk:60-61; upstream samtools bam_plcmd.c mpileup / pileup_seq and htslib
// sam.c resolve_cigar2; format SURVEY.md A.10; restatement oracle/qmo_pileup.c qmo_mpileup_text).  SURVEY 8f-3.
// Same read admission and mate-overlap quality rewrite as pileup.cu (BAQ off, no depth cap).
//
// A column's line lists the reads covering it in coordinate-sorted order, so the text is a function of (column,
// rank of the read in the sorted order).  On the device:
//   1. one warp per pair rewrites the overlapping mates' qualities into a scratch copy (BAM orientation) and notes
//      which records are admitted and how much reference they span;
//   2. the records are sorted by samtools' key (sort.cu);
//   3. one warp per COLUMN looks up the window of sorted records that can reach it (binary search on the sorted start
//      positions, the longest span bounds the window), the lanes take 32 records at a time, find the record's state at
//      the column from its CIGAR and add up the bytes it contributes: line lengths;
//   4. an exclusive scan of the line lengths gives every line its place;
//   5. the same walk again, now writing: a warp scan over the lanes' byte counts places every record's characters.
#include <cub/device/device_scan.cuh>
#include "pipeline.cuh"

namespace {

constexpr int kMaxLen = 512;
constexpr int kWarps = 4;

struct RecInfo { int32_t gstart; int32_t span; };      // forward-strand start (contigs concatenated), reference span; span 0 = not admitted

__device__ __forceinline__ int rpos_walk(const uint32_t *cigar, int nc, int pos, int i)
{   // contig position of query base i (BAM orientation) if it is an M base, else -1
    int x = 0, p = pos;
    for (int k = 0; k < nc; ++k) {
        const int op = cigar[k] & 0xf, len = (int)(cigar[k] >> 4);
        if (op == 0) { if (i < x + len) return p + (i - x); x += len; p += len; }
        else if (op == 1 || op == 4) { if (i < x + len) return -1; x += len; }
        else if (op == 2) p += len;
    }
    return -1;
}
__device__ __forceinline__ int qidx_walk(const uint32_t *cigar, int nc, int pos, int p)
{   // query index of the M base at contig position p, else -1
    int x = 0, pp = pos;
    for (int k = 0; k < nc; ++k) {
        const int op = cigar[k] & 0xf, len = (int)(cigar[k] >> 4);
        if (op == 0) { if (p >= pp && p < pp + len) return x + (p - pp); x += len; pp += len; }
        else if (op == 1 || op == 4) x += len;
        else if (op == 2) { if (p < pp + len) return -1; pp += len; }
    }
    return -1;
}

// step 1: warp per pair (the structure of pileup_kernel: admission, qualities to BAM orientation, overlap rewrite)
__global__ void __launch_bounds__(kWarps * 32)
mplp_prepare_kernel(IndexView V, qm_pileup_opt po, const qm_aln *__restrict__ alns, const uint8_t *__restrict__ codes,
                    const uint8_t *__restrict__ quals, int stride, const int32_t *__restrict__ lens, int64_t n_pairs,
                    uint8_t *__restrict__ tq, RecInfo *__restrict__ info, int *__restrict__ max_span)
{
    __shared__ uint8_t s_q[kWarps][2][kMaxLen];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    int my_max = 0;
    for (int64_t pi = blockIdx.x * (int64_t)kWarps + wib; pi < n_pairs; pi += (int64_t)gridDim.x * kWarps) {
        const qm_aln *g[2] = { alns + 2 * pi, alns + 2 * pi + 1 };
        int flag[2], L[2], nc[2];
        bool ok[2], rev[2];
        __syncwarp();
        for (int e = 0; e < 2; ++e) {
            flag[e] = g[e]->flag; nc[e] = g[e]->n_cigar; L[e] = lens[2 * pi + e];
            rev[e] = (flag[e] & 0x10) != 0;
            ok[e] = !(flag[e] & (0x4 | 0x100 | 0x200 | 0x400)) && nc[e] != 0 && nc[e] != 255 && g[e]->mapq >= po.min_mapq &&
                    !((flag[e] & 0x1) && !(flag[e] & 0x2) && !po.count_orphans) && L[e] <= kMaxLen;
            const uint8_t *qv = quals + (2 * pi + e) * stride;
            if (ok[e]) for (int i = lane; i < L[e]; i += 32) s_q[wib][e][i] = rev[e] ? qv[L[e] - 1 - i] : qv[i];
        }
        __syncwarp();
        const uint8_t *rd[2] = { codes + (2 * pi) * stride, codes + (2 * pi + 1) * stride };
        auto seq_base = [&](int e, int i) {
            const int c = rev[e] ? rd[e][L[e] - 1 - i] : rd[e][i];
            return rev[e] ? (c > 3 ? 4 : 3 - c) : c;
        };
        if (!po.ignore_overlaps && ok[0] && ok[1] && g[0]->rid == g[1]->rid && (flag[0] & 0x2) && !(flag[0] & 0x8) &&
            abs(g[0]->tlen) < 2 * L[0] && abs(g[1]->tlen) < 2 * L[1]) {
            const int p0 = g[0]->pos, p1 = g[1]->pos;
            const int A = (p1 < p0 || (p1 == p0 && (int)rev[1] < (int)rev[0])) ? 1 : 0, B = A ^ 1;
            for (int ia = lane; ia < L[A]; ia += 32) {
                const int p = rpos_walk(g[A]->cigar, nc[A], g[A]->pos, ia);
                if (p < 0) continue;
                const int ib = qidx_walk(g[B]->cigar, nc[B], g[B]->pos, p);
                if (ib < 0) continue;
                const int qa = s_q[wib][A][ia], qb = s_q[wib][B][ib];
                if (seq_base(A, ia) == seq_base(B, ib)) {
                    const int q = qa + qb;
                    s_q[wib][A][ia] = (uint8_t)(q > 200 ? 200 : q); s_q[wib][B][ib] = 0;
                } else if (qa >= qb) { s_q[wib][A][ia] = (uint8_t)(0.8 * qa); s_q[wib][B][ib] = 0; }
                else { s_q[wib][B][ib] = (uint8_t)(0.8 * qb); s_q[wib][A][ia] = 0; }
            }
        }
        __syncwarp();
        for (int e = 0; e < 2; ++e) {
            RecInfo ri; ri.gstart = 0; ri.span = 0;
            if (ok[e]) {
                for (int i = lane; i < L[e]; i += 32) tq[(2 * pi + e) * (int64_t)stride + i] = s_q[wib][e][i];
                int span = 0;
                for (int k = 0; k < nc[e]; ++k) { const int op = g[e]->cigar[k] & 0xf; if (op == 0 || op == 2) span += (int)(g[e]->cigar[k] >> 4); }
                ri.gstart = (int32_t)(V.off[g[e]->rid] + g[e]->pos); ri.span = span;
                my_max = span > my_max ? span : my_max;
            }
            if (lane == 0) info[2 * pi + e] = ri;
        }
    }
    if (lane == 0 && my_max) atomicMax(max_span, my_max);
}

// what the column walk needs of a record, in SORTED order (16 B, read coalesced by the lanes of a column's warp); the
// alignment record itself is only touched for reads with an indel
struct SInfo {
    int32_t gstart;            // forward-strand start, contigs concatenated
    uint16_t span;             // reference span; 0 = not admitted
    uint16_t m0;               // gap-free alignments: query index of the first aligned base (the leading soft clip)
    uint32_t rec;              // index of the record
    uint16_t len;              // read length
    uint8_t mapq, flags;       // flags: 1 = reverse strand, 2 = gap-free ([clip] M [clip])
};

// sorted start positions (records that are not admitted keep their place in the order but never cover a column)
__global__ void mplp_starts_kernel(const uint32_t *__restrict__ perm, const qm_aln *__restrict__ alns, const RecInfo *__restrict__ info,
                                   const int32_t *__restrict__ lens, IndexView V, int64_t n, int32_t *__restrict__ starts, SInfo *__restrict__ sinfo)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= n) return;
    const uint32_t rec = perm[k];
    const qm_aln &a = alns[rec];
    starts[k] = a.rid < 0 ? 0x7fffffff : (int32_t)(V.off[a.rid] + a.pos);      // an unplaced read sits at its mate's position
    const RecInfo ri = info[rec];
    SInfo s;
    s.gstart = ri.gstart; s.span = (uint16_t)ri.span; s.m0 = 0; s.rec = rec; s.len = (uint16_t)lens[rec]; s.mapq = a.mapq;
    s.flags = (a.flag & 0x10) ? 1 : 0;
    if (ri.span > 0) {
        int kk = 0, x = 0;
        const int nc = a.n_cigar;
        if (kk < nc && (a.cigar[kk] & 0xf) == 4) { x = (int)(a.cigar[kk] >> 4); ++kk; }
        if (kk < nc && (a.cigar[kk] & 0xf) == 0) {
            ++kk;
            if (kk < nc && (a.cigar[kk] & 0xf) == 4) ++kk;
            if (kk == nc) { s.flags |= 2; s.m0 = (uint16_t)x; }
        }
    }
    sinfo[k] = s;
}

// sort keys from a caller-given order: rank[r] >= 0 is record r's place, a negative rank puts the record after every ranked one
__global__ void mplp_rank_keys_kernel(const int64_t *__restrict__ rank, int64_t n, uint64_t *__restrict__ keys)
{
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r < n) keys[r] = rank[r] >= 0 ? (uint64_t)rank[r] : (uint64_t)(n + r);
}

__device__ __forceinline__ int n_digits(int v) { int d = 1; while (v >= 10) { v /= 10; ++d; } return d; }

// what a record contributes to the column at contig position p (htslib resolve_cigar2)
struct Entry { bool covers, is_del, head, tail; int qpos, indel; };
__device__ __forceinline__ Entry entry_at(const qm_aln &a, int span, int p)
{
    Entry e; e.covers = false; e.is_del = false; e.head = false; e.tail = false; e.qpos = 0; e.indel = 0;
    if (p < a.pos || p >= a.pos + span) return e;
    int x = a.pos, y = 0;
    const int nc = a.n_cigar;
    for (int k = 0; k < nc; ++k) {
        const int op = a.cigar[k] & 0xf, len = (int)(a.cigar[k] >> 4);
        if (op == 1 || op == 4) { y += len; continue; }
        if (op != 0 && op != 2) continue;
        if (p < x + len) {
            e.covers = true; e.is_del = op == 2; e.qpos = op == 2 ? y : y + (p - x);
            if (p == x + len - 1 && k + 1 < nc) {
                const int op2 = a.cigar[k + 1] & 0xf, l2 = (int)(a.cigar[k + 1] >> 4);
                if (op2 == 2) e.indel = -l2; else if (op2 == 1) e.indel = l2;
            }
            break;
        }
        x += len; if (op == 0) y += len;
    }
    e.head = p == a.pos; e.tail = p == a.pos + span - 1;
    return e;
}

struct NameTab { int32_t off[QM_MAX_CONTIGS + 1]; };

// steps 3 and 5: warp per column.  WRITE = false: line_len[g] (0 = no line);  WRITE = true: the characters.
template <bool WRITE>
__global__ void __launch_bounds__(kWarps * 32)
mplp_column_kernel(IndexView V, qm_pileup_opt po, const qm_aln *__restrict__ alns, const uint8_t *__restrict__ codes,
                   const uint8_t *__restrict__ tq, int stride, const SInfo *__restrict__ sinfo,
                   const int32_t *__restrict__ starts, int64_t n_rec, const int *__restrict__ max_span,
                   const char *__restrict__ names, NameTab NT, int64_t *__restrict__ line_len, int32_t *__restrict__ n_entries,
                   const int64_t *__restrict__ line_off, char *__restrict__ out)
{
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int ms = *max_span;
    for (int64_t g = blockIdx.x * (int64_t)kWarps + wib; g < V.l_pac; g += (int64_t)gridDim.x * kWarps) {
        if (WRITE && line_len[g] == 0) continue;
        // records whose start lies in (g - ms, g]
        int64_t lo, hi;
        { int64_t a = 0, b = n_rec; const int32_t want = (int32_t)(g - ms + 1); while (a < b) { const int64_t m = (a + b) >> 1; if (starts[m] < want) a = m + 1; else b = m; } lo = a; }
        { int64_t a = lo, b = n_rec; const int32_t want = (int32_t)g; while (a < b) { const int64_t m = (a + b) >> 1; if (starts[m] <= want) a = m + 1; else b = m; } hi = a; }
        int rid = 0;
        for (int c = 0; c < V.n_contigs; ++c) if (g >= V.off[c] && g < V.off[c] + V.len[c]) rid = c;
        const int p = (int)(g - V.off[rid]);
        const int64_t clen = V.len[rid];
        const int refc = V.refb[g];
        int64_t b_off = 0, q_off = 0;          // WRITE: where the next base-string / quality byte of this line goes
        if (WRITE) {
            const int name_len = NT.off[rid + 1] - NT.off[rid];
            const int cnt = n_entries[g];
            char *o = out + line_off[g];
            const int hdr = name_len + 1 + n_digits(p + 1) + 1 + 1 + 1 + n_digits(cnt) + 1;
            if (lane == 0) {
                int w = 0;
                for (int i = 0; i < name_len; ++i) o[w++] = names[NT.off[rid] + i];
                o[w++] = '\t';
                { int v = p + 1, d = n_digits(v); for (int i = d - 1; i >= 0; --i) { o[w + i] = (char)('0' + v % 10); v /= 10; } w += d; }
                o[w++] = '\t'; o[w++] = "ACGTN"[refc]; o[w++] = '\t';
                { int v = cnt, d = n_digits(v); for (int i = d - 1; i >= 0; --i) { o[w + i] = (char)('0' + v % 10); v /= 10; } w += d; }
                o[w++] = '\t';
            }
            b_off = line_off[g] + hdr;
            q_off = line_off[g] + line_len[g] - 1 - cnt;      // the quality string ends right before the newline
            if (cnt == 0) {                                   // covered, but every base failed -Q: samtools prints "*" for both strings
                if (lane == 0) { o[hdr] = '*'; o[hdr + 1] = '\t'; o[hdr + 2] = '*'; o[hdr + 3] = '\n'; }
                continue;
            }
            if (lane == 0) { out[q_off - 1] = '\t'; out[line_off[g] + line_len[g] - 1] = '\n'; }
        }
        int tot_b = 0, tot_q = 0, any = 0;
        for (int64_t k0 = lo; k0 < hi; k0 += 32) {
            const int64_t k = k0 + lane;
            int nb = 0, nq = 0, cov = 0;
            Entry e; e.covers = false;
            SInfo si; si.rec = 0; si.span = 0; si.flags = 0; si.len = 0; si.mapq = 0;
            int qual = 0;
            if (k < hi) {
                si = sinfo[k];
                if (si.span > 0 && g < (int64_t)si.gstart + si.span) {
                    if (si.flags & 2) {
                        e.covers = true; e.is_del = false; e.indel = 0; e.qpos = si.m0 + (int)(g - si.gstart);
                        e.head = g == si.gstart; e.tail = g == (int64_t)si.gstart + si.span - 1;
                    } else e = entry_at(alns[si.rec], si.span, p);
                    if (e.covers) {
                        cov = 1;
                        qual = e.qpos < si.len ? tq[(int64_t)si.rec * stride + e.qpos] : 0;
                        if (qual >= po.min_bq) {
                            nq = 1;
                            nb = (e.head ? 2 : 0) + 1 + (e.tail ? 1 : 0);
                            if (e.indel) { const int l = e.indel > 0 ? e.indel : -e.indel; nb += 1 + n_digits(l) + l; }
                        }
                    }
                }
            }
            // inclusive scans over the lanes
            int sb = nb, sq = nq;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int ob = __shfl_up_sync(0xffffffffu, sb, d), oq = __shfl_up_sync(0xffffffffu, sq, d);
                if (lane >= d) { sb += ob; sq += oq; }
            }
            any |= __any_sync(0xffffffffu, cov);
            if (WRITE && nq) {
                const bool rev = (si.flags & 1) != 0;
                const int L = si.len;
                const uint8_t *rd = codes + (int64_t)si.rec * stride;
                auto seq_base = [&](int i) { if (i >= L) return 4; const int c = rev ? rd[L - 1 - i] : rd[i]; return rev ? (c > 3 ? 4 : 3 - c) : c; };
                const char *let = rev ? "acgtn" : "ACGTN";
                char *o = out + b_off + tot_b + (sb - nb);
                int w = 0;
                if (e.head) { o[w++] = '^'; o[w++] = (char)(si.mapq > 93 ? 126 : si.mapq + 33); }
                if (!e.is_del) { const int cc = seq_base(e.qpos); o[w++] = (cc < 4 && cc == refc) ? (rev ? ',' : '.') : let[cc]; }
                else o[w++] = '*';
                if (e.indel) {
                    const int l = e.indel > 0 ? e.indel : -e.indel, d = n_digits(l);
                    o[w++] = e.indel > 0 ? '+' : '-';
                    { int v = l; for (int i = d - 1; i >= 0; --i) { o[w + i] = (char)('0' + v % 10); v /= 10; } w += d; }
                    if (e.indel > 0) for (int j = 1; j <= l; ++j) o[w++] = let[seq_base(e.qpos + j)];
                    else for (int j = 1; j <= l; ++j) o[w++] = p + j < clen ? let[V.refb[g + j]] : let[4];
                }
                if (e.tail) o[w++] = '$';
                out[q_off + tot_q + (sq - 1)] = (char)(qual + 33 < 126 ? qual + 33 : 126);
            }
            tot_b += __shfl_sync(0xffffffffu, sb, 31);
            tot_q += __shfl_sync(0xffffffffu, sq, 31);
        }
        if (!WRITE && lane == 0) {
            int64_t len = 0;
            if (any) {
                const int name_len = NT.off[rid + 1] - NT.off[rid];
                len = name_len + 1 + n_digits(p + 1) + 1 + 1 + 1 + n_digits(tot_q) + 1 + tot_b + 1 + tot_q + 1;
                if (tot_q == 0) len += 2;                     // "*" for the empty base string and the empty quality string
            }
            line_len[g] = len;
            n_entries[g] = tot_q;
        }
    }
}

// Text pileup of the device-resident records of one sample.  *d_text points into library scratch (valid until the next
// call on this context that produces text); *h_bytes = its length.  names: contig names, '\0'-terminated, n_contigs of them.
// d_rank NULL: reads reach a column in samtools' sort order (ties in record order); else in the order of d_rank.
int mplp_text(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns, const uint8_t *d_codes,
              const uint8_t *d_quals, int32_t stride, const int32_t *d_lens, int64_t n_pairs, const char *const *names,
              const int64_t *d_rank, const char **d_text, int64_t *h_bytes, void *stream)
{
    if (!ctx || !idx || !po || !names || !d_text || !h_bytes || n_pairs < 0 || (n_pairs > 0 && (!d_alns || !d_codes || !d_quals || !d_lens)))
        return QM_EINVAL;
    *d_text = nullptr; *h_bytes = 0;
    if (n_pairs == 0) return QM_OK;
    if (stride > kMaxLen) return qm_fail(ctx, QM_ELIMIT, "qm_mpileup_text: reads longer than %d bases", kMaxLen);
    if (idx->v.l_pac >= 0x7fffffffll || 2 * n_pairs > 0xffffffffll) return qm_fail(ctx, QM_ELIMIT, "qm_mpileup_text: reference or batch too large");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const IndexView &V = idx->v;
    const int64_t n = 2 * n_pairs, l_pac = V.l_pac;
    NameTab NT;
    std::string all;
    for (int c = 0; c < V.n_contigs; ++c) { NT.off[c] = (int32_t)all.size(); all += names[c] ? names[c] : ""; }
    NT.off[V.n_contigs] = (int32_t)all.size();
    // scratch 16: tweaked qualities | record info | keys | perm | starts | line lengths | line offsets | entry counts | names | misc | cub temp
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    size_t cub_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, (int64_t *)nullptr, (int64_t *)nullptr, (int)(l_pac + 1), st);
    const size_t o_tq = 0, o_info = o_tq + al((size_t)n * stride), o_keys = o_info + al((size_t)n * sizeof(RecInfo));
    const size_t o_perm = o_keys + al((size_t)n * 8), o_starts = o_perm + al((size_t)n * 4), o_sinfo = o_starts + al((size_t)n * 4);
    const size_t o_len = o_sinfo + al((size_t)n * sizeof(SInfo));
    const size_t o_off = o_len + al((size_t)(l_pac + 1) * 8), o_cnt = o_off + al((size_t)(l_pac + 1) * 8), o_names = o_cnt + al((size_t)l_pac * 4);
    const size_t o_misc = o_names + al(all.size() + 1), o_cub = o_misc + 256;
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 16, o_cub + al(cub_bytes), &p);
    if (rc) return rc;
    char *b = (char *)p;
    uint8_t *tq = (uint8_t *)(b + o_tq);
    RecInfo *info = (RecInfo *)(b + o_info);
    uint64_t *keys = (uint64_t *)(b + o_keys);
    uint32_t *perm = (uint32_t *)(b + o_perm);
    int32_t *starts = (int32_t *)(b + o_starts), *cnt = (int32_t *)(b + o_cnt);
    int64_t *line_len = (int64_t *)(b + o_len), *line_off = (int64_t *)(b + o_off);
    char *d_names = b + o_names;
    SInfo *sinfo = (SInfo *)(b + o_sinfo);
    int *max_span = (int *)(b + o_misc);
    QM_CUDA(ctx, cudaMemsetAsync(max_span, 0, 256, st));
    QM_CUDA(ctx, cudaMemsetAsync(line_len + l_pac, 0, 8, st));
    QM_CUDA(ctx, cudaMemcpyAsync(d_names, all.data(), all.size(), cudaMemcpyHostToDevice, st));
    const int blocks = ctx->sm_count * 8;
    mplp_prepare_kernel<<<blocks, kWarps * 32, 0, st>>>(V, *po, d_alns, d_codes, d_quals, stride, d_lens, n_pairs, tq, info, max_span);
    int key_bits = 0;
    if (d_rank) {
        mplp_rank_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_rank, n, keys);
        key_bits = 1;
        while (key_bits < 63 && ((uint64_t)2 * n >> key_bits)) ++key_bits;
    } else {
        rc = qm_aln_sort_keys(ctx, idx, d_alns, n, keys, &key_bits, stream);
        if (rc) return rc;
    }
    rc = qm_sort_pairs(ctx, keys, perm, n, key_bits, stream);
    if (rc) return rc;
    mplp_starts_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(perm, d_alns, info, d_lens, V, n, starts, sinfo);
    mplp_column_kernel<false><<<blocks, kWarps * 32, 0, st>>>(V, *po, d_alns, d_codes, tq, stride, sinfo, starts, n, max_span, d_names, NT,
                                                             line_len, cnt, nullptr, nullptr);
    QM_CUDA(ctx, cub::DeviceScan::ExclusiveSum(b + o_cub, cub_bytes, line_len, line_off, (int)(l_pac + 1), st));
    int64_t total = 0;
    QM_CUDA(ctx, cudaMemcpyAsync(&total, line_off + l_pac, 8, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    void *tp = nullptr;
    rc = qm_scratch_reserve(ctx, 17, (size_t)total + 256, &tp);
    ctx->text_bytes = total;
    if (rc) return rc;
    mplp_column_kernel<true><<<blocks, kWarps * 32, 0, st>>>(V, *po, d_alns, d_codes, tq, stride, sinfo, starts, n, max_span, d_names, NT,
                                                            line_len, cnt, line_off, (char *)tp);
    QM_CUDA(ctx, cudaGetLastError());
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    *d_text = (const char *)tp; *h_bytes = total;
    return QM_OK;
}

}  // namespace

extern "C" {

int qm_mpileup_text(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns, const uint8_t *d_codes,
                    const uint8_t *d_quals, int32_t stride, const int32_t *d_lens, int64_t n_pairs, const char *const *names,
                    const char **d_text, int64_t *h_bytes, void *stream)
{
    return mplp_text(ctx, idx, po, d_alns, d_codes, d_quals, stride, d_lens, n_pairs, names, nullptr, d_text, h_bytes, stream);
}

int qm_mpileup_text_ranked(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *d_alns, const uint8_t *d_codes,
                           const uint8_t *d_quals, int32_t stride, const int32_t *d_lens, int64_t n_pairs, const char *const *names,
                           const int64_t *d_rank, const char **d_text, int64_t *h_bytes, void *stream)
{
    if (!d_rank && n_pairs > 0) return QM_EINVAL;
    return mplp_text(ctx, idx, po, d_alns, d_codes, d_quals, stride, d_lens, n_pairs, names, d_rank, d_text, h_bytes, stream);
}

// host entry for the driver: records, reads and qualities of the whole sample in host memory; the text stays on the device
// until qm_mpileup_text_fetch copies it out (h_out of at least *h_bytes bytes).  Synchronous.
int qm_mpileup_text_host(qm_ctx *ctx, const qm_index *idx, const qm_pileup_opt *po, const qm_aln *h_alns, const uint8_t *h_codes,
                         const uint8_t *h_quals, int32_t stride, const int32_t *h_lens, int64_t n_pairs, const char *const *names,
                         int64_t *h_bytes)
{
    if (!ctx || !idx || !po || !names || !h_bytes || n_pairs < 0 || (n_pairs > 0 && (!h_alns || !h_codes || !h_quals || !h_lens))) return QM_EINVAL;
    *h_bytes = 0;
    if (n_pairs == 0) { ctx->text_bytes = 0; return QM_OK; }
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t n = (size_t)2 * n_pairs;
    const size_t o_alns = 0, o_codes = al(n * sizeof(qm_aln)), o_quals = o_codes + al(n * stride), o_lens = o_quals + al(n * stride);
    void *p = nullptr;
    const int rc = qm_scratch_reserve(ctx, 18, o_lens + al(n * 4), &p);
    if (rc) return rc;
    char *b = (char *)p;
    cudaStream_t st = ctx->own_stream;
    QM_CUDA(ctx, cudaMemcpyAsync(b + o_alns, h_alns, n * sizeof(qm_aln), cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync(b + o_codes, h_codes, n * stride, cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync(b + o_quals, h_quals, n * stride, cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync(b + o_lens, h_lens, n * 4, cudaMemcpyHostToDevice, st));
    const char *d_text = nullptr;
    return qm_mpileup_text(ctx, idx, po, (const qm_aln *)(b + o_alns), (const uint8_t *)(b + o_codes), (const uint8_t *)(b + o_quals), stride,
                           (const int32_t *)(b + o_lens), n_pairs, names, &d_text, h_bytes, st);
}

int qm_mpileup_text_fetch(qm_ctx *ctx, char *h_out, int64_t bytes)
{
    if (!ctx || bytes < 0 || (bytes > 0 && !h_out)) return QM_EINVAL;
    if (bytes > ctx->text_bytes) return qm_fail(ctx, QM_EINVAL, "qm_mpileup_text_fetch: %lld bytes asked, %lld produced", (long long)bytes, (long long)ctx->text_bytes);
    if (bytes == 0) return QM_OK;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    QM_CUDA(ctx, cudaMemcpy(h_out, ctx->scratch[17].ptr, (size_t)bytes, cudaMemcpyDeviceToHost));
    return QM_OK;
}

}  // extern "C"
