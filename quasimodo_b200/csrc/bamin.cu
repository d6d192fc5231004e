// bamin.cu -- records of a coordinate-sorted BAM into the read-batch layout every record consumer takes (the way in for
// `qm_driver pileup`, the per-rule replacement of the reference's rules `mpileup` and `bcftools`, rules/vcfcall.smk:39,115).
//
// The host has inflated the BGZF blocks, validated every record and left out the ones neither mpileup admits; what comes here
// is the uncompressed record stream and the byte offset of each record kept.  On the device:
//   1. one warp per record decodes it into a FILE-ORDER row: qm_aln, base codes 0..4 and qualities in the orientation the read
//      was sequenced in (a reverse-strand record is reverse-complemented back), its length and a 64-bit hash of its name;
//   2. (hash, file index) pairs are sorted (sort.cu); within a run of equal hashes the names are compared byte for byte, and the
//      two primary records of a name (0x40 / 0x80, neither 0x100 nor 0x800) become one pair.  Every other record is a pair of
//      its own with an empty placeholder mate (flag 0x4, no CIGAR, length 0);
//   3. pair i is the i-th pair in the file order of its first record, which goes to row 2i (the mate-overlap rewrite breaks a
//      tie of position and strand in favour of row 2i, as htslib favours the read already in its overlap hash); a gather lays
//      the rows out and keeps each row's file index;
//   4. the depth cap (qm_depth_cap) runs over the file-order rows, consecutive rows standing in as pseudo-pairs: htslib's cap
//      depends on the order of the reads in the file, and the cap looks at every read alone.  Its verdict moves to the pair
//      layout through the permutation.
#include <cub/device/device_scan.cuh>
#include "pipeline.cuh"

namespace {

__device__ __forceinline__ uint32_t ld_u32(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }
__device__ __forceinline__ uint32_t ld_u16(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8; }

// SAM's 4-bit base codes -> 0..4: '=' and the IUPAC codes are N (htslib seq_nt16_int)
__constant__ uint8_t kNt16Code[16] = {4, 0, 1, 4, 2, 4, 4, 4, 3, 4, 4, 4, 4, 4, 4, 4};

__device__ __forceinline__ void placeholder(qm_aln &a)
{
    memset(&a, 0, sizeof a);
    a.rid = -1; a.pos = -1; a.flag = 0x4; a.mate_rid = -1; a.mate_pos = -1;
}

// the value of an integer tag, or 0 when the record has none (bwa's NM / AS / XS are 'c' 'C' 's' 'S' 'i' 'I')
__device__ int32_t aux_int(const uint8_t *p, const uint8_t *end, char t0, char t1)
{
    while (p + 3 <= end) {
        const char a = (char)p[0], b = (char)p[1], ty = (char)p[2];
        p += 3;
        int32_t v = 0;
        int sz = 0;
        switch (ty) {
        case 'A': case 'c': case 'C': sz = 1; v = ty == 'c' ? (int32_t)(int8_t)p[0] : (int32_t)p[0]; break;
        case 's': case 'S': sz = 2; v = ty == 's' ? (int32_t)(int16_t)ld_u16(p) : (int32_t)ld_u16(p); break;
        case 'i': case 'I': case 'f': sz = 4; v = (int32_t)ld_u32(p); break;
        case 'Z': case 'H': while (p + sz < end && p[sz]) ++sz; ++sz; break;
        case 'B': {
            const char sub = (char)p[0];
            const int es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4;
            sz = 5 + es * (int)ld_u32(p + 1);
            break;
        }
        default: return 0;                                 // malformed: no tag
        }
        if (a == t0 && b == t1) return (ty == 'A' || ty == 'f' || ty == 'Z' || ty == 'H' || ty == 'B') ? 0 : v;
        p += sz;
    }
    return 0;
}

// step 1: one warp per file-order row.  Rows [n, n_rows) are placeholders (the pad of an odd record count).
__global__ void __launch_bounds__(128)
bam_decode_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ rec_off, int64_t n, int64_t n_rows, int stride,
                  int hash_bits, qm_aln *__restrict__ alns, uint8_t *__restrict__ codes, uint8_t *__restrict__ quals,
                  int32_t *__restrict__ lens, uint64_t *__restrict__ hash)
{
    const int lane = threadIdx.x & 31;
    const int64_t f = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (f >= n_rows) return;
    uint8_t *c = codes + f * stride, *q = quals + f * stride;
    if (f >= n) {
        for (int i = lane; i < stride; i += 32) { c[i] = 4; q[i] = 0; }
        if (lane == 0) { qm_aln a; placeholder(a); alns[f] = a; lens[f] = 0; hash[f] = ~0ull; }
        return;
    }
    const uint8_t *r = bytes + rec_off[f];
    const int l_name = r[12], n_cig = (int)ld_u16(r + 16);
    const int flag = (int)ld_u16(r + 18), L = (int)ld_u32(r + 20);
    const int64_t o_seq = 36 + l_name + 4 * n_cig, o_qual = o_seq + (L + 1) / 2;
    const bool rev = (flag & 0x10) != 0;
    for (int i = lane; i < stride; i += 32) {
        if (i < L) {
            const int s = rev ? L - 1 - i : i;                 // as sequenced: a reverse-strand record read backwards, complemented
            const int code = kNt16Code[(r[o_seq + (s >> 1)] >> ((s & 1) ? 0 : 4)) & 15];
            c[i] = rev ? (code < 4 ? 3 - code : 4) : code;
            q[i] = r[o_qual + s];
        } else { c[i] = 4; q[i] = 0; }
    }
    if (lane != 0) return;
    qm_aln a;
    memset(&a, 0, sizeof a);
    a.rid = (int32_t)ld_u32(r + 4); a.pos = (int32_t)ld_u32(r + 8);
    a.mapq = r[13]; a.flag = (uint16_t)flag;
    a.mate_rid = (int32_t)ld_u32(r + 24); a.mate_pos = (int32_t)ld_u32(r + 28); a.tlen = (int32_t)ld_u32(r + 32);
    // CIGAR: '=' and 'X' are M, H is dropped, neighbours of one kind merge (the host refused N, P and more than QM_MAX_CIGAR ops)
    int nc = 0;
    for (int k = 0; k < n_cig; ++k) {
        const uint32_t w = ld_u32(r + 36 + l_name + 4 * k);
        int op = (int)(w & 0xf);
        const uint32_t len = w >> 4;
        if (op == 5 || len == 0) continue;
        if (op == 7 || op == 8) op = 0;
        if (nc > 0 && (int)(a.cigar[nc - 1] & 0xf) == op) { a.cigar[nc - 1] += len << 4; continue; }
        if (nc < QM_MAX_CIGAR) a.cigar[nc++] = len << 4 | (uint32_t)op;
    }
    a.n_cigar = (uint8_t)nc;
    a.qb = 0; a.qe = L;
    const uint8_t *aux = r + o_qual + L, *end = r + 4 + ld_u32(r);
    a.nm = aux_int(aux, end, 'N', 'M'); a.score = aux_int(aux, end, 'A', 'S'); a.sub = aux_int(aux, end, 'X', 'S');
    alns[f] = a;
    lens[f] = L;
    uint64_t h = 1469598103934665603ull;                           // FNV-1a over the name without its NUL
    for (int i = 0; i + 1 < l_name; ++i) { h ^= r[36 + i]; h *= 1099511628211ull; }
    hash[f] = hash_bits >= 64 ? h : h & ((1ull << hash_bits) - 1);
}

__device__ __forceinline__ bool pairing_primary(const qm_aln &a)
{
    const int m = a.flag & 0xc0;
    return (m == 0x40 || m == 0x80) && !(a.flag & 0x900);
}

__device__ bool same_name(const uint8_t *bytes, const int64_t *rec_off, int64_t f, int64_t g)
{
    const uint8_t *a = bytes + rec_off[f], *b = bytes + rec_off[g];
    if (a[12] != b[12]) return false;
    for (int i = 0; i + 1 < a[12]; ++i) if (a[36 + i] != b[36 + i]) return false;
    return true;
}

// step 2: sorted position k (keys[k] = hash, perm[k] = file index).  partner[f] = file index of f's mate, -1 = f stays alone:
// f and g pair iff they are the only two primary records of their name and one is the first, the other the last segment
__global__ void __launch_bounds__(256)
bam_pair_kernel(const uint8_t *__restrict__ bytes, const int64_t *__restrict__ rec_off, const qm_aln *__restrict__ alns,
                const uint64_t *__restrict__ keys, const uint32_t *__restrict__ perm, int64_t n, int32_t *__restrict__ partner)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int64_t f = perm[k];
    partner[f] = -1;
    const qm_aln &a = alns[f];
    if (!pairing_primary(a)) return;
    const uint64_t h = keys[k];
    int64_t lo = k, hi = k + 1;
    while (lo > 0 && keys[lo - 1] == h) --lo;
    while (hi < n && keys[hi] == h) ++hi;
    int64_t mate = -1;
    int found = 0;
    for (int64_t j = lo; j < hi && found < 2; ++j) {
        if (j == k) continue;
        const int64_t g = perm[j];
        if (!pairing_primary(alns[g]) || !same_name(bytes, rec_off, f, g)) continue;
        mate = g; ++found;
    }
    if (found == 1 && (alns[mate].flag & 0xc0) != (a.flag & 0xc0)) partner[f] = (int32_t)mate;
}

// a row opens a pair when it stays alone or comes before its mate in the file
__global__ void __launch_bounds__(256)
bam_leader_kernel(const int32_t *__restrict__ partner, int64_t n, int32_t *__restrict__ lead)
{
    const int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (f < n) lead[f] = partner[f] < 0 || f < partner[f];
}

// step 3: one warp per file-order row that opens a pair; slot 0 = that row, slot 1 = its mate or a placeholder
__global__ void __launch_bounds__(128)
bam_gather_kernel(const qm_aln *__restrict__ f_alns, const uint8_t *__restrict__ f_codes, const uint8_t *__restrict__ f_quals,
                  const int32_t *__restrict__ f_lens, const int32_t *__restrict__ partner, const int32_t *__restrict__ pidx, int64_t n,
                  int stride, qm_aln *__restrict__ alns, uint8_t *__restrict__ codes, uint8_t *__restrict__ quals,
                  int32_t *__restrict__ lens, int64_t *__restrict__ row_file, int64_t *__restrict__ file_row)
{
    const int lane = threadIdx.x & 31;
    const int64_t f = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    if (f >= n) return;
    const int64_t m = partner[f];
    if (m >= 0 && m < f) return;
    const int64_t i = pidx[f];
    for (int e = 0; e < 2; ++e) {
        const int64_t src = e == 0 ? f : m, row = 2 * i + e;
        uint8_t *c = codes + row * stride, *q = quals + row * stride;
        if (src >= 0) {
            const uint8_t *sc = f_codes + src * stride, *sq = f_quals + src * stride;
            for (int j = lane; j < stride; j += 32) { c[j] = sc[j]; q[j] = sq[j]; }
            ((uint32_t *)(alns + row))[lane] = ((const uint32_t *)(f_alns + src))[lane];          // 128 bytes, 4 per lane
        } else {
            for (int j = lane; j < stride; j += 32) { c[j] = 4; q[j] = 0; }
            if (lane == 0) { qm_aln a; placeholder(a); alns[row] = a; }
        }
        if (lane == 0) {
            lens[row] = src >= 0 ? f_lens[src] : 0;
            row_file[row] = src;
            if (src >= 0) file_row[src] = row;
        }
    }
}

// step 4: the cap's verdict on the file-order rows -> the pair layout
__global__ void __launch_bounds__(256)
bam_drop_scatter_kernel(const uint8_t *__restrict__ f_drop, const int64_t *__restrict__ file_row, int64_t n, uint8_t *__restrict__ drop)
{
    const int64_t f = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (f < n) drop[file_row[f]] = f_drop[f];
}

__global__ void __launch_bounds__(256) iota_kernel(uint32_t *v, int64_t n)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) v[i] = (uint32_t)i;
}

inline size_t al256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

extern "C" {

// the body of qm_bam_to_pairs with the name hash cut to hash_bits bits (1..64): the tests pair through colliding hashes with it
int qm_bam_to_pairs_hashbits(qm_ctx *ctx, const qm_index *idx, const uint8_t *d_bytes, const int64_t *d_rec_off, int64_t n_recs,
                             int32_t stride, const qm_pileup_opt *po, int baq, int max_depth, int hash_bits, qm_bam_pairs *out, void *stream)
{
    if (!ctx || !idx || !po || !out || n_recs < 0 || stride < 1 || max_depth < 0 || hash_bits < 1 || hash_bits > 64 ||
        (baq != 0 && baq != 1 && baq != 3) || (n_recs > 0 && (!d_bytes || !d_rec_off)))
        return QM_EINVAL;
    memset(out, 0, sizeof *out);
    out->stride = stride;
    if (stride > 512) return qm_fail(ctx, QM_ELIMIT, "qm_bam_to_pairs: rows of %d bases: reads longer than 512 bases are not supported", stride);
    if (n_recs > 0x7fffffffll) return qm_fail(ctx, QM_ELIMIT, "qm_bam_to_pairs: %lld records: at most 2^31 - 1", (long long)n_recs);
    if (n_recs == 0) return QM_OK;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n = n_recs, nr = (n + 1) & ~(int64_t)1;           // file-order rows, padded to whole pseudo-pairs for the cap
    const size_t sb = (size_t)stride;
    // scratch 38: file-order rows and the pairing state
    size_t cub_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, cub_bytes, (int32_t *)nullptr, (int32_t *)nullptr, (int)(n + 1), st);
    const size_t o_alns = 0, o_codes = al256((size_t)nr * sizeof(qm_aln)), o_quals = o_codes + al256(nr * sb), o_lens = o_quals + al256(nr * sb);
    const size_t o_hash = o_lens + al256((size_t)nr * 4), o_perm = o_hash + al256((size_t)nr * 8), o_partner = o_perm + al256((size_t)nr * 4);
    const size_t o_lead = o_partner + al256((size_t)nr * 4), o_pidx = o_lead + al256((size_t)(n + 1) * 4);
    const size_t o_frow = o_pidx + al256((size_t)(n + 1) * 4), o_fdrop = o_frow + al256((size_t)n * 8), o_cub = o_fdrop + al256((size_t)nr);
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 38, o_cub + al256(cub_bytes), &p);
    if (rc) return rc;
    char *b = (char *)p;
    qm_aln *f_alns = (qm_aln *)(b + o_alns);
    uint8_t *f_codes = (uint8_t *)(b + o_codes), *f_quals = (uint8_t *)(b + o_quals), *f_drop = (uint8_t *)(b + o_fdrop);
    int32_t *f_lens = (int32_t *)(b + o_lens), *partner = (int32_t *)(b + o_partner), *lead = (int32_t *)(b + o_lead), *pidx = (int32_t *)(b + o_pidx);
    uint64_t *hash = (uint64_t *)(b + o_hash);
    uint32_t *perm = (uint32_t *)(b + o_perm);
    int64_t *file_row = (int64_t *)(b + o_frow);
    const int sp = qm_prof_begin(ctx, QM_ST_OTHER, st);
    bam_decode_kernel<<<(unsigned)((nr * 32 + 127) / 128), 128, 0, st>>>(d_bytes, d_rec_off, n, nr, stride, hash_bits, f_alns, f_codes, f_quals, f_lens, hash);
    QM_CUDA(ctx, cudaGetLastError());
    iota_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(perm, n);
    rc = qm_sort_pairs(ctx, hash, perm, n, hash_bits, st);          // stable: a run of equal hashes keeps file order
    if (rc) return rc;
    bam_pair_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_bytes, d_rec_off, f_alns, hash, perm, n, partner);
    bam_leader_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(partner, n, lead);
    QM_CUDA(ctx, cudaMemsetAsync(lead + n, 0, 4, st));
    QM_CUDA(ctx, cub::DeviceScan::ExclusiveSum(b + o_cub, cub_bytes, lead, pidx, (int)(n + 1), st));
    int32_t h_pairs = 0;
    QM_CUDA(ctx, cudaMemcpyAsync(&h_pairs, pidx + n, 4, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    const int64_t np = h_pairs, rows = 2 * np;
    // scratch 39: the pair layout (alns | codes | quals | BAQ-capped quals | lens | row -> file index | drop bytes)
    const size_t l_codes = al256((size_t)rows * sizeof(qm_aln)), l_quals = l_codes + al256(rows * sb), l_baq = l_quals + al256(rows * sb);
    const size_t l_lens = l_baq + (baq ? al256(rows * sb) : 0), l_rowf = l_lens + al256((size_t)rows * 4), l_drop = l_rowf + al256((size_t)rows * 8);
    rc = qm_scratch_reserve(ctx, 39, l_drop + al256((size_t)rows), &p);
    if (rc) return rc;
    char *y = (char *)p;
    qm_aln *alns = (qm_aln *)y;
    uint8_t *codes = (uint8_t *)(y + l_codes), *quals = (uint8_t *)(y + l_quals), *bq = (uint8_t *)(y + l_baq), *drop = (uint8_t *)(y + l_drop);
    int32_t *lens = (int32_t *)(y + l_lens);
    int64_t *row_file = (int64_t *)(y + l_rowf);
    bam_gather_kernel<<<(unsigned)((n * 32 + 127) / 128), 128, 0, st>>>(f_alns, f_codes, f_quals, f_lens, partner, pidx, n, stride, alns, codes,
                                                                       quals, lens, row_file, file_row);
    QM_CUDA(ctx, cudaGetLastError());
    qm_prof_end(ctx, QM_ST_OTHER, sp, st, 6);
    out->n_pairs = np;
    out->d_alns = alns; out->d_codes = codes; out->d_quals = quals; out->d_lens = lens; out->d_row_file = row_file;
    if (max_depth > 0) {
        // htslib's cap over the reads in file order: rows 2j / 2j + 1 of the file-order table are a pseudo-pair, read id = file index
        const qm_aln *fa = f_alns;
        const int64_t npp = nr / 2;
        uint8_t *fd = f_drop;
        int64_t n_capped = 0;
        rc = qm_depth_cap(ctx, po, 1, &fa, &npp, max_depth, &fd, &n_capped, st);
        if (rc) return rc;
        QM_CUDA(ctx, cudaMemsetAsync(drop, 0, (size_t)rows, st));
        bam_drop_scatter_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(f_drop, file_row, n, drop);
        QM_CUDA(ctx, cudaGetLastError());
        out->d_drop = drop;
        out->n_capped = n_capped;
    }
    if (baq) {
        rc = qm_baq_apply(ctx, idx, po, alns, codes, quals, stride, lens, rows, baq, bq, st);
        if (rc) return rc;
        out->d_quals = bq;
    }
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    return QM_OK;
}

int qm_bam_to_pairs(qm_ctx *ctx, const qm_index *idx, const uint8_t *d_bytes, const int64_t *d_rec_off, int64_t n_recs, int32_t stride,
                    const qm_pileup_opt *po, int baq, int max_depth, qm_bam_pairs *out, void *stream)
{
    return qm_bam_to_pairs_hashbits(ctx, idx, d_bytes, d_rec_off, n_recs, stride, po, baq, max_depth, 64, out, stream);
}

// host bytes in: the record stream and the offsets are staged in scratch 37, then as qm_bam_to_pairs on the context's stream
int qm_bam_to_pairs_host(qm_ctx *ctx, const qm_index *idx, const uint8_t *h_bytes, int64_t n_bytes, const int64_t *h_rec_off, int64_t n_recs,
                         int32_t stride, const qm_pileup_opt *po, int baq, int max_depth, qm_bam_pairs *out)
{
    if (!ctx || n_bytes < 0 || n_recs < 0 || (n_bytes > 0 && !h_bytes) || (n_recs > 0 && !h_rec_off)) return QM_EINVAL;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t o_off = al256((size_t)n_bytes);
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 37, o_off + (size_t)n_recs * 8 + 256, &p);
    if (rc) return rc;
    cudaStream_t st = ctx->own_stream;
    const int sp = qm_prof_begin(ctx, QM_ST_H2D, st);
    if (n_bytes) QM_CUDA(ctx, cudaMemcpyAsync(p, h_bytes, (size_t)n_bytes, cudaMemcpyHostToDevice, st));
    if (n_recs) QM_CUDA(ctx, cudaMemcpyAsync((char *)p + o_off, h_rec_off, (size_t)n_recs * 8, cudaMemcpyHostToDevice, st));
    qm_prof_end(ctx, QM_ST_H2D, sp, st, 0);
    return qm_bam_to_pairs(ctx, idx, (const uint8_t *)p, (const int64_t *)((char *)p + o_off), n_recs, stride, po, baq, max_depth, out, st);
}

}  // extern "C"
