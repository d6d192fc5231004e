// fmindex.cu -- bwa's FM-index as a device-resident part of a qm_index (the alternative seeder of fm_core.cuh).
// Two ways in: qm_index_attach_bwa takes the bytes of the reference's own index files (ref/X.bwt and ref/X.sa, written by
// `bwa index`, rules/index.smk:13) -- the drop-in case, a Snakemake deployment already has them next to every genome; and
// qm_index_build_fm rebuilds the same bytes from the genome on the device, which the tests compare with digests of the
// reference's files.  Either way the index lives in device memory only; qm_index_fm_export copies it back as the two files.
//
// The device build (once per genome, on the context's own stream):
//   text     forward strand then its reverse complement, n = 2 l_pac symbols, one byte each;
//   sort     prefix doubling.  Round 0 sorts every suffix by a 37-bit key: its first 16 symbols packed 2 bits each (zeros behind
//            the end) above min(length, 16), so that a suffix that ends sorts before every suffix it is a prefix of.  The rank
//            of a suffix is the first suffix-array slot of its group of equal keys (a suffix alone in its group has its final
//            slot).  Round h then sorts only the suffixes still tied, by (rank[i], rank[i + h] + 1, or 0 when i + h is the end
//            -- the -1 of bwa's comparison), with the stable LSD radix sort of sort.cu over just the bits the largest key
//            needs (qm_sort_ids); the sorted keys land in the group's slots, new ranks are a max-scan of the group starts,
//            the suffixes left alone drop out of the tied list (a sum-scan compacts it), h doubles; done when none is tied;
//   BWT      row r > 0 holds suffix sa[r - 1], row 0 the sentinel suffix; the symbol before each row's suffix, the row of
//            suffix 0 (bwa's primary) not stored; one warp packs 32 words of 16 symbols and counts them per 128 rows;
//            exclusive scans of those counts give the occurrence checkpoints, interleaved with the symbols as fm_core.cuh
//            reads them (per 128 rows four int64 counts, then 8 words of symbols; one more checkpoint at the end);
//   samples  the suffix of every 32nd row.
// Device memory while it runs: about 58 bytes per suffix (2 l_pac suffixes) -- text 1, rank 4, suffix array 4, tied list
// and its slots 2 x 8, keys 8, permutation 4, the radix sort's second buffers 12, scan values 8, plus the result (0.5) --
// so the 2^31 - 1 suffixes the int32 slots and the format's positions hold need about 125 GB.  More is QM_ELIMIT.
#include <string.h>
#include <cub/device/device_scan.cuh>
#include <utility>
#include "pipeline.cuh"

namespace {

constexpr int kFmSaIntv = 32;                 // bwa index's default suffix-array interval

__global__ void __launch_bounds__(256) fm_text_kernel(uint8_t *__restrict__ t, int64_t l_pac)
{   // t[0, l_pac) holds the forward strand; the reverse complement follows it
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < l_pac) t[2 * l_pac - 1 - i] = (uint8_t)(3 - t[i]);
}

__global__ void __launch_bounds__(256) fm_iota_kernel(int32_t *__restrict__ a, int32_t *__restrict__ b, int64_t n)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) a[i] = b[i] = (int32_t)i;
}

// round 0: the first 16 symbols of suffix i, 2 bits each (A beyond the end), then min(n - i, 16) in the low 5 bits
__global__ void __launch_bounds__(256) fm_key16_kernel(const uint8_t *__restrict__ t, int64_t n, uint64_t *__restrict__ keys)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint64_t v = 0;
#pragma unroll
    for (int j = 0; j < 16; ++j) v = v << 2 | (i + j < n ? t[i + j] : 0u);
    keys[i] = v << 5 | (uint64_t)(n - i < 16 ? n - i : 16);
}

// round h: (rank of the suffix, rank of the suffix h behind it + 1, 0 past the end)
__global__ void __launch_bounds__(256)
fm_pair_key_kernel(const int32_t *__restrict__ tied, int64_t m, const int32_t *__restrict__ rank, int64_t n, int64_t h, int bits,
                   uint64_t *__restrict__ keys)
{
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= m) return;
    const int64_t s = tied[j];
    const uint64_t second = s + h < n ? (uint64_t)rank[s + h] + 1 : 0;
    keys[j] = (uint64_t)rank[s] << bits | second;
}

// the sorted tied suffixes into their slots; a group starts where the key changes, its rank is its first slot
__global__ void __launch_bounds__(256)
fm_place_kernel(const int32_t *__restrict__ tied, const uint32_t *__restrict__ perm, const uint64_t *__restrict__ keys,
                const int32_t *__restrict__ slot, int64_t m, int32_t *__restrict__ sorted, int32_t *__restrict__ sa,
                int32_t *__restrict__ start)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= m) return;
    const int32_t s = tied[perm[k]];
    sorted[k] = s;
    sa[slot[k]] = s;
    start[k] = (k == 0 || keys[k] != keys[k - 1]) ? slot[k] : 0;
}

// new ranks; a suffix stays tied unless its group has only it
__global__ void __launch_bounds__(256)
fm_rerank_kernel(const int32_t *__restrict__ sorted, const int32_t *__restrict__ group, const uint64_t *__restrict__ keys, int64_t m,
                 int32_t *__restrict__ rank, int32_t *__restrict__ keep)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k > m) return;
    if (k == m) { keep[m] = 0; return; }
    rank[sorted[k]] = group[k];
    const bool first = k == 0 || keys[k] != keys[k - 1], last = k + 1 == m || keys[k + 1] != keys[k];
    keep[k] = !(first && last);
}

__global__ void __launch_bounds__(256)
fm_compact_kernel(const int32_t *__restrict__ sorted, const int32_t *__restrict__ slot, const int32_t *__restrict__ keep,
                  const int32_t *__restrict__ at, int64_t m, int32_t *__restrict__ tied, int32_t *__restrict__ slot_out)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k >= m || !keep[k]) return;
    tied[at[k]] = sorted[k];
    slot_out[at[k]] = slot[k];
}

struct MaxOp {
    __device__ __forceinline__ int32_t operator()(int32_t a, int32_t b) const { return a > b ? a : b; }
};

// one thread per word of 16 BWT symbols (symbol i is the one before the suffix of row i, or of row i + 1 from bwa's primary on):
// the word goes to its place behind its block's checkpoint, the block's per-symbol counts to cnt[c * (n_blk + 1) + block]
__global__ void __launch_bounds__(256)
fm_bwt_kernel(const uint8_t *__restrict__ t, const int32_t *__restrict__ sa, int64_t n, int64_t primary, int64_t n_words,
              int64_t n_blk, uint32_t *__restrict__ bwt, int32_t *__restrict__ cnt)
{
    const int64_t w = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;          // whole warps: 8 lanes = one 128-row block
    uint32_t word = 0, c4 = 0;                                                 // four 8-bit counts
    if (w < n_words) {
        for (int j = 0; j < 16; ++j) {
            const int64_t i = w * 16 + j;
            if (i >= n) break;
            const int64_t r = i < primary ? i : i + 1;
            const int64_t sfx = r == 0 ? n : sa[r - 1];
            const uint32_t c = t[sfx - 1];
            word |= c << ((15 - j) << 1);
            c4 += 1u << (c << 3);
        }
        bwt[(w >> 3 << 3) + 8 + w] = word;
    }
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) c4 += __shfl_xor_sync(0xffffffffu, c4, o);
    if (w < n_words && (w & 7) == 0) {
        const int64_t b = w >> 3;
#pragma unroll
        for (int c = 0; c < 4; ++c) cnt[c * (n_blk + 1) + b] = (int32_t)(c4 >> (c << 3) & 255u);
    }
}

// checkpoint b (b = n_blk: the one behind the last symbol) from the exclusive scans of the block counts
__global__ void __launch_bounds__(256)
fm_occ_kernel(const int32_t *__restrict__ occ, int64_t n_blk, int64_t n_words, uint32_t *__restrict__ bwt)
{
    const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (b > n_blk) return;
    uint32_t *at = bwt + b * 8 + (b * 8 < n_words ? b * 8 : n_words);
#pragma unroll
    for (int c = 0; c < 4; ++c) { at[2 * c] = (uint32_t)occ[c * (n_blk + 1) + b]; at[2 * c + 1] = 0u; }
}

__global__ void __launch_bounds__(256) fm_sample_kernel(const int32_t *__restrict__ sa, int64_t n_sa, int intv, int64_t *__restrict__ out)
{
    const int64_t k = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (k < n_sa) out[k] = k == 0 ? -1 : (int64_t)sa[k * intv - 1];
}

unsigned blocks(int64_t n) { return (unsigned)((n + 255) / 256); }

}  // namespace

extern "C" {

// h_bwt / h_sa: the two files as bwa 0.7.17 writes them (.bwt: int64 primary, int64 L2[1..4], then per 128 rows four int64
// occurrence counts + eight uint32 words of sixteen 2-bit symbols; .sa: int64 primary, four int64, int64 sa_intv, int64 seq_len,
// then the samples of rows sa_intv, 2 sa_intv, ...).  The index must be of the same genome: seq_len = 2 x l_pac is checked.
int qm_index_attach_bwa(qm_ctx *ctx, qm_index *idx, const uint8_t *h_bwt, int64_t bwt_bytes, const uint8_t *h_sa, int64_t sa_bytes)
{
    if (!ctx || !idx || !h_bwt || !h_sa) return QM_EINVAL;
    if (bwt_bytes < 40 || sa_bytes < 56) return qm_fail(ctx, QM_EINVAL, "qm_index_attach_bwa: truncated index files");
    int64_t hdr[5], sh[7];
    memcpy(hdr, h_bwt, 40);
    memcpy(sh, h_sa, 56);
    FmView F;
    F.primary = hdr[0]; F.L2[0] = 0; memcpy(F.L2 + 1, hdr + 1, 32); F.seq_len = F.L2[4]; F.sa_intv = (int)sh[5];
    if (sh[0] != F.primary || sh[6] != F.seq_len) return qm_fail(ctx, QM_EINVAL, "qm_index_attach_bwa: the .bwt and the .sa are not of one index");
    if (F.seq_len != 2 * idx->v.l_pac)
        return qm_fail(ctx, QM_EINVAL, "qm_index_attach_bwa: the index covers %lld symbols, this genome needs %lld (forward + reverse complement)",
                       (long long)F.seq_len, (long long)(2 * idx->v.l_pac));
    if (F.sa_intv < 1 || (F.sa_intv & (F.sa_intv - 1))) return qm_fail(ctx, QM_EINVAL, "qm_index_attach_bwa: suffix-array interval %d is not a power of two", F.sa_intv);
    const int64_t n_words = (bwt_bytes - 40) / 4, need_words = ((F.seq_len + 127) / 128 + 1) * 8 + (F.seq_len + 15) / 16;
    const int64_t n_sa = (F.seq_len + F.sa_intv) / F.sa_intv;
    if (n_words < need_words - 8 || sa_bytes < 56 + 8 * (n_sa - 1)) return qm_fail(ctx, QM_EINVAL, "qm_index_attach_bwa: index files shorter than their headers say");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    if (idx->d_fm_bwt) { cudaFree(idx->d_fm_bwt); idx->d_fm_bwt = nullptr; }
    if (idx->d_fm_sa) { cudaFree(idx->d_fm_sa); idx->d_fm_sa = nullptr; }
    idx->have_fm = false;
    cudaStream_t st = ctx->own_stream;
    const int64_t minus1 = -1;
    QM_CUDA(ctx, cudaMalloc(&idx->d_fm_bwt, (size_t)n_words * 4 + 64));
    QM_CUDA(ctx, cudaMemsetAsync(idx->d_fm_bwt, 0, (size_t)n_words * 4 + 64, st));
    QM_CUDA(ctx, cudaMemcpyAsync(idx->d_fm_bwt, h_bwt + 40, (size_t)n_words * 4, cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMalloc(&idx->d_fm_sa, (size_t)n_sa * 8));
    QM_CUDA(ctx, cudaMemcpyAsync(idx->d_fm_sa, &minus1, 8, cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync((int64_t *)idx->d_fm_sa + 1, h_sa + 56, (size_t)(n_sa - 1) * 8, cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    F.bwt = (const uint32_t *)idx->d_fm_bwt; F.sa = (const int64_t *)idx->d_fm_sa;
    idx->fm = F;
    idx->fm_words = n_words;
    idx->fm_device = ctx->device;
    idx->have_fm = true;
    return QM_OK;
}

// the same index built on the device from the genome (h_codes as given to qm_index_build)
int qm_index_build_fm(qm_ctx *ctx, qm_index *idx, const uint8_t *h_codes)
{
    if (!ctx || !idx || !h_codes) return QM_EINVAL;
    const int64_t l_pac = idx->v.l_pac, n = 2 * l_pac;
    if (n >= (1ll << 31))
        return qm_fail(ctx, QM_ELIMIT, "qm_index_build_fm: %lld suffixes (forward + reverse complement): at most 2^31 - 1 (32-bit suffix positions)",
                       (long long)n);
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    if (idx->d_fm_bwt) { cudaFree(idx->d_fm_bwt); idx->d_fm_bwt = nullptr; }
    if (idx->d_fm_sa) { cudaFree(idx->d_fm_sa); idx->d_fm_sa = nullptr; }
    idx->have_fm = false;
    cudaStream_t st = ctx->own_stream;
    const int sp = qm_prof_begin(ctx, QM_ST_OTHER, st);
    int bits = 1;                                          // rank + 1 < 2^bits
    while ((n >> bits) != 0) ++bits;
    size_t cub_sum = 0, cub_max = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, cub_sum, (int32_t *)nullptr, (int32_t *)nullptr, (int)(n + 1), st);
    cub::DeviceScan::InclusiveScan(nullptr, cub_max, (int32_t *)nullptr, (int32_t *)nullptr, MaxOp(), (int)n, st);
    size_t cub_bytes = cub_sum > cub_max ? cub_sum : cub_max;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t i4 = al((size_t)(n + 1) * 4);
    const size_t o_t = 0, o_rank = al((size_t)n), o_sa = o_rank + i4, o_tied = o_sa + i4, o_slot = o_tied + i4, o_sorted = o_slot + i4,
                 o_slot2 = o_sorted + i4, o_start = o_slot2 + i4, o_group = o_start + i4, o_perm = o_group + i4, o_keys = o_perm + i4,
                 o_cub = o_keys + al((size_t)n * 8), total = o_cub + al(cub_bytes);
    char *b = nullptr;
    QM_CUDA(ctx, cudaMalloc(&b, total));
    struct Arena { char *p; ~Arena() { cudaFree(p); } } arena{b};
    uint8_t *t = (uint8_t *)(b + o_t);
    int32_t *rank = (int32_t *)(b + o_rank), *sa = (int32_t *)(b + o_sa), *tied = (int32_t *)(b + o_tied), *slot = (int32_t *)(b + o_slot);
    int32_t *sorted = (int32_t *)(b + o_sorted), *slot2 = (int32_t *)(b + o_slot2), *start = (int32_t *)(b + o_start), *group = (int32_t *)(b + o_group);
    uint32_t *perm = (uint32_t *)(b + o_perm);
    uint64_t *keys = (uint64_t *)(b + o_keys);
    int32_t *keep = start, *at = group;                   // reused once the new ranks are out
    int32_t *h_m = (int32_t *)ctx->h_pinned;

    QM_CUDA(ctx, cudaMemcpyAsync(t, h_codes, (size_t)l_pac, cudaMemcpyHostToDevice, st));
    fm_text_kernel<<<blocks(l_pac), 256, 0, st>>>(t, l_pac);
    fm_iota_kernel<<<blocks(n), 256, 0, st>>>(tied, slot, n);
    fm_key16_kernel<<<blocks(n), 256, 0, st>>>(t, n, keys);
    QM_CUDA(ctx, cudaGetLastError());
    int launches = 3;
    int64_t m = n;
    for (int64_t h = 16;; h *= 2) {
        int rc = qm_sort_ids(ctx, keys, perm, m, "qm_index_build_fm", st);
        if (rc) return rc;
        fm_place_kernel<<<blocks(m), 256, 0, st>>>(tied, perm, keys, slot, m, sorted, sa, start);
        QM_CUDA(ctx, cub::DeviceScan::InclusiveScan(b + o_cub, cub_bytes, start, group, MaxOp(), (int)m, st));
        fm_rerank_kernel<<<blocks(m + 1), 256, 0, st>>>(sorted, group, keys, m, rank, keep);
        QM_CUDA(ctx, cub::DeviceScan::ExclusiveSum(b + o_cub, cub_bytes, keep, at, (int)(m + 1), st));
        fm_compact_kernel<<<blocks(m), 256, 0, st>>>(sorted, slot, keep, at, m, tied, slot2);
        QM_CUDA(ctx, cudaGetLastError());
        QM_CUDA(ctx, cudaMemcpyAsync(h_m, at + m, 4, cudaMemcpyDeviceToHost, st));
        QM_CUDA(ctx, cudaStreamSynchronize(st));
        launches += 6;
        std::swap(slot, slot2);
        m = *h_m;
        if (m == 0) break;
        if (h >= n) return qm_fail(ctx, QM_ECUDA, "qm_index_build_fm: %lld suffixes still tied after %lld symbols", (long long)m, (long long)h);
        fm_pair_key_kernel<<<blocks(m), 256, 0, st>>>(tied, m, rank, n, h, bits, keys);
    }
    // every rank is now the suffix's slot: the row of suffix 0 is bwa's primary
    int32_t sa0 = 0;
    QM_CUDA(ctx, cudaMemcpyAsync(h_m, rank, 4, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    sa0 = *h_m;
    const int64_t primary = (int64_t)sa0 + 1, n_words = (n + 15) / 16, n_blk = (n + 127) / 128, all_words = (n_blk + 1) * 8 + n_words;
    const int64_t n_sa = (n + kFmSaIntv) / kFmSaIntv;
    void *d_bwt = nullptr, *d_sa = nullptr;
    QM_CUDA(ctx, cudaMalloc(&d_bwt, (size_t)all_words * 4 + 64));
    idx->d_fm_bwt = d_bwt;
    QM_CUDA(ctx, cudaMalloc(&d_sa, (size_t)n_sa * 8));
    idx->d_fm_sa = d_sa;
    QM_CUDA(ctx, cudaMemsetAsync(d_bwt, 0, (size_t)all_words * 4 + 64, st));
    int32_t *cnt = sorted, *occ = slot2;                  // [symbol][block + 1] counts and their exclusive scans (4 (n_blk + 1) <= n + 1)
    QM_CUDA(ctx, cudaMemsetAsync(cnt, 0, (size_t)4 * (n_blk + 1) * 4, st));
    fm_bwt_kernel<<<blocks((n_words + 31) & ~(int64_t)31), 256, 0, st>>>(t, sa, n, primary, n_words, n_blk, (uint32_t *)d_bwt, cnt);
    for (int c = 0; c < 4; ++c)
        QM_CUDA(ctx, cub::DeviceScan::ExclusiveSum(b + o_cub, cub_bytes, cnt + c * (n_blk + 1), occ + c * (n_blk + 1), (int)(n_blk + 1), st));
    fm_occ_kernel<<<blocks(n_blk + 1), 256, 0, st>>>(occ, n_blk, n_words, (uint32_t *)d_bwt);
    fm_sample_kernel<<<blocks(n_sa), 256, 0, st>>>(sa, n_sa, kFmSaIntv, (int64_t *)d_sa);
    QM_CUDA(ctx, cudaGetLastError());
    uint32_t tail[8];
    QM_CUDA(ctx, cudaMemcpyAsync(tail, (uint32_t *)d_bwt + n_blk * 8 + n_words, 32, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    qm_prof_end(ctx, QM_ST_OTHER, sp, st, launches + 8);
    FmView F;
    F.bwt = (const uint32_t *)d_bwt; F.sa = (const int64_t *)d_sa;
    F.primary = primary; F.seq_len = n; F.sa_intv = kFmSaIntv;
    F.L2[0] = 0;
    for (int c = 0; c < 4; ++c) F.L2[c + 1] = F.L2[c] + (int64_t)tail[2 * c];
    idx->fm = F;
    idx->fm_words = all_words;
    idx->fm_device = ctx->device;
    idx->have_fm = true;
    return QM_OK;
}

// the attached index as the two files bwa would write (sizes with NULL buffers); the bulk comes back from the device here only
int qm_index_fm_export(const qm_index *idx, uint8_t *h_bwt, int64_t *bwt_bytes, uint8_t *h_sa, int64_t *sa_bytes)
{
    if (!idx || !bwt_bytes || !sa_bytes) return QM_EINVAL;
    if (!idx->have_fm) return QM_EINVAL;
    const FmView &F = idx->fm;
    const int64_t n_sa = (F.seq_len + F.sa_intv) / F.sa_intv;
    *bwt_bytes = 40 + idx->fm_words * 4; *sa_bytes = 56 + (n_sa - 1) * 8;
    if (!h_bwt && !h_sa) return QM_OK;
    int prev = 0;
    if (cudaGetDevice(&prev) != cudaSuccess || cudaSetDevice(idx->fm_device) != cudaSuccess) return QM_ECUDA;
    cudaError_t e = cudaSuccess;
    if (h_bwt) {
        const int64_t hdr[5] = {F.primary, F.L2[1], F.L2[2], F.L2[3], F.L2[4]};
        memcpy(h_bwt, hdr, 40);
        e = cudaMemcpyAsync(h_bwt + 40, idx->d_fm_bwt, (size_t)idx->fm_words * 4, cudaMemcpyDeviceToHost, cudaStreamPerThread);
    }
    if (h_sa) {
        const int64_t sh[7] = {F.primary, F.L2[1], F.L2[2], F.L2[3], F.L2[4], F.sa_intv, F.seq_len};
        memcpy(h_sa, sh, 56);
        if (e == cudaSuccess && n_sa > 1)
            e = cudaMemcpyAsync(h_sa + 56, (const int64_t *)idx->d_fm_sa + 1, (size_t)(n_sa - 1) * 8, cudaMemcpyDeviceToHost, cudaStreamPerThread);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamPerThread);
    cudaSetDevice(prev);
    return e == cudaSuccess ? QM_OK : QM_ECUDA;
}

}  // extern "C"
