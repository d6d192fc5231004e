// sort.cu -- coordinate sort of alignment records on the device (the ordering `samtools sort` produces in the
// reference's `bwa` rule, rules/bwa.smk:17; comparator bam1_lt of samtools 1.9 bam_sort.c, SURVEY.md A.7).
//
// Records stay where they are (128 B each): what is sorted is a (64-bit key, 32-bit record index) pair per record,
// with a stable least-significant-digit radix sort, 8 bits per pass, over just the key bits in use (a 235 kb
// genome needs 24 bits -> 3 passes).  Stability gives samtools' tie rule (input order) without carrying the
// index in the key.  Per pass: (1) per-tile digit histograms, (2) one exclusive scan over [digit][tile],
// (3) scatter with a stable in-tile rank: a warp walks its 512 consecutive keys 32 at a time, __match_any_sync
// groups equal digits, the group's first lane bumps the warp's shared counter, ranks follow lane order.
// HBM-bound by construction: 12 B read + 12 B written per record per pass (+ the histogram read).
#include "pipeline.cuh"

namespace {

constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;
constexpr int kSortItems = 16;                                   // keys per lane
constexpr int kSortTile = kSortThreads * kSortItems;             // 4096 keys per block

__global__ void __launch_bounds__(256)
aln_keys_kernel(const qm_aln *__restrict__ alns, int64_t n, int n_contigs, int pos_bits, uint64_t *__restrict__ keys)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t rid = alns[i].rid, pos = alns[i].pos;
    const unsigned flag = alns[i].flag;
    keys[i] = qm_sort_key(rid, pos, (flag & 0x10) != 0, n_contigs, pos_bits);
}

__global__ void __launch_bounds__(kSortThreads)
radix_hist_kernel(const uint64_t *__restrict__ keys, int64_t n, int shift, unsigned *__restrict__ hist, int n_tiles)
{
    __shared__ unsigned h[256];
    h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * kSortTile;
#pragma unroll 4
    for (int k = 0; k < kSortItems; ++k) {
        const int64_t i = base + (int64_t)k * kSortThreads + threadIdx.x;
        if (i < n) atomicAdd(&h[(unsigned)(keys[i] >> shift) & 255u], 1u);
    }
    __syncthreads();
    hist[(size_t)threadIdx.x * n_tiles + blockIdx.x] = h[threadIdx.x];
}

// exclusive scan over [digit][tile] in two small steps (one block walking all 256 x tiles counters took 0.14 ms per pass on a
// 2.7 M-key list, most of the sort): block d scans the tiles of digit d and leaves the digit's total behind the table, then one
// warp-sized step turns the 256 totals into the digits' bases; the scatter adds the two.
__global__ void __launch_bounds__(256) radix_scan_rows_kernel(unsigned *__restrict__ hist, int n_tiles)
{
    __shared__ unsigned warp_sum[8];
    __shared__ unsigned carry;
    unsigned *row = hist + (size_t)blockIdx.x * n_tiles;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n_tiles; c0 += 256) {
        const int i = c0 + threadIdx.x;
        const unsigned v = i < n_tiles ? row[i] : 0u;
        unsigned inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        if (lane == 31) warp_sum[warp] = inc;
        __syncthreads();
        unsigned before = carry;
        for (int w = 0; w < warp; ++w) before += warp_sum[w];
        if (i < n_tiles) row[i] = before + inc - v;
        __syncthreads();
        if (threadIdx.x == 255) carry = before + inc;
        __syncthreads();
    }
    if (threadIdx.x == 0) hist[(size_t)256 * n_tiles + blockIdx.x] = carry;
}
__global__ void __launch_bounds__(256) radix_scan_digits_kernel(unsigned *__restrict__ totals)
{
    __shared__ unsigned s[256];
    s[threadIdx.x] = totals[threadIdx.x];
    __syncthreads();
    unsigned acc = 0;
    for (int d = 0; d < (int)threadIdx.x; ++d) acc += s[d];
    totals[threadIdx.x] = acc;
}

__global__ void __launch_bounds__(kSortThreads)
radix_scatter_kernel(const uint64_t *__restrict__ keys_in, const uint32_t *__restrict__ vals_in /* NULL: iota */, int64_t n,
                     int shift, const unsigned *__restrict__ offs, int n_tiles, uint64_t *__restrict__ keys_out,
                     uint32_t *__restrict__ vals_out)
{
    __shared__ unsigned cnt[kSortWarps][256];
    for (int i = threadIdx.x; i < kSortWarps * 256; i += kSortThreads) (&cnt[0][0])[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    const int64_t base = (int64_t)blockIdx.x * kSortTile + (int64_t)warp * (32 * kSortItems);
    uint64_t key[kSortItems];
    uint32_t val[kSortItems];
    unsigned rank[kSortItems];
#pragma unroll
    for (int k = 0; k < kSortItems; ++k) {
        const int64_t i = base + k * 32 + lane;
        const bool valid = i < n;
        key[k] = valid ? keys_in[i] : ~0ull;
        val[k] = valid ? (vals_in ? vals_in[i] : (uint32_t)i) : 0u;
        const unsigned d = valid ? (unsigned)(key[k] >> shift) & 255u : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int leader = __ffs(peers) - 1;
        unsigned old = 0;
        if (lane == leader && valid) { old = cnt[warp][d]; cnt[warp][d] = old + __popc(peers); }
        old = __shfl_sync(0xffffffffu, old, leader);
        rank[k] = old + __popc(peers & lt);
        __syncwarp();
    }
    __syncthreads();
    {   // digit threadIdx.x: global base of this tile, then the warps in order
        const int d = threadIdx.x;
        unsigned run = offs[(size_t)d * n_tiles + blockIdx.x] + offs[(size_t)256 * n_tiles + d];
#pragma unroll
        for (int w = 0; w < kSortWarps; ++w) { const unsigned t = cnt[w][d]; cnt[w][d] = run; run += t; }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kSortItems; ++k) {
        const int64_t i = base + k * 32 + lane;
        if (i < n) {
            const unsigned d = (unsigned)(key[k] >> shift) & 255u;
            const unsigned o = cnt[warp][d] + rank[k];
            keys_out[o] = key[k];
            vals_out[o] = val[k];
        }
    }
}

__global__ void __launch_bounds__(256)
max_key_kernel(const uint64_t *__restrict__ keys, int64_t n, unsigned long long *__restrict__ mx)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    unsigned long long v = i < n ? keys[i] : 0ull;
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o); v = u > v ? u : v; }
    if ((threadIdx.x & 31) == 0 && v) atomicMax(mx, v);
}

}  // namespace

// The ids of a union of exported tuples (dedup.cu, depthcap.cu), stably sorted over just the bits the largest id needs; d_perm[i] =
// input position of the id at sorted position i.  Ids are int64 values cast to uint64: a negative one is QM_EINVAL.  Synchronous.
int qm_sort_ids(qm_ctx *ctx, uint64_t *d_ids, uint32_t *d_perm, int64_t n, const char *who, cudaStream_t st)
{
    if (n == 0) return QM_OK;
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 33, 256, &p);
    if (rc) return rc;
    unsigned long long *mx = (unsigned long long *)p, h = 0;
    QM_CUDA(ctx, cudaMemsetAsync(mx, 0, 8, st));
    max_key_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_ids, n, mx);
    QM_CUDA(ctx, cudaGetLastError());
    QM_CUDA(ctx, cudaMemcpyAsync(&h, mx, 8, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    if (h >> 63) return qm_fail(ctx, QM_EINVAL, "%s: negative id in the union", who);
    int bits = 1;
    while (bits < 63 && (h >> bits)) ++bits;
    return qm_sort_pairs(ctx, d_ids, d_perm, n, bits, st);
}

extern "C" {

int qm_aln_sort_keys(qm_ctx *ctx, const qm_index *idx, const qm_aln *d_alns, int64_t n, uint64_t *d_keys, int *key_bits, void *stream)
{
    if (!ctx || !idx || n < 0 || (n > 0 && (!d_alns || !d_keys))) return QM_EINVAL;
    int64_t max_len = 0;
    for (int c = 0; c < idx->v.n_contigs; ++c) max_len = idx->v.len[c] > max_len ? idx->v.len[c] : max_len;
    const int pos_bits = qm_sort_pos_bits(max_len);
    if (key_bits) *key_bits = qm_sort_key_bits(idx->v.n_contigs, pos_bits);
    if (n == 0) return QM_OK;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    aln_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_alns, n, idx->v.n_contigs, pos_bits, d_keys);
    QM_CUDA(ctx, cudaGetLastError());
    return QM_OK;
}

int qm_sort_pairs(qm_ctx *ctx, uint64_t *d_keys, uint32_t *d_vals, int64_t n, int key_bits, void *stream)
{
    if (!ctx || n < 0 || key_bits < 1 || key_bits > 64 || (n > 0 && (!d_keys || !d_vals))) return QM_EINVAL;
    if (n > 0xffffffffll) return qm_fail(ctx, QM_ELIMIT, "qm_sort_pairs: more than 2^32 records");
    if (n == 0) return QM_OK;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int n_tiles = (int)((n + kSortTile - 1) / kSortTile);
    const size_t kb = ((size_t)n * 8 + 255) & ~(size_t)255, vb = ((size_t)n * 4 + 255) & ~(size_t)255;
    const size_t hb = ((size_t)256 * n_tiles + 256) * sizeof(unsigned);        // [digit][tile] counters, then the 256 digit bases
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 12, kb + vb + hb, &p);
    if (rc) return rc;
    uint64_t *k_alt = (uint64_t *)p;
    uint32_t *v_alt = (uint32_t *)((char *)p + kb);
    unsigned *hist = (unsigned *)((char *)p + kb + vb);
    const int passes = (key_bits + 7) / 8;
    uint64_t *k_in = d_keys, *k_out = k_alt;
    uint32_t *v_in = nullptr, *v_out = (passes & 1) ? d_vals : v_alt;   // arranged so that the last pass lands in d_vals;
    // with an odd number of passes the keys end in k_alt and are copied back afterwards
    const int sp = qm_prof_begin(ctx, QM_ST_OTHER, st);
    for (int ps = 0; ps < passes; ++ps) {
        const int shift = 8 * ps;
        radix_hist_kernel<<<n_tiles, kSortThreads, 0, st>>>(k_in, n, shift, hist, n_tiles);
        radix_scan_rows_kernel<<<256, 256, 0, st>>>(hist, n_tiles);
        radix_scan_digits_kernel<<<1, 256, 0, st>>>(hist + (size_t)256 * n_tiles);
        radix_scatter_kernel<<<n_tiles, kSortThreads, 0, st>>>(k_in, v_in, n, shift, hist, n_tiles, k_out, v_out);
        uint64_t *tk = k_in; k_in = k_out; k_out = tk;
        v_in = v_out; v_out = (v_out == d_vals) ? v_alt : d_vals;
    }
    qm_prof_end(ctx, QM_ST_OTHER, sp, st, 4 * passes);
    QM_CUDA(ctx, cudaGetLastError());
    if (k_in != d_keys) QM_CUDA(ctx, cudaMemcpyAsync(d_keys, k_in, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
    if (v_in != d_vals) QM_CUDA(ctx, cudaMemcpyAsync(d_vals, v_in, (size_t)n * 4, cudaMemcpyDeviceToDevice, st));
    return QM_OK;
}

// keys on the host in, permutation out: h_perm[i] = input index of the record at sorted position i.  Synchronous.
int qm_sort_keys_host(qm_ctx *ctx, const uint64_t *h_keys, int64_t n, int key_bits, uint32_t *h_perm)
{
    if (!ctx || n < 0 || (n > 0 && (!h_keys || !h_perm))) return QM_EINVAL;
    if (n == 0) return QM_OK;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t kb = ((size_t)n * 8 + 255) & ~(size_t)255;
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 13, kb + (size_t)n * 4, &p);
    if (rc) return rc;
    uint64_t *dk = (uint64_t *)p;
    uint32_t *dv = (uint32_t *)((char *)p + kb);
    cudaStream_t st = ctx->own_stream;
    QM_CUDA(ctx, cudaMemcpyAsync(dk, h_keys, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    rc = qm_sort_pairs(ctx, dk, dv, n, key_bits, st);
    if (rc) return rc;
    QM_CUDA(ctx, cudaMemcpyAsync(h_perm, dv, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    return QM_OK;
}

// page-locked host memory for the driver's read / record buffers (copies then overlap the kernels)
int qm_host_alloc(qm_ctx *ctx, size_t bytes, void **out)
{
    if (!ctx || !out) return QM_EINVAL;
    *out = nullptr;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable);      // page-locked for every device: the multi-GPU driver deals batches to any GPU
    if (e != cudaSuccess) return qm_fail(ctx, QM_ENOMEM, "qm_host_alloc(%zu): %s", bytes, cudaGetErrorString(e));
    return QM_OK;
}

void qm_host_free(qm_ctx *ctx, void *p)
{
    if (!ctx || !p) return;
    cudaSetDevice(ctx->device);
    cudaFreeHost(p);
}

}  // extern "C"
