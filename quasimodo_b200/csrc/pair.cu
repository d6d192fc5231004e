// pair.cu -- paired-end stage: insert-size model, primary marking, pairing, MAPQ, CIGAR/NM, SAM flags.
// Replaces the compute of `bwa mem` worker2 (bwamem_pair.c mem_pestat, mem_pair, mem_sam_pe -- mate rescue
// lives in rescue.cu; bwamem.c mem_mark_primary_se, mem_approx_mapq_se, mem_reg2aln; bwa.c bwa_gen_cigar2;
// ksw.c ksw_global2 -- reference call site rules/bwa.smk:15; semantics SURVEY.md A.4-A.6).
// One thread per pair.  The floating-point pieces (log / erfc) are evaluated on the HOST into small
// tables (same libm as the CPU path) so that the integer MAPQ / pair scores are bit-identical; the
// device only does IEEE add/mul/div on those table values (the library is built with -fmad=false).
#include <math.h>
#include <algorithm>
#include <vector>
#include "pipeline.cuh"

namespace {

constexpr int kMapqTabLen = 1024;
constexpr int kSubnTabLen = 256;

struct PairTables {
    const double *mapq_l;        // [kMapqTabLen]: l < coef_len ? 1 : log(coef_len)/log(l)
    const int *subn;             // [kSubnTabLen]: (int)(4.343*log(n+1)+.499)
    // insert-size models, 4 per model (FF FR RF RR); pair p uses model model_of[p] (model 0 when model_of is NULL: one model
    // for the whole batch).  term + term_off[4 m + d]: .721*log(2*erfc(|ns|/sqrt2))*a of model m, orientation d, dist = low..high
    const qm_pestat *pes;
    const double *term;
    const int64_t *term_off;
    const int32_t *model_of;
};

__device__ __forceinline__ int pair_model(const PairTables &T, int64_t pi) { return T.model_of ? T.model_of[pi] : 0; }


__device__ __forceinline__ uint64_t hash64(uint64_t key)
{
    key += ~(key << 32); key ^= (key >> 22); key += ~(key << 13); key ^= (key >> 8);
    key += (key << 3);   key ^= (key >> 15); key += ~(key << 27); key ^= (key >> 31);
    return key;
}

__device__ int cal_sub(const qm_opt &o, const qm_reg *a, int n)
{
    int j;
    for (j = 1; j < n; ++j) {
        const int b_max = a[j].qb > a[0].qb ? a[j].qb : a[0].qb;
        const int e_min = a[j].qe < a[0].qe ? a[j].qe : a[0].qe;
        if (e_min > b_max) {
            const int l0 = a[0].qe - a[0].qb, lj = a[j].qe - a[j].qb;
            const int min_l = lj < l0 ? lj : l0;
            if (e_min - b_max >= min_l * o.mask_level) break;
        }
    }
    return j < n ? a[j].score : o.min_seed_len * o.a;
}

// insert-size histogram for mem_pestat: hist[chunk][dir][isize] += 1 for every qualifying pair.  model_of (may be NULL: one
// histogram) gives each pair's chunk; the launch covers the pairs of chunks c0.. and hist starts at chunk c0's.
__global__ void pestat_hist_kernel(IndexView V, qm_opt o, const qm_reg *__restrict__ regs, const int32_t *__restrict__ n_regs,
                                   int64_t p0, int64_t n_pairs, const int32_t *__restrict__ model_of, int c0, unsigned *__restrict__ hist)
{
    const int64_t i = p0 + blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= p0 + n_pairs) return;
    const qm_reg *r0 = regs + (2 * i) * QM_MAX_REGS, *r1 = regs + (2 * i + 1) * QM_MAX_REGS;
    const int n0 = n_regs[2 * i], n1 = n_regs[2 * i + 1];
    if (n0 && n1 && !(cal_sub(o, r0, n0) > 0.8 * r0[0].score) && !(cal_sub(o, r1, n1) > 0.8 * r1[0].score) &&
        r0[0].rid == r1[0].rid) {
        int64_t is;
        const int dir = qm_infer_dir(V.l_pac, r0[0].rb, r1[0].rb, &is);
        const int64_t c = model_of ? model_of[i] - c0 : 0;
        if (is && is <= o.max_ins) atomicAdd(&hist[(c * 4 + dir) * (o.max_ins + 1) + is], 1u);
    }
}

// pair p -> the chunk it belongs to (chunk c holds pairs start[c] .. start[c + 1] - 1)
__global__ void chunk_of_kernel(const int64_t *__restrict__ start, int n_chunks, int64_t n_pairs, int32_t *__restrict__ model_of)
{
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    int lo = 0, hi = n_chunks - 1;
    while (lo < hi) { const int m = (lo + hi + 1) >> 1; if (start[m] <= i) lo = m; else hi = m - 1; }
    model_of[i] = lo;
}

// mem_pestat over one histogram per chunk (bwamem_pair.c, bwa 0.7.17 as recalled): block = chunk, thread = orientation.
// Each thread walks its bins in ascending order, the operation order of mem_pestat over its sorted list and of the host
// replay in qm_pestat_sync.  The average's sum is a sum of integers (exact in any order); the variance's sum is not, so it
// is added one pair at a time, as bwa adds it.  Then the orientations with fewer than 5 % of the best one's pairs fail.
__global__ void __launch_bounds__(32)
pestat_model_kernel(const unsigned *__restrict__ hist, int max_ins, int c0, qm_pestat *__restrict__ pes)
{
    __shared__ int64_t s_cnt[4];
    const int d = threadIdx.x;
    const int64_t bins = (int64_t)max_ins + 1;
    qm_pestat r;
    r.low = r.high = r.failed = r.pad = 0; r.avg = r.std = 0;
    if (d < 4) {
        const unsigned *q = hist + ((int64_t)blockIdx.x * 4 + d) * bins;
        int64_t n = 0;
        for (int64_t v = 0; v < bins; ++v) n += q[v];
        s_cnt[d] = n;
        if (n < 10) r.failed = 1;
        else {
            const int64_t k25 = (int)(.25 * n + .499), k75 = (int)(.75 * n + .499);
            int p25 = (int)bins - 1, p75 = (int)bins - 1;
            {
                int64_t c = 0;
                bool h25 = false;
                for (int64_t v = 0; v < bins; ++v) {
                    c += q[v];
                    if (!h25 && c > k25) { p25 = (int)v; h25 = true; }
                    if (c > k75) { p75 = (int)v; break; }
                }
            }
            r.low = (int)(p25 - 2.0 * (p75 - p25) + .499);
            if (r.low < 1) r.low = 1;
            r.high = (int)(p75 + 2.0 * (p75 - p25) + .499);
            int64_t x = 0, sum = 0;
            for (int64_t v = r.low; v <= r.high && v < bins; ++v) { sum += (int64_t)q[v] * v; x += q[v]; }
            r.avg = (double)sum / x;
            for (int64_t v = r.low; v <= r.high && v < bins; ++v) {
                const double dlt = ((double)v - r.avg) * ((double)v - r.avg);
                for (unsigned c = 0; c < q[v]; ++c) r.std = __dadd_rn(r.std, dlt);
            }
            r.std = sqrt(r.std / x);
            r.low = (int)(p25 - 3.0 * (p75 - p25) + .499);
            r.high = (int)(p75 + 3.0 * (p75 - p25) + .499);
            if (r.low > r.avg - 4.0 * r.std) r.low = (int)(r.avg - 4.0 * r.std + .499);
            if (r.high < r.avg + 4.0 * r.std) r.high = (int)(r.avg + 4.0 * r.std + .499);
            if (r.low < 1) r.low = 1;
        }
    }
    __syncthreads();
    if (d < 4) {
        int64_t mx = 0;
        for (int e = 0; e < 4; ++e) mx = s_cnt[e] > mx ? s_cnt[e] : mx;
        if (!r.failed && s_cnt[d] < mx * 0.05) r.failed = 1;
        pes[((int64_t)c0 + blockIdx.x) * 4 + d] = r;
    }
}

// mem_mark_primary_se: sort by (score desc, hash asc), mark secondaries, fill sub / sub_n
__device__ void mark_primary(const qm_opt &o, int n, qm_reg *a, uint64_t id)
{
    if (n == 0) return;
    uint64_t hsh[QM_MAX_REGS];
    int z[QM_MAX_REGS], nz = 0;
    for (int i = 0; i < n; ++i) { a[i].sub = 0; a[i].sub_n = 0; a[i].secondary = -1; hsh[i] = hash64(id + i); }
    for (int i = 1; i < n; ++i) {
        const qm_reg x = a[i];
        const uint64_t hx = hsh[i];
        int j = i - 1;
        while (j >= 0 && !(a[j].score > x.score || (a[j].score == x.score && hsh[j] <= hx))) { a[j + 1] = a[j]; hsh[j + 1] = hsh[j]; --j; }
        a[j + 1] = x; hsh[j + 1] = hx;
    }
    int tmp = o.a + o.b;
    if (o.o_del + o.e_del > tmp) tmp = o.o_del + o.e_del;
    if (o.o_ins + o.e_ins > tmp) tmp = o.o_ins + o.e_ins;
    z[nz++] = 0;
    for (int i = 1; i < n; ++i) {
        int k;
        for (k = 0; k < nz; ++k) {
            const int j = z[k];
            const int b_max = a[j].qb > a[i].qb ? a[j].qb : a[i].qb;
            const int e_min = a[j].qe < a[i].qe ? a[j].qe : a[i].qe;
            if (e_min > b_max) {
                const int li = a[i].qe - a[i].qb, lj = a[j].qe - a[j].qb;
                const int min_l = li < lj ? li : lj;
                if (e_min - b_max >= min_l * o.mask_level) {
                    if (a[j].sub == 0) a[j].sub = a[i].score;
                    if (a[j].score - a[i].score <= tmp) ++a[j].sub_n;
                    break;
                }
            }
        }
        if (k == nz) z[nz++] = i; else a[i].secondary = z[k];
    }
}

__device__ int approx_mapq(const qm_opt &o, const PairTables &T, const qm_reg &a)
{
    int sub = a.sub ? a.sub : o.min_seed_len * o.a;
    if (a.csub > sub) sub = a.csub;
    if (sub >= a.score) return 0;
    const int l = a.qe - a.qb > a.re - a.rb ? a.qe - a.qb : (int)(a.re - a.rb);
    const double identity = 1. - (double)(l * o.a - a.score) / (o.a + o.b) / l;
    int mapq;
    if (a.score == 0) mapq = 0;
    else {
        double tmp = T.mapq_l[l < kMapqTabLen ? l : kMapqTabLen - 1];
        tmp *= identity * identity;
        mapq = (int)(6.02 * (a.score - sub) / o.a * tmp * tmp + .499);
    }
    if (a.sub_n > 0) mapq -= T.subn[a.sub_n < kSubnTabLen ? a.sub_n : kSubnTabLen - 1];
    if (mapq > 60) mapq = 60;
    if (mapq < 0) mapq = 0;
    return mapq;
}

__device__ __forceinline__ int raw_mapq(int diff, int a) { return (int)(6.02 * diff / a + .499); }

struct P128 { uint64_t x, y; };
__device__ __forceinline__ bool p128_gt(const P128 &a, const P128 &b) { return a.x > b.x || (a.x == b.x && a.y > b.y); }

// mem_pair.  Instead of materialising and sorting every candidate pair, keep the best two by (score, hash)
// and count the near-best ones in a second pass over the same enumeration.
__device__ int pair_up(const IndexView &V, const qm_opt &o, const PairTables &T, int model, qm_reg *const a[2], const int n_pri[2],
                       uint64_t id, int *sub, int *n_sub, int z[2])
{
    const qm_pestat *pes = T.pes + 4 * model;
    const int64_t *toff = T.term_off + 4 * model;
    P128 v[2 * QM_MAX_REGS];
    int nv = 0;
    const int64_t l_pac = V.l_pac;
    for (int r = 0; r < 2; ++r)
        for (int i = 0; i < n_pri[r]; ++i) {
            const qm_reg &e = a[r][i];
            const uint64_t fx = e.rb < l_pac ? (uint64_t)e.rb : (uint64_t)((l_pac << 1) - 1 - e.rb);
            v[nv].x = (uint64_t)e.rid << 32 | (fx - (uint64_t)V.off[e.rid]);
            v[nv].y = (uint64_t)e.score << 32 | (uint64_t)(i << 2) | (uint64_t)((e.rb >= l_pac) << 1) | (uint64_t)r;
            ++nv;
        }
    for (int i = 1; i < nv; ++i) { const P128 t = v[i]; int j = i - 1; while (j >= 0 && p128_gt(v[j], t)) { v[j + 1] = v[j]; --j; } v[j + 1] = t; }
    int tmp = o.a + o.b;
    if (o.o_del + o.e_del > tmp) tmp = o.o_del + o.e_del;
    if (o.o_ins + o.e_ins > tmp) tmp = o.o_ins + o.e_ins;
    P128 best = {0, 0}, second = {0, 0};
    int nu = 0, ret = 0;
    *n_sub = 0; *sub = 0;
    for (int pass = 0; pass < 2; ++pass) {
        int y[4] = {-1, -1, -1, -1};
        for (int i = 0; i < nv; ++i) {
            for (int r = 0; r < 2; ++r) {
                const int dir = r << 1 | (int)(v[i].y >> 1 & 1);
                if (pes[dir].failed) continue;
                const int which = r << 1 | ((int)(v[i].y & 1) ^ 1);
                if (y[which] < 0) continue;
                for (int k = y[which]; k >= 0; --k) {
                    if ((int)(v[k].y & 3) != which) continue;
                    const int64_t dist = (int64_t)v[i].x - (int64_t)v[k].x;
                    if (dist > pes[dir].high) break;
                    if (dist < pes[dir].low) continue;
                    const double term = T.term[toff[dir] + (dist - pes[dir].low)];
                    int q = (int)((double)((v[i].y >> 32) + (v[k].y >> 32)) + term + .499);
                    if (q < 0) q = 0;
                    P128 u;
                    u.y = (uint64_t)k << 32 | (uint64_t)i;
                    u.x = (uint64_t)q << 32 | (hash64(u.y ^ id << 8) & 0xffffffffU);
                    if (pass == 0) {
                        ++nu;
                        if (nu == 1 || p128_gt(u, best)) { second = best; best = u; if (nu == 1) second = u; }
                        else if (nu == 2 || p128_gt(u, second)) second = u;
                    } else if (!(u.x == best.x && u.y == best.y)) {
                        if (*sub - (int)(u.x >> 32) <= tmp) ++*n_sub;
                    }
                }
            }
            y[v[i].y & 3] = i;
        }
        if (pass == 0) {
            if (nu == 0) return 0;
            const int i = (int)(best.y >> 32), k = (int)(best.y << 32 >> 32);
            z[v[i].y & 1] = (int)(v[i].y << 32 >> 34);
            z[v[k].y & 1] = (int)(v[k].y << 32 >> 34);
            ret = (int)(best.x >> 32);
            *sub = nu > 1 ? (int)(second.x >> 32) : 0;
            if (nu == 1) break;
        }
    }
    return ret;
}

__device__ __forceinline__ int infer_bw(int l1, int l2, int score, int a, int q, int r)
{
    if (l1 == l2 && l1 * a - score < (q + r - a) << 1) return 0;
    int w = (int)(((double)((l1 < l2 ? l1 : l2) * a - score - q) / r + 2.));
    if (w < abs(l1 - l2)) w = abs(l1 - l2);
    return w;
}

#define QM_NEG_INF (-0x40000000)
#define QM_NEVER   (-0x7ff00000)           // below every value the DP can produce, still safe to subtract from

struct Lut { unsigned lo, hi; };        // 8 score bytes: entries 0..3 = query A,C,G,T, entry 4 = query N
// PTX prmt (default mode): selector nibble bit 3 replicates the sign of the selected byte -> sign-extended score
__device__ __forceinline__ int lut_score(const Lut &L, unsigned sel)
{
    int r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(L.lo), "r"(L.hi), "r"(sel));
    return r;
}

struct SeqPair {            // query / reference bases of one CIGAR task, reversed on the reverse strand
    const uint8_t *q;
    int lq, rlen;
    int64_t rb;
    bool rev;
    const IndexView *V;
    __device__ __forceinline__ int qb(int i) const { return rev ? q[lq - 1 - i] : q[i]; }
    __device__ __forceinline__ int tb(int i) const { return qm_ref_base(*V, rev ? rb + rlen - 1 - i : rb + i); }
};

// a read whose CIGAR needs the banded global DP (everything else is finished by pair_decide_kernel)
struct CigTask {
    int64_t rb, re;
    int32_t read, w2, truesc, regw;
    int32_t wcap, pad;          // equal lengths: no diagonal further than wcap from the main one can hold a better path (cig_gain_cap)
};

// Equal-length tasks: how far from the main diagonal can a path that beats the UNGAPPED alignment stray?
// Such a path has as many inserted query bases as deleted reference bases, >= 1 of each; reaching diagonal d costs at least
// (o_ins + o_del) + (e_ins + e_del) |d|.  All it can win back sits at the n_low main-diagonal positions that score below a
// (mismatch or N): at most a + max(b, 1) each, and one inserted query base is not aligned at all (it gives up a match, or
// wins only b): total gain <= (a + max(b,1)) n_low - a - gap cost.  The largest |d| that leaves the gain positive is
// returned (0: the ungapped alignment is optimal in every band).  ksw_global2 run with band min(w, cap) therefore equals
// the ungapped score exactly when it does with any wider band -- and then its traceback is all-M (ties choose M).
__device__ __forceinline__ int cig_gain_cap(const qm_opt &o, int n_low)
{
    const int mb = o.b > 1 ? o.b : 1;
    const int x = (o.a + mb) * n_low - o.a - o.o_ins - o.o_del, es = o.e_ins + o.e_del;
    if (x <= es) return 0;
    return (x - 1) / es;
}

// band of the first try, exactly as bwa_gen_cigar2 derives it from w2
__device__ __forceinline__ int cig_band(const qm_opt &o, int w2, int lq, int rlen)
{
    if (w2 > o.w << 2) w2 = o.w << 2;
    int max_ins = (int)((double)(((lq + 1) >> 1) * o.a - o.o_ins) / o.e_ins + 1.);
    int max_del = (int)((double)(((lq + 1) >> 1) * o.a - o.o_del) / o.e_del + 1.);
    int max_gap = max_ins > max_del ? max_ins : max_del;
    if (max_gap < 1) max_gap = 1;
    int w = (max_gap + abs(rlen - lq) + 1) >> 1;
    if (w > w2) w = w2;
    const int min_w = abs(rlen - lq) + 3;
    return w < min_w ? min_w : w;
}
// The thread-per-task kernels keep eh[] in 16 bits with -20000 as minus infinity.  That orders like the reference's -2^30 only
// while every real DP value stays well above -20000 and minus infinity less one cell's penalties stays above -32768.  Every
// in-band cell (i, j) is reached by at most min(lq, rlen) diagonal steps and one gap of |i - j|, so no real H, E or F is below
// -(max(b, 1) min(lq, rlen) + the longest gap + one gap opening).  With the default scores that is about -3,100 for 512 bases;
// large penalties (b = 100, gaps 100 + 60 k on a 400-base read: below -24,000) break it, and such tasks go to the warp kernel,
// whose cells are 32-bit.  kCig16Bound leaves room on both sides: NEG16 + a stays below every real value and NEG16 - (b + gap
// opening) above -32768.
constexpr int kCig16Bound = 12000;
__device__ __forceinline__ bool cig_fits16(const qm_opt &o, int lq, int rlen)
{
    const int64_t mb = o.b > 1 ? o.b : 1;
    const int64_t gd = o.o_del + (int64_t)o.e_del * rlen, gi = o.o_ins + (int64_t)o.e_ins * lq;
    const int64_t oe = o.o_del + o.e_del > o.o_ins + o.e_ins ? o.o_del + o.e_del : o.o_ins + o.e_ins;
    return mb * (lq < rlen ? lq : rlen) + (gd > gi ? gd : gi) + oe <= kCig16Bound;
}

// which kernel takes a CIGAR task first: 0 / 1 / 2 = score-only thread-per-task pass with 32 / 48 / 72 circular slots
// (equal lengths, band <= 15 / 23 / 35 -- 35 is the most bwa_gen_cigar2 allows for equal lengths up to 140 bp),
// 3 / 4 / 5 = thread-per-task pass with traceback and 32 / 64 / 128 slots (length difference, band <= 15 / 31 / 63),
// 6 = the warp-per-task kernel with traceback (also every task whose DP values 16-bit cells cannot hold: cig_fits16)
__device__ __forceinline__ int cig_class(const IndexView &V, const qm_opt &o, const CigTask &t, int lq)
{
    const int rlen = (int)(t.re - t.rb);
    if ((t.rb < V.l_pac && t.re > V.l_pac) || !cig_fits16(o, lq, rlen)) return 6;
    int w = cig_band(o, t.w2, lq, rlen);
    if (lq != rlen) return w <= 15 ? 3 : w <= 31 ? 4 : w <= 63 ? 5 : 6;     // traceback needed: thread-per-task kernels by band, else warp
    w = w < t.wcap ? w : t.wcap;            // the score-only pass may narrow its band (cig_gain_cap)
    return w <= 15 ? 0 : w <= 23 ? 1 : w <= 35 ? 2 : 6;
}

constexpr int kCigWarps = 4;                  // warps per block of the CIGAR kernel
constexpr int kDirBytes = 14 * 1024;          // shared-memory direction matrix per warp; larger ones go to global memory
constexpr size_t kOverflowPerWarp = 1u << 20; // global fallback per warp: covers tlen x ncol up to 1 MiB

// ksw_global2 (SURVEY.md A.4) by one warp: column j lives in lane j%32, slot j/32.  E is column-local; the F
// recurrence opens from m only, so inside a 32-column slot it is a max-plus prefix scan with a carry between slots.
// dir: one byte per (row, column - beg(row)), exactly the reference's z[] (bits 0-1 H source, bit 2 E extends,
// bits 4-5 F extends).  Returns H(tlen-1, qlen-1).
template <int C>
__device__ int global_dp_warp(const qm_opt &o, const SeqPair &S, int w, uint8_t *dir, int n_col, int lane)
{
    const unsigned FULL = 0xffffffffu;
    const int qlen = S.lq, tlen = S.rlen;
    const int oe_del = o.o_del + o.e_del, oe_ins = o.o_ins + o.e_ins;
    int Hp[C], E[C], qc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const int j = c * 32 + lane;
        Hp[c] = (j < w && j < qlen) ? -(o.o_ins + o.e_ins * (j + 1)) : QM_NEG_INF;      // H(-1, j) = eh[j+1].h
        E[c] = QM_NEG_INF;
        qc[c] = j < qlen ? S.qb(j) : 4;
    }
    int tb_next = tlen > 0 ? S.tb(0) : 0;
    for (int i = 0; i < tlen; ++i) {
        const int tb = tb_next;
        if (i + 1 < tlen) tb_next = S.tb(i + 1);
        const int beg = i > w ? i - w : 0;
        const int end = i + w + 1 < qlen ? i + w + 1 : qlen;
        uint8_t *drow = dir + (size_t)i * n_col - beg;
        int carry = QM_NEG_INF;                      // F at the first cell of the row
        int prev31 = i == 0 ? 0 : -(o.o_del + o.e_del * i);     // H(i-1, -1); only read when beg == 0
        if (beg > 0) prev31 = QM_NEG_INF;
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const int o31 = __shfl_sync(FULL, Hp[c], 31);        // H(i-1, 32c+31) before this row overwrites it
            const int lo = c * 32;
            if (lo + 32 <= beg || lo >= end) { prev31 = o31; continue; }       // warp-uniform
            const int j = lo + lane;
            const bool act = j >= beg && j < end;
            int diag = __shfl_up_sync(FULL, Hp[c], 1);
            if (lane == 0) diag = prev31;
            prev31 = o31;
            const int s = (tb > 3 || qc[c] > 3) ? -1 : (tb == qc[c] ? o.a : -o.b);
            const int m = diag + s;
            // F: inclusive max-plus scan of the openings g = m - oe_ins over the active lanes
            int x = act ? m - oe_ins : QM_NEVER;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int y = __shfl_up_sync(FULL, x, d);
                if (lane >= d) x = max(x, y - d * o.e_ins);
            }
            int sprev = __shfl_up_sync(FULL, x, 1);              // scan value of the lane to the left
            const int la = beg > lo ? beg - lo : 0;              // first active lane of this slot
            if (lane <= la) sprev = QM_NEVER;
            const int f = max(carry - (lane - la) * o.e_ins, sprev);
            // the cell, in the reference's operation order
            int e = E[c];
            uint8_t d = m >= e ? 0 : 1;
            int h = m >= e ? m : e;
            d = h >= f ? d : 2;
            h = h >= f ? h : f;
            int t = m - oe_del;
            e -= o.e_del;
            if (e > t) d |= 1 << 2; else e = t;
            t = m - oe_ins;
            const int f2 = f - o.e_ins;
            if (f2 > t) d |= 2 << 4;
            if (act) { E[c] = e; Hp[c] = h; drow[j] = d; }
            // F entering the next slot = f after the last cell of this one
            carry = __shfl_sync(FULL, f2 > t ? f2 : t, 31);
        }
    }
    const int jl = qlen - 1;
    int score = QM_NEG_INF;
#pragma unroll
    for (int c = 0; c < C; ++c)
        if ((jl >> 5) == c) score = __shfl_sync(FULL, Hp[c], jl & 31);
    return score;
}

// bwa_gen_cigar2's DP branch + traceback + NM for one task; all lanes return the same values
__device__ int gen_cigar_warp(const IndexView &V, const qm_opt &o, int w_, int l_query, const uint8_t *query, int64_t rb, int64_t re,
                              uint8_t *dir_smem, uint8_t *dir_glob, int lane, int *n_cigar_out, uint32_t *cigar /* shared, per warp */,
                              int *nm_out, int *err)
{
    const unsigned FULL = 0xffffffffu;
    const int rlen = (int)(re - rb);
    SeqPair S;
    S.q = query; S.lq = l_query; S.rlen = rlen; S.rb = rb; S.rev = rb >= V.l_pac; S.V = &V;
    int max_ins = (int)((double)(((l_query + 1) >> 1) * o.a - o.o_ins) / o.e_ins + 1.);
    int max_del = (int)((double)(((l_query + 1) >> 1) * o.a - o.o_del) / o.e_del + 1.);
    int max_gap = max_ins > max_del ? max_ins : max_del;
    if (max_gap < 1) max_gap = 1;
    int w = (max_gap + abs(rlen - l_query) + 1) >> 1;
    if (w > w_) w = w_;
    const int min_w = abs(rlen - l_query) + 3;
    if (w < min_w) w = min_w;
    const int n_col = l_query < 2 * w + 1 ? l_query : 2 * w + 1;
    const size_t need = (size_t)n_col * rlen;
    uint8_t *dir = dir_smem;
    if (need > (size_t)kDirBytes) {
        if (need > kOverflowPerWarp) { if (lane == 0) atomicExch(err, 3); *n_cigar_out = -1; *nm_out = -1; return 0; }
        dir = dir_glob;
    }
    int score;
    if (l_query <= 160) score = global_dp_warp<5>(o, S, w, dir, n_col, lane);
    else if (l_query <= 256) score = global_dp_warp<8>(o, S, w, dir, n_col, lane);
    else if (l_query <= 512) score = global_dp_warp<16>(o, S, w, dir, n_col, lane);
    else { if (lane == 0) atomicExch(err, 2); *n_cigar_out = -1; *nm_out = -1; return 0; }
    __syncwarp();
    // traceback (lane 0), CIGAR built back to front then reversed
    int n = 0;
    if (lane == 0) {
        const int max_cigar = QM_MAX_CIGAR - 2;
        int state = 0, i = rlen - 1, k = (i + w + 1 < l_query ? i + w + 1 : l_query) - 1;
        bool overflow = false;
        uint32_t cur = 0;                            // run being built: len << 4 | op ; 0 = none
        while (i >= 0 && k >= 0) {
            const int lo = i > w ? i - w : 0;
            state = dir[(size_t)i * n_col + (k - lo)] >> (state << 1) & 3;
            const uint32_t op = state == 0 ? 0u : (state == 1 ? 2u : 1u);
            if (cur && (cur & 0xf) == op) cur += 1u << 4;
            else {
                if (cur) { if (n < max_cigar) cigar[n++] = cur; else overflow = true; }
                cur = 1u << 4 | op;
            }
            if (state == 0) { --i; --k; } else if (state == 1) --i; else --k;
        }
        auto push = [&](uint32_t op, int len) {
            if (cur && (cur & 0xf) == op) cur += (uint32_t)len << 4;
            else {
                if (cur) { if (n < max_cigar) cigar[n++] = cur; else overflow = true; }
                cur = (uint32_t)len << 4 | op;
            }
        };
        if (i >= 0) push(2, i + 1);
        if (k >= 0) push(1, k + 1);
        if (cur) { if (n < max_cigar) cigar[n++] = cur; else overflow = true; }
        for (int a = 0; a < n >> 1; ++a) { const uint32_t t = cigar[a]; cigar[a] = cigar[n - 1 - a]; cigar[n - 1 - a] = t; }
        if (overflow) n = -1;
    }
    n = __shfl_sync(FULL, n, 0);
    __syncwarp();
    *n_cigar_out = n;
    int nm = -1;
    if (n > 0) {
        int x = 0, y = 0, n_mm = 0, n_gap = 0;
        for (int k = 0; k < n; ++k) {
            const int op = cigar[k] & 0xf, len = (int)(cigar[k] >> 4);
            if (op == 0) { for (int a = lane; a < len; a += 32) if (S.qb(x + a) != S.tb(y + a)) ++n_mm; x += len; y += len; }
            else if (op == 2) { if (k > 0 && k < n - 1) n_gap += len; y += len; }
            else if (op == 1) { x += len; n_gap += len; }
        }
        nm = __reduce_add_sync(FULL, n_mm) + n_gap;
    }
    *nm_out = nm;
    return score;
}

// Mismatches of an ungapped alignment, four bases per step: query bases q[0 .. lq) against the reference interval that
// starts at rb in bwa's doubled coordinates (reverse strand: the query runs backwards against the complemented forward
// strand).  One thread walks one read, so byte loads cost a 32-byte sector per lane and base; aligned words (only words that
// hold a needed byte are touched) cost a quarter of the requests.  n_low also counts a query N that meets a reference N.
__device__ void count_mismatches(const IndexView &V, const uint8_t *q, int lq, int64_t rb, bool rev, int *n_mm, int *n_low)
{
    const uint8_t *rp = V.refb + (rev ? 2 * V.l_pac - rb - lq : rb);          // forward-strand bases, ascending
    int i = 0, mm = 0, low = 0;
    if (lq >= 4) {
        const uint32_t *rw = (const uint32_t *)((uintptr_t)rp & ~(uintptr_t)3);
        const unsigned rsh = (unsigned)((uintptr_t)rp & 3u) * 8u;
        uint32_t rcur = __ldg(rw);
        const uint8_t *qa = rev ? q + lq - 4 : q;                             // the first group's lowest address
        const uint32_t *qw = (const uint32_t *)((uintptr_t)qa & ~(uintptr_t)3);
        const unsigned qsh = (unsigned)((uintptr_t)qa & 3u) * 8u;
        uint32_t qlo = *qw, qhi = (rev && qsh) ? qw[1] : 0;
        for (; i + 4 <= lq; i += 4) {
            const bool more = i + 8 <= lq;
            uint32_t r4, q4;
            if (rsh) { const uint32_t nx = __ldg(++rw); r4 = __funnelshift_r(rcur, nx, rsh); rcur = nx; }
            else { r4 = rcur; if (more) rcur = __ldg(++rw); }
            if (!rev) {
                if (qsh) { const uint32_t nx = *++qw; q4 = __funnelshift_r(qlo, nx, qsh); qlo = nx; }
                else { q4 = qlo; if (more) qlo = *++qw; }
            } else {                                                          // descending addresses: this group's low word is the next one's high word
                q4 = __byte_perm(qsh ? __funnelshift_r(qlo, qhi, qsh) : qlo, 0, 0x0123);
                r4 ^= 0x03030303u;                                            // complement; a reference N (4) becomes 7 and matches nothing
                qhi = qlo;
                if (more) qlo = *--qw;
            }
            const uint32_t ne = __vcmpne4(q4, r4), big = __vcmpgtu4(q4, 0x03030303u);
            mm += __popc(ne) >> 3; low += __popc(ne | big) >> 3;
        }
    }
    for (; i < lq; ++i) {
        const int qc = rev ? q[lq - 1 - i] : q[i], tc = rev ? 3 - rp[i] : rp[i];
        mm += qc != tc; low += (qc != tc) | (qc > 3);
    }
    *n_mm = mm; *n_low = low;
}

// mem_reg2aln, first half: MAPQ / flags / band inference; reads on the no-DP path (equal lengths, w2 == 0) are
// completed here, the others become CigTasks.  Returns true when a task is needed.
__device__ bool reg_to_aln_prepare(const IndexView &V, const qm_opt &o, const PairTables &T, int l_query, const uint8_t *query,
                                   const qm_reg *ar, qm_aln *a, int *w2_out, int *wcap_out)
{
    qm_aln r = {};
    if (ar == nullptr || ar->rb < 0 || ar->re < 0) { r.rid = -1; r.pos = -1; r.flag |= 0x4; *a = r; return false; }
    const int qb = ar->qb, qe = ar->qe;
    const int64_t rb = ar->rb, re = ar->re;
    r.mapq = ar->secondary < 0 ? (uint8_t)approx_mapq(o, T, *ar) : 0;
    if (ar->secondary >= 0) r.flag |= 0x100;
    int tmp = infer_bw(qe - qb, (int)(re - rb), ar->truesc, o.a, o.o_del, o.e_del);
    int w2 = infer_bw(qe - qb, (int)(re - rb), ar->truesc, o.a, o.o_ins, o.e_ins);
    if (tmp > w2) w2 = tmp;
    if (w2 > o.w) w2 = w2 < ar->w ? w2 : ar->w;
    r.score = ar->score; r.sub = ar->sub > ar->csub ? ar->sub : ar->csub;
    r.qb = qb; r.qe = qe;
    const bool is_rev = rb >= V.l_pac;            // a region never straddles l_pac
    if (is_rev) r.flag |= 0x10;
    *wcap_out = 1 << 20;
    if (qe - qb == (int)(re - rb) && !(rb < V.l_pac && re > V.l_pac)) {
        int n_mm = 0, n_low = 0;                  // q != t (NM); positions scoring below a (mismatch, or N on either side)
        count_mismatches(V, query + qb, qe - qb, rb, is_rev, &n_mm, &n_low);
        const int cap = cig_gain_cap(o, n_low);
        if (w2 == 0 || cap == 0) {
            // bwa_gen_cigar2's shortcut (w2 == 0), or no gapped path can beat the ungapped one in any band (cig_gain_cap):
            // <len>M, NM = mismatches
            r.nm = n_mm;
            const int64_t pos = rb < V.l_pac ? rb : 2 * V.l_pac - 1 - (re - 1);
            int m = 0;
            const int clip5 = is_rev ? l_query - qe : qb, clip3 = is_rev ? qb : l_query - qe;
            if (clip5) r.cigar[m++] = (uint32_t)clip5 << 4 | 4;
            r.cigar[m++] = (uint32_t)(qe - qb) << 4;
            if (clip3) r.cigar[m++] = (uint32_t)clip3 << 4 | 4;
            r.n_cigar = (uint8_t)m;
            r.rid = qm_pos2rid(V, pos);
            r.pos = (int32_t)(pos - V.off[r.rid]);
            *a = r;
            return false;
        }
        *wcap_out = cap;
    }
    r.rid = ar->rid; r.pos = -1; r.n_cigar = 0;
    *a = r;
    *w2_out = w2;
    return true;
}

__device__ __forceinline__ int cigar_rlen(const qm_aln &a)
{
    int l = 0;
    if (a.n_cigar == 255) return 0;
    for (int k = 0; k < a.n_cigar; ++k) { const int op = a.cigar[k] & 0xf; if (op == 0 || op == 2) l += a.cigar[k] >> 4; }
    return l;
}

// flags / mate fields as bwamem.c mem_aln2sam writes them
__device__ void finish_pair(qm_aln *h0, qm_aln *h1, int extra_flag)
{
    qm_aln *const h[2] = { h0, h1 };
    const bool mapped[2] = { h0->rid >= 0, h1->rid >= 0 };
    const bool rev[2] = { (h0->flag & 0x10) != 0, (h1->flag & 0x10) != 0 };
    const int rlen[2] = { cigar_rlen(*h0), cigar_rlen(*h1) };
    const int32_t pos0[2] = { h0->pos, h1->pos };
    const int32_t rid0[2] = { h0->rid, h1->rid };
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        qm_aln *p = h[i];
        const int j = !i;
        p->flag |= 0x1 | (i == 0 ? 0x40 : 0x80) | extra_flag;
        if (!mapped[j]) p->flag |= 0x8;
        if (mapped[j] && rev[j]) p->flag |= 0x20;
        if (!mapped[i] && mapped[j]) { p->rid = rid0[j]; p->pos = pos0[j]; if (rev[j]) p->flag |= 0x10; }
        if (!mapped[i] && !mapped[j]) { p->mate_rid = -1; p->mate_pos = -1; p->tlen = 0; continue; }
        if (mapped[j]) { p->mate_rid = rid0[j]; p->mate_pos = pos0[j]; }
        else { p->mate_rid = rid0[i]; p->mate_pos = pos0[i]; if (rev[i]) p->flag |= 0x20; }
        p->tlen = 0;
        if (mapped[0] && mapped[1] && rid0[0] == rid0[1]) {
            const int64_t p0 = pos0[i] + (rev[i] ? rlen[i] - 1 : 0);
            const int64_t p1 = pos0[j] + (rev[j] ? rlen[j] - 1 : 0);
            p->tlen = (int32_t)(-(p0 - p1 + (p0 > p1 ? 1 : p0 < p1 ? -1 : 0)));
        }
    }
}

// ---- kernel 1 (one thread per pair): primary marking, pairing, MAPQ, no-DP CIGARs, task list ----
// The proper-pair bit (2) and "pairing decided" (4) travel to kernel 3 in the not yet final tlen field of mate 1.
__global__ void __launch_bounds__(128)
pair_decide_kernel(IndexView V, qm_opt o, PairTables T, const uint8_t *__restrict__ codes, int stride,
                   const int32_t *__restrict__ lens, int64_t n_pairs, int64_t pair_id0, qm_reg *__restrict__ regs,
                   int32_t *__restrict__ n_regs, qm_aln *__restrict__ alns, CigTask *__restrict__ tasks, int *__restrict__ n_tasks,
                   int *__restrict__ lists /* [4][list_stride] */, int64_t list_stride, int *__restrict__ n_list /* [4] */)
{
    const int64_t pi = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (pi >= n_pairs) return;
    qm_reg *a[2] = { regs + (2 * pi) * QM_MAX_REGS, regs + (2 * pi + 1) * QM_MAX_REGS };
    const int n[2] = { n_regs[2 * pi], n_regs[2 * pi + 1] };
    int n_pri[2], z[2] = {0, 0};
    const uint8_t *seq[2] = { codes + (2 * pi) * stride, codes + (2 * pi + 1) * stride };
    const int l_seq[2] = { lens[2 * pi], lens[2 * pi + 1] };
    const uint64_t id = (uint64_t)(pair_id0 + pi);
    int extra_flag = 0, o_sc = 0, subo = 0, n_sub = 0;
    bool paired_done = false;
    const qm_reg *chosen[2] = { nullptr, nullptr };
    int q_se[2] = {0, 0};
    mark_primary(o, n[0], a[0], id << 1 | 0);
    mark_primary(o, n[1], a[1], id << 1 | 1);
    n_pri[0] = n[0]; n_pri[1] = n[1];
    if (n_pri[0] && n_pri[1] && (o_sc = pair_up(V, o, T, pair_model(T, pi), a, n_pri, id, &subo, &n_sub, z)) > 0) {
        bool is_multi[2];
        for (int i = 0; i < 2; ++i) {
            int j;
            for (j = 1; j < n_pri[i]; ++j) if (a[i][j].secondary < 0 && a[i][j].score >= o.T) break;
            is_multi[i] = j < n_pri[i];
        }
        if (!(is_multi[0] || is_multi[1])) {
            const int score_un = a[0][0].score + a[1][0].score - o.pen_unpaired;
            if (score_un > subo) subo = score_un;
            int q_pe = raw_mapq(o_sc - subo, o.a);
            if (n_sub > 0) q_pe -= T.subn[n_sub < kSubnTabLen ? n_sub : kSubnTabLen - 1];
            if (q_pe < 0) q_pe = 0;
            if (q_pe > 60) q_pe = 60;
            if (o_sc > score_un) {
                qm_reg *c[2] = { &a[0][z[0]], &a[1][z[1]] };
                for (int i = 0; i < 2; ++i) {
                    if (c[i]->secondary >= 0) { c[i]->sub = a[i][c[i]->secondary].score; c[i]->secondary = -2; }
                    q_se[i] = approx_mapq(o, T, *c[i]);
                }
                for (int i = 0; i < 2; ++i) {
                    q_se[i] = q_se[i] > q_pe ? q_se[i] : q_pe < q_se[i] + 40 ? q_pe : q_se[i] + 40;
                    const int cap = raw_mapq(c[i]->score - c[i]->csub, o.a);
                    if (q_se[i] > cap) q_se[i] = cap;
                }
                extra_flag |= 2;
            } else {
                z[0] = z[1] = 0;
                q_se[0] = approx_mapq(o, T, a[0][0]);
                q_se[1] = approx_mapq(o, T, a[1][0]);
            }
            chosen[0] = &a[0][z[0]]; chosen[1] = &a[1][z[1]];
            paired_done = true;
        }
    }
    if (!paired_done) {
        for (int i = 0; i < 2; ++i) chosen[i] = (n[i] && a[i][0].score >= o.T) ? &a[i][0] : nullptr;
        // (the proper-pair test of this branch needs the final records: kernel 3)
    }
    for (int i = 0; i < 2; ++i) {
        qm_aln h;
        int w2 = 0, wcap = 0;
        const bool need = reg_to_aln_prepare(V, o, T, l_seq[i], seq[i], chosen[i], &h, &w2, &wcap);
        if (paired_done) { h.mapq = (uint8_t)q_se[i]; h.flag &= ~0x100; }
        if (i == 0) h.tlen = extra_flag | (paired_done ? 4 : 0);
        alns[2 * pi + i] = h;
        if (need) {
            CigTask t;
            t.rb = chosen[i]->rb; t.re = chosen[i]->re; t.read = (int32_t)(2 * pi + i); t.w2 = w2;
            t.truesc = chosen[i]->truesc; t.regw = chosen[i]->w; t.wcap = wcap; t.pad = 0;
            const int slot = atomicAdd(n_tasks, 1);
            tasks[slot] = t;
            const int c = cig_class(V, o, t, h.qe - h.qb);
            lists[c * list_stride + atomicAdd(&n_list[c], 1)] = slot;
        }
    }
}

// ---- kernel 2a (one THREAD per task): score-only banded global DP for equal-length tasks ----
// If ksw_global2's optimum equals the score of the ungapped alignment, its traceback is all-M (every cell on the
// main diagonal then has m == H >= e, f, and ties choose M), so CIGAR = <len>M and NM = mismatches: no direction
// matrix, no traceback.  This kernel runs the reference's row/column loop verbatim (no direction bits) with the
// band of eh[] in a circular shared-memory buffer, one task per thread, and finishes every task whose first try
// is final (score >= truesc - a, bwa's retry rule) and gap-free.  Everything else (length difference, wide band,
// retry, real gaps) is left to the warp-per-task kernel with traceback.
constexpr int kCsT = 128;              // threads per block

template <int B>                       // circular slots per thread, needs 2w + 2 <= B
__global__ void __launch_bounds__(kCsT)
cig_score_kernel(IndexView V, qm_opt o, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
                 const CigTask *__restrict__ tasks, const int *__restrict__ mine, const int *__restrict__ n_mine,
                 qm_aln *__restrict__ alns, int *__restrict__ left, int *__restrict__ n_left)
{
    // eh[] in 16 bits (see cig_trace_kernel: -20000 orders like the reference's -2^30); slots (2s, 2s+1) of a thread share
    // one 32-bit word, so lane t always hits bank t
    extern __shared__ short cs_smem[];
    constexpr int NEG16 = -20000;
    short *HS = cs_smem + 2 * threadIdx.x;                     // HS[CX(slot)]  eh[].h
    short *ES = HS + B * kCsT;                                 // ES[CX(slot)]  eh[].e
    unsigned short *SS = (unsigned short *)(HS + 2 * B * kCsT);   // PRMT selector of q[j]
#define CX(sl) ((((sl) >> 1) * (2 * kCsT)) + ((sl) & 1))
    const int n = *n_mine;
    const int oe_del = o.o_del + o.e_del, oe_ins = o.o_ins + o.e_ins;
    for (int li = blockIdx.x * kCsT + threadIdx.x; li < n; li += gridDim.x * kCsT) {
        const int ti = mine[li];
        const CigTask t = tasks[ti];
        qm_aln *rec = alns + t.read;
        const int l_query = lens[t.read];
        const int qb = rec->qb, qe = rec->qe;
        const int lq = qe - qb, rlen = (int)(t.re - t.rb);
        int w = cig_band(o, t.w2, lq, rlen);                // the band pair_decide_kernel classified this task by:
        w = w < t.wcap ? w : t.wcap;                        // bwa's, narrowed to the diagonals a better-than-ungapped path can reach
        SeqPair S;
        S.q = codes + (int64_t)t.read * stride + qb; S.lq = lq; S.rlen = rlen; S.rb = t.rb; S.rev = t.rb >= V.l_pac; S.V = &V;
        // first row of eh[] and the selectors of the columns row 0 can reach
        HS[0] = 0; ES[0] = NEG16;
        for (int j = 1; j <= lq && j <= w; ++j) { HS[CX(j % B)] = (short)-(o.o_ins + o.e_ins * j); ES[CX(j % B)] = NEG16; }
        if (w + 1 <= lq) { HS[CX((w + 1) % B)] = NEG16; ES[CX((w + 1) % B)] = NEG16; }
        for (int j = 0; j < lq && j <= w; ++j) {
            int c = S.qb(j);
            c = c > 4 ? 4 : c;
            SS[CX(j % B)] = (unsigned short)(c * 0x1111 + 0x8880);
        }
        int us = 0, n_mm = 0;                              // ungapped score and mismatches (the main diagonal)
        for (int i = 0; i < rlen; ++i) {
            const int tb = S.tb(i);
            const int beg = i > w ? i - w : 0;
            const int end = i + w + 1 < lq ? i + w + 1 : lq;
            if (i > 0 && i + w < lq) {                     // the column entering the band on the right
                int c = S.qb(i + w);
                c = c > 4 ? 4 : c;
                SS[CX((i + w) % B)] = (unsigned short)(c * 0x1111 + 0x8880);
            }
            Lut L;
            if (tb > 3) { L.lo = 0xffffffffu; L.hi = 0xffffffffu; }
            else {
                const unsigned mis = (unsigned)(-o.b) & 0xffu, mat = (unsigned)o.a & 0xffu;
                unsigned v = mis * 0x01010101u;
                v = (v & ~(0xffu << (8 * tb))) | (mat << (8 * tb));
                L.lo = v; L.hi = 0xffffffffu;
            }
            {   // main-diagonal cell: ungapped score / mismatch bookkeeping
                const unsigned sel = SS[CX(i % B)];
                us += lut_score(L, sel);
                n_mm += (int)(sel & 7u) != tb;
            }
            int f = NEG16;
            int h1 = beg == 0 ? -(o.o_del + o.e_del * (i + 1)) : NEG16;
            int slot = beg % B;                            // slot of column j, advanced with wrap-around
            for (int j = beg; j < end; ++j) {
                const int sl = CX(slot);
                int m = HS[sl], e = ES[sl];
                HS[sl] = (short)h1;
                m += lut_score(L, SS[sl]);
                int h = m >= e ? m : e;
                h = h >= f ? h : f;
                h1 = h;
                int tt = m - oe_del;
                e -= o.e_del;
                e = e > tt ? e : tt;
                ES[sl] = (short)e;
                tt = m - oe_ins;
                f -= o.e_ins;
                f = f > tt ? f : tt;
                if (++slot == B) slot = 0;
            }
            HS[CX(slot)] = (short)h1; ES[CX(slot)] = NEG16;        // slot is now that of column `end` (beg when the row is empty)
        }
        const int score = HS[CX(lq % B)];
        if (score == us) {
            // gap-free in every band (cig_gain_cap), so every retry of mem_reg2aln ends here too: <lq>M with clips
            const bool is_rev = t.rb >= V.l_pac;
            const int64_t pos = t.rb < V.l_pac ? t.rb : 2 * V.l_pac - 1 - (t.re - 1);
            int m = 0;
            const int clip5 = is_rev ? l_query - qe : qb, clip3 = is_rev ? qb : l_query - qe;
            if (clip5) rec->cigar[m++] = (uint32_t)clip5 << 4 | 4;
            rec->cigar[m++] = (uint32_t)lq << 4;
            if (clip3) rec->cigar[m++] = (uint32_t)clip3 << 4 | 4;
            rec->n_cigar = (uint8_t)m;
            const int rid = qm_pos2rid(V, pos);
            rec->rid = rid;
            rec->pos = (int32_t)(pos - V.off[rid]);
            rec->nm = n_mm;
        } else left[atomicAdd(n_left, 1)] = ti;
    }
}
#undef CX

// ---- kernel 2b (one THREAD per task): banded global DP WITH traceback for the tasks the score-only pass could not
// finish (length difference, real gaps).  Same row/column loop plus the reference's direction byte per cell, written
// to a global slab laid out [cell][thread] (a warp's stores for one cell are contiguous); the traceback walks the
// thread's own bytes.  Only the first try is run here: if bwa's retry rule asks for a wider band, or the direction
// matrix does not fit the slab, the task moves on to the warp-per-task kernel. ----
constexpr size_t kTraceCellsPerThread = 32768;      // direction nibbles per thread in the slab (rows x band columns rounded up to 8)

template <int B, int T>                // circular slots (power of two, 2w + 2 <= B), threads per block
__global__ void __launch_bounds__(T)
cig_trace_kernel(IndexView V, qm_opt o, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
                 const CigTask *__restrict__ tasks, const int *__restrict__ mine, const int *__restrict__ n_mine, int wmax,
                 uint8_t *__restrict__ slab, qm_aln *__restrict__ alns, int *__restrict__ next, int *__restrict__ n_next)
{
    // eh[] in 16 bits: cig_class sends a task here only when every real DP value of it is above -kCig16Bound (cig_fits16),
    // so -20000 orders exactly like the reference's -2^30 in every comparison.  Slots (2s, 2s+1) of a thread share one 32-bit word: lane t always hits bank t.
    extern __shared__ short ct_smem[];
    constexpr int NEG16 = -20000;
    short *HS = ct_smem + 2 * threadIdx.x;
    short *ES = HS + B * T;
    unsigned short *SS = (unsigned short *)(HS + 2 * B * T);
#define SX(sl) ((((sl) >> 1) * (2 * T)) + ((sl) & 1))
    // direction nibbles (bits 0-1 source of H, bit 2 E extends, bit 3 F extends), 8 cells per word, each row starting a
    // fresh word, in a slab region of the thread's own: consecutive words of one thread fill whole 32-byte sectors in L2
    // before they are written back (one byte per cell scattered [cell][thread] cost 12 GB of DRAM writes per 2 M pairs)
    uint32_t *dirw = (uint32_t *)slab + ((size_t)blockIdx.x * T + threadIdx.x) * (kTraceCellsPerThread / 8);
    const int n = *n_mine;
    const int oe_del = o.o_del + o.e_del, oe_ins = o.o_ins + o.e_ins;
    for (int li = blockIdx.x * T + threadIdx.x; li < n; li += gridDim.x * T) {
        const int ti = mine[li];
        const CigTask t = tasks[ti];
        qm_aln *rec = alns + t.read;
        const int l_query = lens[t.read];
        const int qb = rec->qb, qe = rec->qe;
        const int lq = qe - qb, rlen = (int)(t.re - t.rb);
        if ((t.rb < V.l_pac && t.re > V.l_pac) || lq <= 0 || rlen <= 0 || lq > 500 || rlen > 1000) { next[atomicAdd(n_next, 1)] = ti; continue; }
        SeqPair S;
        S.q = codes + (int64_t)t.read * stride + qb; S.lq = lq; S.rlen = rlen; S.rb = t.rb; S.rev = t.rb >= V.l_pac; S.V = &V;
        // bwa_gen_cigar2 / mem_reg2aln: first try with the inferred band, doubled (at most twice) while the score stays
        // below truesc - a; the CIGAR is the LAST try's.  A try whose band this kernel cannot hold passes the task on.
        int w2 = t.w2, last_sc = -(1 << 30), it = 0, score = 0, w = 0, n_col = 0, row_words = 0;
        bool pass_on = false;
        for (;;) {
            if (w2 > o.w << 2) w2 = o.w << 2;
            w = cig_band(o, w2, lq, rlen);
            n_col = lq < 2 * w + 1 ? lq : 2 * w + 1;
            row_words = (n_col + 7) >> 3;
            if (w > wmax || (size_t)row_words * rlen > kTraceCellsPerThread / 8) { pass_on = true; break; }
            HS[0] = 0; ES[0] = NEG16;
            for (int j = 1; j <= lq && j <= w; ++j) { HS[SX(j & (B - 1))] = (short)-(o.o_ins + o.e_ins * j); ES[SX(j & (B - 1))] = NEG16; }
            if (w + 1 <= lq) { HS[SX((w + 1) & (B - 1))] = NEG16; ES[SX((w + 1) & (B - 1))] = NEG16; }
            for (int j = 0; j < lq && j <= w; ++j) {
                int c = S.qb(j);
                c = c > 4 ? 4 : c;
                SS[SX(j & (B - 1))] = (unsigned short)(c * 0x1111 + 0x8880);
            }
            for (int i = 0; i < rlen; ++i) {
                const int tb = S.tb(i);
                const int beg = i > w ? i - w : 0;
                const int end = i + w + 1 < lq ? i + w + 1 : lq;
                if (i > 0 && i + w < lq) {
                    int c = S.qb(i + w);
                    c = c > 4 ? 4 : c;
                    SS[SX((i + w) & (B - 1))] = (unsigned short)(c * 0x1111 + 0x8880);
                }
                Lut L;
                if (tb > 3) { L.lo = 0xffffffffu; L.hi = 0xffffffffu; }
                else {
                    const unsigned mis = (unsigned)(-o.b) & 0xffu, mat = (unsigned)o.a & 0xffu;
                    unsigned v = mis * 0x01010101u;
                    v = (v & ~(0xffu << (8 * tb))) | (mat << (8 * tb));
                    L.lo = v; L.hi = 0xffffffffu;
                }
                int f = NEG16;
                int h1 = beg == 0 ? -(o.o_del + o.e_del * (i + 1)) : NEG16;
                uint32_t *drow = dirw + (size_t)i * row_words;
                uint32_t acc = 0;
                int cn = 0;                                     // cells of this row so far
                for (int j = beg; j < end; ++j) {
                    const int sl = SX(j & (B - 1));
                    int m = HS[sl], e = ES[sl];
                    HS[sl] = (short)h1;
                    m += lut_score(L, SS[sl]);
                    uint32_t d = m >= e ? 0u : 1u;
                    int h = m >= e ? m : e;
                    d = h >= f ? d : 2u;
                    h = h >= f ? h : f;
                    h1 = h;
                    int tt = m - oe_del;
                    e -= o.e_del;
                    if (e > tt) d |= 4u; else e = tt;
                    ES[sl] = (short)e;
                    tt = m - oe_ins;
                    f -= o.e_ins;
                    if (f > tt) d |= 8u; else f = tt;
                    acc |= d << (4 * (cn & 7));
                    if ((++cn & 7) == 0) { drow[(cn >> 3) - 1] = acc; acc = 0; }
                }
                if (cn & 7) drow[cn >> 3] = acc;
                const int sl = SX(end & (B - 1));
                HS[sl] = (short)h1; ES[sl] = NEG16;
            }
            score = HS[SX(lq & (B - 1))];
            if (score == last_sc || w2 == o.w << 2) break;
            last_sc = score;
            w2 <<= 1;
            if (!(++it < 3 && score < t.truesc - o.a)) break;
        }
        if (pass_on) { next[atomicAdd(n_next, 1)] = ti; continue; }
        // traceback, CIGAR built back to front
        uint32_t cig[QM_MAX_CIGAR];
        int nc = 0;
        bool overflow = false;
        {
            const int max_cigar = QM_MAX_CIGAR - 2;
            int state = 0, i = rlen - 1, k = (i + w + 1 < lq ? i + w + 1 : lq) - 1;
            uint32_t cur = 0;
            while (i >= 0 && k >= 0) {
                const int lo = i > w ? i - w : 0;
                const uint32_t d = dirw[(size_t)i * row_words + ((k - lo) >> 3)] >> (4 * ((k - lo) & 7));
                state = state == 0 ? (int)(d & 3u) : state == 1 ? (int)((d >> 2) & 1u) : (int)((d >> 3) & 1u) * 2;
                const uint32_t op = state == 0 ? 0u : (state == 1 ? 2u : 1u);
                if (cur && (cur & 0xf) == op) cur += 1u << 4;
                else {
                    if (cur) { if (nc < max_cigar) cig[nc++] = cur; else overflow = true; }
                    cur = 1u << 4 | op;
                }
                if (state == 0) { --i; --k; } else if (state == 1) --i; else --k;
            }
            for (int pass = 0; pass < 2; ++pass) {
                const int len = pass == 0 ? i + 1 : k + 1;
                const uint32_t op = pass == 0 ? 2u : 1u;
                if (len <= 0) continue;
                if (cur && (cur & 0xf) == op) cur += (uint32_t)len << 4;
                else {
                    if (cur) { if (nc < max_cigar) cig[nc++] = cur; else overflow = true; }
                    cur = (uint32_t)len << 4 | op;
                }
            }
            if (cur) { if (nc < max_cigar) cig[nc++] = cur; else overflow = true; }
        }
        if (overflow) {
            rec->rid = -1; rec->pos = -1; rec->flag |= 0x4; rec->flag &= ~0x10; rec->n_cigar = 255; rec->nm = -1;
            rec->score = 0; rec->sub = 0; rec->qb = 0; rec->qe = 0;
            continue;
        }
        // cig[] is in reverse order: operation a of the forward CIGAR is cig[nc - 1 - a]
        int nm = -1;
        if (nc > 0) {
            int x = 0, y = 0, n_mm = 0, n_gap = 0;
            for (int a = 0; a < nc; ++a) {
                const uint32_t c = cig[nc - 1 - a];
                const int op = c & 0xf, len = (int)(c >> 4);
                if (op == 0) { for (int u = 0; u < len; ++u) n_mm += S.qb(x + u) != S.tb(y + u); x += len; y += len; }
                else if (op == 2) { if (a > 0 && a < nc - 1) n_gap += len; y += len; }
                else if (op == 1) { x += len; n_gap += len; }
            }
            nm = n_mm + n_gap;
        }
        const bool is_rev = t.rb >= V.l_pac;
        int64_t pos = t.rb < V.l_pac ? t.rb : 2 * V.l_pac - 1 - (t.re - 1);
        int a0 = 0, a1 = nc;                        // forward-order slice [a0, a1) after squeezing a leading / trailing deletion
        if (nc > 0) {
            if ((cig[nc - 1] & 0xf) == 2) { pos += cig[nc - 1] >> 4; a0 = 1; }
            else if ((cig[0] & 0xf) == 2) a1 = nc - 1;
        }
        int m = 0;
        const int clip5 = is_rev ? l_query - qe : qb, clip3 = is_rev ? qb : l_query - qe;
        if (clip5) rec->cigar[m++] = (uint32_t)clip5 << 4 | 4;
        for (int a = a0; a < a1; ++a) rec->cigar[m++] = cig[nc - 1 - a];
        if (clip3) rec->cigar[m++] = (uint32_t)clip3 << 4 | 4;
        rec->n_cigar = (uint8_t)m;
        const int rid = qm_pos2rid(V, pos);
        rec->rid = rid;
        rec->pos = (int32_t)(pos - V.off[rid]);
        rec->nm = nm;
    }
}
#undef SX

// ---- kernel 2 (one warp per task): banded global DP with traceback, bwa's band-doubling retry, NM, clips ----
__global__ void __launch_bounds__(kCigWarps * 32)
cigar_kernel(IndexView V, qm_opt o, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
             const CigTask *__restrict__ tasks, const int *__restrict__ left, const int *__restrict__ n_left,
             int *__restrict__ cursor, uint8_t *__restrict__ overflow, qm_aln *__restrict__ alns, int *__restrict__ err)
{
    extern __shared__ uint8_t smem[];
    __shared__ uint32_t s_cig[kCigWarps][QM_MAX_CIGAR];
    const int lane = qm_lane(), wib = threadIdx.x >> 5;
    uint8_t *dir_smem = smem + (size_t)wib * kDirBytes;
    uint8_t *dir_glob = overflow + ((size_t)blockIdx.x * kCigWarps + wib) * kOverflowPerWarp;
    const int n = *n_left;
    for (;;) {
        int ti = 0;
        if (lane == 0) ti = atomicAdd(cursor, 1);
        ti = __shfl_sync(0xffffffffu, ti, 0);
        if (ti >= n) break;
        const CigTask t = tasks[left[ti]];
        qm_aln *rec = alns + t.read;
        const int l_query = lens[t.read];
        const int qb = rec->qb, qe = rec->qe;
        const uint8_t *query = codes + (int64_t)t.read * stride + qb;
        int w2 = t.w2, nm = -1, score = 0, last_sc = -(1 << 30), n_cigar = 0;
        int it = 0;
        do {
            if (w2 > o.w << 2) w2 = o.w << 2;
            if (t.rb < V.l_pac && t.re > V.l_pac) { n_cigar = 0; nm = -1; score = 0; }
            else score = gen_cigar_warp(V, o, w2, qe - qb, query, t.rb, t.re, dir_smem, dir_glob, lane, &n_cigar, s_cig[wib], &nm, err);
            if (score == last_sc || w2 == o.w << 2) break;
            last_sc = score;
            w2 <<= 1;
        } while (++it < 3 && score < t.truesc - o.a);
        if (lane == 0) {
            const uint32_t *cig = s_cig[wib];
            if (n_cigar < 0) {       // CIGAR overflow: the read is reported unmapped (mem_reg2aln's fields stay unset)
                rec->rid = -1; rec->pos = -1; rec->flag |= 0x4; rec->flag &= ~0x10; rec->n_cigar = 255; rec->nm = nm;
                rec->score = 0; rec->sub = 0; rec->qb = 0; rec->qe = 0;
            }
            else {
                const bool is_rev = t.rb >= V.l_pac;
                int64_t pos = t.rb < V.l_pac ? t.rb : 2 * V.l_pac - 1 - (t.re - 1);
                int c0 = 0;
                if (n_cigar > 0) {
                    if ((cig[0] & 0xf) == 2) { pos += cig[0] >> 4; c0 = 1; --n_cigar; }
                    else if ((cig[n_cigar - 1] & 0xf) == 2) --n_cigar;
                }
                int m = 0;
                const int clip5 = is_rev ? l_query - qe : qb, clip3 = is_rev ? qb : l_query - qe;
                if (clip5) rec->cigar[m++] = (uint32_t)clip5 << 4 | 4;
                for (int k = 0; k < n_cigar; ++k) rec->cigar[m++] = cig[c0 + k];
                if (clip3) rec->cigar[m++] = (uint32_t)clip3 << 4 | 4;
                rec->n_cigar = (uint8_t)m;
                const int rid = qm_pos2rid(V, pos);
                rec->rid = rid;
                rec->pos = (int32_t)(pos - V.off[rid]);
                rec->nm = nm;
            }
        }
        __syncwarp();
    }
}

// ---- kernel 3 (one thread per pair): proper-pair test of the unpaired branch, SAM flags, mate fields, TLEN ----
// A thread reading and writing its own two 128-byte records straight from global memory costs 32 cache lines per warp
// instruction (measured: 1.06 ms per 2 M pairs, the load/store queue throttled, 1.7 % of the issue slots busy).  The block's
// 256 records are staged in shared memory instead: coalesced word copies in and out, 33 words per record so that the
// threads' accesses to "their" records fall into different banks.
constexpr int kFinT = 128, kAlnWords = (int)(sizeof(qm_aln) / 4), kAlnPad = kAlnWords + 1;
__global__ void __launch_bounds__(kFinT)
pair_finish_kernel(IndexView V, PairTables T, int64_t n_pairs, const qm_reg *__restrict__ regs, qm_aln *__restrict__ alns)
{
    __shared__ uint32_t s_rec[2 * kFinT * kAlnPad];
    const int64_t pair0 = blockIdx.x * (int64_t)kFinT;
    const int64_t n_here = n_pairs - pair0 < kFinT ? n_pairs - pair0 : kFinT;
    const int n_words = (int)(2 * n_here) * kAlnWords;
    uint32_t *g = (uint32_t *)(alns + 2 * pair0);
    for (int w = threadIdx.x; w < n_words; w += kFinT) s_rec[(w / kAlnWords) * kAlnPad + (w % kAlnWords)] = g[w];
    __syncthreads();
    if (threadIdx.x < n_here) {
        const int64_t pi = pair0 + threadIdx.x;
        qm_aln *h0 = (qm_aln *)(s_rec + (2 * threadIdx.x) * kAlnPad), *h1 = (qm_aln *)(s_rec + (2 * threadIdx.x + 1) * kAlnPad);
        int extra_flag = h0->tlen & 2;
        const bool paired_done = (h0->tlen & 4) != 0;
        h0->tlen = 0;
        if (!paired_done && h0->rid == h1->rid && h0->rid >= 0) {
            int64_t dist;
            const int d = qm_infer_dir(V.l_pac, regs[(2 * pi) * QM_MAX_REGS].rb, regs[(2 * pi + 1) * QM_MAX_REGS].rb, &dist);
            const qm_pestat &pe = T.pes[4 * pair_model(T, pi) + d];
            if (!pe.failed && dist >= pe.low && dist <= pe.high) extra_flag |= 2;
        }
        finish_pair(h0, h1, extra_flag);
    }
    __syncthreads();
    for (int w = threadIdx.x; w < n_words; w += kFinT) g[w] = s_rec[(w / kAlnWords) * kAlnPad + (w % kAlnWords)];
}

}  // namespace

extern "C" {

int qm_pestat_sync(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const qm_reg *d_regs, const int32_t *d_n_regs,
                   int64_t n_pairs, qm_pestat pes[4], void *stream)
{
    if (!ctx || !idx || !opt || !pes || n_pairs < 0 || (n_pairs > 0 && (!d_regs || !d_n_regs))) return QM_EINVAL;
    if (opt->max_ins < 1 || opt->max_ins > (1 << 20)) return qm_fail(ctx, QM_ELIMIT, "qm_pestat_sync: max_ins must be in [1, 2^20]");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    // device: one histogram of insert sizes per orientation; host: the percentile / moment arithmetic of
    // mem_pestat replayed over the histogram in ascending order (same operation order as over the sorted list)
    const size_t bins = (size_t)opt->max_ins + 1;
    std::vector<unsigned> h(4 * bins, 0u);
    if (n_pairs > 0) {
        void *p = nullptr;
        int rc = qm_scratch_reserve(ctx, 4, 4 * bins * sizeof(unsigned), &p);
        if (rc) return rc;
        QM_CUDA(ctx, cudaMemsetAsync(p, 0, 4 * bins * sizeof(unsigned), st));
        const int tpb = 128;
        const int sp = qm_prof_begin(ctx, QM_ST_PAIR, st);
        pestat_hist_kernel<<<(unsigned)((n_pairs + tpb - 1) / tpb), tpb, 0, st>>>(idx->v, *opt, d_regs, d_n_regs, 0, n_pairs, nullptr, 0, (unsigned *)p);
        qm_prof_end(ctx, QM_ST_PAIR, sp, st, 1);
        QM_CUDA(ctx, cudaMemcpyAsync(h.data(), p, 4 * bins * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
        QM_CUDA(ctx, cudaStreamSynchronize(st));
    }
    int64_t cnt[4], max = 0;
    for (int d = 0; d < 4; ++d) {
        qm_pestat *r = &pes[d];
        r->low = r->high = r->failed = r->pad = 0; r->avg = r->std = 0;
        const unsigned *q = h.data() + (size_t)d * bins;
        int64_t n = 0;
        for (size_t v = 0; v < bins; ++v) n += q[v];
        cnt[d] = n;
        if (n > max) max = n;
        if (n < 10) { r->failed = 1; continue; }
        auto nth = [&](int64_t k) {       // value at rank k of the ascending list
            int64_t c = 0;
            for (size_t v = 0; v < bins; ++v) { c += q[v]; if (c > k) return (int)v; }
            return (int)bins - 1;
        };
        const int p25 = nth((int)(.25 * n + .499)), p75 = nth((int)(.75 * n + .499));
        r->low = (int)(p25 - 2.0 * (p75 - p25) + .499);
        if (r->low < 1) r->low = 1;
        r->high = (int)(p75 + 2.0 * (p75 - p25) + .499);
        int64_t x = 0;
        for (int64_t v = r->low; v <= r->high && v < (int64_t)bins; ++v) for (unsigned c = 0; c < q[v]; ++c) { r->avg += (double)v; ++x; }
        r->avg /= x;
        for (int64_t v = r->low; v <= r->high && v < (int64_t)bins; ++v) {
            const double dlt = ((double)v - r->avg) * ((double)v - r->avg);
            for (unsigned c = 0; c < q[v]; ++c) r->std += dlt;
        }
        r->std = sqrt(r->std / x);
        r->low = (int)(p25 - 3.0 * (p75 - p25) + .499);
        r->high = (int)(p75 + 3.0 * (p75 - p25) + .499);
        if (r->low > r->avg - 4.0 * r->std) r->low = (int)(r->avg - 4.0 * r->std + .499);
        if (r->high < r->avg + 4.0 * r->std) r->high = (int)(r->avg + 4.0 * r->std + .499);
        if (r->low < 1) r->low = 1;
    }
    for (int d = 0; d < 4; ++d) if (!pes[d].failed && cnt[d] < max * 0.05) pes[d].failed = 1;
    return QM_OK;
}

// Insert-size models of the chunks of a batch (bwa's mem_process_seqs: one mem_pestat per input chunk, over all of the chunk's
// pairs).  Chunk c holds pairs h_start[c] .. h_start[c + 1] - 1.  Leaves the pair -> chunk map and the models on the device
// (scratch 42: *d_model_of, *d_pes, valid until the next call) and the models in h_pes[4 n_chunks]; synchronous.
int qm_pestat_chunks(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const qm_reg *d_regs, const int32_t *d_n_regs,
                     const int64_t *h_start, int n_chunks, const int32_t **d_model_of, const qm_pestat **d_pes, qm_pestat *h_pes, void *stream)
{
    if (!ctx || !idx || !opt || !h_start || n_chunks < 1 || !d_model_of || !d_pes || !h_pes) return QM_EINVAL;
    if (opt->max_ins < 1 || opt->max_ins > (1 << 20)) return qm_fail(ctx, QM_ELIMIT, "qm_pestat_chunks: max_ins must be in [1, 2^20]");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t n_pairs = h_start[n_chunks];
    // scratch 42: chunk starts | pair -> chunk | models
    const size_t o_map = ((size_t)(n_chunks + 1) * 8 + 255) & ~(size_t)255;
    const size_t o_pes = (o_map + (size_t)(n_pairs > 0 ? n_pairs : 1) * 4 + 255) & ~(size_t)255;
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 42, o_pes + (size_t)n_chunks * 4 * sizeof(qm_pestat), &p);
    if (rc) return rc;
    char *b = (char *)p;
    int64_t *starts = (int64_t *)b;
    int32_t *map = (int32_t *)(b + o_map);
    qm_pestat *pes = (qm_pestat *)(b + o_pes);
    QM_CUDA(ctx, cudaMemcpyAsync(starts, h_start, (size_t)(n_chunks + 1) * 8, cudaMemcpyHostToDevice, st));
    const int tpb = 128;
    const int sp = qm_prof_begin(ctx, QM_ST_PAIR, st);
    if (n_pairs > 0) chunk_of_kernel<<<(unsigned)((n_pairs + 255) / 256), 256, 0, st>>>(starts, n_chunks, n_pairs, map);
    // the histograms of up to 256 MB of chunks at a time ([chunk][4][max_ins + 1] counters)
    const size_t per_chunk = (size_t)4 * (opt->max_ins + 1) * sizeof(unsigned);
    const int group = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_chunks, ((size_t)256 << 20) / per_chunk));
    void *h = nullptr;
    rc = qm_scratch_reserve(ctx, 43, (size_t)group * per_chunk, &h);
    if (rc) return rc;
    for (int c0 = 0; c0 < n_chunks; c0 += group) {
        const int c1 = std::min(n_chunks, c0 + group);
        const int64_t p0 = h_start[c0], np = h_start[c1] - h_start[c0];
        QM_CUDA(ctx, cudaMemsetAsync(h, 0, (size_t)(c1 - c0) * per_chunk, st));
        if (np > 0)
            pestat_hist_kernel<<<(unsigned)((np + tpb - 1) / tpb), tpb, 0, st>>>(idx->v, *opt, d_regs, d_n_regs, p0, np, map, c0, (unsigned *)h);
        pestat_model_kernel<<<(unsigned)(c1 - c0), 32, 0, st>>>((const unsigned *)h, opt->max_ins, c0, pes);
    }
    qm_prof_end(ctx, QM_ST_PAIR, sp, st, 1 + 3 * ((n_chunks + group - 1) / group));
    QM_CUDA(ctx, cudaGetLastError());
    QM_CUDA(ctx, cudaMemcpyAsync(h_pes, pes, (size_t)n_chunks * 4 * sizeof(qm_pestat), cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    *d_model_of = map; *d_pes = pes;
    return QM_OK;
}

// qm_pair_finish with one insert-size model per chunk of the batch: h_pes[4 n_models] on the host (the pairing terms are
// evaluated there), d_pes the same models on the device (NULL: uploaded here), d_model_of each pair's model (NULL: model 0)
int qm_pair_finish_models(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride,
                          const int32_t *d_lens, int64_t n_pairs, int64_t pair_id0, qm_reg *d_regs, int32_t *d_n_regs,
                          const qm_pestat *h_pes, int n_models, const qm_pestat *d_pes, const int32_t *d_model_of, qm_aln *d_alns, void *stream)
{
    if (!ctx || !idx || !opt || !h_pes || n_models < 1 || n_pairs < 0 || (n_pairs > 0 && (!d_codes || !d_lens || !d_regs || !d_n_regs || !d_alns)))
        return QM_EINVAL;
    if (n_pairs == 0) return QM_OK;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (!(opt->flags & QM_F_NO_RESCUE)) {
        const int sr = qm_prof_begin(ctx, QM_ST_RESCUE, st);
        const int rr = qm_mate_rescue_models(ctx, idx, opt, d_codes, stride, d_lens, n_pairs, d_regs, d_n_regs, h_pes, n_models, d_pes, d_model_of,
                                             nullptr, stream);
        qm_prof_end(ctx, QM_ST_RESCUE, sr, st, 3);
        if (rr) return rr;
    }
    // host-evaluated tables (libm): MAPQ length factor, sub_n penalty, pairing term per insert size
    std::vector<double> tab(kMapqTabLen);
    for (int l = 0; l < kMapqTabLen; ++l)
        tab[l] = l < opt->mapq_coef_len ? 1. : log((double)opt->mapq_coef_len) / log((double)l);
    std::vector<int> subn(kSubnTabLen);
    for (int n = 0; n < kSubnTabLen; ++n) subn[n] = (int)(4.343 * log((double)(n + 1)) + .499);
    const int n_pes = 4 * n_models;
    std::vector<int64_t> term_off((size_t)n_pes);
    size_t n_term = 0;
    for (int d = 0; d < n_pes; ++d) {
        term_off[(size_t)d] = (int64_t)n_term;
        if (!h_pes[d].failed && h_pes[d].high >= h_pes[d].low) n_term += (size_t)(h_pes[d].high - h_pes[d].low + 1);
    }
    std::vector<double> term(n_term + 1);
    for (int d = 0; d < n_pes; ++d) {
        const qm_pestat &pe = h_pes[d];
        if (pe.failed || pe.high < pe.low) continue;
        for (int64_t dist = pe.low; dist <= pe.high; ++dist) {
            const double ns = (dist - pe.avg) / pe.std;
            term[term_off[(size_t)d] + (size_t)(dist - pe.low)] = .721 * log(2. * erfc(fabs(ns) * M_SQRT1_2)) * opt->a;
        }
    }
    // scratch 5: tables | counters | task list | per-warp global fallback for oversized direction matrices
    const int cig_blocks = ctx->sm_count * 3;                      // persistent: 3 blocks x 4 warps x 14 KB per SM
    const size_t o_tab = 0, o_subn = o_tab + kMapqTabLen * 8, o_pes = o_subn + kSubnTabLen * 4;
    const size_t o_toff = o_pes + (size_t)n_pes * sizeof(qm_pestat), o_term = o_toff + (size_t)n_pes * 8;
    const size_t o_misc = (o_term + term.size() * 8 + 255) & ~(size_t)255;
    const size_t o_tasks = o_misc + 256;
    const size_t o_left = (o_tasks + (size_t)2 * n_pairs * sizeof(CigTask) + 255) & ~(size_t)255;
    const size_t o_slab = (o_left + (size_t)9 * 2 * n_pairs * sizeof(int) + 255) & ~(size_t)255;
    // thread-per-task traceback kernels (32 / 64 / 128 slots of 6 B per thread): 8 / 4 / 2 blocks of 128 threads per SM
    const int tr_blocks[3] = { ctx->sm_count * 8, ctx->sm_count * 4, ctx->sm_count * 2 };
    const size_t o_over = (o_slab + (size_t)(tr_blocks[0] + tr_blocks[1] + tr_blocks[2]) * 128 * (kTraceCellsPerThread / 2) + 255) & ~(size_t)255;
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 5, o_over + (size_t)cig_blocks * kCigWarps * kOverflowPerWarp, &p);
    if (rc) return rc;
    char *b = (char *)p;
    QM_CUDA(ctx, cudaMemcpyAsync(b + o_tab, tab.data(), kMapqTabLen * 8, cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync(b + o_subn, subn.data(), kSubnTabLen * 4, cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync(b + o_pes, h_pes, (size_t)n_pes * sizeof(qm_pestat), cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync(b + o_toff, term_off.data(), (size_t)n_pes * 8, cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync(b + o_term, term.data(), term.size() * 8, cudaMemcpyHostToDevice, st));
    QM_CUDA(ctx, cudaMemsetAsync(b + o_misc, 0, 256, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));      // the host vectors above go out of scope
    PairTables T;
    T.mapq_l = (const double *)(b + o_tab); T.subn = (const int *)(b + o_subn);
    T.pes = (const qm_pestat *)(b + o_pes); T.term_off = (const int64_t *)(b + o_toff); T.term = (const double *)(b + o_term);
    T.model_of = d_model_of;
    int *n_tasks = (int *)(b + o_misc), *cursor = (int *)(b + o_misc + 8), *err = (int *)(b + o_misc + 16);
    // task lists of 2 n_pairs slots each, see the launches below; counters n_list[0..8]
    int *n_list = (int *)(b + o_misc + 32), *lists = (int *)(b + o_left);
    const int64_t lstride = 2 * n_pairs;
    CigTask *tasks = (CigTask *)(b + o_tasks);
    const unsigned grid = (unsigned)((n_pairs + 127) / 128);
    static bool attr_set[64] = {};              // per device: function attributes belong to a device's context, and one
                                                // process may drive several GPUs (qm_driver --gpus)
    if (!attr_set[ctx->device & 63]) {
        QM_CUDA(ctx, cudaFuncSetAttribute(cigar_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCigWarps * kDirBytes));
        QM_CUDA(ctx, cudaFuncSetAttribute(cig_score_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 32 * kCsT * 6));
        QM_CUDA(ctx, cudaFuncSetAttribute(cig_score_kernel<48>, cudaFuncAttributeMaxDynamicSharedMemorySize, 48 * kCsT * 6));
        QM_CUDA(ctx, cudaFuncSetAttribute(cig_score_kernel<72>, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * kCsT * 6));
        QM_CUDA(ctx, cudaFuncSetAttribute(cig_trace_kernel<64, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 128 * 6));
        QM_CUDA(ctx, cudaFuncSetAttribute(cig_trace_kernel<128, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 128 * 6));
        attr_set[ctx->device & 63] = true;
    }
    const int sp = qm_prof_begin(ctx, QM_ST_PAIR, st);
    pair_decide_kernel<<<grid, 128, 0, st>>>(idx->v, *opt, T, d_codes, stride, d_lens, n_pairs, pair_id0, d_regs, d_n_regs, d_alns,
                                             tasks, n_tasks, lists, lstride, n_list);
    // Eight independent kernels, none of which fills the GPU alone (shared memory caps the resident warps): side streams,
    // as the extension classes do.  [0..2] score-only pass by band (equal lengths); [3..5] thread-per-task traceback by band
    // (length difference); [6] warp-per-task traceback for what kernel 1 already knows to be too wide.  What the score-only
    // kernels cannot finish lands in list 7, what the thread-per-task traceback kernels cannot hold in list 8: two more
    // warp-per-task launches behind the join.
    int *cursor2 = (int *)(b + o_misc + 12), *cursor3 = (int *)(b + o_misc + 20);
    uint8_t *slab = (uint8_t *)(b + o_slab);
    const size_t slab_per_thread = kTraceCellsPerThread / 2;
    QM_CUDA(ctx, cudaEventRecord(ctx->ev_fork, st));
    for (int c = 0; c < 7; ++c) {
        cudaStream_t sc = ctx->side[c];
        QM_CUDA(ctx, cudaStreamWaitEvent(sc, ctx->ev_fork, 0));
        const int *mine = lists + c * lstride, *n_mine = n_list + c;
        auto blocks_for = [&](size_t sm) { return (unsigned)(ctx->sm_count * (int)std::min<size_t>(16, (227u * 1024u) / (sm + 1024))); };
        switch (c) {
        case 0: cig_score_kernel<32><<<blocks_for(32 * kCsT * 6), kCsT, 32 * kCsT * 6, sc>>>(idx->v, *opt, d_codes, stride, d_lens, tasks, mine, n_mine, d_alns, lists + 7 * lstride, n_list + 7); break;
        case 1: cig_score_kernel<48><<<blocks_for(48 * kCsT * 6), kCsT, 48 * kCsT * 6, sc>>>(idx->v, *opt, d_codes, stride, d_lens, tasks, mine, n_mine, d_alns, lists + 7 * lstride, n_list + 7); break;
        case 2: cig_score_kernel<72><<<blocks_for(72 * kCsT * 6), kCsT, 72 * kCsT * 6, sc>>>(idx->v, *opt, d_codes, stride, d_lens, tasks, mine, n_mine, d_alns, lists + 7 * lstride, n_list + 7); break;
        case 3: cig_trace_kernel<32, 128><<<tr_blocks[0], 128, 32 * 128 * 6, sc>>>(idx->v, *opt, d_codes, stride, d_lens, tasks, mine, n_mine, 15, slab, d_alns,
                                                                                  lists + 8 * lstride, n_list + 8); break;
        case 4: cig_trace_kernel<64, 128><<<tr_blocks[1], 128, 64 * 128 * 6, sc>>>(idx->v, *opt, d_codes, stride, d_lens, tasks, mine, n_mine, 31,
                                                                                  slab + (size_t)tr_blocks[0] * 128 * slab_per_thread, d_alns, lists + 8 * lstride, n_list + 8); break;
        case 5: cig_trace_kernel<128, 128><<<tr_blocks[2], 128, 128 * 128 * 6, sc>>>(idx->v, *opt, d_codes, stride, d_lens, tasks, mine, n_mine, 63,
                                                                                    slab + (size_t)(tr_blocks[0] + tr_blocks[1]) * 128 * slab_per_thread, d_alns,
                                                                                    lists + 8 * lstride, n_list + 8); break;
        default: cigar_kernel<<<cig_blocks, kCigWarps * 32, kCigWarps * kDirBytes, sc>>>(idx->v, *opt, d_codes, stride, d_lens, tasks, mine, n_mine, cursor2,
                                                                                       (uint8_t *)(b + o_over), d_alns, err); break;
        }
        QM_CUDA(ctx, cudaEventRecord(ctx->ev_join[c], sc));
        QM_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_join[c], 0));
    }
    cigar_kernel<<<cig_blocks, kCigWarps * 32, kCigWarps * kDirBytes, st>>>(idx->v, *opt, d_codes, stride, d_lens, tasks, lists + 8 * lstride, n_list + 8,
                                                                          cursor3, (uint8_t *)(b + o_over), d_alns, err);
    cigar_kernel<<<cig_blocks, kCigWarps * 32, kCigWarps * kDirBytes, st>>>(idx->v, *opt, d_codes, stride, d_lens, tasks, lists + 7 * lstride, n_list + 7,
                                                                          cursor, (uint8_t *)(b + o_over), d_alns, err);
    pair_finish_kernel<<<(unsigned)((n_pairs + kFinT - 1) / kFinT), kFinT, 0, st>>>(idx->v, T, n_pairs, d_regs, d_alns);
    qm_prof_end(ctx, QM_ST_PAIR, sp, st, 11);
    QM_CUDA(ctx, cudaGetLastError());
    int h_err = 0;
    QM_CUDA(ctx, cudaMemcpyAsync(&h_err, err, 4, cudaMemcpyDeviceToHost, st));
    QM_CUDA(ctx, cudaStreamSynchronize(st));
    if (h_err) return qm_fail(ctx, QM_ELIMIT, "qm_pair_finish: traceback scratch exhausted (code %d)", h_err);
    return QM_OK;
}

int qm_pair_finish(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride,
                   const int32_t *d_lens, int64_t n_pairs, int64_t pair_id0, qm_reg *d_regs, int32_t *d_n_regs,
                   const qm_pestat pes[4], qm_aln *d_alns, void *stream)
{
    if (!pes) return QM_EINVAL;
    return qm_pair_finish_models(ctx, idx, opt, d_codes, stride, d_lens, n_pairs, pair_id0, d_regs, d_n_regs, pes, 1, nullptr, nullptr, d_alns, stream);
}

}  // extern "C"
