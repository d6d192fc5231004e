// rescue.cu -- mate rescue: bwamem_pair.c mem_matesw as driven by mem_sam_pe, with ksw.c ksw_align2 (KSW_XSUBO |
// KSW_XSTART | min_seed_len * a) as the local alignment.  Reference call site rules/bwa.smk:15 (`bwa mem` runs it for
// every pair in which an end has no region at a proper distance from a region of its mate); semantics SURVEY.md A.6 and
// the restatement oracle/qmo_mem.c matesw / oracle/qmo_ksw.c qmo_ksw_align2.
//
// Few pairs need it (1 - 4 % on the BASELINE configs), each of them needs a 150 x ~450 cell local alignment plus the
// reversed pass that finds its start, and the outcome of one alignment decides whether the next one of the pair runs
// at all.  So: a scan kernel lists the pairs in which the first alignment would run; a persistent kernel gives each
// listed pair to one WARP, which walks the pair's anchors in bwa's order.  The alignment itself is a wavefront over
// the warp: lane l owns C consecutive query columns (H and E of its columns in registers), at step s it computes row
// s - l, and the row's state at the strip boundary (H, F, running row maximum and its first column) moves to lane
// l + 1 by shuffle; lane 31 closes a row: best score / first row / first column, the log of rows above min score
// that gives the sub-optimal score, the early stop of the reversed pass.  Target window and query sit in shared memory.
#include <stdlib.h>
#include "pipeline.cuh"

namespace {

constexpr int kResWarps = 8;                 // warps per block
constexpr int kResMaxWindow = 4096;          // = QMO_RESCUE_MAX_WINDOW: longer windows are not searched
constexpr int kResMaxQuery = 512;
constexpr int kResLog = kResMaxWindow;       // log entries per warp (at most one per row)
constexpr int kNoLimit = 0x10000;

struct SwOut { int score, te, qe, score2, te2, tb, qb; };

// One pass of the local recurrence over target rows [0, tlen) and query columns [0, qlen), both read from shared
// memory through (base, step): element i is base[i * step].  minsc: rows whose maximum reaches it are logged in
// log[] as (imax << 16 | row), same merge rule as ksw_u8's b[]; endsc: stop at the first row whose maximum reaches it.
// All lanes return the same (score, te, qe, n_log).
// Per cell 10 integer instructions: compare + select (score), viaddmax.relu + max (H), shift-add + max (row maximum
// and its FIRST column as one key: imax << 16 | 0xffff - column), sub + viaddmax twice (E and F; neither is clamped at
// zero as the byte-wide upstream loop does: both stay >= -(gap open + extend) and no non-positive value can win a cell).
template <int C>
__device__ void local_pass_warp(const qm_opt &o, const uint8_t *qbase, int qstep, int qlen, const uint8_t *tbase, int tstep, int tlen,
                                int minsc, int endsc, uint32_t *log, int &score, int &te, int &qe, int &n_log, long long &cells)
{
    const int lane = threadIdx.x & 31;
    const int c0 = lane * C;
    const int oe_del = o.o_del + o.e_del, oe_ins = o.o_ins + o.e_ins, ne_del = -o.e_del, ne_ins = -o.e_ins, sa = o.a;
    int q[C], msk[C], H[C], E[C], kcol[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const int code = c0 + c < qlen ? qbase[(c0 + c) * qstep] : 5;
        q[c] = code < 4 ? code : 8;                                  // N and padding equal no target base
        msk[c] = code == 5 ? -30000 : code == 4 ? -1 : -o.b;         // the score of a column when the bases differ
        H[c] = 0; E[c] = 0; kcol[c] = 0xffff - (c0 + c);
    }
    constexpr uint32_t kKey0 = 0x0000ffffu;                          // row maximum 0, no column
    uint32_t out_hf = 0, out_key = kKey0;                            // H of my last column | F leaving it << 16; running key
    int left_prev = 0;
    int gmax = 0, g_te = -1, g_qe = -1, nl = 0, last_row = -2, last_sc = 0;
    bool done = false;
    const int n_steps = tlen + 31;
    for (int s = 0; s < n_steps; ++s) {
        uint32_t in_hf = __shfl_up_sync(0xffffffffu, out_hf, 1), key = __shfl_up_sync(0xffffffffu, out_key, 1);
        if (lane == 0) { in_hf = 0; key = kKey0; }
        const int i = s - lane;
        if (i >= 0 && i < tlen) {
            const int tb = tbase[i * tstep];
            int diag = left_prev, f = (int)in_hf >> 16;
            left_prev = (int)(in_hf & 0xffffu);
#define QM_RES_CELL(SC)                                                                  \
            {                                                                            \
                int h = __viaddmax_s32_relu(diag, (SC), E[c]);                            \
                diag = H[c];                                                             \
                h = max(h, f);                                                           \
                H[c] = h;                                                                \
                key = max(key, ((uint32_t)h << 16) + (uint32_t)kcol[c]);                  \
                E[c] = __viaddmax_s32(E[c], ne_del, h - oe_del);                          \
                f = __viaddmax_s32(f, ne_ins, h - oe_ins);                                \
            }
            if (tb < 4) {
#pragma unroll
                for (int c = 0; c < C; ++c) QM_RES_CELL(q[c] == tb ? sa : msk[c])
            } else {                                            // N in the reference: -1 against every real base
#pragma unroll
                for (int c = 0; c < C; ++c) QM_RES_CELL(msk[c] < -1000 ? msk[c] : -1)
            }
#undef QM_RES_CELL
            out_hf = (uint32_t)H[C - 1] | ((uint32_t)f << 16); out_key = key;
            if (lane == 31) {                               // the row is complete
                const int imax = (int)(key >> 16), imax_j = 0xffff - (int)(key & 0xffffu);
                if (imax >= minsc) {
                    if (nl == 0 || last_row + 1 != i) { if (nl < kResLog) log[nl] = (uint32_t)imax << 16 | (uint32_t)i; ++nl; last_row = i; last_sc = imax; }
                    else if (last_sc < imax) { log[nl - 1] = (uint32_t)imax << 16 | (uint32_t)i; last_row = i; last_sc = imax; }
                }
                if (imax > gmax) { gmax = imax; g_te = i; g_qe = imax_j; if (gmax >= endsc) done = true; }
            }
        }
        if (endsc < kNoLimit && __shfl_sync(0xffffffffu, (int)done, 31)) break;
    }
    score = __shfl_sync(0xffffffffu, gmax, 31);
    te = __shfl_sync(0xffffffffu, g_te, 31);
    qe = __shfl_sync(0xffffffffu, g_qe, 31);
    n_log = __shfl_sync(0xffffffffu, nl, 31);
    // executed cells as the reference loop counts them: whole rows up to and including the row that stopped the pass
    cells += (long long)qlen * (endsc < kNoLimit && score >= endsc ? te + 1 : tlen);
}

// ksw_align2 on sequences staged in shared memory: seq[0..l_ms) (as searched) against win[0..tlen)
template <int C>
__device__ SwOut sw_align2_warp(const qm_opt &o, const uint8_t *seq, int l_ms, const uint8_t *win, int tlen, int minsc, uint32_t *log, long long &cells)
{
    SwOut r;
    int n_log;
    r.score2 = -1; r.te2 = -1; r.tb = -1; r.qb = -1;
    local_pass_warp<C>(o, seq, 1, l_ms, win, 1, tlen, minsc, kNoLimit, log, r.score, r.te, r.qe, n_log, cells);
    __syncwarp();
    if (n_log > 0) {
        // best logged row further than `score` rows from te, first one on ties: lanes take entries round-robin and keep
        // their earliest best, then the warp reduces on (score desc, entry index asc)
        const int lane = threadIdx.x & 31;
        const int max_sc = o.a > 1 ? o.a : 1;
        const int mx = (r.score + max_sc - 1) / max_sc, low = r.te - mx, high = r.te + mx;
        int best = -1, best_at = 0x7fffffff, best_row = -1;
        for (int e = lane; e < n_log; e += 32) {
            const uint32_t v = log[e];
            const int row = (int)(v & 0xffffu), sc = (int)(v >> 16);
            if ((row < low || row > high) && sc > best) { best = sc; best_at = e; best_row = row; }
        }
#pragma unroll
        for (int d = 16; d; d >>= 1) {
            const int ob = __shfl_xor_sync(0xffffffffu, best, d), oa = __shfl_xor_sync(0xffffffffu, best_at, d), orow = __shfl_xor_sync(0xffffffffu, best_row, d);
            if (ob > best || (ob == best && oa < best_at)) { best = ob; best_at = oa; best_row = orow; }
        }
        if (best > r.score2) { r.score2 = best; r.te2 = best_row; }
    }
    if (r.score < minsc || r.te < 0) return r;
    int sc2, te2, qe2, nl2;
    local_pass_warp<C>(o, seq + r.qe, -1, r.qe + 1, win + r.te, -1, r.te + 1, kNoLimit, r.score, log, sc2, te2, qe2, nl2, cells);
    if (sc2 == r.score) { r.tb = r.te - te2; r.qb = r.qe - qe2; }
    return r;
}

// insert-size models, 4 per model; pair p searches with model model_of[p] (model 0 when model_of is NULL)
struct PesArg {
    const qm_pestat *pes;
    const int32_t *model_of;
    __device__ __forceinline__ const qm_pestat *of(int64_t pi) const { return pes + 4 * (model_of ? model_of[pi] : 0); }
};

// orientations (bit r) in which the anchor at arb needs no alignment: no usable model, or a region of the mate at a proper distance
__device__ __forceinline__ int served_dirs(const IndexView &V, const qm_pestat *pes, int64_t arb, const qm_reg *ma, int n_ma)
{
    int skip = 0;
    for (int r = 0; r < 4; ++r) if (pes[r].failed) skip |= 1 << r;
    for (int i = 0; i < n_ma; ++i) {
        int64_t dist;
        const int r = qm_infer_dir(V.l_pac, arb, ma[i].rb, &dist);
        if (dist >= pes[r].low && dist <= pes[r].high) skip |= 1 << r;
    }
    return skip;
}

// the window orientation r implies for a mate of l_ms bases around an anchor at arb on contig arid (mem_matesw +
// bns_fetch_seq); false: nothing to align there
__device__ __forceinline__ bool rescue_window(const IndexView &V, const qm_opt &o, const qm_pestat *pes, int64_t arb, int arid, int r, int l_ms,
                                              int max_query, int64_t &rb, int64_t &re, bool &is_rev)
{
    const int64_t l_pac = V.l_pac;
    is_rev = (r >> 1) != (r & 1);                         // the mate is searched as its reverse complement
    const bool is_larger = !(r >> 1);                     // the mate lies at the larger coordinate
    if (!is_rev) {
        rb = is_larger ? arb + pes[r].low : arb - pes[r].high;
        re = (is_larger ? arb + pes[r].high : arb - pes[r].low) + l_ms;
    } else {
        rb = (is_larger ? arb + pes[r].low : arb - pes[r].high) - l_ms;
        re = is_larger ? arb + pes[r].high : arb - pes[r].low;
    }
    if (rb < 0) rb = 0;
    if (re > l_pac << 1) re = l_pac << 1;
    int rid = -1;
    if (rb < re) {                                        // the contig and strand of the midpoint
        const int64_t mid = (rb + re) >> 1;
        const bool mrev = mid >= l_pac;
        rid = qm_pos2rid(V, mrev ? 2 * l_pac - 1 - mid : mid);
        int64_t far_beg = V.off[rid], far_end = far_beg + V.len[rid];
        if (mrev) { const int64_t x = far_beg; far_beg = (l_pac << 1) - far_end; far_end = (l_pac << 1) - x; }
        if (rb < far_beg) rb = far_beg;
        if (re > far_end) re = far_end;
    }
    return arid == rid && re - rb >= o.min_seed_len && re - rb <= kResMaxWindow && l_ms <= max_query;
}

// The alignments of a pair depend on one another only through WHETHER they run (an earlier hit can serve the
// orientation a later anchor would have searched); what an alignment finds depends on its window alone.  So every
// alignment the lists would trigger as they stand is run up front, one warp each, and the pass that walks the
// anchors in bwa's order only looks the results up (and runs the rare alignment that becomes necessary later itself).
struct ResTask { int32_t pair; int32_t tr; };          // tr = anchor slot (end << 4 | index) << 2 | orientation
struct ResOut { int32_t score, te, qe, score2, te2, tb, qb; int32_t cells; };     // cells < 2^31: 512 x 4096 x 2 passes

// thread per pair: the alignments to run up front, in (anchor, orientation) order, as one block of the task list
__global__ void __launch_bounds__(128)
rescue_scan_kernel(IndexView V, qm_opt o, PesArg P, int64_t n_pairs, int max_query, const qm_reg *__restrict__ regs, const int32_t *__restrict__ n_regs,
                   const int32_t *__restrict__ lens, int *__restrict__ list, int2 *__restrict__ blocks, ResTask *__restrict__ tasks, int cap_tasks,
                   int *__restrict__ ctr)
{
    const int64_t pi = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (pi >= n_pairs) return;
    const qm_pestat *pes = P.of(pi);
    int k = 0, base = 0;
    for (int pass = 0; pass < 2; ++pass) {              // count, then write
        int w = 0;
        for (int i = 0; i < 2; ++i) {
            const qm_reg *a = regs + (2 * pi + i) * QM_MAX_REGS, *ma = regs + (2 * pi + !i) * QM_MAX_REGS;
            const int n = n_regs[2 * pi + i], n_ma = n_regs[2 * pi + !i], l_ms = lens[2 * pi + !i];
            for (int j = 0; j < n; ++j) {
                if (a[j].score < a[0].score - o.pen_unpaired) continue;
                const int skip = served_dirs(V, pes, a[j].rb, ma, n_ma);
                if (skip == 15) continue;
                for (int r = 0; r < 4; ++r) {
                    int64_t rb, re;
                    bool is_rev;
                    if ((skip >> r & 1) || !rescue_window(V, o, pes, a[j].rb, a[j].rid, r, l_ms, max_query, rb, re, is_rev)) continue;
                    if (pass && base + w < cap_tasks) { ResTask t; t.pair = k ? (int)pi : -1; t.tr = ((i << 4 | j) << 2) | r; tasks[base + w] = t; }
                    ++w;
                }
            }
        }
        if (!pass) {
            k = w;
            if (k == 0) return;                          // nothing runs, nothing changes
            base = atomicAdd(ctr + 1, k);
            if (base > cap_tasks) base = cap_tasks;      // (the counter can run past the list, never wrap: <= 128 per pair)
            if (base + k > cap_tasks) k = 0;             // no room: slots taken are marked void, the pair aligns as it goes
            const int item = atomicAdd(ctr, 1);
            list[item] = (int)pi;
            blocks[item] = make_int2(base, k);
        }
    }
}

// stage window and mate in shared memory and align (all lanes get the result)
template <int C>
__device__ ResOut run_alignment(const IndexView &V, const qm_opt &o, const uint8_t *ms, int l_ms, int64_t rb, int64_t re, bool is_rev,
                                uint8_t *win, uint8_t *seq, uint32_t *log)
{
    const int lane = threadIdx.x & 31;
    const int tlen = (int)(re - rb);
    __syncwarp();
    for (int x = lane; x < tlen; x += 32) win[x] = (uint8_t)qm_ref_base(V, rb + x);
    for (int x = lane; x < l_ms; x += 32) { const int c = ms[is_rev ? l_ms - 1 - x : x]; seq[x] = (uint8_t)(is_rev ? (c < 4 ? 3 - c : 4) : c); }
    __syncwarp();
    long long cells = 0;
    const SwOut a = sw_align2_warp<C>(o, seq, l_ms, win, tlen, o.min_seed_len * o.a, log, cells);
    ResOut r;
    r.score = a.score; r.te = a.te; r.qe = a.qe; r.score2 = a.score2; r.te2 = a.te2; r.tb = a.tb; r.qb = a.qb; r.cells = (int32_t)cells;
    return r;
}

// warp per task of the up-front list
template <int C>                        // query columns per lane: reads of up to 32 * C bases
__global__ void __launch_bounds__(kResWarps * 32, C <= 5 ? 4 : C <= 8 ? 3 : 2)
rescue_align_kernel(IndexView V, qm_opt o, PesArg P, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
                    const qm_reg *__restrict__ regs, const ResTask *__restrict__ tasks, int cap_tasks, int *__restrict__ ctr,
                    uint32_t *__restrict__ logs, ResOut *__restrict__ out)
{
    __shared__ uint8_t s_win[kResWarps][kResMaxWindow];
    __shared__ uint8_t s_seq[kResWarps][kResMaxQuery];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint32_t *log = logs + (size_t)(blockIdx.x * kResWarps + wib) * kResLog;
    const int total = ctr[1] < cap_tasks ? ctr[1] : cap_tasks;
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(ctr + 2, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= total) break;
        const ResTask t = tasks[item];
        if (t.pair < 0) continue;
        const int slot = t.tr >> 2, r = t.tr & 3, i = slot >> 4, j = slot & 15;
        const qm_reg *a = regs + (2 * (int64_t)t.pair + i) * QM_MAX_REGS + j;
        const int l_ms = lens[2 * (int64_t)t.pair + !i];
        int64_t rb, re;
        bool is_rev;
        rescue_window(V, o, P.of(t.pair), a->rb, a->rid, r, l_ms, 32 * C, rb, re, is_rev);
        const ResOut res = run_alignment<C>(V, o, codes + (2 * (int64_t)t.pair + !i) * stride, l_ms, rb, re, is_rev, s_win[wib], s_seq[wib], log);
        if (lane == 0) out[item] = res;
    }
}

// warp per listed pair: mem_sam_pe's loop over the anchors, mem_matesw per anchor
template <int C>
__global__ void __launch_bounds__(kResWarps * 32, C <= 5 ? 4 : C <= 8 ? 3 : 2)
rescue_apply_kernel(IndexView V, qm_opt o, PesArg P, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
                    qm_reg *__restrict__ regs, int32_t *__restrict__ n_regs, const int *__restrict__ list, const int2 *__restrict__ blocks,
                    const ResTask *__restrict__ tasks, const ResOut *__restrict__ results, int *__restrict__ ctr, uint32_t *__restrict__ logs,
                    unsigned long long *__restrict__ stats)
{
    __shared__ uint8_t s_win[kResWarps][kResMaxWindow];
    __shared__ uint8_t s_seq[kResWarps][kResMaxQuery];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    uint32_t *log = logs + (size_t)(blockIdx.x * kResWarps + wib) * kResLog;
    const int total = ctr[0];
    const int64_t l_pac = V.l_pac;
    long long cells = 0;
    int n_sw = 0;
    for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(ctr + 3, 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= total) break;
        const int64_t pi = list[item];
        const int2 blk = blocks[item];
        const qm_pestat *pes = P.of(pi);
        int next = 0;                                   // first result of the pair's block not yet passed
        // anchors: lane t holds anchor j = t & 15 of end t >> 4 as the lists were BEFORE any rescue
        int64_t my_rb = 0;
        int my_rid = -1;
        bool my_ok = false;
        {
            const int i = lane >> 4, j = lane & 15;
            const qm_reg *a = regs + (2 * pi + i) * QM_MAX_REGS;
            if (j < n_regs[2 * pi + i] && a[j].score >= a[0].score - o.pen_unpaired) { my_ok = true; my_rb = a[j].rb; my_rid = a[j].rid; }
        }
        __syncwarp();
        for (int t = 0; t < 32; ++t) {
            if (!__shfl_sync(0xffffffffu, (int)my_ok, t)) continue;
            const int i = t >> 4;
            const int64_t arb = __shfl_sync(0xffffffffu, my_rb, t);
            const int arid = __shfl_sync(0xffffffffu, my_rid, t);
            qm_reg *ma = regs + (2 * pi + !i) * QM_MAX_REGS;
            int n_ma = n_regs[2 * pi + !i];
            const int l_ms = lens[2 * pi + !i];
            // orientations already served by a region of the mate (lanes over the mate's regions)
            int skip = 0;
            for (int r = 0; r < 4; ++r) if (pes[r].failed) skip |= 1 << r;
            {
                int mine = 0;
                if (lane < n_ma) {
                    int64_t dist;
                    const int r = qm_infer_dir(l_pac, arb, ma[lane].rb, &dist);
                    if (dist >= pes[r].low && dist <= pes[r].high) mine = 1 << r;
                }
#pragma unroll
                for (int d = 16; d; d >>= 1) mine |= __shfl_xor_sync(0xffffffffu, mine, d);
                skip |= mine;
            }
            if (skip == 15) continue;
            int n = 0;
            for (int r = 0; r < 4; ++r) {
                if (skip >> r & 1) continue;
                int64_t rb, re;
                bool is_rev;
                if (rescue_window(V, o, pes, arb, arid, r, l_ms, 32 * C, rb, re, is_rev)) {
                    const int want = (t << 2) | r;
                    while (next < blk.y && tasks[blk.x + next].tr < want) ++next;       // run up front, not needed after all
                    ResOut aln;
                    if (next < blk.y && tasks[blk.x + next].tr == want) aln = results[blk.x + next++];
                    else aln = run_alignment<C>(V, o, codes + (2 * pi + !i) * (int64_t)stride, l_ms, rb, re, is_rev, s_win[wib], s_seq[wib], log);
                    cells += aln.cells;
                    if (lane == 0 && aln.score >= o.min_seed_len && aln.qb >= 0) {
                        qm_reg b;
                        b.rid = arid;
                        b.qb = is_rev ? l_ms - (aln.qe + 1) : aln.qb;
                        b.qe = is_rev ? l_ms - aln.qb : aln.qe + 1;
                        b.rb = is_rev ? (l_pac << 1) - (rb + aln.te + 1) : rb + aln.tb;
                        b.re = is_rev ? (l_pac << 1) - (rb + aln.tb) : rb + aln.te + 1;
                        b.score = aln.score; b.truesc = 0; b.sub = 0; b.csub = aln.score2; b.sub_n = 0; b.w = 0;
                        b.seedcov = (int)((b.re - b.rb < b.qe - b.qb ? b.re - b.rb : b.qe - b.qb) >> 1);
                        b.secondary = -1; b.seedlen0 = 0;
                        int at = 0;
                        while (at < n_ma && ma[at].score >= b.score) ++at;      // behind the entries that score at least as much
                        if (n_ma < QM_MAX_REGS) ++n_ma;                         // a full list loses its last entry
                        if (at < n_ma) {
                            for (int x = n_ma - 1; x > at; --x) ma[x] = ma[x - 1];
                            ma[at] = b;
                        }
                    }
                    ++n; ++n_sw;
                }
                if (n) {
                    if (lane == 0) n_ma = qm_sort_dedup(o, n_ma, ma);
                    n_ma = __shfl_sync(0xffffffffu, n_ma, 0);
                }
                __syncwarp();
            }
            if (lane == 0) n_regs[2 * pi + !i] = n_ma;
            __syncwarp();
        }
    }
    if (lane == 0 && stats && (n_sw || cells)) { atomicAdd(stats, (unsigned long long)n_sw); atomicAdd(stats + 1, (unsigned long long)cells); }
}

}  // namespace

extern "C" {

// mate rescue with one insert-size model per chunk of the batch: h_pes[4 n_models] on the host, d_pes the same on the device
// (NULL: uploaded here), d_model_of each pair's model (NULL: model 0)
int qm_mate_rescue_models(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride, const int32_t *d_lens,
                          int64_t n_pairs, qm_reg *d_regs, int32_t *d_n_regs, const qm_pestat *h_pes, int n_models, const qm_pestat *d_pes,
                          const int32_t *d_model_of, int64_t *d_stats, void *stream)
{
    const qm_pestat *pes = h_pes;
    if (!ctx || !idx || !opt || !pes || n_models < 1 || n_pairs < 0 || (n_pairs > 0 && (!d_codes || !d_lens || !d_regs || !d_n_regs))) return QM_EINVAL;
    if (n_pairs == 0) return QM_OK;
    if (n_pairs > (1ll << 24)) return qm_fail(ctx, QM_ELIMIT, "qm_mate_rescue: more than 2^24 pairs in one call");
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    bool any = false;
    for (int d = 0; d < 4 * n_models; ++d) any |= !pes[d].failed;
    if (!any) return QM_OK;                       // no usable insert-size model: every orientation is skipped
    if (stride > kResMaxQuery) return qm_fail(ctx, QM_ELIMIT, "qm_mate_rescue: reads longer than %d bases", kResMaxQuery);
    const int blocks = ctx->sm_count * (stride <= 160 ? 4 : stride <= 256 ? 3 : 2);
    // scratch 14: counters | pair list | task blocks of the pairs | tasks | results | per-warp row logs
    // The up-front task list holds 4 tasks per pair of the batch (a pair can have 32 anchors x 4 orientations, a batch in
    // which few pairs need rescue -- every realistic one -- uses a small part of it); a pair whose block does not fit is
    // not run up front, the apply pass then aligns for it as it goes.
    // QM_RESCUE_INLINE=1 (test knob): an empty list, every alignment is run by the apply pass as it goes
    const size_t cap_tasks = getenv("QM_RESCUE_INLINE") ? 0 : (size_t)n_pairs * 4 + 1024;
    const size_t o_list = 256, o_blk = (o_list + (size_t)n_pairs * sizeof(int) + 255) & ~(size_t)255;
    const size_t o_task = (o_blk + (size_t)n_pairs * sizeof(int2) + 255) & ~(size_t)255;
    const size_t o_res = (o_task + cap_tasks * sizeof(ResTask) + 255) & ~(size_t)255;
    const size_t o_log = (o_res + cap_tasks * sizeof(ResOut) + 255) & ~(size_t)255;
    const size_t o_pes = o_log + (size_t)blocks * kResWarps * kResLog * sizeof(uint32_t);
    void *p = nullptr;
    const int rc = qm_scratch_reserve(ctx, 14, o_pes + (d_pes ? 0 : (size_t)n_models * 4 * sizeof(qm_pestat)), &p);
    if (rc) return rc;
    char *b = (char *)p;
    int *ctr = (int *)b;                              // [0] listed pairs, [1] tasks, [2] task cursor, [3] pair cursor
    int *list = (int *)(b + o_list);
    int2 *blk = (int2 *)(b + o_blk);
    ResTask *tasks = (ResTask *)(b + o_task);
    ResOut *results = (ResOut *)(b + o_res);
    uint32_t *logs = (uint32_t *)(b + o_log);
    unsigned long long *stats = (unsigned long long *)d_stats;
    QM_CUDA(ctx, cudaMemsetAsync(b, 0, 256, st));
    PesArg P;
    P.model_of = d_model_of;
    P.pes = d_pes;
    if (!d_pes) {
        QM_CUDA(ctx, cudaMemcpyAsync(b + o_pes, h_pes, (size_t)n_models * 4 * sizeof(qm_pestat), cudaMemcpyHostToDevice, st));
        P.pes = (const qm_pestat *)(b + o_pes);
    }
    // reads are at most `stride` long: 5 / 8 / 16 query columns per lane
    const int C = stride <= 160 ? 5 : stride <= 256 ? 8 : 16;
    rescue_scan_kernel<<<(unsigned)((n_pairs + 127) / 128), 128, 0, st>>>(idx->v, *opt, P, n_pairs, 32 * C, d_regs, d_n_regs, d_lens, list, blk, tasks, (int)cap_tasks, ctr);
#define QM_RES_LAUNCH(C_)                                                                                                                   \
    do {                                                                                                                                    \
        rescue_align_kernel<C_><<<blocks, kResWarps * 32, 0, st>>>(idx->v, *opt, P, d_codes, stride, d_lens, d_regs, tasks, (int)cap_tasks, ctr, logs, results); \
        rescue_apply_kernel<C_><<<blocks, kResWarps * 32, 0, st>>>(idx->v, *opt, P, d_codes, stride, d_lens, d_regs, d_n_regs, list, blk, tasks,    \
                                                                  results, ctr, logs, stats);                                               \
    } while (0)
    if (C == 5) QM_RES_LAUNCH(5); else if (C == 8) QM_RES_LAUNCH(8); else QM_RES_LAUNCH(16);
#undef QM_RES_LAUNCH
    QM_CUDA(ctx, cudaGetLastError());
    return QM_OK;
}

int qm_mate_rescue(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride, const int32_t *d_lens,
                   int64_t n_pairs, qm_reg *d_regs, int32_t *d_n_regs, const qm_pestat pes[4], int64_t *d_stats, void *stream)
{
    return qm_mate_rescue_models(ctx, idx, opt, d_codes, stride, d_lens, n_pairs, d_regs, d_n_regs, pes, 1, nullptr, nullptr, d_stats, stream);
}

}  // extern "C"
