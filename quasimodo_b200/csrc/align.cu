// align.cu -- single-end alignment stage: seeding, chaining, the per-read extension state machine and
// redundancy removal.  Replaces the compute of `bwa mem -k 31` worker1 (bwamem.c mem_align1_core:
// mem_chain -> mem_chain_flt -> mem_chain2aln -> mem_sort_dedup_patch; reference call site
// rules/bwa.smk:15; semantics SURVEY.md A.2, A.5).
//
// Layout of the work on the GPU:
//   pack_reads_kernel   a block's rows staged by one cp.async.bulk copy, every read packed to 2 bits per base + N flags.
//   seed_walk_kernel    PERSISTENT, one lane per read at a time: 2-bit k-mers of both strands probe the L2-resident hash
//                       index behind a Bloom filter; a hit that is the k-mer's only one is followed 32 bases per step
//                       against the packed reference; consecutive hits on one diagonal are merged into maximal exact
//                       matches; a lane that finishes its read takes the next one off a cursor.
//   plan_kernel         one thread per read: seeds sorted, chained and the chains filtered exactly as bwa does; the
//                       result is a per-read "plan" = the order in which mem_chain2aln visits the seeds.
//   (seed_chain_kernel  the three in one, one read per thread: the form of round 1, kept for A/B runs and very long rows.)
//   advance_kernel      one thread per read: a small state machine that walks the plan, applies
//                       mem_chain2aln's "already covered" test against the read's regions so far and
//                       emits at most one extension task (left or right) per round; it consumes the
//                       previous task's result first (right depends on left).
//   ext3_kernel / ext_kernel<C>   extend3.cu / extend.cu: all tasks of a round, sorted; a thread per PAIR of tasks (packed
//                       s16x2 DPX cells) for the big classes, a warp per task for small rounds and long queries.
//   spec_* / tail_kernel   the last reads of a batch: every remaining seed's extensions ahead of the state machine, or one warp
//                       per read without further host round trips.
//   The host loops advance -> extend until no read emits a task (one 24-byte read-back per round).
// Tasks reference the read batch and the reference in place (ExtTaskI, QM_EXTI_INDIRECT); no sequence
// bytes are materialised.
#include <stdlib.h>
#include <algorithm>
#include "pipeline.cuh"
#include "ext_warp.cuh"

namespace {

enum { PH_NEXT = 0, PH_WAIT_LEFT = 1, PH_WAIT_RIGHT = 2, PH_RIGHT = 3, PH_DONE = 4 };

struct ReadState {
    int16_t cursor;
    uint8_t phase, n_av;
    int32_t task;
};

constexpr int kPlanSkipped = 0x8000;

__device__ __forceinline__ int max_gap_for(const qm_opt &o, int qlen)
{
    const int l_del = (int)((double)(qlen * o.a - o.o_del) / o.e_del + 1.);
    const int l_ins = (int)((double)(qlen * o.a - o.o_ins) / o.e_ins + 1.);
    int l = l_del > l_ins ? l_del : l_ins;
    l = l > 1 ? l : 1;
    return l < o.w << 1 ? l : o.w << 1;
}

// ---- seeding: all maximal exact matches of length >= k on both strands ----
// Every k-mer of the read is looked up on both strands (oracle: qmo_collect_seeds).  Most look-ups are avoided
// without changing the result:
//  * when the previous k-mer had exactly one hit, at forward reference position p, and the next read base continues
//    that match, the next k-mer EQUALS the reference k-mer next to p; if the index says that k-mer is unique and its
//    reverse complement absent (IndexView::uniqp), both look-ups are known: one hit, there.  This is decided for 32
//    positions at a time: read, reference and bitmap are 2-bit / 1-bit packed, one XOR + count-trailing-zeros gives
//    the length of the continuing run;
//  * a k-mer whose canonical form misses the Bloom filter occurs on neither strand.
// The read is packed once into shared memory (2 bits per base + an N bitmap); k-mers are cut out of the packed words,
// so no rolling state ties one position to the next and whole runs can be skipped.
constexpr int kWalkRange = 64;             // reads a warp of the walk kernel takes off the global cursor at a time
constexpr int kBloomBatch = 8;             // filter look-ups in flight per thread behind a mismatch (collect_seeds)
constexpr int kSeedThreads = 128;          // most a block may have (launch bounds); launched with kSeedThreadsDefault

struct PackedRead {                 // per-thread view of the block's shared arrays, [word][thread]
    uint64_t *bits;                 // base j at bits 2*(j&31) of word j>>5
    uint64_t *nmask;                // bit j&63 of word j>>6: base j is N
    int ts;                         // threads per block = stride of both arrays
    __device__ __forceinline__ uint64_t get2(int b) const
    {   // 32 bases starting at base b (words past the read are zero)
        const int w = b >> 5, sh = 2 * (b & 31);
        const uint64_t lo = bits[w * ts];
        return sh ? (lo >> sh) | (bits[(w + 1) * ts] << (64 - sh)) : lo;
    }
    __device__ __forceinline__ uint64_t getn(int b) const
    {   // N flags of 64 bases starting at base b
        const int w = b >> 6, sh = b & 63;
        const uint64_t lo = nmask[w * ts];
        return sh ? (lo >> sh) | (nmask[(w + 1) * ts] << (64 - sh)) : lo;
    }
};

__device__ __forceinline__ uint64_t ref_get2(const IndexView &V, int64_t b)
{   // 32 reference bases starting at forward position b >= -32
    return qm_get2_padded(V.ref2p, b);
}
__device__ __forceinline__ uint32_t uniq_get(const uint32_t *__restrict__ map, int64_t b)
{   // flags of the 32 k-mers starting at forward positions b .. b+31, b >= -32 (map = V.uniqp or V.uniq2p)
    const int64_t x = b + 32;
    const uint32_t *w = map + (x >> 5);
    return __funnelshift_r(__ldg(w), __ldg(w + 1), (unsigned)(x & 31));
}

__device__ void pack_read(const uint8_t *__restrict__ rd, int len, int n_words, int n_nwords, PackedRead &R)
{
    for (int w = 0; w < n_words; ++w) R.bits[w * R.ts] = 0;
    for (int w = 0; w < n_nwords; ++w) R.nmask[w * R.ts] = 0;
    uint64_t acc = 0, nacc = 0;
    int j = 0;
    auto put = [&](unsigned c) {
        acc |= (uint64_t)(c & 3u) << (2 * (j & 31));
        nacc |= (uint64_t)(c >> 2) << (j & 63);
        ++j;
        if ((j & 31) == 0) { R.bits[((j >> 5) - 1) * R.ts] = acc; acc = 0; }
        if ((j & 63) == 0) { R.nmask[((j >> 6) - 1) * R.ts] = nacc; nacc = 0; }
    };
    // head bytes up to 4-byte alignment, then whole words (4 bases per load), then the tail
    while (j < len && ((uintptr_t)(rd + j) & 3u)) put(rd[j]);
    while (j + 4 <= len) {
        const uint32_t w4 = *(const uint32_t *)(rd + j);
        // gather the four 2-bit codes / the four N flags (code 4) with one multiply each
        const uint32_t c4 = ((w4 & 0x03030303u) * 0x01041040u) >> 24;
        const uint32_t n4 = (((w4 >> 2) & 0x01010101u) * 0x10204080u) >> 28;
        if ((j & 31) <= 28 && (j & 63) <= 60) {
            acc |= (uint64_t)c4 << (2 * (j & 31));
            nacc |= (uint64_t)n4 << (j & 63);
            j += 4;
            if ((j & 31) == 0) { R.bits[((j >> 5) - 1) * R.ts] = acc; acc = 0; }
            if ((j & 63) == 0) { R.nmask[((j >> 6) - 1) * R.ts] = nacc; nacc = 0; }
        } else {
            put(w4 & 0xffu); put((w4 >> 8) & 0xffu); put((w4 >> 16) & 0xffu); put(w4 >> 24);
        }
    }
    while (j < len) put(rd[j]);
    if (j & 31) R.bits[(j >> 5) * R.ts] = acc;
    if (j & 63) R.nmask[(j >> 6) * R.ts] = nacc;
}

// The walk over one read's k-mer positions as a resumable state: seed_walk_step is one trip of the loop, so that a lane of the
// persistent kernel can take its next read the moment this one is finished instead of idling until the warp's slowest read ends.
struct SeedWalk {
    qm_seed *S;                     // the read's seed slots (global memory)
    int n, q, q_last;               // seeds so far, next k-mer start, last k-mer start (q > q_last: finished)
    int64_t trk_p;                  // forward position of the previous k-mer's only hit, -1 = none / several
    int64_t trk_p2;                 // >= 0: the previous k-mer had one hit per strand, trk_p (as is) and trk_p2 (reverse complement)
    int trk_pass;                   // strand of a lone hit: 0 = read k-mer as is, 1 = reverse complement
    // 2..4 hits of any strand mix (repeats in a few copies): all of them tracked, in look-up order
    int nt;
    int64_t tp[4];
    unsigned tpass;                 // bit t: strand of tracked hit t
    // the seed each strand is currently growing lives in registers (a clean read extends ONE seed ~120 times);
    // S[] in global memory is only touched when a seed is created, looked for, or handed back
    // (two named copies, one per strand, picked with selects: an array indexed by the strand would live in local memory)
    struct Cur { int64_t diag; int idx, len, qnext; } cur0, cur1;
    int last_ext;                   // start of the last k-mer that created or extended ANY seed (-2 = none yet): a hit at q can only
                                    // continue a seed when last_ext == q - 1, otherwise the seed list need not be searched
    int miss_run;                   // the last filter look-up missed (or a tracked match just broke): the next look-ups come in batches
};

// index of the seed on diagonal `diag` whose last k-mer starts at q - 1, or -1; S[0..n) scanned four entries per round trip
__device__ __forceinline__ int seed_find(const qm_seed *S, int n, int64_t diag, int q, int k)
{
    for (int m0 = 0; m0 < n; m0 += 4) {
        // (8-byte loads: a caller's seed array is only as aligned as the struct)
        int64_t rb[4];
        int2 ql[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const qm_seed *e = &S[m0 + i < QM_MAX_SEEDS ? m0 + i : QM_MAX_SEEDS - 1];
            rb[i] = e->rbeg; ql[i] = *(const int2 *)&e->qbeg;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (m0 + i < n && rb[i] - ql[i].x == diag && ql[i].x + ql[i].y - k + 1 == q) return m0 + i;
    }
    return -1;
}

__device__ __forceinline__ void seed_walk_init(SeedWalk &W, qm_seed *S, int len, int k)
{
    W.S = S; W.n = 0; W.q = 0; W.q_last = len - k;
    W.trk_p = -1; W.trk_p2 = -1; W.trk_pass = 0; W.nt = 0; W.tpass = 0;
    W.tp[0] = W.tp[1] = W.tp[2] = W.tp[3] = 0;
    W.cur0.diag = W.cur1.diag = 0;
    W.cur0.idx = W.cur1.idx = -1; W.cur0.len = W.cur1.len = 0; W.cur0.qnext = W.cur1.qnext = 0;
    W.miss_run = 0; W.last_ext = -2;
}

// the read's seed list and the two growing seeds (one per strand)
struct SeedList {
    const IndexView &V;
    SeedWalk &W;
    __device__ __forceinline__ void flush() const
    {
        if (W.cur0.idx >= 0) W.S[W.cur0.idx].len = W.cur0.len;
        if (W.cur1.idx >= 0) W.S[W.cur1.idx].len = W.cur1.len;
    }
    // is strand `pass` growing a seed on `diag` whose next k-mer starts at qq?
    __device__ __forceinline__ bool cur_is(int pass, int64_t diag, int qq) const
    {
        const int idx = pass ? W.cur1.idx : W.cur0.idx, qn = pass ? W.cur1.qnext : W.cur0.qnext;
        const int64_t d = pass ? W.cur1.diag : W.cur0.diag;
        return idx >= 0 && d == diag && qn == qq;
    }
    __device__ __forceinline__ void cur_grow(int pass, int m) const
    {
        if (pass) { W.cur1.len += m; W.cur1.qnext += m; } else { W.cur0.len += m; W.cur0.qnext += m; }
    }
    __device__ __forceinline__ void cur_set(int pass, int idx, int len, int64_t diag, int qnext) const
    {
        if (pass) { W.cur1.idx = idx; W.cur1.len = len; W.cur1.diag = diag; W.cur1.qnext = qnext; }
        else { W.cur0.idx = idx; W.cur0.len = len; W.cur0.diag = diag; W.cur0.qnext = qnext; }
    }
    __device__ __forceinline__ void add_hit(int pass, int64_t p, int q, bool single) const
    {
        const int k = V.k;
        qm_seed *S = W.S;
        const int64_t rpos = pass ? 2 * V.l_pac - p - k : p;
        const int64_t diag = rpos - q;
        if (single && cur_is(pass, diag, q)) { cur_grow(pass, 1); W.last_ext = q; return; }
        flush();
        const int m = W.last_ext >= q - 1 ? seed_find(S, W.n, diag, q, k) : -1;
        W.last_ext = q;
        if (m >= 0) { const int len = S[m].len + 1; S[m].len = len; cur_set(pass, m, len, diag, q + 1); }
        else if (W.n < QM_MAX_SEEDS) {
            S[W.n].rbeg = rpos; S[W.n].qbeg = q; S[W.n].len = k;
            cur_set(pass, W.n++, k, diag, q + 1);
        }
    }
};

// one trip: positions q .. of the read are decided (at least one), W.q moves on
__device__ __forceinline__ void seed_walk_step(const IndexView &V, const qm_opt &o, SeedWalk &W, const uint32_t *__restrict__ bloom /* V.bloom, or NULL */,
                                               const PackedRead &R, int bloom_batch)
{
    const int k = V.k;
    const uint32_t occ_cap = (uint32_t)(o.max_occ < QM_OCC_CAP ? o.max_occ : QM_OCC_CAP);
    const uint64_t mask = k < 32 ? ((1ull << (2 * k)) - 1) : ~0ull;
    const uint64_t kbits = k < 64 ? ((1ull << k) - 1) : ~0ull;
    qm_seed *S = W.S;
    int &n = W.n, &q = W.q, &trk_pass = W.trk_pass, &nt = W.nt;
    const int q_last = W.q_last;
    int64_t &trk_p = W.trk_p, &trk_p2 = W.trk_p2;
    int64_t (&tp)[4] = W.tp;
    unsigned &tpass = W.tpass;
    const SeedList SL = {V, W};
    auto flush = [&]() { SL.flush(); };
    auto cur_is = [&](int pass, int64_t diag, int qq) { return SL.cur_is(pass, diag, qq); };
    auto cur_grow = [&](int pass, int m) { SL.cur_grow(pass, m); };
    auto cur_set = [&](int pass, int idx, int len, int64_t diag, int qnext) { SL.cur_set(pass, idx, len, diag, qnext); };
    auto add_hit = [&](int pass, int64_t p, int q, bool single) { SL.add_hit(pass, p, q, single); };
    if (nt >= 2) {
        // every hit of position q-1 is tracked: position q+j has exactly these hits, one step further, as long as the new
        // read base continues ALL of them and the index says the reference k-mer there occurs nt times in total
        const int nb = q + k - 1;
        const uint64_t rbits = R.get2(nb);
        const uint32_t nbits = (uint32_t)R.getn(nb);
        int m = nbits ? __ffs((int)nbits) - 1 : 32;
        if (m > q_last - q + 1) m = q_last - q + 1;
        {
            const uint32_t *map = V.cnteqp[nt - 2];
            const uint32_t cm = (tpass & 1u) ? __brev(uniq_get(map, tp[0] - 32)) : uniq_get(map, tp[0] + 1);
            const int m_c = ~cm ? __ffs((int)~cm) - 1 : 32;
            m = m < m_c ? m : m_c;
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            if (t >= nt) break;
            const bool r = (tpass >> t) & 1u;
            const uint64_t x = rbits ^ (r ? ~qm_grouprev(ref_get2(V, tp[t] - 32)) : ref_get2(V, tp[t] + k));
            const uint64_t mm = (x | (x >> 1)) & 0x5555555555555555ull;
            const int m_b = mm ? (__ffsll((long long)mm) - 1) >> 1 : 32;
            const int64_t lim = r ? tp[t] : V.l_pac - k - tp[t];
            m = m < m_b ? m : m_b; m = (int64_t)m > lim ? (int)lim : m;
        }
        if (m > 0) {
            W.last_ext = q + m - 1;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                if (t >= nt) break;
                const int pass = (int)((tpass >> t) & 1u);
                const int64_t rpos = pass ? 2 * V.l_pac - tp[t] - k : tp[t];             // of the hit at q-1
                const int64_t diag = rpos - (q - 1);
                if (cur_is(pass, diag, q)) cur_grow(pass, m);
                else {
                    flush();
                    const int sidx = seed_find(S, n, diag, q, k);
                    if (sidx >= 0) { const int len = S[sidx].len + m; S[sidx].len = len; cur_set(pass, sidx, len, diag, q + m); }
                }
                tp[t] += pass ? -m : m;
            }
            q += m;
            if (m == 32) return;
            if (q > q_last) return;
        }
        // position q does not continue all of them: the general path below decides
        W.miss_run = 1;
    }
    if (trk_p >= 0) {
        // How many of the positions q, q+1, ... continue the match of position q-1 (at most 32 per step).  Tracked is
        // either the ONLY hit of that k-mer (trk_p on strand trk_pass; trk_p2 < 0) or its only hit on EACH strand
        // (forward-strand hit at trk_p, reverse-complement hit at trk_p2: inverted repeats).
        const int nb = q + k - 1;                   // index of the first new read base
        const uint64_t rbits = R.get2(nb);
        const uint32_t nbits = (uint32_t)R.getn(nb);
        int m = nbits ? __ffs((int)nbits) - 1 : 32;
        if (m > q_last - q + 1) m = q_last - q + 1;
        const bool two = trk_p2 >= 0;
        if (two || !trk_pass) {                     // a forward-strand hit at trk_p: positions p+1 .. l_pac-k
            const uint64_t x = rbits ^ ref_get2(V, trk_p + k);
            const uint64_t mm = (x | (x >> 1)) & 0x5555555555555555ull;
            const uint32_t ub = uniq_get(two ? V.uniq2p : V.uniqp, trk_p + 1);
            const int m_b = mm ? (__ffsll((long long)mm) - 1) >> 1 : 32, m_u = ~ub ? __ffs((int)~ub) - 1 : 32;
            const int64_t lim = V.l_pac - k - trk_p;
            m = m < m_b ? m : m_b; m = m < m_u ? m : m_u; m = (int64_t)m > lim ? (int)lim : m;
        }
        if (two || trk_pass) {                      // a reverse-complement hit at pr: positions pr-1 .. 0
            const int64_t pr = two ? trk_p2 : trk_p;
            const uint64_t x = rbits ^ ~qm_grouprev(ref_get2(V, pr - 32));
            const uint64_t mm = (x | (x >> 1)) & 0x5555555555555555ull;
            const int m_b = mm ? (__ffsll((long long)mm) - 1) >> 1 : 32;
            m = m < m_b ? m : m_b; m = (int64_t)m > pr ? (int)pr : m;
            if (!two) {
                const uint32_t ub = __brev(uniq_get(V.uniqp, pr - 32));
                const int m_u = ~ub ? __ffs((int)~ub) - 1 : 32;
                m = m < m_u ? m : m_u;
            }
        }
        if (m > 0) {
            auto grow = [&](int pass, int64_t p) {
                const int64_t rpos = pass ? 2 * V.l_pac - p - k : p;                 // of the hit at q-1
                if (cur_is(pass, rpos - (q - 1), q)) cur_grow(pass, m);
            };
            W.last_ext = q + m - 1;
            if (two) { grow(0, trk_p); grow(1, trk_p2); trk_p += m; trk_p2 -= m; }
            else { grow(trk_pass, trk_p); trk_p = trk_pass ? trk_p - m : trk_p + m; }
            q += m;
            if (m == 32) return;
            if (q > q_last) return;
        }
        // position q does not continue the match: the general path below decides (a mismatch: ~k positions in a row will miss)
        W.miss_run = 1;
    }
    const uint64_t nm = R.getn(q) & kbits;
    if (nm) {                                       // an N inside the k-mer: skip every k-mer that covers it
        trk_p = -1; trk_p2 = -1; nt = 0;
        q += 64 - __clzll((long long)nm);
        return;
    }
    if (bloom) {
        // A k-mer whose canonical form misses the filter occurs on neither strand: no table probe (the common case for
        // the k - 1 k-mers that cover a mismatch).  The filter words of kBloomBatch consecutive positions are fetched
        // TOGETHER: behind a mismatch ~k positions in a row miss, and probing them one by one is a chain of ~k dependent
        // L2 round trips per mismatch -- the bulk of this kernel's time -- where the batch pays one round trip per
        // kBloomBatch positions.  Only positions whose k-mer holds no N are in a batch (nm == 0 covers the first).
        // (one position at a time until a look-up misses: at a read's start and behind a repeat the first look-up usually hits)
        const int want = W.miss_run ? bloom_batch : 1;
        int gmax = q_last - q + 1 < want ? q_last - q + 1 : want;
        {
            const uint64_t nn = R.getn(q) >> k;                    // N flags of the bases behind the first k-mer
            const int free_n = nn ? __ffsll((long long)nn) : 64;   // positions q .. q+free_n-1 have an N-free k-mer
            gmax = gmax < free_n ? gmax : free_n;
        }
        uint32_t bw[kBloomBatch][3], bs[kBloomBatch][3];
#pragma unroll
        for (int g = 0; g < kBloomBatch; ++g) {
            if (g < gmax) {
                const uint64_t vg = R.get2(q + g) & mask;
                const uint64_t fg = qm_grouprev(vg) >> (64 - 2 * k), rg = ~vg & mask;
                uint32_t bp[3];
                qm_bloom_pos(fg < rg ? fg : rg, V.bloom_bits, bp);
#pragma unroll
                for (int t = 0; t < 3; ++t) { bw[g][t] = __ldg(&bloom[bp[t] >> 5]); bs[g][t] = bp[t] & 31; }
            }
        }
        unsigned hitmask = 0;
#pragma unroll
        for (int g = 0; g < kBloomBatch; ++g)
            if (g < gmax) hitmask |= ((bw[g][0] >> bs[g][0]) & (bw[g][1] >> bs[g][1]) & (bw[g][2] >> bs[g][2]) & 1u) << g;
        const int lead = hitmask ? __ffs((int)hitmask) - 1 : gmax;             // positions in a row that miss
        W.miss_run = lead == gmax;
        if (lead > 0) {
            trk_p = -1; trk_p2 = -1; nt = 0;
            q += lead;
            if (lead == gmax) return;
        }
        // position q passed the filter (and its k-mer holds no N)
    }
    const uint64_t v = R.get2(q) & mask;            // first base in the lowest bits
    const uint64_t fw = qm_grouprev(v) >> (64 - 2 * k);  // first base in the highest bits: the table's key order
    const uint64_t rc = ~v & mask;                  // reverse complement in the same order
    // the first table slot of both strands, fetched together (two dependent L2 round trips become one)
    const uint64_t slot0[2] = {(fw * 0x9E3779B97F4A7C15ull) >> V.shift, (rc * 0x9E3779B97F4A7C15ull) >> V.shift};
    const uint4 ent0[2] = {__ldg(&V.table[slot0[0]]), __ldg(&V.table[slot0[1]])};
    int n_hits = 0, one_pass = 0, n_pass[2] = {0, 0};
    int64_t one_p = -1, p_of[2] = {-1, -1};
    bool ignored = false;
    nt = 0; tpass = 0;
#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
        uint32_t first, cnt;
        if (!qm_idx_lookup_from(V, pass ? rc : fw, pass ? slot0[1] : slot0[0], pass ? ent0[1] : ent0[0], first, cnt)) continue;
        if (cnt > occ_cap) { n_hits += 2; ignored = true; continue; }          // ignored k-mer: nothing of this position is tracked
        for (uint32_t t = 0; t < cnt; ++t) {
            const int64_t p = cnt == 1 ? (int64_t)first : (int64_t)V.pos[first + t];
            add_hit(pass, p, q, cnt == 1);
            one_p = p; one_pass = pass; p_of[pass] = p;
            if (nt < 4) { if (nt == 0) tp[0] = p; else if (nt == 1) tp[1] = p; else if (nt == 2) tp[2] = p; else tp[3] = p; tpass |= (unsigned)pass << nt; }
            ++nt;
        }
        n_hits += (int)cnt; n_pass[pass] = (int)cnt;
    }
    trk_p = -1; trk_p2 = -1;
    if (n_hits == 1) { trk_p = one_p; trk_pass = one_pass; nt = 0; }
    else if (n_hits == 2 && n_pass[0] == 1 && n_pass[1] == 1) { trk_p = p_of[0]; trk_p2 = p_of[1]; trk_pass = 0; nt = 0; }
    else if (ignored || nt < 2 || nt > 4) nt = 0;                  // (otherwise: 2..4 hits, all tracked)
    ++q;
}

// seeds ordered by (qbeg, rbeg)
__device__ __forceinline__ void seed_sort(qm_seed *S, int n)
{
    for (int i = 1; i < n; ++i) {
        const qm_seed x = S[i];
        int j = i - 1;
        while (j >= 0 && (S[j].qbeg > x.qbeg || (S[j].qbeg == x.qbeg && S[j].rbeg > x.rbeg))) { S[j + 1] = S[j]; --j; }
        S[j + 1] = x;
    }
}

// the end of a read's walk: the growing seeds' lengths handed back; returns the number of seeds (in order of creation when
// `sorted` is false: the persistent kernel leaves the ordering to plan_kernel, where all lanes of a warp sort at the same time)
__device__ __forceinline__ int seed_walk_finish(SeedWalk &W, bool sorted = true)
{
    qm_seed *S = W.S;
    if (W.cur0.idx >= 0) S[W.cur0.idx].len = W.cur0.len;
    if (W.cur1.idx >= 0) S[W.cur1.idx].len = W.cur1.len;
    if (sorted) seed_sort(S, W.n);
    return W.n;
}

__device__ int collect_seeds(const IndexView &V, const qm_opt &o, const uint8_t *__restrict__ rd, int len, qm_seed *S,
                             const uint32_t *__restrict__ bloom /* V.bloom, or NULL */, PackedRead &R, int n_words, int n_nwords,
                             int bloom_batch = kBloomBatch)
{
    pack_read(rd, len, n_words, n_nwords, R);
    SeedWalk W;
    seed_walk_init(W, S, len, V.k);
    while (W.q <= W.q_last) seed_walk_step(V, o, W, bloom, R, bloom_batch);
    return seed_walk_finish(W);
}

__device__ __forceinline__ int seed_rid(const IndexView &V, const qm_seed &s)
{
    const int64_t f = s.rbeg >= V.l_pac ? 2 * V.l_pac - 1 - s.rbeg : s.rbeg;
    return qm_pos2rid(V, f);
}

// chains + filter -> plan (bwamem.c mem_chain, mem_chain_weight, mem_chain_flt, and the visiting order of
// mem_chain2aln).  Returns the number of plan entries.
__device__ int build_plan(const IndexView &V, const qm_opt &o, const qm_seed *S, int ns, uint16_t *plan)
{
    int64_t cpos[QM_MAX_SEEDS];
    uint8_t cfirst[QM_MAX_SEEDS], clast[QM_MAX_SEEDS], order[QM_MAX_SEEDS];
    int8_t crid[QM_MAX_SEEDS], chain_of[QM_MAX_SEEDS];
    int nc = 0;
    for (int i = 0; i < ns; ++i) {
        const qm_seed p = S[i];
        const int rid = seed_rid(V, p);
        int lower = -1;
        for (int kk = 0; kk < nc; ++kk) { if (cpos[order[kk]] <= p.rbeg) lower = kk; else break; }
        int res = 0;      // 0: new chain, 1: contained, 2: appended
        if (lower >= 0) {
            const int c = order[lower];
            const qm_seed first = S[cfirst[c]], last = S[clast[c]];
            const int64_t qend = last.qbeg + last.len, rend = last.rbeg + last.len;
            if (rid == crid[c]) {
                if (p.qbeg >= first.qbeg && p.qbeg + p.len <= qend && p.rbeg >= first.rbeg && p.rbeg + p.len <= rend) res = 1;
                else if ((last.rbeg < V.l_pac || first.rbeg < V.l_pac) && p.rbeg >= V.l_pac) res = 0;
                else {
                    const int64_t x = p.qbeg - last.qbeg, y = p.rbeg - last.rbeg;
                    if (y >= 0 && x - y <= o.w && y - x <= o.w && x - last.len < o.max_chain_gap && y - last.len < o.max_chain_gap) res = 2;
                }
            }
            if (res == 1) { chain_of[i] = -1; continue; }
            if (res == 2) { chain_of[i] = (int8_t)c; clast[c] = (uint8_t)i; continue; }
        }
        cpos[nc] = p.rbeg; crid[nc] = (int8_t)rid; cfirst[nc] = clast[nc] = (uint8_t)i; chain_of[i] = (int8_t)nc;
        const int at = lower + 1;
        for (int kk = nc; kk > at; --kk) order[kk] = order[kk - 1];
        order[at] = (uint8_t)nc++;
    }
    if (nc == 0) return 0;
    // weights (per chain, seeds in seed order)
    int cw[QM_MAX_SEEDS];
    for (int c = 0; c < nc; ++c) {
        int64_t end = 0;
        int w = 0, w2 = 0;
        for (int i = 0; i < ns; ++i) {
            if (chain_of[i] != c) continue;
            const qm_seed s = S[i];
            if (s.qbeg >= end) w += s.len; else if (s.qbeg + s.len > end) w += (int)(s.qbeg + s.len - end);
            if (s.qbeg + s.len > end) end = s.qbeg + s.len;
        }
        end = 0;
        for (int i = 0; i < ns; ++i) {
            if (chain_of[i] != c) continue;
            const qm_seed s = S[i];
            if (s.rbeg >= end) w2 += s.len; else if (s.rbeg + s.len > end) w2 += (int)(s.rbeg + s.len - end);
            if (s.rbeg + s.len > end) end = s.rbeg + s.len;
        }
        cw[c] = w2 < w ? w2 : w;
    }
    // B-tree order, weight filter, stable sort by weight descending
    uint8_t srt[QM_MAX_SEEDS];
    int m = 0;
    for (int kk = 0; kk < nc; ++kk) if (cw[order[kk]] >= o.min_chain_weight) srt[m++] = order[kk];
    for (int i = 1; i < m; ++i) {
        const uint8_t x = srt[i];
        int j = i - 1;
        while (j >= 0 && cw[srt[j]] < cw[x]) { srt[j + 1] = srt[j]; --j; }
        srt[j + 1] = x;
    }
    if (m == 0) return 0;
    uint8_t kept[QM_MAX_SEEDS], kept_idx[QM_MAX_SEEDS];
    int8_t firstsh[QM_MAX_SEEDS];
    for (int i = 0; i < m; ++i) { kept[i] = 0; firstsh[i] = -1; }
    int n_kept = 0;
    kept[0] = 3; kept_idx[n_kept++] = 0;
#define CBEG(i_) (S[cfirst[srt[i_]]].qbeg)
#define CEND(i_) (S[clast[srt[i_]]].qbeg + S[clast[srt[i_]]].len)
    for (int i = 1; i < m; ++i) {
        int large_ovlp = 0, kk;
        for (kk = 0; kk < n_kept; ++kk) {
            const int j = kept_idx[kk];
            const int b_max = CBEG(j) > CBEG(i) ? CBEG(j) : CBEG(i);
            const int e_min = CEND(j) < CEND(i) ? CEND(j) : CEND(i);
            if (e_min > b_max) {
                const int li = CEND(i) - CBEG(i), lj = CEND(j) - CBEG(j);
                const int min_l = li < lj ? li : lj;
                if (e_min - b_max >= min_l * o.mask_level && min_l < o.max_chain_gap) {
                    large_ovlp = 1;
                    if (firstsh[j] < 0) firstsh[j] = (int8_t)i;
                    if (cw[srt[i]] < cw[srt[j]] * o.drop_ratio && cw[srt[j]] - cw[srt[i]] >= o.min_seed_len << 1) break;
                }
            }
        }
        if (kk == n_kept) { kept_idx[n_kept++] = (uint8_t)i; kept[i] = large_ovlp ? 2 : 3; }
    }
#undef CBEG
#undef CEND
    for (int i = 0; i < n_kept; ++i) { const int j = kept_idx[i]; if (firstsh[j] >= 0) kept[firstsh[j]] = 1; }
    // plan: kept chains in sorted order; inside a chain seeds by descending (len, index in chain)
    int np = 0, ord = 0;
    for (int i = 0; i < m; ++i) {
        if (!kept[i]) continue;
        const int c = srt[i];
        const int base = np;
        for (int s = 0; s < ns; ++s) {
            if (chain_of[s] != c) continue;
            // insertion into descending order by (len, within)
            const int len = S[s].len;
            int j = np - 1;
            while (j >= base) {
                const int sj = plan[j] & 63;
                if (S[sj].len > len) break;         // equal length: the later seed (larger index) goes first
                plan[j + 1] = plan[j];
                --j;
            }
            plan[j + 1] = (uint16_t)(s | (ord << 6));
            ++np;
        }
        ++ord;
    }
    return np;
}

// The block's reads are consecutive rows of the batch: one contiguous span of blockDim.x * stride bytes.  One thread asks the
// copy engine for the whole span (cp.async.bulk: a single bulk-copy instruction, completion counted in bytes on an mbarrier)
// and every thread then packs its own read out of shared memory -- instead of 32 lanes walking 32 rows with 4-byte loads,
// ~40 dependent-latency trips through L1 per read.  The span is widened to 16-byte boundaries as the instruction demands;
// the few extra bytes lie inside the same 256-byte allocation granule.
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ const uint8_t *stage_block_reads(const uint8_t *__restrict__ codes, int stride, int64_t first, int n_rows,
                                                            uint8_t *stage, uint64_t *bar)
{
    const uint8_t *src = codes + first * stride;
    const unsigned head = (unsigned)((uintptr_t)src & 15u);
    const unsigned bytes = (head + (unsigned)n_rows * (unsigned)stride + 15u) & ~15u;
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(smem_addr(bar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_addr(bar)), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     :: "r"(smem_addr(stage)), "l"(src - head), "r"(bytes), "r"(smem_addr(bar)) : "memory");
    }
    __syncthreads();                                    // the barrier is initialised and armed for everybody
    unsigned done = 0;
    while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(smem_addr(bar)) : "memory");
    return stage + head;
}

__global__ void __launch_bounds__(kSeedThreads)
seed_chain_kernel(IndexView V, qm_opt o, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
                  int64_t n, qm_seed *__restrict__ seeds, int32_t *__restrict__ n_seeds, uint16_t *__restrict__ plan,
                  uint8_t *__restrict__ n_plan, ReadState *__restrict__ st, bool seeds_only, int n_words, int n_nwords, bool staged,
                  int bloom_batch)
{
    extern __shared__ __align__(16) uint64_t s_read[];   // [n_words][threads] packed bases, [n_nwords][threads] N flags, then the staged rows
    __shared__ uint64_t s_bar;
    const int64_t r0 = blockIdx.x * (int64_t)blockDim.x;
    const int64_t r = r0 + threadIdx.x;
    const uint8_t *rd = codes + r * stride;
    if (staged) {
        const int n_rows = n - r0 < (int64_t)blockDim.x ? (int)(n - r0) : (int)blockDim.x;
        rd = stage_block_reads(codes, stride, r0, n_rows, (uint8_t *)(s_read + (size_t)(n_words + n_nwords) * blockDim.x), &s_bar) +
             (size_t)threadIdx.x * stride;
    }
    if (r >= n) return;
    PackedRead R;
    R.bits = s_read + threadIdx.x;
    R.nmask = s_read + (size_t)n_words * blockDim.x + threadIdx.x;
    R.ts = (int)blockDim.x;
    qm_seed *S = seeds + r * QM_MAX_SEEDS;
    // the filter is read through L1/L2 (a copy in shared memory was measured: the 208 KB carve-out shrinks L1 to the point
    // where the chaining scratch thrashes -- 16.3 -> 23.8 ms per 4 M reads)
    const int ns = collect_seeds(V, o, rd, lens[r], S, V.bloom_bits ? V.bloom : nullptr, R, n_words, n_nwords, bloom_batch);
    n_seeds[r] = ns;
    if (seeds_only) return;
    const int np = build_plan(V, o, S, ns, plan + r * QM_MAX_SEEDS);
    n_plan[r] = (uint8_t)np;
    ReadState s;
    s.cursor = 0; s.phase = PH_NEXT; s.n_av = 0; s.task = -1;
    st[r] = s;
}

// ---- the seeding stage as three kernels (the default): pack, walk, plan ----
// pack_reads_kernel   the block's rows staged by one bulk copy, every thread packs its read (2 bits per base + N flags) and the
//                     block writes the packed words out coalesced: [read][n_words + n_nwords] 64-bit words.
// seed_walk_kernel    PERSISTENT: a lane walks one read's k-mer positions (seed_walk_step) and takes the next read off a global
//                     cursor when it is done.  Reads differ ~30x in work (mismatches, repeats); with one read per thread a warp
//                     lived as long as its slowest read with, on average, 15 of 32 lanes still walking.  Finished lanes wait until
//                     `refill` of them are idle (or nobody works) and fetch together: the refill is a short uniform burst of loads.
// plan_kernel         one thread per read: chains + filter -> plan (build_plan), the state machine's start state.
__global__ void __launch_bounds__(kSeedThreads)
pack_reads_kernel(const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens, int64_t n, uint64_t *__restrict__ packed,
                  int n_words, int n_nwords, bool staged)
{
    extern __shared__ __align__(16) uint64_t s_read[];
    __shared__ uint64_t s_bar;
    const int64_t r0 = blockIdx.x * (int64_t)blockDim.x;
    const int64_t r = r0 + threadIdx.x;
    const int pw = n_words + n_nwords;
    const int n_rows = n - r0 < (int64_t)blockDim.x ? (int)(n - r0) : (int)blockDim.x;
    const uint8_t *rd = codes + r * stride;
    if (staged) rd = stage_block_reads(codes, stride, r0, n_rows, (uint8_t *)(s_read + (size_t)pw * blockDim.x), &s_bar) + (size_t)threadIdx.x * stride;
    if (r < n) {
        PackedRead R;
        R.bits = s_read + threadIdx.x;
        R.nmask = s_read + (size_t)n_words * blockDim.x + threadIdx.x;
        R.ts = (int)blockDim.x;
        pack_read(rd, lens[r], n_words, n_nwords, R);
    }
    __syncthreads();
    uint64_t *out = packed + r0 * pw;
    for (int i = threadIdx.x; i < n_rows * pw; i += blockDim.x) {
        const int t = i / pw, w = i - t * pw;
        out[i] = s_read[(size_t)w * blockDim.x + t];
    }
}

template <int MINB>                                     // resident blocks of 64 threads asked of the compiler (register budget 65536 / 64 / MINB)
__global__ void __launch_bounds__(64, MINB)
seed_walk_kernel(IndexView V, qm_opt o, const uint64_t *__restrict__ packed, const int32_t *__restrict__ lens, int64_t n,
                 qm_seed *__restrict__ seeds, int32_t *__restrict__ n_seeds, int *__restrict__ cursor, int n_words, int n_nwords,
                 int bloom_batch, int refill, unsigned long long *__restrict__ dbg /* QM_SEED_DEBUG: per-read cycle / trip histograms, else NULL */)
{
    extern __shared__ __align__(16) uint64_t s_read[];   // [n_words + n_nwords][threads]: the lane's current read
    long long t_start = 0;
    int n_steps = 0;
    PackedRead R;
    R.bits = s_read + threadIdx.x;
    R.nmask = s_read + (size_t)n_words * blockDim.x + threadIdx.x;
    R.ts = (int)blockDim.x;
    const int pw = n_words + n_nwords;
    const uint32_t *bloom = V.bloom_bits ? V.bloom : nullptr;
    SeedWalk W;
    seed_walk_init(W, nullptr, 0, V.k);
    int64_t r = -1;                                      // the lane's read, -1 = none
    bool exhausted = false;
    int w_next = 0, w_end = 0;                           // the warp's range of reads (the same in every lane)
    bool w_dry = false;                                  // the global cursor has run past the last read
    const unsigned lane = threadIdx.x & 31u;
    for (;;) {
        const bool idle = r < 0;
        const unsigned idle_m = __ballot_sync(0xffffffffu, idle);
        const unsigned want_m = __ballot_sync(0xffffffffu, idle && !exhausted);
        if (idle_m == 0xffffffffu && want_m == 0u) break;
        if (want_m != 0u && (__popc(want_m) >= refill || idle_m == 0xffffffffu)) {
            // (Uniform branch: every lane keeps the same copy of the warp's range.)  The warp owns a range of reads [w_next, w_end)
            // taken off the global cursor kWalkRange at a time: most refills are served without the round trip of a global atomic.
            // When the range holds fewer reads than lanes want, the rest of the lanes are served on the next trip.
            if (w_next >= w_end && !w_dry) {
                int base = 0;
                if (lane == 0) base = atomicAdd(cursor, kWalkRange);
                base = __shfl_sync(0xffffffffu, base, 0);
                w_next = base; w_end = base + kWalkRange;
                if ((int64_t)w_next >= n) { w_dry = true; w_end = w_next; }
                else if ((int64_t)w_end > n) w_end = (int)n;
            }
            const int need = __popc(want_m), have = w_end - w_next;
            const int rank = __popc(want_m & ((1u << lane) - 1u));
            const bool mine = idle && !exhausted;
            const int64_t idx = (int64_t)w_next + rank;
            w_next += need < have ? need : have;
            if (mine && rank >= have) { if (w_dry) exhausted = true; }
            else if (mine) {
                r = idx;
                const uint64_t *src = packed + r * pw;
                for (int w = 0; w < pw; ++w) s_read[(size_t)w * blockDim.x + threadIdx.x] = __ldg(src + w);
                seed_walk_init(W, seeds + r * QM_MAX_SEEDS, lens[r], V.k);
                if (dbg) { t_start = clock64(); n_steps = 0; }
            }
        }
        if (r >= 0) {
            if (W.q <= W.q_last) { seed_walk_step(V, o, W, bloom, R, bloom_batch); ++n_steps; }
            if (W.q > W.q_last) {
                n_seeds[r] = seed_walk_finish(W, false); r = -1;
                if (dbg) {
                    const unsigned long long c = (unsigned long long)(clock64() - t_start);
                    const int bc = 63 - __clzll((long long)(c | 1ull)), bs = 31 - __clz(n_steps | 1);
                    atomicAdd(&dbg[bc & 31], 1ull); atomicAdd(&dbg[32 + (bc & 31)], c);
                    atomicAdd(&dbg[64 + bs], 1ull); atomicAdd(&dbg[96 + bs], c);
                }
            }
        }
    }
}

__global__ void __launch_bounds__(128)
plan_kernel(IndexView V, qm_opt o, int64_t n, qm_seed *__restrict__ seeds, const int32_t *__restrict__ n_seeds,
            uint16_t *__restrict__ plan, uint8_t *__restrict__ n_plan, ReadState *__restrict__ st, bool seeds_only)
{
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n) return;
    seed_sort(seeds + r * QM_MAX_SEEDS, n_seeds[r]);
    if (seeds_only) return;
    const int np = build_plan(V, o, seeds + r * QM_MAX_SEEDS, n_seeds[r], plan + r * QM_MAX_SEEDS);
    n_plan[r] = (uint8_t)np;
    ReadState s;
    s.cursor = 0; s.phase = PH_NEXT; s.n_av = 0; s.task = -1;
    st[r] = s;
}

// packed (n * (n_words + n_nwords) words of scratch) and cursor (one int of scratch) select the three-kernel form; without them
// (or with QM_SEED_PERSIST=0, for A/B measurements) the one-read-per-thread kernel runs
static cudaError_t launch_seed_chain(qm_ctx *ctx, const IndexView &V, const qm_opt &o, const uint8_t *codes, int stride, const int32_t *lens,
                                     int64_t n, qm_seed *seeds, int32_t *n_seeds, uint16_t *plan, uint8_t *n_plan, ReadState *st,
                                     bool seeds_only, cudaStream_t stream, uint64_t *packed = nullptr, int *cursor = nullptr)
{
    // packed read: one word per 32 bases + one spare (windows may start at the last base), N flags per 64 bases + one spare
    const int n_words = (stride + 31) / 32 + 2, n_nwords = (stride + 63) / 64 + 2;
    static const int threads = getenv("QM_SEED_THREADS") ? std::max(32, std::min(kSeedThreads, atoi(getenv("QM_SEED_THREADS")) & ~31)) : 64;   // tuning knob; 64: a block
    // lives as long as its slowest read (repeats), and smaller blocks give their slots back sooner (7.47 -> 7.13 ms per 4 M reads; 32: 7.35)
    const size_t smem_packed = (size_t)(n_words + n_nwords) * threads * sizeof(uint64_t);
    size_t smem = smem_packed;
    // the block's rows staged by one bulk copy (QM_SEED_STAGE=0: per-thread loads, for A/B measurements); very long rows stay
    // with the per-thread loads (the default 48 KB of dynamic shared memory)
    static const bool want_stage = !(getenv("QM_SEED_STAGE") && atoi(getenv("QM_SEED_STAGE")) == 0);
    const size_t stage_bytes = (size_t)threads * stride + 32;
    const bool staged = want_stage && smem + stage_bytes <= 40 * 1024;
    if (staged) smem += stage_bytes;
    static const int bloom_batch = getenv("QM_BLOOM_BATCH") ? std::max(1, std::min(kBloomBatch, atoi(getenv("QM_BLOOM_BATCH")))) : kBloomBatch;   // tuning knob
    static const bool want_persist = !(getenv("QM_SEED_PERSIST") && atoi(getenv("QM_SEED_PERSIST")) == 0);
    static const int refill = getenv("QM_SEED_REFILL") ? std::max(1, std::min(32, atoi(getenv("QM_SEED_REFILL")))) : 8;                           // tuning knob
    const unsigned blocks = (unsigned)((n + threads - 1) / threads);
    if (packed && cursor && want_persist && smem_packed <= 40 * 1024 && n <= 0x7fffffff - (1 << 22)) {
        cudaError_t e = cudaMemsetAsync(cursor, 0, sizeof(int), stream);
        if (e != cudaSuccess) return e;
        pack_reads_kernel<<<blocks, threads, smem, stream>>>(codes, stride, lens, n, packed, n_words, n_nwords, staged);
        // the walk is bound by the latency of dependent L2 look-ups: resident warps matter more than registers per thread
        static const int minb = getenv("QM_SEED_MINB") ? atoi(getenv("QM_SEED_MINB")) : 8;                                                        // tuning knob: 8 / 12 / 16
        auto walk = minb >= 16 ? seed_walk_kernel<16> : minb >= 12 ? seed_walk_kernel<12> : seed_walk_kernel<8>;
        const int wt = 64;                             // (its launch bounds)
        const size_t smem_walk = (size_t)(n_words + n_nwords) * wt * sizeof(uint64_t);
        static int per_sm[64] = {};                    // resident blocks of the walk kernel per SM, per device
        int &ps = per_sm[ctx->device & 63];
        if (ps == 0) {
            e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ps, walk, wt, smem_walk);
            if (e != cudaSuccess) return e;
            if (ps < 1) ps = 1;
        }
        const unsigned walk_blocks = std::min<unsigned>((unsigned)((n + wt - 1) / wt), (unsigned)(ctx->sm_count * ps));
        static const bool debug = getenv("QM_SEED_DEBUG") != nullptr;       // diagnostics: where the walk's time goes, read by read
        unsigned long long *dbg = nullptr;
        if (debug) { cudaMalloc(&dbg, 128 * 8); cudaMemsetAsync(dbg, 0, 128 * 8, stream); }
        walk<<<walk_blocks, wt, smem_walk, stream>>>(V, o, packed, lens, n, seeds, n_seeds, cursor, n_words, n_nwords, bloom_batch, refill, dbg);
        if (debug) {
            unsigned long long h[128];
            cudaMemcpyAsync(h, dbg, sizeof(h), cudaMemcpyDeviceToHost, stream); cudaStreamSynchronize(stream); cudaFree(dbg);
            fprintf(stderr, "[qm seed walk] %lld reads, %u blocks; per read: log2(cycles) bucket: reads, share of all cycles | log2(trips) bucket: reads, mean cycles\n", (long long)n, walk_blocks);
            unsigned long long tot = 0;
            for (int b = 0; b < 32; ++b) tot += h[32 + b];
            for (int b = 0; b < 32; ++b)
                if (h[b] || h[64 + b])
                    fprintf(stderr, "[qm seed walk]  2^%-2d cycles: %9llu reads %5.1f %% | 2^%-2d trips: %9llu reads, mean %10.0f cycles, %5.1f %%\n", b, h[b],
                            tot ? 100.0 * h[32 + b] / tot : 0.0, b, h[64 + b], h[64 + b] ? (double)h[96 + b] / h[64 + b] : 0.0, tot ? 100.0 * h[96 + b] / tot : 0.0);
        }
        plan_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(V, o, n, seeds, n_seeds, plan, n_plan, st, seeds_only);
        return cudaGetLastError();
    }
    seed_chain_kernel<<<blocks, threads, smem, stream>>>(
        V, o, codes, stride, lens, n, seeds, n_seeds, plan, n_plan, st, seeds_only, n_words, n_nwords, staged, bloom_batch);
    return cudaGetLastError();
}

// ---- bwa's own seeds (opt.flags & QM_F_FM_SEEDS): FM-index search of fm_core.cuh, one thread per read, then the same
// chaining.  The seeds come in mem_chain's order (not sorted by position): build_plan takes them as they are, like bwa. ----
struct CtgView { int n; const int64_t *off, *len; int64_t l_pac; };

__global__ void __launch_bounds__(128)
fm_seed_kernel(IndexView V, FmView F, qm_opt o, int max_mem_intv, const uint8_t *__restrict__ codes, int stride,
               const int32_t *__restrict__ lens, int64_t n, qm_seed *__restrict__ seeds, int32_t *__restrict__ n_seeds,
               uint16_t *__restrict__ plan, uint8_t *__restrict__ n_plan, ReadState *__restrict__ st, bool seeds_only)
{
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (r >= n) return;
    CtgView G = {V.n_contigs, V.off, V.len, V.l_pac};
    FmSeedOut tmp[QM_MAX_SEEDS];
    const int ns = fm_collect_seeds(F, G, o.min_seed_len, o.max_occ, max_mem_intv, lens[r], codes + r * stride, 1, tmp, QM_MAX_SEEDS);
    qm_seed *S = seeds + r * QM_MAX_SEEDS;
    for (int i = 0; i < ns; ++i) { qm_seed s; s.rbeg = tmp[i].rbeg; s.qbeg = tmp[i].qbeg; s.len = tmp[i].len; S[i] = s; }
    n_seeds[r] = ns;
    if (seeds_only) return;
    const int np = build_plan(V, o, S, ns, plan + r * QM_MAX_SEEDS);
    n_plan[r] = (uint8_t)np;
    ReadState s;
    s.cursor = 0; s.phase = PH_NEXT; s.n_av = 0; s.task = -1;
    st[r] = s;
}

static cudaError_t launch_fm_seed(const qm_index *idx, const qm_opt &o, const uint8_t *codes, int stride, const int32_t *lens, int64_t n,
                                  qm_seed *seeds, int32_t *n_seeds, uint16_t *plan, uint8_t *n_plan, ReadState *st, bool seeds_only,
                                  cudaStream_t stream)
{
    const int max_mem_intv = (o.flags & QM_F_FM_NO_ROUND3) ? 0 : 20;          // bwa's max_mem_intv
    fm_seed_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(idx->v, idx->fm, o, max_mem_intv, codes, stride, lens, n, seeds, n_seeds,
                                                                      plan, n_plan, st, seeds_only);
    return cudaGetLastError();
}

struct RoundCounters {        // zeroed before every advance round; the host reads back the first kRoundHeader bytes
    int class_count[kExtCtr];     // tasks per query-length class
    int class_cursor[kExtCtr];    // work cursors of the extension kernels
    int n_tasks;
    int tail_cursor;
    int max_score;            // max over the round's tasks of h0 + qlen * a: <= 255 lets the extension kernel hold eh[] in bytes
    int pad[5];
    int fb[2 * kExtCtr];      // fallback lists of the paired extension kernel: counts, then cursors
};
constexpr size_t kRoundHeader = (2 * kExtCtr + 8) * sizeof(int);

// the chain's reference window (mem_chain2aln rmax[], clamped to the contig as bns_fetch_seq does) and contig
struct ChainWin { int64_t rmax0, rmax1; int rid; };
__device__ ChainWin chain_window(const IndexView &V, const qm_opt &o, int lq, const qm_seed *S, const uint16_t *PL, int np, int chain,
                                 const qm_seed &sd)
{
    const int64_t l_pac = V.l_pac;
    int64_t rmax0 = l_pac << 1, rmax1 = 0;
    qm_seed first_seed = sd;
    int first_idx = 1 << 30;
    for (int i = 0; i < np; ++i) {
        if (((PL[i] >> 6) & 63) != chain) continue;
        const int si = PL[i] & 63;
        const qm_seed t = S[si];
        const int64_t b = t.rbeg - (t.qbeg + max_gap_for(o, t.qbeg));
        const int tail = lq - t.qbeg - t.len;
        const int64_t e = t.rbeg + t.len + (tail + max_gap_for(o, tail));
        rmax0 = b < rmax0 ? b : rmax0;
        rmax1 = e > rmax1 ? e : rmax1;
        if (si < first_idx) { first_idx = si; first_seed = t; }     // seed 0 of the chain = lowest seed index
    }
    rmax0 = rmax0 > 0 ? rmax0 : 0;
    rmax1 = rmax1 < l_pac << 1 ? rmax1 : l_pac << 1;
    if (rmax0 < l_pac && l_pac < rmax1) { if (first_seed.rbeg < l_pac) rmax1 = l_pac; else rmax0 = l_pac; }
    ChainWin W;
    const bool rev = first_seed.rbeg >= l_pac;
    const int64_t f = rev ? 2 * l_pac - 1 - first_seed.rbeg : first_seed.rbeg;
    W.rid = qm_pos2rid(V, f);
    int64_t far_beg = V.off[W.rid], far_end = V.off[W.rid] + V.len[W.rid];
    if (rev) { const int64_t t = far_beg; far_beg = (l_pac << 1) - far_end; far_end = (l_pac << 1) - t; }
    W.rmax0 = rmax0 > far_beg ? rmax0 : far_beg;
    W.rmax1 = rmax1 < far_end ? rmax1 : far_end;
    return W;
}
// the two extensions of a seed (mem_chain2aln): left of it (query and target reversed), then right of it with the left score as h0.
// A task is a function of the seed and its chain alone -- which is what lets the tail of a batch run them ahead of the
// state machine (spec_* kernels below).
__device__ __forceinline__ void left_task(const qm_opt &o, const uint8_t *query, const qm_seed &sd, const ChainWin &W, ExtTaskI *t)
{
    t->q = query + sd.qbeg - 1; t->qstep = -1; t->qlen = sd.qbeg;
    t->t = nullptr; t->t0 = sd.rbeg - 1; t->tstep = -1; t->tlen = (int)(sd.rbeg - W.rmax0);
    t->h0 = sd.len * o.a; t->w = o.w; t->end_bonus = o.pen_clip5;
    t->flags = QM_EXT_BAND_RETRY | QM_EXTI_INDIRECT;
}
__device__ __forceinline__ void right_task(const qm_opt &o, const uint8_t *query, int lq, const qm_seed &sd, const ChainWin &W, int h0,
                                           ExtTaskI *t)
{
    const int qe = sd.qbeg + sd.len;
    const int64_t re = sd.rbeg + sd.len;
    t->q = query + qe; t->qstep = 1; t->qlen = lq - qe;
    t->t = nullptr; t->t0 = re; t->tstep = 1; t->tlen = (int)(W.rmax1 - re);
    t->h0 = h0; t->w = o.w; t->end_bonus = o.pen_clip3;
    t->flags = QM_EXT_BAND_RETRY | QM_EXT_PREV_H0 | QM_EXTI_INDIRECT;
}

// ---- mem_chain2aln as a per-read state machine ----
// Consumes the result of the read's pending extension (xres, when the state is a WAIT state), then walks the plan
// until the next extension task is known (returns true, task in *t_out) or the read is finished (returns false,
// regions sorted / de-duplicated, *n_regs_out set).
__device__ bool advance_read(const IndexView &V, const qm_opt &o, const uint8_t *query, int lq, const qm_seed *S, uint16_t *PL,
                             int np, ReadState &s, qm_reg *av, int32_t *n_regs_out, const qm_ext_result *xres, int64_t r,
                             ExtTaskI *t_out, unsigned long long *cells /* caller's local sum, may be NULL */)
{
    if (s.phase == PH_WAIT_LEFT) {
        const qm_ext_result x = *xres;
        const qm_seed sd = S[PL[s.cursor] & 63];
        qm_reg *a = &av[s.n_av];
        if (cells) *cells += (unsigned long long)x.cells;
        a->score = x.score; a->w = x.w_used;
        if (x.gscore <= 0 || x.gscore <= x.score - o.pen_clip5) { a->qb = sd.qbeg - x.qle; a->rb = sd.rbeg - x.tle; a->truesc = x.score; }
        else { a->qb = 0; a->rb = sd.rbeg - x.gtle; a->truesc = x.gscore; }
        s.phase = PH_RIGHT;
    } else if (s.phase == PH_WAIT_RIGHT) {
        const qm_ext_result x = *xres;
        const qm_seed sd = S[PL[s.cursor] & 63];
        qm_reg *a = &av[s.n_av];
        const int sc0 = a->score;        // score before the right extension (= the task's h0)
        if (cells) *cells += (unsigned long long)x.cells;
        const int qe = sd.qbeg + sd.len;
        const int64_t re = sd.rbeg + sd.len;
        a->score = x.score;
        if (x.gscore <= 0 || x.gscore <= x.score - o.pen_clip3) { a->qe = qe + x.qle; a->re = re + x.tle; a->truesc += x.score - sc0; }
        else { a->qe = lq; a->re = re + x.gtle; a->truesc += x.gscore - sc0; }
        if (x.w_used > a->w) a->w = x.w_used;
        s.phase = PH_NEXT + 100;       // finalize marker
    }

    for (;;) {
        if (s.phase == PH_NEXT + 100) {
            // finalize the region in av[n_av]: seed coverage over the chain's seeds
            const int ent = PL[s.cursor];
            const int chain = (ent >> 6) & 63;
            qm_reg *a = &av[s.n_av];
            int cov = 0;
            for (int i = 0; i < np; ++i) {
                if (((PL[i] >> 6) & 63) != chain) continue;
                const qm_seed t = S[PL[i] & 63];
                if (t.qbeg >= a->qb && t.qbeg + t.len <= a->qe && t.rbeg >= a->rb && t.rbeg + t.len <= a->re) cov += t.len;
            }
            a->seedcov = cov;
            a->seedlen0 = S[ent & 63].len;
            ++s.n_av; ++s.cursor;
            s.phase = PH_NEXT;
        }
        if (s.phase == PH_NEXT) {
            // next seed of the plan that is not already explained by an existing region
            bool have = false;
            while (s.cursor < np) {
                const int ent = PL[s.cursor];
                const int chain = (ent >> 6) & 63;
                const qm_seed sd = S[ent & 63];
                int i;
                for (i = 0; i < s.n_av; ++i) {
                    const qm_reg *p = &av[i];
                    if (sd.rbeg < p->rb || sd.rbeg + sd.len > p->re || sd.qbeg < p->qb || sd.qbeg + sd.len > p->qe) continue;
                    if (sd.len - p->seedlen0 > .1 * lq) continue;
                    int qd = sd.qbeg - p->qb;
                    int64_t rd = sd.rbeg - p->rb;
                    int mg = max_gap_for(o, qd < rd ? qd : (int)rd);
                    int w = mg < p->w ? mg : p->w;
                    if (qd - rd < w && rd - qd < w) break;
                    qd = p->qe - (sd.qbeg + sd.len); rd = p->re - (sd.rbeg + sd.len);
                    mg = max_gap_for(o, qd < rd ? qd : (int)rd);
                    w = mg < p->w ? mg : p->w;
                    if (qd - rd < w && rd - qd < w) break;
                }
                bool skip = false;
                if (i < s.n_av) {
                    // covered: extend anyway only if an earlier-visited, extended seed of this chain overlaps it on
                    // a different diagonal
                    int j;
                    for (j = s.cursor - 1; j >= 0; --j) {
                        const int ej = PL[j];
                        if (((ej >> 6) & 63) != chain) break;       // plan entries of one chain are contiguous
                        if (ej & kPlanSkipped) continue;
                        const qm_seed t = S[ej & 63];
                        if (t.len < sd.len * .95) continue;
                        if (sd.qbeg <= t.qbeg && sd.qbeg + sd.len - t.qbeg >= sd.len >> 2 && t.qbeg - sd.qbeg != t.rbeg - sd.rbeg) break;
                        if (t.qbeg <= sd.qbeg && t.qbeg + t.len - sd.qbeg >= sd.len >> 2 && sd.qbeg - t.qbeg != sd.rbeg - t.rbeg) break;
                    }
                    if (j < 0 || ((PL[j] >> 6) & 63) != chain) skip = true;
                }
                if (!skip && s.n_av >= QM_MAX_REGS) skip = true;       // documented hard cap
                if (skip) { PL[s.cursor] = (uint16_t)(ent | kPlanSkipped); ++s.cursor; continue; }
                have = true;
                break;
            }
            if (!have) {
                *n_regs_out = qm_sort_dedup(o, s.n_av, av);
                s.phase = PH_DONE;
                return false;
            }
        }
        const int ent = PL[s.cursor];
        const qm_seed sd = S[ent & 63];
        const ChainWin W = chain_window(V, o, lq, S, PL, np, (ent >> 6) & 63, sd);
        const int rid = W.rid;
        ExtTaskI t;
        bool emit = false;
        if (s.phase == PH_NEXT) {
            qm_reg *a = &av[s.n_av];
            qm_reg z = {};
            z.w = o.w; z.score = z.truesc = -1; z.rid = rid; z.secondary = -1;
            *a = z;
            if (sd.qbeg) {
                left_task(o, query, sd, W, &t);
                emit = true;
                s.phase = PH_WAIT_LEFT;
            } else {
                a->score = a->truesc = sd.len * o.a; a->qb = 0; a->rb = sd.rbeg;
                s.phase = PH_RIGHT;
            }
        }
        if (s.phase == PH_RIGHT) {
            qm_reg *a = &av[s.n_av];
            if (sd.qbeg + sd.len != lq) {
                right_task(o, query, lq, sd, W, a->score, &t);
                emit = true;
                s.phase = PH_WAIT_RIGHT;
            } else {
                a->qe = lq; a->re = sd.rbeg + sd.len;
                s.phase = PH_NEXT + 100;
                continue;
            }
        }
        if (emit) {
            t.pad[0] = (int)r; t.pad[1] = 0;
            *t_out = t;
            return true;
        }
    }
}

// The round's counters sit at a handful of addresses (task count, 10 class counts, 512 length bins, the cell total, the
// score maximum) and every read that emits a task used to hit five of them with its own atomic: two million same-address
// atomics per round, serialised in L2.  They are combined first -- per block in shared memory for the bins, per warp for
// the task slots, the cell sum and the maximum -- so that a block issues a few dozen global atomics instead of hundreds.
__global__ void __launch_bounds__(128)
advance_kernel(IndexView V, qm_opt o, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
               int64_t n, const qm_seed *__restrict__ seeds, uint16_t *__restrict__ plan, const uint8_t *__restrict__ n_plan,
               ReadState *__restrict__ st, qm_reg *__restrict__ regs, int32_t *__restrict__ n_regs,
               const qm_ext_result *__restrict__ res, ExtTaskI *__restrict__ tasks, uint64_t *__restrict__ keys,
               RoundCounters *__restrict__ ctr, unsigned long long *__restrict__ cells)
{
    __shared__ int s_class[kExtCtr];
    if (threadIdx.x < kExtCtr) s_class[threadIdx.x] = 0;
    __syncthreads();
    const int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int lane = qm_lane();
    ReadState s;
    bool live = r < n;
    if (live) { s = st[r]; live = s.phase != PH_DONE; }
    ExtTaskI t;
    unsigned long long my_cells = 0;
    bool emit = false;
    if (live)
        emit = advance_read(V, o, codes + r * stride, lens[r], seeds + r * QM_MAX_SEEDS, plan + r * QM_MAX_SEEDS, n_plan[r], s,
                            regs + r * QM_MAX_REGS, n_regs + r, s.task >= 0 ? res + s.task : nullptr, r, &t, &my_cells);
    // task slots: one atomic per warp
    const unsigned em = __ballot_sync(0xffffffffu, emit);
    int base = 0;
    if (lane == 0 && em) base = atomicAdd(&ctr->n_tasks, __popc(em));
    base = __shfl_sync(0xffffffffu, base, 0);
    int score = 0;
    if (emit) {
        const int slot = base + __popc(em & ((1u << lane) - 1u));
        tasks[slot] = t;
        keys[slot] = qm_ext_sort_key(t.qlen, t.tlen, t.h0);
        atomicAdd(&s_class[qm_ext_class(t.qlen)], 1);
        score = t.h0 + t.qlen * o.a;
        s.task = slot;
    }
    if (live) st[r] = s;
    const int wmax = __reduce_max_sync(0xffffffffu, score);
    if (lane == 0 && wmax > 0) atomicMax(&ctr->max_score, wmax);
    if (cells) {
        // 64-bit sum over the warp
        unsigned long long v = my_cells;
        for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
        if (lane == 0 && v) atomicAdd(cells, v);
    }
    __syncthreads();
    if (threadIdx.x < kExtCtr && s_class[threadIdx.x]) atomicAdd(&ctr->class_count[threadIdx.x], s_class[threadIdx.x]);
}

// ---- tail: the reads still active after the bulk rounds (reads with many chains, up to 2 x QM_MAX_REGS dependent
// extensions each) are finished by ONE WARP PER READ without further host round trips: the warp runs the pending
// extension with the warp-wide kernel body (ext_warp.cuh), lane 0 feeds the result to the state machine, repeat. ----
template <int C>
__device__ __forceinline__ qm_ext_result tail_extend(const ExtParams &P, const IndexView &V, const ExtTaskI &t, int lane)
{
    SeqFetch F;
    F.q = t.q; F.t = t.t; F.t0 = t.t0; F.qstep = t.qstep; F.tstep = t.tstep;
    F.indirect = (t.flags & QM_EXTI_INDIRECT) != 0; F.V = &V;
    ExtState r;
    int w_used = t.w, cells = 0, prev = (t.flags & QM_EXT_PREV_H0) ? t.h0 : -1;
    const int tries = (t.flags & QM_EXT_BAND_RETRY) ? 2 : 1;
    for (int a = 0; a < tries; ++a) {
        w_used = t.w << a;
        r = ext_run<C>(P, F, t.qlen, t.tlen, t.h0, w_used, t.end_bonus, lane);
        cells += r.cells;
        if (r.score == prev || r.max_off < (w_used >> 1) + (w_used >> 2)) break;
        prev = r.score;
    }
    qm_ext_result x;
    x.score = r.score; x.qle = r.qle; x.tle = r.tle; x.gtle = r.gtle; x.gscore = r.gscore; x.max_off = r.max_off;
    x.w_used = w_used; x.cells = cells;
    return x;
}

constexpr int kTailWarps = 4;
constexpr int kTailMinTasks = 32768;        // a round with fewer tasks hands the still-active reads to tail_kernel

// MAXC = 4: only queries of <= 127 bases (every extension of a 150-base read) -- the warp-wide extension then keeps four
// column slots per lane in registers instead of sixteen and four times as many warps fit on an SM.  A read whose next
// extension is longer is parked (its state written back, the task appended to `over`) for the MAXC = 16 launch behind.
template <int MAXC>
__global__ void __launch_bounds__(kTailWarps * 32)
tail_kernel(IndexView V, qm_opt o, ExtParams P, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
            const qm_seed *__restrict__ seeds, uint16_t *__restrict__ plan, const uint8_t *__restrict__ n_plan,
            ReadState *__restrict__ st, qm_reg *__restrict__ regs, int32_t *__restrict__ n_regs,
            const ExtTaskI *__restrict__ tasks, int n_tasks_host, const int *__restrict__ n_tasks_dev, int *__restrict__ cursor,
            unsigned long long *__restrict__ cells, ExtTaskI *__restrict__ over, int *__restrict__ n_over)
{
    __shared__ ExtTaskI s_task[kTailWarps];
    __shared__ qm_ext_result s_res[kTailWarps];
    __shared__ int s_more[kTailWarps];
    const int lane = qm_lane(), wib = threadIdx.x >> 5;
    const int n_tasks = n_tasks_dev ? *n_tasks_dev : n_tasks_host;
    unsigned long long my_cells = 0;               // lane 0: executed cells of this warp's reads, added once at the end
    for (;;) {
        int slot = 0;
        if (lane == 0) slot = atomicAdd(cursor, 1);
        slot = __shfl_sync(0xffffffffu, slot, 0);
        if (slot >= n_tasks) break;
        if (lane == 0) s_task[wib] = tasks[slot];
        __syncwarp();
        const int64_t r = s_task[wib].pad[0];
        ReadState s;
        if (lane == 0) s = st[r];
        bool parked = false;
        for (;;) {
            const ExtTaskI t = s_task[wib];
            if (MAXC < 16 && t.qlen > 127) {            // too long for this instantiation: park the read (warp-uniform)
                if (lane == 0) { const int k = atomicAdd(n_over, 1); over[k] = t; s.task = k; st[r] = s; }
                parked = true;
                break;
            }
            qm_ext_result x;
            // column slots per lane by query length (warp-uniform): every row costs C cell updates per lane whatever the band
            if (t.qlen <= 31) x = tail_extend<1>(P, V, t, lane);
            else if (t.qlen <= 63) x = tail_extend<2>(P, V, t, lane);
            else if (t.qlen <= 95) x = tail_extend<3>(P, V, t, lane);
            else if (MAXC < 16 || t.qlen <= 127) x = tail_extend<4>(P, V, t, lane);
            else if (t.qlen <= 287) x = tail_extend<9>(P, V, t, lane);
            else x = tail_extend<16>(P, V, t, lane);
            __syncwarp();
            if (lane == 0) {
                s_res[wib] = x;
                ExtTaskI nt;
                const bool more = advance_read(V, o, codes + r * stride, lens[r], seeds + r * QM_MAX_SEEDS, plan + r * QM_MAX_SEEDS,
                                               n_plan[r], s, regs + r * QM_MAX_REGS, n_regs + r, &s_res[wib], r, &nt, &my_cells);
                if (more) s_task[wib] = nt;
                s_more[wib] = more ? 1 : 0;
            }
            __syncwarp();
            if (!s_more[wib]) break;
        }
        if (lane == 0 && !parked) { s.task = -1; st[r] = s; }
        __syncwarp();
    }
    if (lane == 0 && cells && my_cells) atomicAdd(cells, my_cells);
}

// ---- speculative finish of a batch's last reads ----
// After the bulk rounds only reads with many seeds are left (tandem repeats, terminal repeats: up to 2 x QM_MAX_REGS DEPENDENT
// extensions each), and the batch waits for the longest such chain: extension after extension, each ~150 rows of a latency-bound
// kernel (round 1's tail_kernel: 3.3 ms for 2 % of the cells, plus the three small rounds before it).  But an extension task is
// a function of its seed and chain alone (left_task / right_task); what depends on earlier results is only whether
// mem_chain2aln SKIPS the seed.  So every remaining seed of these reads is extended ahead of time, all at once, by the
// throughput kernels -- left sides in one launch group, right sides (h0 = the left score) in a second -- and the state machine
// then runs to the end on results that are already there.  Results of seeds it skips are discarded (and not counted as cells).
// Same regions as the serial order, bit for bit; the dependent chain shrinks from dozens of extensions to two.
constexpr int kSpecMinTasks = 1 << 17;       // a round with fewer tasks switches to this mode (rows of the directory)
constexpr int kSpecCap = 1 << 20;             // tasks per launch group
constexpr int kSpecDirRow = 2 * QM_MAX_SEEDS; // directory entries per read: [plan index][side]
static_assert(QM_MAX_SEEDS <= 64, "plan index must fit the 6 bits of ExtTaskI::pad[1]");

struct SpecScratch {
    ExtTaskI *tasks;            // [2 * kSpecCap]: group A (pending + left sides + right sides of seeds without a left), group B at kSpecCap
    qm_ext_result *res;         // [2 * kSpecCap]
    uint64_t *keys;             // [2 * kSpecCap]
    int *lists;                 // [2 * kSpecCap] sorted lists, then the fallback lists [2][kExtClasses][kSpecCap]
    int *dir;                   // [kSpecMinTasks][kSpecDirRow]: slot of the task of (read, plan index, side), -1 = none
    int *meta;                  // [kSpecMinTasks]: lo | hi << 8: plan indices [lo, hi) of the read are in the directory
    ExtTaskI *next_tasks;       // [kSpecMinTasks]: what the next pass starts from (reads that ran past their directory)
    uint64_t *next_keys;
    RoundCounters *ctr;         // [3]: group A, group B, next pass
};

__device__ __forceinline__ void spec_emit(const ExtTaskI &t, int slot, ExtTaskI *tasks, uint64_t *keys, RoundCounters *ctr, const qm_opt &o)
{
    tasks[slot] = t;
    keys[slot] = qm_ext_sort_key(t.qlen, t.tlen, t.h0);
    atomicAdd(&ctr->class_count[qm_ext_class(t.qlen)], 1);
    atomicMax(&ctr->max_score, t.h0 + t.qlen * o.a);
}

// one thread per pending task (= per active read): enter it and every later seed of the read's plan into group A
__global__ void __launch_bounds__(128)
spec_plan_kernel(IndexView V, qm_opt o, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
                 const qm_seed *__restrict__ seeds, const uint16_t *__restrict__ plan, const uint8_t *__restrict__ n_plan,
                 const ReadState *__restrict__ st, int n_active, int depth, SpecScratch X)
{
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_active) return;
    RoundCounters *ctr = X.ctr;
    const int64_t r = X.tasks[row].pad[0];
    const ReadState s = st[r];
    const qm_seed *S = seeds + r * QM_MAX_SEEDS;
    const uint16_t *PL = plan + r * QM_MAX_SEEDS;
    const int np = n_plan[r], lq = lens[r];
    const uint8_t *query = codes + r * stride;
    int *d = X.dir + (size_t)row * kSpecDirRow;
    const int lo = s.cursor, side0 = s.phase == PH_WAIT_RIGHT ? 1 : 0;
    d[2 * lo + side0] = row; d[2 * lo + 1 - side0] = -1;
    X.tasks[row].pad[1] = row << 8 | lo << 1 | side0;
    int hi = lo + 1;
    for (int i = lo + 1; i < np && i <= lo + depth; ++i) {
        const int ent = PL[i];
        const qm_seed sd = S[ent & 63];
        int side = -1;
        ExtTaskI t;
        if (sd.qbeg) side = 0; else if (sd.qbeg + sd.len != lq) side = 1;
        if (side >= 0) {
            const int slot = atomicAdd(&ctr->n_tasks, 1);
            if (slot >= kSpecCap) break;                // group full: the rest of this read waits for the next pass
            const ChainWin W = chain_window(V, o, lq, S, PL, np, (ent >> 6) & 63, sd);
            if (side == 0) left_task(o, query, sd, W, &t); else right_task(o, query, lq, sd, W, sd.len * o.a, &t);
            t.pad[0] = (int)r; t.pad[1] = row << 8 | i << 1 | side;
            spec_emit(t, slot, X.tasks, X.keys, ctr, o);
            d[2 * i + side] = slot; d[2 * i + 1 - side] = -1;
        } else { d[2 * i] = -1; d[2 * i + 1] = -1; }
        hi = i + 1;
    }
    X.meta[row] = lo | hi << 8;
}

// one thread per task of group A: a left side that has run gives its seed's right side (group B)
__global__ void __launch_bounds__(128)
spec_right_kernel(IndexView V, qm_opt o, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
                  const qm_seed *__restrict__ seeds, const uint16_t *__restrict__ plan, const uint8_t *__restrict__ n_plan, int n_a, SpecScratch X)
{
    const int ta = blockIdx.x * blockDim.x + threadIdx.x;
    if (ta >= n_a) return;
    const int tag = X.tasks[ta].pad[1];
    if (tag & 1) return;
    const int i = (tag >> 1) & 63, row = tag >> 8;
    const int64_t r = X.tasks[ta].pad[0];
    const qm_seed *S = seeds + r * QM_MAX_SEEDS;
    const uint16_t *PL = plan + r * QM_MAX_SEEDS;
    const int ent = PL[i], lq = lens[r];
    const qm_seed sd = S[ent & 63];
    if (sd.qbeg + sd.len == lq) return;
    RoundCounters *ctr = X.ctr + 1;
    const int slot = atomicAdd(&ctr->n_tasks, 1);       // <= n_a <= kSpecCap
    const ChainWin W = chain_window(V, o, lq, S, PL, n_plan[r], (ent >> 6) & 63, sd);
    ExtTaskI t;
    right_task(o, codes + r * stride, lq, sd, W, X.res[ta].score, &t);
    t.pad[0] = (int)r; t.pad[1] = row << 8 | i << 1 | 1;
    spec_emit(t, slot, X.tasks + kSpecCap, X.keys + kSpecCap, ctr, o);
    X.dir[(size_t)row * kSpecDirRow + 2 * i + 1] = kSpecCap + slot;
}

// one thread per active read: the state machine, fed from the directory, to the end of the plan (or of the directory)
__global__ void __launch_bounds__(128)
spec_finish_kernel(IndexView V, qm_opt o, const uint8_t *__restrict__ codes, int stride, const int32_t *__restrict__ lens,
                   const qm_seed *__restrict__ seeds, uint16_t *__restrict__ plan, const uint8_t *__restrict__ n_plan,
                   ReadState *__restrict__ st, qm_reg *__restrict__ regs, int32_t *__restrict__ n_regs, int n_active, SpecScratch X,
                   unsigned long long *__restrict__ cells)
{
    const int row = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long my_cells = 0;
    if (row < n_active) {
        const int64_t r = X.tasks[row].pad[0];
        ReadState s = st[r];
        const int meta = X.meta[row], lo = meta & 255, hi = meta >> 8;
        const int *d = X.dir + (size_t)row * kSpecDirRow;
        const qm_ext_result *xres = X.res + row;
        RoundCounters *ctr = X.ctr + 2;
        for (;;) {
            ExtTaskI t;
            const bool more = advance_read(V, o, codes + r * stride, lens[r], seeds + r * QM_MAX_SEEDS, plan + r * QM_MAX_SEEDS, n_plan[r],
                                           s, regs + r * QM_MAX_REGS, n_regs + r, xres, r, &t, &my_cells);
            if (!more) { s.task = -1; break; }
            const int i = s.cursor, side = s.phase == PH_WAIT_RIGHT ? 1 : 0;
            const int slot = (i >= lo && i < hi) ? d[2 * i + side] : -1;
            if (slot < 0) {                              // past the directory: this task opens the read's next pass
                const int k = atomicAdd(&ctr->n_tasks, 1);
                spec_emit(t, k, X.next_tasks, X.next_keys, ctr, o);
                s.task = k;
                break;
            }
            xres = X.res + slot;
        }
        st[r] = s;
    }
    if (cells) {
        unsigned long long v = my_cells;
        for (int dd = 16; dd > 0; dd >>= 1) v += __shfl_down_sync(0xffffffffu, v, dd);
        if (qm_lane() == 0 && v) atomicAdd(cells, v);
    }
}

constexpr int kMaxStride = 512;               // longest row the read-level entries take (the extension's queries stop at QM_EXT_MAX_QLEN)
constexpr int64_t kSeBatch = 1 << 22;         // a round with fewer tasks hands the still-active reads to tail_kernel       // reads per internal round-trip (bounds scratch memory)

struct SeScratch {
    qm_seed *seeds; int32_t *n_seeds; uint16_t *plan; uint8_t *n_plan; ReadState *st;
    ExtTaskI *tasks; qm_ext_result *res; int *lists; uint64_t *keys; RoundCounters *ctr; RoundCounters *h_ctr;
    uint64_t *packed; size_t packed_words; int *cursors;        // the seeding stage's packed reads (per read: packed_words) and read cursors
};

int se_scratch(qm_ctx *ctx, int64_t nb, int stride, SeScratch *sc)
{
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_seeds = take((size_t)nb * QM_MAX_SEEDS * sizeof(qm_seed));
    const size_t o_ns = take((size_t)nb * 4);
    const size_t o_plan = take((size_t)nb * QM_MAX_SEEDS * 2);
    const size_t o_np = take((size_t)nb);
    const size_t o_st = take((size_t)nb * sizeof(ReadState));
    const size_t o_tasks = take((size_t)(nb + kTailMinTasks) * sizeof(ExtTaskI));       // + the tail kernel's parked tasks
    const size_t o_res = take((size_t)nb * sizeof(qm_ext_result));
    const size_t o_lists = take((size_t)nb * (1 + kExtClasses) * 4);   // the round's sorted task list, then the fallback lists
    const size_t o_keys = take((size_t)nb * 8);
    const size_t o_ctr = take(sizeof(RoundCounters));
    const size_t pw = (size_t)((stride + 31) / 32 + 2 + (stride + 63) / 64 + 2);
    const size_t o_packed = take((size_t)nb * pw * 8), o_cursors = take(64 * sizeof(int));
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 3, off, &p);
    if (rc) return rc;
    char *b = (char *)p;
    sc->seeds = (qm_seed *)(b + o_seeds); sc->n_seeds = (int32_t *)(b + o_ns); sc->plan = (uint16_t *)(b + o_plan);
    sc->n_plan = (uint8_t *)(b + o_np); sc->st = (ReadState *)(b + o_st); sc->tasks = (ExtTaskI *)(b + o_tasks);
    sc->res = (qm_ext_result *)(b + o_res); sc->lists = (int *)(b + o_lists); sc->keys = (uint64_t *)(b + o_keys); sc->ctr = (RoundCounters *)(b + o_ctr);
    sc->packed = (uint64_t *)(b + o_packed); sc->packed_words = pw; sc->cursors = (int *)(b + o_cursors);
    return QM_OK;
}

// have all pieces of the batch the host entry announced arrived?
bool se_parts_landed(qm_ctx *ctx)
{
    for (int pt = 0; pt < ctx->se_n_parts; ++pt)
        if (cudaEventQuery(ctx->se_part_ev[pt]) != cudaSuccess) { (void)cudaGetLastError(); return false; }
    return true;
}

int spec_scratch(qm_ctx *ctx, SpecScratch *X)
{
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_tasks = take((size_t)2 * kSpecCap * sizeof(ExtTaskI)), o_res = take((size_t)2 * kSpecCap * sizeof(qm_ext_result));
    const size_t o_keys = take((size_t)2 * kSpecCap * 8), o_lists = take((size_t)(2 + 2 * kExtClasses) * kSpecCap * 4);
    const size_t o_dir = take((size_t)kSpecMinTasks * kSpecDirRow * 4), o_meta = take((size_t)kSpecMinTasks * 4);
    const size_t o_nt = take((size_t)kSpecMinTasks * sizeof(ExtTaskI)), o_nk = take((size_t)kSpecMinTasks * 8), o_ctr = take(3 * sizeof(RoundCounters));
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 26, off, &p);
    if (rc) return rc;
    char *b = (char *)p;
    X->tasks = (ExtTaskI *)(b + o_tasks); X->res = (qm_ext_result *)(b + o_res); X->keys = (uint64_t *)(b + o_keys); X->lists = (int *)(b + o_lists);
    X->dir = (int *)(b + o_dir); X->meta = (int *)(b + o_meta); X->next_tasks = (ExtTaskI *)(b + o_nt); X->next_keys = (uint64_t *)(b + o_nk);
    X->ctr = (RoundCounters *)(b + o_ctr);
    return QM_OK;
}

// sort one launch group by (query length, rows, seed score) and run it through the class kernels
int spec_run_group(qm_ctx *ctx, const ExtParams &P, const IndexView &V, SpecScratch &X, int g, int n, const RoundCounters *h_ctr, cudaStream_t st)
{
    const size_t base = (size_t)g * kSpecCap;
    int sp = qm_prof_begin(ctx, QM_ST_ADVANCE, st);
    int rc = qm_sort_pairs(ctx, X.keys + base, (uint32_t *)(X.lists + base), n, kExtSortKeyBits, st);
    qm_prof_end(ctx, QM_ST_ADVANCE, sp, st, 0);
    if (rc) return rc;
    int64_t list_off[kExtClasses];
    int n_launch = 0;
    { int64_t acc = 0; for (int c = 0; c < kExtClasses; ++c) { list_off[c] = acc; acc += h_ctr->class_count[c]; n_launch += h_ctr->class_count[c] > 0; } }
    sp = qm_prof_begin(ctx, QM_ST_EXTEND, st);
    rc = qm_ext_launch_classes(ctx, P, V, X.tasks + base, X.lists + base, kSpecCap, X.ctr[g].class_count, X.ctr[g].class_cursor, h_ctr->class_count,
                               X.res + base, X.lists + (size_t)(2 + g * kExtClasses) * kSpecCap, X.ctr[g].fb, st, h_ctr->max_score <= 255, list_off);
    qm_prof_end(ctx, QM_ST_EXTEND, sp, st, n_launch);
    return rc;
}

// the reads still active (their pending tasks are sc.tasks[0 .. n_active), counters sc.ctr) run to the end of their plans
int spec_finish_batch(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const ExtParams &P, const uint8_t *codes, int stride, const int32_t *lens,
                      const SeScratch &sc, qm_reg *regs, int32_t *n_regs, int64_t *d_cells, RoundCounters *h_ctr, int n_active, cudaStream_t st)
{
    SpecScratch X;
    int rc = spec_scratch(ctx, &X);
    if (rc) return rc;
    static const int depth = getenv("QM_SPEC_DEPTH") ? atoi(getenv("QM_SPEC_DEPTH")) : QM_MAX_SEEDS;      // test knob: seeds entered ahead per pass
    static const bool spec_log = getenv("QM_ROUND_LOG") != nullptr;
    QM_CUDA(ctx, cudaMemcpyAsync(X.tasks, sc.tasks, (size_t)n_active * sizeof(ExtTaskI), cudaMemcpyDeviceToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync(X.keys, sc.keys, (size_t)n_active * 8, cudaMemcpyDeviceToDevice, st));
    QM_CUDA(ctx, cudaMemcpyAsync(X.ctr, sc.ctr, sizeof(RoundCounters), cudaMemcpyDeviceToDevice, st));
    for (int pass = 0; pass < 4 * QM_MAX_REGS + 8; ++pass) {
        const unsigned grid = (unsigned)((n_active + 127) / 128);
        int sp = qm_prof_begin(ctx, QM_ST_ADVANCE, st);
        QM_CUDA(ctx, cudaMemsetAsync(X.ctr + 1, 0, 2 * sizeof(RoundCounters), st));
        spec_plan_kernel<<<grid, 128, 0, st>>>(idx->v, *opt, codes, stride, lens, sc.seeds, sc.plan, sc.n_plan, sc.st, n_active, depth, X);
        qm_prof_end(ctx, QM_ST_ADVANCE, sp, st, 1);
        QM_CUDA(ctx, cudaMemcpyAsync(h_ctr, X.ctr, kRoundHeader, cudaMemcpyDeviceToHost, st));
        QM_CUDA(ctx, cudaStreamSynchronize(st));
        const int n_a = h_ctr->n_tasks < kSpecCap ? h_ctr->n_tasks : kSpecCap;
        if (spec_log) fprintf(stderr, "[qm spec pass %d] reads %d group A %d", pass, n_active, n_a);
        rc = spec_run_group(ctx, P, idx->v, X, 0, n_a, h_ctr, st);
        if (rc) return rc;
        sp = qm_prof_begin(ctx, QM_ST_ADVANCE, st);
        spec_right_kernel<<<(unsigned)((n_a + 127) / 128), 128, 0, st>>>(idx->v, *opt, codes, stride, lens, sc.seeds, sc.plan, sc.n_plan, n_a, X);
        qm_prof_end(ctx, QM_ST_ADVANCE, sp, st, 1);
        QM_CUDA(ctx, cudaMemcpyAsync(h_ctr, X.ctr + 1, kRoundHeader, cudaMemcpyDeviceToHost, st));
        QM_CUDA(ctx, cudaStreamSynchronize(st));
        const int n_b = h_ctr->n_tasks;
        if (spec_log) fprintf(stderr, " group B %d", n_b);
        if (n_b > 0) {
            rc = spec_run_group(ctx, P, idx->v, X, 1, n_b, h_ctr, st);
            if (rc) return rc;
        }
        sp = qm_prof_begin(ctx, QM_ST_ADVANCE, st);
        spec_finish_kernel<<<grid, 128, 0, st>>>(idx->v, *opt, codes, stride, lens, sc.seeds, sc.plan, sc.n_plan, sc.st, regs, n_regs, n_active, X,
                                                 (unsigned long long *)d_cells);
        qm_prof_end(ctx, QM_ST_ADVANCE, sp, st, 1);
        QM_CUDA(ctx, cudaMemcpyAsync(h_ctr, X.ctr + 2, kRoundHeader, cudaMemcpyDeviceToHost, st));
        QM_CUDA(ctx, cudaStreamSynchronize(st));
        if (spec_log) fprintf(stderr, " -> next %d\n", h_ctr->n_tasks);
        if (h_ctr->n_tasks == 0) return QM_OK;
        n_active = h_ctr->n_tasks;
        QM_CUDA(ctx, cudaMemcpyAsync(X.tasks, X.next_tasks, (size_t)n_active * sizeof(ExtTaskI), cudaMemcpyDeviceToDevice, st));
        QM_CUDA(ctx, cudaMemcpyAsync(X.keys, X.next_keys, (size_t)n_active * 8, cudaMemcpyDeviceToDevice, st));
        QM_CUDA(ctx, cudaMemcpyAsync(X.ctr, X.ctr + 2, sizeof(RoundCounters), cudaMemcpyDeviceToDevice, st));
    }
    return qm_fail(ctx, QM_ECUDA, "spec_finish_batch: reads still active after %d passes", 4 * QM_MAX_REGS + 8);
}

}  // namespace

extern "C" {

int qm_collect_seeds(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride,
                     const int32_t *d_lens, int64_t n_reads, qm_seed *d_seeds, int32_t *d_n_seeds, void *stream)
{
    if (!ctx || !idx || !opt || n_reads < 0 || (n_reads > 0 && (!d_codes || !d_lens || !d_seeds || !d_n_seeds)))
        return QM_EINVAL;
    if (opt->min_seed_len != idx->v.k) return qm_fail(ctx, QM_EINVAL, "index built with k=%d but min_seed_len=%d", idx->v.k, opt->min_seed_len);
    if (stride > kMaxStride) return qm_fail(ctx, QM_ELIMIT, "qm_collect_seeds: rows of %d bases: reads longer than %d bases are not supported", stride, kMaxStride);
    if (n_reads == 0) return QM_OK;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    if (opt->flags & QM_F_FM_SEEDS) {
        if (!idx->have_fm) return qm_fail(ctx, QM_EINVAL, "QM_F_FM_SEEDS needs an FM-index: qm_index_attach_bwa or qm_index_build_fm first");
        QM_CUDA(ctx, launch_fm_seed(idx, *opt, d_codes, stride, d_lens, n_reads, d_seeds, d_n_seeds, nullptr, nullptr, nullptr, true, (cudaStream_t)stream));
        return QM_OK;
    }
    // scratch of the three-kernel form: the packed reads and the read cursor
    const size_t pw = (size_t)((stride + 31) / 32 + 2 + (stride + 63) / 64 + 2);
    void *p = nullptr;
    int rc = qm_scratch_reserve(ctx, 3, (size_t)n_reads * pw * 8 + 256, &p);
    if (rc) return rc;
    QM_CUDA(ctx, launch_seed_chain(ctx, idx->v, *opt, d_codes, stride, d_lens, n_reads, d_seeds, d_n_seeds, nullptr, nullptr, nullptr, true,
                                   (cudaStream_t)stream, (uint64_t *)((char *)p + 256), (int *)p));
    return QM_OK;
}

int qm_align_se(qm_ctx *ctx, const qm_index *idx, const qm_opt *opt, const uint8_t *d_codes, int32_t stride,
                const int32_t *d_lens, int64_t n_reads, qm_reg *d_regs, int32_t *d_n_regs, int64_t *d_cells, void *stream)
{
    if (!ctx || !idx || !opt || n_reads < 0 || (n_reads > 0 && (!d_codes || !d_lens || !d_regs || !d_n_regs)))
        return QM_EINVAL;
    if (opt->min_seed_len != idx->v.k) return qm_fail(ctx, QM_EINVAL, "index built with k=%d but min_seed_len=%d", idx->v.k, opt->min_seed_len);
    if (opt->e_ins <= 0 || opt->e_del <= 0) return qm_fail(ctx, QM_EINVAL, "gap extension penalties must be > 0");
    if (stride > kMaxStride) return qm_fail(ctx, QM_ELIMIT, "qm_align_se: rows of %d bases: reads longer than %d bases are not supported", stride, kMaxStride);
    if (n_reads == 0) return QM_OK;
    QM_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t nbmax = n_reads < kSeBatch ? n_reads : kSeBatch;
    SeScratch sc;
    int rc = se_scratch(ctx, nbmax, stride, &sc);
    if (rc) return rc;
    static_assert(kRoundHeader <= 8192, "round header must fit the context's pinned buffer");
    RoundCounters *h_ctr = (RoundCounters *)ctx->h_pinned;          // only the first kRoundHeader bytes are ever read back
    const ExtParams P = qm_ext_params(opt);
    const int tpb = 128;
    for (int64_t b0 = 0; b0 < n_reads; b0 += kSeBatch) {
        const int64_t nb = n_reads - b0 < kSeBatch ? n_reads - b0 : kSeBatch;
        const unsigned grid = (unsigned)((nb + tpb - 1) / tpb);
        const uint8_t *codes = d_codes + b0 * stride;
        const int32_t *lens = d_lens + b0;
        int sp = qm_prof_begin(ctx, QM_ST_SEED, st);
        int n_seed_launches = 0;
        if (opt->flags & QM_F_FM_SEEDS) {
            if (!idx->have_fm) return qm_fail(ctx, QM_EINVAL, "QM_F_FM_SEEDS needs an FM-index: qm_index_attach_bwa or qm_index_build_fm first");
            for (int pt = 0; pt < ctx->se_n_parts; ++pt) QM_CUDA(ctx, cudaStreamWaitEvent(st, ctx->se_part_ev[pt], 0));
            if (ctx->se_pk && b0 == 0) QM_CUDA(ctx, qm_unpack_reads_launch(ctx->se_pk, ctx->se_mk, stride, ctx->se_sp, ctx->se_sm, n_reads, (uint8_t *)d_codes, st));
            QM_CUDA(ctx, launch_fm_seed(idx, *opt, codes, stride, lens, nb, sc.seeds, sc.n_seeds, sc.plan, sc.n_plan, sc.st, false, st));
            n_seed_launches = 1;
        } else if (ctx->se_n_parts > 0 && b0 == 0 && n_reads <= kSeBatch && !se_parts_landed(ctx)) {
            // the batch is still arriving piece by piece (host entry): seed each piece as soon as its copy has landed.  Each piece
            // is launched on a side stream of its own: one thread per read leaves every launch a tail of slow reads (repeats),
            // and eight launches in one stream paid eight tails (+4.3 ms per 4 M reads); side by side the next piece fills it.
            int64_t r0 = 0;
            QM_CUDA(ctx, cudaEventRecord(ctx->ev_fork, st));
            for (int pt = 0; pt < ctx->se_n_parts; ++pt) {
                const int64_t r1 = ctx->se_part_end[pt] < nb ? ctx->se_part_end[pt] : nb;
                cudaStream_t ss = ctx->side[pt % 12];
                if (r1 > r0) {
                    QM_CUDA(ctx, cudaStreamWaitEvent(ss, ctx->ev_fork, 0));
                    QM_CUDA(ctx, cudaStreamWaitEvent(ss, ctx->se_part_ev[pt], 0));
                    if (ctx->se_pk) QM_CUDA(ctx, qm_unpack_reads_launch(ctx->se_pk + r0 * ctx->se_sp, ctx->se_mk + r0 * ctx->se_sm, stride, ctx->se_sp, ctx->se_sm,
                                                                        r1 - r0, (uint8_t *)codes + r0 * stride, ss));
                    QM_CUDA(ctx, launch_seed_chain(ctx, idx->v, *opt, codes + r0 * stride, stride, lens + r0, r1 - r0, sc.seeds + r0 * QM_MAX_SEEDS,
                                                   sc.n_seeds + r0, sc.plan + r0 * QM_MAX_SEEDS, sc.n_plan + r0, sc.st + r0, false, ss,
                                                   sc.packed + r0 * sc.packed_words, sc.cursors + 1 + pt % 32));
                    QM_CUDA(ctx, cudaEventRecord(ctx->ev_join[pt % 12], ss));
                    QM_CUDA(ctx, cudaStreamWaitEvent(st, ctx->ev_join[pt % 12], 0));
                    ++n_seed_launches;
                    r0 = r1;
                } else {
                    QM_CUDA(ctx, cudaStreamWaitEvent(st, ctx->se_part_ev[pt], 0));
                }
            }
            if (r0 < nb) return qm_fail(ctx, QM_EINVAL, "qm_align_se: the announced pieces cover %lld of %lld reads", (long long)r0, (long long)nb);
        } else {
            // (a chunk whose pieces have all landed already -- every chunk of a host call but the first -- is seeded in one launch)
            for (int pt = 0; pt < ctx->se_n_parts; ++pt) QM_CUDA(ctx, cudaStreamWaitEvent(st, ctx->se_part_ev[pt], 0));
            if (ctx->se_pk && b0 == 0) QM_CUDA(ctx, qm_unpack_reads_launch(ctx->se_pk, ctx->se_mk, stride, ctx->se_sp, ctx->se_sm, n_reads, (uint8_t *)d_codes, st));
            QM_CUDA(ctx, launch_seed_chain(ctx, idx->v, *opt, codes, stride, lens, nb, sc.seeds, sc.n_seeds, sc.plan, sc.n_plan, sc.st, false, st,
                                           sc.packed, sc.cursors));
            n_seed_launches = 1;
        }
        ctx->se_n_parts = 0; ctx->se_pk = ctx->se_mk = nullptr;
        qm_prof_end(ctx, QM_ST_SEED, sp, st, n_seed_launches);
        // each read has at most 2 x QM_MAX_REGS dependent tasks, so the loop always ends on one of its breaks; if it did not, reads
        // would be left unfinished, and that is an error as it is in spec_finish_batch
        bool finished = false;
        for (int round = 0; round < 4 * QM_MAX_REGS + 8; ++round) {
            sp = qm_prof_begin(ctx, QM_ST_ADVANCE, st);
            cudaMemsetAsync(sc.ctr, 0, sizeof(RoundCounters), st);
            advance_kernel<<<grid, tpb, 0, st>>>(idx->v, *opt, codes, stride, lens, nb, sc.seeds, sc.plan, sc.n_plan, sc.st,
                                                 d_regs + b0 * QM_MAX_REGS, d_n_regs + b0, sc.res, sc.tasks, sc.keys,
                                                 sc.ctr, (unsigned long long *)d_cells);
            qm_prof_end(ctx, QM_ST_ADVANCE, sp, st, 1);
            cudaMemcpyAsync(h_ctr, sc.ctr, kRoundHeader, cudaMemcpyDeviceToHost, st);
            cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) { return qm_fail(ctx, QM_ECUDA, "qm_align_se round %d: %s", round, cudaGetErrorString(e)); }
            if (h_ctr->n_tasks == 0) { finished = true; break; }
            static const bool round_log = getenv("QM_ROUND_LOG") != nullptr;       // diagnostics: the round's task counts per class
            if (round_log) {
                fprintf(stderr, "[qm round %d] tasks %d max_score %d classes", round, h_ctr->n_tasks, h_ctr->max_score);
                for (int c = 0; c < kExtClasses; ++c) fprintf(stderr, " %d", h_ctr->class_count[c]);
                fprintf(stderr, "\n");
            }
            // (both thresholds follow the batch: they were tuned on 4 M reads, and a 200 k-read batch that switched modes at the same task
            // counts spent its whole first round in the speculative finish: 9.2 against 7.6 ms per 100 k pairs)
            static const int tail_env = getenv("QM_TAIL_MIN") ? atoi(getenv("QM_TAIL_MIN")) : -1;       // tuning knob
            const int tail_min = tail_env >= 0 ? tail_env : (int)std::min<int64_t>(kTailMinTasks, std::max<int64_t>(2048, nb / 64));
            if (h_ctr->n_tasks < tail_min) {
                // few reads left: finish them on the device, one warp per read, no more round trips
                sp = qm_prof_begin(ctx, QM_ST_EXTEND, st);
                int blocks = (h_ctr->n_tasks + kTailWarps - 1) / kTailWarps;
                if (blocks > ctx->sm_count * 6) blocks = ctx->sm_count * 6;
                ExtTaskI *over = sc.tasks + nb;
                int *n_over = &sc.ctr->pad[0], *cursor2 = &sc.ctr->pad[1];
                tail_kernel<4><<<blocks, kTailWarps * 32, 0, st>>>(idx->v, *opt, P, codes, stride, lens, sc.seeds, sc.plan, sc.n_plan,
                                                                   sc.st, d_regs + b0 * QM_MAX_REGS, d_n_regs + b0, sc.tasks, h_ctr->n_tasks, nullptr,
                                                                   &sc.ctr->tail_cursor, (unsigned long long *)d_cells, over, n_over);
                // reads parked because an extension is longer than 127 bases (none for 150-base reads)
                tail_kernel<16><<<ctx->sm_count * 2, kTailWarps * 32, 0, st>>>(idx->v, *opt, P, codes, stride, lens, sc.seeds, sc.plan, sc.n_plan,
                                                                               sc.st, d_regs + b0 * QM_MAX_REGS, d_n_regs + b0, over, 0, n_over,
                                                                               cursor2, (unsigned long long *)d_cells, nullptr, nullptr);
                qm_prof_end(ctx, QM_ST_EXTEND, sp, st, 2);
                finished = true;
                break;
            }
            // between the two thresholds: every remaining seed ahead of the state machine (spec_finish_batch).  Below tail_min the
            // serial warp-per-read tail above is quicker: two launch groups of the throughput kernels cost ~1 ms whatever they hold.
            static const bool spec_on = !(getenv("QM_SPEC") && atoi(getenv("QM_SPEC")) == 0);       // QM_SPEC=0: the serial tail of round 1
            static const int spec_env = getenv("QM_SPEC_MIN") ? std::min(atoi(getenv("QM_SPEC_MIN")), kSpecMinTasks) : -1;   // tuning knob
            const int spec_min = spec_env >= 0 ? spec_env : (int)std::min<int64_t>(kSpecMinTasks, std::max<int64_t>(8192, nb / 8));
            if (spec_on && h_ctr->n_tasks < spec_min) {
                rc = spec_finish_batch(ctx, idx, opt, P, codes, stride, lens, sc, d_regs + b0 * QM_MAX_REGS, d_n_regs + b0, d_cells, h_ctr,
                                       h_ctr->n_tasks, st);
                if (rc) return rc;
                finished = true;
                break;
            }
            // The round's tasks sorted by (query length, rows, seed score): the classes become contiguous runs of one list, the
            // two tasks a thread of the packed kernel takes are near twins (same columns, same rows, same band) and the lanes of
            // a warp finish together.  Stable LSD radix sort of 24-bit keys (sort.cu), values = task indices.
            sp = qm_prof_begin(ctx, QM_ST_ADVANCE, st);
            rc = qm_sort_pairs(ctx, sc.keys, (uint32_t *)sc.lists, h_ctr->n_tasks, kExtSortKeyBits, st);
            qm_prof_end(ctx, QM_ST_ADVANCE, sp, st, 0);
            if (rc) return rc;
            int64_t list_off[kExtClasses];
            { int64_t acc = 0; for (int c = 0; c < kExtClasses; ++c) { list_off[c] = acc; acc += h_ctr->class_count[c]; } }
            sp = qm_prof_begin(ctx, QM_ST_EXTEND, st);
            int n_launch = 0;
            for (int c = 0; c < kExtClasses; ++c) n_launch += h_ctr->class_count[c] > 0;
            rc = qm_ext_launch_classes(ctx, P, idx->v, sc.tasks, sc.lists, nb, sc.ctr->class_count, sc.ctr->class_cursor,
                                       h_ctr->class_count, sc.res, sc.lists + nb, sc.ctr->fb, st,
                                       h_ctr->max_score <= 255, list_off);
            qm_prof_end(ctx, QM_ST_EXTEND, sp, st, n_launch);
            if (rc) return rc;
        }
        if (!finished) return qm_fail(ctx, QM_ECUDA, "qm_align_se: reads still active after %d rounds", 4 * QM_MAX_REGS + 8);
    }
    QM_CUDA(ctx, cudaGetLastError());
    return QM_OK;
}

}  // extern "C"
