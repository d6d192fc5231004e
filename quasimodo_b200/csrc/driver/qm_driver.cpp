// qm_driver -- C++ host driver over the C-ABI (include/quasimodo_b200.h): the file-level drop-in for the
// reference's read-level rules.  It owns no arithmetic of the hot path: alignment, counting, calling and the
// coordinate sort all run in libquasimodo_b200.so on the B200; this file is file formats and plumbing.
//
//   qm_driver sample   --ref REF.fa[,MORE.fa...] --r1 R1.fq[.gz] --r2 R2.fq[.gz] [--sample NAME]
//                      [--bam OUT.bam] [--counts OUT.tsv] [--vcf OUT.vcf [--vcf-gz 0]] [--gpu I | --gpus A,B,..|A-B] [-t THREADS] [-w BAND]
//                      [--rmdup 1 [--rmdup-bam OUT.rmdup.bam] [--metrics FILE]] [--no-rescue 1] [--mpileup OUT.mpileup]
//                      [--bwa-index PREFIX | --fm-seeds 1] [--indels 0] [--max-depth N] [--baq 1]
//                      [-A -B -O -E -L -U -T -d -c -D -W: bwa mem's options of the same letters, -A scaling the others as bwa does]
//                      [-q / --min-mapq N] [-Q / --min-bq N] [--count-orphans 1] [--ignore-overlaps 1]: the mpileups' -q -Q -A -x
//                      [--stage-ms 1: per-stage device time (CUDA events) of every GPU in the log]
//                      [--benchmark FILE (every command): wall time, peak memory, I/O and CPU load as a Snakemake benchmark TSV]
//                      [-K INT: bwa mem -K, input chunks of INT bases, each paired against its own insert-size model (mem_pestat over
//                       all of its pairs), as bwa does; the default is one model per sample from its first QM_PESTAT_PAIRS pairs (DESIGN.md 5.3)]
//                      [-I mean[,std[,max[,min]]]: bwa mem -I, the FR insert-size model given instead of estimated]
//                      [--print-options 1: print the alignment options the command line resolves to and exit (host only)]
//        an option the command does not know is a usage error
//        --mpileup: the text pileup of `samtools mpileup -f ref bam` (rules/vcfcall.smk:39, input of the VarScan rule) with -B
//        semantics, formatted on the device (with --rmdup 1: of the duplicate-free records, as the reference's rule reads them)
//        --no-rescue 1 = bwa mem -S (mate rescue off; on by default as in the reference's command line)
//        --rmdup: duplicates are marked on the device with picard MarkDuplicates' rule (rules/rmdup.smk:13-16) before
//        anything is counted, as in the reference where every caller reads the .rmdup.bam; --bam still holds all records
//        (duplicates flagged 0x400), --rmdup-bam is the REMOVE_DUPLICATES=true file.  With --gpus the reads and records stay on
//        their GPUs: duplicates and the --max-depth cap are decided over small per-pair / per-read tuples all-gathered over NCCL,
//        so every output is the one-GPU output
//        --decontam A.fa[,B.fa] [--decontam2 C.fa[,D.fa]] [--clean-r1 F --clean-r2 F]: rules rm_phix and rm_human_ecoli
//        (rules/decontamination.smk:15-17,43-48) in the same job, in front of the target: each raw batch is aligned against pass 1's
//        genome (its own index, filter-mode sample and insert-size model; bwa's options, not --bwa-index / --fm-seeds), the pairs
//        whose records are both unmapped are gathered on the host, still packed, and go on to pass 2, then to the target, whose pair
//        ids count the kept pairs.  Every output equals `decontam` (pass 1) | `decontam` (pass 2) | `sample` on the cleaned FASTQ,
//        with --gpus too; --clean-r1/-r2 write that cleaned FASTQ.  Not with --keep-contigs.  With -K every stage cuts bwa's chunks
//        over its own input (pass 2 over pass 1's survivors, the target over pass 2's), on one GPU
//        = rules/bwa.smk:15-18 (bwa mem | samtools view | samtools sort | samtools index -> BAM + BAI),
//          rules/vcfcall.smk:39 (pileup path: count TSV, SURVEY.md B.3) and rules/vcfcall.smk:115-117 (VCF)
//   qm_driver decontam --ref CONTAMINANT.fa[,MORE.fa] --r1 .. --r2 .. --out-r1 CLEAN1.fq --out-r2 CLEAN2.fq
//                      [--keep-contigs N]
//        = rules/decontamination.smk:15-17 / 43-48: keep the pairs whose BOTH records are unmapped
//          ((flag & 12) == 12 && !(flag & 256)), re-emitted as FASTQ with /1 /2 names, as sequenced.
//          With --keep-contigs N the first N contigs of the (concatenated) reference are the target genome and
//          a pair is dropped iff a mate maps to a later (contaminant) contig: one pass instead of three.
//   qm_driver pileup   --ref REF.fa[,MORE.fa...] --bam IN.bam [--counts OUT.tsv] [--vcf OUT.vcf [--vcf-gz 0]] [--mpileup OUT.mpileup]
//                      [--max-depth N] [--baq 1] [-q -Q --count-orphans 1 --ignore-overlaps 1] [--min-dp --min-alt --min-af] [--indels 0]
//                      [--sample NAME] [--gpu I] [-t THREADS] [--stage-ms 1]
//        = rules/vcfcall.smk:39 (`mpileup`: samtools mpileup -f ref {rmdup.bam}) and rules/vcfcall.smk:115-119 (`bcftools`): the
//          count TSV, VCF (+ .gz + .tbi) and text pileup of an existing coordinate-sorted BAM, through the writers of `sample`, with
//          the same defaults (BAQ off, no depth cap); the BAM of `sample` read back gives `sample`'s bytes.  The file is inflated
//          and validated on the host before a CUDA context exists (a bad file exits 2 with or without a GPU); the records are
//          decoded and paired on the device (qm_bam_to_pairs); the depth cap follows the file's order of the reads.
//   qm_driver rmdup    --bam IN.bam --rmdup-bam OUT.bam [--metrics FILE] [--sample LIB] [--gpu I] [-t THREADS] [--stage-ms 1]
//        = rules/rmdup.smk:13-16 (`picard MarkDuplicates REMOVE_DUPLICATES=true` on {sample}.{ref_name}.bam): the records of an
//          existing coordinate-sorted BAM without its duplicates, byte for byte (0x400 cleared), the input's header plus one @PG
//          line, the .bai and the duplication metrics.  Inflated and validated on the host before a CUDA context exists; the
//          decision runs on the device (qm_bam_mark_duplicates), ties going to the file order of the sorted BAM as in picard
//   qm_driver index    --ref X.fa [--prefix P] [--gpu I] [-t THREADS]
//        = rules/index.smk:12-14 (`bwa index` + `samtools faidx`): bwa's five index files P.bwt, P.sa (suffix array, BWT,
//          checkpoints and samples built on the device, qm_index_build_fm), P.pac, P.ann, P.amb, and X.fa.fai; --prefix defaults
//          to the FASTA path, as in bwa.  The FASTA is read and validated on the host before a CUDA context exists (A/C/G/T only,
//          line lengths samtools faidx accepts, at most QM_MAX_CONTIGS contigs, 2 x length < 2^31)
//   qm_driver bam-from-records --ref .. --r1 .. --r2 .. --alns ALNS.bin [--perm PERM.bin] --bam OUT.bam
//        = the BAM/BAI writer alone on given qm_aln records (test entry; with --perm no GPU is touched)
//   qm_driver fastq-check --r1 .. --r2 .. [-t THREADS] [-K N [--batch-pairs M]]
//        = the FASTQ side alone (host only): the two mate files parsed and validated as `sample` would, pairs / bases / parse rate;
//          with -K the sizes in pairs of bwa mem's input chunks of N bases, cut as `sample -K N` cuts them
//
// Exit status: 0 ok, 1 usage, 2 I/O or format error, 3 library/CUDA error (message on stderr), so a failing job
// fails its Snakemake rule exactly like a failing `bwa`.
#include <zlib.h>
#include <fcntl.h>
#include <unistd.h>
#include <cerrno>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdarg>
#include <ctime>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/quasimodo_b200.h"

namespace {

[[noreturn]] void die(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    fprintf(stderr, "qm_driver: ");
    vfprintf(stderr, fmt, ap);
    fprintf(stderr, "\n");
    va_end(ap);
    exit(code);
}

// ------------------------------------------------------------------------------------------------
// line reader over zlib (reads plain and gzip files alike)
struct LineReader {
    gzFile f = nullptr;                   // gzip input
    int fd = -1;                          // plain input: read(2) straight into the buffer (zlib's transparent mode copies every byte twice)
    std::string path;
    std::vector<char> buf;
    size_t pos = 0, len = 0;
    explicit LineReader(const std::string &p) : path(p), buf(4 << 20)
    {
        fd = open(p.c_str(), O_RDONLY);
        if (fd < 0) die(2, "cannot open %s", p.c_str());
        unsigned char magic[2] = {0, 0};
        const ssize_t got = pread(fd, magic, 2, 0);
        if (got == 2 && magic[0] == 0x1f && magic[1] == 0x8b) {
            close(fd); fd = -1;
            f = gzopen(p.c_str(), "rb");
            if (!f) die(2, "cannot open %s", p.c_str());
            gzbuffer(f, 1 << 20);
        }
    }
    ~LineReader() { if (f) gzclose(f); if (fd >= 0) close(fd); }
    LineReader(const LineReader &) = delete;
    LineReader &operator=(const LineReader &) = delete;
    bool fill()
    {
        long n;
        if (f) n = gzread(f, buf.data(), (unsigned)buf.size());
        else do { n = (long)read(fd, buf.data(), buf.size()); } while (n < 0 && errno == EINTR);
        if (n < 0) die(2, "read error in %s", path.c_str());
        pos = 0; len = (size_t)n;
        return n > 0;
    }
    // next line as a view into the buffer (valid until the next call), without the terminator; false at end of file.  A line that
    // crosses the end of the buffer is assembled in `spill`.
    std::string spill;
    bool next_view(const char *&p, size_t &n)
    {
        if (pos == len && !fill()) return false;
        const char *s = buf.data() + pos;
        const char *nl = (const char *)memchr(s, '\n', len - pos);
        if (nl) {
            p = s; n = (size_t)(nl - s);
            pos += n + 1;
            if (n && p[n - 1] == '\r') --n;
            return true;
        }
        if (!next(spill)) return false;
        p = spill.data(); n = spill.size();
        return true;
    }
    // next line without the terminator; false at end of file
    bool next(std::string &out)
    {
        out.clear();
        bool got = false;
        for (;;) {
            if (pos == len && !fill()) return got;
            got = true;
            const char *s = buf.data() + pos;
            const char *nl = (const char *)memchr(s, '\n', len - pos);
            if (nl) {
                out.append(s, nl - s);
                pos += (size_t)(nl - s) + 1;
                if (!out.empty() && out.back() == '\r') out.pop_back();
                return true;
            }
            out.append(s, len - pos);
            pos = len;
        }
    }
};

struct Genome {
    std::vector<std::string> names;
    std::vector<int64_t> lens, offs;
    std::vector<uint8_t> codes;            // 0..3, contigs concatenated
};

void read_fasta(const std::string &path, Genome &g)
{
    LineReader rd(path);
    std::string ln;
    int8_t lut[256];
    memset(lut, -1, sizeof lut);
    lut['A'] = lut['a'] = 0; lut['C'] = lut['c'] = 1; lut['G'] = lut['g'] = 2; lut['T'] = lut['t'] = 3;
    bool open = false;
    while (rd.next(ln)) {
        if (ln.empty()) continue;
        if (ln[0] == '>') {
            if (open) g.lens.back() = (int64_t)g.codes.size() - g.offs.back();
            size_t e = 1;
            while (e < ln.size() && !isspace((unsigned char)ln[e])) ++e;
            g.names.push_back(ln.substr(1, e - 1));      // bwa: name up to the first whitespace (.ann / .fai column 1)
            g.offs.push_back((int64_t)g.codes.size());
            g.lens.push_back(0);
            open = true;
        } else {
            if (!open) die(2, "%s: sequence before the first '>' line", path.c_str());
            for (char c : ln) {
                const int8_t v = lut[(unsigned char)c];
                if (v < 0) die(2, "%s: base '%c' in contig %s: only A/C/G/T references are supported (bwa would draw a random base)",
                               path.c_str(), c, g.names.back().c_str());
                g.codes.push_back((uint8_t)v);
            }
        }
    }
    if (open) g.lens.back() = (int64_t)g.codes.size() - g.offs.back();
    if (g.names.empty()) die(2, "%s: no contigs", path.c_str());
}

// ------------------------------------------------------------------------------------------------
// one batch of read pairs in the library's layout (reads 2i / 2i+1 are mates) + names
struct Batch {
    int64_t n_pairs = 0;
    int32_t stride = 0;
    uint8_t *codes = nullptr, *quals = nullptr;      // page-locked (qm_host_alloc)
    uint8_t *bases2 = nullptr, *nmask = nullptr;      // the packed form of codes that crosses the link (2 bits per base + an N bit)
    int32_t *lens = nullptr;
    qm_aln *alns = nullptr;
    std::string names;                                // NUL-separated, one per pair
    std::vector<uint32_t> name_off;
    std::vector<int64_t> chunks;                      // -K: the sizes in pairs of bwa's input chunks the batch consists of
};

struct FastqPairReader {
    LineReader r1, r2;
    std::string h, s, p, q;
    FastqPairReader(const std::string &a, const std::string &b) : r1(a), r2(b) {}
    static bool record(LineReader &r, std::string &h, std::string &s, std::string &p, std::string &q)
    {
        if (!r.next(h)) return false;
        while (h.empty()) if (!r.next(h)) return false;
        if (h[0] != '@') die(2, "%s: FASTQ header expected, got '%.40s'", r.path.c_str(), h.c_str());
        if (!r.next(s) || !r.next(p) || !r.next(q)) die(2, "%s: truncated FASTQ record", r.path.c_str());
        if (p.empty() || p[0] != '+') die(2, "%s: '+' line expected", r.path.c_str());
        if (s.size() != q.size()) die(2, "%s: sequence and quality lengths differ in %s", r.path.c_str(), h.c_str());
        return true;
    }
};

// one mate file's share of a batch, flat: record i's bases are seq[soff[i] .. soff[i+1]), its qualities the same range of qual, its
// cleaned name names + noff[i] (NUL-terminated).  No allocation per record: the line buffers are reused, the arrays grow amortised.
struct Side {
    std::vector<char> names, seq, qual;
    std::vector<uint64_t> soff;
    std::vector<uint32_t> noff;
    size_t n = 0;
    void clear() { names.clear(); seq.clear(); qual.clear(); soff.assign(1, 0); noff.clear(); n = 0; }
    size_t len(size_t i) const { return (size_t)(soff[i + 1] - soff[i]); }
};

struct RawBatch { Side a, b; size_t size() const { return a.n; } };

int g_threads = 8;                                  // -t: host threads for parsing, packing, record encoding, BGZF

// run fn(begin, end) over [0, n) on up to g_threads threads
template <class F> void parallel_ranges(size_t n, F fn)
{
    const size_t nt = std::max<size_t>(1, std::min<size_t>((size_t)g_threads, n / 4096 + 1));
    if (nt == 1) { fn((size_t)0, n); return; }
    std::vector<std::thread> pool;
    for (size_t t = 0; t < nt; ++t) pool.emplace_back([=]() { fn(n * t / nt, n * (t + 1) / nt); });
    for (auto &th : pool) th.join();
}

// one FASTQ record appended to a side; false at the end of the file
bool read_record(LineReader &r, Side &v)
{
    const char *p = nullptr;
    size_t n = 0;
    if (!r.next_view(p, n)) return false;
    while (n == 0) if (!r.next_view(p, n)) return false;                // blank lines between records
    if (p[0] != '@') die(2, "%s: FASTQ header expected, got '%.*s'", r.path.c_str(), (int)std::min<size_t>(n, 40), p);
    // bwa: the name up to the first whitespace, a trailing /<digit> dropped (bwa.c trim_readno; SURVEY.md B.8)
    size_t e = 1;
    while (e < n && !isspace((unsigned char)p[e])) ++e;
    if (e > 3 && p[e - 2] == '/' && isdigit((unsigned char)p[e - 1])) e -= 2;
    v.noff.push_back((uint32_t)v.names.size());
    v.names.insert(v.names.end(), p + 1, p + e);
    v.names.push_back('\0');
    if (!r.next_view(p, n)) die(2, "%s: truncated FASTQ record", r.path.c_str());
    const size_t sl = n;
    v.seq.insert(v.seq.end(), p, p + n);
    if (!r.next_view(p, n)) die(2, "%s: truncated FASTQ record", r.path.c_str());
    if (n == 0 || p[0] != '+') die(2, "%s: '+' line expected", r.path.c_str());
    if (!r.next_view(p, n)) die(2, "%s: truncated FASTQ record", r.path.c_str());
    if (n != sl) die(2, "%s: sequence and quality lengths differ in @%s", r.path.c_str(), v.names.data() + v.noff.back());
    v.qual.insert(v.qual.end(), p, p + n);
    v.soff.push_back((uint64_t)v.seq.size());
    ++v.n;
    return true;
}

// bwa mem's input chunks (-K): bseq_read (bwa.c, bwa 0.7.17 as recalled) reads pairs in order and adds both mates' lengths to a
// running sum; a chunk ends after the first pair at which the sum reaches K, and the next one starts from zero.  *sum carries an
// open chunk's sum into the next call; chunks gets the sizes (in pairs) of the chunks that end among pairs [from, n).
void cut_chunks(const RawBatch &b, size_t from, int64_t K, int64_t *sum, int64_t *open, std::vector<int64_t> &chunks)
{
    for (size_t i = from; i < b.a.n; ++i) {
        *sum += (int64_t)(b.a.len(i) + b.b.len(i));
        ++*open;
        if (*sum >= K) { chunks.push_back(*open); *sum = 0; *open = 0; }
        else if (*open >= QM_CHUNK_MAX_PAIRS)
            die(1, "option -K: a chunk of %lld bases runs past %d pairs, the most one chunk may hold (QM_CHUNK_MAX_PAIRS); choose a smaller -K",
                (long long)K, QM_CHUNK_MAX_PAIRS);
    }
}

// reads up to max_pairs pairs; mates are matched by file order (bwa's rule), not by name.  The two files are read (and
// inflated) side by side: the second mate's file has a thread of its own.  With K > 0 (bwa mem -K) the batch is then read on,
// pair by pair, to the end of bwa's chunk it stops in, so that it holds whole chunks; *chunks gets their sizes in pairs (the
// last one of the input is whatever remains).
bool read_batch(FastqPairReader &fr, int64_t max_pairs, RawBatch &out, int64_t K = 0, std::vector<int64_t> *chunks = nullptr)
{
    // a record's four lines are consumed as they are read (a view dies with the next read): one copy from the file buffer into the
    // side's arrays, no string per line
    auto side = [max_pairs](LineReader &r, Side &v) {
        v.clear();
        while ((int64_t)v.n < max_pairs) {
            if (!read_record(r, v)) return;
            if (v.n == 1 && max_pairs <= ((int64_t)1 << 23)) {
                // the first record sizes the batch's arrays (address space only: no growth by doubling, no copies of what was read)
                const size_t m = (size_t)max_pairs, sl = v.len(0);
                v.seq.reserve(m * (sl + 1)); v.qual.reserve(m * (sl + 1));
                v.names.reserve(m * (v.names.size() + 2)); v.soff.reserve(m + 1); v.noff.reserve(m);
            }
        }
    };
    std::thread t2([&]() { side(fr.r2, out.b); });
    side(fr.r1, out.a);
    t2.join();
    if (out.a.n < out.b.n) die(2, "%s has more records than %s", fr.r2.path.c_str(), fr.r1.path.c_str());
    if (out.a.n > out.b.n) die(2, "%s has fewer records than %s", fr.r2.path.c_str(), fr.r1.path.c_str());
    if (K > 0) {
        chunks->clear();
        int64_t sum = 0, open = 0;
        cut_chunks(out, 0, K, &sum, &open, *chunks);
        while (open > 0) {
            const bool g1 = read_record(fr.r1, out.a), g2 = read_record(fr.r2, out.b);
            if (g1 != g2) die(2, "%s has %s records than %s", fr.r2.path.c_str(), g1 ? "fewer" : "more", fr.r1.path.c_str());
            if (!g1) { chunks->push_back(open); break; }
            cut_chunks(out, out.a.n - 1, K, &sum, &open, *chunks);
        }
    }
    // bwa refuses mates whose names differ once /1 and /2 are dropped (bwamem_pair.c mem_sam_pe: "paired reads have different
    // names"): files that went out of step pair every read with a stranger and still align -- fail like bwa instead
    std::atomic<size_t> first_bad{out.a.n};
    parallel_ranges(out.a.n, [&](size_t b, size_t e) {
        for (size_t i = b; i < e; ++i)
            if (strcmp(out.a.names.data() + out.a.noff[i], out.b.names.data() + out.b.noff[i]) != 0) {
                size_t cur = first_bad.load();
                while (i < cur && !first_bad.compare_exchange_weak(cur, i)) {}
                return;
            }
    });
    if (first_bad.load() < out.a.n) {
        const size_t i = first_bad.load();
        die(2, "paired reads have different names: \"%s\" (%s), \"%s\" (%s)", out.a.names.data() + out.a.noff[i], fr.r1.path.c_str(),
            out.b.names.data() + out.b.noff[i], fr.r2.path.c_str());
    }
    return out.a.n > 0;
}

struct Lib {
    qm_ctx *ctx = nullptr;
    void check(int rc, const char *what)
    {
        if (rc != QM_OK) die(3, "%s failed (%d): %s", what, rc, ctx ? qm_last_error(ctx) : "no context");
    }
};

void pack_batch(Lib &L, const RawBatch &raw, bool want_alns, Batch &b)
{
    static uint8_t lut[256];
    static bool init = false;
    if (!init) {
        memset(lut, 4, sizeof lut);
        lut['A'] = lut['a'] = 0; lut['C'] = lut['c'] = 1; lut['G'] = lut['g'] = 2; lut['T'] = lut['t'] = 3;
        init = true;
    }
    const Side *sd[2] = {&raw.a, &raw.b};
    b.n_pairs = (int64_t)raw.size();
    size_t mx = 1;
    for (int m = 0; m < 2; ++m)
        for (size_t i = 0; i < sd[m]->n; ++i) mx = std::max(mx, sd[m]->len(i));
    if (mx > 500) die(2, "read of %zu bases: reads longer than 500 bp are not supported", mx);
    b.stride = (int32_t)((mx + 15) & ~(size_t)15);
    const size_t nb = (size_t)2 * b.n_pairs * b.stride;
    void *p = nullptr;
    L.check(qm_host_alloc(L.ctx, nb, &p), "qm_host_alloc"); b.codes = (uint8_t *)p;
    L.check(qm_host_alloc(L.ctx, nb, &p), "qm_host_alloc"); b.quals = (uint8_t *)p;
    L.check(qm_host_alloc(L.ctx, (size_t)2 * b.n_pairs * sizeof(int32_t), &p), "qm_host_alloc"); b.lens = (int32_t *)p;
    if (want_alns) { L.check(qm_host_alloc(L.ctx, (size_t)2 * b.n_pairs * sizeof(qm_aln), &p), "qm_host_alloc"); b.alns = (qm_aln *)p; }
    // the pair's name is the first mate's (bwa prints one name for both records)
    b.names.assign(raw.a.names.begin(), raw.a.names.end());
    b.name_off = raw.a.noff;
    parallel_ranges(raw.size(), [&](size_t i0, size_t i1) {
        for (size_t i = i0; i < i1; ++i) {
            for (int m = 0; m < 2; ++m) {
                const char *s = sd[m]->seq.data() + sd[m]->soff[i], *q = sd[m]->qual.data() + sd[m]->soff[i];
                uint8_t *c = b.codes + (2 * i + m) * b.stride, *qq = b.quals + (2 * i + m) * b.stride;
                const size_t n = sd[m]->len(i);
                for (size_t j = 0; j < n; ++j) {
                    c[j] = lut[(unsigned char)s[j]];
                    const int v = (int)(unsigned char)q[j] - 33;
                    qq[j] = (uint8_t)(v < 0 ? 0 : v > 93 ? 93 : v);
                }
                memset(c + n, 4, (size_t)b.stride - n);
                memset(qq + n, 0, (size_t)b.stride - n);
                b.lens[2 * i + m] = (int32_t)n;
            }
        }
    });
    // codes stay on the host for the BAM records; the device receives 3 bits per base instead of 8
    L.check(qm_host_alloc(L.ctx, (size_t)2 * b.n_pairs * (b.stride / 4), &p), "qm_host_alloc"); b.bases2 = (uint8_t *)p;
    L.check(qm_host_alloc(L.ctx, (size_t)2 * b.n_pairs * (b.stride / 8), &p), "qm_host_alloc"); b.nmask = (uint8_t *)p;
    L.check(qm_pack_reads_host(b.codes, b.stride, 2 * b.n_pairs, b.bases2, b.nmask), "qm_pack_reads_host");
}

void free_batch(Lib &L, Batch &b)
{
    qm_host_free(L.ctx, b.codes); qm_host_free(L.ctx, b.quals); qm_host_free(L.ctx, b.lens); qm_host_free(L.ctx, b.alns);
    qm_host_free(L.ctx, b.bases2); qm_host_free(L.ctx, b.nmask);
    b.bases2 = b.nmask = nullptr;
    b.codes = b.quals = nullptr; b.lens = nullptr; b.alns = nullptr;
    std::string().swap(b.names);
    std::vector<uint32_t>().swap(b.name_off);
}

// The pairs of src[k] whose byte keep[k][p] is set (keep[k] == nullptr: all of them), in order, as one batch at the largest stride
// among the sources: packed bases, N mask, qualities, codes, lengths and names are copied as they are, the rows padded as pack_batch
// pads them (N bases, quality 0).  A threaded host gather; the records are not carried (alns stays unset).
void gather_pairs(Lib &L, const std::vector<const Batch *> &src, const std::vector<const uint8_t *> &keep, Batch &out)
{
    std::vector<std::pair<uint32_t, int64_t>> sel;            // (source, pair)
    int32_t stride = 16;
    for (size_t k = 0; k < src.size(); ++k) {
        for (int64_t p = 0; p < src[k]->n_pairs; ++p) if (!keep[k] || keep[k][p]) sel.emplace_back((uint32_t)k, p);
        if (src[k]->n_pairs) stride = std::max(stride, src[k]->stride);
    }
    const size_t n = sel.size(), sp = (size_t)stride / 4, sm = (size_t)stride / 8;
    out.n_pairs = (int64_t)n;
    out.stride = stride;
    void *p = nullptr;
    L.check(qm_host_alloc(L.ctx, 2 * n * stride, &p), "qm_host_alloc"); out.codes = (uint8_t *)p;
    L.check(qm_host_alloc(L.ctx, 2 * n * stride, &p), "qm_host_alloc"); out.quals = (uint8_t *)p;
    L.check(qm_host_alloc(L.ctx, 2 * n * sizeof(int32_t), &p), "qm_host_alloc"); out.lens = (int32_t *)p;
    L.check(qm_host_alloc(L.ctx, 2 * n * sp, &p), "qm_host_alloc"); out.bases2 = (uint8_t *)p;
    L.check(qm_host_alloc(L.ctx, 2 * n * sm, &p), "qm_host_alloc"); out.nmask = (uint8_t *)p;
    auto name = [&](size_t i) { const Batch &b = *src[sel[i].first]; return b.names.data() + b.name_off[(size_t)sel[i].second]; };
    std::vector<uint32_t> nl(n);
    parallel_ranges(n, [&](size_t i0, size_t i1) { for (size_t i = i0; i < i1; ++i) nl[i] = (uint32_t)strlen(name(i)) + 1; });
    out.name_off.resize(n);
    uint32_t o = 0;
    for (size_t i = 0; i < n; ++i) { out.name_off[i] = o; o += nl[i]; }
    out.names.resize(o);
    parallel_ranges(n, [&](size_t i0, size_t i1) {
        for (size_t i = i0; i < i1; ++i) {
            const Batch &b = *src[sel[i].first];
            memcpy(&out.names[out.name_off[i]], name(i), nl[i]);
            const size_t bs = (size_t)b.stride, bp = bs / 4, bm = bs / 8;
            for (int m = 0; m < 2; ++m) {
                const size_t r = (size_t)(2 * sel[i].second + m), w = 2 * i + m;
                memcpy(out.codes + w * stride, b.codes + r * bs, bs); memset(out.codes + w * stride + bs, 4, stride - bs);
                memcpy(out.quals + w * stride, b.quals + r * bs, bs); memset(out.quals + w * stride + bs, 0, stride - bs);
                memcpy(out.bases2 + w * sp, b.bases2 + r * bp, bp); memset(out.bases2 + w * sp + bp, 0, sp - bp);
                memcpy(out.nmask + w * sm, b.nmask + r * bm, bm); memset(out.nmask + w * sm + bm, 0xff, sm - bm);
                out.lens[w] = b.lens[r];
            }
        }
    });
}

// Pair ids of `sample --decontam` across the GPU workers.  A pair's id in a stage is its index in that stage's input (in the
// three-job chain: its index in the FASTQ the stage reads), so batch i takes its ids of a stage once batch i - 1 has taken its own.
// Channel s < number of stages: ids of stage s; one more channel orders the writes of the cleaned FASTQ.
struct Ledger {
    std::mutex m;
    std::condition_variable cv;
    std::vector<int64_t> turn, total;                        // per channel: the batch whose turn it is, pairs taken so far
    int64_t begin(int ch, int64_t i)
    {
        std::unique_lock<std::mutex> lk(m);
        cv.wait(lk, [&]() { return turn[(size_t)ch] == i; });
        return total[(size_t)ch];
    }
    void end(int ch, int64_t n)
    {
        { std::lock_guard<std::mutex> lk(m); total[(size_t)ch] += n; ++turn[(size_t)ch]; }
        cv.notify_all();
    }
    int64_t take(int ch, int64_t i, int64_t n) { const int64_t t = begin(ch, i); end(ch, n); return t; }
};

// ------------------------------------------------------------------------------------------------
// BGZF writer (SURVEY.md B.7): blocks of <= 0xff00 bytes, raw deflate level 1, compressed by a thread team,
// written in order; remembers each block's file offset so that virtual offsets can be resolved afterwards
struct BgzfWriter {
    static constexpr size_t kBlock = 0xff00;
    FILE *fp = nullptr;
    std::string path;
    int threads = 1, level = 1;
    std::vector<std::vector<uint8_t>> pending;
    std::vector<uint8_t> cur;
    std::vector<uint64_t> block_off;                  // file offset of every block written or pending
    uint64_t file_off = 0;
    size_t blocks_done = 0;
    BgzfWriter(const std::string &p, int t, int lvl) : path(p), threads(t < 1 ? 1 : t), level(lvl)
    {
        fp = fopen(p.c_str(), "wb");
        if (!fp) die(2, "cannot create %s", p.c_str());
        cur.reserve(kBlock);
    }
    static void compress(const std::vector<uint8_t> &in, std::vector<uint8_t> &out, int level)
    {
        out.resize(18 + compressBound((uLong)in.size()) + 8 + 64);
        static const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
        memcpy(out.data(), hdr, 16);
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        if (deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) die(2, "deflateInit2 failed");
        zs.next_in = (Bytef *)in.data(); zs.avail_in = (uInt)in.size();
        zs.next_out = out.data() + 18; zs.avail_out = (uInt)(out.size() - 18 - 8);
        if (deflate(&zs, Z_FINISH) != Z_STREAM_END) die(2, "deflate failed");
        const size_t clen = zs.total_out;
        deflateEnd(&zs);
        const size_t total = 18 + clen + 8;
        if (total > 65536) die(2, "BGZF block does not fit");
        out[16] = (uint8_t)((total - 1) & 0xff); out[17] = (uint8_t)((total - 1) >> 8);
        const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), in.data(), (uInt)in.size()), isz = (uint32_t)in.size();
        memcpy(out.data() + 18 + clen, &crc, 4);
        memcpy(out.data() + 18 + clen + 4, &isz, 4);
        out.resize(total);
    }
    void drain()
    {
        if (pending.empty()) return;
        std::vector<std::vector<uint8_t>> outv(pending.size());
        std::atomic<size_t> next{0};
        auto work = [&]() {
            for (;;) {
                const size_t i = next.fetch_add(1);
                if (i >= pending.size()) break;
                compress(pending[i], outv[i], level);
            }
        };
        const int nt = (int)std::min<size_t>((size_t)threads, pending.size());
        std::vector<std::thread> team;
        for (int t = 1; t < nt; ++t) team.emplace_back(work);
        work();
        for (auto &t : team) t.join();
        for (auto &o : outv) {
            block_off.push_back(file_off);
            if (fwrite(o.data(), 1, o.size(), fp) != o.size()) die(2, "write error on %s", path.c_str());
            file_off += o.size();
        }
        blocks_done += pending.size();
        pending.clear();
    }
    void close_block()
    {
        if (cur.empty()) return;
        pending.push_back(cur);
        cur.clear();
        if (pending.size() >= (size_t)threads * 16) drain();
    }
    // index of the block the next byte goes to, and the offset inside it
    void tell(uint64_t &block, uint32_t &off) const { block = blocks_done + pending.size(); off = (uint32_t)cur.size(); }
    // keep a record inside one block when it fits in one (htslib's bgzf_flush_try)
    void reserve(size_t n) { if (cur.size() + n > kBlock) close_block(); }
    void write(const void *p, size_t n)
    {
        const uint8_t *s = (const uint8_t *)p;
        while (n) {
            const size_t k = std::min(n, kBlock - cur.size());
            cur.insert(cur.end(), s, s + k);
            s += k; n -= k;
            if (cur.size() == kBlock) close_block();
        }
    }
    void finish()
    {
        close_block();
        drain();
        static const uint8_t eof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        block_off.push_back(file_off);
        if (fwrite(eof, 1, 28, fp) != 28 || fclose(fp) != 0) die(2, "write error on %s", path.c_str());
        fp = nullptr;
    }
    uint64_t voffset(uint64_t block, uint32_t off) const { return (block_off[block] << 16) | off; }
};

// ------------------------------------------------------------------------------------------------
// BAM records + BAI (SURVEY.md B.7)
inline int reg2bin(int64_t beg, int64_t end)
{
    --end;
    if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}

struct RecRef {                       // one alignment record = (batch, read index inside the batch)
    const Batch *b;
    int64_t r;
};

struct BamIndexEntry { int32_t rid; int32_t beg, end; uint16_t bin; bool mapped; uint64_t blk0; uint32_t off0; uint64_t blk1; uint32_t off1; };

inline void put32(std::vector<uint8_t> &v, uint32_t x) { uint8_t b[4]; memcpy(b, &x, 4); v.insert(v.end(), b, b + 4); }
inline void put16(std::vector<uint8_t> &v, uint16_t x) { uint8_t b[2]; memcpy(b, &x, 2); v.insert(v.end(), b, b + 2); }

void put_tag_int(std::vector<uint8_t> &v, const char *tag, int64_t x)
{   // smallest fitting integer type, like htslib's bam_aux_append of SAM "i" values
    v.push_back((uint8_t)tag[0]); v.push_back((uint8_t)tag[1]);
    if (x >= 0) {
        if (x <= 0xff) { v.push_back('C'); v.push_back((uint8_t)x); }
        else if (x <= 0xffff) { v.push_back('S'); put16(v, (uint16_t)x); }
        else { v.push_back('I'); put32(v, (uint32_t)x); }
    } else {
        if (x >= -128) { v.push_back('c'); v.push_back((uint8_t)(int8_t)x); }
        else if (x >= -32768) { v.push_back('s'); put16(v, (uint16_t)(int16_t)x); }
        else { v.push_back('i'); put32(v, (uint32_t)(int32_t)x); }
    }
}

std::string cigar_string(const qm_aln &a)
{
    std::string s;
    char tmp[16];
    for (int k = 0; k < a.n_cigar; ++k) {
        snprintf(tmp, sizeof tmp, "%u%c", a.cigar[k] >> 4, "MIDNSHP=X"[a.cigar[k] & 15]);
        s += tmp;
    }
    return s;
}

int cigar_ref_len(const qm_aln &a)
{
    int n = 0;
    for (int k = 0; k < a.n_cigar; ++k) { const int op = a.cigar[k] & 15; if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) n += a.cigar[k] >> 4; }
    return n;
}

// one BAM record into `out` (without the leading block_size); returns the reference span end for the index
void encode_record(const Genome &g, const RecRef &rr, std::vector<uint8_t> &out, BamIndexEntry &ie)
{
    const Batch &b = *rr.b;
    const int64_t r = rr.r;
    const qm_aln &a = b.alns[r], &m = b.alns[r ^ 1];
    const int l_seq = b.lens[r];
    const uint8_t *codes = b.codes + r * b.stride, *quals = b.quals + r * b.stride;
    const char *name = b.names.data() + b.name_off[r >> 1];
    const size_t l_name = strlen(name) + 1;
    const bool mapped = !(a.flag & 0x4);
    const bool cig_ok = a.n_cigar != 255;
    const int n_cig = mapped && cig_ok ? a.n_cigar : 0;
    const int rlen = mapped ? cigar_ref_len(a) : 0;
    const int64_t end = a.pos + (rlen > 0 ? rlen : 1);
    const int bin = reg2bin(a.pos, end);
    out.clear();
    put32(out, (uint32_t)a.rid);
    put32(out, (uint32_t)a.pos);
    out.push_back((uint8_t)l_name);
    out.push_back(a.mapq);
    put16(out, (uint16_t)bin);
    put16(out, (uint16_t)n_cig);
    put16(out, a.flag);
    put32(out, (uint32_t)l_seq);
    put32(out, (uint32_t)a.mate_rid);
    put32(out, (uint32_t)a.mate_pos);
    put32(out, (uint32_t)a.tlen);
    out.insert(out.end(), (const uint8_t *)name, (const uint8_t *)name + l_name);
    for (int k = 0; k < n_cig; ++k) put32(out, a.cigar[k]);
    // SEQ / QUAL as SAM stores them: reverse-complemented / reversed for reverse-strand records
    const bool rev = (a.flag & 0x10) != 0;            // bwa mem_aln2sam: an unmapped read placed at its reverse-strand mate carries 0x10 and is stored reverse-complemented too
    static const uint8_t nib[5] = {1, 2, 4, 8, 15};
    std::vector<uint8_t> seq((size_t)l_seq);
    for (int j = 0; j < l_seq; ++j) {
        const uint8_t c = rev ? codes[l_seq - 1 - j] : codes[j];
        seq[j] = rev ? (c < 4 ? (uint8_t)(3 - c) : 4) : c;
    }
    for (int j = 0; j < l_seq; j += 2) out.push_back((uint8_t)(nib[seq[j]] << 4 | (j + 1 < l_seq ? nib[seq[j + 1]] : 0)));
    for (int j = 0; j < l_seq; ++j) out.push_back(rev ? quals[l_seq - 1 - j] : quals[j]);
    // tags in bwa's order (mem_aln2sam): NM, MD (mapped), MC (mate mapped), AS, XS
    if (n_cig > 0) {
        put_tag_int(out, "NM", a.nm);
        std::string md;
        const uint8_t *ref = g.codes.data() + g.offs[a.rid] + a.pos;
        int x = 0, y = 0, u = 0;
        char tmp[16];
        for (int k = 0; k < n_cig; ++k) {
            const int op = a.cigar[k] & 15, len = (int)(a.cigar[k] >> 4);
            if (op == 0) {
                for (int i = 0; i < len; ++i) {
                    if (seq[x + i] != ref[y + i]) { snprintf(tmp, sizeof tmp, "%d%c", u, "ACGTN"[ref[y + i]]); md += tmp; u = 0; }
                    else ++u;
                }
                x += len; y += len;
            } else if (op == 2) {
                if (k > 0 && k < n_cig - 1) {                // bwa_gen_cigar2 ignores leading / trailing deletions
                    snprintf(tmp, sizeof tmp, "%d^", u); md += tmp;
                    for (int i = 0; i < len; ++i) md.push_back("ACGTN"[ref[y + i]]);
                    u = 0;
                }
                y += len;
            } else if (op == 1 || op == 4) x += len;
        }
        snprintf(tmp, sizeof tmp, "%d", u); md += tmp;
        out.push_back('M'); out.push_back('D'); out.push_back('Z');
        out.insert(out.end(), md.begin(), md.end()); out.push_back(0);
    }
    if (!(m.flag & 0x4) && m.n_cigar != 255 && m.n_cigar > 0) {
        const std::string mc = cigar_string(m);
        out.push_back('M'); out.push_back('C'); out.push_back('Z');
        out.insert(out.end(), mc.begin(), mc.end()); out.push_back(0);
    }
    if (a.score >= 0) put_tag_int(out, "AS", a.score);
    if (a.sub >= 0) put_tag_int(out, "XS", a.sub);
    ie.rid = a.rid; ie.beg = a.pos; ie.end = (int32_t)end; ie.bin = (uint16_t)bin; ie.mapped = mapped;
}

void write_bai(const std::string &path, const Genome &g, const std::vector<BamIndexEntry> &ents, const BgzfWriter &bw)
{
    FILE *fp = fopen(path.c_str(), "wb");
    if (!fp) die(2, "cannot create %s", path.c_str());
    auto w32 = [&](uint32_t x) { fwrite(&x, 4, 1, fp); };
    auto w64 = [&](uint64_t x) { fwrite(&x, 8, 1, fp); };
    fwrite("BAI\1", 1, 4, fp);
    w32((uint32_t)g.names.size());
    size_t e = 0;
    uint64_t n_no_coor = 0;
    for (size_t c = 0; c < g.names.size(); ++c) {
        std::map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins;
        const size_t n_win = (size_t)((g.lens[c] + 16383) >> 14);
        std::vector<uint64_t> lin(n_win, ~0ull);
        uint64_t off_beg = ~0ull, off_end = 0, n_map = 0, n_unmap = 0;
        int last_bin = -1;
        for (; e < ents.size() && ents[e].rid == (int32_t)c; ++e) {
            const BamIndexEntry &x = ents[e];
            const uint64_t v0 = bw.voffset(x.blk0, x.off0), v1 = bw.voffset(x.blk1, x.off1);
            auto &ch = bins[x.bin];
            if (last_bin == (int)x.bin && !ch.empty()) ch.back().second = v1;       // consecutive records of one bin: one chunk
            else ch.emplace_back(v0, v1);
            last_bin = x.bin;
            const size_t w0 = (size_t)(x.beg >> 14), w1 = (size_t)((x.end - 1) >> 14);
            for (size_t w = w0; w <= w1 && w < n_win; ++w) if (lin[w] == ~0ull) lin[w] = v0;
            if (off_beg == ~0ull) off_beg = v0;
            off_end = v1;
            if (x.mapped) ++n_map; else ++n_unmap;
        }
        size_t used = n_win;
        while (used > 0 && lin[used - 1] == ~0ull) --used;
        for (size_t w = 0; w < used; ++w) if (lin[w] == ~0ull) lin[w] = w ? lin[w - 1] : 0;
        const bool any = off_beg != ~0ull;
        w32((uint32_t)(bins.size() + (any ? 1 : 0)));
        for (auto &kv : bins) {
            w32(kv.first); w32((uint32_t)kv.second.size());
            for (auto &ch : kv.second) { w64(ch.first); w64(ch.second); }
        }
        if (any) { w32(37450); w32(2); w64(off_beg); w64(off_end); w64(n_map); w64(n_unmap); }   // samtools' metadata pseudo-bin
        w32((uint32_t)used);
        for (size_t w = 0; w < used; ++w) w64(lin[w]);
    }
    for (; e < ents.size(); ++e) ++n_no_coor;
    w64(n_no_coor);
    if (fclose(fp) != 0) die(2, "write error on %s", path.c_str());
}

void write_bam(const std::string &path, const Genome &g, const std::deque<Batch> &batches, const std::vector<uint32_t> &perm,
               const std::vector<int64_t> &batch_first_read, const std::string &cmdline, int threads)
{
    BgzfWriter bw(path, threads, 1);
    std::string text = "@HD\tVN:1.6\tSO:coordinate\n";
    for (size_t c = 0; c < g.names.size(); ++c) text += "@SQ\tSN:" + g.names[c] + "\tLN:" + std::to_string(g.lens[c]) + "\n";
    text += "@PG\tID:quasimodo_b200\tPN:quasimodo_b200\tVN:0.1\tCL:" + cmdline + "\n";
    std::vector<uint8_t> hdr;
    hdr.insert(hdr.end(), {'B', 'A', 'M', 1});
    put32(hdr, (uint32_t)text.size());
    hdr.insert(hdr.end(), text.begin(), text.end());
    put32(hdr, (uint32_t)g.names.size());
    for (size_t c = 0; c < g.names.size(); ++c) {
        put32(hdr, (uint32_t)g.names[c].size() + 1);
        hdr.insert(hdr.end(), g.names[c].begin(), g.names[c].end()); hdr.push_back(0);
        put32(hdr, (uint32_t)g.lens[c]);
    }
    bw.write(hdr.data(), hdr.size());
    bw.close_block();                                  // records start on a block boundary, as samtools writes them
    // Records are encoded (SEQ / QUAL orientation, NM / MD against the reference, tags: ~2 us each) by `threads` workers, a wave of
    // chunks at a time; the writer thread then only copies the finished bytes into the BGZF blocks and notes the virtual offsets.
    // (One thread encoding 2 M records took 4.8 of the 7.9 s a 1 M-pair sample needed from FASTQ to every output.)
    std::vector<BamIndexEntry> ents(perm.size());
    const size_t kChunk = 16384;
    const size_t n_chunks = (perm.size() + kChunk - 1) / kChunk;
    const size_t wave = (size_t)std::max(1, threads) * 2;
    std::vector<std::vector<uint8_t>> bytes(wave);
    std::vector<std::vector<uint32_t>> sizes(wave);
    auto encode_chunk = [&](size_t c, std::vector<uint8_t> &out, std::vector<uint32_t> &sz) {
        out.clear(); sz.clear();
        std::vector<uint8_t> rec;
        const size_t i0 = c * kChunk, i1 = std::min(perm.size(), i0 + kChunk);
        for (size_t i = i0; i < i1; ++i) {
            const int64_t gr = perm[i];
            const size_t bi = (size_t)(std::upper_bound(batch_first_read.begin(), batch_first_read.end(), gr) - batch_first_read.begin()) - 1;
            RecRef rr{&batches[bi], gr - batch_first_read[bi]};
            encode_record(g, rr, rec, ents[i]);
            sz.push_back((uint32_t)rec.size());
            out.insert(out.end(), rec.begin(), rec.end());
        }
    };
    for (size_t c0 = 0; c0 < n_chunks; c0 += wave) {
        const size_t nw = std::min(wave, n_chunks - c0);
        std::atomic<size_t> next{0};
        std::vector<std::thread> pool;
        const int nt = (int)std::min<size_t>((size_t)std::max(1, threads), nw);
        for (int t = 0; t < nt; ++t)
            pool.emplace_back([&]() { for (size_t k; (k = next.fetch_add(1)) < nw;) encode_chunk(c0 + k, bytes[k], sizes[k]); });
        for (auto &th : pool) th.join();
        for (size_t k = 0; k < nw; ++k) {
            const uint8_t *p = bytes[k].data();
            size_t i = (c0 + k) * kChunk;
            for (uint32_t bs : sizes[k]) {
                bw.reserve((size_t)bs + 4);
                bw.tell(ents[i].blk0, ents[i].off0);
                bw.write(&bs, 4);
                bw.write(p, bs);
                bw.tell(ents[i].blk1, ents[i].off1);
                p += bs; ++i;
            }
        }
    }
    bw.finish();
    write_bai(path + ".bai", g, ents, bw);
}

// ------------------------------------------------------------------------------------------------
// text outputs: count TSV (SURVEY.md B.3) and caller VCF (B.4) -- same bytes as quasimodo_b200/formats.py
void write_count_tsv(const std::string &path, const Genome &g, const std::vector<int32_t> &rows)
{
    FILE *fp = fopen(path.c_str(), "w");
    if (!fp) die(2, "cannot create %s", path.c_str());
    std::vector<char> buf(1 << 22);
    setvbuf(fp, buf.data(), _IOFBF, buf.size());
    fputs("chrom\tpos\tref\tdepth\tA_f\tC_f\tG_f\tT_f\tN_f\tdel_f\tA_r\tC_r\tG_r\tT_r\tN_r\tdel_r\tins_start\tdel_start\traw_depth\tread_starts\n", fp);
    for (size_t c = 0; c < g.names.size(); ++c)
        for (int64_t i = 0; i < g.lens[c]; ++i) {
            const int32_t *r = rows.data() + (size_t)(g.offs[c] + i) * QM_NCH;
            int64_t depth = 0;
            for (int k = 0; k < 5; ++k) depth += r[k] + r[6 + k];
            fprintf(fp, "%s\t%lld\t%c\t%lld", g.names[c].c_str(), (long long)(i + 1), "ACGT"[g.codes[g.offs[c] + i]], (long long)depth);
            for (int k = 0; k < QM_NCH; ++k) fprintf(fp, "\t%d", r[k]);
            fputc('\n', fp);
        }
    if (fclose(fp) != 0) die(2, "write error on %s", path.c_str());
}

std::string trim_float3(double x)
{   // Python: f"{x:.3f}".rstrip("0").rstrip(".")
    char tmp[64];
    snprintf(tmp, sizeof tmp, "%.3f", x);
    std::string s = tmp;
    while (!s.empty() && s.back() == '0') s.pop_back();
    if (!s.empty() && s.back() == '.') s.pop_back();
    return s;
}

// --gpus: batches are dealt round-robin, batch i to GPU i % n_gpu; a GPU keeps the records of its batches in the order it got them
int batch_gpu(int64_t batch, int n_gpu) { return (int)(batch % n_gpu); }

// where each batch's records lie among those its GPU kept (qm_sample_kept_alns_host): {GPU, first record} per batch, batch i having
// gone to GPU batch_dev[i]
std::vector<std::pair<int, int64_t>> batch_sources(const std::vector<int64_t> &batch_pairs, const std::vector<int> &batch_dev, int n_gpu)
{
    std::vector<std::pair<int, int64_t>> src(batch_pairs.size());
    std::vector<int64_t> next((size_t)n_gpu, 0);
    for (size_t i = 0; i < batch_pairs.size(); ++i) {
        const int d = batch_dev[i];
        src[i] = {d, next[(size_t)d]};
        next[(size_t)d] += 2 * batch_pairs[i];
    }
    return src;
}

// the same for batches dealt round-robin
std::vector<std::pair<int, int64_t>> batch_sources(const std::vector<int64_t> &batch_pairs, int n_gpu)
{
    std::vector<int> dev(batch_pairs.size());
    for (size_t i = 0; i < dev.size(); ++i) dev[i] = batch_gpu((int64_t)i, n_gpu);
    return batch_sources(batch_pairs, dev, n_gpu);
}

// An indel allele that passes the caller's thresholds (same rule as the SNPs: raw depth at the anchor >= min_dp, supporting
// reads >= min_alt and >= min_af x depth), as the VCF shows it: anchor base first, POS = anchor (the convention of
// program/mummer2vcf.py for the truth set and of bcftools).
struct IndelCall { qm_indel a; int dp; double af, qual; };

// two allele tables sorted by key -> one sorted table, the counts of an allele both hold added up
std::vector<qm_indel> merge_indel_tables(const std::vector<qm_indel> &a, const qm_indel *b, int64_t nb)
{
    std::vector<qm_indel> out;
    out.reserve(a.size() + (size_t)nb);
    size_t i = 0;
    int64_t j = 0;
    while (i < a.size() || j < nb) {
        if (j >= nb || (i < a.size() && a[i].key < b[j].key)) out.push_back(a[i++]);
        else if (i >= a.size() || b[j].key < a[i].key) out.push_back(b[j++]);
        else {
            qm_indel x = a[i++];
            x.n_fwd += b[j].n_fwd; x.n_rev += b[j].n_rev;
            ++j;
            out.push_back(x);
        }
    }
    return out;
}

void write_vcf(const std::string &path, const Genome &g, const std::string &sample, const std::string &ref_path,
               const std::vector<qm_call> &calls, const std::vector<IndelCall> &indels)
{
    FILE *fp = fopen(path.c_str(), "w");
    if (!fp) die(2, "cannot create %s", path.c_str());
    fprintf(fp, "##fileformat=VCFv4.2\n##FILTER=<ID=PASS,Description=\"All filters passed\">\n"
                "##source=quasimodo_b200 (threshold caller on bcftools-mpileup-style counts; QUAL is not bcftools call QUAL)\n"
                "##reference=file://%s\n", ref_path.c_str());
    for (size_t c = 0; c < g.names.size(); ++c) fprintf(fp, "##contig=<ID=%s,length=%lld>\n", g.names[c].c_str(), (long long)g.lens[c]);
    fprintf(fp, "##INFO=<ID=DP,Number=1,Type=Integer,Description=\"Raw read depth\">\n"
                "##INFO=<ID=AF,Number=1,Type=Float,Description=\"Alternate allele fraction among bases passing the BQ filter\">\n"
                "##INFO=<ID=DP4,Number=4,Type=Integer,Description=\"ref-forward, ref-reverse, alt-forward, alt-reverse bases\">\n");
    if (!indels.empty())
        fprintf(fp, "##INFO=<ID=INDEL,Number=0,Type=Flag,Description=\"Indicates that the variant is an INDEL.\">\n"
                    "##INFO=<ID=IDV,Number=1,Type=Integer,Description=\"Reads supporting the indel (forward + reverse)\">\n"
                    "##INFO=<ID=ADF,Number=1,Type=Integer,Description=\"Supporting forward reads\">\n"
                    "##INFO=<ID=ADR,Number=1,Type=Integer,Description=\"Supporting reverse reads\">\n");
    fprintf(fp, "##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">\n"
                "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t%s\n", sample.c_str());
    size_t k = 0;
    auto put_indel = [&](const IndelCall &x) {
        const qm_indel &a = x.a;
        const uint8_t *ref = g.codes.data() + g.offs[a.rid] + a.pos;
        std::string r(1, "ACGT"[ref[0]]), alt(1, "ACGT"[ref[0]]);
        if (a.type == 1) { for (int i = 1; i <= a.len && a.pos + i < g.lens[a.rid]; ++i) r.push_back("ACGT"[ref[i]]); }
        else for (int i = 0; i < a.len; ++i) alt.push_back(i < QM_INDEL_SEQ_BASES && !(a.has_n) ? "ACGT"[(a.seq >> (2 * i)) & 3] : 'N');
        fprintf(fp, "%s\t%d\t.\t%s\t%s\t%s\tPASS\tINDEL;DP=%d;AF=%.3f;IDV=%d;ADF=%d;ADR=%d\tGT\t1\n", g.names[a.rid].c_str(), a.pos + 1, r.c_str(),
                alt.c_str(), trim_float3(x.qual).c_str(), x.dp, x.af, a.n_fwd + a.n_rev, a.n_fwd, a.n_rev);
    };
    for (const qm_call &c : calls) {
        while (k < indels.size() && (indels[k].a.rid < c.rid || (indels[k].a.rid == c.rid && indels[k].a.pos < c.pos))) put_indel(indels[k++]);
        fprintf(fp, "%s\t%d\t.\t%c\t%c\t%s\tPASS\tDP=%d;AF=%.3f;DP4=%d,%d,%d,%d\tGT\t1\n", g.names[c.rid].c_str(), c.pos + 1,
                "ACGT"[c.ref], "ACGT"[c.alt], trim_float3((double)c.qual).c_str(), c.dp, (double)c.af, c.ad_ref_f, c.ad_ref_r, c.ad_alt_f, c.ad_alt_r);
    }
    while (k < indels.size()) put_indel(indels[k++]);
    if (fclose(fp) != 0) die(2, "write error on %s", path.c_str());
}

// bgzip + tabix of a VCF (rule `bcftools`: `bgzip -c vcf > vcf.gz; tabix -p vcf vcf.gz`, rules/vcfcall.smk:118-119; the same two
// commands close rule `genome_diff`, rules/genome_diff.smk:24-25).  The .tbi is the tabix index of the spec: BGZF-compressed,
// format 2 (VCF: sequence column 1, begin column 2, meta char '#'), the UCSC binning of BAI with 16 kb linear windows, one
// entry per data line covering [POS-1, POS-1 + len(REF)), sequences listed in order of first appearance, htslib's
// pseudo-bin 37450 with the sequence's file range and record count.
void write_vcf_gz_tbi(const std::string &vcf_path, const std::string &gz_path, int threads)
{
    FILE *in = fopen(vcf_path.c_str(), "r");
    if (!in) die(2, "cannot open %s", vcf_path.c_str());
    BgzfWriter bw(gz_path, threads, 6);
    struct Ent { int ref; int64_t beg, end; uint64_t blk0; uint32_t off0; uint64_t blk1; uint32_t off1; };
    std::vector<Ent> ents;
    std::vector<std::string> names;
    std::map<std::string, int> name_id;
    char *line = nullptr;
    size_t cap = 0;
    ssize_t len;
    while ((len = getline(&line, &cap, in)) > 0) {
        if (line[0] != '#') {
            const char *t1 = (const char *)memchr(line, '\t', (size_t)len);
            const char *t2 = t1 ? (const char *)memchr(t1 + 1, '\t', (size_t)(line + len - t1 - 1)) : nullptr;
            const char *t3 = t2 ? (const char *)memchr(t2 + 1, '\t', (size_t)(line + len - t2 - 1)) : nullptr;
            const char *t4 = t3 ? (const char *)memchr(t3 + 1, '\t', (size_t)(line + len - t3 - 1)) : nullptr;
            if (!t4) die(2, "%s: malformed VCF line", vcf_path.c_str());
            const std::string chrom(line, (size_t)(t1 - line));
            auto it = name_id.find(chrom);
            if (it == name_id.end()) { it = name_id.emplace(chrom, (int)names.size()).first; names.push_back(chrom); }
            Ent e;
            e.ref = it->second;
            e.beg = atoll(t1 + 1) - 1;
            e.end = e.beg + std::max<int64_t>(1, (int64_t)(t4 - t3 - 1));
            if (!ents.empty() && (e.ref < ents.back().ref || (e.ref == ents.back().ref && e.beg < ents.back().beg)))
                die(2, "%s: records are not sorted by position: cannot index", vcf_path.c_str());
            bw.reserve((size_t)len);
            bw.tell(e.blk0, e.off0);
            bw.write(line, (size_t)len);
            bw.tell(e.blk1, e.off1);
            ents.push_back(e);
        } else bw.write(line, (size_t)len);
    }
    free(line);
    fclose(in);
    bw.finish();
    std::vector<uint8_t> out;
    auto w32 = [&](uint32_t x) { put32(out, x); };
    auto w64 = [&](uint64_t x) { uint8_t b[8]; memcpy(b, &x, 8); out.insert(out.end(), b, b + 8); };
    out.insert(out.end(), {'T', 'B', 'I', 1});
    w32((uint32_t)names.size());
    w32(2); w32(1); w32(2); w32(0); w32('#'); w32(0);
    size_t l_nm = 0;
    for (auto &n : names) l_nm += n.size() + 1;
    w32((uint32_t)l_nm);
    for (auto &n : names) { out.insert(out.end(), n.begin(), n.end()); out.push_back(0); }
    size_t e = 0;
    for (size_t c = 0; c < names.size(); ++c) {
        std::map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins;
        std::vector<uint64_t> lin;
        uint64_t off_beg = ~0ull, off_end = 0, n_rec = 0;
        int last_bin = -1;
        for (; e < ents.size() && ents[e].ref == (int)c; ++e) {
            const Ent &x = ents[e];
            const uint64_t v0 = bw.voffset(x.blk0, x.off0), v1 = bw.voffset(x.blk1, x.off1);
            const int bin = reg2bin(x.beg, x.end);
            auto &ch = bins[(uint32_t)bin];
            if (last_bin == bin && !ch.empty()) ch.back().second = v1;
            else ch.emplace_back(v0, v1);
            last_bin = bin;
            const size_t w0 = (size_t)(x.beg >> 14), w1 = (size_t)((x.end - 1) >> 14);
            if (lin.size() <= w1) lin.resize(w1 + 1, ~0ull);
            for (size_t w = w0; w <= w1; ++w) if (lin[w] == ~0ull) lin[w] = v0;
            if (off_beg == ~0ull) off_beg = v0;
            off_end = v1;
            ++n_rec;
        }
        for (size_t w = 0; w < lin.size(); ++w) if (lin[w] == ~0ull) lin[w] = w ? lin[w - 1] : 0;
        w32((uint32_t)bins.size() + 1);
        for (auto &kv : bins) {
            w32(kv.first); w32((uint32_t)kv.second.size());
            for (auto &ch : kv.second) { w64(ch.first); w64(ch.second); }
        }
        w32(37450); w32(2); w64(off_beg); w64(off_end); w64(n_rec); w64(0);
        w32((uint32_t)lin.size());
        for (uint64_t v : lin) w64(v);
    }
    w64(0);                                            // n_no_coor
    BgzfWriter tw(gz_path + ".tbi", 1, 6);
    tw.write(out.data(), out.size());
    tw.finish();
}

void write_fastq_pair(FILE *f1, FILE *f2, const Batch &b, int64_t pi)
{
    const char *name = b.names.data() + b.name_off[pi];
    FILE *fs[2] = {f1, f2};
    std::string s, q;
    for (int m = 0; m < 2; ++m) {
        const int64_t r = 2 * pi + m;
        const int l = b.lens[r];
        s.resize((size_t)l); q.resize((size_t)l);
        for (int j = 0; j < l; ++j) { s[j] = "ACGTN"[b.codes[r * b.stride + j]]; q[j] = (char)(b.quals[r * b.stride + j] + 33); }
        fprintf(fs[m], "@%s/%d\n%s\n+\n%s\n", name, m + 1, s.c_str(), q.c_str());   // bedtools bamtofastq: /1 /2 appended
    }
}

// ------------------------------------------------------------------------------------------------
struct Args {
    std::map<std::string, std::string> kv;
    std::string get(const std::string &k, const std::string &d = "") const { auto it = kv.find(k); return it == kv.end() ? d : it->second; }
    bool has(const std::string &k) const { return kv.count(k) != 0; }
};

Args parse_args(int argc, char **argv, int first)
{
    Args a;
    for (int i = first; i < argc; ++i) {
        std::string k = argv[i];
        if (k.size() < 2 || k[0] != '-') die(1, "unexpected argument '%s'", k.c_str());
        k = k.substr(k[1] == '-' ? 2 : 1);
        if (i + 1 >= argc) die(1, "option --%s needs a value", k.c_str());
        a.kv[k] = argv[++i];
    }
    return a;
}

// an option the command does not know is a usage error (a typo such as --min-qual must not silently run with the default)
void require_known(const Args &a, const char *cmd, const std::vector<const char *> &known)
{
    for (auto &kv : a.kv) {
        bool ok = false;
        for (const char *k : known) ok = ok || kv.first == k;
        if (!ok) die(1, "%s: unknown option '%s%s'", cmd, kv.first.size() > 1 ? "--" : "-", kv.first.c_str());
    }
}

// a whole non-negative decimal number or a usage error (atoi would read "6x" as 6 and "x" as 0)
int32_t parse_int(const std::string &opt, const std::string &v)
{
    if (v.empty() || v.size() > 9 || v.find_first_not_of("0123456789") != std::string::npos)
        die(1, "option -%s: '%s' is not a non-negative integer", opt.c_str(), v.c_str());
    return (int32_t)atol(v.c_str());
}

std::vector<std::string> split(const std::string &s, char sep);

// bwa mem's scoring and filtering options on top of the defaults of `bwa mem -k 31` (rules/bwa.smk:15), with bwa's own letters
// and bwa's rule for -A (fastmap.c main_mem): the match score scales -T -d -B -O -E -L -U unless they are given themselves;
// -O / -E / -L take "INT[,INT]" (deletion,insertion; 5',3').
void apply_bwa_options(const Args &a, qm_opt &o)
{
    auto one = [&](const char *k, int32_t &x) { if (a.has(k)) x = parse_int(k, a.get(k)); return a.has(k); };
    auto two = [&](const char *k, int32_t &x, int32_t &y) {
        if (!a.has(k)) return false;
        const auto v = split(a.get(k), ',');
        if (v.size() > 2) die(1, "option -%s takes INT[,INT]", k);
        x = y = parse_int(k, v[0]);
        if (v.size() == 2) y = parse_int(k, v[1]);
        return true;
    };
    one("w", o.w);
    one("k", o.min_seed_len);
    one("c", o.max_occ);
    one("W", o.min_chain_weight);
    if (a.has("D")) {
        char *end = nullptr;
        const std::string v = a.get("D");
        o.drop_ratio = strtof(v.c_str(), &end);
        if (v.empty() || *end || !(o.drop_ratio >= 0.f && o.drop_ratio <= 1.f)) die(1, "option -D: '%s' is not a fraction in [0, 1]", v.c_str());
    }
    const bool hB = one("B", o.b), hT = one("T", o.T), hd = one("d", o.zdrop), hU = one("U", o.pen_unpaired);
    const bool hO = two("O", o.o_del, o.o_ins), hE = two("E", o.e_del, o.e_ins), hL = two("L", o.pen_clip5, o.pen_clip3);
    if (one("A", o.a)) {
        if (!hB) o.b *= o.a;
        if (!hT) o.T *= o.a;
        if (!hO) { o.o_del *= o.a; o.o_ins *= o.a; }
        if (!hE) { o.e_del *= o.a; o.e_ins *= o.a; }
        if (!hd) o.zdrop *= o.a;
        if (!hL) { o.pen_clip5 *= o.a; o.pen_clip3 *= o.a; }
        if (!hU) o.pen_unpaired *= o.a;
    }
    if (o.a < 1) die(1, "option -A: the match score must be at least 1");
    if (o.w < 1) die(1, "option -w: the band width must be at least 1");
    if (o.max_occ < 1) die(1, "option -c: at least 1");
    if (o.min_seed_len < 8 || o.min_seed_len > 31) die(1, "option -k: 8 <= k <= 31 (the k-mer index packs a seed into 62 bits)");
}

// bwa mem -K INT and -I mean[,std[,max[,min]]] (fastmap.c, bwa 0.7.17 as recalled).  -K: bwa's input chunks hold K bases
// instead of 10^7 x threads, and each is paired against its own insert-size model (0: the driver's default, one model per sample
// from its first QM_PESTAT_PAIRS pairs).  -I: the model is given, not estimated: only FR (pes[1]) is set, std defaults to
// 0.1 x mean, high = (int)(mean + 4 std + .499), low = (int)(mean - 4 std + .499) clamped to >= 1 (bwa's rounding idiom), and an
// explicit max and min replace them; the other three orientations fail.  bwa reads the fields with strtod and takes any
// punctuation followed by a digit as the separator; what bwa would silently ignore (trailing text, a mean <= 0, min > max) is a
// usage error here.
struct PairOptions { int64_t K = 0; bool has_I = false; qm_pestat pes[4]; };

PairOptions parse_pair_options(const Args &a)
{
    PairOptions r;
    if (a.has("K")) {
        const std::string v = a.get("K");
        if (v.empty() || v.size() > 15 || v.find_first_not_of("0123456789") != std::string::npos || atoll(v.c_str()) < 1)
            die(1, "option -K: '%s' is not a positive integer (bases per input chunk)", v.c_str());
        r.K = atoll(v.c_str());
    }
    for (auto &pe : r.pes) { memset(&pe, 0, sizeof pe); pe.failed = 1; }
    if (a.has("I")) {
        const std::string v = a.get("I");
        const char *q = v.c_str();
        char *p = nullptr;
        qm_pestat &f = r.pes[1];
        auto bad = [&]() { die(1, "option -I: '%s' is not mean[,std[,max[,min]]]", v.c_str()); };
        auto next_field = [&]() { return *p != 0 && ispunct((unsigned char)*p) && isdigit((unsigned char)p[1]); };
        f.failed = 0;
        f.avg = strtod(q, &p);
        if (p == q || !(f.avg > 0) || !std::isfinite(f.avg)) bad();
        f.std = f.avg * .1;
        if (next_field()) f.std = strtod(p + 1, &p);
        f.high = (int)(f.avg + 4. * f.std + .499);
        f.low = (int)(f.avg - 4. * f.std + .499);
        if (f.low < 1) f.low = 1;
        if (next_field()) f.high = (int)(strtod(p + 1, &p) + .499);
        if (next_field()) f.low = (int)(strtod(p + 1, &p) + .499);
        if (*p != 0 || !(f.std >= 0) || !std::isfinite(f.std) || f.high < f.low || f.low < 0) bad();
        r.has_I = true;
    }
    return r;
}

// the admission options of both mpileups (rules/vcfcall.smk:39,115 pass none: the defaults), under the tools' names:
// -q / --min-mapq, -Q / --min-bq, --count-orphans 1 (-A), --ignore-overlaps 1 (-x)
void apply_mpileup_options(const Args &a, qm_pileup_opt &p)
{
    for (const char *k : {"min-mapq", "q"}) if (a.has(k)) p.min_mapq = parse_int(k, a.get(k));
    for (const char *k : {"min-bq", "Q"}) if (a.has(k)) p.min_bq = parse_int(k, a.get(k));
    if (a.has("count-orphans")) p.count_orphans = parse_int("count-orphans", a.get("count-orphans")) != 0;
    if (a.has("ignore-overlaps")) p.ignore_overlaps = parse_int("ignore-overlaps", a.get("ignore-overlaps")) != 0;
    if (p.min_mapq > 255 || p.min_bq > 93) die(1, "option -q is at most 255 and option -Q at most 93");
}

void print_options(const qm_opt &o, const qm_pileup_opt &p, const PairOptions &po)
{
    printf("q=%d Q=%d count-orphans=%d ignore-overlaps=%d ", p.min_mapq, p.min_bq, p.count_orphans, p.ignore_overlaps);
    printf("A=%d B=%d O=%d,%d E=%d,%d L=%d,%d U=%d T=%d d=%d w=%d k=%d c=%d D=%g W=%d flags=%d", o.a, o.b, o.o_del, o.o_ins, o.e_del, o.e_ins,
           o.pen_clip5, o.pen_clip3, o.pen_unpaired, o.T, o.zdrop, o.w, o.min_seed_len, o.max_occ, (double)o.drop_ratio, o.min_chain_weight, o.flags);
    if (po.K) printf(" K=%lld", (long long)po.K);                     // -K / -I only when given
    if (po.has_I) printf(" I=%.17g,%.17g,%d,%d", po.pes[1].avg, po.pes[1].std, po.pes[1].high, po.pes[1].low);
    printf("\n");
}

std::vector<std::string> split(const std::string &s, char sep)
{
    std::vector<std::string> out;
    size_t p = 0;
    for (;;) {
        const size_t q = s.find(sep, p);
        out.push_back(s.substr(p, q == std::string::npos ? q : q - p));
        if (q == std::string::npos) break;
        p = q + 1;
    }
    return out;
}

void check_refs(const Genome &g);

void load_refs(const std::string &spec, Genome &g)
{
    for (auto &p : split(spec, ',')) read_fasta(p, g);
    check_refs(g);
}

// a contaminant pass's genome (--decontam / --decontam2): as load_refs, an empty contig named with its file and option
void load_pass_refs(const char *opt, const std::string &spec, Genome &g)
{
    for (auto &p : split(spec, ',')) {
        const size_t c0 = g.names.size();
        read_fasta(p, g);
        for (size_t i = c0; i < g.names.size(); ++i)
            if (g.lens[i] <= 0) die(2, "--%s %s: contig %s is empty", opt, p.c_str(), g.names[i].c_str());
    }
    check_refs(g);
}

void check_refs(const Genome &g)
{
    if (g.names.size() > QM_MAX_CONTIGS) die(2, "%zu contigs: at most %d are supported", g.names.size(), QM_MAX_CONTIGS);
    for (size_t i = 0; i < g.names.size(); ++i) {
        if (g.lens[i] <= 0) die(2, "contig %s is empty", g.names[i].c_str());
        // the BAI / TBI binning scheme (and with it `samtools index`, `tabix -p vcf`) ends at 2^29 bases per contig
        if (g.lens[i] > ((int64_t)1 << 29)) die(2, "contig %s has %lld bases: BAI / TBI indexes address at most 2^29 per contig", g.names[i].c_str(), (long long)g.lens[i]);
        for (size_t j = 0; j < i; ++j) if (g.names[j] == g.names[i]) die(2, "contig name %s occurs twice in the reference", g.names[i].c_str());
    }
}

int sort_key_bits(const Genome &g, int &pos_bits)
{
    int64_t mx = 0;
    for (auto l : g.lens) mx = std::max(mx, l);
    pos_bits = qm_sort_pos_bits(mx);
    return qm_sort_key_bits((int)g.names.size(), pos_bits);
}

template <class T> std::vector<T> read_binary(const std::string &path);

// the duplication metrics of `sample --rmdup 1 --metrics` and `rmdup --metrics` (picard's file, reduced to what is decided here)
void write_dup_metrics(const std::string &path, const std::string &library, int64_t n_examined, int64_t n_dup)
{
    FILE *fm = fopen(path.c_str(), "w");
    if (!fm) die(2, "cannot create %s", path.c_str());
    fprintf(fm, "## METRICS CLASS\tquasimodo_b200.DuplicationMetrics\nLIBRARY\tREAD_PAIRS_EXAMINED\tREAD_PAIR_DUPLICATES\tPERCENT_DUPLICATION\n"
                "%s\t%lld\t%lld\t%.6f\n", library.c_str(), (long long)n_examined, (long long)n_dup,
            n_examined ? (double)n_dup / (double)n_examined : 0.0);
    fclose(fm);
}

// wall clock of the run's phases, one line on stderr at the end (where a sample's file-level time goes)
struct PhaseClock {
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now(), last = t0;
    std::string line;
    void mark(const char *name)
    {
        const auto now = std::chrono::steady_clock::now();
        char buf[64];
        snprintf(buf, sizeof buf, "%s%s %.2f", line.empty() ? "" : ", ", name, std::chrono::duration<double>(now - last).count());
        line += buf;
        last = now;
    }
    void report()
    {
        fprintf(stderr, "[qm_driver] phases (s): %s; total %.2f\n", line.c_str(), std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
    }
};

// --stage-ms 1: the library's CUDA-event stage timers of one GPU, one line in the log
void print_stage_ms(Lib &L, int dev)
{
    static const char *const kStage[QM_N_STAGES] = {"seed+chain", "advance", "extend", "pair+cigar", "pileup", "h2d", "d2h", "other", "rescue"};
    double ms[QM_N_STAGES];
    int64_t launches[QM_N_STAGES];
    L.check(qm_profile_collect(L.ctx, ms, launches), "qm_profile_collect");
    std::string line;
    double tot = 0;
    int64_t nl = 0;
    for (int i = 0; i < QM_N_STAGES; ++i) {
        char buf[64];
        snprintf(buf, sizeof buf, "%s%s %.1f", i ? ", " : "", kStage[i], ms[i]);
        line += buf;
        tot += ms[i];
        nl += launches[i];
    }
    fprintf(stderr, "[qm_driver] GPU %d stages (ms of device time): %s; total %.1f in %lld launches\n", dev, line.c_str(), tot, (long long)nl);
}

// The outputs of the reference's rules `mpileup` and `bcftools` from a counted sample (smps[0]: count tensor and indel allele
// table; with several GPUs the counts are summed already and the indel tables of smps[1..] are merged here): the count TSV
// (--counts), the calls and indel records as VCF (--vcf, + .gz and .tbi unless --vcf-gz 0) and the text pileup (--mpileup).
// make_text() leaves the text pileup on the device (qm_mpileup_text*) and returns its length.  `sample` and `pileup` both
// write through here, so that the same counts give the same bytes.
void write_outputs(const Args &a, const Genome &g, std::vector<Lib> &Ls, const std::vector<qm_index *> &idxs, const std::vector<qm_sample *> &smps,
                   int threads, const std::function<int64_t()> &make_text)
{
    Lib &L = Ls[0];
    qm_sample *smp = smps[0];
    qm_index *idx = idxs[0];
    const int n_gpu = (int)smps.size();
    const std::string counts = a.get("counts"), vcf = a.get("vcf"), mpileup = a.get("mpileup");
    if (!counts.empty()) {
        std::vector<int32_t> rows(g.codes.size() * QM_NCH);
        L.check(qm_sample_counts_host(smp, rows.data()), "qm_sample_counts_host");
        write_count_tsv(counts, g, rows);
    }
    if (!vcf.empty()) {
        qm_call_opt copt; qm_call_opt_default(&copt);
        if (a.has("min-dp")) copt.min_dp = atoi(a.get("min-dp").c_str());
        if (a.has("min-alt")) copt.min_alt = atoi(a.get("min-alt").c_str());
        if (a.has("min-af")) copt.min_af = (float)atof(a.get("min-af").c_str());
        std::vector<qm_call> calls(g.codes.size() * 3 + 16);                   // at most 3 alternative bases per position
        int64_t nc = 0;
        L.check(qm_sample_call_snps_host(smp, &copt, calls.data(), (int64_t)calls.size(), &nc), "qm_sample_call_snps_host");
        calls.resize((size_t)nc);
        // indel records (--indels 0 leaves them out): the sample's allele table against the raw depth at the anchor
        std::vector<IndelCall> icalls;
        if (atoi(a.get("indels", "1").c_str())) {
            std::vector<qm_indel> tab((size_t)1 << 18);
            int64_t nt = 0;
            L.check(qm_indel_table_fetch_host(qm_sample_indel_table(smp), idx, tab.data(), (int64_t)tab.size(), &nt), "qm_indel_table_fetch_host");
            if (n_gpu > 1) {
                // the sparse part of the merge (SURVEY.md 8e: "host merge of the sparse indel-allele table"): every GPU tallied the
                // alleles of its own batches; the tables (a few thousand records, sorted by key) are added up by key here
                tab.resize((size_t)nt);
                std::vector<qm_indel> other((size_t)1 << 18);
                for (int d = 1; d < n_gpu; ++d) {
                    int64_t no = 0;
                    Ls[d].check(qm_indel_table_fetch_host(qm_sample_indel_table(smps[d]), idxs[d], other.data(), (int64_t)other.size(), &no), "qm_indel_table_fetch_host");
                    tab = merge_indel_tables(tab, other.data(), no);
                }
                nt = (int64_t)tab.size();
            }
            std::vector<int32_t> rows(g.codes.size() * QM_NCH);
            L.check(qm_sample_counts_host(smp, rows.data()), "qm_sample_counts_host");
            for (int64_t i = 0; i < nt; ++i) {
                const qm_indel &x = tab[(size_t)i];
                const int dp = rows[(size_t)(g.offs[x.rid] + x.pos) * QM_NCH + 14], ad = x.n_fwd + x.n_rev;
                if (dp < copt.min_dp || ad < copt.min_alt || (double)ad < (double)copt.min_af * dp) continue;
                IndelCall c;
                c.a = x; c.dp = dp; c.af = dp > 0 ? (double)ad / dp : 0.0;
                const double f = c.af > 1.0 ? 1.0 : c.af, e = 0.002;     // same Chernoff-bound QUAL as the SNP records
                double kl = f > 0 ? f * log(f / e) : 0.0;
                if (f < 1.0) kl += (1.0 - f) * log((1.0 - f) / (1.0 - e));
                const double q = f > e ? 4.342944819032518 * dp * kl : 0.0;
                c.qual = q > 999.0 ? 999.0 : q;
                icalls.push_back(c);
            }
        }
        write_vcf(vcf, g, a.get("sample", "sample"), split(a.get("ref"), ',')[0], calls, icalls);
        // rule `bcftools` declares vcf_bgz = vcf + ".gz" and tabix-indexes it (rules/vcfcall.smk:107,118-119): written unless --vcf-gz 0
        if (atoi(a.get("vcf-gz", "1").c_str())) write_vcf_gz_tbi(vcf, vcf + ".gz", threads);
    }
    if (!mpileup.empty()) {
        const int64_t bytes = make_text();
        std::vector<char> text((size_t)bytes);
        L.check(qm_mpileup_text_fetch(L.ctx, text.data(), bytes), "qm_mpileup_text_fetch");
        FILE *fp = fopen(mpileup.c_str(), "w");
        if (!fp || (bytes && fwrite(text.data(), 1, (size_t)bytes, fp) != (size_t)bytes) || fclose(fp) != 0) die(2, "cannot write %s", mpileup.c_str());
        fprintf(stderr, "[qm_driver] text pileup: %lld bytes\n", (long long)bytes);
    }
}

// one contaminant pass of `sample --decontam` (rule rm_phix) or `--decontam2` (rule rm_human_ecoli): its genome and, per GPU, its
// index and filter-mode sample
struct Pass {
    Genome g;
    std::vector<qm_index *> idxs;
    std::vector<qm_sample *> smps;
};

int cmd_sample(const Args &a, const std::string &cmdline, bool decontam)
{
    PhaseClock pc;
    std::vector<const char *> known = {
        "ref", "r1", "r2", "sample", "bam", "counts", "vcf", "vcf-gz", "out-r1", "out-r2", "keep-contigs", "gpu", "gpus", "t", "threads",
        "batch-pairs", "rmdup", "rmdup-bam", "metrics", "no-rescue", "mpileup", "bwa-index", "fm-seeds", "indels", "max-depth", "baq",
        "min-mapq", "q", "min-bq", "Q", "count-orphans", "ignore-overlaps", "min-dp", "min-alt", "min-af", "print-options", "stage-ms",
        "w", "k", "c", "W", "D", "A", "B", "O", "E", "L", "U", "T", "d", "K", "I"};
    if (!decontam) known.insert(known.end(), {"decontam", "decontam2", "clean-r1", "clean-r2"});
    require_known(a, decontam ? "decontam" : "sample", known);
    // --decontam A.fa[,B.fa] [--decontam2 C.fa[,D.fa]]: rules rm_phix and rm_human_ecoli in this job, in front of the target
    // (--clean-r1 / --clean-r2: what the last pass keeps, as FASTQ)
    if (a.has("decontam2") && !a.has("decontam")) die(1, "--decontam2 needs --decontam (it is the second pass)");
    if (a.has("clean-r1") != a.has("clean-r2")) die(1, "--clean-r1 and --clean-r2 go together");
    if (a.has("clean-r1") && !a.has("decontam")) die(1, "--clean-r1 / --clean-r2 need --decontam");
    if (a.has("decontam") && a.has("keep-contigs")) die(1, "--decontam and --keep-contigs exclude each other (exact passes or the fused approximation)");
    const PairOptions pair_opts = parse_pair_options(a);
    const int64_t K = pair_opts.K;
    if (atoi(a.get("print-options", "0").c_str())) {   // host only: the alignment options this command line resolves to
        qm_opt o; qm_opt_default(&o);
        apply_bwa_options(a, o);
        if (atoi(a.get("no-rescue", "0").c_str())) o.flags |= QM_F_NO_RESCUE;
        if (a.has("bwa-index") || atoi(a.get("fm-seeds", "0").c_str())) o.flags |= QM_F_FM_SEEDS;
        qm_pileup_opt po; qm_pileup_opt_default(&po);
        apply_mpileup_options(a, po);
        print_options(o, po, pair_opts);
        return 0;
    }
    if (!a.has("ref") || !a.has("r1") || !a.has("r2")) die(1, "--ref, --r1 and --r2 are required");
    const std::string bam = a.get("bam"), counts = a.get("counts"), vcf = a.get("vcf"), o1 = a.get("out-r1"), o2 = a.get("out-r2");
    if (decontam && (o1.empty() || o2.empty())) die(1, "decontam needs --out-r1 and --out-r2");
    const int threads = std::max(1, atoi(a.get("t", a.get("threads", "4")).c_str()));
    g_threads = threads;
    // the insert-size model is fixed from the first QM_PESTAT_PAIRS pairs handed in: batches are never smaller than that,
    // so the records do not depend on the batch size
    const int64_t batch_pairs = std::max<int64_t>(QM_PESTAT_PAIRS, atoll(a.get("batch-pairs", "2000000").c_str()));
    const int keep_contigs = atoi(a.get("keep-contigs", "0").c_str());
    Genome g;
    load_refs(a.get("ref"), g);
    std::vector<Pass> passes;
    for (const char *k : {"decontam", "decontam2"})
        if (a.has(k)) { passes.emplace_back(); load_pass_refs(k, a.get(k), passes.back().g); }
    // --gpus A,B,C or A-B: one context, index and sample per GPU in this one process; batches are dealt round-robin, the
    // count tensors merged with one NCCL all-reduce (north_star).  --gpu I: the single-GPU form.
    std::vector<int> devs;
    if (a.has("gpus")) {
        for (auto &tok : split(a.get("gpus"), ',')) {
            const size_t dash = tok.find('-');
            if (dash != std::string::npos && dash > 0) { for (int d = atoi(tok.substr(0, dash).c_str()); d <= atoi(tok.substr(dash + 1).c_str()); ++d) devs.push_back(d); }
            else if (!tok.empty()) devs.push_back(atoi(tok.c_str()));
        }
        if (devs.empty()) die(1, "--gpus: no device given");
        for (size_t i = 0; i < devs.size(); ++i) {
            if (devs[i] < 0 || devs[i] > 1023) die(1, "--gpus: '%s' names no device list (A,B,.. or A-B)", a.get("gpus").c_str());
            for (size_t j = 0; j < i; ++j) if (devs[j] == devs[i]) die(1, "--gpus: device %d is listed twice", devs[i]);
        }
        if (decontam && devs.size() > 1) die(1, "decontam runs on one GPU (--gpu I)");
        if (K && a.has("decontam") && devs.size() > 1) die(1, "sample --decontam with -K runs on one GPU (--gpu I)");
    } else devs.push_back(atoi(a.get("gpu", "0").c_str()));
    const int n_gpu = (int)devs.size();
    std::vector<Lib> Ls((size_t)n_gpu);
    for (int d = 0; d < n_gpu; ++d) {
        const int rc = qm_ctx_create(devs[d], &Ls[d].ctx);
        if (rc != QM_OK) die(3, "qm_ctx_create(%d) failed (%d): no usable B200 (there is no CPU fallback)", devs[d], rc);
    }
    // --stage-ms 1: the library's CUDA-event stage timers on, one line per GPU in the log at the end (what a Snakemake
    // `benchmark:` file cannot show: where inside the job the device time went)
    const bool stage_ms = atoi(a.get("stage-ms", "0").c_str()) != 0;
    if (stage_ms) for (int d = 0; d < n_gpu; ++d) Ls[d].check(qm_profile_enable(Ls[d].ctx, 1), "qm_profile_enable");
    Lib &L = Ls[0];
    qm_opt opt; qm_opt_default(&opt);
    apply_bwa_options(a, opt);
    if (atoi(a.get("no-rescue", "0").c_str())) opt.flags |= QM_F_NO_RESCUE;          // bwa mem -S
    qm_pileup_opt popt; qm_pileup_opt_default(&popt);
    apply_mpileup_options(a, popt);
    // --bwa-index PREFIX: seeds through bwa's own index files PREFIX.bwt + PREFIX.sa (what `bwa index` left next to the genome,
    // rules/index.smk:13) -- bwa-mem's seeds (SMEMs, re-seeding, third round) instead of the k-mer hash index's exact matches;
    // --fm-seeds 1 rebuilds the same index from the FASTA when the files are not at hand
    std::vector<uint8_t> bwt_file, sa_file;
    const bool fm_build = atoi(a.get("fm-seeds", "0").c_str()) != 0;
    if (a.has("bwa-index")) {
        bwt_file = read_binary<uint8_t>(a.get("bwa-index") + ".bwt");
        sa_file = read_binary<uint8_t>(a.get("bwa-index") + ".sa");
    }
    const qm_opt pass_opt = opt;                       // the passes take bwa's options, not the target's seeding through bwa's index
    if (a.has("bwa-index") || fm_build) opt.flags |= QM_F_FM_SEEDS;
    std::vector<qm_index *> idxs((size_t)n_gpu, nullptr);
    std::vector<qm_sample *> smps((size_t)n_gpu, nullptr);
    for (int d = 0; d < n_gpu; ++d) {
        Ls[d].check(qm_index_build(Ls[d].ctx, g.codes.data(), (int)g.names.size(), g.lens.data(), opt.min_seed_len, &idxs[d]), "qm_index_build");
        if (!bwt_file.empty())
            Ls[d].check(qm_index_attach_bwa(Ls[d].ctx, idxs[d], bwt_file.data(), (int64_t)bwt_file.size(), sa_file.data(), (int64_t)sa_file.size()), "qm_index_attach_bwa");
        else if (fm_build) Ls[d].check(qm_index_build_fm(Ls[d].ctx, idxs[d], g.codes.data()), "qm_index_build_fm");
        Ls[d].check(qm_sample_begin(Ls[d].ctx, idxs[d], &opt, &popt, &smps[d]), "qm_sample_begin");
        if (pair_opts.has_I) Ls[d].check(qm_sample_set_pestat(smps[d], pair_opts.pes), "qm_sample_set_pestat");    // bwa mem -I
    }
    for (auto &ps : passes) {
        ps.idxs.assign((size_t)n_gpu, nullptr);
        ps.smps.assign((size_t)n_gpu, nullptr);
        for (int d = 0; d < n_gpu; ++d) {
            Ls[d].check(qm_index_build(Ls[d].ctx, ps.g.codes.data(), (int)ps.g.names.size(), ps.g.lens.data(), pass_opt.min_seed_len, &ps.idxs[d]),
                        "qm_index_build");
            Ls[d].check(qm_sample_begin(Ls[d].ctx, ps.idxs[d], &pass_opt, &popt, &ps.smps[d]), "qm_sample_begin");
            Ls[d].check(qm_sample_set_filter(ps.smps[d], 1), "qm_sample_set_filter");
            if (pair_opts.has_I) Ls[d].check(qm_sample_set_pestat(ps.smps[d], pair_opts.pes), "qm_sample_set_pestat");
        }
    }
    qm_index *idx = idxs[0];
    pc.mark("context + reference + index");
    qm_sample *smp = smps[0];

    const bool rmdup = !decontam && atoi(a.get("rmdup", "0").c_str()) != 0;
    const std::string rmdup_bam = a.get("rmdup-bam"), metrics = a.get("metrics");
    if (!rmdup && (!rmdup_bam.empty() || !metrics.empty())) die(1, "--rmdup-bam / --metrics need --rmdup 1");
    if (rmdup) for (int d = 0; d < n_gpu; ++d) Ls[d].check(qm_sample_set_rmdup(smps[d], 1), "qm_sample_set_rmdup");
    // --max-depth N: bcftools mpileup -d N (htslib's order-dependent depth cap); 0 / absent = no cap (DESIGN.md 5)
    const int max_depth = atoi(a.get("max-depth", "0").c_str());
    if (max_depth < 0) die(1, "--max-depth must be >= 0");
    if (max_depth > 0) for (int d = 0; d < n_gpu; ++d) Ls[d].check(qm_sample_set_max_depth(smps[d], max_depth), "qm_sample_set_max_depth");
    const bool deferred = rmdup || max_depth > 0;      // counting waits for the whole sample (qm_sample_finish / _finish_comm)
    // --baq 1: base alignment quality on, as both mpileups of the reference flow run (no -B at rules/vcfcall.smk:39,115): extended BAQ
    // caps the base qualities the counts, the calls and the text pileup see.  Off by default (the parity configuration is -B).
    const int baq = atoi(a.get("baq", "0").c_str()) ? 3 : 0;
    if (baq) for (int d = 0; d < n_gpu; ++d) Ls[d].check(qm_sample_set_baq(smps[d], baq), "qm_sample_set_baq");
    const std::string mpileup = a.get("mpileup");
    const bool want_bam = !bam.empty() || !rmdup_bam.empty();
    const bool want_batches = want_bam || !mpileup.empty();
    const bool keep = want_batches || decontam;       // records / reads needed after the batch loop
    FastqPairReader fr(a.get("r1"), a.get("r2"));
    std::deque<Batch> batches;                        // (a deque: the workers hold references while more batches arrive)
    std::vector<int> batch_dev;                       // the GPU each of them went to
    std::vector<int64_t> first_read;
    RawBatch raw;
    std::vector<int64_t> chunks;                      // -K: the chunks of the batch read last
    int64_t n_pairs = 0, kept = 0;
    FILE *f1 = nullptr, *f2 = nullptr;
    if (decontam) {
        f1 = fopen(o1.c_str(), "w"); f2 = fopen(o2.c_str(), "w");
        if (!f1 || !f2) die(2, "cannot create %s / %s", o1.c_str(), o2.c_str());
    }
    // one host thread per GPU (a context is not thread-safe, distinct contexts are independent); worker d holds at most one batch
    std::vector<std::thread> workers((size_t)n_gpu);
    std::vector<Batch *> in_flight((size_t)n_gpu, nullptr);
    auto join_worker = [&](int d) {
        if (workers[d].joinable()) workers[d].join();
        if (in_flight[d] && !want_batches) { free_batch(Ls[d], *in_flight[d]); }
        in_flight[d] = nullptr;
    };
    int64_t n_batches = 0;
    const auto t_loop = std::chrono::steady_clock::now();
    if (!passes.empty()) {
        // Stage s < P is contaminant pass s + 1, stage P the target.  Each stage fixes its insert-size model from the first batch it
        // gets, which must hold QM_PESTAT_PAIRS pairs or the whole rest of its input, as the stage's first FASTQ batch in the chain
        // does.  Until every stage has had such a batch the raw batches run here on GPU 0, and what a stage still without a model
        // receives waits in pend[s] (carried over to the next raw batch); then the models go to every GPU and each raw batch runs all
        // stages on its own GPU's worker while the next one is read.
        const int P = (int)passes.size();
        std::vector<std::vector<Batch>> pend((size_t)P + 1);
        std::vector<int64_t> pend_n((size_t)P + 1, 0), n_in((size_t)P + 1, 0);
        std::vector<bool> fixed((size_t)P + 1, false);
        const std::string c1 = a.get("clean-r1"), c2 = a.get("clean-r2");
        FILE *fc1 = nullptr, *fc2 = nullptr;
        if (!c1.empty()) {
            fc1 = fopen(c1.c_str(), "w"); fc2 = fopen(c2.c_str(), "w");
            if (!fc1 || !fc2) die(2, "cannot create %s / %s", c1.c_str(), c2.c_str());
        }
        // a pass on GPU d: `in` aligned with pair ids from id0, its kept pairs gathered into `out`, `in` released
        auto run_pass = [&](int d, int s, Batch &in, int64_t id0, Batch &out) {
            std::vector<uint8_t> kb((size_t)in.n_pairs);
            if (in.n_pairs > 0) {
                qm_sample *ps = passes[(size_t)s].smps[(size_t)d];
                if (K) Ls[d].check(qm_sample_set_chunks(ps, in.chunks.data(), (int64_t)in.chunks.size()), "qm_sample_set_chunks");
                Ls[d].check(qm_sample_add_pairs_host_packed(ps, in.bases2, in.nmask, in.quals, in.stride, in.lens, in.n_pairs, id0, nullptr),
                            "qm_sample_add_pairs_host_packed");
                Ls[d].check(qm_sample_keep_host(ps, kb.data(), in.n_pairs, nullptr), "qm_sample_keep_host");
            }
            gather_pairs(Ls[d], {&in}, {kb.data()}, out);
            free_batch(Ls[d], in);
        };
        // the target on GPU d: records as `sample` keeps them; the batch is then stored (BAM / text pileup) or released
        auto run_target = [&](int d, Batch &b, int64_t id0) {
            void *p = nullptr;
            if (keep) { Ls[d].check(qm_host_alloc(Ls[d].ctx, (size_t)2 * b.n_pairs * sizeof(qm_aln), &p), "qm_host_alloc"); b.alns = (qm_aln *)p; }
            if (b.n_pairs > 0 && K) Ls[d].check(qm_sample_set_chunks(smps[d], b.chunks.data(), (int64_t)b.chunks.size()), "qm_sample_set_chunks");
            if (b.n_pairs > 0)
                Ls[d].check(qm_sample_add_pairs_host_packed(smps[d], b.bases2, b.nmask, b.quals, b.stride, b.lens, b.n_pairs, id0, b.alns),
                            "qm_sample_add_pairs_host_packed");
        };
        auto write_clean = [&](const Batch &b) { if (fc1) for (int64_t p = 0; p < b.n_pairs; ++p) write_fastq_pair(fc1, fc2, b, p); };
        auto store = [&](int d, Batch &b, Batch *slot) {
            if (slot) *slot = std::move(b);
            else free_batch(Ls[d], b);
        };
        // startup (GPU 0): `cur` enters stage s (eof: no more input, a stage without a model takes what it has)
        auto advance = [&](int s, Batch cur, bool has, bool eof) {
            for (; s <= P; ++s) {
                if (!fixed[(size_t)s]) {
                    if (has) { pend_n[(size_t)s] += cur.n_pairs; pend[(size_t)s].push_back(std::move(cur)); }
                    if (pend_n[(size_t)s] < QM_PESTAT_PAIRS && !eof) return;
                    std::vector<Batch> &q = pend[(size_t)s];
                    if (q.empty()) return;
                    if (q.size() == 1) cur = std::move(q[0]);
                    else {
                        std::vector<const Batch *> src;
                        for (auto &x : q) src.push_back(&x);
                        Batch m;
                        gather_pairs(L, src, std::vector<const uint8_t *>(q.size(), nullptr), m);
                        for (auto &x : q) free_batch(L, x);
                        cur = std::move(m);
                        const std::string stage = s < P ? "pass " + std::to_string(s + 1) : std::string("the target");
                        fprintf(stderr, "[qm_driver] decontam: the first batch of %s (%lld pairs) carries over the pairs of %zu raw batches\n",
                                stage.c_str(), (long long)cur.n_pairs, q.size());
                    }
                    q.clear();
                    pend_n[(size_t)s] = 0;
                    fixed[(size_t)s] = true;
                    has = true;
                }
                const int64_t id0 = n_in[(size_t)s];
                n_in[(size_t)s] += cur.n_pairs;
                if (s < P) {
                    Batch out;
                    run_pass(0, s, cur, id0, out);
                    cur = std::move(out);
                } else {
                    Batch *slot = nullptr;
                    if (want_batches) { batches.emplace_back(); batch_dev.push_back(0); slot = &batches.back(); }
                    run_target(0, cur, id0);
                    write_clean(cur);
                    store(0, cur, slot);
                }
            }
        };
        // -K (GPU 0): every stage cuts bwa's chunks over its own input stream -- pass 1 over the FASTQ, pass 2 over pass 1's survivors,
        // the target over pass 2's -- as the chain `decontam -K | decontam -K | sample -K` does.  What a stage receives waits in
        // pend[s] (which always starts at a chunk start) until chunks close; the closed chunks run as one add call, the open one's
        // pairs stay for the next batch; eof: the rest is the stage's last chunk.
        auto advance_k = [&](int s, Batch cur, bool has, bool eof) {
            for (; s <= P; ++s) {
                std::vector<Batch> &q = pend[(size_t)s];
                if (has && cur.n_pairs > 0) q.push_back(std::move(cur));
                else if (has) free_batch(L, cur);
                has = false;
                std::vector<int64_t> chunks;
                int64_t sum = 0, open = 0, done = 0;
                for (const Batch &x : q)
                    for (int64_t p = 0; p < x.n_pairs; ++p) {
                        sum += x.lens[2 * p] + x.lens[2 * p + 1];
                        ++open;
                        if (sum >= K) { chunks.push_back(open); done += open; sum = 0; open = 0; }
                        else if (open >= QM_CHUNK_MAX_PAIRS)
                            die(1, "option -K: a chunk of %lld bases runs past %d pairs, the most one chunk may hold (QM_CHUNK_MAX_PAIRS); "
                                   "choose a smaller -K", (long long)K, QM_CHUNK_MAX_PAIRS);
                    }
                if (eof && open) { chunks.push_back(open); done += open; open = 0; }
                if (done == 0) { if (eof) continue; return; }
                // the closed chunks' pairs as one batch, the open chunk's pairs as the new pend[s]
                std::vector<const Batch *> src;
                std::vector<std::vector<uint8_t>> head_mask(q.size()), rest_mask(q.size());
                std::vector<const uint8_t *> hm, rm;
                int64_t left = done;
                for (size_t k = 0; k < q.size(); ++k) {
                    src.push_back(&q[k]);
                    head_mask[k].assign((size_t)q[k].n_pairs, 0);
                    rest_mask[k].assign((size_t)q[k].n_pairs, 1);
                    for (int64_t p = 0; p < q[k].n_pairs && left > 0; ++p, --left) { head_mask[k][(size_t)p] = 1; rest_mask[k][(size_t)p] = 0; }
                    hm.push_back(head_mask[k].data()); rm.push_back(rest_mask[k].data());
                }
                Batch head, rest;
                gather_pairs(L, src, hm, head);
                if (open > 0) gather_pairs(L, src, rm, rest);
                for (auto &x : q) free_batch(L, x);
                q.clear();
                pend_n[(size_t)s] = rest.n_pairs;
                if (rest.n_pairs > 0) q.push_back(std::move(rest));
                head.chunks = std::move(chunks);
                const int64_t id0 = n_in[(size_t)s];
                n_in[(size_t)s] += head.n_pairs;
                if (s < P) {
                    Batch out;
                    run_pass(0, s, head, id0, out);
                    cur = std::move(out);
                    has = true;
                } else {
                    Batch *slot = nullptr;
                    if (want_batches) { batches.emplace_back(); batch_dev.push_back(0); slot = &batches.back(); }
                    run_target(0, head, id0);
                    write_clean(head);
                    store(0, head, slot);
                }
            }
        };
        Ledger ledger;
        int64_t n_par = 0;                              // raw batches run by the workers
        while (read_batch(fr, batch_pairs, raw)) {
            const bool startup = !std::all_of(fixed.begin(), fixed.end(), [](bool f) { return f; });
            const int d = startup ? 0 : batch_gpu(n_batches, n_gpu);
            join_worker(d);
            Batch b;
            pack_batch(Ls[d], raw, false, b);
            ++n_batches;
            if (K) { advance_k(0, std::move(b), true, false); continue; }
            if (startup) {
                advance(0, std::move(b), true, false);
                if (std::all_of(fixed.begin(), fixed.end(), [](bool f) { return f; })) {
                    // every stage has its model: every GPU gets it, the ledger starts where the startup left off
                    for (int s = 0; s <= P && n_gpu > 1; ++s) {
                        qm_sample *s0 = s < P ? passes[(size_t)s].smps[0] : smp;
                        qm_pestat pes[4];
                        L.check(qm_sample_get_pestat(s0, pes), "qm_sample_get_pestat");
                        for (int e = 1; e < n_gpu; ++e)
                            Ls[e].check(qm_sample_set_pestat(s < P ? passes[(size_t)s].smps[(size_t)e] : smps[e], pes), "qm_sample_set_pestat");
                    }
                    ledger.turn.assign((size_t)P + 2, 0);
                    ledger.total = n_in;
                    ledger.total.push_back(0);
                }
                continue;
            }
            Batch *slot = nullptr;
            if (want_batches) { batches.emplace_back(); batch_dev.push_back(d); slot = &batches.back(); }
            const int64_t j = n_par++;
            workers[d] = std::thread([&, d, j, slot, cur = std::move(b)]() mutable {
                for (int s = 0; s < P; ++s) {
                    const int64_t id0 = ledger.take(s, j, cur.n_pairs);
                    Batch out;
                    run_pass(d, s, cur, id0, out);
                    cur = std::move(out);
                }
                run_target(d, cur, ledger.take(P, j, cur.n_pairs));
                ledger.begin(P + 1, j);
                write_clean(cur);
                ledger.end(P + 1, 0);
                store(d, cur, slot);
            });
        }
        for (int d = 0; d < n_gpu; ++d) join_worker(d);
        if (K) advance_k(0, Batch(), false, true);
        else if (n_par > 0) n_in.assign(ledger.total.begin(), ledger.total.begin() + P + 1);
        else for (int s = 0; s <= P; ++s) if (!fixed[(size_t)s]) { advance(s, Batch(), false, true); break; }
        if (fc1 && (fclose(fc1) != 0 || fclose(fc2) != 0)) die(2, "write error on %s / %s", c1.c_str(), c2.c_str());
        for (int s = 0; s < P; ++s)
            fprintf(stderr, "[qm_driver] decontam pass %d: %lld of %lld pairs kept\n", s + 1, (long long)n_in[(size_t)s + 1], (long long)n_in[(size_t)s]);
        n_pairs = n_in[(size_t)P];
        int64_t r0 = 0;
        for (auto &b : batches) { first_read.push_back(r0); r0 += 2 * b.n_pairs; }
    } else while (read_batch(fr, batch_pairs, raw, K, &chunks)) {
        const int d = batch_gpu(n_batches, n_gpu);
        join_worker(d);
        batches.emplace_back();
        batch_dev.push_back(d);
        Batch &b = batches.back();
        pack_batch(Ls[d], raw, keep, b);
        // -K: the batch holds whole chunks of bwa's (read_batch), so whole chunks are dealt to the GPUs; each GPU estimates the
        // models of its own chunks and none is broadcast
        if (K) b.chunks = chunks;
        const int64_t pair0 = n_pairs;
        if (n_batches == 0 || decontam) {
            // (later batches go to a worker thread, also with one GPU: the next batch is read and packed while this one is on the device)
            // the first batch fixes the sample's insert-size model (its first QM_PESTAT_PAIRS pairs): every GPU gets that model
            // before it sees a batch of its own, so the records do not depend on the number of GPUs
            if (K) L.check(qm_sample_set_chunks(smp, b.chunks.data(), (int64_t)b.chunks.size()), "qm_sample_set_chunks");
            L.check(qm_sample_add_pairs_host_packed(smp, b.bases2, b.nmask, b.quals, b.stride, b.lens, b.n_pairs, pair0, b.alns), "qm_sample_add_pairs_host_packed");
            if (n_gpu > 1 && !K) {
                qm_pestat pes[4];
                L.check(qm_sample_get_pestat(smp, pes), "qm_sample_get_pestat");
                for (int e = 1; e < n_gpu; ++e) Ls[e].check(qm_sample_set_pestat(smps[e], pes), "qm_sample_set_pestat");
            }
        } else {
            in_flight[d] = &b;
            workers[d] = std::thread([&Ls, &smps, d, &b, pair0, K]() {
                if (K) Ls[d].check(qm_sample_set_chunks(smps[d], b.chunks.data(), (int64_t)b.chunks.size()), "qm_sample_set_chunks");
                Ls[d].check(qm_sample_add_pairs_host_packed(smps[d], b.bases2, b.nmask, b.quals, b.stride, b.lens, b.n_pairs, pair0, b.alns), "qm_sample_add_pairs_host_packed");
            });
        }
        if (decontam) {
            for (int64_t p = 0; p < b.n_pairs; ++p) {
                const qm_aln &x = b.alns[2 * p], &y = b.alns[2 * p + 1];
                bool ok;
                if (keep_contigs > 0)      // fused pass: drop iff a mate sits on a contaminant contig
                    ok = !(!(x.flag & 4) && x.rid >= keep_contigs) && !(!(y.flag & 4) && y.rid >= keep_contigs);
                else                       // samtools view -f 12 -F 256 on each record
                    ok = (x.flag & 12) == 12 && !(x.flag & 256) && (y.flag & 12) == 12 && !(y.flag & 256);
                if (ok) { write_fastq_pair(f1, f2, b, p); ++kept; }
            }
        }
        first_read.push_back(2 * n_pairs);
        n_pairs += b.n_pairs;
        ++n_batches;
        if (!want_batches && in_flight[d] == nullptr) { free_batch(Ls[d], b); }
        if (!want_batches && n_gpu == 1 && in_flight[d] == nullptr) { batches.pop_back(); batch_dev.pop_back(); }
    }
    for (int d = 0; d < n_gpu; ++d) join_worker(d);
    const double loop_s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_loop).count();
    pc.mark("FASTQ -> records + counts");
    if (decontam) {
        if (fclose(f1) != 0 || fclose(f2) != 0) die(2, "write error on the cleaned FASTQ files");
        fprintf(stderr, "[qm_driver] decontam: %lld of %lld pairs kept\n", (long long)kept, (long long)n_pairs);
    }
    int64_t cells = 0;
    for (int d = 0; d < n_gpu; ++d) {
        int64_t c = 0;
        Ls[d].check(qm_sample_stats_sync(smps[d], nullptr, &c, nullptr), "qm_sample_stats_sync");
        cells += c;
    }
    fprintf(stderr, "[qm_driver] %lld pairs aligned, %lld extension cells\n", (long long)n_pairs, (long long)cells);
    fprintf(stderr, "[qm_driver] %d GPU(s), %lld batch(es): %.2f s from the first read to the last record, %.3f M pairs/s, %.1f G extension cells/s "
                    "(FASTQ parsing included)\n", n_gpu, (long long)n_batches, loop_s, loop_s > 0 ? n_pairs / loop_s / 1e6 : 0.0,
            loop_s > 0 ? cells / loop_s / 1e9 : 0.0);
    if (stage_ms) for (int d = 0; d < n_gpu; ++d) print_stage_ms(Ls[d], devs[d]);
    int64_t n_dup = 0, n_capped = 0;
    if (n_gpu > 1) {
        // per-GPU int32 count tensors -> one NCCL all-reduce over NVLink; every GPU ends up with the sample's totals.  Deferred
        // counting first: every GPU marks duplicates and applies the cap over the tuples of the whole sample, counts its survivors
        std::vector<qm_ctx *> ctxs;
        for (auto &x : Ls) ctxs.push_back(x.ctx);
        std::vector<qm_comm *> comms((size_t)n_gpu, nullptr);
        L.check(qm_comm_init_all(n_gpu, ctxs.data(), comms.data()), "qm_comm_init_all");
        std::vector<std::thread> team;
        std::vector<int64_t> nd((size_t)n_gpu, 0), ncap((size_t)n_gpu, 0);
        for (int d = 0; d < n_gpu; ++d)
            team.emplace_back([&, d]() {
                if (deferred) Ls[d].check(qm_sample_finish_comm(smps[d], comms[d], &nd[(size_t)d], &ncap[(size_t)d], nullptr), "qm_sample_finish_comm");
                Ls[d].check(qm_counts_allreduce(Ls[d].ctx, comms[d], qm_sample_counts(smps[d]), (int64_t)QM_NCH * (int64_t)g.codes.size(), nullptr),
                            "qm_counts_allreduce");
                Ls[d].check(qm_sample_stats_sync(smps[d], nullptr, nullptr, nullptr), "qm_sample_stats_sync");
            });
        for (auto &t : team) t.join();
        for (auto c : comms) qm_comm_destroy(c);
        n_dup = nd[0]; n_capped = ncap[0];                 // sample-wide, the same on every GPU
        fprintf(stderr, "[qm_driver] count tensors of %d GPUs merged (ncclAllReduce, int32 sum, %lld values)\n", n_gpu,
                (long long)QM_NCH * (long long)g.codes.size());
    } else if (deferred) L.check(qm_sample_finish(smp, &n_dup, &n_capped, nullptr), "qm_sample_finish");
    if (deferred) {
        if (rmdup) fprintf(stderr, "[qm_driver] rmdup: %lld of %lld pairs are duplicates\n", (long long)n_dup, (long long)n_pairs);
        if (max_depth > 0) fprintf(stderr, "[qm_driver] depth cap %d: %lld reads dropped by the pileup iterator\n", max_depth, (long long)n_capped);
    }
    if (rmdup) {
        if (want_batches) {                            // final flags of every record, batch by batch, from the GPU that held the batch
            std::vector<int64_t> bp;
            for (auto &b : batches) bp.push_back(b.n_pairs);
            const auto src = batch_sources(bp, batch_dev, n_gpu);
            std::vector<std::vector<qm_aln>> all((size_t)n_gpu);
            for (size_t i = 0; i < bp.size(); ++i) all[(size_t)src[i].first].resize((size_t)(src[i].second + 2 * bp[i]));
            for (int d = 0; d < n_gpu; ++d)
                Ls[d].check(qm_sample_kept_alns_host(smps[d], all[(size_t)d].data(), (int64_t)all[(size_t)d].size()), "qm_sample_kept_alns_host");
            for (size_t i = 0; i < bp.size(); ++i)
                memcpy(batches[i].alns, all[(size_t)src[i].first].data() + src[i].second, (size_t)2 * bp[i] * sizeof(qm_aln));
        }
        if (!metrics.empty()) write_dup_metrics(metrics, a.get("sample", "sample"), n_pairs, n_dup);
    }

    pc.mark("merge / deferred counting");
    write_outputs(a, g, Ls, idxs, smps, threads, [&]() {
        // text pileup (samtools mpileup format) of the whole sample: records, reads and qualities go to the device once more,
        // at one common stride; the text comes back in one piece
        int32_t stride = 1;
        for (auto &b : batches) stride = std::max(stride, b.stride);
        std::vector<qm_aln> alns((size_t)2 * n_pairs);
        std::vector<uint8_t> codes((size_t)2 * n_pairs * stride, 4), quals((size_t)2 * n_pairs * stride, 0);
        std::vector<int32_t> lens((size_t)2 * n_pairs);
        size_t r0 = 0;
        for (auto &b : batches) {
            for (int64_t r = 0; r < 2 * b.n_pairs; ++r) {
                alns[r0 + r] = b.alns[r]; lens[r0 + r] = b.lens[r];
                memcpy(&codes[(r0 + r) * stride], b.codes + (size_t)r * b.stride, (size_t)b.lens[r]);
                memcpy(&quals[(r0 + r) * stride], b.quals + (size_t)r * b.stride, (size_t)b.lens[r]);
            }
            r0 += (size_t)2 * b.n_pairs;
        }
        std::vector<const char *> nm;
        for (auto &s : g.names) nm.push_back(s.c_str());
        if (baq) {                                   // samtools mpileup without -B: the text shows the capped qualities
            std::vector<uint8_t> capped(quals.size());
            L.check(qm_baq_apply_host(L.ctx, idx, &popt, alns.data(), codes.data(), quals.data(), stride, lens.data(), 2 * n_pairs, baq, capped.data()),
                    "qm_baq_apply_host");
            quals.swap(capped);
        }
        int64_t bytes = 0;
        L.check(qm_mpileup_text_host(L.ctx, idx, &popt, alns.data(), codes.data(), quals.data(), stride, lens.data(), n_pairs, nm.data(), &bytes),
                "qm_mpileup_text_host");
        return bytes;
    });
    pc.mark("count TSV + calls + VCF + text pileup");
    if (want_bam) {
        // coordinate sort on the device: keys from the records, stable radix sort, gather through the permutation
        int pos_bits = 0;
        const int key_bits = sort_key_bits(g, pos_bits);
        std::vector<uint64_t> keys((size_t)2 * n_pairs);
        size_t k = 0;
        for (auto &b : batches)
            for (int64_t r = 0; r < 2 * b.n_pairs; ++r, ++k)
                keys[k] = qm_sort_key(b.alns[r].rid, b.alns[r].pos, (b.alns[r].flag & 0x10) != 0, (int)g.names.size(), pos_bits);
        std::vector<uint32_t> perm(keys.size());
        L.check(qm_sort_keys_host(L.ctx, keys.data(), (int64_t)keys.size(), key_bits, perm.data()), "qm_sort_keys_host");
        pc.mark("coordinate sort");
        if (!bam.empty()) write_bam(bam, g, batches, perm, first_read, cmdline, threads);
        pc.mark("BAM + BAI");
        if (!rmdup_bam.empty()) {                      // REMOVE_DUPLICATES=true: the same order without the flagged records
            std::vector<uint32_t> kept_perm;
            kept_perm.reserve(perm.size());
            for (uint32_t gr : perm) {
                const size_t bi = (size_t)(std::upper_bound(first_read.begin(), first_read.end(), (int64_t)gr) - first_read.begin()) - 1;
                if (!(batches[bi].alns[gr - first_read[bi]].flag & 0x400)) kept_perm.push_back(gr);
            }
            write_bam(rmdup_bam, g, batches, kept_perm, first_read, cmdline, threads);
        }
    }
    for (auto &b : batches) free_batch(L, b);
    for (int d = 0; d < n_gpu; ++d) {
        for (auto &ps : passes) { qm_sample_destroy(ps.smps[(size_t)d]); qm_index_destroy(Ls[d].ctx, ps.idxs[(size_t)d]); }
        qm_sample_destroy(smps[d]);
        qm_index_destroy(Ls[d].ctx, idxs[d]);
        qm_ctx_destroy(Ls[d].ctx);
    }
    pc.mark("release");
    pc.report();
    return 0;
}

template <class T> std::vector<T> read_binary(const std::string &path)
{
    FILE *fp = fopen(path.c_str(), "rb");
    if (!fp) die(2, "cannot open %s", path.c_str());
    fseek(fp, 0, SEEK_END);
    const long sz = ftell(fp);
    fseek(fp, 0, SEEK_SET);
    if (sz < 0 || (size_t)sz % sizeof(T)) die(2, "%s: size is not a multiple of %zu", path.c_str(), sizeof(T));
    std::vector<T> v((size_t)sz / sizeof(T));
    if (!v.empty() && fread(v.data(), sizeof(T), v.size(), fp) != v.size()) die(2, "read error in %s", path.c_str());
    fclose(fp);
    return v;
}

// the BAM/BAI writer alone: records given as a binary file of qm_aln (2 per pair, input order)
int cmd_bam_from_records(const Args &a, const std::string &cmdline)
{
    require_known(a, "bam-from-records", {"ref", "r1", "r2", "alns", "perm", "bam", "gpu", "t"});
    if (!a.has("ref") || !a.has("r1") || !a.has("r2") || !a.has("alns") || !a.has("bam")) die(1, "--ref --r1 --r2 --alns --bam are required");
    Genome g;
    load_refs(a.get("ref"), g);
    std::vector<qm_aln> alns = read_binary<qm_aln>(a.get("alns"));
    FastqPairReader fr(a.get("r1"), a.get("r2"));
    RawBatch raw;
    read_batch(fr, (int64_t)1 << 40, raw);
    if (raw.size() * 2 != alns.size()) die(2, "%zu records for %zu pairs", alns.size(), raw.size());
    // host-only path: plain memory instead of page-locked buffers, no context
    Batch b;
    b.n_pairs = (int64_t)raw.size();
    const Side *sd[2] = {&raw.a, &raw.b};
    size_t mx = 1;
    for (int m = 0; m < 2; ++m)
        for (size_t i = 0; i < sd[m]->n; ++i) mx = std::max(mx, sd[m]->len(i));
    b.stride = (int32_t)mx;
    std::vector<uint8_t> codes(2 * raw.size() * mx, 4), quals(2 * raw.size() * mx, 0);
    std::vector<int32_t> lens(2 * raw.size());
    static uint8_t lut[256];
    memset(lut, 4, sizeof lut);
    lut['A'] = lut['a'] = 0; lut['C'] = lut['c'] = 1; lut['G'] = lut['g'] = 2; lut['T'] = lut['t'] = 3;
    b.names.assign(raw.a.names.begin(), raw.a.names.end());
    b.name_off = raw.a.noff;
    for (size_t i = 0; i < raw.size(); ++i) {
        for (int m = 0; m < 2; ++m) {
            const char *s = sd[m]->seq.data() + sd[m]->soff[i], *q = sd[m]->qual.data() + sd[m]->soff[i];
            const size_t n = sd[m]->len(i);
            for (size_t j = 0; j < n; ++j) { codes[(2 * i + m) * mx + j] = lut[(unsigned char)s[j]]; quals[(2 * i + m) * mx + j] = (uint8_t)(q[j] - 33); }
            lens[2 * i + m] = (int32_t)n;
        }
    }
    b.codes = codes.data(); b.quals = quals.data(); b.lens = lens.data(); b.alns = alns.data();
    std::vector<uint32_t> perm;
    if (a.has("perm")) perm = read_binary<uint32_t>(a.get("perm"));
    else {
        Lib L;
        int rc = qm_ctx_create(atoi(a.get("gpu", "0").c_str()), &L.ctx);
        if (rc != QM_OK) die(3, "qm_ctx_create failed (%d): no usable B200 (pass --perm to write a BAM without sorting)", rc);
        int pos_bits = 0;
        const int key_bits = sort_key_bits(g, pos_bits);
        std::vector<uint64_t> keys(alns.size());
        for (size_t r = 0; r < alns.size(); ++r) keys[r] = qm_sort_key(alns[r].rid, alns[r].pos, (alns[r].flag & 0x10) != 0, (int)g.names.size(), pos_bits);
        perm.resize(keys.size());
        L.check(qm_sort_keys_host(L.ctx, keys.data(), (int64_t)keys.size(), key_bits, perm.data()), "qm_sort_keys_host");
        qm_ctx_destroy(L.ctx);
    }
    if (perm.size() != alns.size()) die(2, "permutation of %zu entries for %zu records", perm.size(), alns.size());
    std::deque<Batch> batches;
    batches.push_back(b);
    write_bam(a.get("bam"), g, batches, perm, {0}, cmdline, std::max(1, atoi(a.get("t", "2").c_str())));
    return 0;
}


// ------------------------------------------------------------------------------------------------
constexpr int QM_DUP_COORD_BIAS = 4096;          // the end code's coordinate bias (qm_bam_mark_duplicates: -4095 .. 2^26 - 4096)

// BAM reader (`pileup`): the input of the reference's rules `mpileup` and `bcftools` (rules/vcfcall.smk:39,115 read
// {sample}.{ref_name}.rmdup.bam).  Everything here runs before a CUDA context exists, so a bad file fails the same way with
// or without a GPU.
inline uint32_t le16(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8; }
inline uint32_t le32(const uint8_t *p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24; }

// the whole file, BGZF members inflated on the -t threads into one stream.  Every member's gzip header and BC field, its CRC32
// and ISIZE, and the end-of-file block are checked (a file cut at a block boundary still lacks the EOF block).
std::vector<uint8_t> inflate_bgzf(const std::string &path)
{
    std::vector<uint8_t> raw;
    {
        const int fd = open(path.c_str(), O_RDONLY);
        if (fd < 0) die(2, "cannot open %s", path.c_str());
        const off_t sz = lseek(fd, 0, SEEK_END);
        if (sz < 0) die(2, "cannot read %s", path.c_str());
        raw.resize((size_t)sz);
        size_t got = 0;
        while (got < raw.size()) {
            const ssize_t n = pread(fd, raw.data() + got, raw.size() - got, (off_t)got);
            if (n < 0 && errno == EINTR) continue;
            if (n <= 0) die(2, "read error in %s", path.c_str());
            got += (size_t)n;
        }
        close(fd);
    }
    struct Member { size_t off, data, clen, uoff; uint32_t isize; };
    std::vector<Member> mem;
    size_t p = 0, total = 0;
    while (p < raw.size()) {
        const uint8_t *h = raw.data() + p;
        if (raw.size() - p < 18) die(2, "%s: truncated BGZF block at byte %zu", path.c_str(), p);
        if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4))
            die(2, "%s: bad BGZF magic at byte %zu: not a BGZF-compressed BAM", path.c_str(), p);
        const size_t xlen = le16(h + 10);
        size_t bsize = 0;
        for (size_t x = 12; x + 4 <= 12 + xlen && p + x + 4 <= raw.size();) {
            const size_t slen = le16(h + x + 2);
            if (h[x] == 'B' && h[x + 1] == 'C' && slen == 2 && p + x + 6 <= raw.size()) bsize = le16(h + x + 4) + 1;
            x += 4 + slen;
        }
        if (bsize == 0) die(2, "%s: bad BGZF magic at byte %zu: gzip member without a BC field", path.c_str(), p);
        if (bsize < 12 + xlen + 8) die(2, "%s: BGZF block at byte %zu is too short", path.c_str(), p);
        if (p + bsize > raw.size()) die(2, "%s: truncated BGZF block at byte %zu", path.c_str(), p);
        const uint32_t isize = le32(h + bsize - 4);
        if (isize > 65536) die(2, "%s: BGZF block at byte %zu claims %u bytes (at most 65536)", path.c_str(), p, isize);
        mem.push_back({p, p + 12 + xlen, bsize - 12 - xlen - 8, total, isize});
        total += isize;
        p += bsize;
    }
    static const uint8_t kEof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    if (mem.empty() || raw.size() - mem.back().off != 28 || memcmp(raw.data() + mem.back().off, kEof, 28) != 0)
        die(2, "%s: no BGZF end-of-file block: the file is truncated", path.c_str());
    std::vector<uint8_t> out(total);
    std::vector<uint8_t> err(mem.size(), 0);                   // 1 does not inflate to ISIZE, 2 CRC32 mismatch
    std::atomic<size_t> next{0};
    auto work = [&]() {
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        if (inflateInit2(&zs, -15) != Z_OK) return;
        for (size_t i; (i = next.fetch_add(64)) < mem.size();)
            for (size_t k = i; k < std::min(mem.size(), i + 64); ++k) {
                const Member &m = mem[k];
                inflateReset(&zs);
                zs.next_in = raw.data() + m.data; zs.avail_in = (uInt)m.clen;
                zs.next_out = out.data() + m.uoff; zs.avail_out = m.isize;
                uint8_t spare;
                if (m.isize == 0) { zs.next_out = &spare; zs.avail_out = 1; }
                if (inflate(&zs, Z_FINISH) != Z_STREAM_END || zs.total_out != m.isize) { err[k] = 1; continue; }
                const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), out.data() + m.uoff, m.isize);
                if (crc != le32(raw.data() + m.data + m.clen)) err[k] = 2;
            }
        inflateEnd(&zs);
    };
    std::vector<std::thread> team;
    for (int t = 1; t < std::min<int>(g_threads, (int)(mem.size() / 64) + 1); ++t) team.emplace_back(work);
    work();
    for (auto &t : team) t.join();
    for (size_t k = 0; k < mem.size(); ++k) {
        if (err[k] == 1) die(2, "%s: BGZF block at byte %zu does not inflate to its ISIZE of %u bytes", path.c_str(), mem[k].off, mem[k].isize);
        if (err[k] == 2) die(2, "%s: CRC32 mismatch in the BGZF block at byte %zu", path.c_str(), mem[k].off);
    }
    return out;
}

// what the validation walk leaves for the device: the byte offsets of the records the pileup may admit, in file order
struct BamRecords {
    std::vector<int64_t> off;
    int32_t max_len = 0;
    int64_t n_total = 0, n_left_out = 0;
};

// The header must list the FASTA's contigs (names, lengths, order), as bcftools refuses a mismatched -f; then one walk over the
// records: coordinate order (as htslib's pileup checks it: placed records without 0x4, contig, then position), and on every
// record the pileup may admit what the device decode relies on.  Records neither mpileup admits (0x4, 0x100, 0x200, 0x400, no
// contig, no CIGAR) are left out.  Every failure names the read and exits 2.
BamRecords scan_bam(const std::string &path, const std::vector<uint8_t> &d, const Genome &g)
{
    const char *fn = path.c_str();
    if (d.size() < 12 || memcmp(d.data(), "BAM\1", 4) != 0) die(2, "%s: bad BAM magic: not a BAM file", fn);
    size_t p = 8 + (size_t)le32(d.data() + 4);
    if (p + 4 > d.size()) die(2, "%s: truncated BAM header", fn);
    const uint32_t n_ref = le32(d.data() + p);
    p += 4;
    std::vector<std::string> names;
    std::vector<int64_t> lens;
    for (uint32_t i = 0; i < n_ref; ++i) {
        if (p + 4 > d.size()) die(2, "%s: truncated BAM header", fn);
        const size_t ln = le32(d.data() + p);
        if (ln < 1 || p + 8 + ln > d.size()) die(2, "%s: truncated BAM header", fn);
        names.emplace_back((const char *)d.data() + p + 4, ln - 1);
        lens.push_back((int64_t)le32(d.data() + p + 4 + ln));
        p += 8 + ln;
    }
    if (names.size() != g.names.size())
        die(2, "%s: the header lists %zu contigs (@SQ), the reference %zu: the BAM was not aligned to this reference", fn, names.size(), g.names.size());
    for (size_t i = 0; i < names.size(); ++i)
        if (names[i] != g.names[i] || lens[i] != g.lens[i])
            die(2, "%s: @SQ %zu is %s of %lld bp, contig %zu of the reference is %s of %lld bp: the BAM was not aligned to this reference",
                fn, i + 1, names[i].c_str(), (long long)lens[i], i + 1, g.names[i].c_str(), (long long)g.lens[i]);
    // the record offsets (a serial chain of block_size fields) and the coordinate order
    std::vector<int64_t> all;
    int32_t last_tid = -1, last_pos = -1;
    for (; p < d.size();) {
        if (p + 36 > d.size()) die(2, "%s: truncated record at byte %zu of the BAM stream", fn, p);
        const uint8_t *r = d.data() + p;
        const size_t bs = le32(r);
        if (bs < 32 || p + 4 + bs > d.size() || 32 + (size_t)r[12] > bs) die(2, "%s: malformed or truncated record at byte %zu of the BAM stream", fn, p);
        const int32_t tid = (int32_t)le32(r + 4), pos = (int32_t)le32(r + 8);
        if (tid >= 0 && !(le16(r + 18) & 0x4)) {
            if (tid < last_tid || (tid == last_tid && pos < last_pos))
                die(2, "%s: the file is not coordinate-sorted: read %.*s at %s:%d comes after %s:%d", fn, std::max(0, (int)r[12] - 1), (const char *)r + 36,
                    tid < (int32_t)names.size() ? names[(size_t)tid].c_str() : "?", pos + 1, names[(size_t)last_tid].c_str(), last_pos + 1);
            last_tid = tid; last_pos = pos;
        }
        all.push_back((int64_t)p);
        p += 4 + bs;
    }
    // the per-record checks, on the -t threads; the first failure in file order is reported
    std::vector<uint8_t> keep(all.size(), 0);
    std::vector<std::pair<size_t, std::string>> bad;
    std::mutex mu;
    parallel_ranges(all.size(), [&](size_t b, size_t e) {
        for (size_t i = b; i < e; ++i) {
            const uint8_t *r = d.data() + all[i];
            const size_t bs = le32(r), l_name = r[12], n_cig = le16(r + 16);
            const int flag = (int)le16(r + 18);
            const int32_t tid = (int32_t)le32(r + 4), pos = (int32_t)le32(r + 8), l_seq = (int32_t)le32(r + 20);
            const std::string name((const char *)r + 36, l_name ? l_name - 1 : 0);
            auto fail = [&](const std::string &why) { std::lock_guard<std::mutex> lk(mu); bad.emplace_back(i, "read " + name + ": " + why); };
            if (l_seq < 0 || 36 + l_name + 4 * n_cig + (size_t)(l_seq + 1) / 2 + (size_t)l_seq > 4 + bs) { fail("malformed record"); return; }
            if (tid >= (int32_t)names.size()) { fail("contig id " + std::to_string(tid) + " is not in the header"); return; }
            if ((flag & (0x4 | 0x100 | 0x200 | 0x400)) || tid < 0 || n_cig == 0) continue;       // never admitted: left out
            const uint8_t *cig = r + 36 + l_name;
            int n_ops = 0;
            int64_t qlen = 0, span = 0;
            for (size_t k = 0; k < n_cig; ++k) {
                const uint32_t w = le32(cig + 4 * k), op = w & 0xf, len = w >> 4;
                if (op == 3 || op == 6) { fail(std::string("CIGAR operation ") + "MIDNSHP=X"[op] + ": N and P are not supported"); return; }
                if (op > 8) { fail("invalid CIGAR operation"); return; }
                if (op != 5) ++n_ops;
                if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) qlen += len;
                if (op == 0 || op == 2 || op == 7 || op == 8) span += len;
            }
            if (l_seq == 0) { fail("no stored SEQ ('*')"); return; }
            if (r[36 + l_name + 4 * n_cig + (size_t)(l_seq + 1) / 2] == 0xff) { fail("no stored QUAL ('*')"); return; }
            if (l_seq > 512) { fail(std::to_string(l_seq) + " bases: reads longer than 512 bases are not supported"); return; }
            if (n_ops > QM_MAX_CIGAR) { fail(std::to_string(n_ops) + " CIGAR operations: at most " + std::to_string(QM_MAX_CIGAR) + " besides H are supported"); return; }
            if (qlen != l_seq) { fail("CIGAR query length " + std::to_string(qlen) + " differs from the " + std::to_string(l_seq) + " bases of SEQ"); return; }
            if (pos < 0 || pos + span > g.lens[(size_t)tid]) { fail("alignment outside contig " + names[(size_t)tid]); return; }
            keep[i] = 1;
        }
    });
    if (!bad.empty()) {
        auto it = std::min_element(bad.begin(), bad.end(), [](const auto &x, const auto &y) { return x.first < y.first; });
        die(2, "%s: %s", fn, it->second.c_str());
    }
    BamRecords out;
    out.n_total = (int64_t)all.size();
    for (size_t i = 0; i < all.size(); ++i)
        if (keep[i]) { out.off.push_back(all[i]); out.max_len = std::max(out.max_len, (int32_t)le32(d.data() + all[i] + 20)); }
    out.n_left_out = out.n_total - (int64_t)out.off.size();
    return out;
}

// counts, calls and text pileup of an existing coordinate-sorted BAM: rules `mpileup` and `bcftools` one for one
int cmd_pileup(const Args &a)
{
    PhaseClock pc;
    require_known(a, "pileup", {"ref", "bam", "counts", "vcf", "vcf-gz", "mpileup", "max-depth", "baq", "min-mapq", "q", "min-bq", "Q",
                                "count-orphans", "ignore-overlaps", "min-dp", "min-alt", "min-af", "indels", "sample", "gpu", "t", "threads", "stage-ms"});
    if (!a.has("ref") || !a.has("bam")) die(1, "--ref and --bam are required");
    const int threads = std::max(1, atoi(a.get("t", a.get("threads", "4")).c_str()));
    g_threads = threads;
    qm_pileup_opt popt; qm_pileup_opt_default(&popt);
    apply_mpileup_options(a, popt);
    // the defaults of `sample`: no depth cap and BAQ off (the parity configuration); --max-depth caps the counts and calls only
    const int max_depth = a.has("max-depth") ? parse_int("max-depth", a.get("max-depth")) : 0;
    const int baq = a.has("baq") && parse_int("baq", a.get("baq")) ? 3 : 0;
    Genome g;
    load_refs(a.get("ref"), g);
    pc.mark("reference");
    const std::string path = a.get("bam");
    const std::vector<uint8_t> data = inflate_bgzf(path);
    pc.mark("BGZF inflate");
    const BamRecords recs = scan_bam(path, data, g);
    pc.mark("validation walk");
    fprintf(stderr, "[qm_driver] %s: %lld records, %lld left out (unmapped, secondary, QC-failed, duplicate or without CIGAR)\n", path.c_str(),
            (long long)recs.n_total, (long long)recs.n_left_out);
    Lib L;
    const int dev = atoi(a.get("gpu", "0").c_str());
    const int rc = qm_ctx_create(dev, &L.ctx);
    if (rc != QM_OK) die(3, "qm_ctx_create(%d) failed (%d): no usable B200 (there is no CPU fallback)", dev, rc);
    const bool stage_ms = atoi(a.get("stage-ms", "0").c_str()) != 0;
    if (stage_ms) L.check(qm_profile_enable(L.ctx, 1), "qm_profile_enable");
    qm_opt opt; qm_opt_default(&opt);
    std::vector<qm_index *> idxs(1, nullptr);
    std::vector<qm_sample *> smps(1, nullptr);
    L.check(qm_index_build(L.ctx, g.codes.data(), (int)g.names.size(), g.lens.data(), opt.min_seed_len, &idxs[0]), "qm_index_build");
    L.check(qm_sample_begin(L.ctx, idxs[0], &opt, &popt, &smps[0]), "qm_sample_begin");      // holds the count tensor and the indel table
    pc.mark("context + reference on the device");
    const int32_t stride = std::max<int32_t>(16, (recs.max_len + 15) & ~15);
    qm_bam_pairs bp;
    L.check(qm_bam_to_pairs_host(L.ctx, idxs[0], data.data(), (int64_t)data.size(), recs.off.data(), (int64_t)recs.off.size(), stride, &popt, baq,
                                 max_depth, &bp), "qm_bam_to_pairs_host");
    pc.mark("device decode + pairing");
    L.check(qm_pileup_accumulate_masked(L.ctx, idxs[0], &popt, bp.d_alns, bp.d_codes, bp.d_quals, bp.stride, bp.d_lens, bp.n_pairs,
                                        qm_sample_counts(smps[0]), qm_sample_indel_table(smps[0]), bp.d_drop, nullptr), "qm_pileup_accumulate_masked");
    L.check(qm_sample_stats_sync(smps[0], nullptr, nullptr, nullptr), "qm_sample_stats_sync");
    pc.mark("counting");
    fprintf(stderr, "[qm_driver] %lld records in %lld pairs (rows 2i / 2i + 1, a placeholder mate where a record has none)\n",
            (long long)recs.off.size(), (long long)bp.n_pairs);
    if (max_depth > 0) fprintf(stderr, "[qm_driver] depth cap %d: %lld reads dropped by the pileup iterator\n", max_depth, (long long)bp.n_capped);
    std::vector<Lib> Ls(1, L);
    write_outputs(a, g, Ls, idxs, smps, threads, [&]() {
        // the uncapped text pileup, reads in file order at every column as htslib's iterator delivers them
        std::vector<const char *> nm;
        for (auto &s : g.names) nm.push_back(s.c_str());
        const char *d_text = nullptr;
        int64_t bytes = 0;
        L.check(qm_mpileup_text_ranked(L.ctx, idxs[0], &popt, bp.d_alns, bp.d_codes, bp.d_quals, bp.stride, bp.d_lens, bp.n_pairs, nm.data(),
                                       bp.d_row_file, &d_text, &bytes, nullptr), "qm_mpileup_text_ranked");
        return bytes;
    });
    pc.mark("outputs");
    if (stage_ms) print_stage_ms(L, dev);
    qm_sample_destroy(smps[0]);
    qm_index_destroy(L.ctx, idxs[0]);
    qm_ctx_destroy(L.ctx);
    pc.report();
    return 0;
}

// what `rmdup`'s validation walk leaves: the header and the offset of every record in file order
struct DupInput {
    std::string text;                          // header text, trailing NULs dropped
    size_t refs_begin = 0, refs_end = 0;       // the binary reference list (n_ref and its entries) in the stream
    Genome g;                                  // contig names and lengths (no sequence): what the .bai needs
    std::vector<int64_t> off;
    int64_t n_primary = 0;                     // records without 0x100 / 0x800
    std::string library;                       // the LB of the @RG lines, empty without one
};

// {reference span (M D N = X), clipped bases (S H) before the first and after the last other operation} of a CIGAR
inline void cigar_ends(const uint8_t *cig, size_t n_cig, int64_t &span, int64_t &lead, int64_t &trail)
{
    span = lead = trail = 0;
    size_t first = n_cig, last = 0;
    for (size_t k = 0; k < n_cig; ++k) {
        const uint32_t w = le32(cig + 4 * k), op = w & 0xf;
        if (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) span += w >> 4;
        if (op != 4 && op != 5) { if (first == n_cig) first = k; last = k; }
    }
    for (size_t k = 0; k < n_cig; ++k) {
        if (k < first) lead += le32(cig + 4 * k) >> 4;
        else if (k > last) trail += le32(cig + 4 * k) >> 4;
    }
}

// The header: magic, the @SQ limits of the 30-bit end code, one library at most.  Then one walk over the records: well-formed,
// contig ids inside the header, CIGAR operations <= 8, coordinate order with the records without a contig at the end, and an
// unclipped 5' coordinate the end code holds on every placed record.  N and P operations, long reads, many CIGAR operations and a
// missing SEQ or QUAL are fine.  Every failure names the read or the limit and exits 2.
DupInput scan_bam_dup(const std::string &path, const std::vector<uint8_t> &d)
{
    const char *fn = path.c_str();
    DupInput in;
    if (d.size() < 12 || memcmp(d.data(), "BAM\1", 4) != 0) die(2, "%s: bad BAM magic: not a BAM file", fn);
    const size_t l_text = le32(d.data() + 4);
    if (8 + l_text + 4 > d.size()) die(2, "%s: truncated BAM header", fn);
    in.text.assign((const char *)d.data() + 8, l_text);
    while (!in.text.empty() && in.text.back() == '\0') in.text.pop_back();
    size_t p = 8 + l_text;
    in.refs_begin = p;
    const uint32_t n_ref = le32(d.data() + p);
    p += 4;
    for (uint32_t i = 0; i < n_ref; ++i) {
        if (p + 4 > d.size()) die(2, "%s: truncated BAM header", fn);
        const size_t ln = le32(d.data() + p);
        if (ln < 1 || p + 8 + ln > d.size()) die(2, "%s: truncated BAM header", fn);
        in.g.names.emplace_back((const char *)d.data() + p + 4, ln - 1);
        in.g.lens.push_back((int64_t)le32(d.data() + p + 4 + ln));
        p += 8 + ln;
    }
    in.refs_end = p;
    if (n_ref > QM_MAX_CONTIGS) die(2, "%s: the header lists %u contigs (@SQ): duplicate marking supports at most %d", fn, n_ref, QM_MAX_CONTIGS);
    for (size_t i = 0; i < in.g.names.size(); ++i)
        if (in.g.lens[i] >= (1 << 26) - QM_DUP_COORD_BIAS)
            die(2, "%s: @SQ %s has %lld bp: duplicate marking supports contigs under 2^26 - 4096 bases", fn, in.g.names[i].c_str(), (long long)in.g.lens[i]);
    std::vector<std::string> libs;
    for (size_t b = 0; b < in.text.size();) {
        size_t e = in.text.find('\n', b);
        if (e == std::string::npos) e = in.text.size();
        const std::string ln = in.text.substr(b, e - b);
        if (ln.compare(0, 4, "@RG\t") == 0) {
            const size_t k = ln.find("\tLB:");
            if (k != std::string::npos) {
                const std::string lb = ln.substr(k + 4, ln.find('\t', k + 4) - (k + 4));
                if (std::find(libs.begin(), libs.end(), lb) == libs.end()) libs.push_back(lb);
            }
        }
        b = e + 1;
    }
    if (libs.size() > 1) die(2, "%s: the @RG lines name %zu libraries (LB): duplicate marking of one library per file is supported", fn, libs.size());
    if (!libs.empty()) in.library = libs[0];
    // the record offsets (a serial chain of block_size fields), contig ids and the coordinate order
    auto rname = [](const uint8_t *r) { return std::string((const char *)r + 36, r[12] ? r[12] - 1 : 0); };
    int32_t last_tid = -1, last_pos = -1;
    bool no_contig_seen = false;
    for (; p < d.size();) {
        if (p + 36 > d.size()) die(2, "%s: truncated record at byte %zu of the BAM stream", fn, p);
        const uint8_t *r = d.data() + p;
        const size_t bs = le32(r);
        if (bs < 32 || p + 4 + bs > d.size() || 32 + (size_t)r[12] > bs) die(2, "%s: malformed or truncated record at byte %zu of the BAM stream", fn, p);
        const int32_t tid = (int32_t)le32(r + 4), pos = (int32_t)le32(r + 8);
        if (tid < -1 || tid >= (int32_t)n_ref) die(2, "%s: read %s: contig id %d is not in the header", fn, rname(r).c_str(), tid);
        if (tid >= 0) {
            if (no_contig_seen) die(2, "%s: the file is not coordinate-sorted: read %s on %s comes after records without a contig", fn, rname(r).c_str(), in.g.names[(size_t)tid].c_str());
            if (tid < last_tid || (tid == last_tid && pos < last_pos))
                die(2, "%s: the file is not coordinate-sorted: read %s at %s:%d comes after %s:%d", fn, rname(r).c_str(), in.g.names[(size_t)tid].c_str(), pos + 1,
                    in.g.names[(size_t)last_tid].c_str(), last_pos + 1);
            last_tid = tid; last_pos = pos;
        } else no_contig_seen = true;
        in.off.push_back((int64_t)p);
        p += 4 + bs;
    }
    // the per-record checks, on the -t threads; the first failure in file order is reported
    std::vector<std::pair<size_t, std::string>> bad;
    std::atomic<int64_t> n_primary{0};
    std::mutex mu;
    parallel_ranges(in.off.size(), [&](size_t b, size_t e) {
        int64_t np = 0;
        for (size_t i = b; i < e; ++i) {
            const uint8_t *r = d.data() + in.off[i];
            const size_t bs = le32(r), l_name = r[12], n_cig = le16(r + 16);
            const int flag = (int)le16(r + 18);
            const int32_t tid = (int32_t)le32(r + 4), pos = (int32_t)le32(r + 8), l_seq = (int32_t)le32(r + 20);
            auto fail = [&](const std::string &why) { std::lock_guard<std::mutex> lk(mu); bad.emplace_back(i, "read " + rname(r) + ": " + why); };
            if (l_name < 1 || l_seq < 0 || 36 + l_name + 4 * n_cig + (size_t)(l_seq + 1) / 2 + (size_t)l_seq > 4 + bs) { fail("malformed record"); continue; }
            const uint8_t *cig = r + 36 + l_name;
            bool ok = true;
            for (size_t k = 0; k < n_cig && ok; ++k)
                if ((le32(cig + 4 * k) & 0xf) > 8) { fail("invalid CIGAR operation " + std::to_string(le32(cig + 4 * k) & 0xf)); ok = false; }
            if (!ok) continue;
            if (!(flag & 0x900)) ++np;
            if ((flag & 0x4) || tid < 0 || n_cig == 0) continue;
            int64_t span, lead, trail;
            cigar_ends(cig, n_cig, span, lead, trail);
            const int64_t coord = (flag & 0x10) ? pos + span - 1 + trail : pos - lead;
            if (coord + QM_DUP_COORD_BIAS < 0 || coord + QM_DUP_COORD_BIAS >= (1 << 26))
                fail("unclipped 5' coordinate " + std::to_string(coord + 1) + " lies outside what the end code holds (-4095 .. 2^26 - 4096)");
        }
        n_primary += np;
    });
    if (!bad.empty()) {
        auto it = std::min_element(bad.begin(), bad.end(), [](const auto &x, const auto &y) { return x.first < y.first; });
        die(2, "%s: %s", fn, it->second.c_str());
    }
    in.n_primary = n_primary;
    return in;
}

// duplicate marking of an existing coordinate-sorted BAM: rule `rmdup` (picard MarkDuplicates REMOVE_DUPLICATES=true) one for one
int cmd_rmdup(const Args &a, const std::string &cmdline)
{
    PhaseClock pc;
    require_known(a, "rmdup", {"bam", "rmdup-bam", "metrics", "sample", "gpu", "t", "threads", "stage-ms"});
    if (!a.has("bam") || !a.has("rmdup-bam")) die(1, "--bam and --rmdup-bam are required");
    const int threads = std::max(1, atoi(a.get("t", a.get("threads", "4")).c_str()));
    g_threads = threads;
    const std::string path = a.get("bam"), out = a.get("rmdup-bam");
    const std::vector<uint8_t> data = inflate_bgzf(path);
    pc.mark("BGZF inflate");
    const DupInput in = scan_bam_dup(path, data);
    pc.mark("validation walk");
    const int64_t n = (int64_t)in.off.size();
    fprintf(stderr, "[qm_driver] %s: %lld records\n", path.c_str(), (long long)n);
    Lib L;
    const int dev = atoi(a.get("gpu", "0").c_str());
    const int rc = qm_ctx_create(dev, &L.ctx);
    if (rc != QM_OK) die(3, "qm_ctx_create(%d) failed (%d): no usable B200 (there is no CPU fallback)", dev, rc);
    const bool stage_ms = atoi(a.get("stage-ms", "0").c_str()) != 0;
    if (stage_ms) L.check(qm_profile_enable(L.ctx, 1), "qm_profile_enable");
    pc.mark("context");
    std::vector<uint8_t> dup((size_t)n);
    int64_t n_units = 0, n_dup = 0;
    L.check(qm_bam_mark_duplicates_host(L.ctx, data.data(), (int64_t)data.size(), in.off.data(), n, dup.data(), &n_units, &n_dup),
            "qm_bam_mark_duplicates_host");
    pc.mark("H2D + decision");
    int64_t n_removed = 0;
    for (uint8_t v : dup) n_removed += v;
    fprintf(stderr, "[qm_driver] rmdup: %lld of %lld units are duplicates (%lld lone records among the units); %lld records removed\n",
            (long long)n_dup, (long long)n_units, (long long)(2 * n_units - in.n_primary), (long long)n_removed);
    // the input's header plus one @PG line (an ID of its own, PP = the last @PG), then the kept records byte for byte with 0x400 cleared
    std::vector<std::string> pg_ids;
    for (size_t b = 0; b < in.text.size();) {
        size_t e = in.text.find('\n', b);
        if (e == std::string::npos) e = in.text.size();
        const std::string ln = in.text.substr(b, e - b);
        const size_t k = ln.find("\tID:");
        if (ln.compare(0, 4, "@PG\t") == 0 && k != std::string::npos) pg_ids.push_back(ln.substr(k + 4, ln.find('\t', k + 4) - (k + 4)));
        b = e + 1;
    }
    std::string id = "quasimodo_b200.rmdup";
    for (int i = 1; std::find(pg_ids.begin(), pg_ids.end(), id) != pg_ids.end(); ++i) id = "quasimodo_b200.rmdup." + std::to_string(i);
    std::string text = in.text;
    if (!text.empty() && text.back() != '\n') text += '\n';
    text += "@PG\tID:" + id + "\tPN:quasimodo_b200" + (pg_ids.empty() ? "" : "\tPP:" + pg_ids.back()) + "\tVN:0.1\tCL:" + cmdline + "\n";
    BgzfWriter bw(out, threads, 1);
    std::vector<uint8_t> hdr = {'B', 'A', 'M', 1};
    put32(hdr, (uint32_t)text.size());
    hdr.insert(hdr.end(), text.begin(), text.end());
    hdr.insert(hdr.end(), data.begin() + (ptrdiff_t)in.refs_begin, data.begin() + (ptrdiff_t)in.refs_end);
    bw.write(hdr.data(), hdr.size());
    bw.close_block();                                  // records start on a block boundary, as samtools writes them
    std::vector<BamIndexEntry> ents;
    ents.reserve((size_t)(n - n_removed));
    for (int64_t i = 0; i < n; ++i) {
        if (dup[(size_t)i]) continue;
        const uint8_t *r = data.data() + in.off[(size_t)i];
        const size_t bs = le32(r);
        const uint16_t flag = (uint16_t)(le16(r + 18) & ~0x400u);
        BamIndexEntry ie;
        ie.rid = (int32_t)le32(r + 4); ie.beg = (int32_t)le32(r + 8); ie.mapped = !(flag & 0x4);
        int64_t span = 0, lead, trail;
        if (ie.mapped) cigar_ends(r + 36 + r[12], le16(r + 16), span, lead, trail);
        ie.end = (int32_t)(ie.beg + (span > 0 ? span : 1));
        ie.bin = (uint16_t)reg2bin(ie.beg, ie.end);
        bw.reserve(bs + 4);
        bw.tell(ie.blk0, ie.off0);
        bw.write(r, 18);
        bw.write(&flag, 2);
        bw.write(r + 20, bs + 4 - 20);
        bw.tell(ie.blk1, ie.off1);
        ents.push_back(ie);
    }
    bw.finish();
    write_bai(out + ".bai", in.g, ents, bw);
    pc.mark("BAM + BAI");
    if (a.has("metrics")) write_dup_metrics(a.get("metrics"), a.get("sample", in.library.empty() ? "sample" : in.library), n_units, n_dup);
    if (stage_ms) print_stage_ms(L, dev);
    qm_ctx_destroy(L.ctx);
    pc.report();
    return 0;
}
// ------------------------------------------------------------------------------------------------
// `qm_driver index`: rule build_idx (`bwa index X.fa` + `samtools faidx X.fa`) one for one
struct FaiRow { int64_t offset = 0, line_bases = 0, line_bytes = 0; };

// the FASTA as both tools read it; every refusal exits 2 naming the contig, the line or the limit.  A line is counted in bytes with
// its terminator ("\n" or "\r\n"), as the .fai records it; within a contig every line but the last has the first line's length
// and the last is not longer (samtools faidx refuses anything else, a blank line followed by more sequence included).
void read_fasta_for_index(const std::string &path, Genome &g, std::vector<std::string> &annos, std::vector<FaiRow> &fai)
{
    std::string d;
    {
        FILE *fp = fopen(path.c_str(), "rb");
        if (!fp) die(2, "cannot open %s", path.c_str());
        char buf[1 << 16];
        size_t k;
        while ((k = fread(buf, 1, sizeof buf, fp)) > 0) d.append(buf, k);
        const bool bad = ferror(fp) != 0;
        fclose(fp);
        if (bad) die(2, "read error in %s", path.c_str());
    }
    const char *fn = path.c_str();
    if (d.size() >= 2 && (uint8_t)d[0] == 0x1f && (uint8_t)d[1] == 0x8b) die(2, "%s: compressed FASTA: index the plain file", fn);
    int8_t lut[256];
    memset(lut, -1, sizeof lut);
    lut['A'] = lut['a'] = 0; lut['C'] = lut['c'] = 1; lut['G'] = lut['g'] = 2; lut['T'] = lut['t'] = 3;
    int64_t line_no = 0, short_line = 0;              // short_line: the line of this contig that was shorter than the first (0: none)
    bool open = false;
    auto close_contig = [&]() {
        if (!open) return;
        g.lens.back() = (int64_t)g.codes.size() - g.offs.back();
        if (g.lens.back() == 0) die(2, "%s: contig %s has no bases", fn, g.names.back().c_str());
    };
    for (size_t p = 0; p < d.size();) {
        size_t e = d.find('\n', p);
        const bool terminated = e != std::string::npos;
        if (!terminated) e = d.size();
        const int64_t bytes = (int64_t)(e - p) + (terminated ? 1 : 0);
        size_t len = e - p;
        if (len && d[p + len - 1] == '\r') --len;
        ++line_no;
        const char *ln = d.data() + p;
        if (len && ln[0] == '>') {
            close_contig();
            size_t a = 1;
            while (a < len && !isspace((unsigned char)ln[a])) ++a;
            std::string name(ln + 1, a - 1), anno = a < len ? std::string(ln + a + 1, len - a - 1) : std::string();
            if (name.empty()) die(2, "%s: line %lld: a '>' line without a name", fn, (long long)line_no);
            for (auto &other : g.names) if (other == name) die(2, "%s: line %lld: contig name %s occurs twice", fn, (long long)line_no, name.c_str());
            if (g.names.size() == QM_MAX_CONTIGS) die(2, "%s: line %lld: more than %d contigs: at most %d are supported", fn, (long long)line_no, QM_MAX_CONTIGS, QM_MAX_CONTIGS);
            g.names.push_back(name);
            annos.push_back(anno);
            g.offs.push_back((int64_t)g.codes.size());
            g.lens.push_back(0);
            FaiRow r;
            r.offset = (int64_t)(e + (terminated ? 1 : 0));
            fai.push_back(r);
            open = true;
            short_line = 0;
        } else {
            if (!open) {
                if (len == 0) { p = e + 1; continue; }         // blank lines before the first header
                die(2, "%s: line %lld: sequence before the first '>' line", fn, (long long)line_no);
            }
            FaiRow &r = fai.back();
            if (len > 0) {
                if (short_line) die(2, "%s: contig %s: line %lld is shorter than the contig's first line and more sequence follows it (samtools faidx refuses different line lengths)",
                                    fn, g.names.back().c_str(), (long long)short_line);
                if (r.line_bases == 0) { r.line_bases = (int64_t)len; r.line_bytes = terminated ? bytes : (int64_t)len + 1; }
                else if ((int64_t)len > r.line_bases || (terminated && bytes - (int64_t)len != r.line_bytes - r.line_bases))
                    die(2, "%s: contig %s: line %lld has %lld bases, the contig's first line %lld (samtools faidx refuses different line lengths)",
                        fn, g.names.back().c_str(), (long long)line_no, (long long)len, (long long)r.line_bases);
                for (size_t i = 0; i < len; ++i) {
                    const int8_t v = lut[(unsigned char)ln[i]];
                    if (v < 0) die(2, "%s: line %lld: base '%c' in contig %s: only A/C/G/T references are supported (bwa index would draw a random base)",
                                   fn, (long long)line_no, ln[i], g.names.back().c_str());
                    g.codes.push_back((uint8_t)v);
                }
                if ((int64_t)len < r.line_bases) short_line = line_no;
            } else if (r.line_bases > 0 && !short_line) short_line = line_no;
        }
        if ((int64_t)g.codes.size() >= (1ll << 30))
            die(2, "%s: more than 2^30 - 1 bases: the suffix array of both strands holds at most 2^31 - 1 suffixes", fn);
        p = e + 1;
    }
    close_contig();
    if (g.names.empty()) die(2, "%s: no contigs", fn);
}

void write_file(const std::string &path, const void *data, size_t bytes)
{
    FILE *fp = fopen(path.c_str(), "wb");
    if (!fp || (bytes && fwrite(data, 1, bytes, fp) != bytes) || fclose(fp) != 0) die(2, "cannot write %s", path.c_str());
}

// .pac (bwa bntseq.c): the forward strand, base i in byte i >> 2 at shift ((~i) & 3) << 1, then one zero byte when l_pac % 4 == 0,
// then one byte holding l_pac % 4
std::vector<uint8_t> pack_pac(const std::vector<uint8_t> &codes)
{
    const int64_t l = (int64_t)codes.size();
    std::vector<uint8_t> pac((size_t)((l >> 2) + ((l & 3) ? 1 : 0)), 0);
    for (int64_t i = 0; i < l; ++i) pac[(size_t)(i >> 2)] |= (uint8_t)(codes[(size_t)i] << ((~i & 3) << 1));
    if (l % 4 == 0) pac.push_back(0);
    pac.push_back((uint8_t)(l % 4));
    return pac;
}

int cmd_index(const Args &a)
{
    PhaseClock pc;
    require_known(a, "index", {"ref", "prefix", "t", "threads", "gpu"});
    if (!a.has("ref")) die(1, "--ref is required");
    g_threads = std::max(1, atoi(a.get("t", a.get("threads", "4")).c_str()));
    const std::string fa = a.get("ref"), prefix = a.get("prefix", fa);
    if (prefix.empty()) die(1, "--prefix: empty");
    Genome g;
    std::vector<std::string> annos;
    std::vector<FaiRow> fai;
    read_fasta_for_index(fa, g, annos, fai);
    const int64_t l_pac = (int64_t)g.codes.size();
    pc.mark("FASTA");
    fprintf(stderr, "[qm_driver] %s: %zu contigs, %lld bases\n", fa.c_str(), g.names.size(), (long long)l_pac);
    Lib L;
    const int dev = atoi(a.get("gpu", "0").c_str());
    const int rc = qm_ctx_create(dev, &L.ctx);
    if (rc != QM_OK) die(3, "qm_ctx_create(%d) failed (%d): no usable B200 (there is no CPU fallback)", dev, rc);
    pc.mark("context");
    qm_index *idx = nullptr;
    L.check(qm_index_build(L.ctx, g.codes.data(), (int)g.names.size(), g.lens.data(), 31, &idx), "qm_index_build");
    pc.mark("reference on the device");
    L.check(qm_index_build_fm(L.ctx, idx, g.codes.data()), "qm_index_build_fm");
    pc.mark("suffix array + BWT");
    int64_t nb = 0, ns = 0;
    L.check(qm_index_fm_export(idx, nullptr, &nb, nullptr, &ns), "qm_index_fm_export");
    std::vector<uint8_t> bwt((size_t)nb), sa((size_t)ns);
    L.check(qm_index_fm_export(idx, bwt.data(), &nb, sa.data(), &ns), "qm_index_fm_export");
    qm_index_destroy(L.ctx, idx);
    qm_ctx_destroy(L.ctx);
    write_file(prefix + ".bwt", bwt.data(), bwt.size());
    write_file(prefix + ".sa", sa.data(), sa.size());
    const std::vector<uint8_t> pac = pack_pac(g.codes);
    write_file(prefix + ".pac", pac.data(), pac.size());
    std::string ann = std::to_string(l_pac) + " " + std::to_string(g.names.size()) + " 11\n";
    for (size_t c = 0; c < g.names.size(); ++c) {
        ann += "0 " + g.names[c] + " " + (annos[c].empty() ? std::string("(null)") : annos[c]) + "\n";
        ann += std::to_string(g.offs[c]) + " " + std::to_string(g.lens[c]) + " 0\n";
    }
    write_file(prefix + ".ann", ann.data(), ann.size());
    const std::string amb = std::to_string(l_pac) + " " + std::to_string(g.names.size()) + " 0\n";
    write_file(prefix + ".amb", amb.data(), amb.size());
    std::string fx;
    for (size_t c = 0; c < g.names.size(); ++c)
        fx += g.names[c] + "\t" + std::to_string(g.lens[c]) + "\t" + std::to_string(fai[c].offset) + "\t" + std::to_string(fai[c].line_bases) + "\t" +
              std::to_string(fai[c].line_bytes) + "\n";
    write_file(fa + ".fai", fx.data(), fx.size());
    pc.mark("files");
    pc.report();
    return 0;
}

}  // namespace

// --benchmark FILE (any command): the job's resources in the shape of a Snakemake `benchmark:` file (one header line, one row:
// s, h:m:s, max_rss, max_vms, max_uss, max_pss, io_in, io_out in MB, mean_load in percent), the format
// scripts/resource_benchmark.R reads -- the rule `bwa` this driver replaces has no `benchmark:` of its own (rules/bwa.smk:1-19),
// rules `mpileup` and `bcftools` do (rules/vcfcall.smk:32-33,108-109).  Written when the process ends, whatever its exit status.
std::string g_benchmark_path;
std::chrono::steady_clock::time_point g_benchmark_t0;
clock_t g_benchmark_cpu0;

void write_benchmark()
{
    if (g_benchmark_path.empty()) return;
    const double wall = std::chrono::duration<double>(std::chrono::steady_clock::now() - g_benchmark_t0).count();
    auto proc_kb = [](const char *file, const char *key) {           // "Key:   12345 kB" lines of /proc/self/{status,smaps_rollup}
        double v = 0;
        if (FILE *fh = fopen(file, "r")) {
            char ln[256];
            const size_t kl = strlen(key);
            while (fgets(ln, sizeof ln, fh)) if (!strncmp(ln, key, kl) && ln[kl] == ':') v += atof(ln + kl + 1);
            fclose(fh);
        }
        return v;
    };
    const double rss = proc_kb("/proc/self/status", "VmHWM") / 1024, vms = proc_kb("/proc/self/status", "VmPeak") / 1024;
    const double pss = proc_kb("/proc/self/smaps_rollup", "Pss") / 1024;
    const double uss = (proc_kb("/proc/self/smaps_rollup", "Private_Clean") + proc_kb("/proc/self/smaps_rollup", "Private_Dirty")) / 1024;
    const double io_in = proc_kb("/proc/self/io", "rchar") / (1024.0 * 1024.0), io_out = proc_kb("/proc/self/io", "wchar") / (1024.0 * 1024.0);
    const double cpu = (double)(clock() - g_benchmark_cpu0) / CLOCKS_PER_SEC;      // process CPU time since main(), every thread
    FILE *fh = fopen(g_benchmark_path.c_str(), "w");
    if (!fh) { fprintf(stderr, "qm_driver: cannot create %s\n", g_benchmark_path.c_str()); return; }
    const long ws = (long)wall;
    fprintf(fh, "s\th:m:s\tmax_rss\tmax_vms\tmax_uss\tmax_pss\tio_in\tio_out\tmean_load\n");
    fprintf(fh, "%.4f\t%ld:%02ld:%02ld\t%.2f\t%.2f\t%.2f\t%.2f\t%.2f\t%.2f\t%.2f\n", wall, ws / 3600, ws / 60 % 60, ws % 60, rss, vms, uss, pss, io_in, io_out,
            wall > 0 ? 100.0 * cpu / wall : 0.0);
    fclose(fh);
}

int main(int argc, char **argv)
{
    g_benchmark_t0 = std::chrono::steady_clock::now();
    g_benchmark_cpu0 = clock();
    if (argc < 2) die(1, "usage: qm_driver sample|decontam|pileup|rmdup|index|bam-from-records|vcf-index|fastq-check|selftest [options]   (%s)", qm_version());
    std::string cmdline;
    for (int i = 0; i < argc; ++i) { if (i) cmdline += ' '; cmdline += argv[i]; }
    const std::string cmd = argv[1];
    Args a = parse_args(argc, argv, 2);
    if (a.has("benchmark")) {
        g_benchmark_path = a.get("benchmark");
        a.kv.erase("benchmark");
        atexit(write_benchmark);
    }
    if (cmd == "sample") return cmd_sample(a, cmdline, false);
    if (cmd == "decontam") return cmd_sample(a, cmdline, true);
    if (cmd == "bam-from-records") return cmd_bam_from_records(a, cmdline);
    if (cmd == "pileup") return cmd_pileup(a);
    if (cmd == "rmdup") return cmd_rmdup(a, cmdline);
    if (cmd == "index") return cmd_index(a);
    if (cmd == "fastq-check") {                        // host only: parse the two mate files as `sample` would, report what is there
        // -K N: bwa mem's input chunks of N bases as `sample -K N` cuts them, one line "chunks: size size ..." (pairs per chunk)
        require_known(a, "fastq-check", {"r1", "r2", "t", "threads", "K", "batch-pairs"});
        if (!a.has("r1") || !a.has("r2")) die(1, "--r1 --r2 are required");
        g_threads = std::max(1, atoi(a.get("t", a.get("threads", "4")).c_str()));
        const int64_t K = parse_pair_options(a).K;
        const int64_t batch = std::max<int64_t>(1, atoll(a.get("batch-pairs", "2000000").c_str()));
        FastqPairReader fr(a.get("r1"), a.get("r2"));
        RawBatch raw;
        int64_t n_pairs = 0, bases = 0;
        size_t mx = 0;
        std::vector<int64_t> chunks, all_chunks;
        const auto t0 = std::chrono::steady_clock::now();
        while (read_batch(fr, batch, raw, K, &chunks)) {
            all_chunks.insert(all_chunks.end(), chunks.begin(), chunks.end());
            n_pairs += (int64_t)raw.size();
            bases += (int64_t)raw.a.seq.size() + (int64_t)raw.b.seq.size();
            for (const Side *sd : {&raw.a, &raw.b}) for (size_t i = 0; i < sd->n; ++i) mx = std::max(mx, sd->len(i));
        }
        const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        printf("%lld pairs, %lld bases, longest read %zu, parsed in %.2f s (%.3f M pairs/s)\n", (long long)n_pairs, (long long)bases, mx, dt,
               dt > 0 ? (double)n_pairs / dt / 1e6 : 0.0);
        if (K) {
            printf("chunks:");
            for (int64_t c : all_chunks) printf(" %lld", (long long)c);
            printf("\n");
        }
        return 0;
    }
    if (cmd == "vcf-index") {                          // bgzip -c X > X.gz; tabix -p vcf X.gz  (host only: rules/vcfcall.smk:118-119, rules/genome_diff.smk:24-25)
        require_known(a, "vcf-index", {"vcf", "out", "t"});
        if (!a.has("vcf")) die(1, "--vcf is required");
        write_vcf_gz_tbi(a.get("vcf"), a.get("out", a.get("vcf") + ".gz"), std::max(1, atoi(a.get("t", "2").c_str())));
        return 0;
    }
    if (cmd == "selftest") {                           // host-only checks of the driver's own helpers (tests/test_driver_cpu.py)
        auto rec = [](uint64_t key, int f, int r) { qm_indel x; memset(&x, 0, sizeof x); x.key = key; x.n_fwd = f; x.n_rev = r; return x; };
        const std::vector<qm_indel> A = {rec(3, 1, 0), rec(7, 2, 2), rec(9, 0, 1)}, B = {rec(1, 1, 1), rec(7, 0, 3), rec(9, 4, 0), rec(12, 1, 0)};
        const std::vector<qm_indel> M = merge_indel_tables(A, B.data(), (int64_t)B.size());
        const int64_t want[5][3] = {{1, 1, 1}, {3, 1, 0}, {7, 2, 5}, {9, 4, 1}, {12, 1, 0}};
        bool ok = M.size() == 5;
        for (size_t i = 0; ok && i < 5; ++i) ok = (int64_t)M[i].key == want[i][0] && M[i].n_fwd == want[i][1] && M[i].n_rev == want[i][2];
        ok = ok && merge_indel_tables(A, nullptr, 0).size() == 3 && merge_indel_tables({}, B.data(), 4).size() == 4 && merge_indel_tables({}, nullptr, 0).empty();
        if (!ok) die(2, "selftest: merge_indel_tables is wrong");
        // batch -> (GPU, first record among that GPU's kept records) for batches of 3, 5, 2, 7, 4 pairs
        const std::vector<int64_t> bp = {3, 5, 2, 7, 4};
        const std::vector<std::pair<int, int64_t>> w1 = {{0, 0}, {0, 6}, {0, 16}, {0, 20}, {0, 34}}, w2 = {{0, 0}, {1, 0}, {0, 6}, {1, 10}, {0, 10}},
                                                   w3 = {{0, 0}, {1, 0}, {2, 0}, {0, 6}, {1, 10}}, w8 = {{0, 0}, {1, 0}, {2, 0}, {3, 0}, {4, 0}};
        ok = batch_sources(bp, 1) == w1 && batch_sources(bp, 2) == w2 && batch_sources(bp, 3) == w3 && batch_sources(bp, 8) == w8 &&
             batch_sources({}, 2).empty();
        if (!ok) die(2, "selftest: batch_sources is wrong");
        printf("selftest ok\n");
        return 0;
    }
    die(1, "unknown command '%s'", cmd.c_str());
}
