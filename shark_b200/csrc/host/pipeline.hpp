// Host pipeline stages of shark-b200 around the device calls (SURVEY.md 8f.1/8f.2):
//
//   RecordSource x {1,2}  ->  Batcher  ->  [shk_reads_submit_packed / shk_reads_collect]  ->  Writer
//   (fastpipe.hpp: parallel    (a thread +    (the caller's thread)                            (a thread +
//    scan of mapped files)      the pool)                                                       the pool)
//
// Batcher = FastqSplitter::operator() called until it returns an empty batch (main.cpp:66-77,
// FastqSplitter.hpp:47-93).  Every chunk leaves the batcher in the PACKED form of shk_reads_submit_packed
// (2-bit code + validity bit per base, the -q masking rule of FastqSplitter.hpp:104-109 folded in): the
// device never sees text or qualities.  Two ways to build a chunk:
//   bulk   runs of plain records (status >= 0, no NUL bytes - all of a well-formed FASTQ file): offsets by a
//          parallel prefix sum over the record lengths, then the pool packs 64 KiB pieces of the chunk's
//          joined text (mate1 [+ 'N' + mate2]) straight from the mapped input; no text staging, the writer
//          later takes names, sequences and qualities from the records themselves;
//   exact  outcome by outcome, with the reference's behaviour at failed reads, NUL bytes (C-string
//          semantics of FastqSplitter.hpp:56) and the end of the input; builds the text in a staging buffer
//          and packs that.  A bulk chunk ends where the next outcome needs this path.
// Batches: ReadOutput's consecutive-name dedup resets per 50 000-read batch (ReadOutput.hpp:41); a batch may
// span chunks (chunks are bounded by reads AND by bytes), so the batcher marks the batch starts inside every
// chunk and the writer carries the last kept name across chunks.
// Writer = ReadOutput::operator() (ReadOutput.hpp:37-50): formats ranges of a chunk's reads in parallel from
// the compact results (one 16-bit word per read + a list for ties), writes with pwrite at precomputed
// offsets when the descriptor is seekable, in order otherwise.
#pragma once
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/vfs.h>
#include <unistd.h>

#include <algorithm>
#include <cerrno>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

#include "fastpipe.hpp"

namespace shkhost {

// SHK_TIMING: seconds spent per host stage (diagnostics; printed by the CLI at exit)
struct StageTimes {
    double scan_wait = 0, flatten = 0, offsets = 0, pack = 0, exact = 0, format = 0, output = 0;
};
inline StageTimes &stage_times()
{
    static StageTimes t;
    return t;
}
inline double stage_now()
{
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

constexpr unsigned kBatch = 50000;  // FastqSplitter batch (main.cpp:215): ReadOutput's dedup resets per batch
constexpr uint32_t kGeneNone = 0xFFFFu, kGeneMulti = 0xFFFEu;  // SHK_GENE_NONE / SHK_GENE_MULTI

struct AssocPair {  // layout of shk_assoc
    uint32_t read_idx, gene_idx;
};

// shk_host_pack(seq, qual, min_quality, n, codes, valid, parallel = 0): the library's packer, or a restatement
// where the library is not linked (host_tools)
using PackFn = void (*)(const uint8_t *seq, const uint8_t *qual, int32_t min_quality, uint64_t n, uint64_t *codes,
                        uint32_t *valid);

template <class Alloc>
struct Staging {
    uint8_t *p = nullptr;
    size_t cap = 0;
    bool external = false;  // the bytes belong to someone else (a slot of the memory shared with the device process)
    void use(void *mem, size_t bytes)
    {
        if (p && !external) Alloc::free(p);
        p = (uint8_t *)mem;
        cap = bytes;
        external = true;
    }
    void reserve(size_t n, size_t keep_bytes)
    {
        if (n <= cap) return;
        if (external) {  // sized for the largest chunk by whoever provided it
            fprintf(stderr, "shark: internal error: a chunk outgrew its shared buffer (%zu > %zu bytes)\n", n, cap);
            abort();
        }
        size_t want = cap ? cap : (1u << 20);
        while (want < n) want *= 2;
        uint8_t *q = (uint8_t *)Alloc::alloc(want);
        if (p) {
            if (keep_bytes) memcpy(q, p, keep_bytes);
            Alloc::free(p);
        }
        p = q;
        cap = want;
    }
    ~Staging()
    {
        if (p && !external) Alloc::free(p);
    }
};

// What ReadOutput needs for one read of an exact-path chunk besides the sequence text (which is in Chunk::seq).
struct ReadMeta {
    const char *name1 = nullptr, *qual1 = nullptr, *name2 = nullptr, *qual2 = nullptr;
    uint32_t nlen1 = 0, qlen1 = 0, nlen2 = 0, qlen2 = 0;
    uint32_t len1 = 0;  // length of mate 1 in the joined text (mate 2 = total - len1 - 1)
};

template <class Alloc>
struct Chunk {
    // what the device gets (both kinds of chunk)
    Staging<Alloc> off, codes, valid;   // uint32 offsets [n + 1], uint64 code words, uint32 validity words
    // bulk chunks: the records themselves
    bool bulk = false;
    std::vector<const Rec *> r1, r2;
    // exact chunks: joined text, qualities for the packer, per-read output fields
    Staging<Alloc> seq, qual;
    std::vector<ReadMeta> meta;
    std::vector<uint32_t> batch_start;  // read indices where a 50 000-read batch begins
    std::vector<std::shared_ptr<Block>> keep;
    // results in the compact form: views (into the memory shared with the device process, or into the vectors
    // below), valid until the chunk is recycled
    const uint16_t *gene16 = nullptr;
    const AssocPair *multi = nullptr;
    size_t n_multi = 0;
    const uint32_t *scores = nullptr;  // with a scores output: per read {len, cov, hits, n_best} (shk_read_score)
    std::vector<uint16_t> gene16_v;
    std::vector<AssocPair> multi_v;
    std::vector<uint32_t> scores_v;
    void results_from_vectors()
    {
        gene16 = gene16_v.data();
        multi = multi_v.data();
        n_multi = multi_v.size();
        scores = scores_v.empty() ? nullptr : scores_v.data();
    }
    int slot = -1;  // shared slot this chunk's buffers live in (two-process CLI)
    uint32_t n = 0;
    uint64_t bytes = 0;
    bool last = false;
    uint64_t index = 0;
    void clear()
    {
        r1.clear();
        r2.clear();
        meta.clear();
        batch_start.clear();
        keep.clear();
        gene16_v.clear();
        multi_v.clear();
        scores_v.clear();
        gene16 = nullptr, multi = nullptr, n_multi = 0, scores = nullptr;
        bulk = false;
        n = 0;
        bytes = 0;
        last = false;
    }
    const uint32_t *offsets() const { return (const uint32_t *)off.p; }
    uint64_t groups() const { return (bytes + 31) / 32; }
};

template <class Alloc>
class Batcher {
public:
    Batcher(const char *path1, const char *path2, int32_t min_quality, PackFn pack)
        : s1_(path1), min_quality_(min_quality), with_qual_((min_quality & 0xFF) != 0), pack_(pack)
    {
        if (path2) s2_.reset(new RecordSource(path2));
    }
    bool files_ok() const { return s1_.ok() && (!s2_ || s2_->ok()); }
    void start()
    {
        s1_.start();
        if (s2_) s2_->start();
    }

    // Fills one chunk (at most max_reads reads and max_bytes bytes of joined text); returns false when the
    // input is exhausted (the chunk may still hold reads).
    bool fill(Chunk<Alloc> &ch, unsigned max_reads, uint64_t max_bytes)
    {
        ch.clear();
        if (finished_) return false;
        static const bool no_bulk = getenv("SHK_NO_BULK") && atoi(getenv("SHK_NO_BULK")) != 0;
        const double t0 = stage_now();
        size_t n = no_bulk ? 0 : s1_.clean_run(max_reads);
        if (s2_ && n) n = std::min(n, s2_->clean_run(n));
        stage_times().scan_wait += stage_now() - t0;
        if (n) {
            fill_bulk(ch, n, max_bytes);
            if (ch.n) return true;  // (a first read longer than max_bytes: the exact path reports it)
        }
        const double t1 = stage_now();
        const bool more = fill_exact(ch, max_reads, max_bytes);
        stage_times().exact += stage_now() - t1;
        return more;
    }
    const char *error() const { return error_.empty() ? nullptr : error_.c_str(); }

private:
    // ---- bulk ----------------------------------------------------------------------------------------------
    void fill_bulk(Chunk<Alloc> &ch, size_t n, uint64_t max_bytes)
    {
        const bool paired = (bool)s2_;
        // the records, without consuming them yet: the byte bound may cut the chunk short
        const double t_a = stage_now();
        std::vector<Span> sp1, sp2;
        std::vector<std::shared_ptr<Block>> keep1, keep2;
        peek_spans(s1_, n, sp1, keep1);
        if (paired) peek_spans(*s2_, n, sp2, keep2);
        ch.r1.resize(n);
        if (paired) ch.r2.resize(n);
        flatten(sp1, ch.r1);
        if (paired) flatten(sp2, ch.r2);
        const double t_b = stage_now();
        stage_times().flatten += t_b - t_a;
        // offsets: per-range byte sums, their prefix, then the fill - all ranges in parallel
        ch.off.reserve((n + 2) * 4, 0);
        uint32_t *off = (uint32_t *)ch.off.p;
        const size_t n_ranges = std::min<size_t>(64, (n + 4095) / 4096);
        const size_t per = (n + n_ranges - 1) / n_ranges;
        std::vector<uint64_t> sum(n_ranges + 1, 0);
        auto len_of = [&](size_t i) -> uint64_t {
            return paired ? (uint64_t)ch.r1[i]->seq_len + 1 + ch.r2[i]->seq_len : ch.r1[i]->seq_len;
        };
        WorkPool::instance().run(n_ranges, [&](size_t t) {
            uint64_t s = 0;
            for (size_t i = t * per, e = std::min(n, i + per); i < e; ++i) s += len_of(i);
            sum[t + 1] = s;
        });
        for (size_t t = 0; t < n_ranges; ++t) sum[t + 1] += sum[t];
        // byte bound: the longest prefix of reads whose text fits (ranges first, then inside the range)
        size_t n_fit = n;
        if (sum[n_ranges] > max_bytes) {
            size_t t = 0;
            while (sum[t + 1] <= max_bytes) ++t;
            uint64_t s = sum[t];
            size_t i = t * per;
            for (; i < n && s + len_of(i) <= max_bytes; ++i) s += len_of(i);
            n_fit = i;
        }
        if (n_fit == 0) {
            ch.clear();
            return;
        }
        WorkPool::instance().run(n_ranges, [&](size_t t) {
            uint64_t s = sum[t];
            for (size_t i = t * per, e = std::min(n_fit, i + per); i < e; ++i) {
                off[i] = (uint32_t)s;
                s += len_of(i);
            }
        });
        uint64_t total = 0;
        {
            const size_t t = (n_fit - 1) / per;
            total = sum[t];
            for (size_t i = t * per; i < n_fit; ++i) total += len_of(i);
        }
        off[n_fit] = (uint32_t)total;
        n = n_fit;
        ch.r1.resize(n);
        if (paired) ch.r2.resize(n);
        // consume what the chunk holds
        {
            std::vector<Span> dummy;
            s1_.take(n, dummy, ch.keep);
            if (paired) {
                dummy.clear();
                s2_->take(n, dummy, ch.keep);
            }
        }
        ch.bulk = true;
        ch.n = (uint32_t)n;
        ch.bytes = total;
        for (size_t i = (kBatch - batch_got_) % kBatch; i < n; i += kBatch) ch.batch_start.push_back((uint32_t)i);
        batch_got_ = (unsigned)((batch_got_ + n) % kBatch);
        const double t_c = stage_now();
        stage_times().offsets += t_c - t_b;
        pack_bulk(ch);
        stage_times().pack += stage_now() - t_c;
    }
    static void peek_spans(RecordSource &s, size_t n, std::vector<Span> &spans, std::vector<std::shared_ptr<Block>> &keep)
    {
        s.peek_run(n, spans, keep);
    }
    static void flatten(const std::vector<Span> &spans, std::vector<const Rec *> &out)
    {
        // ranges of the flat array in parallel; a span is found by binary search over the span starts
        std::vector<size_t> start(spans.size() + 1, 0);
        for (size_t i = 0; i < spans.size(); ++i) start[i + 1] = start[i] + spans[i].n;
        const size_t n = out.size();
        const size_t n_ranges = std::min<size_t>(64, (n + 8191) / 8192);
        const size_t per = (n + n_ranges - 1) / n_ranges;
        WorkPool::instance().run(n_ranges, [&](size_t t) {
            size_t i = t * per;
            const size_t e = std::min(n, i + per);
            size_t sp = (size_t)(std::upper_bound(start.begin(), start.end(), i) - start.begin()) - 1;
            while (i < e) {
                const size_t in_span = i - start[sp], m = std::min(e - i, spans[sp].n - in_span);
                const Rec *r = spans[sp].recs + in_span;
                for (size_t j = 0; j < m; ++j) out[i + j] = r + j;
                i += m;
                ++sp;
            }
        });
    }
    // Bytes [a, b) of the joined text / quality string of a bulk chunk, gathered from the records.
    void gather(const Chunk<Alloc> &ch, uint64_t a, uint64_t b, uint8_t *seq, uint8_t *qual) const
    {
        const bool paired = (bool)s2_;
        const uint32_t *off = ch.offsets();
        size_t i = (size_t)(std::upper_bound(off, off + ch.n + 1, (uint32_t)a) - off) - 1;
        uint64_t pos = a;
        while (pos < b) {
            const Rec &x = *ch.r1[i];
            const uint64_t r0 = off[i], r_end = off[i + 1];
            const uint64_t lo = pos - r0, hi = std::min(b, r_end) - r0;  // range inside this read's text
            auto piece = [&](const char *src, uint64_t at, uint64_t len, uint8_t *dst_base) {  // src covers [at, at + len)
                const uint64_t s = std::max(lo, at), e = std::min(hi, at + len);
                if (s < e) memcpy(dst_base + (r0 + s - a), src + (s - at), e - s);
            };
            piece(x.seq, 0, x.seq_len, seq);
            if (paired) {
                const Rec &y = *ch.r2[i];
                if (lo <= x.seq_len && x.seq_len < hi) seq[r0 + x.seq_len - a] = 'N';  // FastqSplitter.hpp:63,83
                piece(y.seq, (uint64_t)x.seq_len + 1, y.seq_len, seq);
            }
            if (qual) {
                // string(qual1) [+ "\33" + string(qual2)] (FastqSplitter.hpp:84); mask_seq walks the QUAL string
                // (FastqSplitter.hpp:104-108): positions it does not reach are never masked -> 0x7f
                const uint64_t total = r_end - r0;
                memset(qual + (r0 + lo - a), 0x7f, hi - lo);
                const uint64_t c1 = std::min<uint64_t>(x.qual_len, total);
                piece(x.qual, 0, c1, qual);
                if (paired) {
                    const Rec &y = *ch.r2[i];
                    uint64_t w = c1;
                    if (w < total) {
                        if (lo <= w && w < hi) qual[r0 + w - a] = 0x1B;
                        ++w;
                    }
                    piece(y.qual, w, std::min<uint64_t>(y.qual_len, total - w), qual);
                }
            }
            pos = r0 + hi;
            ++i;
        }
    }
    void pack_bulk(Chunk<Alloc> &ch)
    {
        const uint64_t groups = ch.groups();
        ch.codes.reserve(groups * 8 + 64, 0);
        ch.valid.reserve(groups * 4 + 64, 0);
        constexpr uint64_t kPiece = 64u << 10;  // bytes of text per task (a multiple of 32)
        const size_t n_pieces = (size_t)((ch.bytes + kPiece - 1) / kPiece);
        WorkPool::instance().run(n_pieces, [&](size_t t) {
            thread_local std::vector<uint8_t> stage_seq, stage_qual;
            const uint64_t a = (uint64_t)t * kPiece, b = std::min(ch.bytes, a + kPiece);
            stage_seq.resize(kPiece + 64);
            if (with_qual_) stage_qual.resize(kPiece + 64);
            gather(ch, a, b, stage_seq.data(), with_qual_ ? stage_qual.data() : nullptr);
            pack_(stage_seq.data(), with_qual_ ? stage_qual.data() : nullptr, min_quality_, b - a,
                  (uint64_t *)ch.codes.p + a / 32, (uint32_t *)ch.valid.p + a / 32);
        });
    }

    // ---- exact -----------------------------------------------------------------------------------------------
    // One batch at most (the bulk path takes over again at the next batch start if the stream is plain there).
    bool fill_exact(Chunk<Alloc> &ch, unsigned max_reads, uint64_t max_bytes)
    {
        max_reads_ = max_reads;
        max_bytes_ = max_bytes;
        if (batch_got_ == 0) ch.batch_start.push_back(0);
        bool more = true;
        while (ch.n < max_reads) {
            const Rec a = s1_.peek();
            if (a.status < 0) {
                s1_.consume();
                if (!end_batch()) more = false;
                break;
            }
            const std::shared_ptr<Block> ba = s1_.block();
            Rec b;
            std::shared_ptr<Block> bb;
            if (s2_) {
                b = s2_->peek();
                if (b.status < 0) {  // mate 1 is dropped (FastqSplitter.hpp:61)
                    s1_.consume();
                    s2_->consume();
                    if (!end_batch()) more = false;
                    break;
                }
                bb = s2_->block();
            }
            const uint32_t l1 = clen(a.seq, a.seq_len, ba->has_nul), l2 = s2_ ? clen(b.seq, b.seq_len, bb->has_nul) : 0;
            const uint64_t total = s2_ ? (uint64_t)l1 + 1 + l2 : l1;
            if (total > max_bytes) {
                error_ = "a read of " + std::to_string(total) + " bytes exceeds the chunk capacity of " + std::to_string(max_bytes) +
                         " bytes (--chunk-reads sizes it)";
                finished_ = true;
                return false;
            }
            if (ch.bytes + total > max_bytes) break;  // chunk full: the batch goes on in the next chunk
            hold(ch, ba);
            if (s2_) hold(ch, bb);
            s1_.consume();
            if (s2_) s2_->consume();
            append(ch, a, ba->has_nul, b, s2_ ? bb->has_nul : false);
            if (++batch_got_ == kBatch) {
                batch_got_ = 0;
                break;  // a batch start: the bulk path may take over
            }
        }
        if (!more) finished_ = true;
        if (ch.n) {
            const uint64_t groups = ch.groups();
            ch.codes.reserve(groups * 8 + 64, 0);
            ch.valid.reserve(groups * 4 + 64, 0);
            pack_(ch.seq.p, with_qual_ ? ch.qual.p : nullptr, min_quality_, ch.bytes, (uint64_t *)ch.codes.p, (uint32_t *)ch.valid.p);
        }
        return more;
    }
    // A failed read ends the current batch (FastqSplitter.hpp:53,61); a batch that ends empty ends the input
    // (the reference's worker returns, main.cpp:70).
    bool end_batch()
    {
        if (batch_got_ == 0) return false;
        batch_got_ = 0;
        return true;
    }
    static void hold(Chunk<Alloc> &ch, const std::shared_ptr<Block> &b)
    {
        // blocks arrive in order per stream: at most the last two entries can be this block
        const size_t k = ch.keep.size();
        if (k >= 1 && ch.keep[k - 1] == b) return;
        if (k >= 2 && ch.keep[k - 2] == b) return;
        ch.keep.push_back(b);
    }
    // C-string semantics of the reference (FastqSplitter.hpp:56: `seq1->seq.s` as const char*)
    static uint32_t clen(const char *s, uint32_t n, bool may_have_nul)
    {
        if (!may_have_nul) return n;
        const void *z = memchr(s, 0, n);
        return z ? (uint32_t)((const char *)z - s) : n;
    }
    void append(Chunk<Alloc> &ch, const Rec &a, bool nul_a, const Rec &b, bool nul_b)
    {
        const bool paired = (bool)s2_;
        const uint32_t l1 = clen(a.seq, a.seq_len, nul_a), l2 = paired ? clen(b.seq, b.seq_len, nul_b) : 0;
        const size_t total = paired ? (size_t)l1 + 1 + l2 : l1;
        if (ch.n == 0) {
            ch.off.reserve(((size_t)std::min<unsigned>(max_reads_, kBatch) + 2) * 4, 0);
            ((uint32_t *)ch.off.p)[0] = 0;
        }
        ch.off.reserve(((size_t)ch.n + 2) * 4, ((size_t)ch.n + 1) * 4);
        uint32_t *off = (uint32_t *)ch.off.p;
        ch.seq.reserve(ch.bytes + total + 64, ch.bytes);
        uint8_t *d = ch.seq.p + ch.bytes;
        memcpy(d, a.seq, l1);
        if (paired) {
            d[l1] = 'N';  // FastqSplitter.hpp:63,83
            memcpy(d + l1 + 1, b.seq, l2);
        }
        // qualities: mask_seq walks the QUAL string (FastqSplitter.hpp:104-108); positions it does
        // not reach are never masked -> pad with 0x7f, which is not < any mq
        const uint32_t ql1 = clen(a.qual, a.qual_len, nul_a), ql2 = paired ? clen(b.qual, b.qual_len, nul_b) : 0;
        if (with_qual_) {
            ch.qual.reserve(ch.bytes + total + 64, ch.bytes);
            uint8_t *q = ch.qual.p + ch.bytes;
            if (!paired) {
                const size_t c1 = ql1 < total ? ql1 : total;
                memcpy(q, a.qual, c1);
                if (c1 < total) memset(q + c1, 0x7f, total - c1);
            } else {
                // string(qual1) + "\33" + string(qual2), FastqSplitter.hpp:84
                size_t w = 0;
                const size_t c1 = ql1 < total ? ql1 : total;
                memcpy(q, a.qual, c1);
                w = c1;
                if (w < total) q[w++] = 0x1B;
                const size_t c2 = ql2 < total - w ? ql2 : total - w;
                memcpy(q + w, b.qual, c2);
                w += c2;
                if (w < total) memset(q + w, 0x7f, total - w);
            }
        }
        ReadMeta m;
        m.name1 = a.name;
        m.nlen1 = clen(a.name, a.name_len, nul_a);
        m.qual1 = a.qual;
        m.qlen1 = ql1;
        if (paired) {
            m.name2 = b.name;
            m.nlen2 = clen(b.name, b.name_len, nul_b);
            m.qual2 = b.qual;
            m.qlen2 = ql2;
        }
        m.len1 = l1;
        ch.meta.push_back(m);
        ch.bytes += total;
        ++ch.n;
        off[ch.n] = (uint32_t)ch.bytes;
    }

    RecordSource s1_;
    std::unique_ptr<RecordSource> s2_;
    int32_t min_quality_;
    bool with_qual_;
    PackFn pack_;
    unsigned max_reads_ = 0;
    uint64_t max_bytes_ = 0;
    unsigned batch_got_ = 0;  // reads of the running batch so far
    bool finished_ = false;
    std::string error_;
};

// Buffered writer over a file descriptor.
class OutBuf {
public:
    explicit OutBuf(int fd, size_t cap = 8u << 20) : fd_(fd), buf_(new char[cap]), cap_(cap) {}
    ~OutBuf() { flush(); }
    void put(const void *p, size_t n)
    {
        if (n > cap_ - len_) {
            flush();
            if (n >= cap_) {
                raw(p, n);
                return;
            }
        }
        memcpy(buf_.get() + len_, p, n);
        len_ += n;
    }
    void putc(char c)
    {
        if (len_ == cap_) flush();
        buf_[len_++] = c;
    }
    void flush()
    {
        if (len_) raw(buf_.get(), len_);
        len_ = 0;
    }
    int fd() const { return fd_; }

private:
    void raw(const void *p, size_t n)
    {
        const char *c = (const char *)p;
        while (fd_ >= 0 && n) {
            const ssize_t w = ::write(fd_, c, n);
            if (w <= 0) {
                if (w < 0 && errno == EINTR) continue;
                return;  // like the reference, output errors are not reported
            }
            c += w;
            n -= (size_t)w;
        }
    }
    int fd_;
    std::unique_ptr<char[]> buf_;
    size_t cap_, len_ = 0;
};

// ReadOutput::operator() (ReadOutput.hpp:37-50) for one chunk's results in the compact form.  An optional fourth
// output (fd_scores >= 0, the chunks carry score records) gets one line per reported read, in the order of the ssv:
// `<name> <len> <cov> <hits> <n_best>`, name = the ssv's first field (shk_read_score, include/shark_b200.h).
template <class Alloc>
class Writer {
public:
    static constexpr int kOuts = 4;  // ssv, FASTQ 1, FASTQ 2, scores
    Writer(int fd_ssv, int fd_out1, int fd_out2, const std::vector<std::string> &legend, bool paired, int fd_scores = -1)
        : legend_(legend), paired_(paired), ssv_(fd_ssv), out1_(fd_out1), out2_(fd_out2), scores_(fd_scores), has1_(fd_out1 >= 0),
          has2_(fd_out2 >= 0 && paired), has3_(fd_scores >= 0)
    {
        for (const std::string &g : legend_) legend_len_.push_back((uint32_t)strlen(g.c_str()));
        // Files on tmpfs are written through shared mappings: the threads of the pool fault pages in
        // concurrently (7 GB/s on the B200 host), while write / pwrite to one file serialise on its inode lock
        // (4-5 GB/s).  On disk-backed file systems write(2) into the page cache is the faster way (6.7 vs
        // 3-4 GB/s there; profiles/iobench_r2.txt), so everything else is formatted into a private buffer and
        // written in order.  SHK_OUT=map / write forces either.
        const char *mode = getenv("SHK_OUT");
        const int fds[kOuts] = {fd_ssv, has1_ ? fd_out1 : -1, has2_ ? fd_out2 : -1, fd_scores};
        for (int f = 0; f < kOuts; ++f) {
            struct stat st;
            struct statfs sf;
            const bool can = fds[f] >= 0 && fstat(fds[f], &st) == 0 && S_ISREG(st.st_mode) && lseek(fds[f], 0, SEEK_CUR) >= 0 &&
                             (fcntl(fds[f], F_GETFL) & O_ACCMODE) == O_RDWR;
            const bool tmpfs = can && fstatfs(fds[f], &sf) == 0 && (unsigned long)sf.f_type == 0x01021994ul;  // TMPFS_MAGIC
            mappable_[f] = can && (mode ? !strcmp(mode, "map") : tmpfs);
        }
        populate_ = getenv("SHK_OUT_POPULATE") && atoi(getenv("SHK_OUT_POPULATE")) != 0;
    }
    ~Writer()
    {
        stop_prefault();
        stop_async();
    }
    // Pre-faulting.  Writing a fresh file on tmpfs costs a page allocation per 4 KiB, at most ~7 GB/s on the B200
    // host however many threads fault - the writer's whole budget.  The device needs a second or so to come up,
    // during which nothing can be written yet: `expect[f]` > 0 (an upper bound of output f's size - the filtered
    // FASTQ is never longer than its input) makes a few threads allocate that many bytes of the file ahead of the
    // writer, so that the writer's own stores find the pages in place.  A touch is an atomic `or 0` on one byte
    // per page: it allocates the page and can never change what the writer has already stored there.  The file is
    // cut to its real length at the end (flush()).  Only for mapped outputs, and only if the file system has
    // room for twice the bound.
    void start_prefault(const uint64_t expect[3], int n_threads)  // (ssv and FASTQ outputs)
    {
        OutBuf *outs[3] = {&ssv_, &out1_, &out2_};
        for (int f = 0; f < 3; ++f) {
            if (!expect[f] || !mappable_[f] || n_threads < 1) continue;
            struct statfs sf;
            if (fstatfs(outs[f]->fd(), &sf) != 0 || (uint64_t)sf.f_bavail * (uint64_t)sf.f_bsize < 2 * expect[f]) continue;
            char *p = window(f, (size_t)expect[f]);  // grows the file and maps [pos, pos + expect)
            if (!p) continue;
            pre_[f].base = p;
            pre_[f].len = expect[f];
            for (int t = 0; t < n_threads; ++t)
                pre_threads_.emplace_back([this, f] {
                    constexpr uint64_t kStep = 4u << 20;
                    const long page = sysconf(_SC_PAGESIZE);
                    for (;;) {
                        const uint64_t a = pre_[f].cursor.fetch_add(kStep);
                        if (a >= pre_[f].len || pre_stop_.load()) return;
                        const uint64_t b = std::min(pre_[f].len, a + kStep);
                        if ((off_t)b <= win_[f].pos - win_[f].start0) continue;  // the writer is past this piece already
                        for (uint64_t o = a; o < b; o += (uint64_t)page)
                            __atomic_fetch_or((unsigned char *)pre_[f].base + o, 0, __ATOMIC_RELAXED);
                    }
                });
        }
    }
    void stop_prefault()
    {
        pre_stop_.store(true);
        for (auto &t : pre_threads_) t.join();
        pre_threads_.clear();
    }
    void flush()
    {
        stop_prefault();
        stop_async();
        OutBuf *outs[kOuts] = {&ssv_, &out1_, &out2_, &scores_};
        for (int f = 0; f < kOuts; ++f) {
            outs[f]->flush();
            if (win_[f].base) {  // the file was grown ahead of the data: cut it to what was written
                if (ftruncate(outs[f]->fd(), win_[f].pos) != 0) {
                }
                lseek(outs[f]->fd(), win_[f].pos, SEEK_SET);
                // the windows themselves are left to the end of the process (unmapping gigabytes of dirty pages
                // costs tens of milliseconds that nobody needs to wait for)
            }
        }
    }
    void write(const Chunk<Alloc> &ch)
    {
        if (ch.n == 0) return;
        // ranges of reads; pass 1 sizes every range's share of the three outputs, pass 2 formats it in place:
        // straight into a shared mapping of the grown file when the descriptor is a regular file (page faults of
        // different threads proceed in parallel, whereas write / pwrite to one file serialise on the inode
        // lock), else into a private buffer that is then written in order
        const size_t n_ranges = std::min<size_t>((size_t)WorkPool::instance().size() * 4, ((size_t)ch.n + 8191) / 8192);
        const size_t per = ((size_t)ch.n + n_ranges - 1) / n_ranges;
        const double t_f = stage_now();
        std::vector<size_t> at[kOuts];
        for (auto &v : at) v.assign(n_ranges + 1, 0);
        WorkPool::instance().run(n_ranges, [&](size_t t) {
            const uint32_t a = (uint32_t)(t * per), b = (uint32_t)std::min<size_t>(ch.n, (t + 1) * per);
            CountSink c[kOuts];
            format(ch, a, b, c[0], c[1], c[2], c[3]);
            for (int f = 0; f < kOuts; ++f) at[f][t + 1] = c[f].n;
        });
        for (auto &v : at)
            for (size_t t = 0; t < n_ranges; ++t) v[t + 1] += v[t];
        OutBuf *outs[kOuts] = {&ssv_, &out1_, &out2_, &scores_};
        char *dst[kOuts] = {nullptr, nullptr, nullptr, nullptr};  // where byte 0 of this chunk's share of output f goes
        bool mapped[kOuts] = {false, false, false, false};
        for (int f = 0; f < kOuts; ++f) {
            const size_t total = at[f][n_ranges];
            if (!total || (f == 1 && !has1_) || (f == 2 && !has2_) || (f == 3 && !has3_)) continue;
            if (mappable_[f] && (total >= (1u << 16) || win_[f].base)) dst[f] = window(f, total);
            mapped[f] = dst[f] != nullptr;
            if (!dst[f]) {
                // private buffer, written out in order - by the background thread when the descriptor is never mapped
                // (a pipe, a file opened write-only by the shell: the ssv on stdout), so that write(2) of this chunk
                // overlaps the formatting of the next; two buffers per output take turns
                std::vector<char> &buf = priv_[f][priv_turn_[f]];
                wait_async(priv_job_[f][priv_turn_[f]]);
                if (buf.size() < total) buf.resize(total);
                dst[f] = buf.data();
            }
        }
        WorkPool::instance().run(n_ranges, [&](size_t t) {
            const uint32_t a = (uint32_t)(t * per), b = (uint32_t)std::min<size_t>(ch.n, (t + 1) * per);
            WriteSink w[kOuts];
            for (int f = 0; f < kOuts; ++f) w[f].p = dst[f] ? dst[f] + at[f][t] : nullptr;
#ifdef MADV_POPULATE_WRITE
            if (populate_)  // allocate this range's pages of the file in one call instead of one fault per page
                for (int f = 0; f < kOuts; ++f)
                    if (mapped[f] && at[f][t + 1] > at[f][t]) {
                        const uintptr_t pg = (uintptr_t)sysconf(_SC_PAGESIZE);
                        const uintptr_t lo = (uintptr_t)(dst[f] + at[f][t]) / pg * pg, hi = (uintptr_t)(dst[f] + at[f][t + 1]);
                        madvise((void *)lo, hi - lo, MADV_POPULATE_WRITE);
                    }
#endif
            format(ch, a, b, w[0], w[1], w[2], w[3]);
        });
        const double t_o = stage_now();
        stage_times().format += t_o - t_f;
        for (int f = 0; f < kOuts; ++f) {
            const size_t total = at[f][n_ranges];
            if (!dst[f] || !total) continue;
            if (mapped[f]) {
                win_[f].pos += (off_t)total;
            } else if (!mappable_[f]) {
                priv_job_[f][priv_turn_[f]] = submit_async(outs[f], dst[f], total);
                priv_turn_[f] ^= 1;
            } else {
                outs[f]->put(dst[f], total);
            }
        }
        stage_times().output += stage_now() - t_o;
        // the name ReadOutput's `previd` holds at the end of this chunk, for the first read of the next one
        update_carry(ch);
    }

private:
    struct CountSink {
        size_t n = 0;
        void put(const void *, size_t len) { n += len; }
        void putc(char) { ++n; }
    };
    struct WriteSink {
        char *p = nullptr;
        void put(const void *src, size_t len)
        {
            memcpy(p, src, len);
            p += len;
        }
        void putc(char c) { *p++ = c; }
    };
    struct Fields {
        const char *name1, *seq1, *qual1, *name2, *seq2, *qual2;
        uint32_t nlen1, slen1, qlen1, nlen2, slen2, qlen2;
    };
    static Fields fields(const Chunk<Alloc> &ch, uint32_t r, bool paired)
    {
        Fields f{};
        if (ch.bulk) {
            const Rec &x = *ch.r1[r];
            f.name1 = x.name, f.nlen1 = x.name_len, f.seq1 = x.seq, f.slen1 = x.seq_len, f.qual1 = x.qual, f.qlen1 = x.qual_len;
            if (paired) {
                const Rec &y = *ch.r2[r];
                f.name2 = y.name, f.nlen2 = y.name_len, f.seq2 = y.seq, f.slen2 = y.seq_len, f.qual2 = y.qual, f.qlen2 = y.qual_len;
            }
        } else {
            const ReadMeta &m = ch.meta[r];
            const uint32_t *off = ch.offsets();
            const char *s = (const char *)ch.seq.p + off[r];
            f.name1 = m.name1, f.nlen1 = m.nlen1, f.seq1 = s, f.slen1 = m.len1, f.qual1 = m.qual1, f.qlen1 = m.qlen1;
            if (paired) {
                f.name2 = m.name2, f.nlen2 = m.nlen2, f.seq2 = s + m.len1 + 1, f.slen2 = off[r + 1] - off[r] - m.len1 - 1;
                f.qual2 = m.qual2, f.qlen2 = m.qlen2;
            }
        }
        return f;
    }
    // start of the batch that read r belongs to, or -1 when that batch began in an earlier chunk
    static int64_t batch_begin(const Chunk<Alloc> &ch, uint32_t r)
    {
        auto it = std::upper_bound(ch.batch_start.begin(), ch.batch_start.end(), r);
        return it == ch.batch_start.begin() ? -1 : (int64_t) * (it - 1);
    }
    template <class Sink>
    static void put_u32(Sink &o, uint32_t v)
    {
        char d[10];
        int n = 0;
        do {
            d[9 - n++] = (char)('0' + v % 10u);
            v /= 10u;
        } while (v);
        o.put(d + 10 - n, (size_t)n);
    }
    template <class Sink>
    void format(const Chunk<Alloc> &ch, uint32_t a, uint32_t b, Sink &ssv, Sink &o1, Sink &o2, Sink &sc) const
    {
        // ReadOutput's previd (ReadOutput.hpp:41,44-48) entering this range: the name of the previous kept read of
        // the same batch - earlier in this chunk, or carried over from the previous chunk
        const char *previd = "";  // `string previd = ""`: an empty name at the start of a batch equals it
        uint32_t prevlen = 0;
        {
            const int64_t bb = batch_begin(ch, a);
            int64_t i = (int64_t)a - 1;
            for (; i >= 0 && i >= bb; --i)
                if (ch.gene16[(size_t)i] != kGeneNone) break;
            if (i >= 0 && i >= bb) {
                const Fields f = fields(ch, (uint32_t)i, paired_);
                previd = f.name1, prevlen = f.nlen1;
            } else if (bb < 0 && carry_valid_) {
                previd = carry_.data(), prevlen = (uint32_t)carry_.size();
            }
        }
        size_t next_batch = (size_t)(std::upper_bound(ch.batch_start.begin(), ch.batch_start.end(), a) - ch.batch_start.begin());
        const AssocPair *m_end = ch.multi + ch.n_multi;
        const AssocPair *m_it = std::lower_bound(ch.multi, m_end, a, [](const AssocPair &p, uint32_t r) { return p.read_idx < r; });
        for (uint32_t r = a; r < b; ++r) {
            if (next_batch < ch.batch_start.size() && ch.batch_start[next_batch] == r) {
                previd = "", prevlen = 0;  // `string previd = ""` per ReadOutput call = per batch
                ++next_batch;
            }
            const uint32_t g16 = ch.gene16[r];
            if (g16 == kGeneNone) continue;
            const Fields f = fields(ch, r, paired_);
            auto line = [&](uint32_t g) {
                ssv.put(f.name1, f.nlen1);
                ssv.putc(' ');
                if (g < legend_.size()) ssv.put(legend_[g].data(), legend_len_[g]);
                ssv.putc('\n');
            };
            if (g16 != kGeneMulti) {
                line(g16);
            } else {
                for (; m_it != m_end && m_it->read_idx == r; ++m_it) line(m_it->gene_idx);
            }
            if (has3_ && ch.scores) {
                const uint32_t *s = ch.scores + 4 * (size_t)r;
                sc.put(f.name1, f.nlen1);
                for (int i = 0; i < 4; ++i) {
                    sc.putc(' ');
                    put_u32(sc, s[i]);
                }
                sc.putc('\n');
            }
            // FASTQ once per read unless its name equals the previous printed id (ReadOutput.hpp:44-48)
            const bool same = prevlen == f.nlen1 && memcmp(previd, f.name1, prevlen) == 0;
            if (!same) {
                if (has1_) record(o1, f.name1, f.nlen1, f.seq1, f.slen1, f.qual1, f.qlen1);
                if (has2_) record(o2, f.name2, f.nlen2, f.seq2, f.slen2, f.qual2, f.qlen2);
            }
            previd = f.name1, prevlen = f.nlen1;
        }
    }
    template <class Sink>
    static void record(Sink &o, const char *name, uint32_t nlen, const char *seq, uint32_t slen, const char *qual, uint32_t qlen)
    {
        o.putc('@');
        o.put(name, nlen);
        o.putc('\n');
        o.put(seq, slen);
        o.put("\n+\n", 3);
        o.put(qual, qlen);
        o.putc('\n');
    }
    void update_carry(const Chunk<Alloc> &ch)
    {
        const int64_t bb = batch_begin(ch, ch.n - 1);  // the batch that is running at the end of the chunk
        int64_t i = (int64_t)ch.n - 1;
        for (; i >= 0 && i >= bb; --i)
            if (ch.gene16[(size_t)i] != kGeneNone) break;
        if (i >= 0 && i >= bb) {
            const Fields f = fields(ch, (uint32_t)i, paired_);
            carry_.assign(f.name1, f.nlen1);
            carry_valid_ = true;
        } else if (bb >= 0) {
            carry_valid_ = false;  // a batch began in this chunk and has printed nothing yet
        }  // else: the batch came from an earlier chunk and printed nothing here - the carry stands
    }

    const std::vector<std::string> &legend_;
    std::vector<uint32_t> legend_len_;
    bool paired_;
    OutBuf ssv_, out1_, out2_, scores_;
    bool has1_, has2_, has3_;
    // Output through mappings: the file is grown a window (1 GiB) at a time and the window mapped once; chunks
    // are formatted into it back to back.  -> address of the next `total` bytes of output f (nullptr: cannot map).
    struct Window {
        char *base = nullptr;  // mapping of [start, start + len)
        off_t start = 0, len = 0, pos = 0;  // pos = file offset of the next output byte
        off_t start0 = 0;                   // file offset where the first window's data began (pre-faulting)
    };
    struct Prefault {
        char *base = nullptr;
        uint64_t len = 0;
        std::atomic<uint64_t> cursor{0};
    };
    Prefault pre_[3];
    std::vector<std::thread> pre_threads_;
    std::atomic<bool> pre_stop_{false};
    char *window(int f, size_t total)
    {
        OutBuf *outs[kOuts] = {&ssv_, &out1_, &out2_, &scores_};
        Window &w = win_[f];
        const int fd = outs[f]->fd();
        if (!w.base) {
            outs[f]->flush();
            w.pos = lseek(fd, 0, SEEK_CUR);
            if (w.pos < 0) return nullptr;
            w.start0 = w.pos;
        }
        if (!w.base || w.pos + (off_t)total > w.start + w.len) {
            const off_t page = (off_t)sysconf(_SC_PAGESIZE), start = w.pos / page * page;
            const off_t len = std::max<off_t>((off_t)1 << 30, (w.pos - start) + (off_t)total);
            if (ftruncate(fd, start + len) != 0) return w.base ? (abort_windows(f), nullptr) : nullptr;
            void *mm = mmap(nullptr, (size_t)len, PROT_READ | PROT_WRITE, MAP_SHARED, fd, start);
            if (mm == MAP_FAILED) return w.base ? (abort_windows(f), nullptr) : nullptr;
            w.base = (char *)mm;  // (the previous window stays mapped: see flush())
            w.start = start;
            w.len = len;
        }
        return w.base + (w.pos - w.start);
    }
    void abort_windows(int f)  // mapping failed mid-way: continue with write(2) at the current position
    {
        OutBuf *outs[kOuts] = {&ssv_, &out1_, &out2_, &scores_};
        if (ftruncate(outs[f]->fd(), win_[f].pos) != 0) {
        }
        lseek(outs[f]->fd(), win_[f].pos, SEEK_SET);
        win_[f] = Window{};
        mappable_[f] = false;
    }
    Window win_[kOuts];
    bool mappable_[kOuts] = {false, false, false, false};  // a regular file opened read-write (a shared mapping needs both)
    bool populate_ = false;
    std::vector<char> priv_[kOuts][2];
    int priv_turn_[kOuts] = {0, 0, 0, 0};
    uint64_t priv_job_[kOuts][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};
    // background write(2) of private buffers, in submission order
    struct AsyncJob {
        OutBuf *ob;
        const char *p;
        size_t n;
    };
    std::thread async_thread_;
    std::mutex async_mu_;
    std::condition_variable async_cv_;
    std::deque<AsyncJob> async_q_;
    uint64_t async_submitted_ = 0, async_done_ = 0;
    bool async_stop_ = false;
    uint64_t submit_async(OutBuf *ob, const char *p, size_t n)
    {
        std::unique_lock<std::mutex> lk(async_mu_);
        if (!async_thread_.joinable())
            async_thread_ = std::thread([this] {
                std::unique_lock<std::mutex> lk2(async_mu_);
                for (;;) {
                    async_cv_.wait(lk2, [&] { return async_stop_ || !async_q_.empty(); });
                    if (async_q_.empty()) return;
                    const AsyncJob j = async_q_.front();
                    async_q_.pop_front();
                    lk2.unlock();
                    j.ob->put(j.p, j.n);
                    lk2.lock();
                    ++async_done_;
                    async_cv_.notify_all();
                }
            });
        async_q_.push_back(AsyncJob{ob, p, n});
        const uint64_t id = ++async_submitted_;
        async_cv_.notify_all();
        return id;
    }
    void wait_async(uint64_t id)
    {
        if (!id) return;
        std::unique_lock<std::mutex> lk(async_mu_);
        async_cv_.wait(lk, [&] { return async_done_ >= id; });
    }
    void stop_async()
    {
        {
            std::unique_lock<std::mutex> lk(async_mu_);
            async_cv_.wait(lk, [&] { return async_done_ >= async_submitted_; });
            async_stop_ = true;
            async_cv_.notify_all();
        }
        if (async_thread_.joinable()) async_thread_.join();
        async_stop_ = false;
    }
    std::string carry_;
    bool carry_valid_ = false;
};

}  // namespace shkhost
