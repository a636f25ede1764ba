// shark-b200: command-line drop-in for the reference's `shark` (main.cpp:83-240) on top of the
// C ABI of libshark_b200.so.  Same options (argument_parser.hpp:29-174), same stdout ssv
// (ReadOutput.hpp:43), same filtered FASTQ files (ReadOutput.hpp:44-47), same stderr stage
// stamps.  The host does what the north star leaves on the host: FASTA/FASTQ parsing
// (ingest.hpp, fastpipe.hpp), batching into packed chunks (FastaSplitter.hpp / FastqSplitter.hpp) and
// output (ReadOutput.hpp); everything between goes through shk_index_build / shk_reads_submit_packed /
// shk_reads_collect.  Extensions (not in the reference): --gpus N, --chunk-reads N, --sharded-build
// (with --gpus N: every GPU indexes one gene shard, filters OR-merged over NVLink, instead of build +
// replicate), --save-index FILE / --load-index FILE (the reference rebuilds its index on every run;
// the gene names still come from -r), --wide-ids (32-bit gene ids: references of more than 65536 records, which
// the reference's 16-bit ids cannot index - small_vector.hpp:46; without the flag such inputs end with an error),
// --scores FILE (one line `<name> <len> <cov> <hits> <n_best>` per reported read, in the order of the ssv: the numbers
// behind each answer, from which any -c / -s can be applied afterwards - shk_read_score, include/shark_b200.h).
//
// Pipeline (pipeline.hpp, fastpipe.hpp, ingest.hpp): plain input files are memory-mapped and scanned by
// the host pool in parallel (compressed ones by a streaming scanner per file); a batcher thread turns runs
// of records into chunks in the packed form of shk_reads_submit_packed (2-bit code + validity bit per base,
// the pool packs 64 KiB pieces straight from the mapped input); the main thread submits chunk i+1 to a free
// slot before it collects chunk i (double buffering per GPU, chunks round-robin over GPUs); a writer thread
// formats the compact results in parallel and writes them in chunk order, which reproduces the reference's
// `-t 1` output order.  Scanning and packing start with the process, concurrently with CUDA start-up and
// the index build.
#include <fcntl.h>
#include <getopt.h>
#include <malloc.h>
#include <signal.h>
#include <sys/mman.h>
#include <sys/wait.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <iostream>
#include <memory>
#include <mutex>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/shark_b200.h"
#include "pipeline.hpp"

namespace {

// The reference's usage text is part of its observable behaviour (-h, argument errors).
const char *USAGE_MESSAGE =
    "Usage: shark -r <references> -1 <sample1> [OPTIONAL ARGUMENTS]\n"
    "\n"
    "Arguments:\n"
    "      -r, --reference                   reference sequences in FASTA format (can be gzipped)\n"
    "      -1, --sample1                     sample in FASTQ (can be gzipped)\n"
    "\n"
    "Optional arguments:\n"
    "      -h, --help                        display this help and exit\n"
    "      -2, --sample2                     second sample in FASTQ (optional, can be gzipped)\n"
    "      -o, --out1                        first output sample in FASTQ (default: sharked_sample.1)\n"
    "      -p, --out2                        second output sample in FASTQ (default: sharked_sample.2)\n"
    "      -k, --kmer-size                   size of the kmers to index (default:17, max:31)\n"
    "      -c, --confidence                  confidence for associating a read to a gene (default:0.6)\n"
    "      -b, --bf-size                     bloom filter size in GB (default:1)\n"
    "      -q, --min-base-quality            minimum base quality (assume FASTQ Illumina 1.8+ Phred scale, default:0, i.e., no filtering)\n"
    "      -s, --single                      report an association only if a single gene is found\n"
    "      -t, --threads                     number of threads (default:1)\n"
    "      -v, --verbose                     verbose mode\n";

struct Options {
    std::string fasta_path, sample1_path, sample2_path, out1_path, out2_path;
    bool paired = false;
    unsigned k = 17;
    double c = 0.6;
    uint64_t bf_size = 1ull << 33;
    char min_quality = 0;
    bool single = false, verbose = false;
    int n_threads = 1;
    int gpus = 1;                   // extension
    unsigned chunk_reads = 1000000; // extension
    bool sharded_build = false;     // extension
    bool wide_ids = false;          // extension: more than 65536 reference records (SHK_F_WIDE_IDS)
    std::string save_index, load_index;  // extensions
    std::string scores_path;        // extension: per-read score records (SHK_F_SCORES)
};

[[noreturn]] void usage_error(const char *msg, bool with_usage)
{
    if (with_usage) std::cerr << USAGE_MESSAGE;
    std::cerr << msg << std::endl << "aborting..." << std::endl;
    exit(EXIT_FAILURE);
}

// The reference's options (argument_parser.hpp:65-82) and ours, one row each: getopt value, long name, whether
// it takes an argument, and what it does with the argument (an istringstream, so that e.g. "-k 17abc" parses
// like the reference does; validation and messages as in argument_parser.hpp:84-166).
struct OptionRow {
    int key;
    const char *long_name;
    bool has_arg;
    void (*apply)(Options &, std::istringstream &);
};
const OptionRow kOptions[] = {
    {'r', "reference", true, [](Options &o, std::istringstream &a) { a >> o.fasta_path; }},
    {'t', "threads", true,
     [](Options &o, std::istringstream &a) {
         a >> o.n_threads;
         if (o.n_threads <= 0) {
             std::cerr << "USAGE_MESSAGE";  // sic: argument_parser.hpp:94
             usage_error("shark: at least 1 thread is required.", false);
         }
     }},
    {'1', "sample1", true, [](Options &o, std::istringstream &a) { a >> o.sample1_path; }},
    {'2', "sample2", true,
     [](Options &o, std::istringstream &a) {
         a >> o.sample2_path;
         o.paired = true;
     }},
    {'o', "out1", true, [](Options &o, std::istringstream &a) { a >> o.out1_path; }},
    {'p', "out2", true, [](Options &o, std::istringstream &a) { a >> o.out2_path; }},
    {'k', "kmer-size", true,
     [](Options &o, std::istringstream &a) {
         a >> o.k;
         if (o.k == 0 || o.k > 31) usage_error("shark: k must be in the range [1, 31].", true);
     }},
    {'c', "confidence", true,
     [](Options &o, std::istringstream &a) {
         a >> o.c;
         if (o.c < 0 || o.c > 1) usage_error("shark: c must be in the range [0, 1].", false);
     }},
    {'b', "bf-size", true,
     [](Options &o, std::istringstream &a) {
         a >> o.bf_size;
         o.bf_size = o.bf_size * (1ull << 33);  // "GB": argument_parser.hpp:130-134
     }},
    {'q', "min-base-quality", true,
     [](Options &o, std::istringstream &a) {
         int mq = 0;
         a >> mq;
         if (mq < 0) usage_error("shark: q must be a positive value.", true);
         o.min_quality = static_cast<char>(mq);
     }},
    {'s', "single", false, [](Options &o, std::istringstream &) { o.single = true; }},
    {'v', "verbose", false, [](Options &o, std::istringstream &) { o.verbose = true; }},
    {'h', "help", false,
     [](Options &, std::istringstream &) {
         std::cerr << USAGE_MESSAGE;
         exit(EXIT_SUCCESS);
     }},
    {1000, "gpus", true, [](Options &o, std::istringstream &a) { a >> o.gpus; }},
    {1001, "chunk-reads", true, [](Options &o, std::istringstream &a) { a >> o.chunk_reads; }},
    {1002, "sharded-build", false, [](Options &o, std::istringstream &) { o.sharded_build = true; }},
    {1003, "save-index", true, [](Options &o, std::istringstream &a) { a >> o.save_index; }},
    {1004, "load-index", true, [](Options &o, std::istringstream &a) { a >> o.load_index; }},
    {1005, "wide-ids", false, [](Options &o, std::istringstream &) { o.wide_ids = true; }},
    {1006, "scores", true, [](Options &o, std::istringstream &a) { a >> o.scores_path; }},
};

Options parse_arguments(int argc, char **argv)
{
    Options opt;
    std::string shortopts;
    std::vector<struct option> longopts;
    for (const OptionRow &row : kOptions) {
        if (row.key < 256) {
            shortopts += (char)row.key;
            if (row.has_arg) shortopts += ':';
        }
        longopts.push_back({row.long_name, row.has_arg ? required_argument : no_argument, nullptr, row.key});
    }
    longopts.push_back({nullptr, 0, nullptr, 0});
    for (int ch; (ch = getopt_long(argc, argv, shortopts.c_str(), longopts.data(), nullptr)) != -1;) {
        std::istringstream arg(optarg != nullptr ? optarg : "");
        const OptionRow *row = nullptr;
        for (const OptionRow &r : kOptions)
            if (r.key == ch) row = &r;
        if (!row) {
            std::cerr << "shark : unknown argument" << std::endl;
            std::cerr << "\n" << USAGE_MESSAGE;
            exit(EXIT_FAILURE);
        }
        row->apply(opt, arg);
    }
    if (opt.fasta_path.empty() || opt.sample1_path.empty()) {
        std::cerr << "shark : missing required files" << std::endl;
        std::cerr << "\n" << USAGE_MESSAGE;
        exit(EXIT_FAILURE);
    }
    if (opt.out1_path.empty()) opt.out1_path = "sharked_sample.1";
    if (opt.out2_path.empty() && !opt.sample2_path.empty()) opt.out2_path = "sharked_sample.2";
    if (opt.gpus < 1) opt.gpus = 1;
    return opt;
}

auto start_t = std::chrono::high_resolution_clock::now();
void pelapsed(const std::string &s)  // main.cpp:49-54
{
    auto now_t = std::chrono::high_resolution_clock::now();
    std::cerr << "[shark/" << s << "] Time elapsed "
              << std::chrono::duration_cast<std::chrono::milliseconds>(now_t - start_t).count() / 1000 << std::endl;
}

// SHK_TIMING=1: millisecond stamps of the host stages on stderr (not part of the reference's output)
const bool g_timing = getenv("SHK_TIMING") != nullptr;
void tstamp(const char *what)
{
    if (!g_timing) return;
    auto now_t = std::chrono::high_resolution_clock::now();
    fprintf(stderr, "[shark-b200/timing] %-28s %8.1f ms\n", what,
            std::chrono::duration_cast<std::chrono::microseconds>(now_t - start_t).count() / 1000.0);
}

[[noreturn]] void die(const std::string &msg)
{
    std::cerr << "shark: " << msg << std::endl;
    fflush(nullptr);
    _exit(EXIT_FAILURE);  // worker threads may be running: no static destructors under their feet
}

using shkhost::kBatch;

// Staging memory of the exact-path chunks (text, qualities); the packed chunks themselves live in the memory shared
// with the device process.  Ordinary memory: the host process never calls into CUDA.
struct HostAlloc {
    static void *alloc(size_t n)
    {
        void *q = nullptr;
        if (posix_memalign(&q, 4096, n) != 0) die("out of memory");
        return q;
    }
    static void free(void *p) { ::free(p); }
};
using Chunk = shkhost::Chunk<HostAlloc>;
using Batcher = shkhost::Batcher<HostAlloc>;
using Writer = shkhost::Writer<HostAlloc>;
static_assert(sizeof(shkhost::AssocPair) == sizeof(shk_assoc), "AssocPair mirrors shk_assoc");
static_assert(shkhost::kGeneNone == SHK_GENE_NONE && shkhost::kGeneMulti == SHK_GENE_MULTI, "compact result markers");

void pack_piece(const uint8_t *seq, const uint8_t *qual, int32_t min_quality, uint64_t n, uint64_t *codes, uint32_t *valid)
{
    shk_host_pack(seq, qual, min_quality, n, codes, valid, 0);  // the caller is one of the pool's threads already
}

// Simple blocking queue for the hand-offs between the pipeline threads.
template <class T>
class Channel {
public:
    void push(T v)
    {
        std::unique_lock<std::mutex> lk(mu_);
        q_.push_back(std::move(v));
        cv_.notify_all();
    }
    T pop()
    {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return !q_.empty(); });
        T v = std::move(q_.front());
        q_.pop_front();
        return v;
    }

private:
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<T> q_;
};

#define SHK_TRY(ctx, call)                                                              \
    do {                                                                                \
        int rc_ = (call);                                                               \
        if (rc_ != SHK_OK) die(std::string(#call " failed: ") + shk_last_error(ctx));   \
    } while (0)

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// Two processes.  The process the user starts is the HOST process: it scans the sample files, builds the packed
// chunks, formats and writes the output.  Before it creates a single thread it forks the DEVICE process, which
// owns everything CUDA: device contexts, index build, shk_reads_submit_packed / shk_reads_collect.  Why two:
//   * CUDA start-up (0.4 - 2 s on these boxes) reserves and maps address space for most of that time with the
//     process's memory-map lock held, and every page fault of every other thread of the SAME process waits for
//     it - measured: not one chunk of the sample was packed before the context was up, although the packing
//     threads had the cores to themselves.  In its own process the host pipeline runs at full speed meanwhile.
//   * When the last output byte is written the host process returns; what is left - unmapping, freeing and the
//     driver taking the device context apart, about half a second - is the device process's business, which
//     finishes on its own ("detached tear-down").
// The two share one anonymous mapping created before the fork: per chunk buffer a slot with the packed chunk
// (offsets, code words, validity words; host -> device) and the compact results (one 16-bit word per read + the
// list for ties, and with --scores the score records, 16 bytes per read; device -> host).  Two pipes carry the small messages.  SHK_ONE_PROCESS=1 runs the device side as
// a thread of the host process instead (same protocol; for debuggers and sanitizers).
// ---------------------------------------------------------------------------------------------------------
struct SlotView {
    uint32_t *off;
    uint64_t *codes;
    uint32_t *valid;
    uint16_t *gene16;
    shkhost::AssocPair *multi;
    uint32_t *scores;  // nullptr without --scores
};
struct SharedLayout {
    char *base = nullptr;
    size_t n_slots = 0, slot_bytes = 0;
    size_t off_bytes = 0, codes_bytes = 0, valid_bytes = 0, gene_bytes = 0, multi_cap = 0, scores_bytes = 0;
    static size_t round(size_t n) { return (n + 4095) / 4096 * 4096; }
    void plan(size_t slots, size_t max_reads, uint64_t max_bytes, bool scores)
    {
        n_slots = slots;
        const size_t groups = (size_t)((max_bytes + 31) / 32) + 2;
        off_bytes = round((max_reads + 2) * 4);
        codes_bytes = round(groups * 8 + 64);
        valid_bytes = round(groups * 4 + 64);
        gene_bytes = round((max_reads + 64) * 2);
        multi_cap = max_reads;  // entries; a chunk with more ties than reads sends the rest through the pipe
        scores_bytes = scores ? round(max_reads * sizeof(shk_read_score)) : 0;
        slot_bytes = off_bytes + codes_bytes + valid_bytes + gene_bytes + round(multi_cap * sizeof(shkhost::AssocPair)) + scores_bytes;
    }
    bool map()
    {
        void *m = mmap(nullptr, n_slots * slot_bytes, PROT_READ | PROT_WRITE, MAP_SHARED | MAP_ANONYMOUS | MAP_NORESERVE, -1, 0);
        if (m == MAP_FAILED) return false;
        base = (char *)m;
        return true;
    }
    SlotView slot(size_t i) const
    {
        char *p = base + i * slot_bytes;
        SlotView v;
        v.off = (uint32_t *)p;
        v.codes = (uint64_t *)(p + off_bytes);
        v.valid = (uint32_t *)(p + off_bytes + codes_bytes);
        v.gene16 = (uint16_t *)(p + off_bytes + codes_bytes + valid_bytes);
        v.multi = (shkhost::AssocPair *)(p + off_bytes + codes_bytes + valid_bytes + gene_bytes);
        v.scores = scores_bytes ? (uint32_t *)(p + slot_bytes - scores_bytes) : nullptr;
        return v;
    }
};

enum : uint32_t { kMsgChunk = 1, kMsgEnd = 2, kMsgReady = 3, kMsgResult = 4, kMsgDone = 5 };
struct Msg {  // both directions; well below PIPE_BUF, so a write is atomic
    uint32_t kind = 0, slot = 0;
    uint32_t n_reads = 0, n_genes = 0;
    uint64_t n_bytes = 0, n_multi = 0, tail = 0;  // tail: multi entries that follow on the pipe (beyond the slot's capacity)
};

bool write_all(int fd, const void *p, size_t n)
{
    const char *c = (const char *)p;
    while (n) {
        const ssize_t w = write(fd, c, n);
        if (w <= 0) {
            if (w < 0 && errno == EINTR) continue;
            return false;
        }
        c += w;
        n -= (size_t)w;
    }
    return true;
}
bool read_all(int fd, void *p, size_t n)
{
    char *c = (char *)p;
    while (n) {
        const ssize_t r = read(fd, c, n);
        if (r <= 0) {
            if (r < 0 && errno == EINTR) continue;
            return false;
        }
        c += r;
        n -= (size_t)r;
    }
    return true;
}

// ---- the device side -----------------------------------------------------------------------------------------
// Reference -> index on every GPU; then chunks as they are announced on `in`, results announced on `out`.
void device_main(const Options &opt, const SharedLayout &shm, unsigned chunk_reads, uint64_t max_chunk_bytes, int in, int out)
{
    const int32_t min_quality = (int32_t)(unsigned char)opt.min_quality;
    // the driver initialises every visible device: name only the ones this run uses (a second per GPU saved on
    // an 8-GPU box); a CUDA_VISIBLE_DEVICES set by the user stands
    {
        std::string vis;
        for (int g = 0; g < opt.gpus; ++g) vis += (g ? "," : "") + std::to_string(g);
        setenv("CUDA_VISIBLE_DEVICES", vis.c_str(), 0);
    }
    // FastaSplitter (FastaSplitter.hpp:42-54) -> concatenated records, parsed while the contexts come up.
    // Unlike the reference (which ignores open failures and later segfaults) we fail cleanly.
    std::vector<uint8_t> ref_bases;
    std::vector<uint64_t> rec_off{0};
    uint32_t n_records = 0;
    std::thread ref_thread([&] {
        shkhost::RecordSource ref(opt.fasta_path.c_str());
        if (!ref.ok()) die("cannot open reference " + opt.fasta_path);
        ref.start();
        for (;;) {
            const shkhost::Rec r = ref.peek();
            if (r.status < 0) break;  // `while ((seq_len = kseq_read(seq)) >= 0)`, FastaSplitter.hpp:46
            const void *zs = memchr(r.seq, 0, r.seq_len);  // `seq->seq.s` as a C string (FastaSplitter.hpp:49)
            const size_t l = zs ? (size_t)((const char *)zs - r.seq) : r.seq_len;
            ref_bases.insert(ref_bases.end(), r.seq, r.seq + l);
            rec_off.push_back(ref_bases.size());
            ++n_records;
            ref.consume();
        }
        tstamp("reference parsed");
    });
    std::vector<shk_ctx *> ctxs((size_t)opt.gpus, nullptr);
    for (int g = 0; g < opt.gpus; ++g) {
        shk_params p;
        memset(&p, 0, sizeof p);
        p.k = opt.k;
        p.c = opt.c;
        p.bf_bits = opt.bf_size;
        p.min_quality = min_quality;
        p.single = opt.single ? 1 : 0;
        p.device = g;
        p.n_slots = 2;
        p.max_reads_per_chunk = chunk_reads;
        p.max_bytes_per_chunk = max_chunk_bytes;
        p.flags = SHK_F_COMPACT_RESULTS | (opt.wide_ids ? SHK_F_WIDE_IDS : 0u) | (opt.scores_path.empty() ? 0u : SHK_F_SCORES);
        if (shk_create(&p, &ctxs[g]) != SHK_OK) die(std::string("shk_create: ") + shk_last_error(nullptr));
    }
    tstamp("contexts created");
    ref_thread.join();
    shk_index_info info;
    bool replicated = false;
    if (!opt.load_index.empty()) {
        SHK_TRY(ctxs[0], shk_index_load(ctxs[0], opt.load_index.c_str(), &info));
        if (info.n_records != n_records)
            die("index " + opt.load_index + " was built from " + std::to_string(info.n_records) + " records, " +
                opt.fasta_path + " has " + std::to_string(n_records));
    } else if (opt.sharded_build && opt.gpus > 1) {
        SHK_TRY(ctxs[0], shk_index_build_sharded(ctxs.data(), (uint32_t)opt.gpus, ref_bases.data(), rec_off.data(), n_records, &info));
        replicated = true;
    } else {
        SHK_TRY(ctxs[0], shk_index_build(ctxs[0], ref_bases.data(), rec_off.data(), n_records, &info));
    }
    tstamp("index built");
    if (!opt.save_index.empty()) {
        SHK_TRY(ctxs[0], shk_index_save(ctxs[0], opt.save_index.c_str()));
        tstamp("index saved");
    }
    if (!replicated)
        for (int g = 1; g < opt.gpus; ++g) SHK_TRY(ctxs[g], shk_index_replicate(ctxs[0], ctxs[g]));
    tstamp("index ready");
    std::vector<uint8_t>().swap(ref_bases);
    Msg ready;
    ready.kind = kMsgReady;
    ready.n_genes = info.n_genes;
    if (!write_all(out, &ready, sizeof ready)) _exit(EXIT_FAILURE);

    struct InFlight {
        uint32_t shm_slot;
        int gpu;
        uint32_t slot;
    };
    std::deque<InFlight> inflight;
    const size_t max_inflight = (size_t)opt.gpus * 2;
    uint64_t submitted = 0;
    double t_submit = 0, t_collect = 0;
    auto drain_one = [&] {
        const InFlight f = inflight.front();
        inflight.pop_front();
        shk_chunk_result res;
        const double t0 = shkhost::stage_now();
        SHK_TRY(ctxs[f.gpu], shk_reads_collect(ctxs[f.gpu], f.slot, &res));
        t_collect += shkhost::stage_now() - t0;
        // the slot's result buffers are reused by its next submit: the compact results go to the shared slot
        const SlotView v = shm.slot(f.shm_slot);
        memcpy(v.gene16, res.gene16, (size_t)res.n_reads * 2);
        const uint64_t in_slot = std::min<uint64_t>(res.n_multi, shm.multi_cap);
        if (in_slot) memcpy(v.multi, res.multi, in_slot * sizeof(shk_assoc));
        if (v.scores) {
            const shk_read_score *sc = nullptr;
            uint32_t n_sc = 0;
            SHK_TRY(ctxs[f.gpu], shk_reads_scores(ctxs[f.gpu], f.slot, &sc, &n_sc));
            memcpy(v.scores, sc, (size_t)n_sc * sizeof(shk_read_score));
        }
        Msg m;
        m.kind = kMsgResult;
        m.slot = f.shm_slot;
        m.n_reads = res.n_reads;
        m.n_multi = res.n_multi;
        m.tail = res.n_multi - in_slot;
        if (!write_all(out, &m, sizeof m) || (m.tail && !write_all(out, res.multi + in_slot, m.tail * sizeof(shk_assoc)))) _exit(EXIT_FAILURE);
    };
    for (;;) {
        Msg c;
        if (!read_all(in, &c, sizeof c)) _exit(EXIT_FAILURE);  // the host process is gone
        if (c.kind == kMsgEnd) break;
        if (submitted == 0) tstamp("first chunk submitted");
        if (inflight.size() == max_inflight) drain_one();
        const int gpu = (int)(submitted % (uint64_t)opt.gpus);
        const uint32_t slot = (uint32_t)((submitted / (uint64_t)opt.gpus) % 2);
        const SlotView v = shm.slot(c.slot);
        const double t0 = shkhost::stage_now();
        SHK_TRY(ctxs[gpu], shk_reads_submit_packed(ctxs[gpu], slot, v.codes, v.valid, v.off, c.n_reads));
        t_submit += shkhost::stage_now() - t0;
        inflight.push_back({c.slot, gpu, slot});
        ++submitted;
    }
    while (!inflight.empty()) drain_one();
    tstamp("last chunk collected");
    if (g_timing) fprintf(stderr, "[shark-b200/timing] device side: %llu chunks, submit %.0f ms, collect %.0f ms\n",
                          (unsigned long long)submitted, t_submit * 1e3, t_collect * 1e3);
    Msg d;
    d.kind = kMsgDone;
    write_all(out, &d, sizeof d);
    if (getenv("SHK_CLEAN_EXIT")) {
        for (auto *c : ctxs) shk_destroy(c);
    }
}

int main(int argc, char *argv[])
{
    // the record arrays and staging buffers of the pipeline are megabytes each and are recycled chunk after chunk:
    // keep them in the heap (fresh anonymous mappings would cost a page fault per 4 KiB every time)
    mallopt(M_MMAP_THRESHOLD, 32 << 20);
    mallopt(M_TRIM_THRESHOLD, 1 << 30);
    const Options opt = parse_arguments(argc, argv);

    if (opt.verbose) {  // main.cpp:113-123
        std::cerr << "Reference texts: " << opt.fasta_path << std::endl;
        std::cerr << "Sample 1: " << opt.sample1_path << std::endl;
        if (opt.paired) std::cerr << "Sample 2: " << opt.sample2_path << std::endl;
        std::cerr << "K-mer length: " << opt.k << std::endl;
        std::cerr << "Threshold value: " << opt.c << std::endl;
        std::cerr << "Only single associations: " << (opt.single ? "Yes" : "No") << std::endl;
        std::cerr << "Minimum base quality: " << static_cast<int>(opt.min_quality) << std::endl;
        std::cerr << std::endl;
    }
    if (opt.n_threads > 1) shkhost::set_ingest_threads(opt.n_threads);  // -t: inflate threads for blocked-gzip samples
    const unsigned chunk_reads = std::max(1000u, opt.chunk_reads);
    // slot buffers are sized by this; a chunk is closed early when its text would not fit
    const uint64_t max_chunk_bytes = std::min<uint64_t>(0xF0000000ull, std::max<uint64_t>((uint64_t)chunk_reads * 640, 64ull << 20));
    // chunk buffers: what the GPUs have in flight (2 each) + the writer's + enough for the host side to keep packing
    // while the device process is still starting up (the device side drains them in a few milliseconds each)
    size_t n_bufs = std::max<size_t>((size_t)opt.gpus * 2 + 3, 16);
    if (const char *ev = getenv("SHK_CHUNK_BUFFERS")) {
        const long v = atol(ev);
        if (v >= (long)opt.gpus * 2 + 2 && v <= 256) n_bufs = (size_t)v;
    }
    // the sample files are opened (and mapped) before the device process exists, so that a missing file ends the
    // run here; no thread runs yet
    const int32_t min_quality = (int32_t)(unsigned char)opt.min_quality;
    Batcher batcher(opt.sample1_path.c_str(), opt.paired ? opt.sample2_path.c_str() : nullptr, min_quality, pack_piece);
    if (!batcher.files_ok()) die("cannot open sample file(s)");
    {  // unlike the reference (which ignores open failures and later segfaults) a missing reference ends the run here
        const int fd = open(opt.fasta_path.c_str(), O_RDONLY);
        if (fd < 0) die("cannot open reference " + opt.fasta_path);
        close(fd);
    }
    SharedLayout shm;
    shm.plan(n_bufs, chunk_reads, max_chunk_bytes, !opt.scores_path.empty());
    if (!shm.map()) die("cannot map the chunk buffers");
    int h2d[2], d2h[2];
    if (pipe(h2d) != 0 || pipe(d2h) != 0) die("cannot create pipes");
    signal(SIGPIPE, SIG_IGN);
    fflush(nullptr);
    const bool one_process = getenv("SHK_ONE_PROCESS") && atoi(getenv("SHK_ONE_PROCESS")) != 0;
    pid_t child = -1;
    std::thread device_thread;
    if (one_process) {
        device_thread = std::thread([&] { device_main(opt, shm, chunk_reads, max_chunk_bytes, h2d[0], d2h[1]); });
    } else {
        child = fork();  // before this process has any thread
        if (child < 0) die("cannot fork the device process");
        if (child == 0) {
            close(h2d[1]);
            close(d2h[0]);
            device_main(opt, shm, chunk_reads, max_chunk_bytes, h2d[0], d2h[1]);
            fflush(nullptr);
            _exit(0);  // tear-down of the device context happens here, after the host process has returned
        }
        close(h2d[0]);
        close(d2h[1]);
    }
    // the device process ended without finishing its job: pass its fate on
    auto device_failed = [&]() -> int {
        if (child > 0) {
            int status = 0;
            while (waitpid(child, &status, 0) < 0 && errno == EINTR) {
            }
            if (WIFEXITED(status) && WEXITSTATUS(status) != 0) return WEXITSTATUS(status);
            if (WIFSIGNALED(status)) {
                signal(WTERMSIG(status), SIG_DFL);
                raise(WTERMSIG(status));
            }
        }
        return EXIT_FAILURE;
    };

    // ---- host side: scanners -> batcher thread -> (device process) -> writer thread
    // The device process's start-up is the critical path of a run and is mostly one thread deep; the host side
    // has a dozen threads that would happily take every core.  They run at a lower priority (threads created
    // from here on inherit it), so that the scheduler serves the device process first.
    if (!one_process && !(getenv("SHK_HOST_NICE") && atoi(getenv("SHK_HOST_NICE")) == 0)) {
        errno = 0;
        if (nice(getenv("SHK_HOST_NICE") ? atoi(getenv("SHK_HOST_NICE")) : 10) == -1 && errno != 0) {
        }
    }
    batcher.start();
    std::vector<std::unique_ptr<Chunk>> pool;
    Channel<Chunk *> free_q, write_q;
    for (size_t i = 0; i < n_bufs; ++i) {
        pool.emplace_back(new Chunk);
        Chunk &c = *pool.back();
        const SlotView v = shm.slot(i);
        c.slot = (int)i;
        c.off.use(v.off, shm.off_bytes);
        c.codes.use(v.codes, shm.codes_bytes);
        c.valid.use(v.valid, shm.valid_bytes);
        free_q.push(&c);
    }
    std::atomic<uint64_t> chunks_sent{0};
    std::atomic<bool> input_done{false};
    std::thread parser([&] {  // builds chunks and announces them to the device process
        for (;;) {
            Chunk *ch = free_q.pop();
            const bool more = batcher.fill(*ch, chunk_reads, max_chunk_bytes);
            if (batcher.error()) die(batcher.error());
            if (ch->n) {
                Msg m;
                m.kind = kMsgChunk;
                m.slot = (uint32_t)ch->slot;
                m.n_reads = ch->n;
                m.n_bytes = ch->bytes;
                chunks_sent.fetch_add(1);
                if (!write_all(h2d[1], &m, sizeof m)) break;  // the device process is gone: the reader below reports it
            } else {
                ch->clear();
                free_q.push(ch);
            }
            if (!more) break;
        }
        input_done.store(true);
        Msg e;
        e.kind = kMsgEnd;
        write_all(h2d[1], &e, sizeof e);
        tstamp("all chunks packed");
    });

    // legend_ID (FastaSplitter.hpp:48): every record's name, in file order
    std::vector<std::string> legend_ID;
    {
        shkhost::RecordSource ref(opt.fasta_path.c_str());
        if (ref.ok()) ref.start();  // (a reference that cannot be opened: the device process says so and ends the run)
        for (; ref.ok();) {
            const shkhost::Rec r = ref.peek();
            if (r.status < 0) break;
            const void *zn = memchr(r.name, 0, r.name_len);  // `seq->name.s` as a C string
            legend_ID.emplace_back(r.name, zn ? (size_t)((const char *)zn - r.name) : r.name_len);
            ref.consume();
        }
    }
    const int fd1 = opt.out1_path.empty() ? -1 : open(opt.out1_path.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0666);
    const int fd2 = (!opt.paired || opt.out2_path.empty()) ? -1 : open(opt.out2_path.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0666);
    const int fd_scores = opt.scores_path.empty() ? -1 : open(opt.scores_path.c_str(), O_RDWR | O_CREAT | O_TRUNC, 0666);
    if (!opt.scores_path.empty() && fd_scores < 0) die("cannot create " + opt.scores_path);
    Writer writer(STDOUT_FILENO, fd1, fd2, legend_ID, opt.paired, fd_scores);
    if (!(getenv("SHK_PREFAULT") && atoi(getenv("SHK_PREFAULT")) == 0)) {
        // the filtered FASTQ of a FASTQ sample is never longer than the sample (pipeline.hpp, Writer::start_prefault)
        auto plain_size = [](const std::string &path) -> uint64_t {
            shkhost::MappedFile m(path.c_str());  // maps only plain regular files
            return m.ok() && m.size() > 0 && m.data()[0] == '@' ? (uint64_t)m.size() : 0;
        };
        const uint64_t expect[3] = {0, fd1 >= 0 ? plain_size(opt.sample1_path) : 0, fd2 >= 0 ? plain_size(opt.sample2_path) : 0};
        writer.start_prefault(expect, std::max(1, shkhost::host_threads() / (opt.paired ? 8 : 4)));
    }
    std::thread writer_thread([&] {
        for (;;) {
            Chunk *ch = write_q.pop();
            if (!ch) break;
            writer.write(*ch);
            ch->clear();  // releases the scanner blocks
            free_q.push(ch);
        }
        writer.flush();
    });

    // results, in the order the chunks were sent
    uint64_t total_reads = 0, chunks_done = 0;
    bool got_ready = false, got_done = false;
    for (;;) {
        Msg m;
        if (!read_all(d2h[0], &m, sizeof m)) break;
        if (m.kind == kMsgReady) {
            got_ready = true;
            pelapsed("Transcript file processed");
            pelapsed("First switch performed");
            pelapsed("BF created from transcripts (" + std::to_string(m.n_genes) + " genes)");
            pelapsed("Second switch performed");
            continue;
        }
        if (m.kind == kMsgDone) {
            got_done = true;
            break;
        }
        if (m.kind != kMsgResult || m.slot >= n_bufs) break;
        Chunk *ch = pool[m.slot].get();
        const SlotView v = shm.slot(m.slot);
        ch->gene16 = v.gene16;
        ch->scores = v.scores;
        if (m.tail) {  // more ties than the slot holds: the whole list, slot part + pipe part, in the chunk's own vector
            ch->multi_v.resize((size_t)m.n_multi);
            memcpy(ch->multi_v.data(), v.multi, (size_t)(m.n_multi - m.tail) * sizeof(shkhost::AssocPair));
            if (!read_all(d2h[0], ch->multi_v.data() + (m.n_multi - m.tail), (size_t)m.tail * sizeof(shkhost::AssocPair))) break;
            ch->multi = ch->multi_v.data();
        } else {
            ch->multi = v.multi;
        }
        ch->n_multi = (size_t)m.n_multi;
        total_reads += ch->n;
        ++chunks_done;
        write_q.push(ch);
    }
    if (!got_ready || !got_done) {
        fflush(nullptr);
        _exit(device_failed());
    }
    tstamp("last results received");
    parser.join();
    write_q.push(nullptr);
    writer_thread.join();
    if (fd1 >= 0) close(fd1);
    if (fd2 >= 0) close(fd2);
    if (fd_scores >= 0) close(fd_scores);
    tstamp("output written");
    if (g_timing) {
        const shkhost::StageTimes &st = shkhost::stage_times();
        fprintf(stderr, "[shark-b200/timing] reads %llu in %llu chunks, %d host threads\n", (unsigned long long)total_reads,
                (unsigned long long)chunks_done, shkhost::host_threads());
        fprintf(stderr, "[shark-b200/timing] batcher: waiting for the scanners %.0f ms, record arrays %.0f ms, offsets %.0f ms, packing %.0f ms, "
                        "exact path %.0f ms; writer: formatting %.0f ms, output %.0f ms\n",
                st.scan_wait * 1e3, st.flatten * 1e3, st.offsets * 1e3, st.pack * 1e3, st.exact * 1e3, st.format * 1e3, st.output * 1e3);
    }
    pelapsed("Sample completed");
    pelapsed("Association done");
    fflush(nullptr);
    if (one_process) {
        device_thread.join();
        if (getenv("SHK_CLEAN_EXIT")) {
            pool.clear();
            return 0;
        }
    }
    // the process ends here: its mappings and staging memory go with it; the device process tidies up by itself
    _exit(0);
}
