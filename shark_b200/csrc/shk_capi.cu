// C ABI of libshark_b200.so (include/shark_b200.h): contexts, slots, streams, copies.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <algorithm>
#include <string>
#include <thread>
#include <vector>

#include <sched.h>

#include "shk_hostpack.h"
#include "shk_internal.h"

namespace shk {

static std::mutex g_err_mu;
static char g_err[512] = {0};

void set_global_error(const char *msg)
{
    std::lock_guard<std::mutex> lk(g_err_mu);
    snprintf(g_err, sizeof g_err, "%s", msg);
}

int fail(shk_ctx *ctx, int code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) snprintf(ctx->err, sizeof ctx->err, "%s", buf);
    set_global_error(buf);
    return code;
}

static void free_slot(Slot &s)
{
    cudaFree(s.d_seq);
    cudaFree(s.d_qual);
    cudaFree(s.d_off);
    cudaFree(s.d_rec);
    cudaFree(s.d_pool);
    cudaFree(s.d_slow_list);
    cudaFree(s.d_slow2_list);
    cudaFree(s.d_tile_sums);
    cudaFree(s.d_tile_base);
    cudaFree(s.d_counters);
    cudaFree(s.d_gene16);
    cudaFree(s.d_multi);
    cudaFree(s.d_slow_table);
    cudaFree(s.d_slow_stamp);
    cudaFreeHost(s.h_counters);
    cudaFreeHost(s.h_gene16);
    cudaFreeHost(s.h_multi);
    free(s.h_assoc);
    free(s.h_keep);
    cudaFreeHost(s.h_pack);
    cudaFree(s.d_pack);
    cudaFree(s.d_scores);
    cudaFreeHost(s.h_scores);
    if (s.ev_start) cudaEventDestroy(s.ev_start);
    if (s.ev_k0) cudaEventDestroy(s.ev_k0);
    if (s.ev_ka) cudaEventDestroy(s.ev_ka);
    if (s.ev_k1) cudaEventDestroy(s.ev_k1);
    if (s.ev_done) cudaEventDestroy(s.ev_done);
    if (s.stream) cudaStreamDestroy(s.stream);
    s = Slot{};
}

// SHK_TIMING=1: stderr stamps of the start-up steps (diagnostics only)
static void tmark(const char *what)
{
    static const bool on = getenv("SHK_TIMING") != nullptr;
    static const auto t0 = std::chrono::steady_clock::now();
    if (on)
        fprintf(stderr, "[libshark_b200/timing] %-24s +%8.1f ms\n", what,
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
}


// Pinned staging memory should live on the NUMA node the GPU hangs off: a host-to-device copy that
// crosses the socket interconnect shares its bandwidth with every other GPU's copies (the 4-GPU
// bench loses ~13 % of its end-to-end rate to that).  While a pinned allocation is made for the
// CURRENT device, the calling thread is confined to that node's CPUs, so that the pages the driver
// faults in and pins are local (first touch); the previous affinity is restored afterwards.  No
// libnuma and no set_mempolicy (containers filter it); if sysfs does not describe the topology
// this is a no-op.  SHK_NUMA=0 disables it.
class NumaLocalScope {
public:
    NumaLocalScope()
    {
        static const bool enabled = !(getenv("SHK_NUMA") && atoi(getenv("SHK_NUMA")) == 0);
        int dev = 0;
        char bus[32] = {0};
        if (!enabled || cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetPCIBusId(bus, sizeof bus, dev) != cudaSuccess) {
            cudaGetLastError();
            return;
        }
        for (char *c = bus; *c; ++c)
            if (*c >= 'A' && *c <= 'F') *c = (char)(*c - 'A' + 'a');  // sysfs spells bus ids in lower case
        int node = -1;
        if (!read_int((std::string("/sys/bus/pci/devices/") + bus + "/numa_node").c_str(), node) || node < 0) return;
        cpu_set_t want;
        CPU_ZERO(&want);
        if (!read_cpulist(("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist").c_str(), want)) return;
        if (sched_getaffinity(0, sizeof saved_, &saved_) != 0) return;
        cpu_set_t both;
        CPU_AND(&both, &want, &saved_);  // never leave the cpuset the process was given
        if (CPU_COUNT(&both) == 0) return;
        active_ = sched_setaffinity(0, sizeof both, &both) == 0;
        node_ = node;
    }
    ~NumaLocalScope()
    {
        if (active_) sched_setaffinity(0, sizeof saved_, &saved_);
    }
    int node() const { return active_ ? node_ : -1; }

private:
    static bool read_int(const char *path, int &v)
    {
        FILE *f = fopen(path, "r");
        if (!f) return false;
        const bool ok = fscanf(f, "%d", &v) == 1;
        fclose(f);
        return ok;
    }
    static bool read_cpulist(const char *path, cpu_set_t &set)  // "0-31,64-95"
    {
        FILE *f = fopen(path, "r");
        if (!f) return false;
        char buf[4096];
        const bool got = fgets(buf, sizeof buf, f) != nullptr;
        fclose(f);
        if (!got) return false;
        int n = 0;
        for (char *p = buf; *p && *p != '\n';) {
            char *e;
            long a = strtol(p, &e, 10), b = a;
            if (e == p) break;
            if (*e == '-') {
                p = e + 1;
                b = strtol(p, &e, 10);
            }
            for (long c = a; c <= b && c < CPU_SETSIZE; ++c) CPU_SET((int)c, &set), ++n;
            p = *e == ',' ? e + 1 : e;
        }
        return n > 0;
    }
    cpu_set_t saved_;
    bool active_ = false;
    int node_ = -1;
};

static cudaError_t pinned_alloc(void **ptr, size_t bytes)
{
    NumaLocalScope numa;
    static const bool verbose = getenv("SHK_TIMING") != nullptr;
    if (verbose) fprintf(stderr, "[libshark_b200/numa] pinned %zu bytes on node %d\n", bytes, numa.node());
    return cudaMallocHost(ptr, bytes ? bytes : 1);
}

// The pack threads are created on first use and inherit the creating thread's affinity for good: create them
// while confined to the GPU's NUMA node, next to the pinned staging buffers they read and write.
static void start_pack_pool_numa_local()
{
    NumaLocalScope numa;
    (void)host_pack_threads();
}

static int alloc_slot(shk_ctx *ctx, Slot &s)
{
    const uint64_t R = ctx->max_reads, B = ctx->max_bytes;
    const uint64_t tiles = (R + kReadsPerTile - 1) / kReadsPerTile;
    SHK_CUDA(ctx, cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    SHK_CUDA(ctx, cudaEventCreate(&s.ev_start));
    SHK_CUDA(ctx, cudaEventCreate(&s.ev_k0));
    SHK_CUDA(ctx, cudaEventCreate(&s.ev_ka));
    SHK_CUDA(ctx, cudaEventCreate(&s.ev_k1));
    SHK_CUDA(ctx, cudaEventCreate(&s.ev_done));
    // d_seq / d_qual (text chunks) are allocated by the first text submit: a caller that only ever submits packed
    // chunks (the CLI) neither waits for them at start-up nor holds them
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_off, (R + 1) * 4));
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_rec, R * sizeof(uint2)));
    s.pool_cap = (uint32_t)std::max<uint64_t>(R / 2, 4096);
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_pool, (uint64_t)s.pool_cap * 4));
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_slow_list, R * 4));
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_slow2_list, R * 4));
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_tile_sums, (tiles + 1) * 4));
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_tile_base, (tiles + 1) * 4));
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_counters, sizeof(ChunkCounters)));
    s.multi_cap = R / 4 + 1024;
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_multi, s.multi_cap * sizeof(shk_assoc)));
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_gene16, (R + 64) * 2));
    SHK_CUDA(ctx, pinned_alloc((void **)&s.h_counters, sizeof(ChunkCounters)));
    s.h_multi_cap = s.multi_cap;
    SHK_CUDA(ctx, pinned_alloc((void **)&s.h_multi, s.h_multi_cap * sizeof(shk_assoc)));
    SHK_CUDA(ctx, pinned_alloc((void **)&s.h_gene16, (R + 64) * 2));
    if (ctx->scores) {
        SHK_CUDA(ctx, cudaMalloc((void **)&s.d_scores, R * sizeof(uint4)));
        SHK_CUDA(ctx, pinned_alloc((void **)&s.h_scores, R * sizeof(shk_read_score)));
    }
    // packed reads: + 2 groups so that the kernels' prefetch of the following group stays inside
    s.pack_groups_cap = (B + 31) / 32 + 2;
    SHK_CUDA(ctx, cudaMalloc((void **)&s.d_pack, s.pack_groups_cap * 12));
    SHK_CUDA(ctx, cudaMemset(s.d_pack, 0, s.pack_groups_cap * 12));
    if (ctx->host_pack) {
        start_pack_pool_numa_local();
        SHK_CUDA(ctx, pinned_alloc((void **)&s.h_pack, s.pack_groups_cap * 12));
    }
    return SHK_OK;
}

static ReadKernelArgs make_args(shk_ctx *ctx, Slot &s)
{
    ReadKernelArgs a{};
    a.seq = s.d_seq;
    a.qual = s.has_qual ? s.d_qual : nullptr;
    a.off = s.d_off;
    a.n_reads = s.n_reads;
    a.pcodes = s.d_pack;
    a.pvalid = reinterpret_cast<const uint32_t *>(s.d_pack + s.pack_groups_cap);
    a.pack_first = s.pack_first;
    a.pack_base = s.pack_base;
    a.sectors = ctx->index.sectors;
    a.entries = ctx->index.entries;
    a.csr_off = ctx->index.csr_off;
    a.csr_ids = ctx->index.csr_ids;
    a.csr_ids32 = ctx->index.csr_ids32;
    a.wide = ctx->index.csr_ids32 != nullptr || ctx->index.info.id_bits == 32;
    a.geom = ctx->index.geom;
    a.front = ctx->index.front;
    a.fgeom = ctx->index.fgeom;
    a.estream = ctx->index.estream;
    a.ref2 = ctx->index.ref2;
    a.coarse = ctx->index.coarse;
    a.refr = ctx->index.refr;
    a.front_plain = ctx->index.front_plain;
    a.ebits = ctx->index.ebits;
    a.ref_total = ctx->index.egeom.total;
    a.coarse_rel = ctx->index.egeom.enabled ? ctx->index.fgeom.shift - ctx->index.egeom.coarse_shift : 0;
    a.coarse_key_shift = kFrontKeyShift + ctx->index.egeom.coarse_shift;
    a.n_genes = ctx->index.info.n_genes;
    a.k = (int)ctx->params.k;
    a.c = ctx->params.c;
    // `const char mq = min_quality + 33` with min_quality a (signed) char: FastqSplitter.hpp:75
    a.mq = (int)(signed char)(unsigned char)((ctx->params.min_quality & 0xFF) + 33);
    a.single = ctx->params.single ? 1 : 0;
    a.pol_first = ctx->pol_first;
    a.pol_last = ctx->pol_last;
    a.rec = s.d_rec;
    a.pool = s.d_pool;
    a.pool_cap = s.pool_cap;
    a.slow_list = s.d_slow_list;
    a.slow2_list = s.d_slow2_list;
    a.tile_sums = s.d_tile_sums;
    a.counters = s.d_counters;
    a.slow_table = s.d_slow_table;
    a.slow_stamp = s.d_slow_stamp;
    a.n_slow_slabs = ctx->n_slow_slabs;
    a.tile_base = s.d_tile_base;
    a.gene16 = s.d_gene16;
    a.multi = s.d_multi;
    a.scores = s.d_scores;
    return a;
}

// The exact-path tables depend on the number of gene indices -> (re)allocated after a build,
// one set per slot because the slots' kernels run concurrently.
static int ensure_slow_table(shk_ctx *ctx)
{
    if (int rc = index_derive_bulk(ctx)) return rc;  // every path to a ready index ends here
    const uint64_t ng = std::max<uint32_t>(ctx->index.info.n_genes, 1);
    // as many concurrent exact-path warps as 128 MiB of tables allow, at most 4 per SM
    uint64_t slabs = std::min<uint64_t>((uint64_t)ctx->sm_count * 4, (128ull << 20) / (ng * sizeof(uint4)));
    slabs = std::max<uint64_t>(slabs, 8);
    ctx->n_slow_slabs = (uint32_t)slabs;
    for (uint32_t i = 0; i < ctx->n_slots; ++i) {
        Slot &s = ctx->slots[i];
        cudaFree(s.d_slow_table);
        cudaFree(s.d_slow_stamp);
        s.d_slow_table = nullptr;
        s.d_slow_stamp = nullptr;
        SHK_CUDA(ctx, cudaMalloc((void **)&s.d_slow_table, slabs * ng * sizeof(uint4)));
        SHK_CUDA(ctx, cudaMalloc((void **)&s.d_slow_stamp, slabs * 4));
        SHK_CUDA(ctx, cudaMemset(s.d_slow_table, 0, slabs * ng * sizeof(uint4)));
        SHK_CUDA(ctx, cudaMemset(s.d_slow_stamp, 0, slabs * 4));
    }
    return SHK_OK;
}

static int enqueue_chunk_kernels(shk_ctx *ctx, Slot &s)
{
    s.collected = false;
    SHK_CUDA(ctx, cudaMemsetAsync(s.d_counters, 0, sizeof(ChunkCounters), s.stream));
    ReadKernelArgs a = make_args(ctx, s);
    s.launches += (uint32_t)launch_read_kernels(ctx, a, s.multi_cap, s.stream, s.ev_k0, s.ev_ka, s.ev_k1);
    SHK_CUDA(ctx, cudaGetLastError());
    SHK_CUDA(ctx, cudaMemcpyAsync(s.h_counters, s.d_counters, sizeof(ChunkCounters), cudaMemcpyDeviceToHost, s.stream));
    // Results follow on the stream, before the host knows their size: the per-read words, and as many multi
    // entries as the previous chunks produced per read (+10 %); the rest - if any - is fetched by
    // shk_reads_collect.  This keeps the read-back off the collecting thread's critical path and lets it
    // overlap the other slots' kernels.
    const double per_read = ctx->multi_per_read.load();
    uint64_t pre = per_read < 0 ? s.n_reads / 8 : (uint64_t)(per_read * 1.10 * s.n_reads) + 1024;
    pre = std::min(pre, std::min(s.multi_cap, s.h_multi_cap));
    if (!s.n_reads) pre = 0;
    if (s.n_reads) SHK_CUDA(ctx, cudaMemcpyAsync(s.h_gene16, s.d_gene16, (size_t)s.n_reads * 2, cudaMemcpyDeviceToHost, s.stream));
    if (pre) SHK_CUDA(ctx, cudaMemcpyAsync(s.h_multi, s.d_multi, pre * sizeof(shk_assoc), cudaMemcpyDeviceToHost, s.stream));
    s.pre_multi = pre;
    ctx->d2h_bytes += pre * sizeof(shk_assoc) + (uint64_t)s.n_reads * 2 + sizeof(ChunkCounters);
    if (s.h_scores && s.n_reads) {
        SHK_CUDA(ctx, cudaMemcpyAsync(s.h_scores, s.d_scores, (size_t)s.n_reads * sizeof(shk_read_score), cudaMemcpyDeviceToHost,
                                      s.stream));
        ctx->d2h_bytes += (uint64_t)s.n_reads * sizeof(shk_read_score);
    }
    SHK_CUDA(ctx, cudaEventRecord(s.ev_done, s.stream));
    return SHK_OK;
}

static int check_chunk(shk_ctx *ctx, uint32_t slot, const uint32_t *off, uint32_t n_reads, const uint8_t *qual,
                       bool packed_input = false)
{
    if (!ctx) return SHK_E_ARG;
    if (slot >= ctx->n_slots) return fail(ctx, SHK_E_ARG, "slot %u out of range (n_slots=%u)", slot, ctx->n_slots);
    if (!ctx->index.built) return fail(ctx, SHK_E_STATE, "no index: call shk_index_build first");
    if (ctx->slots[slot].pending)
        return fail(ctx, SHK_E_STATE, "slot %u has an uncollected chunk: call shk_reads_collect first", slot);
    if (n_reads > ctx->max_reads)
        return fail(ctx, SHK_E_CAPACITY, "chunk of %u reads exceeds max_reads_per_chunk=%u", n_reads, ctx->max_reads);
    if (n_reads && !off) return fail(ctx, SHK_E_ARG, "read_offsets is NULL");
    if (n_reads && (uint64_t)off[n_reads] > ctx->max_bytes)
        return fail(ctx, SHK_E_CAPACITY, "chunk of %u bytes exceeds max_bytes_per_chunk=%llu", off[n_reads],
                    (unsigned long long)ctx->max_bytes);
    if (!packed_input && (ctx->params.min_quality & 0xFF) != 0 && !qual && n_reads)
        return fail(ctx, SHK_E_ARG, "min_quality != 0 needs the quality bytes");
    return SHK_OK;
}

// Split upload (SHK_F_HOST_PACK): share x of a chunk's n bases that the host packs.  Packing more relieves the
// link (0.375 bytes per base instead of b = 1, or 2 with qualities) and loads the submitting thread.  x balances
// the two per chunk:   host  x n / P + h0   =   link  ((1 - x) b + 0.375 x) n / B
// with P the packing rate (measured, smoothed), h0 the submitting thread's other work per chunk (measured:
// cycle time minus packing minus the time blocked on the device in shk_reads_collect), B the link rate
// (SHK_PCIE_GBS, default 53: what the plain path measures on a B200 host).  Measured (profiles/
// hostpack_r1_v13.md): the balance point is within a few percent of the best fixed share on C2, C3 and C4.
// shk_params.host_pack_permille fixes x instead.
static double now_secs()
{
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

static double pack_fraction(shk_ctx *ctx, bool has_qual, uint64_t n)
{
    if (ctx->params.host_pack_permille) return std::min(1.0, ctx->params.host_pack_permille / 1000.0);
    static const double B_max = [] {
        const char *ev = getenv("SHK_PCIE_GBS");
        const double v = ev ? atof(ev) : 0;
        return (v > 1 ? v : 53.0) * 1e9;
    }();
    PackControl &pc = ctx->pack;
    if (pc.link <= 0) pc.link = B_max;
    const double t = now_secs();
    if (pc.last_submit > 0) {
        const double cycle = t - pc.last_submit;
        const double h = cycle - pc.last_pack_secs - pc.blocked_secs;
        if (cycle < 1.0 && h >= 0) pc.h0 = 0.7 * pc.h0 + 0.3 * std::min(h, 5e-3);  // (a long pause is not a cycle)
        // The link rate is not a constant of the machine: GPUs behind one PCIe switch share an uplink, all ranks of
        // a host share its memory system (measured: 53 GB/s for one rank alone, 20 GB/s per rank with eight).  The
        // submitting thread sees which resource binds: blocked in shk_reads_collect for a good part of the cycle =
        // the device side (the link) is behind -> the link is slower than assumed, pack more; hardly ever blocked =
        // the host is behind -> assume a faster link, pack less.
        if (cycle < 1.0 && cycle > 0) {
            const double blocked = pc.blocked_secs / cycle;
            if (blocked > 0.25) pc.link = std::max(4e9, pc.link * 0.92);
            else if (blocked < 0.08) pc.link = std::min(B_max, pc.link * 1.04);
        }
    }
    pc.last_submit = t;
    pc.blocked_secs = 0;
    pc.last_pack_secs = 0;
    const double B = pc.link;
    const double b = has_qual ? 2.0 : 1.0;
    const double P = pc.rate > 0 ? pc.rate : 3e9 * host_pack_threads() / b;  // first chunk: a guess
    const double nn = (double)n;
    pc.x = std::min(1.0, std::max(0.05, (b * nn / B - pc.h0) / (nn / P + (b - 0.375) * nn / B)));
    return pc.x;
}

// Copies `groups` code words and validity words of a packed stream into the slot's device buffers.
static int enqueue_packed_copy(shk_ctx *ctx, Slot &s, const uint64_t *codes, const uint32_t *valid, uint64_t groups)
{
    if (!groups) return SHK_OK;
    SHK_CUDA(ctx, cudaMemcpyAsync(s.d_pack, codes, groups * 8, cudaMemcpyHostToDevice, s.stream));
    SHK_CUDA(ctx, cudaMemcpyAsync(reinterpret_cast<uint32_t *>(s.d_pack + s.pack_groups_cap), valid, groups * 4,
                                  cudaMemcpyHostToDevice, s.stream));
    ctx->h2d_bytes += groups * 12;
    return SHK_OK;
}

static int enqueue_upload(shk_ctx *ctx, Slot &s, const uint8_t *seq, const uint8_t *qual, const uint32_t *off,
                          uint32_t n_reads, bool allow_pack)
{
    s.n_reads = n_reads;
    s.collected = false;
    s.n_bytes = n_reads ? off[n_reads] : 0;
    s.has_qual = (ctx->params.min_quality & 0xFF) != 0;
    s.launches = 0;
    s.pack_first = 0xFFFFFFFFu;
    s.pack_base = 0;
    SHK_CUDA(ctx, cudaEventRecord(s.ev_start, s.stream));
    if (!n_reads) return SHK_OK;
    SHK_CUDA(ctx, cudaMemcpyAsync(s.d_off, off, ((uint64_t)n_reads + 1) * 4, cudaMemcpyHostToDevice, s.stream));
    ctx->h2d_bytes += ((uint64_t)n_reads + 1) * 4;
    uint32_t r_split = n_reads;  // reads [0, r_split) cross the link as text, the rest packed by the host
    if (allow_pack && ctx->host_pack && s.n_bytes) {
        // Split upload: the first reads of the chunk cross the link as they are (asynchronous copy from the
        // caller's buffer), the rest is packed to 3 bits per base by the host cores WHILE that copy runs and
        // classified by the packed variant of the kernels.  The split point balances the two resources (see
        // pack_fraction()) and sits at a read that starts a tile of kReadsPerTile reads.
        const double x = pack_fraction(ctx, s.has_qual, s.n_bytes);
        const uint64_t want = (uint64_t)((1.0 - x) * (double)s.n_bytes);
        r_split = (uint32_t)(std::upper_bound(off, off + n_reads + 1, (uint32_t)std::min<uint64_t>(want, 0xFFFFFFFFull)) - off);
        r_split = r_split ? r_split - 1 : 0;                 // last read starting at or before `want`
        r_split = r_split / kReadsPerTile * kReadsPerTile;
    }
    const uint64_t S = off[r_split];  // text bytes
    if (S && !s.d_seq) SHK_CUDA(ctx, cudaMalloc((void **)&s.d_seq, ctx->max_bytes + 64));
    if (S && s.has_qual && !s.d_qual) SHK_CUDA(ctx, cudaMalloc((void **)&s.d_qual, ctx->max_bytes + 64));
    if (S) {
        SHK_CUDA(ctx, cudaMemcpyAsync(s.d_seq, seq, S, cudaMemcpyHostToDevice, s.stream));
        if (s.has_qual) SHK_CUDA(ctx, cudaMemcpyAsync(s.d_qual, qual, S, cudaMemcpyHostToDevice, s.stream));
        ctx->h2d_bytes += S * (s.has_qual ? 2 : 1);
    }
    if (r_split == 0) s.has_qual = false;  // nothing is text: the packed part carries its masking
    if (r_split < n_reads) {
        const uint64_t n = s.n_bytes - S;
        const uint64_t groups = (n + 31) / 32;
        const int mq = (int)(signed char)(unsigned char)((ctx->params.min_quality & 0xFF) + 33);
        uint32_t *h_valid = reinterpret_cast<uint32_t *>(s.h_pack + s.pack_groups_cap);
        const double t0 = now_secs();
        host_pack_parallel(seq + S, qual && (ctx->params.min_quality & 0xFF) ? qual + S : nullptr, mq, n, s.h_pack, h_valid);
        const double secs = now_secs() - t0;
        ctx->pack.last_pack_secs = secs;
        if (secs > 0 && n >= (1u << 20))
            ctx->pack.rate = ctx->pack.rate > 0 ? 0.7 * ctx->pack.rate + 0.3 * (double)n / secs : (double)n / secs;
        s.pack_first = r_split;
        s.pack_base = (uint32_t)S;
        return enqueue_packed_copy(ctx, s, s.h_pack, h_valid, groups);
    }
    return SHK_OK;
}

// A chunk that arrives packed (shk_reads_submit_packed / shk_reads_upload_packed).
static int enqueue_upload_packed(shk_ctx *ctx, Slot &s, const uint64_t *codes, const uint32_t *valid, const uint32_t *off,
                                 uint32_t n_reads)
{
    s.n_reads = n_reads;
    s.collected = false;
    s.n_bytes = n_reads ? off[n_reads] : 0;
    s.has_qual = false;
    s.launches = 0;
    s.pack_first = 0;
    s.pack_base = 0;
    SHK_CUDA(ctx, cudaEventRecord(s.ev_start, s.stream));
    if (!n_reads) return SHK_OK;
    SHK_CUDA(ctx, cudaMemcpyAsync(s.d_off, off, ((uint64_t)n_reads + 1) * 4, cudaMemcpyHostToDevice, s.stream));
    ctx->h2d_bytes += ((uint64_t)n_reads + 1) * 4;
    return enqueue_packed_copy(ctx, s, codes, valid, (s.n_bytes + 31) / 32);
}

}  // namespace shk

using namespace shk;

static_assert(sizeof(shk_read_score) == sizeof(uint4), "the kernels store a score record as one uint4");
static_assert(sizeof(shk_index_info) == 96 && sizeof(shk_shard_mem) == 240 && sizeof(shk_chunk_result) == 112, "layouts mirrored in shark_b200/capi.py");

extern "C" {

int shk_abi_version(void) { return SHK_ABI_VERSION; }

const char *shk_last_error(const shk_ctx *ctx) { return ctx ? ctx->err : g_err; }

int shk_create(const shk_params *p, shk_ctx **out)
{
    if (!p || !out) return fail(nullptr, SHK_E_ARG, "NULL argument");
    *out = nullptr;
    if (p->k == 0 || p->k > 31) return fail(nullptr, SHK_E_ARG, "k must be in the range [1, 31]");
    if (!(p->c >= 0.0 && p->c <= 1.0)) return fail(nullptr, SHK_E_ARG, "c must be in the range [0, 1]");
    if (p->bf_bits < 64) return fail(nullptr, SHK_E_ARG, "bf_bits must be >= 64");
    if ((p->flags & SHK_F_EXTEND_ON) && (p->flags & SHK_F_EXTEND_OFF))
        return fail(nullptr, SHK_E_ARG, "SHK_F_EXTEND_ON and SHK_F_EXTEND_OFF are exclusive");
    if (p->flags & ~(SHK_F_EXTEND_ON | SHK_F_EXTEND_OFF | SHK_F_HOST_PACK | SHK_F_COMPACT_RESULTS | SHK_F_WIDE_IDS | SHK_F_SCORES))
        return fail(nullptr, SHK_E_ARG, "unknown flag bits");
    if ((p->flags & SHK_F_WIDE_IDS) && (p->flags & SHK_F_EXTEND_ON))
        return fail(nullptr, SHK_E_ARG, "SHK_F_WIDE_IDS has no extension structures (SHK_F_EXTEND_ON)");
    const uint64_t n_words = (p->bf_bits + 31) / 32;
    const uint64_t n_sectors = (n_words + kWordsPerSector - 1) / kWordsPerSector;
    if (n_sectors * 8 > 0xFFFFFFFFull)
        return fail(nullptr, SHK_E_LIMIT, "bf_bits=%llu: filters above ~2^36.8 bits (-b 14) are not supported",
                    (unsigned long long)p->bf_bits);
    tmark("shk_create enter");
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    tmark("device count");
    if (e != cudaSuccess || n_dev == 0)
        return fail(nullptr, SHK_E_CUDA, "no CUDA device (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    if (p->device < 0 || p->device >= n_dev) return fail(nullptr, SHK_E_ARG, "device %d out of range", p->device);
    shk_ctx *ctx = new (std::nothrow) shk_ctx;
    if (!ctx) return fail(nullptr, SHK_E_NOMEM, "out of host memory");
    ctx->params = *p;
    ctx->device = p->device;
    ctx->host_pack = (p->flags & SHK_F_HOST_PACK) != 0;
    ctx->compact_results = (p->flags & SHK_F_COMPACT_RESULTS) != 0;
    ctx->wide_ids = (p->flags & SHK_F_WIDE_IDS) != 0;
    ctx->scores = (p->flags & SHK_F_SCORES) != 0;
    if (const char *ev = getenv("SHK_HOST_PACK")) ctx->host_pack = atoi(ev) != 0;  // tuning override
    int rc = SHK_OK;
    auto bail = [&](int code) {
        shk_destroy(ctx);
        return code;
    };
    if (cudaSetDevice(ctx->device) != cudaSuccess) return bail(fail(nullptr, SHK_E_CUDA, "cudaSetDevice failed"));
    cudaFree(nullptr);
    tmark("primary context");
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, ctx->device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    FilterGeom &g = ctx->index.geom;
    g.bf_bits = p->bf_bits;
    g.n_sectors = n_sectors;
    if ((p->bf_bits & (p->bf_bits - 1)) == 0) {
        g.mod_kind = MOD_POW2;
        g.pow2_mask = p->bf_bits - 1;
    } else if ((p->bf_bits & ((1ULL << 33) - 1)) == 0 && (p->bf_bits >> 33) < (1ULL << 31)) {
        g.mod_kind = MOD_B33;
        g.b33 = (uint32_t)(p->bf_bits >> 33);
    } else {
        g.mod_kind = MOD_GENERIC;
    }
    ctx->n_slots = p->n_slots ? p->n_slots : 2;
    ctx->max_reads = p->max_reads_per_chunk ? p->max_reads_per_chunk : (1u << 20);
    ctx->max_bytes = p->max_bytes_per_chunk ? p->max_bytes_per_chunk : 320ull * ctx->max_reads;
    if (ctx->max_bytes >= (1ull << 32)) return bail(fail(nullptr, SHK_E_LIMIT, "max_bytes_per_chunk must be < 4 GiB"));
    if (cudaStreamCreateWithFlags(&ctx->build_stream, cudaStreamNonBlocking) != cudaSuccess)
        return bail(fail(nullptr, SHK_E_CUDA, "cudaStreamCreate failed"));
    rc = fetch_cache_policies(ctx);
    if (rc) {
        set_global_error(ctx->err);
        return bail(rc);
    }
    // BF bloom(opt::bf_size): the filter, zero-initialised (bloomfilter.h:48-53)
    e = cudaMalloc((void **)&ctx->index.sectors, n_sectors * 32);
    if (e != cudaSuccess)
        return bail(fail(nullptr, SHK_E_NOMEM, "cannot allocate %llu bytes for the filter: %s",
                         (unsigned long long)(n_sectors * 32), cudaGetErrorString(e)));
    cudaMemset(ctx->index.sectors, 0, n_sectors * 32);
    tmark("filter allocated");
    ctx->slots = new (std::nothrow) Slot[ctx->n_slots];
    if (!ctx->slots) return bail(fail(nullptr, SHK_E_NOMEM, "out of host memory"));
    for (uint32_t i = 0; i < ctx->n_slots; ++i) {
        rc = alloc_slot(ctx, ctx->slots[i]);
        if (rc) {
            set_global_error(ctx->err);
            return bail(rc);
        }
    }
    tmark("slots allocated");
    *out = ctx;
    return SHK_OK;
}

void shk_destroy(shk_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->slots) {
        for (uint32_t i = 0; i < ctx->n_slots; ++i) free_slot(ctx->slots[i]);
        delete[] ctx->slots;
    }
    staged_free(ctx);
    shard_free(ctx);
    cudaFree(ctx->index.sectors);
    cudaFree(ctx->index.entries);
    cudaFree(ctx->index.csr_off);
    cudaFree(ctx->index.csr_ids);
    cudaFree(ctx->index.csr_ids32);
    cudaFree(ctx->index.front);
    cudaFree(ctx->index.estream);
    cudaFree(ctx->index.ref2);
    cudaFree(ctx->index.coarse);
    cudaFree(ctx->index.refr);
    cudaFree(ctx->index.ebits);
    cudaFree(ctx->index.front_plain);
    if (ctx->build_stream) cudaStreamDestroy(ctx->build_stream);
    if (ctx->ev_t0) cudaEventDestroy(ctx->ev_t0);
    if (ctx->ev_t1) cudaEventDestroy(ctx->ev_t1);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->timer_stream) cudaStreamDestroy(ctx->timer_stream);
    delete ctx;
}

int shk_index_build(shk_ctx *ctx, const uint8_t *ref_bases, const uint64_t *rec_offsets, uint32_t n_records,
                    shk_index_info *info)
{
    if (!ctx || !rec_offsets) return fail(ctx, SHK_E_ARG, "NULL argument");
    if (rec_offsets[n_records] && !ref_bases) return fail(ctx, SHK_E_ARG, "ref_bases is NULL");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    staged_free(ctx);
    ctx->staged.mode = 0;
    int rc = index_build_device(ctx, ref_bases, rec_offsets, n_records);
    if (rc) return rc;
    ctx->staged.mode = 2;
    ctx->staged.hashed = true;
    rc = ensure_slow_table(ctx);
    if (rc) return rc;
    if (info) *info = ctx->index.info;
    return SHK_OK;
}

int shk_index_info_get(const shk_ctx *ctx, shk_index_info *info)
{
    if (!ctx || !info) return SHK_E_ARG;
    if (!ctx->index.built) return SHK_E_STATE;
    *info = ctx->index.info;
    return SHK_OK;
}

// ---- staged build: the reference's functor protocol (shk_index.cu, "Staged build") ----------
int shk_kmer_hashes(shk_ctx *ctx, const uint8_t *bases, const uint64_t *rec_offsets, uint32_t n_records, uint64_t *hashes,
                    uint64_t cap, uint64_t *n_hashes)
{
    if (!ctx || !rec_offsets || !n_hashes) return fail(ctx, SHK_E_ARG, "NULL argument");
    if (rec_offsets[n_records] && !bases) return fail(ctx, SHK_E_ARG, "bases is NULL");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    return kmer_hashes_device(ctx, bases, rec_offsets, n_records, hashes, cap, n_hashes);
}

int shk_bf_add_at(shk_ctx *ctx, const uint64_t *positions, uint64_t n)
{
    if (!ctx || (n && !positions)) return fail(ctx, SHK_E_ARG, "NULL argument");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    return staged_add_at(ctx, positions, n);
}

int shk_bf_switch_mode(shk_ctx *ctx, int new_mode, uint64_t *n_set_bits)
{
    if (!ctx) return fail(ctx, SHK_E_ARG, "NULL argument");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = staged_switch_mode(ctx, new_mode, n_set_bits);
    if (rc) return rc;
    return ctx->staged.mode == 2 ? ensure_slow_table(ctx) : SHK_OK;
}

int shk_bf_add_to_kmer(shk_ctx *ctx, const uint64_t *kmers, uint64_t n, int32_t input_idx)
{
    if (!ctx || (n && !kmers)) return fail(ctx, SHK_E_ARG, "NULL argument");
    if (ctx->wide_ids) return fail(ctx, SHK_E_STATE, "the staged protocol is the reference's (16-bit ids): not available with SHK_F_WIDE_IDS");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    return staged_add_to_kmer(ctx, kmers, n, input_idx);
}

int shk_bf_mode(const shk_ctx *ctx) { return ctx ? ctx->staged.mode : SHK_E_ARG; }

int shk_set_options(shk_ctx *ctx, uint32_t k, double c, int32_t min_quality, int32_t single)
{
    if (!ctx) return fail(ctx, SHK_E_ARG, "NULL argument");
    if (k == 0 || k > 31) return fail(ctx, SHK_E_ARG, "k must be in the range [1, 31]");
    if (!(c >= 0.0 && c <= 1.0)) return fail(ctx, SHK_E_ARG, "c must be in the range [0, 1]");
    if (k != ctx->params.k && ctx->staged.hashed)
        return fail(ctx, SHK_E_STATE, "k cannot change from %u to %u once k-mers have been hashed", ctx->params.k, k);
    for (uint32_t i = 0; i < ctx->n_slots; ++i)
        if (ctx->slots[i].pending) return fail(ctx, SHK_E_STATE, "a chunk is in flight on slot %u", i);
    ctx->params.k = k;
    ctx->params.c = c;
    ctx->params.min_quality = min_quality;
    ctx->params.single = single;
    return SHK_OK;
}

int shk_index_export(shk_ctx *ctx, uint64_t *set_bit_pos, uint32_t *offsets, uint16_t *ids)
{
    if (!ctx) return SHK_E_ARG;
    if (!ctx->index.built) return fail(ctx, SHK_E_STATE, "no index");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    return index_export_device(ctx, set_bit_pos, offsets, ids, nullptr);
}

int shk_index_export_wide(shk_ctx *ctx, uint64_t *set_bit_pos, uint32_t *offsets, uint32_t *ids)
{
    if (!ctx) return SHK_E_ARG;
    if (!ctx->index.built) return fail(ctx, SHK_E_STATE, "no index");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    return index_export_device(ctx, set_bit_pos, offsets, nullptr, ids);
}

int shk_index_views_get(shk_ctx *ctx, shk_index_views *v)
{
    if (!ctx || !v) return SHK_E_ARG;
    if (!ctx->index.built && !ctx->index.entries) return fail(ctx, SHK_E_STATE, "no index");
    const DeviceIndex &ix = ctx->index;
    v->dev_ptr[0] = ix.sectors;
    v->bytes[0] = ix.geom.n_sectors * 32;
    v->dev_ptr[1] = ix.entries;
    v->bytes[1] = (ix.info.n_set_bits + 1) * 8;
    v->dev_ptr[2] = ix.csr_off;
    v->bytes[2] = (ix.info.n_set_bits + 1) * 4;
    const bool wide = ix.info.id_bits == 32;
    v->dev_ptr[3] = wide ? (void *)ix.csr_ids32 : (void *)ix.csr_ids;
    v->bytes[3] = std::max<uint64_t>(ix.info.tot_ids, 1) * (wide ? 4 : 2);
    v->dev_ptr[4] = ix.front;
    v->bytes[4] = ix.fgeom.n_entries * 16 * ix.fgeom.stride;
    const bool ext = ix.egeom.enabled != 0;
    v->dev_ptr[5] = ext ? ix.estream : nullptr;
    v->bytes[5] = ext ? ix.egeom.estream_words * 8 : 0;
    v->dev_ptr[6] = ext ? ix.ref2 : nullptr;
    v->bytes[6] = ext ? ix.egeom.ref2_words * 8 : 0;
    v->dev_ptr[7] = ext ? ix.coarse : nullptr;
    v->bytes[7] = ext ? ix.egeom.coarse_words * 4 : 0;
    v->info = ix.info;
    return SHK_OK;
}

int shk_index_adopt(shk_ctx *ctx, const shk_index_info *info)
{
    if (!ctx || !info) return SHK_E_ARG;
    if (info->bf_bits != ctx->index.geom.bf_bits)
        return fail(ctx, SHK_E_ARG, "bf_bits mismatch between source index and this context");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    DeviceIndex &ix = ctx->index;
    if (info->id_bits != 16 && info->id_bits != 32) return fail(ctx, SHK_E_ARG, "index info: id_bits must be 16 or 32");
    if ((info->id_bits == 32) != ctx->wide_ids)
        return fail(ctx, SHK_E_ARG, "the index holds %u-bit gene ids, this context was created %s SHK_F_WIDE_IDS", info->id_bits,
                    ctx->wide_ids ? "with" : "without");
    cudaFree(ix.entries);
    cudaFree(ix.csr_off);
    cudaFree(ix.csr_ids);
    cudaFree(ix.csr_ids32);
    ix.entries = nullptr, ix.csr_off = nullptr, ix.csr_ids = nullptr, ix.csr_ids32 = nullptr;
    ix.built = false;
    ix.info = *info;
    SHK_CUDA(ctx, cudaMalloc((void **)&ix.entries, (info->n_set_bits + 1) * 8));
    SHK_CUDA(ctx, cudaMalloc((void **)&ix.csr_off, (info->n_set_bits + 1) * 4));
    if (info->id_bits == 32) SHK_CUDA(ctx, cudaMalloc((void **)&ix.csr_ids32, std::max<uint64_t>(info->tot_ids, 1) * 4));
    else SHK_CUDA(ctx, cudaMalloc((void **)&ix.csr_ids, std::max<uint64_t>(info->tot_ids, 1) * 2));
    return index_alloc_front(ctx);
}

int shk_index_finalize(shk_ctx *ctx)
{
    if (!ctx) return SHK_E_ARG;
    if (!ctx->index.entries) return fail(ctx, SHK_E_STATE, "shk_index_adopt was not called");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    SHK_CUDA(ctx, cudaDeviceSynchronize());
    ctx->index.built = true;
    ctx->staged.mode = 2;
    ctx->staged.hashed = true;
    return ensure_slow_table(ctx);
}

int shk_index_replicate(shk_ctx *src, shk_ctx *dst)
{
    if (!src || !dst || src == dst) return fail(dst, SHK_E_ARG, "bad contexts");
    if (!src->index.built) return fail(dst, SHK_E_STATE, "source context has no index");
    int rc = shk_index_adopt(dst, &src->index.info);
    if (rc) return rc;
    shk_index_views vs, vd;
    if ((rc = shk_index_views_get(src, &vs)) != 0) return rc;
    if ((rc = shk_index_views_get(dst, &vd)) != 0) return rc;
    SHK_CUDA(dst, cudaSetDevice(dst->device));
    int can = 0;
    if (src->device != dst->device && cudaDeviceCanAccessPeer(&can, dst->device, src->device) == cudaSuccess && can) {
        cudaError_t e = cudaDeviceEnablePeerAccess(src->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
        else cudaGetLastError();
    }
    for (int i = 0; i < SHK_INDEX_N_VIEWS; ++i) {
        if (!vs.bytes[i]) continue;
        if (vs.bytes[i] != vd.bytes[i]) return fail(dst, SHK_E_STATE, "index view %d size mismatch", i);
        SHK_CUDA(dst, cudaMemcpyPeerAsync(vd.dev_ptr[i], dst->device, vs.dev_ptr[i], src->device, vs.bytes[i],
                                          dst->build_stream));
    }
    SHK_CUDA(dst, cudaStreamSynchronize(dst->build_stream));
    return shk_index_finalize(dst);
}

// ---- sharded index build (shk_index.cu, "Sharded build") ---------------------------------------
static int shard_guard(shk_ctx *ctx)
{
    if (!ctx) return SHK_E_ARG;
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    return SHK_OK;
}

int shk_shard_cuts(const uint64_t *rec_offsets, uint32_t n_records, uint32_t n_shards, uint64_t *cuts)
{
    if (!rec_offsets || !cuts || n_shards == 0) return fail(nullptr, SHK_E_ARG, "bad argument");
    shard_cuts_host(rec_offsets, n_records, n_shards, cuts);
    return SHK_OK;
}

int shk_shard_begin(shk_ctx *ctx, const uint8_t *ref_bases, const uint64_t *rec_offsets, uint32_t n_records, uint32_t shard,
                    uint32_t n_shards, shk_shard_mem *mine)
{
    if (!ctx || !rec_offsets || !mine) return fail(ctx, SHK_E_ARG, "NULL argument");
    if (rec_offsets[n_records] && !ref_bases) return fail(ctx, SHK_E_ARG, "ref_bases is NULL");
    int rc = shard_guard(ctx);
    if (rc) return rc;
    staged_free(ctx);
    ctx->staged.mode = 0;
    return shard_begin(ctx, ref_bases, rec_offsets, n_records, shard, n_shards, mine);
}

int shk_shard_open(shk_ctx *ctx, const shk_shard_mem *peer, shk_shard_mem *opened)
{
    if (!ctx || !peer || !opened) return fail(ctx, SHK_E_ARG, "NULL argument");
    int rc = shard_guard(ctx);
    return rc ? rc : shard_open(ctx, peer, opened);
}

int shk_shard_close(shk_ctx *ctx, shk_shard_mem *opened)
{
    if (!ctx || !opened) return fail(ctx, SHK_E_ARG, "NULL argument");
    int rc = shard_guard(ctx);
    return rc ? rc : shard_close(ctx, opened);
}

int shk_shard_merge(shk_ctx *ctx, int phase, const shk_shard_mem *all)
{
    if (!ctx || !all || (phase != 1 && phase != 2)) return fail(ctx, SHK_E_ARG, "bad argument");
    int rc = shard_guard(ctx);
    return rc ? rc : shard_merge(ctx, phase, all);
}

int shk_shard_rank(shk_ctx *ctx)
{
    int rc = shard_guard(ctx);
    return rc ? rc : shard_rank(ctx);
}

int shk_shard_finish(shk_ctx *ctx, const shk_shard_mem *all, shk_index_info *info)
{
    if (!ctx || !all) return fail(ctx, SHK_E_ARG, "NULL argument");
    int rc = shard_guard(ctx);
    if (rc) return rc;
    if ((rc = shard_finish(ctx, all)) != 0) return rc;
    ctx->staged.mode = 2;
    ctx->staged.hashed = true;
    if ((rc = ensure_slow_table(ctx)) != 0) return rc;
    if (info) *info = ctx->index.info;
    return SHK_OK;
}

int shk_shard_end(shk_ctx *ctx)
{
    int rc = shard_guard(ctx);
    if (rc) return rc;
    shard_free(ctx);
    return SHK_OK;
}

int shk_index_build_sharded(shk_ctx **ctxs, uint32_t n, const uint8_t *ref_bases, const uint64_t *rec_offsets,
                            uint32_t n_records, shk_index_info *info)
{
    if (!ctxs || n == 0 || !ctxs[0]) return fail(nullptr, SHK_E_ARG, "no contexts");
    for (uint32_t i = 0; i < n; ++i)
        if (!ctxs[i]) return fail(ctxs[0], SHK_E_ARG, "context %u is NULL", i);
    std::vector<shk_shard_mem> mem(n);
    std::vector<std::vector<shk_shard_mem>> seen(n, std::vector<shk_shard_mem>(n));
    std::vector<int> rcs(n, 0);
    // one host thread per context per step; joining the threads is the barrier
    auto step = [&](auto &&fn) {
        std::vector<std::thread> th;
        for (uint32_t i = 0; i < n; ++i) {
            auto body = [&, i] {
                if (rcs[i] == 0) rcs[i] = fn(i);
            };
            try {
                th.emplace_back(body);
            } catch (...) {  // no thread to be had: run this context's step on the calling thread
                body();
            }
        }
        for (auto &t : th) t.join();
        for (uint32_t i = 0; i < n; ++i)
            if (rcs[i]) return rcs[i];
        return 0;
    };
    int rc = step([&](uint32_t i) { return shk_shard_begin(ctxs[i], ref_bases, rec_offsets, n_records, i, n, &mem[i]); });
    if (!rc)
        rc = step([&](uint32_t i) {
            for (uint32_t j = 0; j < n; ++j) {
                int r = shk_shard_open(ctxs[i], &mem[j], &seen[i][j]);
                if (r) return r;
            }
            return shk_shard_merge(ctxs[i], 1, seen[i].data());
        });
    if (!rc)
        rc = step([&](uint32_t i) {
            int r = shk_shard_merge(ctxs[i], 2, seen[i].data());
            return r ? r : shk_shard_rank(ctxs[i]);
        });
    if (!rc) rc = step([&](uint32_t i) { return shk_shard_finish(ctxs[i], seen[i].data(), nullptr); });
    for (uint32_t i = 0; i < n; ++i) shk_shard_end(ctxs[i]);
    if (rc) {
        for (uint32_t i = 0; i < n; ++i)
            if (rcs[i] && i != 0) snprintf(ctxs[0]->err, sizeof ctxs[0]->err, "context %u: %.480s", i, ctxs[i]->err);
        return rc;
    }
    if (info) *info = ctxs[0]->index.info;
    return SHK_OK;
}

// ---- index serialisation -------------------------------------------------------------------------
namespace {
struct IndexFileHeader {
    char magic[8];  // "SHKIDX\0\0"
    uint32_t abi, k;
    uint64_t bf_bits;
    uint64_t view_bytes[SHK_INDEX_N_VIEWS];
    uint64_t checksum;  // FNV-1a (64-bit words) over all view payloads in order
    shk_index_info info;
};
constexpr size_t kIoPiece = 64u << 20;

uint64_t fnv1a_words(uint64_t h, const uint8_t *p, size_t n)
{
    size_t i = 0;
    for (; i + 8 <= n; i += 8) {
        uint64_t w;
        memcpy(&w, p + i, 8);
        h = (h ^ w) * 0x100000001B3ull;
    }
    for (; i < n; ++i) h = (h ^ p[i]) * 0x100000001B3ull;
    return h;
}
}  // namespace

int shk_index_save(shk_ctx *ctx, const char *path)
{
    if (!ctx || !path) return fail(ctx, SHK_E_ARG, "NULL argument");
    if (!ctx->index.built) return fail(ctx, SHK_E_STATE, "no index to save");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    shk_index_views v;
    int rc = shk_index_views_get(ctx, &v);
    if (rc) return rc;
    IndexFileHeader h{};
    memcpy(h.magic, "SHKIDX\0\0", 8);
    h.abi = SHK_ABI_VERSION;
    h.k = ctx->params.k;
    h.bf_bits = ctx->index.geom.bf_bits;
    h.info = v.info;
    for (int i = 0; i < SHK_INDEX_N_VIEWS; ++i) h.view_bytes[i] = v.bytes[i];
    FILE *f = fopen(path, "wb");
    if (!f) return fail(ctx, SHK_E_ARG, "cannot open %s for writing", path);
    void *stage = nullptr;
    if (cudaMallocHost(&stage, kIoPiece) != cudaSuccess) {
        fclose(f);
        return fail(ctx, SHK_E_NOMEM, "cannot allocate the staging buffer");
    }
    bool ok = fwrite(&h, sizeof h, 1, f) == 1;
    uint64_t sum = 0xCBF29CE484222325ull;
    for (int i = 0; ok && i < SHK_INDEX_N_VIEWS; ++i)
        for (uint64_t a = 0; ok && a < v.bytes[i]; a += kIoPiece) {
            const size_t nb = (size_t)std::min<uint64_t>(kIoPiece, v.bytes[i] - a);
            ok = cudaMemcpy(stage, (const uint8_t *)v.dev_ptr[i] + a, nb, cudaMemcpyDeviceToHost) == cudaSuccess;
            if (ok) {
                sum = fnv1a_words(sum, (const uint8_t *)stage, nb);
                ok = fwrite(stage, 1, nb, f) == nb;
            }
        }
    h.checksum = sum;
    ok = ok && fseek(f, 0, SEEK_SET) == 0 && fwrite(&h, sizeof h, 1, f) == 1;
    ok = (fclose(f) == 0) && ok;
    cudaFreeHost(stage);
    cudaGetLastError();
    if (!ok) return fail(ctx, SHK_E_ARG, "writing %s failed", path);
    return SHK_OK;
}

int shk_index_load(shk_ctx *ctx, const char *path, shk_index_info *info)
{
    if (!ctx || !path) return fail(ctx, SHK_E_ARG, "NULL argument");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    FILE *f = fopen(path, "rb");
    if (!f) return fail(ctx, SHK_E_ARG, "cannot open %s", path);
    IndexFileHeader h{};
    auto bad = [&](const char *why) {
        fclose(f);
        ctx->index.built = false;
        return fail(ctx, SHK_E_ARG, "%s: %s", path, why);
    };
    if (fread(&h, sizeof h, 1, f) != 1 || memcmp(h.magic, "SHKIDX\0\0", 8) != 0) return bad("not a shark-b200 index file");
    if (h.abi != SHK_ABI_VERSION) return bad("written by another ABI version");
    if (h.k != ctx->params.k) return bad("built with another k");
    if (h.bf_bits != ctx->index.geom.bf_bits || h.info.bf_bits != h.bf_bits) return bad("built with another filter size");
    staged_free(ctx);
    int rc = shk_index_adopt(ctx, &h.info);
    if (rc) {
        fclose(f);
        return rc;
    }
    shk_index_views v;
    if ((rc = shk_index_views_get(ctx, &v)) != 0) {
        fclose(f);
        return rc;
    }
    for (int i = 0; i < SHK_INDEX_N_VIEWS; ++i)
        if (v.bytes[i] != h.view_bytes[i]) return bad("view sizes do not match the header");
    void *stage = nullptr;
    if (cudaMallocHost(&stage, kIoPiece) != cudaSuccess) {
        fclose(f);
        return fail(ctx, SHK_E_NOMEM, "cannot allocate the staging buffer");
    }
    bool ok = true;
    uint64_t sum = 0xCBF29CE484222325ull;
    for (int i = 0; ok && i < SHK_INDEX_N_VIEWS; ++i)
        for (uint64_t a = 0; ok && a < v.bytes[i]; a += kIoPiece) {
            const size_t nb = (size_t)std::min<uint64_t>(kIoPiece, v.bytes[i] - a);
            ok = fread(stage, 1, nb, f) == nb;
            if (ok) {
                sum = fnv1a_words(sum, (const uint8_t *)stage, nb);
                ok = cudaMemcpy((uint8_t *)v.dev_ptr[i] + a, stage, nb, cudaMemcpyHostToDevice) == cudaSuccess;
            }
        }
    cudaFreeHost(stage);
    cudaGetLastError();
    if (!ok) return bad("truncated file or copy failure");
    if (sum != h.checksum) return bad("checksum mismatch");
    fclose(f);
    if ((rc = shk_index_finalize(ctx)) != 0) return rc;
    if (info) *info = ctx->index.info;
    return SHK_OK;
}

int shk_probe(shk_ctx *ctx, const uint64_t *kmers, uint64_t n, int64_t *rank, uint32_t *begin, uint32_t *len)
{
    if (!ctx || (n && (!kmers || !rank || !begin || !len))) return fail(ctx, SHK_E_ARG, "NULL argument");
    if (!ctx->index.built) return fail(ctx, SHK_E_STATE, "no index");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    return probe_device(ctx, kmers, n, rank, begin, len);
}

int shk_probe_bench(shk_ctx *ctx, const uint64_t *kmers, uint64_t n, uint32_t reps, float *ms, uint64_t *n_hits)
{
    if (!ctx || !kmers || !n) return fail(ctx, SHK_E_ARG, "bad argument");
    if (!ctx->index.built) return fail(ctx, SHK_E_STATE, "no index");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    return probe_bench_device(ctx, kmers, n, reps ? reps : 3, ms, n_hits);
}

int shk_random_sector_bench(shk_ctx *ctx, uint64_t n_loads, uint64_t span_bytes, uint64_t seed, float *ms)
{
    if (!ctx || !n_loads) return fail(ctx, SHK_E_ARG, "bad argument");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    return random_sector_bench_device(ctx, n_loads, span_bytes, seed, ms);
}

int shk_alloc_pinned(void **ptr, size_t bytes)
{
    if (!ptr) return SHK_E_ARG;
    cudaError_t e = pinned_alloc(ptr, bytes);
    if (e != cudaSuccess) return fail(nullptr, SHK_E_NOMEM, "cudaMallocHost(%zu) failed: %s", bytes, cudaGetErrorString(e));
    return SHK_OK;
}

int shk_free_pinned(void *ptr)
{
    if (ptr) cudaFreeHost(ptr);
    return SHK_OK;
}

int shk_reads_submit(shk_ctx *ctx, uint32_t slot, const uint8_t *seq, const uint8_t *qual, const uint32_t *off,
                     uint32_t n_reads)
{
    int rc = check_chunk(ctx, slot, off, n_reads, qual);
    if (rc) return rc;
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    Slot &s = ctx->slots[slot];
    rc = enqueue_upload(ctx, s, seq, qual, off, n_reads, true);
    if (rc) return rc;
    rc = enqueue_chunk_kernels(ctx, s);
    if (rc) return rc;
    s.pending = true;
    return SHK_OK;
}

int shk_reads_submit_packed(shk_ctx *ctx, uint32_t slot, const uint64_t *codes, const uint32_t *valid, const uint32_t *off,
                            uint32_t n_reads)
{
    int rc = check_chunk(ctx, slot, off, n_reads, nullptr, true);
    if (rc) return rc;
    if (n_reads && off[n_reads] && (!codes || !valid)) return fail(ctx, SHK_E_ARG, "codes / valid is NULL");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    Slot &s = ctx->slots[slot];
    rc = enqueue_upload_packed(ctx, s, codes, valid, off, n_reads);
    if (rc) return rc;
    rc = enqueue_chunk_kernels(ctx, s);
    if (rc) return rc;
    s.pending = true;
    return SHK_OK;
}

int shk_reads_upload(shk_ctx *ctx, uint32_t slot, const uint8_t *seq, const uint8_t *qual, const uint32_t *off,
                     uint32_t n_reads)
{
    int rc = check_chunk(ctx, slot, off, n_reads, qual);
    if (rc) return rc;
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    Slot &s = ctx->slots[slot];
    rc = enqueue_upload(ctx, s, seq, qual, off, n_reads, false);  // kernel-only timing of the text form
    if (rc) return rc;
    SHK_CUDA(ctx, cudaStreamSynchronize(s.stream));
    s.pending = false;
    return SHK_OK;
}

int shk_reads_upload_packed(shk_ctx *ctx, uint32_t slot, const uint64_t *codes, const uint32_t *valid, const uint32_t *off,
                            uint32_t n_reads)
{
    int rc = check_chunk(ctx, slot, off, n_reads, nullptr, true);
    if (rc) return rc;
    if (n_reads && off[n_reads] && (!codes || !valid)) return fail(ctx, SHK_E_ARG, "codes / valid is NULL");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    Slot &s = ctx->slots[slot];
    rc = enqueue_upload_packed(ctx, s, codes, valid, off, n_reads);
    if (rc) return rc;
    SHK_CUDA(ctx, cudaStreamSynchronize(s.stream));
    s.pending = false;
    return SHK_OK;
}

int shk_reads_analyze_resident(shk_ctx *ctx, uint32_t slot)
{
    if (!ctx || slot >= ctx->n_slots) return fail(ctx, SHK_E_ARG, "bad slot");
    if (!ctx->index.built) return fail(ctx, SHK_E_STATE, "no index");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    Slot &s = ctx->slots[slot];
    if (s.pending) return fail(ctx, SHK_E_STATE, "slot %u has an uncollected chunk: call shk_reads_collect first", slot);
    s.launches = 0;
    SHK_CUDA(ctx, cudaEventRecord(s.ev_start, s.stream));
    int rc = enqueue_chunk_kernels(ctx, s);
    if (rc) return rc;
    s.pending = true;
    return SHK_OK;
}

int shk_result_expand(const shk_chunk_result *res, shk_assoc *assoc, uint8_t *keep)
{
    if (!res || (res->n_reads && !res->gene16) || (res->n_multi && !res->multi)) return fail(nullptr, SHK_E_ARG, "bad result");
    uint64_t o = 0, m = 0;
    for (uint32_t r = 0; r < res->n_reads; ++r) {
        const uint32_t g = res->gene16[r];
        if (keep) keep[r] = g != SHK_GENE_NONE;
        if (g == SHK_GENE_NONE) continue;
        if (g != SHK_GENE_MULTI) {
            if (assoc) assoc[o] = shk_assoc{r, g};
            ++o;
        } else {
            for (; m < res->n_multi && res->multi[m].read_idx == r; ++m, ++o)
                if (assoc) assoc[o] = res->multi[m];
        }
    }
    if (o != res->n_assoc || m != res->n_multi) return fail(nullptr, SHK_E_STATE, "inconsistent compact result");
    return SHK_OK;
}

int shk_reads_collect(shk_ctx *ctx, uint32_t slot, shk_chunk_result *out)
{
    if (!ctx || slot >= ctx->n_slots || !out) return fail(ctx, SHK_E_ARG, "bad argument");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    Slot &s = ctx->slots[slot];
    if (!s.pending) return fail(ctx, SHK_E_STATE, "slot %u has no submitted chunk", slot);
    for (int attempt = 0;; ++attempt) {
        const double t_block = ctx->host_pack ? now_secs() : 0;
        SHK_CUDA(ctx, cudaEventSynchronize(s.ev_done));
        if (ctx->host_pack) ctx->pack.blocked_secs += now_secs() - t_block;  // feeds pack_fraction()
        const ChunkCounters &c = *s.h_counters;
        if (c.pool_overflow) {
            // more tied winners than the pool holds: grow it and run the chunk again (exact)
            if (attempt > 8) return fail(ctx, SHK_E_NOMEM, "tie pool keeps overflowing");
            uint64_t want = std::max<uint64_t>((uint64_t)c.pool_used * 2, (uint64_t)s.pool_cap * 4);
            if (want > 0xFFFFFFF0ull) return fail(ctx, SHK_E_LIMIT, "tie pool would exceed 2^32 entries");
            cudaFree(s.d_pool);
            s.d_pool = nullptr;
            SHK_CUDA(ctx, cudaMalloc((void **)&s.d_pool, want * 4));
            s.pool_cap = (uint32_t)want;
            int rc = enqueue_chunk_kernels(ctx, s);
            if (rc) return rc;
            continue;
        }
        if (c.n_multi > s.multi_cap) {
            uint64_t want = c.n_multi + c.n_multi / 8 + 1024;
            cudaFree(s.d_multi);
            s.d_multi = nullptr;
            SHK_CUDA(ctx, cudaMalloc((void **)&s.d_multi, want * sizeof(shk_assoc)));
            s.multi_cap = want;
            ReadKernelArgs a = make_args(ctx, s);
            s.launches += (uint32_t)launch_scatter(ctx, a, s.multi_cap, s.stream);
            SHK_CUDA(ctx, cudaGetLastError());
            SHK_CUDA(ctx, cudaEventRecord(s.ev_done, s.stream));
            s.pre_multi = 0;  // the list was rebuilt in a new buffer: fetch all of it below
            continue;
        }
        break;
    }
    const ChunkCounters c = *s.h_counters;
    if (c.n_multi > s.h_multi_cap) {
        cudaFreeHost(s.h_multi);
        s.h_multi = nullptr;
        s.h_multi_cap = c.n_multi + c.n_multi / 8 + 1024;
        SHK_CUDA(ctx, pinned_alloc((void **)&s.h_multi, s.h_multi_cap * sizeof(shk_assoc)));
        s.pre_multi = 0;
    }
    if (c.n_multi > s.pre_multi) {  // what the read-back enqueued with the kernels did not cover
        SHK_CUDA(ctx, cudaMemcpyAsync(s.h_multi + s.pre_multi, s.d_multi + s.pre_multi,
                                      (c.n_multi - s.pre_multi) * sizeof(shk_assoc), cudaMemcpyDeviceToHost, s.stream));
        ctx->d2h_bytes += (c.n_multi - s.pre_multi) * sizeof(shk_assoc);
        SHK_CUDA(ctx, cudaStreamSynchronize(s.stream));
    }
    if (s.n_reads) ctx->multi_per_read.store((double)c.n_multi / (double)s.n_reads);
    float k_ms = 0, t_ms = 0, p_ms = 0;
    cudaEventElapsedTime(&k_ms, s.ev_k0, s.ev_k1);
    cudaEventElapsedTime(&p_ms, s.ev_k0, s.ev_ka);
    cudaEventElapsedTime(&t_ms, s.ev_start, s.ev_done);
    memset(out, 0, sizeof *out);
    out->n_assoc = c.n_assoc;
    out->gene16 = s.h_gene16;
    out->multi = s.h_multi;
    out->n_multi = c.n_multi;
    out->n_kept = c.n_kept;
    out->n_reads = s.n_reads;
    out->n_slow_reads = c.n_slow;
    out->n_probes = c.n_probes;
    out->n_hits = c.n_hits;
    out->analyze_ms = k_ms;
    out->probe_kernel_ms = p_ms;
    out->total_ms = t_ms;
    out->kernel_launches = s.launches;
    out->n_extended = c.n_extended;
    out->n_table_loads = c.n_table_loads;
    s.pending = false;
    s.collected = true;
    if (!ctx->compact_results) {
        // the classic form of the ABI: association list + keep flags, expanded here on the calling thread
        if (c.n_assoc > s.h_assoc_cap || !s.h_assoc) {
            free(s.h_assoc);
            s.h_assoc_cap = c.n_assoc + c.n_assoc / 8 + 1024;
            s.h_assoc = (shk_assoc *)malloc(s.h_assoc_cap * sizeof(shk_assoc));
            if (!s.h_assoc) return fail(ctx, SHK_E_NOMEM, "out of host memory");
        }
        if (!s.h_keep) {
            s.h_keep = (uint8_t *)malloc((size_t)ctx->max_reads + 64);
            if (!s.h_keep) return fail(ctx, SHK_E_NOMEM, "out of host memory");
        }
        if (shk_result_expand(out, s.h_assoc, s.h_keep) != SHK_OK)
            return fail(ctx, SHK_E_STATE, "inconsistent compact result on slot %u", slot);
        out->assoc = s.h_assoc;
        out->keep = s.h_keep;
    }
    return SHK_OK;
}

int shk_reads_scores(shk_ctx *ctx, uint32_t slot, const shk_read_score **scores, uint32_t *n_reads)
{
    if (!ctx || slot >= ctx->n_slots || !scores || !n_reads) return fail(ctx, SHK_E_ARG, "bad argument");
    if (!ctx->scores) return fail(ctx, SHK_E_STATE, "the context was created without SHK_F_SCORES");
    const Slot &s = ctx->slots[slot];
    if (!s.collected) return fail(ctx, SHK_E_STATE, "slot %u has no collected chunk", slot);
    *scores = s.h_scores;
    *n_reads = s.n_reads;
    return SHK_OK;
}

// second ? ev_t1 : ev_t0 <- a point after everything enqueued so far on every slot stream (and the
// build stream)
static int timer_mark(shk_ctx *ctx, bool second)
{
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!ctx->timer_stream) {
        SHK_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->timer_stream, cudaStreamNonBlocking));
        SHK_CUDA(ctx, cudaEventCreate(&ctx->ev_t0));
        SHK_CUDA(ctx, cudaEventCreate(&ctx->ev_t1));
        SHK_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming));
    }
    cudaEvent_t ev = second ? ctx->ev_t1 : ctx->ev_t0;
    for (uint32_t i = 0; i <= ctx->n_slots; ++i) {
        cudaStream_t st = i < ctx->n_slots ? ctx->slots[i].stream : ctx->build_stream;
        SHK_CUDA(ctx, cudaEventRecord(ctx->ev_join, st));
        SHK_CUDA(ctx, cudaStreamWaitEvent(ctx->timer_stream, ctx->ev_join, 0));
    }
    SHK_CUDA(ctx, cudaEventRecord(ev, ctx->timer_stream));
    return SHK_OK;
}

int shk_device_timer_start(shk_ctx *ctx)
{
    if (!ctx) return SHK_E_ARG;
    int rc = timer_mark(ctx, false);
    if (rc) return rc;
    // work enqueued from now on must not start before the mark
    for (uint32_t i = 0; i < ctx->n_slots; ++i) SHK_CUDA(ctx, cudaStreamWaitEvent(ctx->slots[i].stream, ctx->ev_t0, 0));
    return SHK_OK;
}

int shk_device_timer_stop(shk_ctx *ctx, float *ms)
{
    if (!ctx || !ms) return SHK_E_ARG;
    if (!ctx->ev_t0) return fail(ctx, SHK_E_STATE, "shk_device_timer_start was not called");
    int rc = timer_mark(ctx, true);
    if (rc) return rc;
    SHK_CUDA(ctx, cudaEventSynchronize(ctx->ev_t1));
    SHK_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev_t0, ctx->ev_t1));
    return SHK_OK;
}

uint64_t shk_h2d_bytes(const shk_ctx *ctx) { return ctx ? ctx->h2d_bytes.load() : 0; }
uint64_t shk_d2h_bytes(const shk_ctx *ctx) { return ctx ? ctx->d2h_bytes.load() : 0; }

int shk_upload_stats(const shk_ctx *ctx, double *packed_share, double *pack_gbases_per_s)
{
    if (!ctx) return SHK_E_ARG;
    if (packed_share)
        *packed_share = !ctx->host_pack ? 0.0
                        : ctx->params.host_pack_permille ? ctx->params.host_pack_permille / 1000.0 : ctx->pack.x;
    if (pack_gbases_per_s) *pack_gbases_per_s = ctx->pack.rate * 1e-9;
    return SHK_OK;
}

int shk_set_upload_mode(shk_ctx *ctx, uint32_t host_pack, uint32_t permille)
{
    if (!ctx || permille > 1000) return fail(ctx, SHK_E_ARG, "bad argument");
    SHK_CUDA(ctx, cudaSetDevice(ctx->device));
    for (uint32_t i = 0; i < ctx->n_slots; ++i)
        if (ctx->slots[i].pending) return fail(ctx, SHK_E_STATE, "slot %u has a chunk in flight", i);
    if (host_pack) start_pack_pool_numa_local();
    if (host_pack)
        for (uint32_t i = 0; i < ctx->n_slots; ++i) {
            Slot &s = ctx->slots[i];
            if (!s.h_pack) SHK_CUDA(ctx, pinned_alloc((void **)&s.h_pack, s.pack_groups_cap * 12));
        }
    ctx->host_pack = host_pack != 0;
    ctx->params.host_pack_permille = permille;
    ctx->pack = PackControl{};
    return SHK_OK;
}

int shk_host_pack(const uint8_t *seq, const uint8_t *qual, int32_t min_quality, uint64_t n, uint64_t *codes, uint32_t *valid,
                  int32_t parallel)
{
    if ((n && !seq) || !codes || !valid) return fail(nullptr, SHK_E_ARG, "NULL argument");
    const int mq = (int)(signed char)(unsigned char)((min_quality & 0xFF) + 33);
    const uint8_t *q = (min_quality & 0xFF) != 0 ? qual : nullptr;
    if ((min_quality & 0xFF) != 0 && !qual && n) return fail(nullptr, SHK_E_ARG, "min_quality != 0 needs the quality bytes");
    if (parallel) host_pack_parallel(seq, q, mq, n, codes, valid);
    else host_pack(seq, q, mq, n, codes, valid);
    return SHK_OK;
}

const char *shk_host_pack_info(int32_t *n_threads)
{
    if (n_threads) *n_threads = host_pack_threads();
    return host_pack_isa();
}

uint64_t shk_kernel_launches(const shk_ctx *ctx) { return ctx ? ctx->launches.load() : 0; }

}  // extern "C"
