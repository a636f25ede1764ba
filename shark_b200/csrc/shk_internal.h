// Host-side internals shared by the translation units of libshark_b200.so.
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>

#include "../../include/shark_b200.h"
#include "shk_device.cuh"

namespace shk {

// Device-resident index (the reference's class BF in mode 2, bloomfilter.h:36-203).
struct DeviceIndex {
    FilterGeom geom{};
    uint32_t *sectors = nullptr;  // n_sectors * 8 words (filter bits + in-sector rank)
    uint64_t *entries = nullptr;  // one per set bit
    uint32_t *csr_off = nullptr;  // n_set + 1
    uint16_t *csr_ids = nullptr;  // tot_ids
    uint32_t *csr_ids32 = nullptr;  // tot_ids, instead of csr_ids with SHK_F_WIDE_IDS
    uint4 *front = nullptr;       // front table, fgeom.n_entries x 16 bytes (x 32 with anchors)
    FrontGeom fgeom{};
    // anchor-and-extend structures (only when info.extend; layouts in shk_device.cuh)
    uint64_t *estream = nullptr;  // 4 bits per reference position: base code + two extension flags
    uint64_t *ref2 = nullptr;     // 2-bit packed reference, 32 bases per word (anchor verification)
    uint32_t *coarse = nullptr;   // coarse miss filter: one bit per 2^coarse_shift filter positions
    // derived from estream whenever an index becomes ready (index_derive_bulk): the inputs of the bulk
    // classification kernel (shk_bulk.cu).  Never serialised, broadcast or exported.
    uint64_t *refr = nullptr;     // reference in the layout of the packed reads (base t at bits 2*(t&31) of word
                                  // (t>>5)+kDerivedPad, codes A0 C1 T2 G3), zero words on both sides
    uint32_t *ebits = nullptr;    // E[t] (shk_device.cuh) at bit t&31 of word (t>>5)+kDerivedPad
    uint4 *front_plain = nullptr; // slots of every front-table entry without the anchors (16-byte stride): what the
                                  // text kernel probes when the table is L2-sized (info.plain_front)
    uint64_t derived_bytes = 0;   // bytes of refr + ebits + front_plain (part of info.device_bytes)
    ExtGeom egeom{};
    shk_index_info info{};
    bool built = false;
};

// Counters the classification kernels maintain per chunk (device, mirrored to pinned host).
struct ChunkCounters {
    unsigned long long n_probes;
    unsigned long long n_hits;
    unsigned long long n_assoc;
    unsigned int pool_used;   // entries of the tie pool in use
    unsigned int n_slow;      // reads queued for the exact large-table path
    unsigned int pool_overflow;
    unsigned int n_slow2;     // reads the middle path handed on to the exact path
    unsigned long long n_extended;    // windows resolved by extension (no table access)
    unsigned long long n_table_loads; // front-table entries loaded by the fast kernel (extension mode)
    unsigned long long n_multi;       // entries of the `multi` list (associations of reads marked kGeneMulti)
    unsigned long long n_kept;        // reads with at least one association
};

struct ReadKernelArgs {
    // inputs
    const uint8_t *seq;
    const uint8_t *qual;  // nullptr when min_quality == 0
    const uint32_t *off;
    uint32_t n_reads;
    // packed part of the chunk: reads [pack_first, n_reads) live in the packed stream (2-bit code + validity bit
    // per base, shk_hostpack.h), whose position 0 is text offset pack_base = off[pack_first]; reads before
    // pack_first are text.  pack_first is a multiple of kReadsPerTile (or >= n_reads: no packed part).
    const uint64_t *pcodes;
    const uint32_t *pvalid;
    uint32_t pack_first, pack_base;
    uint32_t r0, r1;  // reads [r0, r1) of one launch of the fast kernel (r0 a multiple of kReadsPerTile)
    // index
    const uint32_t *sectors;
    const uint64_t *entries;
    const uint32_t *csr_off;
    const uint16_t *csr_ids;
    const uint32_t *csr_ids32;  // SHK_F_WIDE_IDS: 32-bit ids, wide entries, no front table (wide != 0)
    uint32_t wide;
    FilterGeom geom;
    const uint4 *front;
    FrontGeom fgeom;
    const uint64_t *estream;
    const uint64_t *ref2;
    const uint32_t *coarse;
    const uint64_t *refr;       // bulk kernel: see DeviceIndex
    const uint4 *front_plain;   // non-null: thread-per-read kernels probe this table (16-byte entries), no extension
    const uint32_t *ebits;
    uint64_t ref_total;         // reference bases
    uint32_t coarse_rel;        // fgeom.shift - coarse_shift: coarse index = bucket << rel | offset >> coarse_shift
    uint32_t coarse_key_shift;  // kFrontKeyShift + coarse_shift (the offset sits in the key)
    uint32_t n_genes;
    // options
    int k;
    double c;
    int mq;  // (signed char)(min_quality + 33), FastqSplitter.hpp:75
    int single;
    // L2 cache-hint descriptors (createpolicy results, fetched once per context): as kernel
    // parameters they reach the loads through uniform registers without per-load moves
    uint64_t pol_first, pol_last;
    // outputs
    uint2 *rec;              // per read: x = association count, y = gene id (count==1) or pool offset
    uint32_t *pool;          // winners of reads with >= 2 associations, ascending gene id
    uint32_t pool_cap;
    uint32_t *slow_list;     // read indices the fast path gave up on (middle path input)
    uint32_t *slow2_list;    // read indices the middle path gave up on (exact path input)
    uint32_t *tile_sums;     // `multi` entries per tile of kReadsPerTile reads
    ChunkCounters *counters;
    // exact-path scratch
    uint4 *slow_table;       // n_slow_slabs * n_genes entries {stamp, cov, hits, last}
    uint32_t *slow_stamp;    // per slab
    uint32_t n_slow_slabs;
    // compaction outputs (compact result form, include/shark_b200.h)
    uint32_t *tile_base;
    uint16_t *gene16;        // per read: gene index, SHK_GENE_NONE or SHK_GENE_MULTI
    shk_assoc *multi;        // associations of the SHK_GENE_MULTI reads, ordered by read then gene
    // SHK_F_SCORES: per read {len, cov, hits, n_best} (shk_read_score), written by the kernel that settles the read;
    // nullptr without the flag (the kernels without scores never touch it)
    uint4 *scores;
};

constexpr uint32_t kReadsPerTile = 128;  // one CTA of the fast kernel: 128 threads = 128 reads
constexpr uint32_t kDerivedPad = 2;     // zero words in front of refr / ebits (a read may overhang the reference)
constexpr uint32_t kDerivedTail = 4;    // and behind
constexpr uint32_t kMaxFastLen = 1024;  // longer reads take the exact path (32 chunks x 32)

struct Slot {
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_start = nullptr, ev_k0 = nullptr, ev_ka = nullptr, ev_k1 = nullptr, ev_done = nullptr;
    // device
    uint8_t *d_seq = nullptr, *d_qual = nullptr;
    uint32_t *d_off = nullptr;
    uint2 *d_rec = nullptr;
    uint32_t *d_pool = nullptr;
    uint32_t pool_cap = 0;
    uint32_t *d_slow_list = nullptr, *d_slow2_list = nullptr;
    uint32_t *d_tile_sums = nullptr, *d_tile_base = nullptr;
    ChunkCounters *d_counters = nullptr;
    uint16_t *d_gene16 = nullptr;    // compact per-read results
    shk_assoc *d_multi = nullptr;    // associations of the SHK_GENE_MULTI reads
    uint64_t multi_cap = 0;
    uint4 *d_slow_table = nullptr;   // exact-path tables: private to the slot (slots run concurrently)
    uint32_t *d_slow_stamp = nullptr;
    // pinned host
    ChunkCounters *h_counters = nullptr;
    uint16_t *h_gene16 = nullptr;
    shk_assoc *h_multi = nullptr;
    uint64_t h_multi_cap = 0;
    uint64_t pre_multi = 0;  // multi entries whose read-back was enqueued with the kernels
    // ordinary host memory: the expanded form (without SHK_F_COMPACT_RESULTS), filled by shk_reads_collect
    shk_assoc *h_assoc = nullptr;
    uint64_t h_assoc_cap = 0;
    uint8_t *h_keep = nullptr;
    // packed reads: codes (8 bytes per 32 bases) then validity words (4 bytes); d_pack always exists,
    // h_pack is the pinned staging of the split upload (SHK_F_HOST_PACK)
    uint64_t *h_pack = nullptr, *d_pack = nullptr;
    uint64_t pack_groups_cap = 0;
    uint32_t pack_first = 0xFFFFFFFFu, pack_base = 0;  // this chunk: reads >= pack_first are packed
    // SHK_F_SCORES only: one record per read, read back with the other results
    uint4 *d_scores = nullptr;
    shk_read_score *h_scores = nullptr;
    // state
    uint32_t n_reads = 0;
    uint64_t n_bytes = 0;
    bool has_qual = false;
    bool pending = false;
    bool collected = false;  // the results of the slot's last chunk are on the host (shk_reads_scores)
    uint32_t launches = 0;
};

}  // namespace shk

namespace shk {
// Staged build = the reference's BF protocol (bloomfilter.h:57-75,112-184): mode 0 set bits,
// mode 1 attach gene ids, mode 2 query.  Mode 1 keeps (rank, gene) pairs on the device.
struct StagedBuild {
    int mode = 0;
    bool hashed = false;          // a window was hashed with params.k: k is frozen
    uint32_t n_set = 0;
    int32_t last_idx = -1;        // largest input_idx seen by add_to_kmer
    uint32_t *cnt = nullptr;      // occurrences per rank (n_set + 1)
    uint32_t *pair_rank = nullptr;
    uint16_t *pair_gene = nullptr;
    uint64_t n_pairs = 0, cap = 0;
};
}  // namespace shk

namespace shk {
struct ShardBuild;  // sharded build state (shk_index.cu)
// Split upload (SHK_F_HOST_PACK): measurements behind the share of a chunk that the host packs
// (pack_fraction() in shk_capi.cu).  One submitting thread per context.
struct PackControl {
    double x = 0;               // current share
    double rate = 0;            // packing rate, bases/s (smoothed)
    double h0 = 3e-4;           // submitting thread's other work per chunk, seconds (smoothed)
    double last_submit = 0;     // host clock of the previous packed submit
    double last_pack_secs = 0;  // packing time of that submit
    double blocked_secs = 0;    // time blocked on the device in shk_reads_collect since then
    double link = 0;            // current estimate of this context's share of the host-to-device link, bytes/s
};
}

struct shk_ctx {
    shk_params params{};
    shk::StagedBuild staged;
    shk::ShardBuild *shard = nullptr;
    int device = 0;
    int sm_count = 148;
    shk::DeviceIndex index;
    shk::Slot *slots = nullptr;
    uint32_t n_slots = 0;
    uint32_t max_reads = 0;
    uint64_t max_bytes = 0;
    uint32_t n_slow_slabs = 0;
    std::atomic<uint64_t> launches{0};
    cudaStream_t build_stream = nullptr;
    cudaStream_t timer_stream = nullptr;  // shk_device_timer_*: joins every slot stream
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr, ev_join = nullptr;
    uint64_t pol_first = 0, pol_last = 0;  // createpolicy evict_first / evict_last descriptors
    bool host_pack = false;                // shk_reads_submit packs the text on the host cores first
    std::atomic<uint64_t> h2d_bytes{0};    // bytes shk_reads_submit / upload copied to the device
    std::atomic<uint64_t> d2h_bytes{0};    // result bytes copied back
    std::atomic<double> multi_per_read{-1.0};  // last chunk's multi entries per read: sizes the early read-back
    bool compact_results = false;          // SHK_F_COMPACT_RESULTS
    bool wide_ids = false;                 // SHK_F_WIDE_IDS
    bool scores = false;                   // SHK_F_SCORES
    shk::PackControl pack;                 // split upload: feedback state of the packed share
    char err[512] = {0};
};

namespace shk {

void set_global_error(const char *msg);
int fail(shk_ctx *ctx, int code, const char *fmt, ...);

#define SHK_CUDA(ctx, call)                                                                              \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            return shk::fail(ctx, SHK_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                             __FILE__, __LINE__);                                                        \
    } while (0)

// shk_index.cu
int index_build_device(shk_ctx *ctx, const uint8_t *ref_bases, const uint64_t *rec_off, uint32_t n_records);
int index_alloc_front(shk_ctx *ctx);  // sizes fgeom from info and allocates the table
int index_derive_bulk(shk_ctx *ctx);  // refr / ebits from estream (no-op without the extension structures)
int index_export_device(shk_ctx *ctx, uint64_t *pos, uint32_t *off, uint16_t *ids, uint32_t *ids32);
int probe_device(shk_ctx *ctx, const uint64_t *kmers, uint64_t n, int64_t *rank, uint32_t *begin, uint32_t *len);
int probe_bench_device(shk_ctx *ctx, const uint64_t *kmers, uint64_t n, uint32_t reps, float *ms, uint64_t *hits);
int random_sector_bench_device(shk_ctx *ctx, uint64_t n_loads, uint64_t span_bytes, uint64_t seed, float *ms);
// staged build (the reference's functor protocol)
int kmer_hashes_device(shk_ctx *ctx, const uint8_t *bases, const uint64_t *rec_off, uint32_t n_rec, uint64_t *hashes,
                       uint64_t cap, uint64_t *n_hashes);
int staged_add_at(shk_ctx *ctx, const uint64_t *positions, uint64_t n);
int staged_switch_mode(shk_ctx *ctx, int new_mode, uint64_t *n_set_bits);
int staged_add_to_kmer(shk_ctx *ctx, const uint64_t *kmers, uint64_t n, int32_t input_idx);
void staged_free(shk_ctx *ctx);
// sharded build (SURVEY.md 8e second mode)
int shard_begin(shk_ctx *ctx, const uint8_t *ref_bases, const uint64_t *rec_off, uint32_t n_rec, uint32_t shard,
                uint32_t n_shards, shk_shard_mem *mine);
int shard_open(shk_ctx *ctx, const shk_shard_mem *peer, shk_shard_mem *opened);
int shard_close(shk_ctx *ctx, shk_shard_mem *opened);
int shard_merge(shk_ctx *ctx, int phase, const shk_shard_mem *all);
int shard_rank(shk_ctx *ctx);
int shard_finish(shk_ctx *ctx, const shk_shard_mem *all);
void shard_free(shk_ctx *ctx);
void shard_cuts_host(const uint64_t *rec_off, uint32_t n_rec, uint32_t n_shards, uint64_t *cuts);

// shk_reads.cu
// Enqueues the classification kernels of one chunk on `st`; returns the number of launches.
int launch_read_kernels(shk_ctx *ctx, const ReadKernelArgs &a, uint64_t assoc_cap, cudaStream_t st, cudaEvent_t ev_k0,
                        cudaEvent_t ev_ka, cudaEvent_t ev_k1);
int launch_scatter(shk_ctx *ctx, const ReadKernelArgs &a, uint64_t assoc_cap, cudaStream_t st);
// shk_bulk.cu: the bulk classification kernel for packed reads over the extension structures
bool bulk_enabled();
template <bool SCORES>
void launch_bulk_kernel(const ReadKernelArgs &a, cudaStream_t st, unsigned blocks);
int fetch_cache_policies(shk_ctx *ctx);

}  // namespace shk
