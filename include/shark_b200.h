/*
 * shark_b200.h - C ABI of the B200-native implementation of Shark's k-mer Bloom-filter
 * hot path (index build -> probe + rank -> per-read classification).
 *
 * The reference (AlgoLab/shark) has no plugin/FFI interface: its stages are C++ functors wired
 * together in main.cpp.  Each entry point below names the reference interface it replaces
 * (file:line relative to the reference tree).  Plain pointers and sizes only; no exceptions
 * cross this boundary.  Every function returns SHK_OK (0) or a negative shk_status;
 * shk_last_error() gives the message.  There is NO CPU fallback: without a CUDA device every
 * compute call fails with SHK_E_CUDA.
 *
 * Threading: a context belongs to one CUDA device.  Calls on the same context must be
 * serialised by the caller, except that slots are independent: one host thread may submit to
 * slot 0 while another collects slot 1.
 */
#ifndef SHARK_B200_H
#define SHARK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SHK_ABI_VERSION 5

typedef enum shk_status {
    SHK_OK = 0,
    SHK_E_ARG = -1,      /* invalid argument (k outside [1,31], c outside [0,1], ...)            */
    SHK_E_CUDA = -2,     /* CUDA runtime/driver failure, or no device                             */
    SHK_E_STATE = -3,    /* call out of order (e.g. reads submitted before the index exists)      */
    SHK_E_CAPACITY = -4, /* chunk larger than the slot capacity given at shk_create               */
    SHK_E_LIMIT = -5,    /* input exceeds a documented limit (e.g. > 65536 gene indices)          */
    SHK_E_NOMEM = -6
} shk_status;

typedef struct shk_ctx shk_ctx;

/* Options of one run = the reference's `opt::` globals (argument_parser.hpp:49-63). */
typedef struct shk_params {
    uint32_t k;                   /* -k, 1..31 (argument_parser.hpp:113-120)                       */
    double c;                     /* -c, [0,1]; used as `max >= c*len` in IEEE double
                                     (ReadAnalyzer.hpp:104)                                          */
    uint64_t bf_bits;             /* Bloom filter size in bits.  The CLI passes -b * 2^33
                                     (argument_parser.hpp:130-134); any value >= 64 is accepted    */
    int32_t min_quality;          /* -q as the reference stores it: low 8 bits = its `char`
                                     (argument_parser.hpp:144); 0 = no masking                     */
    int32_t single;               /* -s (ReadAnalyzer.hpp:104)                                     */
    int32_t device;               /* CUDA device ordinal                                           */
    uint32_t n_slots;             /* chunk slots for double buffering (0 -> 2)                     */
    uint32_t max_reads_per_chunk; /* slot capacity in reads   (0 -> 1<<20)                         */
    uint64_t max_bytes_per_chunk; /* slot capacity in sequence bytes (0 -> 320 * max_reads)        */
    uint32_t flags;               /* SHK_F_*; 0 = defaults                                         */
    uint32_t host_pack_permille;  /* with SHK_F_HOST_PACK: share of each chunk the host packs, in
                                     1/1000; 0 = balanced automatically against the link           */
    uint32_t reserved[6];         /* must be zero                                                  */
} shk_params;

/* shk_params.flags.  Anchor-and-extend (DESIGN.md 2.5, 3): results are identical on every path.  Default (neither flag):
 * the extension structures are built; packed reads (shk_reads_submit_packed, the packed part of a split upload) are
 * classified by the bulk kernel over them, text reads by the thread-per-read kernel - extending when the front table is
 * too large to stay in L2, window by window over a slots-only copy of it otherwise (shk_index_info.plain_front). */
#define SHK_F_EXTEND_ON 1u  /* build the structures; the thread-per-read kernel extends whatever the table size */
#define SHK_F_EXTEND_OFF 2u /* never build them: every read is classified window by window               */
/* Split upload: the plain path is PCIe-bound at 3-5 x below the kernels' rate, with the host cores idle.
 * With this flag shk_reads_submit sends the first part of a chunk as it is and, WHILE that copy runs,
 * reduces the rest to what the kernels use of a text byte - one validity bit (after the -q masking rule,
 * FastqSplitter.hpp:104-109) and a 2-bit code - on the host cores (AVX2, all pack threads, blocking); that
 * part crosses the link at 0.375 bytes per base instead of 1 (2 with qualities) and is classified by the
 * packed variant of the kernels (the chunk is split at a read boundary: text reads and packed reads).  The split point balances host and link (measured packing rate; host_pack_permille
 * fixes it).  Results are identical (the parity suite runs both ways). */
#define SHK_F_HOST_PACK 4u
/* Results stay in the compact form in which they cross the link (shk_chunk_result.gene16 / multi): assoc and
 * keep are NULL and shk_reads_collect does no per-read host work.  Without the flag shk_reads_collect expands
 * the compact form into assoc / keep on the calling thread (about 1 ms per million reads). */
#define SHK_F_COMPACT_RESULTS 8u
/* Lifts two limits of the reference (SURVEY.md 8f.4) - an opt-in extension, the default stays as the reference
 * is: gene ids are 32 bits wide instead of the 16 of small_vector_t::push_back(uint16_t) / vector<uint16_t>
 * (small_vector.hpp:46, bloomfilter.h:45), so that more than 65536 reference records can be indexed; and the
 * id total is bounded by the 32 bits of the list offsets instead of the reference's `int tot_idx`
 * (bloomfilter.h:130).  Without the flag such inputs fail with SHK_E_LIMIT.  With it the index keeps the
 * reference's structures (filter + rank, per-bit entries, CSR with uint32 ids; shk_index_export_wide) but not
 * the 16-bit accelerators built on top of them, every read is classified through the reference-shaped probe
 * (warp per read), results arrive through the `multi` list, and the staged functor protocol
 * (shk_bf_add_to_kmer) is not available. */
#define SHK_F_WIDE_IDS 16u
/* Keep a score record per read (shk_read_score, shk_reads_scores): the numbers behind each read's yes/no answer,
 * so that a caller can classify a sample once and apply any -c and -s afterwards (INTEGRATION.md 3).  16 bytes per
 * read more cross the link; without the flag nothing is written, allocated or copied. */
#define SHK_F_SCORES 32u
/* Count reads per gene on the device (shk_gene_counts): every chunk's reported associations are added into two 64-bit
 * counters per gene index that stay on the device, so that a caller gets the per-gene table of a whole sample without
 * walking gene16 / multi (INTEGRATION.md 3).  One more kernel launch per chunk; without the flag nothing is launched or
 * allocated. */
#define SHK_F_GENE_COUNTS 128u
/* Count reads per equivalence class on the device (shk_eq_classes): the set of genes a reported read is associated
 * with, and the number of reads with exactly that set, over a whole sample (INTEGRATION.md 3).  Needs
 * SHK_F_GENE_COUNTS (the singleton classes are its `unique` counters).  The insert pass runs inside K8; a device hash
 * table grows as classes appear.  Without the flag nothing is launched, allocated or copied. */
#define SHK_F_EQ_CLASSES 512u

/* Compact per-read result words (shk_chunk_result.gene16). */
#define SHK_GENE_NONE 0xFFFFu  /* no association: the read is not reported                                */
#define SHK_GENE_MULTI 0xFFFEu /* the read's associations are in shk_chunk_result.multi (two or more
                                  genes tie, or its single gene index is one of these two values)       */

typedef struct shk_index_info {
    uint32_t n_records;  /* FASTA records given (= legend_ID.size(), FastaSplitter.hpp:48)         */
    uint32_t n_genes;    /* final `nidx` (main.cpp:186): indices 0..n_genes-1 are in use           */
    uint64_t n_set_bits; /* num_kmer = rank(size) (bloomfilter.h:122)                              */
    uint64_t tot_ids;    /* tot_idx = total length of all gene-id lists (bloomfilter.h:130-133)    */
    uint64_t n_windows;  /* k-mer occurrences hashed in each pass                                  */
    uint64_t bf_bits;
    uint64_t device_bytes; /* HBM held by the index                                               */
    float build_ms;        /* device time of the whole build: CUDA-event segments that exclude the
                              host gaps between phases (allocations, read-backs of counts)         */
    uint32_t front_shift;  /* front table: log2(positions per bucket)                              */
    uint64_t front_entries; /* front table: entries (buckets + overflow records)                  */
    uint64_t ref_bases;    /* bases of the concatenated reference (extension structures)           */
    uint32_t extend;       /* 1 = the index carries the anchor-and-extend structures: front-table
                              entries are 32 bytes (slots + anchors), views 5-7 are present        */
    uint32_t coarse_shift; /* log2(filter positions per bit of the coarse miss filter)             */
    float build_wall_ms;   /* host clock around the same build, allocations included               */
    uint32_t n_shards;     /* 1 = built by shk_index_build; n = sharded build over n contexts;
                              0 = staged protocol / adopted                                         */
    uint32_t id_bits;      /* width of a gene id in the CSR: 16, or 32 with SHK_F_WIDE_IDS            */
    uint32_t plain_front;  /* 1 = the table is L2-sized and no flag forces a path: text reads are classified
                              over a derived slots-only copy of the front table (16-byte entries, stays in
                              L2), packed reads by the bulk kernel over the extension structures.  Set by
                              every context for itself when its index becomes ready (was `reserved`)    */
} shk_index_info;

/* One association = one line of the reference's stdout (ReadOutput.hpp:43): read `read_idx`
 * of the chunk goes with reference record `gene_idx`; the NAME to print is legend[gene_idx]
 * (ReadAnalyzer.hpp:106 - including the reference's index/name desync, SURVEY.md App. C Q1). */
typedef struct shk_assoc {
    uint32_t read_idx;
    uint32_t gene_idx;
} shk_assoc;

typedef struct shk_chunk_result {
    uint64_t n_assoc;       /* associations, ordered by read_idx then gene_idx                     */
    const shk_assoc *assoc; /* library-owned host memory, valid until the slot's next submit; NULL
                               with SHK_F_COMPACT_RESULTS                                           */
    const uint8_t *keep;    /* n_reads flags: 1 = read has >= 1 association (is written to the
                               filtered FASTQ, ReadOutput.hpp:44-47); NULL with SHK_F_COMPACT_RESULTS */
    uint32_t n_reads;
    uint32_t n_slow_reads;  /* reads that took the exact large-table path                          */
    uint64_t n_probes;      /* valid k-mer windows probed (counted on the device)                  */
    uint64_t n_hits;        /* probes that found a set bit                                         */
    float analyze_ms;       /* device time of the classification kernels (CUDA events)             */
    float total_ms;         /* device time H2D + kernels + D2H of counters                         */
    uint32_t kernel_launches;
    float probe_kernel_ms;  /* device time of the dominant kernel alone (analyze_reads_kernel)     */
    uint64_t n_extended;    /* probes resolved by anchor-and-extend, without a table access        */
    uint64_t n_table_loads; /* front-table entries the fast kernel loaded (extension mode only;
                               the rest of the probes were answered by the coarse miss filter)     */
    /* The compact form - what actually crosses the link (2 bytes per read + 8 per tied association instead
     * of 8 per association + 1 per read): what ReadOutput needs per read is "which gene, if any"
     * (ReadOutput.hpp:37-50), and all but a few percent of the kept reads have exactly one. */
    const uint16_t *gene16; /* n_reads words: gene index, SHK_GENE_NONE or SHK_GENE_MULTI; library-owned
                               pinned host memory, valid until the slot's next submit               */
    const shk_assoc *multi; /* the associations of the SHK_GENE_MULTI reads, ordered by read_idx then
                               gene_idx (same lifetime)                                             */
    uint64_t n_multi;
    uint64_t n_kept;        /* reads with >= 1 association                                         */
} shk_chunk_result;

/* Expands a compact result into the association list (n_assoc entries) and the keep flags (n_reads); either
 * output may be NULL.  Pure host function. */
int shk_result_expand(const shk_chunk_result *result, shk_assoc *assoc, uint8_t *keep);

/* The numbers behind one read's answer (SHK_F_SCORES).  A read is reported iff
 *     n_best > 0  &&  (double)cov >= c * len  &&  (!single || n_best == 1)
 * (c * len the IEEE double product, ReadAnalyzer.hpp:104), and a reported read has exactly n_best associations.
 * None of the four depends on c or -s: a run at c = 0 without -s, filtered by this rule, gives the run at any
 * (c, -s) association for association. */
typedef struct shk_read_score {
    uint32_t len;    /* valid bases after the -q masking: ReadAnalyzer's len (ReadAnalyzer.hpp:46-49)              */
    uint32_t cov;    /* coverage of the best gene (`max`, ReadAnalyzer.hpp:90-102); 0 if no gene was hit           */
    uint32_t hits;   /* k-mer hits of the best gene (`maxk`); 0 if no gene was hit                                 */
    uint32_t n_best; /* genes tied at (cov, hits), BEFORE the threshold and -s; 0 if no gene was hit              */
} shk_read_score;
/* After shk_reads_collect(slot): n_reads records, one per read of the chunk in read order, in library-owned pinned
 * memory, valid until the slot's next submit (same lifetime as gene16).  A read without a window of k valid bases
 * gets {len, 0, 0, 0}.  SHK_E_STATE for a context created without SHK_F_SCORES or before the slot is collected. */
int shk_reads_scores(shk_ctx *ctx, uint32_t slot, const shk_read_score **scores, uint32_t *n_reads);

/* Per-gene read counts (SHK_F_GENE_COUNTS), for every gene index g in [0, n_genes):
 *     unique[g]  reported reads whose only association is g (a single winner whose index is SHK_GENE_MULTI or
 *                SHK_GENE_NONE travels through `multi` but counts here)
 *     shared[g]  reported reads that have g among two or more tied associations
 * so that unique[g] + shared[g] = the associations {read, g} that shk_reads_collect returned, under the context's -c,
 * -s and -q.  Every chunk adds to the counters once, including chunks that shk_reads_collect had to run again, and
 * every shk_reads_analyze_resident adds again (the same resident chunk analysed n times counts n times).  The counters
 * are zeroed whenever an index becomes ready and by shk_gene_counts_reset, which with SHK_F_EQ_CLASSES also empties the
 * class table (its singletons are these counters).  n must equal shk_index_info.n_genes;
 * either pointer may be NULL.  SHK_E_STATE for a context created without the flag, without an index, or while a slot
 * has an uncollected chunk.  The read-back counts in shk_d2h_bytes. */
int shk_gene_counts(shk_ctx *ctx, uint64_t *unique, uint64_t *shared, uint32_t n);
int shk_gene_counts_reset(shk_ctx *ctx);

/* Reads per equivalence class (SHK_F_EQ_CLASSES).  A reported read's class is the set of its n_best associations in
 * ascending gene index order, under the context's -c, -s and -q; class i is ids[offsets[i], offsets[i+1]) and
 * counts[i] reads had exactly that set.  Classes come in lexicographic order of their id lists; singletons are
 * included ({g} counts unique[g] of shk_gene_counts), classes with no read are not.  So the classes containing g add up
 * to unique[g] + shared[g], and the counts to the n_kept of the chunks.  Accumulation and reset are those of
 * shk_gene_counts: every chunk adds once, every shk_reads_analyze_resident adds again, and the table is emptied
 * whenever an index becomes ready and by shk_gene_counts_reset.  Two calls: with NULL arrays only *n_classes and
 * *n_ids are set; then arrays of n_classes + 1, n_ids and n_classes entries (cap_classes >= n_classes, cap_ids >= n_ids,
 * SHK_E_CAPACITY otherwise, with the sizes set; ids and counts may be NULL when they would be empty).  SHK_E_STATE for a context created without the flag, without an index,
 * or while a slot has an uncollected chunk.  The read-back counts in shk_d2h_bytes. */
int shk_eq_classes(shk_ctx *ctx, uint64_t *n_classes, uint64_t *n_ids, uint64_t *offsets, uint32_t *ids, uint64_t *counts,
                   uint64_t cap_classes, uint64_t cap_ids);

/* ---- lifetime ------------------------------------------------------------------------ */

/* Replaces `parse_arguments` validation + `BF bloom(opt::bf_size)` (main.cpp:84,108;
 * bloomfilter.h:48-53).  Allocates the filter in HBM and the chunk slots. */
int shk_create(const shk_params *params, shk_ctx **out);
void shk_destroy(shk_ctx *ctx);
/* Message of the last failure on this context (ctx may be NULL: last failure of shk_create). */
const char *shk_last_error(const shk_ctx *ctx);
int shk_abi_version(void);

/* ---- index build ---------------------------------------------------------------------- */

/* Replaces pass 1 (FastaSplitter -> KmerBuilder::operator() KmerBuilder.hpp:40-72 ->
 * BloomfilterFiller::operator() BloomfilterFiller.hpp:38-46 -> BF::add_at bloomfilter.h:57-59),
 * BF::switch_mode(1) (bloomfilter.h:112-125), pass 2 (main.cpp:154-189 -> BF::add_to_kmer
 * bloomfilter.h:61-75) and BF::switch_mode(2) (bloomfilter.h:126-184).
 * ref_bases: the record sequences exactly as parsed (case and non-ACGT bytes preserved),
 * concatenated; rec_offsets[n_records+1] are byte offsets.  Host pointers.  The caller keeps
 * legend_ID (the record names). */
int shk_index_build(shk_ctx *ctx, const uint8_t *ref_bases, const uint64_t *rec_offsets, uint32_t n_records,
                    shk_index_info *info);
int shk_index_info_get(const shk_ctx *ctx, shk_index_info *info);

/* Downloads the index in the reference's logical form, for parity checks:
 * set_bit_pos[n_set_bits] ascending (the 1s of `_bf`), offsets[n_set_bits+1]
 * (offsets[r] = select(r)+1 over `_bv`, bloomfilter.h:142-148), ids[tot_ids] (`_index_kmer`).
 * Any pointer may be NULL. */
int shk_index_export(shk_ctx *ctx, uint64_t *set_bit_pos, uint32_t *offsets, uint16_t *ids);
/* The same with 32-bit ids: works for both id widths (ids of a 16-bit index are widened); shk_index_export
 * returns SHK_E_STATE for an index built with SHK_F_WIDE_IDS when ids != NULL. */
int shk_index_export_wide(shk_ctx *ctx, uint64_t *set_bit_pos, uint32_t *offsets, uint32_t *ids);

/* Replication across GPUs (one context per GPU, SURVEY.md 8e).  The arrays that define the
 * index are exposed as device buffers so that the host can move them with any transport
 * (ncclBroadcast over NVLink, cudaMemcpyPeer): call shk_index_views on the source context,
 * shk_index_adopt (allocates same-sized buffers) + shk_index_views on each destination, copy
 * every view, then shk_index_finalize on the destinations. */
#define SHK_INDEX_N_VIEWS 8
typedef struct shk_index_views {
    void *dev_ptr[SHK_INDEX_N_VIEWS]; /* 0 filter sectors, 1 per-bit entries, 2 CSR offsets, 3 CSR ids,
                                         4 front table; when info.extend: 5 reference stream (base +
                                         extension flags per position), 6 2-bit packed reference,
                                         7 coarse miss filter (bytes = 0 otherwise) */
    uint64_t bytes[SHK_INDEX_N_VIEWS];
    shk_index_info info;
} shk_index_views;
int shk_index_views_get(shk_ctx *ctx, shk_index_views *views);
int shk_index_adopt(shk_ctx *ctx, const shk_index_info *info);
int shk_index_finalize(shk_ctx *ctx);
/* Same replication for two contexts of ONE process (the multi-GPU CLI): adopt + peer copies over
 * NVLink (cudaMemcpyPeerAsync) + finalize. */
int shk_index_replicate(shk_ctx *src, shk_ctx *dst);

/* ---- sharded index build (SURVEY.md 8e second mode, 8f.3) ------------------------------- */
/* The north star's alternative to broadcasting a finished index: every context (= GPU) enumerates
 * the k-mers of ONE shard of the reference records into its own filter (pass 1 of the reference,
 * KmerBuilder.hpp:40-72 -> bloomfilter.h:57-59, over a subset of the genes); the filters are then
 * OR-merged with a P2P kernel over NVLink (NCCL has no bitwise-OR reduction): phase 1 reduces
 * slice i of every peer's filter into context i, phase 2 gathers the reduced slices.  Every
 * context then builds the same rank directory (bloomfilter.h:121-124), converts its own windows to
 * ranks, gathers the other shards' ranks and finishes pass 2 locally.  The result on every context
 * is bit-identical to shk_index_build (tests/test_gpu_shard.py).
 *
 * Protocol, with a barrier across all contexts wherever a line says so (every call returns with
 * its device work finished, so a host-side barrier is enough):
 *     shk_shard_begin                       each context; fills its shk_shard_mem
 *     (exchange the shk_shard_mem structs; other processes: shk_shard_open on each peer's)
 *     -- barrier --  shk_shard_merge(1)  -- barrier --  shk_shard_merge(2)  shk_shard_rank
 *     -- barrier --  shk_shard_finish    -- barrier --  shk_shard_close / shk_shard_end
 * `all` is an array of n_shards structs indexed by shard whose dev_ptr are usable from the
 * calling process (entry [own shard] is ignored). */
typedef struct shk_shard_mem {
    void *dev_ptr[3];           /* 0 filter sectors, 1 per-position window array, 2 per-record
                                   window flags; valid in the process named by pid                 */
    uint8_t ipc_handle[3][64];  /* cudaIpcMemHandle_t of each, for peers in other processes        */
    int64_t pid;                /* owning process; negative after shk_shard_open mapped it         */
    int32_t device;
    uint32_t shard;
    uint32_t ipc_ok;            /* 0: the handles could not be exported (same-process use only)    */
    uint32_t reserved;
} shk_shard_mem;
/* How the reference is cut: cuts[n_shards+1] positions at record boundaries, balanced by bases
 * (shard s enumerates the windows ending in [cuts[s], cuts[s+1])).  Pure host function. */
int shk_shard_cuts(const uint64_t *rec_offsets, uint32_t n_records, uint32_t n_shards, uint64_t *cuts);
int shk_shard_begin(shk_ctx *ctx, const uint8_t *ref_bases, const uint64_t *rec_offsets, uint32_t n_records,
                    uint32_t shard, uint32_t n_shards, shk_shard_mem *mine);
/* Makes a peer's buffers addressable from this context: peer access for a context of the same
 * process, cudaIpcOpenMemHandle for another process.  `opened` receives the usable struct. */
int shk_shard_open(shk_ctx *ctx, const shk_shard_mem *peer, shk_shard_mem *opened);
int shk_shard_close(shk_ctx *ctx, shk_shard_mem *opened);
int shk_shard_merge(shk_ctx *ctx, int phase, const shk_shard_mem *all);
int shk_shard_rank(shk_ctx *ctx);
int shk_shard_finish(shk_ctx *ctx, const shk_shard_mem *all, shk_index_info *info);
int shk_shard_end(shk_ctx *ctx);
/* The whole protocol for n contexts of ONE process (the multi-GPU CLI; also several contexts on one
 * device), one host thread per context, barriers between the steps.  info (may be NULL) receives
 * context 0's. */
int shk_index_build_sharded(shk_ctx **ctxs, uint32_t n, const uint8_t *ref_bases, const uint64_t *rec_offsets,
                            uint32_t n_records, shk_index_info *info);

/* ---- index serialisation (SURVEY.md 8f.3) ------------------------------------------------- */
/* The reference rebuilds its index on every run (main.cpp:128-193).  These two calls write the
 * finished device index to a file and load it into a context created with the same k and bf_bits:
 * header (magic, ABI version, k, shk_index_info, view sizes, FNV-1a checksum of the payload)
 * followed by the raw views of shk_index_views_get.  A load that does not match (k, bf_bits, ABI
 * version, checksum, truncated file) fails with SHK_E_ARG and leaves the context without an index. */
int shk_index_save(shk_ctx *ctx, const char *path);
int shk_index_load(shk_ctx *ctx, const char *path, shk_index_info *info);

/* ---- staged index build: the reference's own functor protocol ------------------------- */
/* The same index, built through the calls the reference's main.cpp makes (SURVEY.md 8b, seam 2),
 * so that KmerBuilder / BloomfilterFiller / class BF can be replaced one for one
 * (include/shark_b200_functors.hpp does exactly that).  A context starts in mode 0 with an empty
 * filter; shk_index_build above is the one-call equivalent of the whole protocol and may be used
 * instead, not in between. */

/* KmerBuilder::operator() (KmerBuilder.hpp:40-72): XXH64 (not reduced modulo the filter size) of
 * every canonical k-mer of the given records, records in order, windows in text order; k is
 * shk_params.k.  hashes[cap] is a host buffer; *n_hashes is always set to the number of windows;
 * SHK_E_CAPACITY when cap is too small (cap = total bases always suffices). */
int shk_kmer_hashes(shk_ctx *ctx, const uint8_t *bases, const uint64_t *rec_offsets, uint32_t n_records,
                    uint64_t *hashes, uint64_t cap, uint64_t *n_hashes);
/* BloomfilterFiller::operator() -> BF::add_at (BloomfilterFiller.hpp:38-46, bloomfilter.h:57-59):
 * `_bf[p % _size] = 1` for n positions (host pointer).  Mode 0 only (SHK_E_STATE otherwise; the
 * reference would silently corrupt its rank structure). */
int shk_bf_add_at(shk_ctx *ctx, const uint64_t *positions, uint64_t n);
/* BF::switch_mode (bloomfilter.h:112-184): 0 -> 1 builds the rank directory, 1 -> 2 flattens the
 * lists into the CSR (+ entries + front table) and makes the context ready for reads.  Any other
 * transition returns SHK_E_STATE (the reference returns false).  n_set_bits (may be NULL)
 * receives num_kmer (bloomfilter.h:122). */
int shk_bf_switch_mode(shk_ctx *ctx, int new_mode, uint64_t *n_set_bits);
/* BF::add_to_kmer (bloomfilter.h:61-75): hash % size of n canonical k-mers (host pointer), rank of
 * each position, gene id `input_idx` appended to that list unless it is already its last
 * element.  Mode 1 only.  input_idx must be in [0, 65535] (small_vector.hpp:46) and must not
 * decrease from call to call (the reference's pass 2 counts up, main.cpp:159-187), which makes
 * "append unless last" the same as "sorted unique". */
int shk_bf_add_to_kmer(shk_ctx *ctx, const uint64_t *kmers, uint64_t n, int32_t input_idx);
/* Current mode (0, 1, 2); 2 also after shk_index_build / shk_index_finalize. */
int shk_bf_mode(const shk_ctx *ctx);
/* ReadAnalyzer's constructor arguments (ReadAnalyzer.hpp:34-35) arrive after BF's: k, c, -s and
 * the masking threshold may be (re)set while no chunk is in flight.  k may only change before the
 * first window is hashed. */
int shk_set_options(shk_ctx *ctx, uint32_t k, double c, int32_t min_quality, int32_t single);

/* ---- probe (test / roofline entry) ---------------------------------------------------- */

/* Replaces BF::get_index (bloomfilter.h:78-102) for n canonical k-mers (host pointers):
 * rank[i] = 0-based index of the set bit or -1 for a miss; [begin, begin+len) is the id range
 * in `ids` as exported above (the reference's inclusive iterator pair, Q10). */
int shk_probe(shk_ctx *ctx, const uint64_t *canonical_kmers, uint64_t n, int64_t *rank, uint32_t *list_begin,
              uint32_t *list_len);

/* Probe throughput through the hot path's own access sequence (filter word -> sector/rank ->
 * entry): uploads n canonical k-mers once, runs the probe kernel reps times on the resident
 * array, reports the best kernel time (CUDA events) and the number of hits. */
int shk_probe_bench(shk_ctx *ctx, const uint64_t *canonical_kmers, uint64_t n, uint32_t reps, float *ms,
                    uint64_t *n_hits);

/* Measurement only (SURVEY.md 2.3 kernel B0): n_loads independent random 32-byte sector loads
 * over the first `span_bytes` of the filter allocation (0 = all of it). */
int shk_random_sector_bench(shk_ctx *ctx, uint64_t n_loads, uint64_t span_bytes, uint64_t seed, float *ms);

/* ---- pinned staging memory ------------------------------------------------------------ */
/* Page-locked host memory for chunk staging.  The pages are placed on the NUMA node of the calling
 * thread's CURRENT CUDA device (the device of the last shk_create / cudaSetDevice on that thread), so
 * that copies do not cross the socket interconnect; SHK_NUMA=0 turns the placement off. */
int shk_alloc_pinned(void **ptr, size_t bytes);
int shk_free_pinned(void *ptr);

/* ---- read classification -------------------------------------------------------------- */

/* Replaces FastqSplitter's masking rule (FastqSplitter.hpp:104-109), ReadAnalyzer::operator()
 * (ReadAnalyzer.hpp:39-110) and the ordering contract of ReadOutput (ReadOutput.hpp:40-49) for
 * one chunk of reads in SoA form:
 *   seq           concatenated read texts; a paired read is mate1 + 'N' + mate2
 *                 (FastqSplitter.hpp:63,83)
 *   qual          same layout (joiner byte 0x1B, FastqSplitter.hpp:84); may be NULL when
 *                 min_quality == 0 (the reference never looks at qualities then)
 *   read_offsets  n_reads+1 byte offsets into seq/qual
 * Host pointers (pinned memory makes the copies asynchronous); they must stay valid until the slot is
 * collected.  Asynchronous on the slot's stream: returns once the work is enqueued (with SHK_F_HOST_PACK the
 * packing of the chunk's second part happens inside this call, on the pack threads).  A slot must be
 * collected before it is submitted to again (SHK_E_STATE otherwise). */
int shk_reads_submit(shk_ctx *ctx, uint32_t slot, const uint8_t *seq, const uint8_t *qual,
                     const uint32_t *read_offsets, uint32_t n_reads);
/* The same chunk already reduced to what the kernels use of a text byte - 2-bit code and validity bit,
 * exactly what shk_host_pack produces from (seq, qual, min_quality) of the call above: codes[ceil(n/32)]
 * 64-bit words, valid[ceil(n/32)] 32-bit words, n = read_offsets[n_reads].  The -q masking rule
 * (FastqSplitter.hpp:104-109) is already in the validity bits, so qualities never cross the link; the
 * classification kernels read this form directly (0.375 bytes per base).  This is what the CLI's batcher
 * emits while it copies records. */
int shk_reads_submit_packed(shk_ctx *ctx, uint32_t slot, const uint64_t *codes, const uint32_t *valid,
                            const uint32_t *read_offsets, uint32_t n_reads);
/* Blocks until the slot's chunk is done and returns its result. */
int shk_reads_collect(shk_ctx *ctx, uint32_t slot, shk_chunk_result *result);

/* Same work split for kernel-only timing: upload copies the chunk to HBM and waits;
 * analyze_resident runs only the kernels on the resident chunk (repeatable). */
int shk_reads_upload(shk_ctx *ctx, uint32_t slot, const uint8_t *seq, const uint8_t *qual,
                     const uint32_t *read_offsets, uint32_t n_reads);
int shk_reads_upload_packed(shk_ctx *ctx, uint32_t slot, const uint64_t *codes, const uint32_t *valid,
                            const uint32_t *read_offsets, uint32_t n_reads);
int shk_reads_analyze_resident(shk_ctx *ctx, uint32_t slot);

/* Device-side stopwatch over ALL slots of a context (CUDA events, no host clock): start records
 * an event after everything enqueued so far; stop records one after everything enqueued since, on
 * every slot stream, waits for it and returns the elapsed device time.  bench.py times its steps
 * with this pair. */
int shk_device_timer_start(shk_ctx *ctx);
int shk_device_timer_stop(shk_ctx *ctx, float *ms);

/* The packing step of SHK_F_HOST_PACK as a pure host function (tests, tools): per text byte i, after
 * the masking rule when min_quality != 0 (`seq[i] -= 64` where `qual[i] < q+33`), valid bit i % 32 of
 * valid[i / 32] = byte is one of ACGTacgt, code at bits 2 (i % 32) of codes[i / 32] = (byte >> 1) & 3
 * (A 0, C 1, T 2, G 3; 0 when invalid).  Both arrays have ceil(n / 32) words.  parallel != 0 uses the
 * process-wide pack threads.  Needs no GPU. */
int shk_host_pack(const uint8_t *seq, const uint8_t *qual, int32_t min_quality, uint64_t n, uint64_t *codes,
                  uint32_t *valid, int32_t parallel);
/* "avx512", "avx2" or "scalar"; n_threads (may be NULL) receives the size of the pack pool. */
const char *shk_host_pack_info(int32_t *n_threads);

/* Switches the split upload (SHK_F_HOST_PACK, host_pack_permille) on or off while no chunk is in flight. */
int shk_set_upload_mode(shk_ctx *ctx, uint32_t host_pack, uint32_t permille);

/* Split upload diagnostics: the share of a chunk currently packed by the host (0 when off) and the last
 * measured packing rate in 10^9 bases per second.  Either pointer may be NULL. */
int shk_upload_stats(const shk_ctx *ctx, double *packed_share, double *pack_gbases_per_s);

/* Bytes that shk_reads_submit / shk_reads_upload copied host -> device on this context so far. */
uint64_t shk_h2d_bytes(const shk_ctx *ctx);
/* Result bytes (associations, keep flags, counters, score records, gene counts, class tables) copied device -> host on this context so far.  The
 * read-back of a chunk is enqueued with its kernels, sized by the previous chunks' associations per read;
 * shk_reads_collect fetches what that did not cover. */
uint64_t shk_d2h_bytes(const shk_ctx *ctx);

/* Kernel launches issued by this context so far (for bench accounting). */
uint64_t shk_kernel_launches(const shk_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* SHARK_B200_H */
