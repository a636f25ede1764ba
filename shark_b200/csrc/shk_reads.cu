// Read classification on the device: replaces FastqSplitter's masking rule, ReadAnalyzer::operator()
// and the ordering contract of ReadOutput.  Citations are reference file:line.
//
// Kernels of one chunk (all on the slot's stream):
//   analyze_reads_kernel   K6, one THREAD per read: mask, rolling canonical k-mers, front-table probe
//                          (one 16-byte load per k-mer), per-gene coverage/hits in a
//                          register-resident 4-gene table, argmax, threshold (packed reads over the
//                          extension structures take K6b analyze_bulk_kernel instead, shk_bulk.cu)
//   analyze_mid_kernel     K6m, one WARP per read the fast kernels give up on (more than 4 genes, a
//                          list longer than 4, or a text longer than 1024 bytes), per-gene state in a
//                          shared-memory table; with SHK_F_WIDE_IDS every read (all_reads_slow_kernel)
//   analyze_slow_kernel    K6x, exact warp-per-read path with a dense per-gene table for the reads
//                          K6m cannot hold (more than kMidMaxGenes genes)
//   scan_tile_sums_kernel  exclusive scan of the per-tile association counts
//   scatter_assoc_kernel   ordered (read_idx, gene_idx) list + keep flags
//   gene_counts_kernel     K8, SHK_F_GENE_COUNTS only: per-gene counts of the chunk's reported reads, added into the
//                          context's device counters; with EQ (SHK_F_EQ_CLASSES) it also inserts every tied read's
//                          winner list into the context's class table
//   eq_leftover_kernel     SHK_F_EQ_CLASSES: inserts the reads K8 left over, without a probe limit
//   eq_rehash_kernel       SHK_F_EQ_CLASSES: moves the class table into one twice the size
#include "shk_internal.h"
#include "shk_scan.cuh"
#include "shk_reads.cuh"

#include <algorithm>
#include <cstdlib>

namespace shk {

// Ids of a per-bit entry, for the warp-per-read kernels: list length and id number t (shk_device.cuh).
template <bool WIDE>
__device__ __forceinline__ uint32_t list_len(uint64_t e)
{
    return WIDE ? wide_entry_len(e) : entry_len(e);
}
template <bool WIDE>
__device__ __forceinline__ uint32_t list_id(const ReadKernelArgs &a, uint64_t e, uint32_t ln, uint32_t t)
{
    if (WIDE) return ln == 1 ? entry_lo(e) : a.csr_ids32[entry_lo(e) + t];
    if (t == 0) return entry_id0(e);
    return ln == 2 ? entry_lo(e) : (uint32_t)a.csr_ids[entry_lo(e) + t];
}

__device__ __forceinline__ uint64_t shfl64(uint64_t v, int src)
{
    uint32_t lo = __shfl_sync(kFull, (uint32_t)v, src);
    uint32_t hi = __shfl_sync(kFull, (uint32_t)(v >> 32), src);
    return ((uint64_t)hi << 32) | lo;
}

// One 32-position chunk of a read text: load, mask (FastqSplitter.hpp:104-109), validity and
// 2-bit codes (kmer_utils.hpp:29-41), pack to 64 bits, and for the lane's window
// [pos-k+1, pos] the hashed filter position.  Returns the lane's window validity.
struct ChunkState {
    uint64_t prevP;  // packed codes of the previous chunk (base i at bits 63-2i..62-2i)
    uint32_t prevV;  // validity mask of the previous chunk
};

template <bool HAS_QUAL, int MOD>
__device__ __forceinline__ bool chunk_window(const ReadKernelArgs &a, uint32_t off0, uint32_t n, int chunk, int lane,
                                             ChunkState &cs, uint32_t &len, uint32_t &pw, uint32_t &bit, bool packed)
{
    const uint32_t pos = (uint32_t)chunk * 32u + (uint32_t)lane;
    bool valid = false;
    uint32_t code = 0;
    if (packed) {  // warp-uniform: the read lives in the packed stream (masking already folded into the validity bits)
        if (pos < n) {
            const uint32_t ap = off0 - a.pack_base + pos;
            const uint32_t raw = (uint32_t)(a.pcodes[ap >> 5] >> (2u * (ap & 31u))) & 3u;  // A0 C1 T2 G3
            valid = (a.pvalid[ap >> 5] >> (ap & 31u)) & 1u;
            code = raw ^ (raw >> 1);
        }
    } else {
        uint32_t ch = 0;
        if (pos < n) {
            ch = a.seq[off0 + pos];
            if (HAS_QUAL) {
                int q = (int)(signed char)a.qual[off0 + pos];
                if (q < a.mq) ch = (ch - 64u) & 0xFFu;  // seq[i] = seq[i] - 64
            }
        }
        valid = base_valid(ch);
        code = base_code(ch);
    }
    const uint32_t V = __ballot_sync(kFull, valid);
    len += __popc(V);  // ReadAnalyzer.hpp:46-49
    const uint32_t val = valid ? code << (30 - 2 * (lane & 15)) : 0u;
    const uint32_t hiw = __reduce_or_sync(kFull, lane < 16 ? val : 0u);
    const uint32_t low = __reduce_or_sync(kFull, lane >= 16 ? val : 0u);
    const uint64_t P = ((uint64_t)hiw << 32) | low;
    // window validity: bits [32+lane-k+1, 32+lane] of (prevV : V)
    const int k = a.k;
    const uint64_t VV = (uint64_t)cs.prevV | ((uint64_t)V << 32);
    const uint32_t kbits = (1u << k) - 1u;  // k <= 31
    const bool wv = (((uint32_t)(VV >> (33 + lane - k))) & kbits) == kbits;
    // forward k-mer: low 2k bits of (prevP : P) >> 2*(31-lane)
    const int s = 2 * (31 - lane);
    uint64_t fwd = P >> s;
    if (s) fwd |= cs.prevP << (64 - s);
    fwd &= (1ULL << (2 * k)) - 1ULL;
    pw = 0;
    bit = 0;
    if (wv) {
        uint64_t p = bit_index<MOD>(xxh64_u64(canonical(fwd, k)), a.geom);
        pw = (uint32_t)phys_word(p);
        bit = (uint32_t)(p & 31);
    }
    cs.prevP = P;
    cs.prevV = V;
    return wv;
}

// Reserves room in the tie pool for the `count` winners of a read with >= 2 associations.
// Returns the pool offset (warp-uniform); sets the overflow flag when the pool is exhausted.
__device__ __forceinline__ uint32_t pool_reserve(const ReadKernelArgs &a, uint32_t count, int lane)
{
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(&a.counters->pool_used, count);
    base = __shfl_sync(kFull, base, 0);
    if ((uint64_t)base + count > a.pool_cap) {
        if (lane == 0) a.counters->pool_overflow = 1;
        return 0xFFFFFFFFu;
    }
    return base;
}

// ---------------------------------------------------------------------------------------------
// Fast path: ONE THREAD PER READ.  The thread walks its read exactly like the reference does
// (ReadAnalyzer.hpp:50-87): rolling forward / reverse-complement k-mers (kmer_utils.hpp:73-79), a
// run counter for "k valid bytes in a row" (== build_kmer's restart after a non-ACGT byte,
// kmer_utils.hpp:57-71), one front-table probe per window, and the reference's own sequential
// per-gene update `cov += min(k, pos - last); hits += 1; last = pos` in a 4-gene register table.
// Four consecutive positions (one 32-bit word of text) are processed together so that four
// probes are in flight per thread.  Reads that need more than 4 genes, or are longer than
// kMaxFastLen, go to the exact warp-per-read path.
// ---------------------------------------------------------------------------------------------
constexpr int kFastThreads = 128;
#ifndef SHK_FAST_MIN_BLOCKS
#define SHK_FAST_MIN_BLOCKS 5
#endif
static_assert(kFastThreads == (int)kReadsPerTile, "one CTA of the fast kernel = one scan tile");

// ---------------------------------------------------------------------------------------------
// Fast path, version 4: still one thread per read, restructured around instruction issue (the v3
// profile: 55 % issue-active, 23 of 32 lanes active, 212 instructions per base):
//   * the four bytes of a text word are masked, validated and 2-bit coded together with
//     byte-parallel integer tricks (no per-byte table, no per-byte branches);
//   * rolling, hashing and bucket addressing are unconditional, so the compiler interleaves the
//     four independent XXH64 chains of a word; only the table load is predicated;
//   * the per-gene table keeps its most recent genes in slots 0/1 (a read covers one gene for
//     long stretches): the common update is three predicated integer ops, the shuffle that
//     brings another gene to the front is rare.
// Semantics are those of v3 (ReadAnalyzer.hpp:39-104), reads it cannot hold go to the exact path.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kH4 = 0x80808080u;

// per byte: (signed char)q < mq  ->  0x40 in that byte.  mq4b = (mq replicated) ^ 0x80808080.
__device__ __forceinline__ uint32_t qual_mask4(uint32_t qw, uint32_t mq4b)
{
    const uint32_t a = qw ^ kH4;  // bias to unsigned
    const uint32_t t = (a | kH4) - (mq4b & ~kH4);
    const uint32_t lt = ((~a & mq4b) | (~(a ^ mq4b) & ~t)) & kH4;
    return lt >> 1;
}
// per byte x - m (mod 256) for m < 128: `seq[i] = seq[i] - 64` (FastqSplitter.hpp:106)
__device__ __forceinline__ uint32_t sub_bytes4(uint32_t x, uint32_t m)
{
    const uint32_t t = (x | kH4) - m;
    return (t & ~kH4) | (~(x ^ t) & kH4);
}
// Four bytes -> 2-bit codes (byte b of code4, A0 C1 G2 T3) and a validity word (byte b of x is 0
// iff the byte is one of ACGTacgt): to_int, kmer_utils.hpp:29-41.
__device__ __forceinline__ void codes4(uint32_t w, uint32_t &code4, uint32_t &x)
{
    const uint32_t u = w & 0xDFDFDFDFu;            // fold case
    const uint32_t c4 = (u >> 1) & 0x03030303u;    // A0 C1 T2 G3
    const uint32_t s = c4 | (c4 >> 4);
    const uint32_t sel = __byte_perm(s, 0u, 0x4420u);
    x = u ^ __byte_perm(0x47544341u, 0u, sel);     // the letter each code stands for: "ACTG"
    code4 = c4 ^ ((c4 >> 1) & 0x01010101u);
}


// ---------------------------------------------------------------------------------------------
// Fast path, version 5 = version 4 with a branch-free common case for the table update.  The v4
// profile (profiles/analyze_r1_v4.md) showed 212 instructions per base, of which ~90 are the
// hashing half, and 22 of 32 lanes active: most warps contain a read from a region shared by two
// genes, so the "more than one id" branch ran for nearly every position with one or two lanes.
// Here a min/max network over `slot ^ key` yields the position's smallest two ids A <= B (a
// non-matching slot gives a value >= kFrontLim, a flagged slot a value >= 2^16, so `A == g0`
// alone proves "matching slot, plain id, gene g0"); positions whose ids are all in table slots
// 0/1 - the two most recent genes - are applied with predicated arithmetic.  Everything else (a
// gene entering the table, lists of 3-4 ids, long lists, chained buckets) takes the generic
// path, which for a typical read runs once or twice.
// ---------------------------------------------------------------------------------------------
//
// EXT = anchor-and-extend (layouts and the exactness argument: shk_device.cuh).  Used when the front
// table is DRAM-sized: then the kernel is bound by one random DRAM sector per probe, and most probes
// can be answered without any table access.  A thread that has verified that its current window IS
// the reference window ending at e ("anchored") resolves the next window from one nibble of the
// reference stream: next base equal (complementary on the reverse strand) and the "same gene list as
// the neighbouring reference window" flag set => the window's ids are the previous window's ids.
// Windows that cannot be extended first ask the L2-resident coarse filter whether anything is set near
// their filter position, and only then load their front-table entry (32 bytes = one sector: slots +
// anchors).  Anchors are (re-)established from the last window of a text word.  All of this only
// decides WHERE the ids of a window come from; the ids, and everything downstream, are unchanged.
#ifndef SHK_EXT_MIN_BLOCKS
#define SHK_EXT_MIN_BLOCKS 6
#endif
//
// PACKED: the read comes from the packed stream (64-bit code words + 32-bit validity words per 32 bases,
// shk_hostpack.h) instead of text: no text or quality loads, no byte-parallel decode; the -q masking rule is
// already in the validity bits.  Everything from the rolling k-mers on is the same code.
//
// SCORES: also store each settled read's score record (SHK_F_SCORES); the instantiations without it are the default path.
template <bool HAS_QUAL, int MOD, bool EXT, bool PACKED, bool SCORES>
__global__ void __launch_bounds__(kFastThreads, EXT ? SHK_EXT_MIN_BLOCKS : SHK_FAST_MIN_BLOCKS)
analyze_reads_kernel(const ReadKernelArgs a)
{
    static_assert(!(PACKED && HAS_QUAL), "packed reads carry their masking in the validity bits");
    constexpr uint32_t S = EXT ? 2u : 1u;  // uint4s per front-table entry
    const int lane = threadIdx.x & 31;
    const uint32_t r = a.r0 + blockIdx.x * kFastThreads + threadIdx.x;
    const uint32_t tile = a.r0 / kReadsPerTile + blockIdx.x;
    const uint64_t pol_first = a.pol_first, pol_last = a.pol_last;
    // a DRAM-sized table must not displace the L2-resident streams: its sectors leave first
    const uint64_t pol_front = EXT ? pol_first : pol_last;
    const uint32_t k = (uint32_t)a.k;
    const uint64_t kmask2 = (1ULL << (2 * k)) - 1ULL;
    const int rc_shift = 2 * (int)k - 2;
    const uint32_t fshift = a.fgeom.shift, fmask = a.fgeom.off_mask;
    const uint32_t mq4b = (0x01010101u * (uint32_t)(a.mq & 0xFF)) ^ kH4;
    uint32_t count = 0, payload = 0, my_probes = 0, my_hits = 0, my_ext = 0, my_loads = 0;
    uint4 score = make_uint4(0u, 0u, 0u, 0u);
    bool slow = false;

    if (r < a.r1) {
        const uint32_t off0 = a.off[r];
        const uint32_t n = a.off[r + 1] - off0;
        if (n > kMaxFastLen) {
            slow = true;
        } else {
            Mru4 tab;
            tab.init();
            uint64_t fwd = 0, rc = 0;
            uint32_t run = 0, len = 0;
            // extension state: next reference position to compare, strand, the anchored ids, and
            // the cached word of the reference stream that holds position anc_t
            uint32_t anc_t = 0, anc_dir = 0, prevA = kFrontEmpty, prevB = kFrontEmpty;
            bool anc_on = false;
            uint64_t ew = 0;
            // text: 4 bases = one 32-bit word of the chunk's text; packed: 4 bases = one byte of a code word and
            // one nibble of a validity word.  Either way the walk is over ALIGNED 4-base words; positions of the
            // first and last word that lie outside the read are made invalid.
            const uint32_t src0 = PACKED ? off0 - a.pack_base : off0;
            const uint32_t head = src0 & 3u;
            const uint32_t *seqw = reinterpret_cast<const uint32_t *>(a.seq) + (src0 >> 2);
            const uint32_t *qualw = HAS_QUAL ? reinterpret_cast<const uint32_t *>(a.qual) + (src0 >> 2) : nullptr;
            const uint32_t n_words = (head + n + 3u) >> 2;
            uint32_t w_next = 0, q_next = 0;
            // packed: the next (up to) 8 words of this read - 8 code bytes and 8 validity nibbles - shifted down as
            // they are used.  Every lane reloads at the same iterations (j % 8 == 0), whatever its alignment in the
            // stream: two aligned words each, funnel-shifted to the lane's position.
            uint64_t cw = 0;
            uint32_t vw = 0;
            if (n_words && !PACKED) {
                w_next = ld_text_word(seqw, pol_first);
                if (HAS_QUAL) q_next = ld_text_word(qualw, pol_first);
            }
            for (uint32_t j = 0; j < n_words && !tab.overflow; ++j) {
                // per base b of the word: validity and 2-bit code (A0 C1 G2 T3)
                uint32_t code4, x;
                if (PACKED) {
                    if ((j & 7u) == 0u) {
                        const uint32_t wi = (src0 >> 2) + j;  // this 4-base word = byte wi of the code array
                        const uint32_t gi = wi >> 3, sh = (wi & 7u) * 8u;
                        const uint64_t c_lo = ld_u64_hint(a.pcodes + gi, pol_first), c_hi = ld_u64_hint(a.pcodes + gi + 1, pol_first);
                        const uint32_t v_lo = ld_text_word(a.pvalid + gi, pol_first), v_hi = ld_text_word(a.pvalid + gi + 1, pol_first);
                        cw = sh ? (c_lo >> sh) | (c_hi << (64u - sh)) : c_lo;
                        vw = __funnelshift_r(v_lo, v_hi, sh >> 1);
                    }
                    const uint32_t c8 = (uint32_t)cw & 0xFFu;
                    cw >>= 8;
                    code4 = c8 ^ ((c8 >> 1) & 0x55u);  // A0 C1 T2 G3 -> A0 C1 G2 T3, base b at bits 2b
                    x = vw & 0xFu;                      // bit b = base b is valid
                    vw >>= 4;
                } else {
                    uint32_t w = w_next;
                    const uint32_t qw = q_next;
                    if (j + 1 < n_words) {
                        w_next = ld_text_word(seqw + j + 1, pol_first);
                        if (HAS_QUAL) q_next = ld_text_word(qualw + j + 1, pol_first);
                    }
                    if (HAS_QUAL) w = sub_bytes4(w, qual_mask4(qw, mq4b));
                    codes4(w, code4, x);                    // byte b of x == 0 iff base b is valid
                }
                const uint32_t pos0 = 4u * j - head;  // position of byte 0 (wraps before the read)
                if (j == 0 || j + 1 == n_words) {     // bytes outside the read are not bases
#pragma unroll
                    for (int b = 0; b < 4; ++b)
                        if (pos0 + (uint32_t)b >= n) x = PACKED ? (x & ~(1u << b)) : (x | (0xFFu << (8 * b)));
                }
                if (run + 4u < k) {  // no window can complete in this word (start of a mate): roll only
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const bool valid = PACKED ? ((x >> b) & 1u) != 0u : ((x >> (8 * b)) & 0xFFu) == 0u;
                        const uint64_t code = PACKED ? (code4 >> (2 * b)) & 3u : (code4 >> (8 * b)) & 3u;
                        fwd = ((fwd << 2) | code) & kmask2;
                        rc = (rc >> 2) | ((3ULL ^ code) << rc_shift);
                        run = valid ? run + 1u : 0u;
                        len += valid ? 1u : 0u;
                    }
                    continue;
                }
                uint32_t bucket[4], key[4];
                bool wv[4], ex[4];
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    const bool valid = PACKED ? ((x >> b) & 1u) != 0u : ((x >> (8 * b)) & 0xFFu) == 0u;
                    const uint64_t code = PACKED ? (code4 >> (2 * b)) & 3u : (code4 >> (8 * b)) & 3u;
                    fwd = ((fwd << 2) | code) & kmask2;            // lsappend, kmer_utils.hpp:73-75
                    rc = (rc >> 2) | ((3ULL ^ code) << rc_shift);  // rsprepend(reverse_char), 77-79
                    run = valid ? run + 1u : 0u;                   // build_kmer restart, 57-71
                    len += valid ? 1u : 0u;                        // ReadAnalyzer.hpp:46-49
                    wv[b] = run >= k;
                    ex[b] = false;
                    if (EXT) {
                        // anchored: does the read go on like the reference (and keep its gene list)?
                        const uint32_t nib = (uint32_t)(ew >> ((anc_t & 15u) * 4u));
                        const uint32_t want = (uint32_t)code ^ (anc_dir * 3u);
                        ex[b] = anc_on && valid && ((nib ^ want) & 3u) == 0u && ((nib >> (2u + anc_dir)) & 1u) != 0u;
                        anc_on = ex[b];
                        anc_t += 1u - 2u * anc_dir;
                        if (ex[b] && ((anc_t + anc_dir) & 15u) == 0u)
                            ew = ld_u64_hint(a.estream + ((anc_t + 16u) >> 4), pol_last);
                    }
                    const uint64_t p = bit_index<MOD>(xxh64_u64(fwd < rc ? fwd : rc), a.geom);
                    bucket[b] = (uint32_t)(p >> fshift);
                    key[b] = ex[b] ? 0u : front_key((uint32_t)p & fmask);
                }
                uint4 q[4];
                uint4 an3 = make_uint4(0u, 0u, 0u, 0u);  // anchors of the last window's bucket (same sector as its slots)
                if (EXT) {
                    uint32_t cw[4], cidx[4];
#pragma unroll
                    for (int b = 0; b < 4; ++b) {  // coarse filter word of every window that needs a lookup
                        cidx[b] = (bucket[b] << a.coarse_rel) | (key[b] >> a.coarse_key_shift);
                        cw[b] = 0u;
                        if (wv[b] && !ex[b]) cw[b] = ld_u32_hint(a.coarse + (cidx[b] >> 5), pol_last);
                    }
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        q[b] = make_uint4(kFrontEmpty, kFrontEmpty, kFrontEmpty, kFrontEmpty);
                        if (ex[b]) {
                            q[b] = make_uint4(prevA, prevB, kFrontEmpty, kFrontEmpty);  // key[b] == 0
                            ++my_ext;
                        } else if ((cw[b] >> (cidx[b] & 31u)) & 1u) {
                            q[b] = ld_front(a.front + (uint64_t)bucket[b] * S, pol_front);
                            if (b == 3 && !anc_on) an3 = ld_front(a.front + (uint64_t)bucket[b] * S + 1, pol_front);
                            ++my_loads;
                        }
                    }
                } else {
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        q[b] = make_uint4(kFrontEmpty, kFrontEmpty, kFrontEmpty, kFrontEmpty);
                        if (wv[b]) q[b] = ld_front(a.front + bucket[b], pol_front);
                    }
                }
#pragma unroll
                for (int b = 0; b < 4; ++b) {
                    my_probes += wv[b] ? 1u : 0u;
                    const uint32_t pos = pos0 + (uint32_t)b;
                    const uint32_t kb = key[b];
                    uint4 qq = q[b];
                    uint32_t A, B;
                    uint32_t cur = bucket[b];  // entry that qq came from (anchors)
                    for (;;) {
                        // slot - key: same test and same id as slot ^ key (the key's low 18 bits are 0), but an add the
                        // FMA pipe can take
                        const uint32_t d0 = qq.x - kb, d1 = qq.y - kb, d2 = qq.z - kb, d3 = qq.w - kb;
                        const uint32_t lo01 = min(d0, d1), hi01 = max(d0, d1), lo23 = min(d2, d3), hi23 = max(d2, d3);
                        A = min(lo01, lo23);                        // smallest
                        B = min(max(lo01, lo23), min(hi01, hi23));  // second smallest
                        // not in this record and the bucket goes on (chain pointer: bit 31 set, not
                        // EMPTY): look at the next record.  A 2-id list never straddles records.
                        if (A < kFrontLim || (int32_t)qq.w >= -1) break;
                        cur = qq.w & 0x7FFFFFFFu;
                        qq = ld_front(a.front + (uint64_t)cur * S, pol_front);
                    }
                    const uint4 qfound = qq;  // the record A was found in (anchors)
                    const bool anyA = A < kFrontLim, anyB = B < kFrontLim;
                    const bool a0 = A == tab.g0, a1 = A == tab.g1, b0 = B == tab.g0, b1 = B == tab.g1;
                    my_hits += anyA ? 1u : 0u;
                    if ((!anyA | a0 | a1) & (!anyB | b0 | b1)) {
                        if (a0 | b0) {
                            tab.c0 += min(k, pos - tab.l0);
                            tab.h0 += 1;
                            tab.l0 = pos;
                        }
                        if (a1 | b1) {
                            tab.c1 += min(k, pos - tab.l1);
                            tab.h1 += 1;
                            tab.l1 = pos;
                        }
                    } else {
                        // generic: every slot of the bucket and of its chain, in list order
                        qq = q[b];
                        for (;;) {
#pragma unroll 1
                            for (int i = 0; i < 4; ++i) {
                                const uint32_t sl = i == 0 ? qq.x : (i == 1 ? qq.y : (i == 2 ? qq.z : qq.w));
                                const uint32_t d = sl ^ kb;
                                if (d < kFrontLim) {
                                    if (d & kFrontLongFlag) tab.overflow = true;  // list longer than 4 ids: exact path
                                    else tab.hit(d & 0xFFFFu, pos, k);
                                }
                            }
                            if (!front_is_chain(qq.w)) break;
                            qq = ld_front(a.front + (uint64_t)(qq.w & 0x7FFFFFFFu) * S, pol_front);
                        }
                    }
                    if (EXT && b == 3) {
                        // (re-)anchor on the word's last window: a looked-up hit with plain ids (list of
                        // 1 or 2).  The slot's anchor names a reference window with the same filter bit;
                        // the thread is anchored only if that window IS the read's window (either strand).
                        if (!anc_on && wv[3] && !ex[3] && A < 0x10000u && (B < 0x10000u || B >= kFrontLim) && !tab.overflow) {
                            uint4 an = an3;  // loaded with the bucket; a chained record brings its own
                            if (cur != bucket[3]) an = ld_front(a.front + (uint64_t)cur * S + 1, pol_front);
                            const uint32_t sa = A + kb;  // the slot that produced A (slot - key == A)
                            const uint32_t e = qfound.x == sa ? an.x : (qfound.y == sa ? an.y : (qfound.z == sa ? an.z : an.w));
                            // both candidate stream words travel with the two words of the reference window
                            const uint64_t ew0 = ld_u64_hint(a.estream + ((e + 1u + 16u) >> 4), pol_last);
                            const uint64_t ew1 = ld_u64_hint(a.estream + ((e - k + 16u) >> 4), pol_last);
                            const uint64_t rk = ref2_window(a.ref2, e, kmask2, pol_last);
                            if (rk == fwd) {
                                anc_on = true, anc_dir = 0u, anc_t = e + 1u, ew = ew0;
                            } else if (rk == rc) {
                                anc_on = true, anc_dir = 1u, anc_t = e - k, ew = ew1;
                            }
                            if (anc_on) {
                                prevA = A;
                                prevB = B < 0x10000u ? B : kFrontEmpty;
                            }
                        }
                    }
                }
            }
            if (tab.overflow) {
                slow = true;
            } else {
                finish_read(a, tab, len, count, payload, score);
            }
        }
        if (slow) {
            count = 0;
            payload = 0;
            my_probes = 0, my_hits = 0;  // counted by the kernel that classifies the read
            a.slow_list[atomicAdd(&a.counters->n_slow, 1u)] = r;
        }
        a.rec[r] = make_uint2(count, payload);
        if (SCORES && !slow) a.scores[r] = score;  // (a slow read's record comes from the kernel that settles it)
    }
    flush_warp_counters<EXT>(a, tile, lane, count, payload, my_probes, my_hits, my_ext, my_loads);
}

// ---------------------------------------------------------------------------------------------
// Middle path: one WARP per read the fast path gave up on (more than 4 genes, a list longer than 4
// ids, a text longer than kMaxFastLen), with the per-gene state {gene, cov, hits, last} in a
// 128-slot open-addressing table in shared memory (one per warp).  Windows are probed 32 at a time
// through the reference-shaped structures (filter word -> sector rank -> entry -> CSR ids) and
// applied in read order exactly as ReadAnalyzer.hpp:56-62,79-86 does; the lanes share the (distinct)
// ids of one list.  Reads that touch more than kMidMaxGenes genes go on to the exact path below.
// Thousands of such reads run concurrently (the table is 2 KB per warp), where the dense per-warp
// tables of the exact path allow only a few hundred.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kMidSlots = 128, kMidMaxGenes = 95, kMidWarps = 4;

template <bool HAS_QUAL, int MOD, bool WIDE, bool SCORES>
__global__ void __launch_bounds__(kMidWarps * 32) analyze_mid_kernel(const ReadKernelArgs a)
{
    __shared__ uint4 tables[kMidWarps][kMidSlots];  // {gene (0xFFFFFFFF = free), cov, hits, last}
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t n_slow = a.counters->n_slow;
    const uint32_t total_warps = gridDim.x * kMidWarps;
    const uint64_t pol_first = a.pol_first, pol_last = a.pol_last;
    const Sector *sector_base = reinterpret_cast<const Sector *>(a.sectors);
    uint4 *tab = tables[warp];
    uint32_t *keys = reinterpret_cast<uint32_t *>(tab);  // key of slot s = keys[4 * s]
    const uint32_t k = (uint32_t)a.k;
    unsigned long long probes = 0, hits_total = 0, assoc_total = 0, kept_total = 0;

    for (uint32_t i = blockIdx.x * kMidWarps + warp; i < n_slow; i += total_warps) {
        const uint32_t r = a.slow_list[i];
        const uint32_t off0 = a.off[r];
        const uint32_t n = a.off[r + 1] - off0;
        const bool packed = r >= a.pack_first;
        for (uint32_t s = lane; s < kMidSlots; s += 32) tab[s] = make_uint4(0xFFFFFFFFu, 0u, 0u, 0u);
        __syncwarp();
        uint32_t n_used = 0;
        bool overflow = false;
        const int nch = (int)((n + 31u) >> 5);
        ChunkState cs{0ULL, 0u};
        uint32_t len = 0;
        unsigned long long my_probes = 0, my_hits = 0;
        for (int c = 0; c < nch && !overflow; ++c) {
            uint32_t pw, bit;
            const bool wv = chunk_window<HAS_QUAL, MOD>(a, off0, n, c, lane, cs, len, pw, bit, packed);
            const uint32_t w = wv ? ld_filter_word(a.sectors + pw, pol_first) : 0u;
            const bool hit = wv && ((w >> bit) & 1u);
            my_probes += __popc(__ballot_sync(kFull, wv));
            uint32_t H = __ballot_sync(kFull, hit);
            uint64_t e = 0;
            if (hit) {
                Sector sc = ld_sector(sector_base + (pw >> 3));
                e = ld_u64_hint(a.entries + sector_rank(sc, pw & 7u, bit), pol_last);
            }
            my_hits += __popc(H);
            while (H && !overflow) {  // windows in read order
                const int src = __ffs(H) - 1;
                H &= H - 1;
                const uint64_t el = shfl64(e, src);
                const uint32_t epos = (uint32_t)c * 32u + (uint32_t)src;
                const uint32_t ln = list_len<WIDE>(el);
                for (uint32_t t0 = 0; t0 < ln; t0 += 32) {
                    if (n_used > kMidMaxGenes) {  // at most 32 inserts follow: the table never fills up
                        overflow = true;
                        break;
                    }
                    const uint32_t t = t0 + (uint32_t)lane;
                    bool inserted = false;
                    if (t < ln) {
                        const uint32_t g = list_id<WIDE>(a, el, ln, t);
                        uint32_t s = (g * 0x9E3779B1u) >> 25;  // 7 bits
                        for (;;) {
                            uint32_t key = keys[4 * s];
                            if (key == 0xFFFFFFFFu) {
                                key = atomicCAS(&keys[4 * s], 0xFFFFFFFFu, g);
                                if (key == 0xFFFFFFFFu) {
                                    // fresh map entry: `pos - 0` >= k for every window, so cov = k
                                    tab[s] = make_uint4(g, k, 1u, epos);
                                    inserted = true;
                                    break;
                                }
                            }
                            if (key == g) {
                                uint4 ent = tab[s];
                                ent.y += min(k, epos - ent.w);
                                ent.z += 1u;
                                ent.w = epos;
                                tab[s] = ent;
                                break;
                            }
                            s = (s + 1u) & (kMidSlots - 1u);
                        }
                    }
                    n_used += __popc(__ballot_sync(kFull, inserted));
                    __syncwarp();
                }
            }
        }
        if (overflow) {  // more genes than the table holds: exact path
            if (lane == 0) a.slow2_list[atomicAdd(&a.counters->n_slow2, 1u)] = r;
            __syncwarp();
            continue;
        }
        probes += my_probes;
        hits_total += my_hits;
        // argmax (ReadAnalyzer.hpp:90-102); each lane owns slots lane, lane+32, ...
        uint32_t maxc = 0, maxh = 0;
        for (uint32_t s = lane; s < kMidSlots; s += 32) {
            const uint4 ent = tab[s];
            if (ent.x != 0xFFFFFFFFu && (ent.y > maxc || (ent.y == maxc && ent.z > maxh))) {
                maxc = ent.y;
                maxh = ent.z;
            }
        }
        const uint32_t wmaxc = __reduce_max_sync(kFull, maxc);
        const uint32_t wmaxh = __reduce_max_sync(kFull, maxc == wmaxc ? maxh : 0u);
        uint32_t count = 0, first_gene = 0xFFFFFFFFu;
        for (uint32_t s = lane; s < kMidSlots; s += 32) {
            const uint4 ent = tab[s];
            if (ent.x != 0xFFFFFFFFu && ent.y == wmaxc && ent.z == wmaxh) {
                ++count;
                first_gene = min(first_gene, ent.x);
            }
        }
        count = __reduce_add_sync(kFull, count);
        first_gene = __reduce_min_sync(kFull, first_gene);
        const uint32_t n_best = count;
        if (!read_reported(a, wmaxc, len, n_best)) count = 0;
        uint32_t payload = first_gene;
        if (count >= 2) {
            payload = pool_reserve(a, count, lane);
            if (payload != 0xFFFFFFFFu) {
                // ascending gene order: a winner's place = number of winners with a smaller id
                for (uint32_t s = lane; s < kMidSlots; s += 32) {
                    const uint4 ent = tab[s];
                    if (ent.x != 0xFFFFFFFFu && ent.y == wmaxc && ent.z == wmaxh) {
                        uint32_t place = 0;
                        for (uint32_t u = 0; u < kMidSlots; ++u) {
                            const uint4 o = tab[u];
                            place += (o.x < ent.x && o.y == wmaxc && o.z == wmaxh) ? 1u : 0u;  // free slots: x = 0xFFFFFFFF
                        }
                        a.pool[payload + place] = ent.x;
                    }
                }
            }
        }
        if (lane == 0) {
            a.rec[r] = make_uint2(count, payload);
            if (SCORES) a.scores[r] = make_uint4(len, wmaxc, wmaxh, n_best);
            if (multi_entries(count, payload, a.wide)) atomicAdd(&a.tile_sums[r / kReadsPerTile], count);
            assoc_total += count;
            kept_total += count ? 1u : 0u;
        }
        __syncwarp();
    }
    if (lane == 0) {
        if (probes) atomicAdd(&a.counters->n_probes, probes);
        if (hits_total) atomicAdd(&a.counters->n_hits, hits_total);
        if (assoc_total) atomicAdd(&a.counters->n_assoc, assoc_total);
        if (kept_total) atomicAdd(&a.counters->n_kept, kept_total);
    }
}

// ---------------------------------------------------------------------------------------------
// Exact path: any number of genes, any read length.  One warp per read; a dense per-warp table
// indexed by gene id (ids are 16-bit, small_vector.hpp:46) holds {stamp, cov, hits, last} and is
// updated window by window in read order exactly as ReadAnalyzer.hpp:56-62,79-86 does, the
// lanes sharing the (distinct) ids of one list.  Stamps make clearing unnecessary.
// ---------------------------------------------------------------------------------------------
template <bool HAS_QUAL, int MOD, bool WIDE, bool SCORES>
__global__ void __launch_bounds__(128) analyze_slow_kernel(const ReadKernelArgs a)
{
    const int lane = threadIdx.x & 31;
    const uint32_t slab = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (slab >= a.n_slow_slabs) return;
    const uint32_t n_slow = a.counters->n_slow2;  // what the middle path could not hold
    if (slab >= n_slow) return;
    const uint64_t pol_first = a.pol_first, pol_last = a.pol_last;
    const Sector *sector_base = reinterpret_cast<const Sector *>(a.sectors);
    uint4 *table = a.slow_table + (uint64_t)slab * a.n_genes;
    uint32_t stamp = a.slow_stamp[slab];
    const uint32_t k = (uint32_t)a.k;
    unsigned long long probes = 0, hits_total = 0, assoc_total = 0, kept_total = 0;

    for (uint32_t i = slab; i < n_slow; i += a.n_slow_slabs) {
        const uint32_t r = a.slow2_list[i];
        const uint32_t off0 = a.off[r];
        const uint32_t n = a.off[r + 1] - off0;
        const bool packed = r >= a.pack_first;
        if (++stamp == 0) {  // stamp wrapped: clear the slab once
            for (uint32_t g = lane; g < a.n_genes; g += 32) table[g] = make_uint4(0, 0, 0, 0);
            stamp = 1;
            __syncwarp();
        }
        const int nch = (int)((n + 31u) >> 5);
        ChunkState cs{0ULL, 0u};
        uint32_t len = 0;
        for (int c = 0; c < nch; ++c) {
            uint32_t pw, bit;
            const bool wv = chunk_window<HAS_QUAL, MOD>(a, off0, n, c, lane, cs, len, pw, bit, packed);
            const uint32_t w = wv ? ld_filter_word(a.sectors + pw, pol_first) : 0u;
            const bool hit = wv && ((w >> bit) & 1u);
            probes += __popc(__ballot_sync(kFull, wv));
            uint32_t H = __ballot_sync(kFull, hit);
            uint64_t e = 0;
            if (hit) {
                Sector s = ld_sector(sector_base + (pw >> 3));
                e = ld_u64_hint(a.entries + sector_rank(s, pw & 7u, bit), pol_last);
            }
            hits_total += __popc(H);
            while (H) {  // windows in read order
                const int src = __ffs(H) - 1;
                H &= H - 1;
                const uint64_t el = shfl64(e, src);
                const uint32_t epos = (uint32_t)c * 32u + (uint32_t)src;
                const uint32_t ln = list_len<WIDE>(el);
                for (uint32_t t = lane; t < ln; t += 32) {
                    const uint32_t g = list_id<WIDE>(a, el, ln, t);
                    uint4 ent = table[g];
                    if (ent.x != stamp) {
                        // fresh map entry: `pos - 0` >= k for every window, so cov = k
                        ent = make_uint4(stamp, k, 1u, epos);
                    } else {
                        ent.y += min(k, epos - ent.w);
                        ent.z += 1u;
                        ent.w = epos;
                    }
                    table[g] = ent;
                }
                __syncwarp();
            }
        }
        // argmax over the touched genes in ascending id order
        uint32_t maxc = 0, maxh = 0;
        for (uint32_t g = lane; g < a.n_genes; g += 32) {
            const uint4 ent = table[g];
            if (ent.x == stamp && (ent.y > maxc || (ent.y == maxc && ent.z > maxh))) {
                maxc = ent.y;
                maxh = ent.z;
            }
        }
        const uint32_t wmaxc = __reduce_max_sync(kFull, maxc);
        const uint32_t wmaxh = __reduce_max_sync(kFull, maxc == wmaxc ? maxh : 0u);
        uint32_t count = 0;
        uint32_t first_gene = 0xFFFFFFFFu;
        for (uint32_t g0 = 0; g0 < a.n_genes; g0 += 32) {
            const uint32_t g = g0 + lane;
            bool is = false;
            if (g < a.n_genes) {
                const uint4 ent = table[g];
                is = ent.x == stamp && ent.y == wmaxc && ent.z == wmaxh;
            }
            const uint32_t b = __ballot_sync(kFull, is);
            if (b && first_gene == 0xFFFFFFFFu) first_gene = g0 + (uint32_t)(__ffs(b) - 1);
            count += __popc(b);
        }
        const uint32_t n_best = count;
        if (!read_reported(a, wmaxc, len, n_best)) count = 0;
        uint32_t payload = first_gene;
        if (count >= 2) {
            payload = pool_reserve(a, count, lane);
            if (payload != 0xFFFFFFFFu) {
                uint32_t o = payload;
                for (uint32_t g0 = 0; g0 < a.n_genes; g0 += 32) {
                    const uint32_t g = g0 + lane;
                    bool is = false;
                    if (g < a.n_genes) {
                        const uint4 ent = table[g];
                        is = ent.x == stamp && ent.y == wmaxc && ent.z == wmaxh;
                    }
                    const uint32_t b = __ballot_sync(kFull, is);
                    if (is) a.pool[o + __popc(b & ((1u << lane) - 1u))] = g;
                    o += __popc(b);
                }
            }
        }
        if (lane == 0) {
            a.rec[r] = make_uint2(count, payload);
            if (SCORES) a.scores[r] = make_uint4(len, wmaxc, wmaxh, n_best);
            if (multi_entries(count, payload, a.wide)) atomicAdd(&a.tile_sums[r / kReadsPerTile], count);
            assoc_total += count;
            kept_total += count ? 1u : 0u;
        }
        __syncwarp();
    }
    if (lane == 0) {
        a.slow_stamp[slab] = stamp;
        if (probes) atomicAdd(&a.counters->n_probes, probes);
        if (hits_total) atomicAdd(&a.counters->n_hits, hits_total);
        if (assoc_total) atomicAdd(&a.counters->n_assoc, assoc_total);
        if (kept_total) atomicAdd(&a.counters->n_kept, kept_total);
    }
}

// ---------------------------------------------------------------------------------------------
// K7: ordered output in the compact result form.  Per read one 16-bit word: the gene index of its single
// association, SHK_GENE_NONE, or SHK_GENE_MULTI = "see the multi list" (two or more winners - ties - or a
// single gene index that collides with the two marker values).  tile_base = exclusive scan of the per-tile
// multi counts (scan_tile_sums_kernel); every tile then scans its reads and writes the multi entries in read
// order, genes ascending (the order ReadOutput prints them, ReadOutput.hpp:40-49).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kReadsPerTile)
scatter_assoc_kernel(const ReadKernelArgs a, uint64_t multi_cap, const uint32_t *total)
{
    __shared__ uint32_t warp_tot[kReadsPerTile / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t r = blockIdx.x * kReadsPerTile + threadIdx.x;
    uint2 rc = make_uint2(0u, 0u);
    if (r < a.n_reads) rc = a.rec[r];
    const uint32_t m = multi_entries(rc.x, rc.y, a.wide);
    const uint32_t incl = warp_incl_scan(m, lane);
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    uint32_t o = a.tile_base[blockIdx.x] + incl - m;
    for (int w = 0; w < warp; ++w) o += warp_tot[w];
    if (r < a.n_reads) {
        a.gene16[r] = (uint16_t)(rc.x == 0u ? SHK_GENE_NONE : (m ? SHK_GENE_MULTI : rc.y));
        if (m && (uint64_t)o + m <= multi_cap) {
            if (rc.x == 1) {
                a.multi[o] = shk_assoc{r, rc.y};
            } else if ((uint64_t)rc.y + rc.x <= a.pool_cap) {  // pool overflow: the host re-runs the chunk
                for (uint32_t t = 0; t < rc.x; ++t) a.multi[o + t] = shk_assoc{r, a.pool[rc.y + t]};
            }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) a.counters->n_multi = *total;
}

// ---------------------------------------------------------------------------------------------
// K8 (SHK_F_GENE_COUNTS): per-gene counts of the chunk's reported reads, added into counts[0, n_genes) (reads whose only
// association is g) and counts[n_genes, 2 n_genes) (reads with g among two or more tied associations).  Reads rec and
// pool once the classification kernels have settled every read, so it counts exactly what the result lists hold, on
// every path and id width.  No address is hot: the single winners of a warp are merged with __match_any_sync (one add
// per distinct gene), and the genes of one tied read are distinct, so the warp adds them 32 at a time without a
// conflict.  SMEM: the adds go to a per-CTA histogram in shared memory, and every non-zero bin reaches global memory
// once per CTA.  A chunk whose tie pool overflowed adds nothing: the host runs the whole chunk again.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kCountThreads = 256;
constexpr uint32_t kCountSmemGenes = 6144;  // 2 x 6144 32-bit bins = 48 KB, the most static shared memory a kernel may have

// ---------------------------------------------------------------------------------------------
// SHK_F_EQ_CLASSES: the class table (EqTable, shk_internal.h).  One warp inserts one id list: the lanes hash it
// together, probe linearly from a slot the hash picks, and either add 1 to the slot whose published list equals theirs
// (compared id by id: the hash only picks the slots to compare) or claim an empty slot.  A claimer reserves a slot
// (used[1], refused at 3/4 of the slots, so in-flight claims never fill the table) and its arena range before the CAS,
// so a claimed slot is always published: it writes the ids, then off, then len with release semantics.  A warp that
// loses the CAS to a warp inserting the same new list adds to that slot, and its reservations stay unused until the
// next growth compacts the arena: a burst of one new class arriving in many warps at once can use up the arena (or the
// slot budget) and bring a growth forward that the live classes do not need.  No wait is unbounded: a warp that meets an unpublished slot with its hash polls it kEqSpins times and
// then leaves the read over, as it does past kEqProbes slots (K8 only), at the load limit (3/4 of the slots) or with
// the arena full.  Left-over reads go to a slot-private list; shk_reads_collect inserts them in later launches (after
// a kernel boundary every claimed slot is published), growing the table first when a claim was refused.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kEqProbes = 64;
constexpr uint32_t kEqSpins = 2048;
constexpr uint32_t kEqThreads = 256;

__device__ __forceinline__ unsigned long long eq_mix(unsigned long long x)  // splitmix64 finaliser
{
    x ^= x >> 30;
    x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27;
    x *= 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}

__device__ __forceinline__ uint32_t eq_ld_acquire(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void eq_st_release(uint32_t *p, uint32_t v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Warp-collective; every lane gets the same answer: 0 placed, 1 left over, 2 left over and the table must grow.
__device__ __noinline__ int eq_insert(const EqTable t, const uint32_t *__restrict__ ids, uint32_t n, uint32_t max_probes)
{
    const int lane = threadIdx.x & 31;
    unsigned long long h = 0;
    for (uint32_t i = lane; i < n; i += 32) h += eq_mix(((unsigned long long)i << 32 | ids[i]) + 0x9e3779b97f4a7c15ull);
    for (int o = 16; o; o >>= 1) h += __shfl_xor_sync(kFull, h, o);
    h = (eq_mix(h ^ n) & t.hash_mask) + 1u;  // never 0 (empty) unless the mask keeps all 64 bits
    if (!h) h = 1;
    const uint32_t mask = t.cap - 1u;
    uint32_t j = (uint32_t)eq_mix(h) & mask;
    unsigned long long res = ~0ull;  // arena range reserved for a claim
    for (uint32_t p = 0; p < max_probes; ++p, j = (j + 1u) & mask) {
        EqSlot *s = t.slots + j;
        unsigned long long cur = 0;
        if (lane == 0) cur = __ldcg(&s->hash);
        cur = __shfl_sync(kFull, cur, 0);
        if (cur == 0) {
            if (res == ~0ull) {
                int refused = 0;
                if (lane == 0) {  // a slot and an arena range, both reserved before the CAS
                    if (atomicAdd(&t.used[1], 1ull) >= (unsigned long long)t.cap / 4 * 3) refused = 1;
                    else {
                        res = atomicAdd(&t.used[0], (unsigned long long)n);
                        if (res + n > t.arena_cap) refused = 1;
                    }
                    if (refused) atomicExch(&t.used[2], 1ull);
                }
                if (__shfl_sync(kFull, refused, 0)) return 2;
                res = __shfl_sync(kFull, res, 0);
            }
            if (lane == 0) cur = atomicCAS(&s->hash, 0ull, h);
            cur = __shfl_sync(kFull, cur, 0);
            if (cur == 0) {  // claimed: publish
                for (uint32_t i = lane; i < n; i += 32) t.arena[res + i] = ids[i];
                __threadfence();
                __syncwarp();
                if (lane == 0) {
                    s->off = (uint32_t)res;
                    eq_st_release(&s->len, n);
                    atomicAdd(&t.count[j], 1ull);
                }
                return 0;
            }
        }
        if (cur != h) continue;
        uint32_t len = 0;
        if (lane == 0)
            for (uint32_t w = 0; !(len = eq_ld_acquire(&s->len)) && w < kEqSpins; ++w) __nanosleep(128);
        len = __shfl_sync(kFull, len, 0);
        __syncwarp();
        if (!len) return 1;  // still unpublished: a later launch inserts the read
        if (len != n) continue;
        const uint32_t off = __ldcg(&s->off);
        bool same = true;
        for (uint32_t i = lane; i < n; i += 32) same &= __ldcg(t.arena + off + i) == ids[i];
        if (__all_sync(kFull, same)) {
            if (lane == 0) atomicAdd(&t.count[j], 1ull);
            return 0;
        }
    }
    if (max_probes < t.cap) return 1;  // K8's probe limit: the leftover pass probes every slot
    if (lane == 0) atomicExch(&t.used[2], 1ull);  // every slot probed, none free: only a larger table takes the read
    return 2;
}

template <bool SMEM, bool EQ>
__global__ void __launch_bounds__(kCountThreads)
gene_counts_kernel(const uint2 *__restrict__ rec, const uint32_t *__restrict__ pool, uint32_t n_reads, uint32_t n_genes,
                   const ChunkCounters *counters, unsigned long long *counts, const EqTable eq, uint32_t *left,
                   uint32_t *n_left)
{
    __shared__ uint32_t hist[SMEM ? 2 * kCountSmemGenes : 1];
    if (counters->pool_overflow) return;  // the same for every thread of the grid
    if (SMEM) {
        for (uint32_t i = threadIdx.x; i < 2 * n_genes; i += kCountThreads) hist[i] = 0;
        __syncthreads();
    }
    auto add = [&](uint32_t bin, uint32_t v) {
        if (SMEM) atomicAdd(&hist[bin], v);
        else atomicAdd(&counts[bin], (unsigned long long)v);
    };
    const int lane = threadIdx.x & 31;
    for (uint32_t w = blockIdx.x * kCountThreads + (threadIdx.x & ~31u); w < n_reads; w += gridDim.x * kCountThreads) {
        const uint32_t r = w + lane;
        const uint2 rc = r < n_reads ? rec[r] : make_uint2(0u, 0u);
        const uint32_t g = rc.x == 1u ? rc.y : 0xFFFFFFFFu;  // gene ids are < n_genes < 2^32
        const uint32_t peers = __match_any_sync(kFull, g);
        if (g != 0xFFFFFFFFu && lane == __ffs(peers) - 1) add(g, __popc(peers));
        for (uint32_t tied = __ballot_sync(kFull, rc.x >= 2u); tied; tied &= tied - 1u) {
            const int src = __ffs(tied) - 1;
            const uint32_t cnt = __shfl_sync(kFull, rc.x, src), off = __shfl_sync(kFull, rc.y, src);
            for (uint32_t t = lane; t < cnt; t += 32) add(n_genes + pool[off + t], 1u);
            if (EQ && eq_insert(eq, pool + off, cnt, kEqProbes) && lane == 0) left[atomicAdd(n_left, 1u)] = w + src;
        }
    }
    if (SMEM) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < 2 * n_genes; i += kCountThreads)
            if (hist[i]) atomicAdd(&counts[i], (unsigned long long)hist[i]);
    }
}

template <bool EQ>
static void launch_gene_counts(shk_ctx *ctx, const ReadKernelArgs &a, cudaStream_t st, const EqTable &t, const EqPass *eq)
{
    const bool smem = a.n_genes <= kCountSmemGenes;
    const unsigned per_sm = smem ? 4u : 8u;
    const unsigned blocks = std::min<unsigned>((a.n_reads + kCountThreads - 1) / kCountThreads, (unsigned)ctx->sm_count * per_sm);
    uint32_t *left = eq ? eq->left : nullptr, *n_left = eq ? eq->n_left : nullptr;
    if (smem)
        gene_counts_kernel<true, EQ><<<blocks, kCountThreads, 0, st>>>(a.rec, a.pool, a.n_reads, a.n_genes, a.counters,
                                                                     ctx->d_gene_counts, t, left, n_left);
    else
        gene_counts_kernel<false, EQ><<<blocks, kCountThreads, 0, st>>>(a.rec, a.pool, a.n_reads, a.n_genes, a.counters,
                                                                      ctx->d_gene_counts, t, left, n_left);
}

__global__ void __launch_bounds__(kEqThreads)
eq_leftover_kernel(const uint2 *__restrict__ rec, const uint32_t *__restrict__ pool, const uint32_t *__restrict__ in,
                   uint32_t n_in, const EqTable t, uint32_t *out, uint32_t *n_out)
{
    const int lane = threadIdx.x & 31;
    for (uint32_t w = (blockIdx.x * kEqThreads + threadIdx.x) >> 5; w < n_in; w += gridDim.x * (kEqThreads / 32)) {
        const uint32_t r = in[w];
        const uint2 rc = rec[r];
        if (eq_insert(t, pool + rc.y, rc.x, t.cap) && lane == 0) out[atomicAdd(n_out, 1u)] = r;
    }
}

// One thread per slot of `from`; nothing else touches either table meanwhile, and every claimed slot is published.
__global__ void __launch_bounds__(kEqThreads) eq_rehash_kernel(const EqTable from, const EqTable to)
{
    const uint32_t mask = to.cap - 1u;
    for (uint32_t i = blockIdx.x * kEqThreads + threadIdx.x; i < from.cap; i += gridDim.x * kEqThreads) {
        const EqSlot s = from.slots[i];
        if (!s.len) continue;
        const unsigned long long o = atomicAdd(&to.used[0], (unsigned long long)s.len);
        for (uint32_t k = 0; k < s.len; ++k) to.arena[o + k] = from.arena[s.off + k];
        uint32_t j = (uint32_t)eq_mix(s.hash) & mask;
        while (atomicCAS(&to.slots[j].hash, 0ull, s.hash) != 0ull) j = (j + 1u) & mask;  // to.cap > live slots
        to.slots[j].off = (uint32_t)o;
        to.slots[j].len = s.len;
        to.count[j] = from.count[i];
        atomicAdd(&to.used[1], 1ull);
    }
}

static void eq_free(EqTable &t)
{
    cudaFree(t.slots);
    cudaFree(t.count);
    cudaFree(t.arena);
    cudaFree(t.used);
    t.slots = nullptr, t.count = nullptr, t.arena = nullptr, t.used = nullptr;
    t.cap = 0, t.arena_cap = 0;
}

static int eq_alloc_table(shk_ctx *ctx, EqTable &t, uint32_t cap, uint64_t arena_cap)
{
    SHK_CUDA(ctx, cudaMalloc((void **)&t.slots, (size_t)cap * sizeof(EqSlot)));
    SHK_CUDA(ctx, cudaMalloc((void **)&t.count, (size_t)cap * 8));
    SHK_CUDA(ctx, cudaMalloc((void **)&t.arena, arena_cap * 4));
    SHK_CUDA(ctx, cudaMalloc((void **)&t.used, 3 * 8));
    t.cap = cap;
    t.arena_cap = arena_cap;
    SHK_CUDA(ctx, cudaMemsetAsync(t.slots, 0, (size_t)cap * sizeof(EqSlot), ctx->build_stream));
    SHK_CUDA(ctx, cudaMemsetAsync(t.count, 0, (size_t)cap * 8, ctx->build_stream));
    SHK_CUDA(ctx, cudaMemsetAsync(t.used, 0, 3 * 8, ctx->build_stream));
    return SHK_OK;
}

int eq_alloc(shk_ctx *ctx, uint32_t cap, uint64_t arena_cap)
{
    const unsigned long long mask = ctx->eq.hash_mask;
    eq_free(ctx->eq);
    ctx->eq.hash_mask = mask;
    if (int rc = eq_alloc_table(ctx, ctx->eq, cap, arena_cap)) return rc;
    SHK_CUDA(ctx, cudaStreamSynchronize(ctx->build_stream));
    return SHK_OK;
}

int eq_grow(shk_ctx *ctx)
{
    for (uint32_t i = 0; i < ctx->n_slots; ++i) SHK_CUDA(ctx, cudaEventSynchronize(ctx->slots[i].ev_eq));
    EqTable &from = ctx->eq;
    if (from.cap >= (1u << 30) || from.arena_cap >= (1ull << 31))
        return fail(ctx, SHK_E_LIMIT, "the class table would exceed 2^31 slots or 2^32 ids");
    EqTable to;
    to.hash_mask = from.hash_mask;
    if (int rc = eq_alloc_table(ctx, to, from.cap * 2, from.arena_cap * 2)) {
        eq_free(to);
        return rc;
    }
    const unsigned blocks = std::min<unsigned>((from.cap + kEqThreads - 1) / kEqThreads, (unsigned)ctx->sm_count * 8);
    eq_rehash_kernel<<<blocks, kEqThreads, 0, ctx->build_stream>>>(from, to);
    SHK_CUDA(ctx, cudaGetLastError());
    SHK_CUDA(ctx, cudaStreamSynchronize(ctx->build_stream));
    eq_free(from);
    ctx->eq = to;
    ctx->launches += 1;
    return SHK_OK;
}

int eq_leftover_pass(shk_ctx *ctx, const ReadKernelArgs &a, const uint32_t *in, uint32_t n_in, const EqPass &out,
                     cudaStream_t st)
{
    const unsigned blocks = std::min<unsigned>((n_in + kEqThreads / 32 - 1) / (kEqThreads / 32), (unsigned)ctx->sm_count * 8);
    eq_leftover_kernel<<<blocks, kEqThreads, 0, st>>>(a.rec, a.pool, in, n_in, ctx->eq, out.left, out.n_left);
    SHK_CUDA(ctx, cudaGetLastError());
    SHK_CUDA(ctx, cudaEventRecord(out.ev, st));
    ctx->launches += 1;
    return SHK_OK;
}

// SHK_F_WIDE_IDS: there is no front table, every read goes to the middle path.
__global__ void __launch_bounds__(256) all_reads_slow_kernel(const ReadKernelArgs a)
{
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < a.n_reads) {
        a.slow_list[r] = r;
        a.rec[r] = make_uint2(0u, 0u);
    }
    if (r == 0) a.counters->n_slow = a.n_reads;
}

template <bool HAS_QUAL, int MOD, bool SCORES>
static void launch_typed(const ReadKernelArgs &a0, cudaStream_t st, unsigned tiles, unsigned slow_blocks, cudaEvent_t ev_ka)
{
    // middle path: a grid-stride loop over the slow list (its length is only known on the device)
    const unsigned mid_blocks = std::min<unsigned>((tiles * kReadsPerTile + kMidWarps - 1) / kMidWarps, 148u * 8u);
    ReadKernelArgs a = a0;
    if (a.wide) {
        all_reads_slow_kernel<<<(a.n_reads + 255) / 256, 256, 0, st>>>(a);
        if (ev_ka) cudaEventRecord(ev_ka, st);
        analyze_mid_kernel<HAS_QUAL, MOD, true, SCORES><<<mid_blocks, kMidWarps * 32, 0, st>>>(a);
        analyze_slow_kernel<HAS_QUAL, MOD, true, SCORES><<<slow_blocks, 128, 0, st>>>(a);
        return;
    }
    const uint32_t split = std::min(a.pack_first, a.n_reads);
    // The thread-per-read kernels extend only over a DRAM-sized table; an L2-sized one they probe window by window in
    // its slots-only copy (info.plain_front), which is faster there (DESIGN.md 5).
    const bool ext = a.estream && !a.front_plain;
    if (split > 0) {  // text part
        a.r0 = 0;
        a.r1 = split;
        if (a.front_plain) a.front = a.front_plain;
        const unsigned blocks = (split + kReadsPerTile - 1) / kReadsPerTile;
        if (ext) analyze_reads_kernel<HAS_QUAL, MOD, true, false, SCORES><<<blocks, kFastThreads, 0, st>>>(a);
        else analyze_reads_kernel<HAS_QUAL, MOD, false, false, SCORES><<<blocks, kFastThreads, 0, st>>>(a);
        a.front = a0.front;
    }
    if (split < a.n_reads) {  // packed part
        a.r0 = split;
        a.r1 = a.n_reads;
        const unsigned blocks = (a.n_reads - split + kReadsPerTile - 1) / kReadsPerTile;
        if (a.estream && a.refr && bulk_enabled()) {
            launch_bulk_kernel<SCORES>(a, st, blocks);
        } else {
            if (a.front_plain) a.front = a.front_plain;
            if (ext) analyze_reads_kernel<false, MOD, true, true, SCORES><<<blocks, kFastThreads, 0, st>>>(a);
            else analyze_reads_kernel<false, MOD, false, true, SCORES><<<blocks, kFastThreads, 0, st>>>(a);
            a.front = a0.front;
        }
    }
    if (ev_ka) cudaEventRecord(ev_ka, st);
    analyze_mid_kernel<HAS_QUAL, MOD, false, SCORES><<<mid_blocks, kMidWarps * 32, 0, st>>>(a);
    analyze_slow_kernel<HAS_QUAL, MOD, false, SCORES><<<slow_blocks, 128, 0, st>>>(a);
}

template <bool SCORES>
static void launch_classify(const ReadKernelArgs &a, cudaStream_t st, unsigned tiles, unsigned slow_blocks, cudaEvent_t ev_ka)
{
    const bool q = a.qual != nullptr;
    switch (a.geom.mod_kind) {
    case MOD_POW2: q ? launch_typed<true, MOD_POW2, SCORES>(a, st, tiles, slow_blocks, ev_ka) : launch_typed<false, MOD_POW2, SCORES>(a, st, tiles, slow_blocks, ev_ka); break;
    case MOD_B33: q ? launch_typed<true, MOD_B33, SCORES>(a, st, tiles, slow_blocks, ev_ka) : launch_typed<false, MOD_B33, SCORES>(a, st, tiles, slow_blocks, ev_ka); break;
    default: q ? launch_typed<true, MOD_GENERIC, SCORES>(a, st, tiles, slow_blocks, ev_ka) : launch_typed<false, MOD_GENERIC, SCORES>(a, st, tiles, slow_blocks, ev_ka); break;
    }
}

int launch_read_kernels(shk_ctx *ctx, const ReadKernelArgs &a, uint64_t multi_cap, cudaStream_t st, cudaEvent_t ev_k0,
                        cudaEvent_t ev_ka, cudaEvent_t ev_k1, const EqPass *eq)
{
    if (ev_k0) cudaEventRecord(ev_k0, st);
    int launched = 0;
    if (a.n_reads > 0) {
        const unsigned tiles = (a.n_reads + kReadsPerTile - 1) / kReadsPerTile;
        const unsigned slow_blocks = (a.n_slow_slabs + 3) / 4;
        cudaMemsetAsync(a.tile_sums, 0, (size_t)tiles * 4, st);  // the classification kernels add to it
        if (a.scores) launch_classify<true>(a, st, tiles, slow_blocks, ev_ka);
        else launch_classify<false>(a, st, tiles, slow_blocks, ev_ka);
        if (ctx->d_gene_counts && eq) {  // growth frees the table this launch is given
            std::lock_guard<std::mutex> lk(ctx->eq_mu);
            launch_gene_counts<true>(ctx, a, st, ctx->eq, eq);
            cudaEventRecord(eq->ev, st);
        } else if (ctx->d_gene_counts) {
            launch_gene_counts<false>(ctx, a, st, EqTable{}, nullptr);
        }
        // tile_base <- exclusive scan(tile_sums); the grand total lands in tile_base[tiles]
        cudaMemcpyAsync(a.tile_base, a.tile_sums, (size_t)tiles * 4, cudaMemcpyDeviceToDevice, st);
        scan_tile_sums_kernel<<<1, 1024, 0, st>>>(a.tile_base, tiles, a.tile_base + tiles);
        scatter_assoc_kernel<<<tiles, kReadsPerTile, 0, st>>>(a, multi_cap, a.tile_base + tiles);
        const uint32_t split = std::min(a.pack_first, a.n_reads);
        launched = (a.wide ? 5 : 4 + (split > 0 ? 1 : 0) + (split < a.n_reads ? 1 : 0)) + (ctx->d_gene_counts ? 1 : 0);
        ctx->launches += launched;
    }
    else if (ev_ka) cudaEventRecord(ev_ka, st);
    if (ev_k1) cudaEventRecord(ev_k1, st);
    return launched;
}

__global__ void fetch_policies_kernel(uint64_t *out)
{
    out[0] = make_policy_evict_first();
    out[1] = make_policy_evict_last();
}

int fetch_cache_policies(shk_ctx *ctx)
{
    uint64_t *d = nullptr, h[2] = {0, 0};
    SHK_CUDA(ctx, cudaMalloc((void **)&d, 16));
    fetch_policies_kernel<<<1, 1>>>(d);
    cudaError_t e = cudaMemcpy(h, d, 16, cudaMemcpyDeviceToHost);
    cudaFree(d);
    SHK_CUDA(ctx, e);
    ctx->pol_first = h[0];
    ctx->pol_last = h[1];
    return SHK_OK;
}

// Re-runs only the scatter (after the host grew the association buffer).
int launch_scatter(shk_ctx *ctx, const ReadKernelArgs &a, uint64_t multi_cap, cudaStream_t st)
{
    if (a.n_reads == 0) return 0;
    const unsigned tiles = (a.n_reads + kReadsPerTile - 1) / kReadsPerTile;
    scatter_assoc_kernel<<<tiles, kReadsPerTile, 0, st>>>(a, multi_cap, a.tile_base + tiles);
    ctx->launches += 1;
    return 1;
}

}  // namespace shk
