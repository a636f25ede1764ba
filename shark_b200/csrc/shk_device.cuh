// Device-side primitives shared by the index-build and read-classification kernels (sm_100a).
// Citations: reference file:line relative to the reference tree.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace shk {

// ---------------------------------------------------------------------------------------------
// Filter layout in HBM ("rank-in-sector").  The logical bit vector `_bf` of bf_bits bits
// (bloomfilter.h:195-197) is stored as 32-byte sectors = the DRAM access granule:
//     word 0..6 : 224 filter bits   (logical 32-bit word q -> sector q/7, slot q%7)
//     word 7    : number of set bits in all earlier sectors (the rank directory entry)
// so `_bf[p]` and `_brank(p+1)` (bloomfilter.h:89-90, rank_support_v.hpp:114-124) cost ONE
// sector.  Physical word index of logical word q is q + q/7.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kWordsPerSector = 7;

struct __align__(32) Sector {
    uint32_t w[8];
};

enum ModKind : int { MOD_POW2 = 0, MOD_B33 = 1, MOD_GENERIC = 2 };

struct FilterGeom {
    uint64_t bf_bits;
    uint64_t n_sectors;
    uint64_t pow2_mask;  // bf_bits-1 when MOD_POW2
    uint32_t b33;        // bf_bits >> 33 when MOD_B33
    int mod_kind;
};

// XXH64 of one 8-byte little-endian word, seed 0: kmer_utils.hpp:81-83 ->
// xxhash.hpp:459-492 (len < 32: h = PRIME64_5 + len) -> 425-456 (one 8-byte lane + avalanche);
// primes xxhash.hpp:349.
__device__ __forceinline__ uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }

__device__ __forceinline__ uint64_t xxh64_u64(uint64_t v)
{
    constexpr uint64_t P1 = 11400714785074694791ULL, P2 = 14029467366897019727ULL, P3 = 1609587929392839161ULL,
                       P4 = 9650029242287828579ULL, P5 = 2870177450012600261ULL;
    uint64_t h = P5 + 8;
    uint64_t k1 = rotl64(v * P2, 31) * P1;
    h ^= k1;
    h = rotl64(h, 27) * P1 + P4;
    h ^= h >> 33;
    h *= P2;
    h ^= h >> 29;
    h *= P3;
    h ^= h >> 32;
    return h;
}

// hash -> logical bit index: `hash % _size` (bloomfilter.h:58,66,88).
template <int MOD>
__device__ __forceinline__ uint64_t bit_index(uint64_t h, const FilterGeom &g)
{
    if (MOD == MOD_POW2) return h & g.pow2_mask;
    if (MOD == MOD_B33) {
        // bf_bits = b * 2^33: the low 33 bits survive, the high 31 bits reduce mod b
        uint32_t hi = (uint32_t)(h >> 33) % g.b33;
        return ((uint64_t)hi << 33) | (h & ((1ULL << 33) - 1));
    }
    return h % g.bf_bits;
}

// logical bit -> (physical 32-bit word index, bit in word)
__device__ __forceinline__ uint64_t phys_word(uint64_t p)
{
    uint64_t q = p >> 5;
    return q + q / kWordsPerSector;
}

// Base codes: kmer_utils.hpp:29-41 (to_int) minus 1 (kmer_utils.hpp:68).  A/a=0 C/c=1 G/g=2
// T/t=3; everything else (and every byte >= 128) is invalid.
__device__ __forceinline__ bool base_valid(uint32_t ch)
{
    uint32_t u = (ch | 0x20u) - 0x61u;  // 'a' -> 0
    return u < 32u && ((0x00080045u >> u) & 1u);  // a, c, g, t
}
__device__ __forceinline__ uint32_t base_code(uint32_t ch)
{
    uint32_t x = (ch >> 1) & 3u;  // A:0 C:1 G:3 T:2
    return x ^ (x >> 1);          // A:0 C:1 G:2 T:3
}

// Reverse complement of a packed k-mer (kmer_utils.hpp:47-55): complement, reverse the 2-bit
// groups.  brev reverses all 64 bits; swapping the two bits of each pair restores the codes.
__device__ __forceinline__ uint64_t revcompl(uint64_t kmer, int k)
{
    uint64_t x = __brevll(~kmer);
    x = ((x & 0xAAAAAAAAAAAAAAAAULL) >> 1) | ((x & 0x5555555555555555ULL) << 1);
    return x >> (64 - 2 * k);
}

__device__ __forceinline__ uint64_t canonical(uint64_t fwd, int k)
{
    uint64_t rc = revcompl(fwd, k);
    return fwd < rc ? fwd : rc;  // min(kmer, rckmer): KmerBuilder.hpp:48, ReadAnalyzer.hpp:55
}

// ---- loads with Blackwell cache controls ----------------------------------------------------
// One filter word of a random sector: read once, never reused -> keep it out of L1 and mark it
// first to leave L2, so that the small hot arrays (entries, CSR) stay resident.
__device__ __forceinline__ uint32_t ld_filter_word(const uint32_t *p, uint64_t pol_evict_first)
{
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;"
                 : "=r"(r)
                 : "l"(p), "l"(pol_evict_first));
    return r;
}
// Whole 32-byte sector in one 256-bit load (LDG.E.256, sm_100+).
__device__ __forceinline__ Sector ld_sector(const Sector *p)
{
    Sector s;
    asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(s.w[0]), "=r"(s.w[1]), "=r"(s.w[2]), "=r"(s.w[3]), "=r"(s.w[4]), "=r"(s.w[5]), "=r"(s.w[6]),
                   "=r"(s.w[7])
                 : "l"(p));
    return s;
}
__device__ __forceinline__ uint64_t make_policy_evict_last()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint64_t make_policy_evict_first()
{
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ uint32_t ld_u32_hint(const uint32_t *p, uint64_t pol)
{
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ uint64_t ld_u64_hint(const uint64_t *p, uint64_t pol)
{
    uint64_t r;
    asm volatile("ld.global.nc.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(r) : "l"(p), "l"(pol));
    return r;
}

// rank of bit `bit` of slot `slot` inside a loaded sector = set bits strictly before it.
__device__ __forceinline__ uint32_t sector_rank(const Sector &s, uint32_t slot, uint32_t bit)
{
    uint32_t r = s.w[7];
#pragma unroll
    for (uint32_t i = 0; i < kWordsPerSector; ++i) {
        uint32_t m = i < slot ? 0xFFFFFFFFu : (i == slot ? ((1u << bit) - 1u) : 0u);
        r += __popc(s.w[i] & m);
    }
    return r;
}

// ---------------------------------------------------------------------------------------------
// Per-set-bit entry (replaces small_vector_t, small_vector.hpp:25-91, and the select over
// `_bv`, bloomfilter.h:91-94): one 8-byte word per set bit r
//     bits 63..48 : first gene id of the list
//     bits 47..32 : list length - 1
//     bits 31..0  : second gene id when length == 2, CSR begin offset when length >= 3
// so the common lists (1 or 2 genes) need no further memory access.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t make_entry(uint32_t id0, uint32_t len, uint32_t lo)
{
    return ((uint64_t)id0 << 48) | ((uint64_t)(len - 1) << 32) | lo;
}
__device__ __forceinline__ uint32_t entry_id0(uint64_t e) { return (uint32_t)(e >> 48); }
__device__ __forceinline__ uint32_t entry_len(uint64_t e) { return ((uint32_t)(e >> 32) & 0xFFFFu) + 1u; }
__device__ __forceinline__ uint32_t entry_lo(uint64_t e) { return (uint32_t)e; }
// SHK_F_WIDE_IDS (32-bit gene ids): bits 63..32 = list length - 1, bits 31..0 = the id of a one-id list, else the
// CSR begin offset (the ids, first one included, are read from the 32-bit CSR).
__device__ __forceinline__ uint64_t make_wide_entry(uint32_t len, uint32_t lo) { return ((uint64_t)(len - 1) << 32) | lo; }
__device__ __forceinline__ uint32_t wide_entry_len(uint64_t e) { return (uint32_t)(e >> 32) + 1u; }

// ---------------------------------------------------------------------------------------------
// Front table: an exact, L2-sized accelerator in front of the bit vector.  The filter is sparse
// (load 0.03 % .. 1 %), so the set bits themselves fit in tens of MB.  The bit positions are
// uniformly distributed hash values, which makes "bucket = position >> shift" a perfect
// bucketing: bucket b describes positions [b << shift, (b+1) << shift) with four 32-bit slots
//     bit  31     : 0
//     bits 30..18 : position - (b << shift)                       (shift <= 13)
//     bit  17     : the position's list has 3 or 4 ids (set on each of its slots)
//     bit  16     : 0 = (position, gene id in bits 15..0); a position whose list has L <= 4
//                       ids owns L such slots (contiguous, ascending gene id)
//                   1 = the position is set but its list is longer than 4 ids (the fast path
//                       cannot hold it anyway and hands the read to the exact path)
// 0xFFFFFFFF = empty slot.  A bucket that needs more than 4 slots keeps 3 and stores in slot 3 a
// chain pointer (bit 31 set, low 31 bits = index of a 16-byte overflow record with the same
// layout, appended to the same array).  One 16-byte load therefore answers "definitely not set"
// / "set, genes g.." for almost every probe, the rest follows a short chain that is L2-resident
// too - no probe of the fast path touches DRAM-sized structures.  `slot ^ key` is below 2^18 iff
// the slot describes the probed position, and then equals the gene id when no flag is set: the
// fast kernel finds the (up to two) ids of a position with a min/max network, no branches.
// The table is derived from the bit vector + rank + CSR (the reference-shaped index), so results
// are identical by construction.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kFrontEmpty = 0xFFFFFFFFu;
constexpr uint32_t kFrontLongFlag = 0x10000u;
constexpr uint32_t kFrontMultiFlag = 0x20000u;
constexpr uint32_t kFrontKeyShift = 18;
constexpr uint32_t kFrontLim = 1u << kFrontKeyShift;  // slot ^ key < kFrontLim <=> same position
constexpr uint32_t kFrontChainBit = 0x80000000u;
constexpr uint32_t kFrontMaxShift = 13;
constexpr uint32_t kFrontInlineMax = 4;  // longest gene list stored inline

struct FrontGeom {
    uint32_t shift;     // log2(positions per bucket), 5..13
    uint32_t off_mask;  // (1 << shift) - 1
    uint64_t n_buckets;
    uint64_t n_entries;  // buckets + overflow records
    uint32_t stride;     // uint4s per entry: 1 = slots only, 2 = slots + anchors (extension)
    uint32_t pad;
};

// ---------------------------------------------------------------------------------------------
// Anchor-and-extend (exact; used when the front table is DRAM-sized).  Consecutive windows of a
// read that follows the reference need no hashing or table access to be resolved:
//   * every front-table entry becomes 32 bytes = one DRAM sector: its four slots + four anchors;
//     the anchor of a slot is the END position e (in the concatenated reference) of the first
//     reference window whose k-mer maps to the slot's filter position;
//   * ref2 holds the reference 2 bits per base (base x at bits 62-2*(x&31) of word (x>>5)+1), so
//     that the kernel can check that the read window IS that reference window (a read k-mer that
//     merely collides with the filter bit fails this test and is never extended);
//   * estream holds, per reference position t, a nibble {code:2, F0:1, F1:1} (position t at bits
//     4*(t&15) of word (t>>4)+1; word 0 and the tail are zero).  With E[e] = "the windows ending at
//     e-1 and e are both valid and their filter bits carry the same gene-id list":
//         F0[t] = E[t]      forward strand: the window ending at t-1 extends to the one ending at t
//         F1[t] = E[t+k]    reverse strand: the window starting at t+1 extends to the one starting at t
//     An anchored thread therefore resolves its next window with one nibble: base equal (or
//     complementary) and flag set => same k-mer as the next reference window => same filter bit
//     => same list as the window before.  Anything else falls back to the table lookup.
//   * coarse: one bit per 2^coarse_shift filter positions, set iff some position in the group is
//     set; L2-sized, so most misses never touch the DRAM-sized table.
// ---------------------------------------------------------------------------------------------
struct ExtGeom {
    uint64_t total;         // reference bases
    uint64_t estream_words; // total/16 + 3
    uint64_t ref2_words;    // total/32 + 3
    uint64_t coarse_words;  // ((bf_bits >> coarse_shift) + 31)/32 + 1
    uint32_t coarse_shift;
    uint32_t enabled;
};


__device__ __forceinline__ uint32_t front_key(uint32_t off) { return off << kFrontKeyShift; }
// key slot of offset `off` (either kind)?
__device__ __forceinline__ bool front_slot_matches(uint32_t slot, uint32_t key)
{
    return (slot ^ key) < kFrontLim;  // bit 31 clear and offset equal (EMPTY and chains have bit 31 set)
}
__device__ __forceinline__ bool front_is_chain(uint32_t slot) { return (slot & kFrontChainBit) && slot != kFrontEmpty; }

// k-mer (MSB-first, like the rolling forward k-mer) of the reference window ending at e
__device__ __forceinline__ uint64_t ref2_window(const uint64_t *ref2, uint32_t e, uint64_t kmask2, uint64_t pol)
{
    const uint32_t w = (e >> 5) + 1u, r = e & 31u;
    uint64_t lo, hi;
    asm volatile("ld.global.nc.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(lo) : "l"(ref2 + w), "l"(pol));
    asm volatile("ld.global.nc.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(hi) : "l"(ref2 + w - 1), "l"(pol));
    uint64_t v = lo >> (62u - 2u * r);
    if (r != 31u) v |= hi << (2u * r + 2u);
    return v & kmask2;
}

__device__ __forceinline__ uint4 ld_front(const uint4 *p, uint64_t pol)
{
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p), "l"(pol));
    return r;
}
// text words: keep the 128-byte line in L1 (the thread comes back for the next word), but let it
// leave L2 first
__device__ __forceinline__ uint32_t ld_text_word(const uint32_t *p, uint64_t pol_evict_first)
{
    uint32_t r;
    asm volatile("ld.global.nc.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol_evict_first));
    return r;
}

__device__ __forceinline__ uint64_t splitmix64(uint64_t x)
{
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}

}  // namespace shk
