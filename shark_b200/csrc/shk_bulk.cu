// Bulk classification of packed reads over the extension structures (K6b).  Replaces the same reference code as
// analyze_reads_kernel - ReadAnalyzer::operator() (ReadAnalyzer.hpp:39-110) behind FastqSplitter's masking
// (FastqSplitter.hpp:104-109, already folded into the validity bits of the packed form).  Every packed read takes this
// kernel whenever the index carries the extension structures (any table size; SHK_BULK=0 or SHK_F_EXTEND_OFF keep
// analyze_reads_kernel).  Citations are reference file:line.
//
// Why another kernel.  analyze_reads_kernel walks every read base by base and hashes every window, although most
// windows of a read that follows the reference are known without a hash; in its thread-per-read layout a warp pays for
// the union of its lanes' paths, so skipping hashes per lane buys nothing (profiles/analyze_r2.md).  Here the two halves
// of the work are separated and each runs in the layout that suits it:
//
//   * per read, 32 positions at a time (one lane = one read, one round = one 32-base word of every read of the warp):
//     validity runs -> the mask WV of valid windows (build_kmer's restart rule, kmer_utils.hpp:57-71); under the read's
//     current DIAGONAL (a hypothesis "read position q is reference position base +- q") the packed read word is XORed
//     with the packed reference word -> match mask -> D = windows that are, base for base, the reference window on the
//     diagonal -> S = D[p-1] & D[p] & E' = windows whose gene-id list is that of the window before (E: shk_device.cuh).
//     S needs no proof beyond itself: whatever the diagonal is, D says the two read windows ARE the two reference
//     windows, and E says those carry the same list.  The ids of a run of S windows are applied in O(1)
//     (cov += min(k, pos - last) + L - 1, hits += L; the reference's per-window update summed over the run).
//   * all windows that are valid but not S (WV & ~S: the windows covering a mismatch, the first window of a run,
//     every window of a read that follows no reference) are LOOKUPS, and the warp shares them evenly: the lookups of a
//     pass form one list (prefix sum over the lanes' counts), every lane takes an equal slice whoever owns the
//     windows, builds the k-mers from the owners' code words in shared memory (no rolling: a window is a funnel shift),
//     hashes, and tests the coarse filter (the word travels by cp.async while the next item is hashed).  Windows that
//     pass are queued in shared memory; the queue is served 32 entries at a time, one front-table load per lane.  Hits
//     go back to the owner through shared memory.
//   * a read without a working diagonal (the start of a mate, a chimera, an indel) asks for its first window alone
//     (pass 0).  A plain hit whose anchor names a reference window that IS the read's window (checked against refr,
//     either strand) gives the diagonal; the word and the one before are matched again, and only what is still
//     unexplained is looked up (pass 1).  A diagonal found in pass 1 re-matches the word as well, so that the owner
//     applies the hits it explains as one run.
//   * the owner applies hits and runs in window order to the 4-gene table (two hot genes in registers, two cold ones
//     in shared memory) and ends the read with the same code as analyze_reads_kernel (shk_reads.cuh).  Lists of 3 or 4
//     ids are walked by the owner itself; reads it cannot hold (more than 4 genes, a list of more than 4 ids, a run of
//     windows over lists of more than 2 ids, more than kMaxFastLen bases) go to the warp-per-read kernels as before.
//
// Results are those of the reference by construction: the ids of every valid window are either looked up in the exact
// front table or copied from the previous window under a condition that implies equality.
//
// Shape: 4 warps per CTA (one scan tile), 6 CTAs per SM (79 registers, 32 KB of shared memory per CTA).  The kernel is
// bound by instruction issue, by L2 / DRAM latency at 24 warps per SM, and by the instruction cache (38 KB of code:
// nothing in it is unrolled) - the trail of measurements behind each choice is profiles/analyze_r2.md, part 2.
#include "shk_internal.h"
#include "shk_reads.cuh"
#include "shk_scan.cuh"

#include <cstdlib>

namespace shk {

#ifndef SHK_BULK_MIN_BLOCKS
#define SHK_BULK_MIN_BLOCKS 6
#endif
constexpr int kBulkWarps = 4;
constexpr uint32_t kBulkComplex = 0xFFFFFFFEu;  // "ids of the previous window": a list of more than 2 ids
constexpr int kBulkThreads = kBulkWarps * 32;
constexpr uint32_t kBulkQueue = 64;  // ring: fewer than 32 entries wait while up to 32 are pushed
static_assert(kBulkThreads == (int)kReadsPerTile, "one CTA of the bulk kernel = one scan tile");

struct BulkWarp {
    uint64_t cprev[32];            // per lane: code words of the previous and of the current 32 positions of its read
    uint64_t ccur[32];
    unsigned long long cand[32];   // per lane: best diagonal candidate of the round {pos in word:31, strand:1, e:32}
    uint32_t need[32];             // per lane: windows of the round that must be looked up
    uint32_t pre[33];              // exclusive prefix sum of popc(need)
    uint32_t hit[32];              // per lane: looked-up windows that are set in the filter (plain lists)
    uint32_t res[32][32];          // [lane][(pos in word + lane) & 31]: ids of a hit, A | B << 16 (B == A: one id)
    uint32_t cplx[32];             // per lane: hits whose list has more than 2 ids (the owner walks the bucket itself)
    // queue of table loads (windows that passed the coarse filter): bucket, key, owner lane | position << 8
    uint32_t fq_bucket[kBulkQueue], fq_key[kBulkQueue];
    uint16_t fq_who[kBulkQueue];
    uint32_t cw[32];               // per lane: the coarse-filter word of its item in flight (cp.async)
    // owner state that is idle while the warp does lookups (registers there are resident CTAs)
    uint32_t prev_a[32], prev_b[32], last_ev[32];  // ids and end of the last window with ids
    uint16_t n_len[32], n_probes[32], n_hits[32], n_ext[32];  // at most kMaxFastLen each
};

// The per-gene table of the owner (Mru4, shk_reads.cuh) with its two older genes in shared memory: they are touched only
// when the read changes genes, and eight registers more per thread are one more resident CTA per SM.
struct BulkCold {
    uint32_t v[8][kBulkThreads];  // g2 c2 h2 l2 g3 c3 h3 l3, one column per thread
};
struct BulkTab {
    uint32_t g0, c0, h0, l0, g1, c1, h1, l1;
    uint32_t n;
    bool overflow;
    __device__ __forceinline__ void init(BulkCold &cold)
    {
        g0 = g1 = 0xFFFFFFFFu;
        c0 = c1 = h0 = h1 = l0 = l1 = 0u;
        n = 0;
        overflow = false;
        cold.v[0][threadIdx.x] = 0xFFFFFFFFu;
        cold.v[4][threadIdx.x] = 0xFFFFFFFFu;
    }
    __device__ __forceinline__ void hit(BulkCold &cold, uint32_t g, uint32_t pos, uint32_t k)
    {
        if (g == g0) {
            c0 += min(k, pos - l0);
            h0 += 1;
            l0 = pos;
        } else if (g == g1) {
            c1 += min(k, pos - l1);
            h1 += 1;
            l1 = pos;
        } else {
            other(cold, g, pos, k);
        }
    }
    __device__ __forceinline__ void more(uint32_t g, uint32_t d)
    {
        if (g == g0) {
            c0 += d, h0 += d, l0 += d;
        } else {
            c1 += d, h1 += d, l1 += d;
        }
    }
    // Mru4::other with slots 2 and 3 in shared memory
    __device__ __forceinline__ void other(BulkCold &cold,  // (never out of line: a call would put the table on the stack)
                                           uint32_t g, uint32_t pos, uint32_t k)
    {
        const uint32_t t = threadIdx.x;
        uint32_t c = k, h = 1;
        const uint32_t g2 = cold.v[0][t], c2 = cold.v[1][t], h2 = cold.v[2][t], l2 = cold.v[3][t];
        if (g == g2) {
            c = c2 + min(k, pos - l2);
            h = h2 + 1;
        } else {
            if (g == cold.v[4][t]) {
                c = cold.v[5][t] + min(k, pos - cold.v[7][t]);
                h = cold.v[6][t] + 1;
            } else {
                if (n == 4) {
                    overflow = true;
                    return;
                }
                ++n;
            }
            cold.v[4][t] = g2, cold.v[5][t] = c2, cold.v[6][t] = h2, cold.v[7][t] = l2;
        }
        cold.v[0][t] = g1, cold.v[1][t] = c1, cold.v[2][t] = h1, cold.v[3][t] = l1;
        g1 = g0, c1 = c0, h1 = h0, l1 = l0;
        g0 = g, c0 = c, h0 = h, l0 = pos;
    }
    __device__ __forceinline__ Mru4 full(const BulkCold &cold) const
    {
        const uint32_t t = threadIdx.x;
        Mru4 m;
        m.g0 = g0, m.c0 = c0, m.h0 = h0, m.l0 = l0, m.g1 = g1, m.c1 = c1, m.h1 = h1, m.l1 = l1;
        m.g2 = cold.v[0][t], m.c2 = cold.v[1][t], m.h2 = cold.v[2][t], m.l2 = cold.v[3][t];
        m.g3 = cold.v[4][t], m.c3 = cold.v[5][t], m.h3 = cold.v[6][t], m.l3 = cold.v[7][t];
        m.n = n, m.overflow = overflow;
        return m;
    }
};

// reverse the order of the 32 2-bit groups of a word
__device__ __forceinline__ uint64_t pair_reverse(uint64_t x)
{
    x = __brevll(x);
    return ((x >> 1) & 0x5555555555555555ULL) | ((x & 0x5555555555555555ULL) << 1);
}
// bits at even positions of x -> 16 contiguous bits
__device__ __forceinline__ uint32_t squeeze_even(uint32_t x)
{
    x &= 0x55555555u;
    x = (x | (x >> 1)) & 0x33333333u;
    x = (x | (x >> 2)) & 0x0F0F0F0Fu;
    x = (x | (x >> 4)) & 0x00FF00FFu;
    x = (x | (x >> 8)) & 0x0000FFFFu;
    return x;
}
// 32 2-bit groups -> one bit per group: group != 0
__device__ __forceinline__ uint32_t nonzero_pairs(uint64_t x)
{
    const uint64_t nz = x | (x >> 1);
    return squeeze_even((uint32_t)nz) | (squeeze_even((uint32_t)(nz >> 32)) << 16);
}
// bit i of the result: bits [32 + i - k + 1, 32 + i] of (prev : cur) are all set (k <= 32)
__device__ __forceinline__ uint32_t runs_ge(uint32_t prev, uint32_t cur, uint32_t k)
{
    uint64_t r = (uint64_t)prev | ((uint64_t)cur << 32);
    uint32_t have = 1;
    while (2u * have <= k) {  // runs of `have` -> runs of 2 * have
        r &= r << have;
        have *= 2u;
    }
    if (k > have) r &= r << (k - have);  // k - have <= have: the two runs overlap or touch
    return (uint32_t)(r >> 32);
}
// A read's diagonal: read position q <-> reference position base + q (forward) or base - q (reverse strand).
struct Diagonal {
    int64_t base;
    uint32_t dir;
    bool on;
};

// The words of refr / ebits that cover word w of a read under a diagonal, as loaded (the shifts wait until the values
// are used, so that the loads of the NEXT round can be issued before the lookups of this one).
struct RefRaw {
    uint64_t lo, hi;
    uint32_t elo, ehi;
};
__device__ __forceinline__ bool diag_t0(const ReadKernelArgs &a, const Diagonal &dg, uint32_t w, int64_t &t0)
{
    t0 = dg.dir ? dg.base - 32 * (int64_t)w - 31 : dg.base + 32 * (int64_t)w;
    // outside: the arrays have zero words around them, nothing there can match
    return dg.on && t0 >= -32 * (int64_t)kDerivedPad && t0 <= (int64_t)a.ref_total;
}
__device__ __forceinline__ void ref_fetch(const ReadKernelArgs &a, const Diagonal &dg, uint32_t w, uint32_t k, uint64_t pol,
                                          RefRaw &rw)
{
    int64_t t0;
    if (!diag_t0(a, dg, w, t0)) return;
    const uint64_t u = (uint64_t)(t0 + 32 * (int64_t)kDerivedPad), ue = dg.dir ? u + k : u;
    rw.lo = ld_u64_hint(a.refr + (u >> 5), pol);
    rw.hi = ld_u64_hint(a.refr + (u >> 5) + 1, pol);
    rw.elo = ld_u32_hint(a.ebits + (ue >> 5), pol);
    rw.ehi = ld_u32_hint(a.ebits + (ue >> 5) + 1, pol);
}
// Word w of a read under a diagonal: M = positions whose base is valid and equals the reference base (its complement
// on the reverse strand), E = the same-list flag of the window ENDING at each position (shk_device.cuh: forward E[e];
// reverse strand: the read window ending at q is the reference window ending at e = base - q + k - 1 and the window
// before it ends at e + 1, so the flag is E[e + 1]).
__device__ __forceinline__ void match_word(const ReadKernelArgs &a, const Diagonal &dg, uint32_t w, uint64_t C, uint32_t V,
                                           uint32_t k, const RefRaw &rw, uint32_t &M, uint32_t &E)
{
    M = 0u;
    E = 0u;
    int64_t t0;
    if (!diag_t0(a, dg, w, t0) || V == 0u) return;
    const uint64_t u = (uint64_t)(t0 + 32 * (int64_t)kDerivedPad);
    const uint32_t sh = 2u * ((uint32_t)u & 31u);
    uint64_t R = sh ? (rw.lo >> sh) | (rw.hi << (64u - sh)) : rw.lo;
    if (dg.dir) {
        R = pair_reverse(R) ^ 0xAAAAAAAAAAAAAAAAULL;  // complement of A0 C1 T2 G3 = code ^ 2
        E = __brev(__funnelshift_r(rw.elo, rw.ehi, ((uint32_t)u + k) & 31u));
    } else {
        E = __funnelshift_r(rw.elo, rw.ehi, (uint32_t)u & 31u);
    }
    M = V & ~nonzero_pairs(C ^ R);
}

// slots and anchors of a front-table entry (one 32-byte sector) in one load
__device__ __forceinline__ void ld_front_pair(const uint4 *p, uint64_t pol, uint4 &slots, uint4 &anchors)
{
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
                 : "=r"(slots.x), "=r"(slots.y), "=r"(slots.z), "=r"(slots.w), "=r"(anchors.x), "=r"(anchors.y),
                   "=r"(anchors.z), "=r"(anchors.w)
                 : "l"(p), "l"(pol));
}

// The k-mer of the window ENDING at position p of the current word (previous word : current word, LSB first), in the
// reference's code (A0 C1 G2 T3, kmer_utils.hpp:29-41): forward with the first base in the most significant group
// (kmer_utils.hpp:73-75) and its reverse complement (kmer_utils.hpp:47-55).
__device__ __forceinline__ void window_kmers(uint64_t lo, uint64_t hi, uint32_t p, uint32_t k, uint64_t kmask2, uint64_t &fwd,
                                             uint64_t &rcm)
{
    const uint32_t s2 = 2u * (33u + p - k);  // >= 4
    uint64_t X = s2 < 64u ? (lo >> s2) | (hi << (64u - s2)) : hi >> (s2 - 64u);
    X &= kmask2;
    X ^= (X >> 1) & 0x5555555555555555ULL;  // A0 C1 T2 G3 -> A0 C1 G2 T3
    rcm = ~X & kmask2;                       // LSB-first complement = the reverse complement, first base on top
    fwd = pair_reverse(X) >> (64u - 2u * k);
}

// One queued table load per lane: the position's ids go back to the owner of the window; a plain hit of an owner that
// is looking for a diagonal is verified against the reference (the slot's anchor names a reference window with the
// same filter bit; it gives a diagonal only if that window IS the read's window, either strand).
template <int MOD>
__device__ __forceinline__ void serve_queue(const ReadKernelArgs &a, BulkWarp &sh, uint32_t slot, bool valid, uint32_t want,
                                            uint32_t k, uint64_t kmask2, uint64_t pol_front, uint64_t pol_last)
{
    if (!valid) return;
    const uint32_t bucket = sh.fq_bucket[slot], kb = sh.fq_key[slot], who = sh.fq_who[slot];
    const uint32_t ow = who & 31u, p = who >> 8;
    const bool wanted = (want >> ow) & 1u;
    uint4 qq, anc = make_uint4(0u, 0u, 0u, 0u);
    if (wanted) ld_front_pair(a.front + (uint64_t)bucket * 2u, pol_front, qq, anc);  // the anchors sit in the same sector
    else qq = ld_front(a.front + (uint64_t)bucket * 2u, pol_front);
    uint32_t A, B, cur = bucket;
    for (;;) {  // the position's two smallest ids (slot - key; shk_device.cuh), along the bucket's chain
        const uint32_t d0 = qq.x - kb, d1 = qq.y - kb, d2 = qq.z - kb, d3 = qq.w - kb;
        const uint32_t lo01 = min(d0, d1), hi01 = max(d0, d1), lo23 = min(d2, d3), hi23 = max(d2, d3);
        A = min(lo01, lo23);
        B = min(max(lo01, lo23), min(hi01, hi23));
        if (A < kFrontLim || (int32_t)qq.w >= -1) break;
        cur = qq.w & 0x7FFFFFFFu;
        qq = ld_front(a.front + (uint64_t)cur * 2u, pol_front);
    }
    if (A >= kFrontLim) return;
    if (A < 0x10000u && (B < 0x10000u || B >= kFrontLim)) {  // a list of one or two ids
        sh.res[ow][(p + ow) & 31u] = A | ((B < 0x10000u ? B : A) << 16);
        atomicOr(&sh.hit[ow], 1u << p);
        if (wanted) {
            if (cur != bucket) anc = ld_front(a.front + (uint64_t)cur * 2u + 1u, pol_front);
            const uint32_t sa = A + kb;
            const uint32_t e = qq.x == sa ? anc.x : (qq.y == sa ? anc.y : (qq.z == sa ? anc.z : anc.w));
            // the reference window ending at e, from the same array the match words come from (one array less in L2)
            const uint64_t rwi = (uint64_t)(e >> 5) + kDerivedPad;
            uint64_t rk, rk_rc, fwd, rcm;
            window_kmers(ld_u64_hint(a.refr + rwi - 1, pol_last), ld_u64_hint(a.refr + rwi, pol_last), e & 31u, k, kmask2, rk, rk_rc);
            window_kmers(sh.cprev[ow], sh.ccur[ow], p, k, kmask2, fwd, rcm);
            if (rk == fwd) atomicMin(&sh.cand[ow], ((unsigned long long)p << 33) | e);
            else if (rk == rcm) atomicMin(&sh.cand[ow], ((unsigned long long)p << 33) | (1ULL << 32) | e);
        }
    } else {
        atomicOr(&sh.cplx[ow], 1u << p);  // 3 ids or more
    }
}

// SCORES: also store each settled read's score record (SHK_F_SCORES); the instantiations without it are the default path.
template <int MOD, bool SCORES>
__global__ void __launch_bounds__(kBulkThreads, SHK_BULK_MIN_BLOCKS)
analyze_bulk_kernel(const ReadKernelArgs a)
{
    __shared__ BulkWarp shared[kBulkWarps];
    __shared__ BulkCold cold;
    // (opaque to the compiler: under register pressure it would recompute both from %tid before every shared access)
    int lane = threadIdx.x & 31;
    uint32_t warp_in_cta = threadIdx.x >> 5;
    asm volatile("" : "+r"(lane), "+r"(warp_in_cta));
    BulkWarp &sh = shared[warp_in_cta];
    const uint32_t r = a.r0 + blockIdx.x * kBulkThreads + threadIdx.x;
    const uint32_t tile = a.r0 / kReadsPerTile + blockIdx.x;
    const uint64_t pol_first = a.pol_first, pol_last = a.pol_last;
    const uint64_t pol_front = pol_first;  // a DRAM-sized table must not displace the L2-resident arrays
    const uint32_t k = (uint32_t)a.k;
    const uint64_t kmask2 = (1ULL << (2 * k)) - 1ULL;
    const uint32_t fshift = a.fgeom.shift, fmask = a.fgeom.off_mask;

    uint32_t count = 0, payload = 0, my_loads = 0;
    bool slow = false;
    uint32_t n = 0, src0 = 0;
    if (r < a.r1) {
        const uint32_t off0 = a.off[r];
        n = a.off[r + 1] - off0;
        src0 = off0 - a.pack_base;
        if (n > kMaxFastLen) {
            slow = true;
            n = 0;
        }
    }
    const uint32_t my_words = (n + 31u) >> 5;
    const uint32_t rounds = __reduce_max_sync(kFull, my_words);
    // the read's words are loaded one round ahead: round w funnels words gi0 + w and gi0 + w + 1 of the packed stream
    const uint32_t gi0 = src0 >> 5, sb = src0 & 31u;
    uint64_t c_lo = 0, c_hi = 0;
    uint32_t v_lo = 0, v_hi = 0;
    if (my_words) {
        c_lo = ld_u64_hint(a.pcodes + gi0, pol_first), c_hi = ld_u64_hint(a.pcodes + gi0 + 1, pol_first);
        v_lo = ld_text_word(a.pvalid + gi0, pol_first), v_hi = ld_text_word(a.pvalid + gi0 + 1, pol_first);
    }

    BulkTab tab;
    tab.init(cold);
    Diagonal dg{0, 0u, false};
    RefRaw rw{0, 0, 0u, 0u};
    sh.ccur[lane] = 0;  // (the previous word's codes stay in shared memory between rounds)
    uint32_t prevV = 0, prevM = 0, prevDtop = 0;
    sh.prev_a[lane] = kFrontEmpty, sh.prev_b[lane] = kFrontEmpty, sh.last_ev[lane] = 0xFFFFFFF0u;
    sh.n_len[lane] = 0, sh.n_probes[lane] = 0, sh.n_hits[lane] = 0, sh.n_ext[lane] = 0;

    for (uint32_t w = 0; w < rounds; ++w) {
        // ---- the owner's word: validity runs, match runs under the diagonal, what has to be looked up ----
        const bool mine = w < my_words && !tab.overflow;
        uint64_t C = 0;
        uint32_t V = 0;
        if (mine) {
            C = sb ? (c_lo >> (2u * sb)) | (c_hi << (64u - 2u * sb)) : c_lo;
            V = __funnelshift_r(v_lo, v_hi, sb);
            const uint32_t rem = n - 32u * w;  // positions past the read belong to the next one
            if (rem < 32u) V &= (1u << rem) - 1u;
            c_lo = c_hi, v_lo = v_hi;
            if (w + 1u < my_words) {
                c_hi = ld_u64_hint(a.pcodes + gi0 + w + 2u, pol_first);
                v_hi = ld_text_word(a.pvalid + gi0 + w + 2u, pol_first);
            }
        }
        const uint32_t WV = runs_ge(prevV, V, k);
        sh.n_len[lane] += __popc(V);  // ReadAnalyzer.hpp:46-49
        sh.n_probes[lane] += __popc(WV);
        uint32_t M, E;
        match_word(a, dg, w, C, V, k, rw, M, E);
        if (!mine) M = 0u;
        if (mine && w + 1u < my_words) ref_fetch(a, dg, w + 1u, k, pol_last, rw);  // for the next round, unless the diagonal changes
        uint32_t D = runs_ge(prevM, M, k);
        uint32_t S = D & ((D << 1) | prevDtop) & E;
        const uint32_t need = WV & ~S;
        // A read whose diagonal explains nothing in this word takes the anchor of its first plain hit as the next one.
        // It asks for its first window alone (pass 0) and, when that gives a diagonal, matches the word again before
        // the rest is looked up (pass 1) - otherwise every window of the word in which a mate starts would be a lookup.
        bool want_me = WV != 0u && S == 0u;
        uint32_t now = want_me ? need & (0u - need) : need, later = need & ~now;

        sh.cprev[lane] = sh.ccur[lane];
        sh.ccur[lane] = C;
        sh.hit[lane] = 0u;
        sh.cplx[lane] = 0u;
        sh.cand[lane] = ~0ULL;
        for (int pass = 0;; ++pass) {
            sh.need[lane] = now;
            const uint32_t incl = warp_incl_scan((uint32_t)__popc(now), lane);
            sh.pre[lane + 1] = incl;
            if (lane == 0) sh.pre[0] = 0u;
            const uint32_t total = __shfl_sync(kFull, incl, 31);
            const uint32_t want = __ballot_sync(kFull, want_me), nz = __ballot_sync(kFull, now != 0u);
            __syncwarp();

            // ---- the warp's lookups, an equal slice per lane ----
            if (total) {
                const uint32_t per = (total + 31u) >> 5;
                const uint32_t i0 = min(total, (uint32_t)lane * per), i1 = min(total, i0 + per);
                uint32_t left = i1 - i0, o = 0, m = 0;
                if (left) {
#pragma unroll
                    for (uint32_t s = 16; s; s >>= 1)  // the largest o with pre[o] <= i0: the owner of item i0
                        if (sh.pre[o + s] <= i0) o += s;
                    m = sh.need[o];
                    uint32_t j = i0 - sh.pre[o], at = 0, mm = m;  // drop the j lowest set bits of m
#pragma unroll
                    for (uint32_t s = 16; s; s >>= 1) {
                        const uint32_t c = __popc(mm & ((1u << s) - 1u));
                        if (j >= c) {
                            j -= c;
                            mm >>= s;
                            at += s;
                        }
                    }
                    m &= ~0u << at;
                }
                // Windows that pass the coarse filter queue up for the DRAM-sized table; the queue is served 32 entries at a
                // time, one per lane, so that a warp waits for DRAM once per 32 table loads and probes with every lane.
                uint32_t fq_head = 0, fq_n = 0;  // warp-uniform
                // One item per iteration, its coarse word in flight while the next item is hashed (no unrolling: the
                // kernel is bound by latency AND by the instruction cache, profiles/analyze_r2.md).
                // (The coarse word travels by cp.async into the lane's own shared-memory slot: ptxas does not keep a
                // register load in flight across the loop's back edge, an asynchronous copy has no register to wait on.)
                uint32_t q_bucket = 0, q_key = 0, q_who = 0, q_bit = 0;
                bool q_has = false;
                const uint32_t cw_slot = (uint32_t)__cvta_generic_to_shared(&sh.cw[lane]);
                for (uint32_t it = 0; it <= per; ++it) {  // same trip count in every lane
                    // the next item is hashed while the coarse word of the one before is in flight
                    uint32_t n_bucket = 0, n_key = 0, n_who = 0, n_bit = 0;
                    const uint32_t *n_addr = nullptr;
                    if (it < per && left) {
                        while (m == 0u) {  // the next owner that asks for anything
                            o = (uint32_t)__ffs(nz & (0xFFFFFFFEu << o)) - 1u;
                            m = sh.need[o];
                        }
                        const uint32_t p = (uint32_t)__ffs(m) - 1u;
                        m &= m - 1u;
                        --left;
                        uint64_t fwd, rcm;
                        window_kmers(sh.cprev[o], sh.ccur[o], p, k, kmask2, fwd, rcm);
                        const uint64_t pb = bit_index<MOD>(xxh64_u64(fwd < rcm ? fwd : rcm), a.geom);
                        n_bucket = (uint32_t)(pb >> fshift);
                        n_key = front_key((uint32_t)pb & fmask);
                        const uint32_t cidx = (n_bucket << a.coarse_rel) | (n_key >> a.coarse_key_shift);
                        n_bit = cidx & 31u;
                        n_who = o | (p << 8);
                        n_addr = a.coarse + (cidx >> 5);
                    }
                    bool push = false;
                    if (q_has) {
                        asm volatile("cp.async.wait_all;" ::: "memory");
                        push = (sh.cw[lane] >> q_bit) & 1u;
                    }
                    const uint32_t pm = __ballot_sync(kFull, push);
                    if (push) {
                        const uint32_t slot = (fq_head + fq_n + (uint32_t)__popc(pm & ((1u << lane) - 1u))) & (kBulkQueue - 1u);
                        sh.fq_bucket[slot] = q_bucket;
                        sh.fq_key[slot] = q_key;
                        sh.fq_who[slot] = (uint16_t)q_who;
                        ++my_loads;
                    }
                    fq_n += (uint32_t)__popc(pm);
                    if (fq_n >= 32u) {
                        __syncwarp();
                        serve_queue<MOD>(a, sh, (fq_head + (uint32_t)lane) & (kBulkQueue - 1u), true, want, k, kmask2, pol_front, pol_last);
                        __syncwarp();
                        fq_head = (fq_head + 32u) & (kBulkQueue - 1u);
                        fq_n -= 32u;
                    }
                    q_bucket = n_bucket, q_key = n_key, q_who = n_who, q_bit = n_bit;
                    q_has = n_addr != nullptr;
                    if (q_has) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(cw_slot), "l"(n_addr) : "memory");
                }
                if (fq_n) {
                    __syncwarp();
                    serve_queue<MOD>(a, sh, (fq_head + (uint32_t)lane) & (kBulkQueue - 1u), (uint32_t)lane < fq_n, want, k, kmask2, pol_front, pol_last);
                }
            }
            __syncwarp();
            if (want_me) {
                const unsigned long long cd = sh.cand[lane];
                if (cd != ~0ULL) {
                    // A diagonal: the word (and the windows reaching back into the word before) is matched again.  After
                    // pass 0 the runs it explains are no longer looked up; after pass 1 they already were, but the
                    // owner still applies them as runs (a run clears the hits it covers) instead of window by window.
                    const uint32_t e = (uint32_t)cd, pos = 32u * w + (uint32_t)(cd >> 33);
                    dg.on = true;
                    dg.dir = (uint32_t)(cd >> 32) & 1u;
                    dg.base = dg.dir ? (int64_t)e - (int64_t)k + 1 + (int64_t)pos : (int64_t)e - (int64_t)pos;
                    uint32_t pm = 0u, E2;
                    if (w) {
                        ref_fetch(a, dg, w - 1u, k, pol_last, rw);
                        match_word(a, dg, w - 1u, sh.cprev[lane], prevV, k, rw, pm, E2);
                    }
                    ref_fetch(a, dg, w, k, pol_last, rw);
                    match_word(a, dg, w, sh.ccur[lane], V, k, rw, M, E2);
                    if (w + 1u < my_words) ref_fetch(a, dg, w + 1u, k, pol_last, rw);
                    D = runs_ge(pm, M, k);
                    S = D & (D << 1) & E2;  // (nothing is known about the last window of the word before)
                    later = WV & ~S & ~now;
                    want_me = false;
                    sh.cand[lane] = ~0ULL;
                }
            }
            if (pass == 1) break;
            now = later;
            later = 0u;
            if (!__any_sync(kFull, now != 0u)) break;
        }

        // ---- the owner applies hits and runs in window order (ReadAnalyzer.hpp:56-62, 79-86) ----
        if (mine) {
            const uint32_t cplx = sh.cplx[lane];
            uint32_t prevA = sh.prev_a[lane], prevB = sh.prev_b[lane], last_ev = sh.last_ev[lane], my_hits = 0, my_ext = 0;
            uint32_t ev = sh.hit[lane] | cplx | S;
            while (ev && !tab.overflow) {
                const uint32_t p = (uint32_t)__ffs(ev) - 1u, pos = 32u * w + p;
                uint32_t A, B, L;
                if ((S >> p) & 1u) {  // a run of windows with the ids of the window before
                    const uint32_t rest = ~(S >> p);
                    L = rest ? (uint32_t)__ffs(rest) - 1u : 32u;
                    const bool cont = last_ev + 1u == pos;  // (a window without ids before it: none here either)
                    A = cont ? prevA : kFrontEmpty;
                    B = cont ? prevB : kFrontEmpty;
                    my_ext += L;
                    if (cont && prevA == kBulkComplex) {  // a run of lists of 3 ids or more: not held here
                        tab.overflow = true;
                        break;
                    }
                } else if ((cplx >> p) & 1u) {
                    // a list of 3 or 4 ids (or a longer one: exact path): every slot of the bucket and of its chain, in
                    // list order, as analyze_reads_kernel's generic path does
                    const uint32_t s2 = 2u * (33u + p - k);
                    const uint64_t pc = sh.cprev[lane], cc = sh.ccur[lane];
                    uint64_t X = s2 < 64u ? (pc >> s2) | (cc << (64u - s2)) : cc >> (s2 - 64u);
                    X &= kmask2;
                    X ^= (X >> 1) & 0x5555555555555555ULL;
                    const uint64_t rcx = ~X & kmask2, fwx = pair_reverse(X) >> (64u - 2u * k);
                    const uint64_t pb = bit_index<MOD>(xxh64_u64(fwx < rcx ? fwx : rcx), a.geom);
                    const uint32_t kb = front_key((uint32_t)pb & fmask);
                    uint4 qq = ld_front(a.front + (pb >> fshift) * 2u, pol_front);
                    for (;;) {
#pragma unroll 1
                        for (int i = 0; i < 4; ++i) {
                            const uint32_t sl = i == 0 ? qq.x : (i == 1 ? qq.y : (i == 2 ? qq.z : qq.w));
                            const uint32_t d = sl ^ kb;
                            if (d < kFrontLim) {
                                if (d & kFrontLongFlag) tab.overflow = true;
                                else tab.hit(cold, d & 0xFFFFu, pos, k);
                            }
                        }
                        if (!front_is_chain(qq.w)) break;
                        qq = ld_front(a.front + (uint64_t)(qq.w & 0x7FFFFFFFu) * 2u, pol_front);
                    }
                    my_hits += 1u;
                    prevA = kBulkComplex, prevB = kFrontEmpty, last_ev = pos;
                    ev &= ev - 1u;
                    continue;
                } else {
                    const uint32_t rr = sh.res[lane][(p + (uint32_t)lane) & 31u];
                    A = rr & 0xFFFFu;
                    B = rr >> 16;
                    if (B == A) B = kFrontEmpty;
                    // ... and the run of windows with the same ids that follows it, in one step
                    const uint32_t run = p < 31u ? (uint32_t)__ffs(~(S >> (p + 1u))) - 1u : 0u;
                    L = 1u + run;
                    my_ext += run;
                }
                ev &= ~(((L < 32u ? (1u << L) : 0u) - 1u) << p);
                if (A != kFrontEmpty) {
                    my_hits += L;
                    const bool hasB = B != kFrontEmpty;
                    const bool a0 = A == tab.g0, a1 = A == tab.g1, b0 = hasB && B == tab.g0, b1 = hasB && B == tab.g1;
                    if ((a0 | a1) & (!hasB | b0 | b1)) {
                        if (a0 | b0) {
                            tab.c0 += min(k, pos - tab.l0) + (L - 1u);
                            tab.h0 += L;
                            tab.l0 = pos + L - 1u;
                        }
                        if (a1 | b1) {
                            tab.c1 += min(k, pos - tab.l1) + (L - 1u);
                            tab.h1 += L;
                            tab.l1 = pos + L - 1u;
                        }
                    } else {
                        tab.hit(cold, A, pos, k);
                        if (!tab.overflow) tab.more(A, L - 1u);
                        if (hasB && !tab.overflow) {
                            tab.hit(cold, B, pos, k);
                            if (!tab.overflow) tab.more(B, L - 1u);
                        }
                    }
                    prevA = A;
                    prevB = B;
                    last_ev = pos + L - 1u;
                }
            }
            sh.prev_a[lane] = prevA, sh.prev_b[lane] = prevB, sh.last_ev[lane] = last_ev;
            sh.n_hits[lane] += my_hits, sh.n_ext[lane] += my_ext;
        }
        prevV = V;
        prevM = M;
        prevDtop = D >> 31;
    }

    if (r < a.r1) {
        if (tab.overflow) slow = true;
        if (slow) {
            count = 0, payload = 0;
            sh.n_probes[lane] = 0, sh.n_hits[lane] = 0;  // counted by the kernel that classifies the read
            a.slow_list[atomicAdd(&a.counters->n_slow, 1u)] = r;
        } else {
            uint4 score;
            finish_read(a, tab.full(cold), sh.n_len[lane], count, payload, score);
            if (SCORES) a.scores[r] = score;  // (a slow read's record comes from the kernel that settles it)
        }
        a.rec[r] = make_uint2(count, payload);
    }
    flush_warp_counters<true>(a, tile, lane, count, payload, sh.n_probes[lane], sh.n_hits[lane], sh.n_ext[lane], my_loads);
}

// SHK_BULK=1 sends packed reads to this kernel, SHK_BULK=0 keeps them on analyze_reads_kernel<EXT, PACKED> (A/B
// measurements, tests of both kernels); unset = kBulkDefault.
constexpr bool kBulkDefault = true;
bool bulk_enabled()
{
    const char *e = std::getenv("SHK_BULK");
    if (!e || !e[0]) return kBulkDefault;
    return e[0] != '0';
}

template <bool SCORES>
void launch_bulk_kernel(const ReadKernelArgs &a, cudaStream_t st, unsigned blocks)
{
    switch (a.geom.mod_kind) {
    case MOD_POW2: analyze_bulk_kernel<MOD_POW2, SCORES><<<blocks, kBulkThreads, 0, st>>>(a); break;
    case MOD_B33: analyze_bulk_kernel<MOD_B33, SCORES><<<blocks, kBulkThreads, 0, st>>>(a); break;
    default: analyze_bulk_kernel<MOD_GENERIC, SCORES><<<blocks, kBulkThreads, 0, st>>>(a); break;
    }
}
template void launch_bulk_kernel<false>(const ReadKernelArgs &, cudaStream_t, unsigned);
template void launch_bulk_kernel<true>(const ReadKernelArgs &, cudaStream_t, unsigned);

}  // namespace shk
