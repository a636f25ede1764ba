// Pieces shared by the classification kernels (shk_reads.cu, shk_bulk.cu): the register-resident per-gene table of
// the thread-per-read kernels, the reporting rule (threshold, -s), the end of a read (arg-max, rule) and the counter
// flush of the thread-per-read kernels.  Citations are reference file:line.
#pragma once
#include "shk_internal.h"

namespace shk {

constexpr uint32_t kFull = 0xFFFFFFFFu;

// Does a read's result fit the compact per-read form (one 16-bit word), or does it go to the `multi` list?
// (With 32-bit gene ids - SHK_F_WIDE_IDS - every reported read goes to the list.)
__device__ __forceinline__ uint32_t multi_entries(uint32_t count, uint32_t payload, uint32_t wide = 0u)
{
    return (count >= 2u || (count == 1u && (payload >= SHK_GENE_MULTI || wide))) ? count : 0u;
}

// The per-gene state of ReadAnalyzer's std::map (ReadAnalyzer.hpp:52-62,79-86) for reads that touch at most four
// genes, most recent genes first.
struct Mru4 {
    uint32_t g0, c0, h0, l0, g1, c1, h1, l1, g2, c2, h2, l2, g3, c3, h3, l3;
    uint32_t n;
    bool overflow;
    __device__ __forceinline__ void init()
    {
        g0 = g1 = g2 = g3 = 0xFFFFFFFFu;
        c0 = c1 = c2 = c3 = h0 = h1 = h2 = h3 = l0 = l1 = l2 = l3 = 0u;
        n = 0;
        overflow = false;
    }
    // ReadAnalyzer.hpp:57-61 / 80-85.  A fresh std::map entry has last == 0 and `pos - 0 >= k`
    // for every window, so its coverage starts at k.
    __device__ __forceinline__ void hit(uint32_t g, uint32_t pos, uint32_t k)
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
            other(g, pos, k);
        }
    }
    // `d` more consecutive windows of a gene hit() has just seen (it sits in slot 0 or 1): each adds min(k, 1) = 1
    __device__ __forceinline__ void more(uint32_t g, uint32_t d)
    {
        if (g == g0) {
            c0 += d, h0 += d, l0 += d;
        } else {
            c1 += d, h1 += d, l1 += d;
        }
    }
    __device__ __forceinline__ void other(uint32_t g, uint32_t pos, uint32_t k)
    {
        uint32_t c = k, h = 1;
        if (g == g2) {
            c = c2 + min(k, pos - l2);
            h = h2 + 1;
        } else if (g == g3) {
            c = c3 + min(k, pos - l3);
            h = h3 + 1;
            g3 = g2, c3 = c2, h3 = h2, l3 = l2;
        } else {
            if (n == 4) {
                overflow = true;
                return;
            }
            ++n;
            g3 = g2, c3 = c2, h3 = h2, l3 = l2;  // slot 3 was free
        }
        g2 = g1, c2 = c1, h2 = h1, l2 = l1;
        g1 = g0, c1 = c0, h1 = h0, l1 = l0;
        g0 = g, c0 = c, h0 = h, l0 = pos;
    }
};

// Threshold and -s (ReadAnalyzer.hpp:104) for a read whose best genes have coverage `cov` and number `n_best`: is it
// reported (with n_best associations)?  This is the rule the score records promise (INTEGRATION.md §3); `c * len` is
// rounded as the reference's double product.  (No test of cov > 0: every gene in a table has cov >= k >= 1, so
// n_best > 0 implies it.)
__device__ __forceinline__ bool read_reported(const ReadKernelArgs &a, uint32_t cov, uint32_t len, uint32_t n_best)
{
    return n_best > 0 && (double)cov >= __dmul_rn(a.c, (double)len) && (!a.single || n_best == 1);
}

// argmax with ties (ReadAnalyzer.hpp:90-102), then read_reported: -> {count, gene | pool offset},
// and the read's score record {len, cov, hits, n_best} (SHK_F_SCORES; dead code for the kernels that do not store it)
__device__ __forceinline__ void finish_read(const ReadKernelArgs &a, const Mru4 &tab, uint32_t len, uint32_t &count,
                                            uint32_t &payload, uint4 &score)
{
    const uint32_t tg[4] = {tab.g0, tab.g1, tab.g2, tab.g3}, tc[4] = {tab.c0, tab.c1, tab.c2, tab.c3},
                   th[4] = {tab.h0, tab.h1, tab.h2, tab.h3};
    uint32_t maxc = 0, maxh = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        if ((uint32_t)i < tab.n && (tc[i] > maxc || (tc[i] == maxc && th[i] > maxh))) {
            maxc = tc[i];
            maxh = th[i];
        }
    }
    uint32_t wg[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const bool is = (uint32_t)i < tab.n && tc[i] == maxc && th[i] == maxh;
        wg[i] = is ? tg[i] : 0xFFFFFFFFu;
        count += is ? 1u : 0u;
    }
    score = make_uint4(len, maxc, maxh, count);
    if (!read_reported(a, maxc, len, count)) count = 0;
    if (count == 1) {
        payload = min(min(wg[0], wg[1]), min(wg[2], wg[3]));
    } else if (count >= 2) {
        // ascending gene order = std::map order: sort the (at most 4) winners
#define SHK_CSWAP(x, y) { const uint32_t lo_ = min(wg[x], wg[y]), hi_ = max(wg[x], wg[y]); wg[x] = lo_; wg[y] = hi_; }
        SHK_CSWAP(0, 1) SHK_CSWAP(2, 3) SHK_CSWAP(0, 2) SHK_CSWAP(1, 3) SHK_CSWAP(1, 2)
#undef SHK_CSWAP
        payload = atomicAdd(&a.counters->pool_used, count);
        if ((uint64_t)payload + count > a.pool_cap) {
            a.counters->pool_overflow = 1;
            payload = 0xFFFFFFFFu;
        } else {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if ((uint32_t)i < count) a.pool[payload + i] = wg[i];
        }
    }
}

// End of the thread-per-read kernels (K6, K6b): the warp's reads go into the chunk's counters and its multi entries into
// tile_sums, which is zeroed before the launch.  Every warp retires on its own: no warp of a CTA waits at a barrier for
// its slowest sibling.  EXT: also the anchor-and-extend counters.
template <bool EXT>
__device__ __forceinline__ void flush_warp_counters(const ReadKernelArgs &a, uint32_t tile, int lane, uint32_t count,
                                                    uint32_t payload, uint32_t probes, uint32_t hits, uint32_t ext,
                                                    uint32_t loads)
{
    const uint32_t wa = __reduce_add_sync(kFull, count), wp = __reduce_add_sync(kFull, probes),
                   wh = __reduce_add_sync(kFull, hits), wm = __reduce_add_sync(kFull, multi_entries(count, payload)),
                   wk = __popc(__ballot_sync(kFull, count != 0u));
    if (lane == 0) {
        if (wm) atomicAdd(&a.tile_sums[tile], wm);
        if (wa) atomicAdd(&a.counters->n_assoc, (unsigned long long)wa);
        if (wk) atomicAdd(&a.counters->n_kept, (unsigned long long)wk);
        if (wp) atomicAdd(&a.counters->n_probes, (unsigned long long)wp);
        if (wh) atomicAdd(&a.counters->n_hits, (unsigned long long)wh);
    }
    if (EXT) {
        const uint32_t we = __reduce_add_sync(kFull, ext), wl = __reduce_add_sync(kFull, loads);
        if (lane == 0) {
            if (we) atomicAdd(&a.counters->n_extended, (unsigned long long)we);
            if (wl) atomicAdd(&a.counters->n_table_loads, (unsigned long long)wl);
        }
    }
}

}  // namespace shk
