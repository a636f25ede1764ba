"""GPU: every index view word for word against a host restatement, on every route by which an index reaches a context.

The classification kernels read the index through eight device arrays (shk_index_views_get, in the order shk_index_save
writes them): 0 the filter sectors with the rank directory in word 7, 1 the 8-byte entries, 2 the CSR offsets, 3 the CSR
ids, 4 the front table (slots, chain pointers and, with extension, anchors), 5 estream (2-bit base code + F0/F1 per
position), 6 ref2 (2 bits per base), 7 the coarse miss filter.  Several faults in views 4-7 change no classification
result (an anchor other than the first window end, a cleared extension flag, an extra coarse bit) or change it only for
the reads that meet one position (a 2-id list that straddles two records of a chain, a flag set by mistake, a missing
coarse bit), so they are checked here directly.

Each view is read from a file written by shk_index_save (header restated as a ctypes structure) and compared with a
numpy restatement built from the reference and the oracle's index (set bits, offsets, ids).  Placement inside a
front-table bucket follows the order of the build's atomics, so view 4 is decoded into groups of slots and checked for
everything that is determined: record counts, chain pointers, each set bit's group of slots, anchors, the rule that a
2-id group never straddles two records, and where padding may sit.  The word `entries[n_set]` is allocated but never
written, so it is left out of every comparison between builds.

Routes: the one-call build with extension forced on, automatic and forced off; the staged functor protocol; the sharded
build with 1, 2 and 3 contexts (on one device they share it); shk_index_load; shk_index_replicate.  References reach
the build's edges: lists at the 48/49 raw-occurrence switch between insertion sort and the 65 536-bit bitmap, all 65 536
gene indices with ids on the bitmap's word boundaries, k = 1 and 2, a dense filter with long chains, and filter sizes
on the edges of the scan tiles.  Each design is asserted (floors printed) before it is used."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import pyoracle as po
from shark_b200 import capi
from test_functors import _staged_build
from test_gpu_bulk import rc
from test_gpu_parity import ACGT
from test_gpu_shard import _close, _sharks

pytestmark = pytest.mark.gpu

EMPTY = 0xFFFFFFFF
CHAIN = 0x80000000
K_SHORT_LIST = 48      # sort_unique_kernel: longer raw lists take the bitmap kernel
SCAN_TILE = 4096       # kScanTile


class FileHeader(C.Structure):
    """IndexFileHeader of shk_capi.cu"""
    _fields_ = [("magic", C.c_char * 8), ("abi", C.c_uint32), ("k", C.c_uint32), ("bf_bits", C.c_uint64),
                ("view_bytes", C.c_uint64 * 8), ("checksum", C.c_uint64), ("info", capi.IndexInfo)]


def _shark(**kw):
    from shark_b200.engine import Shark
    kw.setdefault("max_reads_per_chunk", 1 << 10)
    return Shark(**kw)


def saved_views(sh, path):
    """save_index -> (header, [view 0 … 7 as uint8 arrays]); the sizes must be those shk_index_views_get reports."""
    sh.save_index(path)
    raw = np.memmap(path, dtype=np.uint8, mode="r")
    hs = C.sizeof(FileHeader)
    h = FileHeader.from_buffer_copy(bytes(raw[:hs]))
    assert h.magic == b"SHKIDX" and h.abi == sh.lib.shk_abi_version() and h.k == sh.k and h.bf_bits == sh.bf_bits
    vb = [int(x) for x in h.view_bytes]
    assert vb == [int(x) for x in sh.index_views().bytes]
    assert len(raw) == hs + sum(vb)
    out, a = [], hs
    for n in vb:
        out.append(raw[a:a + n])
        a += n
    return h, out


def xxh64(v):
    """XXH64 of one 8-byte word, seed 0 (the closed form of shk_device.cuh), vectorised"""
    P1, P2, P3, P4, P5 = (np.uint64(x) for x in (11400714785074694791, 14029467366897019727, 1609587929392839161,
                                                 9650029242287828579, 2870177450012600261))
    rotl = lambda x, r: (x << np.uint64(r)) | (x >> np.uint64(64 - r))
    v = np.asarray(v, np.uint64)
    with np.errstate(over="ignore"):
        h = np.full(v.shape, P5 + np.uint64(8), np.uint64)
        h ^= rotl(v * P2, 31) * P1
        h = rotl(h, 27) * P1 + P4
        h ^= h >> np.uint64(33)
        h *= P2
        h ^= h >> np.uint64(29)
        h *= P3
        h ^= h >> np.uint64(32)
    return h


CODE = np.zeros(256, np.uint64)
for _c, _v in zip(b"ACGTacgt", (0, 1, 2, 3, 0, 1, 2, 3)):
    CODE[_c] = _v


class Restated:
    """The reference, its windows and the oracle's index: everything the views are derived from."""

    def __init__(self, name, records, k, bf_bits, wide=False):
        self.name, self.records, self.k, self.bf_bits = name, records, k, bf_bits
        self.bases, self.rec_off = po.concat_records(records)
        self.total = len(self.bases)
        ora = po.Index(self.bases, self.rec_off, k, bf_bits, wide=wide)
        self.n_genes = ora.n_genes
        self.pos = ora.pos.astype(np.uint64)
        self.off = ora.off.astype(np.int64)
        self.ids = (ora.ids32 if wide else ora.ids).astype(np.int64)
        self.n_set = len(self.pos)
        # windows record by record; gene index = the reference's nidx (a record of length >= k without a window
        # consumes none)
        canon, ends, gene, nidx, g = [], [], [], [], 0
        for r, s in enumerate(records):
            e = po.enumerate_kmers(s, k) if len(s) >= k else (np.zeros(0, np.uint64), np.zeros(0, np.int64))
            if e is None:
                nidx.append(-1)
                continue
            nidx.append(g)
            canon.append(e[0])
            ends.append(e[1] + int(self.rec_off[r]))
            gene.append(np.full(len(e[0]), g, np.int64))
            g += 1
        assert g == self.n_genes
        self.nidx = np.array(nidx, np.int64)
        self.canon = np.concatenate(canon) if canon else np.zeros(0, np.uint64)
        self.ends = np.concatenate(ends) if ends else np.zeros(0, np.int64)
        self.gene = np.concatenate(gene) if gene else np.zeros(0, np.int64)
        sample = np.unique(np.linspace(0, max(len(self.canon) - 1, 0), 64).astype(np.int64))
        h = xxh64(self.canon)
        if len(self.canon):
            assert all(int(h[i]) == po.xxh64_u64(int(self.canon[i])) for i in sample)
        p = h % np.uint64(bf_bits)
        self.rank = np.searchsorted(self.pos, p).astype(np.int64)
        assert (self.rank < self.n_set).all() and (self.pos[np.minimum(self.rank, self.n_set - 1)] == p).all()
        self.raw = np.bincount(self.rank, minlength=self.n_set)
        self.win = np.full(self.total, -1, np.int64)
        self.win[self.ends] = self.rank

    def lens(self, off=None):
        return np.diff(self.off if off is None else off)


# ------------------------------------------------------------------------------------------- expected views
def check_sectors(R, v0):
    words = np.frombuffer(v0, np.uint32)
    n_sec = ((R.bf_bits + 31) // 32 + 6) // 7
    assert len(words) == n_sec * 8
    F = words.reshape(n_sec, 8)
    q = (R.pos >> np.uint64(5)).astype(np.int64)
    uq, inv = np.unique(q, return_inverse=True)
    want = np.zeros(len(uq), np.uint32)
    np.bitwise_or.at(want, inv, (np.uint32(1) << (R.pos & np.uint64(31)).astype(np.uint32)))
    assert np.array_equal(F[uq // 7, uq % 7], want)
    sec_of = R.pos // np.uint64(224)
    nz = 0
    for s0 in range(0, n_sec, 1 << 24):  # piecewise: a b * 2^33 filter has 10^8 sectors
        s1 = min(n_sec, s0 + (1 << 24))
        blk = np.asarray(F[s0:s1])
        nz += np.count_nonzero(blk[:, :7])
        assert np.array_equal(blk[:, 7], np.searchsorted(sec_of, np.arange(s0, s1, dtype=np.uint64)).astype(np.uint32))
    assert nz == len(uq)  # no other filter word has a bit: none at or beyond bf_bits in the last sector


def expected_entries(off, ids, wide):
    ln = np.diff(off)
    idx = np.append(ids, [0, 0]).astype(np.uint64)
    b = off[:-1]
    id0, id1 = idx[np.minimum(b, len(ids))], idx[np.minimum(b + 1, len(ids) + 1)]
    lm1 = np.maximum(ln - 1, 0).astype(np.uint64)
    if wide:
        e = (lm1 << np.uint64(32)) | np.where(ln == 1, id0, b.astype(np.uint64))
    else:
        lo = np.where(ln == 1, np.uint64(0), np.where(ln == 2, id1, b.astype(np.uint64)))
        e = (id0 << np.uint64(48)) | (lm1 << np.uint64(32)) | lo
    return np.where(ln == 0, np.uint64(0), e)


def front_counts(pos, ln, shift, bf_bits):
    nb = (bf_bits + (1 << shift) - 1) >> shift
    bkt = (pos >> np.uint64(shift)).astype(np.int64)
    L = np.where(ln <= 4, ln, 1)
    slots = np.bincount(bkt, weights=L, minlength=nb).astype(np.int64)
    n2 = np.bincount(bkt, weights=(ln == 2), minlength=nb).astype(np.int64)
    records = np.where(slots <= 4, 0, (slots + n2 - 3 + 2) // 3)
    return nb, slots, records


def decode_front(R, v4, info, off, ids, stats):
    """Checks view 4 against the restatement; returns its canonical form (placement order removed)."""
    shift, stride = info.front_shift, (2 if info.extend else 1)
    wpe = 4 * stride
    T = np.frombuffer(v4, np.uint32)
    ln = np.diff(off)
    nb, slots, records = front_counts(R.pos, ln, shift, R.bf_bits)
    assert info.front_entries == nb + records.sum() and len(T) == info.front_entries * wpe
    rb = np.concatenate([[0], np.cumsum(records)[:-1]]).astype(np.int64)
    chained = records > 0
    # chain pointers: slot 3 of a chained bucket and of every record but the last; the last record's slot 3 is empty
    cb = np.nonzero(chained)[0]
    assert np.array_equal(T[cb * wpe + 3], (CHAIN | (nb + rb[cb])).astype(np.uint32))
    rec_of = np.repeat(cb, records[cb])
    ri = np.arange(len(rec_of)) - np.repeat(np.cumsum(records[cb]) - records[cb], records[cb])
    e = nb + rb[rec_of] + ri
    last = ri == records[rec_of] - 1
    want = np.where(last, EMPTY, CHAIN | (e + 1)).astype(np.uint32)
    assert np.array_equal(T[e * wpe + 3], want)
    chain_words = np.concatenate([cb * wpe + 3, e * wpe + 3])
    # logical slots: bucket slots 0-2 (all 4 when unchained), then each record's slots 0-2
    nslot = np.where(chained, 3 + 3 * records, 4)
    B = np.repeat(np.arange(nb), nslot)
    t = np.arange(len(B)) - np.repeat(np.cumsum(nslot) - nslot, nslot)
    u = np.maximum(t - 3, 0)
    word = np.where(~chained[B] | (t < 3), B * wpe + t, (nb + rb[B] + u // 3) * wpe + u % 3)
    assert len(word) + len(chain_words) == info.front_entries * 4
    S = T[word]
    A = T[word + 4] if stride == 2 else None
    if stride == 2:
        assert (T[chain_words + 4] == EMPTY).all()
    ne = S != EMPTY
    assert not (S[ne] & CHAIN).any()
    Sn, Bn, tn = S[ne], B[ne], t[ne]
    key = (Bn << 13) | (Sn >> 18).astype(np.int64)
    start = np.ones(len(key), bool)
    start[1:] = (key[1:] != key[:-1]) | (tn[1:] != tn[:-1] + 1)
    st = np.nonzero(start)[0]
    glen = np.diff(np.append(st, len(key)))
    gkey, gt, gB = key[st], tn[st], Bn[st]
    assert glen.max(initial=1) <= 4
    vals = np.full((len(st), 4), EMPTY, np.uint32)
    anch = np.full((len(st), 4), EMPTY, np.uint32)
    for j in range(4):
        m = glen > j
        vals[m, j] = Sn[st[m] + j]
        if stride == 2:
            anch[m, j] = A[ne][st[m] + j]
    # expected groups, one per set bit, in (bucket, offset) order
    b = off[:-1]
    offs = (R.pos & np.uint64((1 << shift) - 1)).astype(np.int64)
    ekey = ((R.pos >> np.uint64(shift)).astype(np.int64) << 13) | offs
    elen = np.where(ln <= 4, ln, 1)
    evals = np.full((len(ln), 4), EMPTY, np.uint32)
    idp = np.append(ids, [0, 0, 0, 0])
    for j in range(4):
        m = (ln <= 4) & (ln > j)
        evals[m, j] = (offs[m] << 18) | np.where(ln[m] >= 3, 0x20000, 0) | idp[b[m] + j]
    evals[ln > 4, 0] = (offs[ln > 4] << 18) | 0x10000
    eanch = np.full((len(ln), 4), EMPTY, np.uint32)
    if stride == 2:
        first = np.full(R.n_set, EMPTY, np.int64)
        u_r, i_r = np.unique(R.rank, return_index=True)  # windows are in end order: the first one is the smallest end
        first[u_r] = R.ends[i_r]
        for j in range(4):
            m = (ln <= 4) & (ln > j)
            eanch[m, j] = first[m]
    order = np.argsort(gkey, kind="stable")
    assert np.array_equal(gkey[order], ekey), "every set bit appears exactly once, as one contiguous group"
    assert np.array_equal(glen[order], elen)
    assert np.array_equal(vals[order], evals)
    assert np.array_equal(anch[order], eanch)
    # empty slots: inside the used range only as padding at t = 2 (mod 3) right before a 2-id group
    used = np.zeros(nb, np.int64)
    np.maximum.at(used, Bn, tn + 1)
    emp = ~ne & (t < used[B])
    g2 = set(zip(gB[glen == 2].tolist(), gt[glen == 2].tolist()))
    pads = list(zip(B[emp].tolist(), t[emp].tolist()))
    assert all(tt % 3 == 2 and chained[bb] and (bb, tt + 1) in g2 for bb, tt in pads)
    # a 2-id group never straddles the bucket and a record or two records
    assert not ((glen == 2) & chained[gB] & (gt % 3 == 2)).any()
    stats["chained"] = stats.get("chained", 0) + int(chained.sum())
    stats["slots4"] = stats.get("slots4", 0) + int((slots == 4).sum())
    stats["slots5"] = stats.get("slots5", 0) + int((slots == 5).sum())
    stats["max_records"] = max(stats.get("max_records", 0), int(records.max(initial=0)))
    stats["padding"] = stats.get("padding", 0) + len(pads)
    inrec = (gt >= 3) & chained[gB]
    for L_, nm in ((1, "g1"), (2, "g2"), (3, "g3"), (4, "g4")):
        stats[nm + "_in_chain"] = stats.get(nm + "_in_chain", 0) + int((inrec & (glen == L_) & ((vals[:, 0] & 0x10000) == 0)).sum())
    stats["long_in_chain"] = stats.get("long_in_chain", 0) + int((inrec & ((vals[:, 0] & 0x10000) != 0)).sum())
    return records, ekey, vals[order], anch[order]


def ext_flags(R):
    """E[e]: the windows ending at e-1 and e are both valid and their ranks are equal or their id lists are equal."""
    ln = R.lens()
    lid = np.where(ln == 1, R.ids[np.minimum(R.off[:-1], max(len(R.ids) - 1, 0))], -1)
    seen = {}
    for r in np.nonzero(ln != 1)[0]:
        lid[r] = (1 << 40) + seen.setdefault(tuple(R.ids[R.off[r]:R.off[r + 1]].tolist()), len(seen))
    E = np.zeros(R.total, bool)
    a, b = R.win[:-1], R.win[1:]
    both = (a >= 0) & (b >= 0)
    E[1:] = both & ((a == b) | (lid[np.maximum(a, 0)] == lid[np.maximum(b, 0)]))
    return E


def check_ext(R, views, info):
    total, k = R.total, R.k
    code = CODE[R.bases]
    E = ext_flags(R)
    F1 = np.zeros(total, bool)
    F1[:max(total - k, 0)] = E[k:]
    nib = code | (E.astype(np.uint64) << np.uint64(2)) | (F1.astype(np.uint64) << np.uint64(3))
    n16 = (total + 15) // 16
    nib = np.append(nib, np.zeros(n16 * 16 - total, np.uint64)).reshape(n16, 16)
    es = np.zeros(total // 16 + 3, np.uint64)
    es[1:1 + n16] = np.bitwise_or.reduce(nib << (np.uint64(4) * np.arange(16, dtype=np.uint64)), axis=1)
    assert np.array_equal(np.frombuffer(views[5], np.uint64), es)
    n32 = (total + 31) // 32
    c2 = np.append(code, np.zeros(n32 * 32 - total, np.uint64)).reshape(n32, 32)
    r2 = np.zeros(total // 32 + 3, np.uint64)
    r2[1:1 + n32] = np.bitwise_or.reduce(c2 << (np.uint64(62) - np.uint64(2) * np.arange(32, dtype=np.uint64)), axis=1)
    assert np.array_equal(np.frombuffer(views[6], np.uint64), r2)
    cs = info.coarse_shift
    assert cs <= info.front_shift
    cw = np.zeros((((R.bf_bits >> cs) + 32) >> 5) + 1, np.uint32)
    c = (R.pos >> np.uint64(cs)).astype(np.int64)
    np.bitwise_or.at(cw, c >> 5, (np.uint32(1) << (c & 31).astype(np.uint32)))
    assert np.array_equal(np.frombuffer(views[7], np.uint32), cw)
    return E


def check_views(R, views, info, stats, lists=None, wide=False):
    """All eight views of one saved index; -> canonical form for comparisons between routes."""
    off, ids = (R.off, R.ids) if lists is None else lists
    n_set = R.n_set
    assert info.n_set_bits == n_set and info.tot_ids == len(ids) and info.bf_bits == R.bf_bits
    check_sectors(R, views[0])
    ent = np.frombuffer(views[1], np.uint64)
    assert len(ent) == n_set + 1 and np.array_equal(ent[:n_set], expected_entries(off, ids, wide))
    assert np.array_equal(np.frombuffer(views[2], np.uint32), off.astype(np.uint32))
    v3 = np.frombuffer(views[3], np.uint32 if wide else np.uint16)
    assert len(v3) == max(len(ids), 1) and np.array_equal(v3[:len(ids)], ids)
    if wide:
        assert info.front_entries == 0 and all(len(views[i]) == 0 for i in range(4, 8))
        return None
    front = decode_front(R, views[4], info, off, ids, stats)
    if info.extend:
        E = check_ext(R, views, info)
        stats["E"] = int(E.sum())
    else:
        assert all(len(views[i]) == 0 for i in (5, 6, 7))
    return front


def same_canonical(a, b):
    assert len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


def same_bytes(va, vb, n_set, exact=False):
    """Views 0, 2, 3, 5, 6, 7 byte for byte; view 1 up to word n_set (never written by a build); view 4 separately."""
    for i in (0, 2, 3, 5, 6, 7):
        assert np.array_equal(va[i], vb[i]), "view %d" % i
    assert np.array_equal(va[1][:8 * n_set], vb[1][:8 * n_set])
    if exact:
        assert np.array_equal(va[1], vb[1]) and np.array_equal(va[4], vb[4])


# ------------------------------------------------------------------------------------------- routes
def run_routes(R, tmp_path, stats, staged=True, shards=(1, 2, 3), copies=True):
    """One-call (forced on, automatic, forced off), staged, sharded, load, replicate: each decoded and checked; views
    compared between routes."""
    k, bf = R.k, R.bf_bits
    canon, saved = {}, {}
    for ext in (True, None, False):
        with _shark(k=k, bf_bits=bf, extend=ext) as sh:
            info = sh.build_index(R.bases, R.rec_off)
            assert info.extend == (ext is not False)
            assert info.plain_front == int(ext is None and info.front_entries * 16 <= (96 << 20))
            path = str(tmp_path / ("one_%s.shk" % ext))
            h, v = saved_views(sh, path)
            assert len(v[4]) == info.front_entries * 16 * (2 if info.extend else 1)
            canon[ext] = check_views(R, v, h.info, stats if ext else {})  # floors: one build
            saved[ext] = v
            if ext and copies:
                with _shark(k=k, bf_bits=bf) as b:
                    b.load_index(path)
                    _, vl = saved_views(b, str(tmp_path / "loaded.shk"))
                    same_bytes(vl, v, R.n_set, exact=True)
                with _shark(k=k, bf_bits=bf) as c:
                    c._check(c.lib.shk_index_replicate(sh.ctx, c.ctx))
                    hr, vr = saved_views(c, str(tmp_path / "replica.shk"))
                    assert hr.info.extend == 1
                    same_bytes(vr, v, R.n_set, exact=True)
    same_bytes(saved[True], saved[None], R.n_set)
    same_canonical(canon[True], canon[None])
    for i in (0, 2, 3):
        assert np.array_equal(saved[False][i], saved[True][i])
    if staged:
        with _shark(k=k, bf_bits=bf) as sh:
            _staged_build(sh, R.records, k, batch=1 << 13)
            h, v = saved_views(sh, str(tmp_path / "staged.shk"))
            assert h.info.extend == 0 and len(v[4]) == h.info.front_entries * 16
            same_canonical(check_views(R, v, h.info, {}), canon[False])
            same_bytes(v, saved[False], R.n_set)
    for n in shards:
        sharks = _sharks(n, k=k, bf_bits=bf, extend=True)
        try:
            type(sharks[0]).build_index_sharded(sharks, R.bases, R.rec_off)
            for i, sh in enumerate(sharks):
                h, v = saved_views(sh, str(tmp_path / ("shard%d_%d.shk" % (n, i))))
                assert h.info.n_shards == n and h.info.extend == 1
                same_canonical(check_views(R, v, h.info, {}), canon[True])
                same_bytes(v, saved[True], R.n_set)
        finally:
            _close(sharks)


def report(name, floors):
    print("floors %s: %s" % (name, " ".join("%s=%s" % kv for kv in floors.items())))


# ------------------------------------------------------------------------------------------- references
def rnd(rng, n):
    return ACGT[rng.integers(0, 4, int(n))].tobytes()


SEG_COPIES = (2, 3, 4, 5, 48, 49, 130)
REPEATS = (47, 48, 49, 300)


def segment_reference(k, seed):
    """Private random blocks, segments copied into exactly 2 … 130 records (both strands), and k-length pieces repeated
    n times inside one record, separated by N (raw counts at the kShortList switch with one id)."""
    rng = np.random.default_rng(seed)
    n_rec = 140
    recs = [bytearray(rnd(rng, int(rng.integers(60, 120)))) for _ in range(n_rec)]
    for j, m in enumerate(SEG_COPIES):
        seg = rnd(rng, 60)
        for i, g in enumerate(rng.choice(n_rec, m, replace=False)):
            recs[g] += rnd(rng, 7) + (rc(seg) if (i + j) % 2 else seg)
    recs = [bytes(r) + rnd(rng, 20) for r in recs]
    for n in REPEATS:
        piece = rnd(rng, k)
        recs.append(b"N".join([piece] * n))
    return recs


@pytest.mark.parametrize("k", [31, 17, 2])
def test_segment_lists(tmp_path, k):
    recs = segment_reference(k, 40 + k)
    R = Restated("segments_k%d" % k, recs, k, 1 << 24 if k > 2 else 1 << 12)
    ln = R.lens()
    floors = {"n_set": R.n_set, "tot_ids": len(R.ids), "max_len": int(ln.max()), "max_raw": int(R.raw.max())}
    if k > 2:
        # each segment's windows have lists of exactly m ids; each repeated piece one id at n raw occurrences
        for m in SEG_COPIES:
            floors["len%d" % m] = int((ln == m).sum())
            assert floors["len%d" % m] >= 60 - k
        for n in REPEATS:
            floors["raw%d_1id" % n] = int(((R.raw == n) & (ln == 1)).sum())
            assert floors["raw%d_1id" % n] >= 1
        assert ((R.raw > K_SHORT_LIST) & (ln < K_SHORT_LIST)).any() and ((R.raw == K_SHORT_LIST) & (ln > 1)).any()
    else:
        pal = R.canon == np.array([po.revcompl(int(x), k) for x in R.canon], np.uint64)
        floors["palindromes"] = int(pal.sum())
        assert floors["palindromes"] > 0 and (ln > K_SHORT_LIST).all()
    stats = {}
    run_routes(R, tmp_path, stats)
    floors["E"] = stats["E"]
    report(R.name, floors)


def test_k1_record_boundaries(tmp_path):
    """k = 1: every valid byte is a window, so E between the last base of one record and the first of the next follows
    the list rule like any other pair."""
    rng = np.random.default_rng(11)
    recs = [b"ACGTacgtAC", b"TTTTggggNNAC", b"A", b"", b"CAGTNacgGT" * 3, rnd(rng, 50), b"GATTACA", b"n", b"tgca"]
    R = Restated("k1", recs, 1, 1 << 10)
    E = ext_flags(R)
    b = R.rec_off[1:-1].astype(np.int64)
    b = b[(b > 0) & (b < R.total)]
    floors = {"boundaries_E1": int(E[b].sum()), "boundaries_E0": int((~E[b]).sum()), "n_set": R.n_set}
    assert floors["boundaries_E1"] >= 1 and floors["boundaries_E0"] >= 1
    stats = {}
    run_routes(R, tmp_path, stats)
    report(R.name, floors)


LONG_IDS = (0, 31, 32, 65503, 65504, 65534, 65535)


def all_genes_reference(k, seed):
    """65 536 gene indices from tiny records, with records that consume no index (length >= k, no window: the nidx
    `continue`) at record indices 1022 … 1025 and 2046 … 2049 (the block edges of assign_nidx_kernel) and two records
    shorter than k (they consume one).  One k-mer is shared by 60 genes including the bitmap's word and upper-word
    boundaries; a 2-, a 3- and a 4-id list end in 65535."""
    rng = np.random.default_rng(seed)
    genes = [bytearray(rnd(rng, 40)) for _ in range(65536)]
    genes[7] = bytearray(b"ACG")
    genes[40000] = bytearray(b"T" * (k - 1))
    long_piece = rnd(rng, k)
    carriers = sorted(set(LONG_IDS) | set(rng.choice(np.arange(100, 39000), 53, replace=False).tolist()))
    assert len(carriers) == 60
    for g in carriers:
        genes[g] = bytearray(long_piece + b"N" + genes[g])
    for ids in ((65534, 65535), (65533, 65534, 65535), (65532, 65533, 65534, 65535)):
        piece = rnd(rng, k)
        for g in ids:
            genes[g] += b"N" + piece
    quirk = b"ACGTN" * (k // 4 + 2)
    recs, quirk_at = [], (1022, 1023, 1024, 1025, 2046, 2047, 2048, 2049)
    it = iter(genes)
    while len(recs) < 65536 + len(quirk_at):
        recs.append(quirk if len(recs) in quirk_at else bytes(next(it)))
    return recs, long_piece, carriers


def test_all_gene_indices(tmp_path):
    k = 15
    recs, long_piece, carriers = all_genes_reference(k, 7)
    R = Restated("65536_genes", recs, k, 1 << 26)
    assert R.n_genes == 65536 and (R.nidx[[1022, 1023, 1024, 1025, 2046, 2047, 2048, 2049]] == -1).all()
    assert R.nidx[1021] == 1021 and R.nidx[1026] == 1022 and R.nidx[-1] == 65535
    r = int(np.searchsorted(R.pos, xxh64(po.enumerate_kmers(long_piece, k)[0])[0] % np.uint64(R.bf_bits)))
    lst = R.ids[R.off[r]:R.off[r + 1]]
    assert R.raw[r] > K_SHORT_LIST and set(LONG_IDS) <= set(lst.tolist()) and np.array_equal(lst, carriers)
    ln = R.lens()
    last = R.ids[np.maximum(R.off[1:] - 1, 0)]
    floors = {"n_genes": R.n_genes, "long_raw": int(R.raw[r]), "long_len": len(lst)}
    for m in (2, 3, 4):
        floors["len%d_ending_65535" % m] = int(((ln == m) & (last == 65535)).sum())
        assert floors["len%d_ending_65535" % m] >= 1
    stats = {}
    run_routes(R, tmp_path, stats, shards=(3,))
    Rw = Restated("65536_genes_wide", recs, k, R.bf_bits, wide=True)
    with _shark(k=k, bf_bits=R.bf_bits, wide_ids=True) as sh:
        sh.build_index(Rw.bases, Rw.rec_off)
        h, v = saved_views(sh, str(tmp_path / "wide.shk"))
        assert h.info.id_bits == 32
        check_views(Rw, v, h.info, {}, wide=True)
    report(R.name, floors)


def test_dense_chains(tmp_path, monkeypatch):
    """k = 12 at 2^19 bits (about 10 % of the bits set) with 6 keys per bucket: most buckets chain."""
    monkeypatch.setenv("SHK_FRONT_LOAD", "8")
    monkeypatch.delenv("SHK_EXTEND", raising=False)
    rng = np.random.default_rng(3)
    recs = [bytearray(rnd(rng, 1500)) for _ in range(40)]
    for j in range(300):  # short segments shared by 2 … 6 records: lists of every inline length, and long ones
        seg = rnd(rng, 14)
        for g in rng.choice(40, 2 + j % 5, replace=False):
            a = int(rng.integers(0, 1480))
            recs[g][a:a + 14] = seg if j % 2 else rc(seg)
    R = Restated("dense", [bytes(r) for r in recs], 12, 1 << 19)
    stats = {}
    run_routes(R, tmp_path, stats, shards=(2,))
    floors = {k_: stats[k_] for k_ in ("chained", "slots4", "slots5", "max_records", "padding", "g1_in_chain",
                                      "g2_in_chain", "g3_in_chain", "g4_in_chain", "long_in_chain")}
    floors["n_set"] = R.n_set
    report(R.name, floors)
    assert floors["chained"] >= 1000 and floors["slots4"] >= 100 and floors["slots5"] >= 100
    assert floors["max_records"] >= 4 and floors["padding"] >= 1
    assert min(floors[g] for g in ("g1_in_chain", "g2_in_chain", "g3_in_chain", "g4_in_chain", "long_in_chain")) >= 1


TILE_CASES = [224 * 4095 - 5, 224 * 4096 - 5, 224 * 4097 - 5, 224 * (3 * SCAN_TILE + 17) - 3, 1 << 20, 3 << 33]


@pytest.mark.parametrize("bf_bits", TILE_CASES)
def test_scan_tile_edges(tmp_path, bf_bits):
    """The rank directory is an exclusive scan over the sectors in tiles of 4096: filters of 4095, 4096, 4097 and more
    than 3 tiles of sectors (generic modulus, partial last sector), a power of two and a b * 2^33 filter."""
    rng = np.random.default_rng(bf_bits % 1000)
    recs = [rnd(rng, int(rng.integers(100, 900))) for _ in range(60)]
    recs[5] = recs[4][:300] + recs[5][300:]
    R = Restated("bf%d" % bf_bits, recs, 21, bf_bits)
    n_sec = ((bf_bits + 31) // 32 + 6) // 7
    report(R.name, {"n_sectors": n_sec, "tiles": -(-n_sec // SCAN_TILE), "partial_last_sector_bits": bf_bits - 224 * (n_sec - 1)})
    stats = {}
    if bf_bits >= 1 << 33:  # 3.2 GB of sectors per saved index: one route
        path = str(tmp_path / "big.shk")
        with _shark(k=21, bf_bits=bf_bits) as sh:
            sh.build_index(R.bases, R.rec_off)
            h, v = saved_views(sh, path)
            check_views(R, v, h.info, stats)
        del v
        os.remove(path)
        return
    run_routes(R, tmp_path, stats)


def test_staged_add_to_kmer_at_unset_bits(tmp_path):
    """BF::add_to_kmer hashes the k-mer and takes the rank of its position whether or not the bit is set
    (kmer_rank_kernel): an id for an unset position joins the list of the next set bit, and is dropped when no set bit
    follows."""
    rng = np.random.default_rng(21)
    k, bf = 13, 1 << 16
    recs = [rnd(rng, int(rng.integers(200, 600))) for _ in range(20)]
    R = Restated("staged_foreign", recs, k, bf)
    foreign = po.enumerate_kmers(rnd(rng, 40000), k)[0]
    gid = R.n_genes
    p = xxh64(foreign) % np.uint64(bf)
    fr = np.searchsorted(R.pos, p)
    on_set = (fr < R.n_set) & (R.pos[np.minimum(fr, R.n_set - 1)] == p)
    floors = {"unset_joins": int(((fr < R.n_set) & ~on_set).sum()), "set": int(on_set.sum()),
              "dropped": int((fr >= R.n_set).sum())}
    report(R.name, floors)
    assert floors["unset_joins"] >= 1000 and floors["dropped"] >= 1
    keep = fr < R.n_set
    ranks = np.concatenate([R.rank, fr[keep]])
    genes = np.concatenate([R.gene, np.full(int(keep.sum()), gid)])
    pairs = np.unique(ranks * 65536 + genes)
    off = np.concatenate([[0], np.cumsum(np.bincount(pairs // 65536, minlength=R.n_set))]).astype(np.int64)
    ids = (pairs % 65536).astype(np.int64)
    with _shark(k=k, bf_bits=bf) as sh:
        sh.add_at(sh.kmer_hashes(R.bases, R.rec_off))
        sh.switch_mode(1)
        for g, s in zip(R.nidx, recs):
            if g >= 0 and len(s) >= k:
                sh.add_to_kmer(po.enumerate_kmers(s, k)[0], int(g))
        sh.add_to_kmer(foreign, gid)
        sh.switch_mode(2)
        pos, coff, cids = sh.export_index()
        assert np.array_equal(pos, R.pos) and np.array_equal(coff, off) and np.array_equal(cids, ids)
        h, v = saved_views(sh, str(tmp_path / "foreign.shk"))
        check_views(R, v, h.info, {}, lists=(off, ids))
