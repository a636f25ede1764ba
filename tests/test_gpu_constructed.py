"""GPU: the classification kernels on constructed reads, against the oracle.

The reference is built from parts whose k-mer lists are known by construction: every gene record is a private block of
random bases followed by copies of shared segments, each segment copied into exactly m records (m = 2, 3, 4, 5, 31, 32,
33 and 130).  A read is a chosen concatenation of pieces, on either strand, so that it lands on one specific decision of
a kernel: the order in which it visits up to four genes (the register / shared-memory gene tables of K6 and K6b), lists
of 2 … 130 ids, runs of copied windows over such lists, the hand-offs to the warp-per-read kernels (a 5th gene, a list of
more than 4 ids, more than 1024 bytes, 95 … 130 genes), the -c threshold computed in doubles, ties and the hits
tiebreak.  The design of every family is itself checked with the oracle (floors printed and asserted).

Every family runs through K6 on text (extension off, forced on, automatic), K6 on packed reads (SHK_BULK=0), K6b, the
split upload and the wide-id kernels, in several warp layouts and chunk sizes.  Each run is compared with the oracle
read by read (results and score records), chunk by chunk (n_kept, n_assoc, n_multi, the reads handed to the warp-per-read
kernels), and its device counters with counts made without the device: n_probes = windows of k consecutive valid bases,
n_hits = those whose canonical k-mer has a set filter bit.  A set bit always carries at least one id (a record without a
window adds no bits and no id, the nidx rule), so K6's "the front table has an id" and K6m's "the filter bit is set" count
the same windows; the check holds every kernel to the second definition, the one bench.py reports."""
import math

import numpy as np
import pytest

from oracle import pyoracle as po
from test_gpu_bulk import mutate, rc
from test_gpu_parity import ACGT, to_soa
from test_gpu_scores import VALID, oracle_scores, rule

pytestmark = pytest.mark.gpu

BF = 1 << 30          # sparse: a window that is not in the reference rarely finds a set bit
N_PLAIN = 16          # genes 0 … 15 carry the small segments; the order family visits their private blocks
SMALL = {"s2": (0, 1), "s3": (4, 5, 6), "s4": (8, 9, 10, 11), "s5": (12, 13, 14, 15, 3)}
W0 = N_PLAIN + 1      # (record N_PLAIN is all N: it adds no gene id, the ids after it are record index - 1)
WIDE = {"w31": (0, 31), "w32": (31, 63), "w33": (63, 96), "w31b": (96, 127), "w32b": (96, 128), "w33b": (96, 129),
        "w130": (0, 130)}  # gene ranges relative to W0
N_WIDE = 132
PATHS = ["lookup", "extend", "auto", "k6_packed", "bulk", "split", "wide"]


def _shark(**kw):
    from shark_b200.engine import Shark
    return Shark(**kw)


def rnd(rng, n):
    return ACGT[rng.integers(0, 4, int(n))].tobytes()


class SegRef:
    """Records = private block + (spacer + segment) for every segment the record carries + a private tail."""

    def __init__(self, seed):
        rng = np.random.default_rng(seed)
        self.seg = {s: rnd(rng, 200) for s in SMALL}
        self.seg.update({s: rnd(rng, 150) for s in WIDE})
        carriers = {}
        for s, gs in SMALL.items():
            for g in gs:
                carriers.setdefault(g, []).append(s)
        for s, (a, b) in WIDE.items():
            for g in range(a, b):
                carriers.setdefault(W0 + g, []).append(s)
        self.private, self.seg_at, recs = {}, {}, []
        for g in range(W0 + N_WIDE):
            if g == N_PLAIN:
                recs.append(b"N" * 64)
                continue
            rec = rnd(rng, int(rng.integers(300, 400)) if g < N_PLAIN else 100)
            self.private[g] = rec
            for s in carriers.get(g, []):
                rec += rnd(rng, 20)
                self.seg_at[g, s] = len(rec)
                rec += self.seg[s]
            recs.append(rec + rnd(rng, 100))
        self.records = recs
        self.bases, self.rec_off = po.concat_records(recs)
        self.rng = rng

    def piece(self, g, L):
        p = self.private[g]
        st = int(self.rng.integers(0, len(p) - L + 1))
        return p[st:st + L]

    def seg_piece(self, s, L):
        p = self.seg[s]
        st = int(self.rng.integers(0, len(p) - L + 1))
        return p[st:st + L]


def rgs(n, kmax=4):
    """Restricted-growth strings of length n over at most kmax letters: gene-visit patterns up to relabelling."""
    out = []

    def rec(p, m):
        if len(p) == n:
            out.append(tuple(p))
            return
        for a in range(min(m + 1, kmax)):
            rec(p + [a], max(m, a + 1))
    rec([0], 1)
    return out


PATTERNS = [p for n in range(1, 7) for p in rgs(n)]


def substitute(rng, s):
    """One substitution in the middle third of s."""
    j = int(rng.integers(len(s) // 3, max(len(s) // 3 + 1, 2 * len(s) // 3)))
    b = bytearray(s)
    b[j] = int(ACGT[(int(np.nonzero(ACGT == b[j])[0][0]) + int(rng.integers(1, 4))) % 4])
    return bytes(b)


def families(R, k):
    """-> [(text, family, flags)]; flags: 'run' = a run of copied windows over lists of 3 or 4 ids (K6b hands it on)."""
    rng = R.rng
    out = []
    add = lambda t, fam, flag="": out.append((rc(t) if rng.random() < 0.5 else t, fam, flag))
    plain = np.arange(N_PLAIN)
    for pat in PATTERNS:                                   # order: every visit pattern, pieces k-1, k, k+1, 2k
        for L in (k - 1, k, k + 1, 2 * k):
            g = rng.permutation(plain)[:4]
            t = b"".join(R.piece(int(g[a]), L) for a in pat)
            out.append((t, "order", ""))
            out.append((rc(t), "order", ""))
        g = rng.permutation(plain)[:4]                     # one substitution per piece: K6b loses and re-finds its diagonal
        add(b"".join(substitute(rng, R.piece(int(g[a]), 2 * k)) for a in pat), "subs")
        if len(set(pat)) >= 2:                             # a 2-id segment of genes A and B, at every place of the pattern
            g = np.concatenate(([0, 1], rng.permutation(np.arange(2, N_PLAIN))[:2]))
            for at in range(len(pat) + 1):
                ps = [R.piece(int(g[a]), k + 1) for a in pat]
                ps.insert(at, R.seg_piece("s2", 2 * k))
                add(b"".join(ps), "join")
    for s in SMALL:                                        # inside 2 … 5-id segments: ties of 2, 3, 4 genes; 5 = long list
        for L in (k, k + 1, 2 * k, 3 * k, 150):
            for _ in range(4):
                add(R.seg_piece(s, L), "inside")
    for s in ("s2", "s3", "s4"):                           # runs: a private window anchors the diagonal, then the segment
        for g in SMALL[s]:
            rec, at = R.records[g], R.seg_at[g, s]
            for j in range(6):
                pre, post = k + 3 + 7 * j, k + 1 + 11 * j
                flag = "" if s == "s2" else "run"
                out.append((rec[at - pre:at + post], "run", flag))
                end = at + len(R.seg[s])                   # the other strand: the segment's end, then what follows it
                out.append((rc(rec[end - post:end + pre]), "run", flag))
    for n in (4, 5):                                       # exactly 4 and exactly 5 genes
        for _ in range(24):
            g = rng.permutation(plain)[:n]
            order = list(g) + list(g[:int(rng.integers(0, n))])
            add(b"".join(R.piece(int(x), 2 * k) for x in order), "genes%d" % n)
    combos = {95: ["w31", "w32", "w31b", 130], 96: ["w31", "w32", "w33"], 127: ["w31", "w32", "w33", "w31b"],
              128: ["w31", "w32", "w33", "w32b"], 129: ["w31", "w32", "w33", "w33b"], 130: ["w130"]}
    for n, parts in combos.items():                        # 95 … 130 genes: K6m or K6x
        for j in range(8):
            ps = [R.piece(W0 + x, k + 5) if isinstance(x, int) else R.seg_piece(x, k + 5 + j) for x in parts]
            perm = rng.permutation(len(ps))
            add(b"".join(ps[i] for i in perm), "wide%d" % n)
    for n in (1024, 1025):                                 # kMaxFastLen bytes and one more
        for _ in range(6):
            g = rng.permutation(plain)[:3]
            t = b"".join(R.piece(int(g[i % 3]), 2 * k) for i in range(n // (2 * k) + 1))[:n]
            add(t, "len%d" % n)
            if n == 1025:
                m = bytearray(t)
                m[int(rng.integers(100, 900))] = ord("N")
                add(bytes(m), "len1025N")
    for _ in range(24):                                    # equal cov, different hits: the hits tiebreak
        a, b = (int(x) for x in rng.permutation(plain)[:2])
        P = 3 * k
        pa = R.piece(a, P - 1)                             # cov P-1, hits P-k
        pb = bytearray(R.piece(b, P))                      # cov P-1 (one substitution in the middle), hits P-2k+1
        pb[P // 2] = int(ACGT[(int(np.nonzero(ACGT == pb[P // 2])[0][0]) + 1) % 4])
        add(pa + bytes(pb) if rng.random() < 0.5 else bytes(pb) + pa, "hits")
    out += [(b"", "empty", ""), (b"N" * 40, "empty", ""), (b"A", "empty", "")]
    return out


def read_facts(ref, k, seq, off, qual=None, q=0):
    """Per read, without the device: windows of k consecutive valid bases (numpy), windows with a set bit, genes touched,
    longest id list of a window."""
    n = len(off) - 1
    probes, hits, genes, maxlist = (np.zeros(n, np.int64) for _ in range(4))
    for i in range(n):
        t = seq[int(off[i]):int(off[i + 1])]
        if q:
            t = po.mask(t, qual[int(off[i]):int(off[i + 1])], q)
        v = VALID[t].astype(np.int64)
        if len(v) >= k:
            c = np.concatenate(([0], np.cumsum(v)))
            probes[i] = int((c[k:] - c[:-k] == k).sum())
        e = po.enumerate_kmers(t.tobytes(), k)
        km = e[0] if e is not None else np.zeros(0, np.uint64)
        assert len(km) == probes[i], i   # the kernels' run >= k rule is the reference's window enumeration
        if len(km):
            rank, _, ln = ref.probe(km)
            hits[i] = int((rank >= 0).sum())
            maxlist[i] = int(ln.max())
        genes[i] = len(ref.read_table(t.tobytes(), 1 << 12)[0])
    return probes, hits, genes, maxlist


def open_path(monkeypatch, path, **kw):
    """-> (context, packed) for one classification path"""
    monkeypatch.setenv("SHK_BULK", "0" if path == "k6_packed" else "1")
    extend = {"lookup": False, "auto": None, "wide": None}.get(path, True)
    sh = _shark(extend=extend, host_pack=0.5 if path == "split" else False, wide_ids=path == "wide", **kw)
    return sh, path in ("k6_packed", "bulk")


def classify(sh, packed, seq, off, qual):
    """sh.analyze, keeping every chunk's result record."""
    chunks, collect = [], sh.collect
    sh.collect = lambda slot, copy=True: chunks.append(collect(slot, copy)) or chunks[-1]
    try:
        keep, ar, ag, stats = sh.analyze(seq, off, qual, packed=packed)
    finally:
        del sh.collect
    return keep, ar, ag, stats, chunks


class Want:
    """The oracle's view of a read set, in its canonical order."""

    def __init__(self, ref, k, texts, c, single, qual=None, q=0, k6b_extra=None):
        self.seq, self.off = to_soa(texts)
        self.qual, self.q = qual, q
        self.cnt, self.ar, self.ag = ref.analyze(self.seq, self.off, c, qual=qual, min_quality=q, single=single)
        self.scores = oracle_scores(ref, self.seq, self.off, qual, q)
        self.probes, self.hits, self.genes, self.maxlist = read_facts(ref, k, self.seq, self.off, qual, q)
        nbytes = np.diff(self.off.astype(np.int64))
        self.slow_k6 = (self.genes > 4) | (self.maxlist > 4) | (nbytes > 1024)
        # K6b also hands on a run of copied windows over lists of 3 or 4 ids; where the caller does not name those reads,
        # any read with such a list may be one
        self.k6b_exact = k6b_extra is not None
        self.slow_k6b = self.slow_k6 | (k6b_extra if self.k6b_exact else self.maxlist >= 3)

    def layout(self, perm):
        texts = [bytes(self.seq[int(self.off[i]):int(self.off[i + 1])]) for i in perm]
        seq, off = to_soa(texts)
        qual = None
        if self.qual is not None:
            qual = np.concatenate([self.qual[int(self.off[i]):int(self.off[i + 1])] for i in perm] + [np.zeros(0, np.uint8)])
        return seq, off, qual

    def check(self, path, perm, out, sh, wide=False):
        keep, ar, ag, stats, chunks = out
        perm = np.asarray(perm, np.int64)   # (a grouped layout repeats the empty read as padding)
        r0 = perm[ar.astype(np.int64)]
        o = np.lexsort((ag, r0))
        assert np.array_equal(r0[o], self.ar) and np.array_equal(ag[o], self.ag), path
        kp = np.zeros(len(self.cnt), np.uint8)
        kp[perm] = keep
        assert np.array_equal(kp, (self.cnt > 0).astype(np.uint8)), path
        if sh.scores:
            sc = np.zeros_like(self.scores)
            sc[perm] = stats["scores"]
            bad = np.nonzero((sc != self.scores).any(1))[0]
            assert len(bad) == 0, (path, bad[:8], sc[bad[:4]], self.scores[bad[:4]])
        spans = sh.plan_chunks(np.asarray(self.layout_off(perm)))
        assert len(spans) == len(chunks)
        slow = self.slow_k6b if path == "bulk" else self.slow_k6
        for (a, b), ch in zip(spans, chunks):
            idx = perm[a:b]
            cnt = self.cnt[idx].astype(np.int64)
            assert ch["n_reads"] == b - a
            assert (ch["n_kept"], ch["n_assoc"]) == ((cnt > 0).sum(), cnt.sum()), (path, a)
            assert ch["n_multi"] == (cnt.sum() if wide else cnt[cnt >= 2].sum()), (path, a)
            assert (ch["n_probes"], ch["n_hits"]) == (self.probes[idx].sum(), self.hits[idx].sum()), (path, a)
            assert ch["n_extended"] <= ch["n_hits"], (path, a)
            if wide:
                assert ch["n_slow_reads"] == b - a
            elif path == "split" or (path == "bulk" and not self.k6b_exact):
                assert self.slow_k6[idx].sum() <= ch["n_slow_reads"] <= self.slow_k6b[idx].sum(), (path, a)
            else:
                assert ch["n_slow_reads"] == slow[idx].sum(), (path, a, ch["n_slow_reads"], slow[idx].sum())

    def layout_off(self, perm):
        L = np.diff(self.off.astype(np.int64))[np.asarray(perm, np.int64)]
        return np.concatenate(([0], np.cumsum(L))).astype(np.uint64)


def grouped_perm(fams, tile=128):
    """Reads sorted by family, each family padded to whole 128-read tiles with empty reads (index -1)."""
    perm = []
    for f in sorted(set(fams)):
        idx = [i for i, x in enumerate(fams) if x == f]
        perm += idx + [-1] * (-len(idx) % tile)
    return perm


def constructed_text(w, i):
    return w.seq[int(w.off[i]):int(w.off[i + 1])].tobytes()


@pytest.fixture(scope="module", params=[31, 17], ids=["k31", "k17"])
def constructed(request):
    return build_constructed(request.param)


def build_constructed(k):
    R = SegRef(1000 + k)
    reads = families(R, k)
    texts = [t for t, _, _ in reads] + [b""]          # (the last read is the padding of the grouped layout)
    fams = [f for _, f, _ in reads] + ["pad"]
    run = np.array([fl == "run" for _, _, fl in reads] + [False])
    ref = po.Index(R.bases, R.rec_off, k, BF)
    want = {single: Want(ref, k, texts, 0.2, single, k6b_extra=run) for single in (False, True)}
    w = want[False]
    fams_a = np.array(fams)
    # the design, checked with the oracle (floors at about 90 % of what the construction gives)
    floors = {}
    plain_order = fams_a == "order"
    designed = np.array([len(set(p)) for p in PATTERNS for _ in range(8)])
    piece_len = np.array([L for p in PATTERNS for L in (k - 1, k, k + 1, 2 * k) for _ in range(2)])
    ok = (w.genes[plain_order] == designed) | (piece_len < k)
    floors["order reads with their designed gene count"] = (ok.mean(), 0.97)
    floors["order reads touching 4 genes"] = ((w.genes[plain_order] == 4).sum(), 150)
    for n in (4, 5):
        floors["genes%d reads with %d genes" % (n, n)] = ((w.genes[fams_a == "genes%d" % n] == n).mean(), 0.9)
    for n in (95, 96, 127, 128, 129, 130):
        floors["wide%d reads with %d genes" % (n, n)] = ((w.genes[fams_a == "wide%d" % n] == n).mean(), 0.9)
    inside = fams_a == "inside"
    for m in (2, 3, 4, 5):
        floors["inside reads with a %d-id list" % m] = (((w.maxlist == m) & inside).sum(), 18)
        floors["%d-way ties" % m] = ((w.scores[:, 3] == m).sum(), 18)
    floors["run reads over lists of 3 or 4 ids"] = (((w.maxlist >= 3) & run).sum(), run.sum())
    floors["reads K6 hands on"] = (w.slow_k6.sum(), 95)
    floors["4-gene reads K6 keeps"] = (((w.genes == 4) & ~w.slow_k6).sum(), 150)
    floors["reads over 1024 bytes"] = ((np.diff(w.off.astype(np.int64)) > 1024).sum(), 12)
    hb = w.scores[fams_a == "hits"]
    floors["hits-tiebreak reads won by one gene"] = ((hb[:, 3] == 1).mean(), 0.9)
    floors["reads -s drops"] = (((w.cnt > 0) & (want[True].cnt == 0)).sum(), 60)
    hits_tie = 0
    for i in np.nonzero(fams_a == "hits")[0]:
        _, cv, h = ref.read_table(constructed_text(w, i), 64)
        top = cv == cv.max()
        hits_tie += int(top.sum() == 2 and len(set(h[top].tolist())) == 2)
    floors["hits-tiebreak reads: two genes with the best cov, different hits"] = (hits_tie, 12)
    floors["reported reads"] = ((w.cnt > 0).sum(), 1500)
    print("k=%d: %d reads" % (k, len(texts)))
    for name, (v, lo) in floors.items():
        print("  %-45s %s (floor %s)" % (name, v, lo))
        assert v >= lo, (name, v, lo)
    return dict(k=k, R=R, ref=ref, texts=texts, fams=fams, want=want)


@pytest.mark.parametrize("path", PATHS)
def test_constructed_families(monkeypatch, constructed, path):
    """Every family through one path, interleaved and grouped by family, at 1023 reads per chunk (the last warp holds 31
    reads, the last tile 127), at 1025 (last warp 1 read) with score records, and at 1057 (last tile 33 reads) with -s."""
    k, R = constructed["k"], constructed["R"]
    n = len(constructed["texts"])
    rng = np.random.default_rng(k)
    inter = rng.permutation(n)
    grouped = [i if i >= 0 else n - 1 for i in grouped_perm(constructed["fams"][:-1])]
    wide = path == "wide"
    for chunk, scores, single in ((1023, False, False), (1025, True, False), (1057, False, True)):
        want = constructed["want"][single]
        sh, packed = open_path(monkeypatch, path, k=k, c=0.2, bf_bits=BF, single=single, max_reads_per_chunk=chunk,
                               scores=scores)
        with sh:
            info = sh.build_index(R.bases, R.rec_off)
            if path == "auto":
                assert (info.extend, info.plain_front) == (1, 1)
            for perm in (inter, grouped):
                seq, off, qual = want.layout(perm)
                out = classify(sh, packed, seq, off, qual)
                want.check(path, perm, out, sh, wide=wide)
                if scores:
                    stats = out[3]
                    sc = np.zeros_like(want.scores)
                    sc[np.asarray(perm)] = stats["scores"]
                    cnt = np.bincount(np.asarray(perm)[out[1].astype(np.int64)], minlength=n)
                    assert np.array_equal(cnt > 0, rule(sc, 0.2, single))


# ---- the -c boundary ------------------------------------------------------------------------------------------------
C_CASES = [(0.55, 100), (0.55, 180), (0.7, 90), (0.7, 170), (0.57, 100), (0.35, 180), (0.6, 90), (0.3, 190), (0.5, 100),
           (1.0, 100), (1.0, 64)]


def boundary_reads(R, k, q):
    """(c, text, qual): a clean piece of m = ceil(c*L) or ceil(c*L) - 1 bases plus L - m tail bases, so that cov = m and
    len = L; masked bytes (low quality at -q 20, N without -q) sit in the tail, so the text is longer than len."""
    rng = R.rng
    out = []
    for c, L in C_CASES:
        m1 = math.ceil(c * L)
        for m in (m1, m1 - 1):
            if m < k + 2:
                continue
            for j in range(6):
                g = int(rng.integers(0, N_PLAIN))
                p = R.private[g]
                st = int(rng.integers(0, len(p) - m - 1))
                tail = bytearray(rnd(rng, L - m))
                if len(tail) and tail[0] == p[st + m]:      # the tail must not go on like the gene
                    tail[0] = int(ACGT[(int(np.nonzero(ACGT == tail[0])[0][0]) + 1) % 4])
                t = bytearray(p[st:st + m]) + tail
                qu = bytearray([73] * len(t))
                for _ in range(int(rng.integers(1, 4)) if len(tail) else 0):
                    at = int(rng.integers(m + 1, len(t) + 1))
                    t[at:at] = b"A" if q else b"N"
                    qu[at:at] = bytes([33 + 5])
                if j % 2:
                    t, qu = bytearray(rc(bytes(t))), qu[::-1]
                out.append((c, bytes(t), bytes(qu), L, m))
    return out


@pytest.mark.parametrize("q", [20, 0])
def test_c_threshold_boundary(monkeypatch, q):
    """cov = m against c*len in IEEE doubles where the product falls just off an integer (0.55 * 100 = 55.00000000000001,
    0.7 * 90 = 62.99999999999999), with and without -s, on every path; both outcomes occur for every c."""
    k = 31
    R = SegRef(77)
    ref = po.Index(R.bases, R.rec_off, k, BF)
    reads = boundary_reads(R, k, q)
    texts = [t for _, t, _, _, _ in reads]
    qual = np.frombuffer(b"".join(x for _, _, x, _, _ in reads), np.uint8).copy() if q else None
    seq, off = to_soa(texts)
    sc = oracle_scores(ref, seq, off, qual, q)
    design = np.array([(L, m) for _, _, _, L, m in reads])
    assert np.array_equal(sc[:, :2], design), np.nonzero((sc[:, :2] != design).any(1))[0]
    assert (sc[:, 3] == 1).all()
    cs = np.array([c for c, _, _, _, _ in reads])
    for c in sorted(set(cs)):
        keep = rule(sc[cs == c], c, False)
        assert keep.any() and (~keep).any(), c
    f32 = sc[:, 1].astype(np.float32) >= cs.astype(np.float32) * sc[:, 0].astype(np.float32)
    assert (f32 != (sc[:, 1] >= cs * sc[:, 0])).sum() >= 12   # a threshold computed in float decides these differently
    for path in PATHS:
        for single, scores in ((False, True), (True, False)):
            sh, packed = open_path(monkeypatch, path, k=k, c=0.5, bf_bits=BF, min_quality=q, single=single,
                                   max_reads_per_chunk=64, scores=scores)
            with sh:
                sh.build_index(R.bases, R.rec_off)
                for c in sorted(set(cs)):
                    idx = np.nonzero(cs == c)[0]
                    s2, o2 = to_soa([texts[i] for i in idx])
                    q2 = np.concatenate([qual[int(off[i]):int(off[i + 1])] for i in idx]) if q else None
                    cnt0, ar0, ag0 = ref.analyze(s2, o2, c, qual=q2, min_quality=q, single=single)
                    sh.set_options(c=c, single=single)
                    keep, ar, ag, stats = sh.analyze(s2, o2, q2, packed=packed)
                    assert np.array_equal(keep, (cnt0 > 0).astype(np.uint8)), (path, c, single)
                    assert np.array_equal(ar, ar0) and np.array_equal(ag, ag0), (path, c, single)
                    assert np.array_equal(keep.astype(bool), rule(sc[idx], c, single)), (path, c, single)
                    if scores:
                        assert np.array_equal(stats["scores"], sc[idx]), (path, c)


# ---- uniform warps ----------------------------------------------------------------------------------------------------
def test_uniform_warps(monkeypatch):
    """Warps whose 32 reads all take the same path, on a dense filter (k = 12 at 2^19 bits, about 11 % of the bits set:
    the coarse filter passes nearly every window).  The reference has 4 records, so no read can reach a 5th gene or a
    list of 5 ids: every read stays in K6 / K6b for all of its windows.  32 background reads of 1024 bases per warp
    (every window is a lookup, about one in nine passes to the table), 31 empty or all-N reads and one long read, 32
    copies of one read, gene pieces of 1024 bases; through every path."""
    rng = np.random.default_rng(5)
    k, bf = 12, 1 << 19
    genes = [rnd(rng, 15000) for _ in range(4)]
    bases, rec_off = po.concat_records(genes)
    ref = po.Index(bases, rec_off, k, bf)
    assert ref.n_set > bf // 16
    texts = [rnd(rng, 1024) for _ in range(128)]                       # background, one whole tile
    for j in range(8):                                                 # one long read among 31 empty ones
        g = genes[j % 4]
        warp = [b"" if i % 2 else b"N" * int(rng.integers(1, 200)) for i in range(32)]
        st = int(rng.integers(0, 14000))
        warp[(5 * j) % 32] = g[st:st + int(rng.integers(600, 1025))]
        texts += warp
    for t in (genes[0][:150], genes[1][:1024], rc(genes[2][100:1124]), rnd(rng, 1024), mutate(rng, genes[3][:1000])):
        texts += [t] * 32                                              # 32 copies of one read
    texts += [genes[i % 4][int(st):][:1024] for i, st in enumerate(rng.integers(0, 13900, 64))]   # gene pieces
    want = Want(ref, k, texts, 0.3, False)
    bg = slice(0, 128)
    print("dense filter: %d of %d bits set; background reads: %.3f of their windows hit, up to %d genes, lists up to %d "
          "ids; %d reads with a list of 3 or 4 ids" % (ref.n_set, bf, want.hits[bg].sum() / want.probes[bg].sum(),
                                                       want.genes[bg].max(), want.maxlist[bg].max(), (want.maxlist >= 3).sum()))
    assert (want.probes[bg] == 1024 - k + 1).all() and want.hits[bg].sum() > 0.08 * want.probes[bg].sum()
    assert not want.slow_k6.any() and want.genes.max() <= 4 and want.maxlist.max() <= 4
    perm = np.arange(len(texts))
    for path in PATHS:
        sh, packed = open_path(monkeypatch, path, k=k, c=0.3, bf_bits=bf, max_reads_per_chunk=512, scores=True)
        with sh:
            sh.build_index(bases, rec_off)
            out = classify(sh, packed, *want.layout(perm))
            want.check(path, perm, out, sh, wide=path == "wide")
            if path != "wide":   # no read leaves the fast kernels: they walk every window of every lane
                assert [ch["n_slow_reads"] for ch in out[4]] == [0] * len(out[4]), path


# ---- tie-saturated chunks ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("scores", [False, True], ids=["plain", "scores"])
@pytest.mark.parametrize("path", ["extend", "bulk", "wide"])
def test_tie_saturated_chunks(monkeypatch, path, scores):
    """Chunks in which every read is a 2-, 4- or 130-way tie overflow the tie pool (max(R/2, 4096) entries: the chunk
    runs again) and the multi list (R/4 + 1024: it is scattered again into a larger buffer).  The order of chunks on one
    context varies what the read-back enqueued with the kernels (sized by the previous chunks) covers: a tie-free chunk
    then a saturated one (it falls short), two saturated ones (the second, on the other slot, prefetches all of its old
    list, then meets a re-scatter), a tie-free one (it overshoots), a saturated one on grown buffers."""
    k, Rc = 21, 2048
    R = SegRef(21)
    ref = po.Index(R.bases, R.rec_off, k, BF)
    rng = np.random.default_rng(3)
    free = [R.piece(int(g), 60) for g in rng.integers(0, N_PLAIN, Rc)]
    sat = lambda: [rc(x) if rng.random() < 0.5 else x for x in
                   (R.seg_piece(("s2", "s4", "w130")[i % 3], 60) for i in range(Rc))]
    calls = [free, sat(), sat() + sat(), free, sat()]
    sh, packed = open_path(monkeypatch, path, k=k, c=0.5, bf_bits=BF, max_reads_per_chunk=Rc, scores=scores)
    with sh:
        sh.build_index(R.bases, R.rec_off)
        # the launches of a chunk that needs no recovery: a few tie-free reads on the fresh slot
        want = Want(ref, k, free[:64], 0.5, False)
        out = classify(sh, packed, *want.layout(np.arange(64)))
        want.check(path, np.arange(64), out, sh, wide=path == "wide")
        normal = out[4][0]["kernel_launches"]
        # a re-run adds the chunk's launches again, a re-scatter one more; with wide ids every reported read is a multi
        # entry, so the tie-free chunk (2048 entries) is scattered again too
        expect = [[normal + (path == "wide")], [2 * normal + 1], [normal, 2 * normal + 1], [normal], [normal]]
        for texts, launches in zip(calls, expect):
            want = Want(ref, k, texts, 0.5, False)
            perm = np.arange(len(texts))
            out = classify(sh, packed, *want.layout(perm))
            want.check(path, perm, out, sh, wide=path == "wide")
            assert [ch["kernel_launches"] for ch in out[4]] == launches, (normal, [ch["kernel_launches"] for ch in out[4]])
