"""The front-table and coarse-filter geometry of the extension structures, swept on references small enough to check
every read against the oracle.

The classification kernels find a window's coarse-filter bit as (bucket << coarse_rel) | (offset >> coarse_shift), with
coarse_rel = front shift - coarse shift (shk_bulk.cu, shk_reads.cu; the arguments come from make_args in
shk_capi.cu).  A full-size reference sets the geometry: C2 runs at (front shift, coarse shift) = (11, 5), C3 at (8, 5),
C4 at (8, 7), a whole transcriptome clamps the coarse shift to the front shift (coarse_rel 0).  The tuning variables
SHK_FRONT_LOAD and SHK_COARSE_LOG2, read only by the index build (front_geometry, build_front in shk_index.cu), give
each of these geometries to a reference of ~66 k keys.  Every case asserts the geometry it got, so that a clamp cannot
silently turn it into another case, and then checks the index, BF::get_index and the reads through the three kernels
that read the structures: the thread-per-read kernel on text (K6) and on packed reads (SHK_BULK=0), and the bulk
kernel (K6b) - each bit for bit against the oracle."""
import numpy as np
import pytest

from oracle import pyoracle as po
from test_gpu_bulk import stress_reads
from test_gpu_parity import quals_for, quirky_reference, rnd_genes, sample_reads, to_soa

pytestmark = pytest.mark.gpu

# front shift, coarse shift, bf_bits, k, -q, -s, SHK_COARSE_LOG2 (None: lg(bf_bits) - coarse shift)
CASES = [
    (8, 7, 1 << 31, 31, 0, False, None),          # C4's: coarse_rel 1
    (8, 5, 536870909, 21, 20, True, None),        # C3's, with -q 20 and -s
    (11, 5, 1073741789, 21, 0, False, None),      # C2's
    (5, 5, 67108859, 31, 0, False, None),         # coarse_rel 0 ...
    (8, 8, 1 << 30, 21, 0, False, 20),            # ... through the clamp of the coarse shift to the front shift
    (13, 13, 3 << 33, 31, 0, False, None),
    (12, 12, 3 << 33, 21, 20, False, None),
    (5, 0, 1 << 26, 21, 0, False, None),          # one coarse bit per filter position
    (13, 0, 1 << 30, 31, 0, False, None),
    (12, 3, 3 << 33, 21, 0, True, None),
    (6, 2, 16777213, 31, 0, False, None),
    (9, 0, 1 << 22, 21, 0, False, None),          # ~8 keys per bucket: most of the table is overflow records
]
CHAINED = (9, 0, 1 << 22)
MOD = {0: "pow2", 1: "b33", 2: "generic"}


def _lg(n):
    """smallest lg with 2^lg >= n (build_front)"""
    return max(0, (int(n) - 1).bit_length())


def _mod(bf_bits):
    """bit_index variant (shk_capi.cu): power of two, b * 2^33, or a generic modulus"""
    if bf_bits & (bf_bits - 1) == 0:
        return 0
    return 1 if bf_bits % (1 << 33) == 0 else 2


def _case_id(c):
    fs, cs, bf, k, q, single, _ = c
    return "f%d_c%d_%s_k%d%s%s" % (fs, cs, MOD[_mod(bf)], k, "_q%d" % q if q else "", "_s" if single else "")


def _inputs(rng, k, q):
    genes = quirky_reference(rng)
    genes += rnd_genes(rng, 20, 1500, 3000)
    genes[45] = genes[44][:700] + genes[45][700:]           # copies: the anchor of a shared window names the first gene
    genes[47] = genes[46][300:1200] + genes[47][900:]
    bases, rec_off = po.concat_records(genes)
    texts = stress_reads(rng, [g.upper() for g in genes], 6000, k)
    texts += sample_reads(rng, genes, 1000, 100, paired=True)
    texts += [b"", b"A", b"ACGT" * 8]
    seq, off = to_soa(texts)
    qual = quals_for(rng, texts) if q else None
    return genes, bases, rec_off, seq, off, qual


@pytest.mark.parametrize("case", CASES, ids=_case_id)
def test_geometry_parity(monkeypatch, case):
    from shark_b200.engine import Shark
    fs, cs, bf_bits, k, q, single, coarse_log2 = case
    c = 0.6
    rng = np.random.default_rng(100 * fs + cs)
    genes, bases, rec_off, seq, off, qual = _inputs(rng, k, q)
    ref = po.Index(bases, rec_off, k, bf_bits)

    # the geometry: front_geometry takes the largest shift with 2^shift <= load * bf_bits / n_set (at least 5, at most
    # 13); build_front takes coarse shift = min(lg(bf_bits) - coarse_log2, front shift)
    load = 1.5 * (1 << fs) * ref.n_set / bf_bits
    assert 0.01 < load < 64, load
    coarse_log2 = _lg(bf_bits) - cs if coarse_log2 is None else coarse_log2
    assert 20 <= coarse_log2 <= 32, coarse_log2
    monkeypatch.setenv("SHK_FRONT_LOAD", "%.9g" % load)
    monkeypatch.setenv("SHK_COARSE_LOG2", str(coarse_log2))
    monkeypatch.delenv("SHK_EXTEND", raising=False)
    with Shark(k=k, c=c, bf_bits=bf_bits, min_quality=q, single=single, max_reads_per_chunk=1500, extend=True,
               compact=True) as sh:
        info = sh.build_index(bases, rec_off)
        assert (info.extend, info.front_shift, info.coarse_shift) == (1, fs, cs)
        n_buckets = -(-bf_bits // (1 << fs))
        assert info.front_entries >= n_buckets
        if (fs, cs, bf_bits) == CHAINED:
            assert info.front_entries - n_buckets >= 0.1 * n_buckets, (info.front_entries, n_buckets)

        # index and BF::get_index
        assert (info.n_genes, info.n_set_bits, info.tot_ids) == (ref.n_genes, ref.n_set, ref.tot_ids)
        pos, coff, ids = sh.export_index()
        assert np.array_equal(pos, ref.pos) and np.array_equal(coff, ref.off) and np.array_equal(ids, ref.ids)
        kmers = [rng.integers(0, 1 << 62, 20000, dtype=np.uint64) & np.uint64((1 << (2 * k)) - 1)]
        for s in genes:
            e = po.enumerate_kmers(s, k)
            if e is not None:
                kmers.append(e[0])
        kmers = np.concatenate(kmers)
        rank, begin, ln = sh.get_index(kmers)
        r0, b0, l0 = ref.probe(kmers)
        assert np.array_equal(rank, r0) and np.array_equal(begin, b0) and np.array_equal(ln, l0)
        assert (r0 >= 0).sum() > 50_000

        # the reads through K6 on text, K6b and K6 on packed reads
        cnt0, ar0, ag0 = ref.analyze(seq, off, c, qual=qual, min_quality=q, single=single)
        assert len(ar0) > 1000
        stats = {}
        for label, packed, bulk in (("K6 text", False, "1"), ("K6b", True, "1"), ("K6 packed", True, "0")):
            monkeypatch.setenv("SHK_BULK", bulk)
            keep, ar, ag, st = sh.analyze(seq, off, qual, packed=packed)
            assert np.array_equal(keep, (cnt0 > 0).astype(np.uint8)), label
            assert np.array_equal(ar, ar0), label
            assert np.array_equal(ag, ag0), label
            assert st["n_extended"] > 0, label
            stats[label] = st
    for label, st in stats.items():
        assert (st["n_probes"], st["n_hits"]) == (stats["K6b"]["n_probes"], stats["K6b"]["n_hits"]), label
    print("[geometry] %s: front shift %d, coarse shift %d, %d buckets, %d entries, extended/hits %s" % (
        _case_id(case), info.front_shift, info.coarse_shift, n_buckets, info.front_entries,
        " ".join("%s %.2f" % (lb, st["n_extended"] / max(st["n_hits"], 1)) for lb, st in stats.items())))
