"""bench.py's workloads through every path it times, checked against the oracle on the benchmark's own reads and index.

bench.py reports the reads resident in HBM in the packed form as `value`: the bulk kernel (K6b, shk_bulk.cu) over the
index geometry that only a full-size reference produces (table below).  Its own checks compare step totals between
forms; this file compares every result, read by read:

  * the index export against the oracle's, in full (at C4: 56 M set bits);
  * every path bench.py times - resident text, resident packed, text submit with plain and split upload, packed
    submit, K6 on packed reads (SHK_BULK=0), the expanded result form - bit for bit against each other, per chunk;
  * the packed resident result against the oracle on a sample of reads: a prefix of the first chunk, the tail of the
    second (ragged) chunk, seeded random reads and reads the GPU reported as tied.

The workloads are bench.WORKLOADS themselves, two chunks of bench.CHUNK_READS + 333 333 reads built by
bench.make_workload (the same bytes, pinned chunk lists and host-packed copies that bench.py times)."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

# (front shift, coarse shift, plain_front) that front_geometry (shk_index.cu) and build_front give for the key count of
# each workload's reference: C2 ~2.8 M keys in 2^33 bits, C3 14 149 337 in 2^33, C4 56 413 906 in 2^35.  coarse_rel =
# front shift - coarse shift is 6, 3 and 1; C2's front table fits L2 (text reads probe its slots-only copy).
GEOMETRY = {"c2": (11, 5, 1), "c3": (8, 5, 0), "c4": (8, 7, 0)}
EXTRA_READS = 333_333    # the second chunk is ragged
PASSES = 3
ORACLE_HEAD, ORACLE_TAIL, ORACLE_RANDOM, ORACLE_TIED = 65_536, 16_384, 16_384, 4_096

# Non-vacuity floors, about half of what a run on one B200 showed:
#   kept: share of the oracle sample with at least one association (observed C2 0.904, C3 0.834, C4 0.904)
#   tied: reads of the sample with two or more genes (C2 12 118, C4 10 208); for -s workloads (C3), reads of the first
#         16 384 of the sample that -s drops because their best genes tie (1 080)
#   extended: n_extended / n_hits of the packed resident path (C2 0.977, C3 0.977, C4 0.978)
FLOORS = {"c2": dict(kept=0.45, tied=6000, extended=0.45),
          "c3": dict(kept=0.42, tied=540, extended=0.45),
          "c4": dict(kept=0.45, tied=5000, extended=0.45)}
TUNING_VARS = ("SHK_FRONT_LOAD", "SHK_COARSE_LOG2", "SHK_EXTEND", "SHK_BULK")


def _shark(wl, n_chunks, W, compact=True):
    """The context bench.run_workload creates."""
    import bench
    from shark_b200.engine import Shark
    return Shark(k=wl["k"], c=wl["c"], bf_bits=wl["b"] << 33, min_quality=wl["q"], single=wl["single"],
                 n_slots=max(n_chunks, 2), max_reads_per_chunk=bench.CHUNK_READS, max_bytes_per_chunk=bench.CHUNK_READS * W,
                 extend=None, compact=compact)


def _resident(sh, chunks, packed, passes=PASSES):
    """Uploads every chunk once, then `passes` passes of analyze_resident + collect -> list per pass of per-chunk results."""
    for i, c in enumerate(chunks):
        (sh.upload_packed if packed else sh.upload)(i, *c)
    out = []
    for _ in range(passes):
        for i in range(len(chunks)):
            sh.analyze_resident(i)
        out.append([sh.collect(i, copy=True) for i in range(len(chunks))])
    return out


def _oracle_lists(ref, wl, text, qual, idx, threads):
    """The oracle on reads `idx` (sorted) of the fixed-width block -> (kept bool[len(idx)], position in idx of every
    association, gene of every association), in read order, genes ascending."""
    W = text.shape[1]
    pieces = np.array_split(np.arange(len(idx)), threads)

    def one(p):
        sel = idx[p]
        off = np.arange(len(sel) + 1, dtype=np.uint64) * np.uint64(W)
        q = None if qual is None else qual[sel].reshape(-1)
        cnt, ar, ag = ref.analyze(text[sel].reshape(-1), off, wl["c"], qual=q, min_quality=wl["q"], single=wl["single"])
        return cnt > 0, ar.astype(np.int64) + (int(p[0]) if len(p) else 0), ag

    with ThreadPoolExecutor(threads) as ex:   # ctypes releases the GIL; shko_analyze allocates per call
        res = list(ex.map(one, [p for p in pieces if len(p)]))
    return np.concatenate([r[0] for r in res]), np.concatenate([r[1] for r in res]), np.concatenate([r[2] for r in res])


@pytest.mark.parametrize("name", ["c2", "c3", "c4"])
def test_workload_paths_equal_oracle(name, monkeypatch):
    import bench
    from shark_b200 import capi
    from shark_b200.engine import Shark
    for v in TUNING_VARS:
        monkeypatch.delenv(v, raising=False)
    wl = bench.WORKLOADS[name]
    threads = max(1, min(16, len(os.sched_getaffinity(0))))
    wd = bench.make_workload(wl, 0, bench.CHUNK_READS + EXTRA_READS, min(8, threads))
    try:
        chunks, packed, W = wd["chunks"], wd["packed"], wd["W"]
        n_chunks = len(chunks)
        assert n_chunks == 2 and chunks[1][3] == EXTRA_READS
        firsts = np.cumsum([0] + [c[3] for c in chunks])
        n = int(firsts[-1])
        ref = po.Index(wd["bases"], wd["rec_off"], wl["k"], wl["b"] << 33)

        paths = {}
        with _shark(wl, n_chunks, W) as sh:
            # ---- index: the geometry the benchmark runs, and the whole CSR against the oracle
            info = sh.build_index(wd["bases"], wd["rec_off"])
            assert (info.extend, info.front_shift, info.coarse_shift, info.plain_front) == (1, *GEOMETRY[name])
            assert (info.n_genes, info.n_set_bits, info.tot_ids) == (ref.n_genes, ref.n_set, ref.tot_ids)
            pos, off, ids = sh.export_index()
            assert np.array_equal(pos, ref.pos)
            assert np.array_equal(off, ref.off)
            assert np.array_equal(ids, ref.ids)
            del pos, off, ids

            # ---- every path bench.py times
            for p, res in enumerate(_resident(sh, chunks, packed=False)):
                paths["resident text, pass %d" % p] = res
            for p, res in enumerate(_resident(sh, packed, packed=True)):
                paths["resident packed, pass %d" % p] = res
            # plain text upload; split upload (the host packs part of every chunk: text reads go to K6, packed ones to
            # K6b within one chunk), auto-balanced and at a fixed half
            for label, mode in (("plain", False), ("split", True), ("split 0.5", 0.5)):
                sh.set_upload_mode(mode)
                paths["text submit, %s upload" % label] = sh.analyze_chunks(chunks)
            sh.set_upload_mode(False)
            paths["packed submit"] = sh.analyze_chunks(packed, packed=True)
            monkeypatch.setenv("SHK_BULK", "0")   # read at every launch: the thread-per-read kernel on packed reads
            for p, res in enumerate(_resident(sh, packed, packed=True)):
                paths["resident packed K6, pass %d" % p] = res
            monkeypatch.delenv("SHK_BULK")
        head = paths["resident packed, pass 0"]

        # ---- all paths, all passes: bit-identical results and the same window counts, chunk by chunk
        for label, res in paths.items():
            assert len(res) == n_chunks, label
            for i, (r, h) in enumerate(zip(res, head)):
                assert r["n_reads"] == chunks[i][3], (label, i)
                assert np.array_equal(r["gene16"], h["gene16"]), (label, i)
                assert np.array_equal(r["multi"], h["multi"]), (label, i)
                assert (r["n_probes"], r["n_hits"]) == (h["n_probes"], h["n_hits"]), (label, i)

        # ---- the expanded result form of the same context configuration
        with _shark(wl, n_chunks, W, compact=False) as sh:
            sh.build_index(wd["bases"], wd["rec_off"])
            for i, (r, h) in enumerate(zip(_resident(sh, packed, packed=True, passes=1)[0], head)):
                ridx, gidx, keep = Shark.expand(h)
                assert np.array_equal(r["read_idx"], ridx), i
                assert np.array_equal(r["gene_idx"], gidx), i
                assert np.array_equal(r["keep"], keep), i
                assert np.array_equal(r["gene16"], h["gene16"]) and np.array_equal(r["multi"], h["multi"]), i

        # ---- the headline form against the oracle, read by read, on a sample
        gene16 = np.concatenate([h["gene16"] for h in head])
        exp = [Shark.expand(h) for h in head]
        g_read = np.concatenate([e[0].astype(np.int64) + int(f) for e, f in zip(exp, firsts)])
        g_gene = np.concatenate([e[1] for e in exp])
        rng = np.random.default_rng(2024)
        tied = np.nonzero(gene16 == capi.GENE_MULTI)[0]
        idx = np.unique(np.concatenate([
            np.arange(ORACLE_HEAD), np.arange(n - ORACLE_TAIL, n), rng.choice(n, ORACLE_RANDOM, replace=False),
            rng.choice(tied, min(ORACLE_TIED, len(tied)), replace=False)]))
        text = wd["keep"][0].u8[: n * W].reshape(n, W)
        qual = wd["keep"][1].u8[: n * W].reshape(n, W) if wl["q"] else None
        kept0, at0, ag0 = _oracle_lists(ref, wl, text, qual, idx, threads)
        sel = np.isin(g_read, idx)
        assert np.array_equal(gene16[idx] != capi.GENE_NONE, kept0)
        assert np.array_equal(np.searchsorted(idx, g_read[sel]), at0)
        assert np.array_equal(g_gene[sel], ag0)

        # ---- non-vacuity
        n_tied = int(np.isin(idx, tied).sum())
        if wl["single"]:   # -s reports no ties: what is checked is that it drops the reads whose best genes tie
            assert n_tied == 0
            first = idx[:16_384]
            _, at1, _ = _oracle_lists(ref, dict(wl, single=False), text, qual, first, threads)
            n_tied = int((np.bincount(at1, minlength=len(first)) > 1).sum())
        hits = sum(h["n_hits"] for h in head)
        extended = sum(h["n_extended"] for h in head) / max(hits, 1)
        print("[workloads] %s: %d reads sampled, kept %.3f, tied %d%s, extended/hits %.3f" % (
            name, len(idx), kept0.mean(), n_tied, " (without -s)" if wl["single"] else "", extended))
        floor = FLOORS[name]
        assert kept0.mean() >= floor["kept"]
        assert n_tied >= floor["tied"]
        assert extended >= floor["extended"]
    finally:
        for b in wd["keep"]:
            if b is not None:
                b.free()
