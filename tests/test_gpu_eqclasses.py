"""GPU: reads per equivalence class accumulated on the device (SHK_F_EQ_CLASSES, shk_eq_classes, the CLI's --eqclasses).

A reported read's class is the tuple of its associations in ascending gene order; the expected table groups the oracle's
association list by read and counts each tuple.  Every check also holds the table against the same run's gene counts
(singleton {g} = unique[g]; the classes containing g add up to unique[g] + shared[g]) and its own association list
(sum of counts = reported reads, sum of count * |S| = associations).  Covered: every submit path and kernel at several -c
and with -s, wide ids, constructed tie families, tens of thousands of classes (the table grows and the leftover pass
runs), equal hashes of unequal lists (SHK_EQ_HASH_BITS), both recoveries of shk_reads_collect, resident analysis, every
route to a ready index, two contexts, the errors, the default path, and the CLI."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import GOLDEN, edge_cases, example_cases, flags_to_kwargs, stage_edge, stage_example
from oracle import pyoracle as po
from oracle import shark_text as st
from test_gpu_constructed import BF, N_PLAIN, SegRef, families, open_path, classify
from test_gpu_bulk import rc
from test_gpu_counts import CLI, run_cli
from test_gpu_parity import ACGT, CASES, to_soa
from test_gpu_scores import CASE_IDS, _case_inputs

pytestmark = pytest.mark.gpu


def _shark(**kw):
    from shark_b200.engine import Shark
    return Shark(**kw)


def classes_of(ar, ag):
    """{tuple of genes: reads} from an association list ordered by read then gene."""
    ar, ag = np.asarray(ar, np.int64), np.asarray(ag, np.int64)
    out = {}
    if len(ar):
        for grp in np.split(ag, np.flatnonzero(np.diff(ar)) + 1):
            t = tuple(int(g) for g in grp)
            out[t] = out.get(t, 0) + 1
    return out


def table(sh):
    """The device table as [(tuple, count)], checked for its own form: ascending lists, sorted, no zero counts."""
    offsets, ids, counts = sh.eq_classes()
    assert offsets.dtype == np.uint64 and ids.dtype == np.uint32 and counts.dtype == np.uint64
    assert len(offsets) == len(counts) + 1 and offsets[0] == 0 and offsets[-1] == len(ids)
    rows = [(tuple(int(g) for g in ids[offsets[i]:offsets[i + 1]]), int(counts[i])) for i in range(len(counts))]
    keys = [r[0] for r in rows]
    assert keys == sorted(keys) and len(set(keys)) == len(keys) and all(c > 0 for _, c in rows)
    assert all(len(k) >= 1 and list(k) == sorted(set(k)) for k in keys)
    return rows


def assert_classes(sh, want, what="", single=False):
    """The table equals `want` ({tuple: count}) and agrees with the same context's gene counts."""
    rows = table(sh)
    got = dict(rows)
    if got != want:
        miss = [(k, want[k], got.get(k)) for k in sorted(want) if got.get(k) != want[k]][:4]
        extra = [(k, got[k]) for k in sorted(got) if k not in want][:4]
        raise AssertionError((what, len(got), len(want), miss, extra))
    u, s = sh.gene_counts()
    tot = np.zeros(len(u), np.uint64)
    sing = np.zeros(len(u), np.uint64)
    for k, c in rows:
        tot[list(k)] += np.uint64(c)
        if len(k) == 1:
            sing[k[0]] = c
    assert np.array_equal(sing, u) and np.array_equal(tot, u + s), what
    if single:
        assert all(len(k) == 1 for k, _ in rows), what
    return rows


def totals(rows):
    return sum(c for _, c in rows), sum(c * len(k) for k, c in rows)


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_eq_parity(monkeypatch, case):
    """The parity cases through text (lookup, extend, auto), packed (K6b, and K6 with SHK_BULK=0) and the split upload."""
    bases, rec_off, seq, off, qual = _case_inputs(case)
    ref = po.Index(bases, rec_off, case["k"], case["bf_bits"])
    cnt0, ar0, ag0 = ref.analyze(seq, off, case["c"], qual=qual, min_quality=case["q"], single=case["single"])
    want = classes_of(ar0, ag0)
    kw = dict(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], min_quality=case["q"], single=case["single"],
              max_reads_per_chunk=1024, gene_counts=True, eq_classes=True)
    for path in ("lookup", "extend", "auto", "bulk", "k6_packed", "split"):
        sh, packed = open_path(monkeypatch, path, **kw)
        with sh:
            sh.build_index(bases, rec_off)
            assert table(sh) == [], path
            keep, ar, ag, stats, chunks = classify(sh, packed, seq, off, qual)
            assert np.array_equal(ar, ar0) and np.array_equal(ag, ag0), path
            rows = assert_classes(sh, want, path, case["single"])
            assert totals(rows) == (sum(ch["n_kept"] for ch in chunks), sum(ch["n_assoc"] for ch in chunks)), path
            assert totals(rows) == (int(keep.sum()), len(ar)), path
            if case["single"]:
                u = sh.gene_counts()[0]
                assert rows == [((g,), int(u[g])) for g in np.flatnonzero(u)]


@pytest.mark.parametrize("path", ["auto", "bulk", "wide"])
def test_eq_constructed_families(monkeypatch, path):
    """Ties inside 2 ... 5-id segments, 31/32/33- and 130-way ties, reads of 1024/1025 bytes and of 95 ... 130 genes
    (K6m / K6x), at several -c and with -s on one context (set_options + reset between them)."""
    k = 17
    R = SegRef(1000 + k)
    texts = [t for t, f, _ in families(R, k)]
    texts += [R.seg_piece("w130", 60) for _ in range(20)]
    seq, off = to_soa(texts)
    ref = po.Index(R.bases, R.rec_off, k, BF)
    sh, packed = open_path(monkeypatch, path, k=k, c=0.2, bf_bits=BF, max_reads_per_chunk=256, eq_classes=True)
    with sh:
        sh.build_index(R.bases, R.rec_off)
        for c in (0.0, 0.2, 0.5, 0.8):
            for single in (False, True):
                cnt0, ar0, ag0 = ref.analyze(seq, off, c, single=single)
                want = classes_of(ar0, ag0)
                if c == 0.2 and not single:
                    sizes = {len(t) for t in want}
                    assert {2, 3, 4, 5, 130} <= sizes and max(sizes) >= 130, sorted(sizes)
                sh.reset_gene_counts()
                assert table(sh) == []
                sh.set_options(c=c, single=single)
                sh.analyze(seq, off, packed=packed)
                assert_classes(sh, want, (path, c, single), single)


def test_eq_wide_ids():
    """SHK_F_WIDE_IDS with 70 000 records: ids above 65 535 and 300-way ties among them."""
    rng = np.random.default_rng(70)
    genes = [ACGT[rng.integers(0, 4, int(rng.integers(36, 60)))].tobytes() for _ in range(70000)]
    for i in range(0, 3000, 7):
        genes[65536 + i] = genes[i][:30] + genes[65536 + i][30:]
    core = ACGT[rng.integers(0, 4, 40)].tobytes()
    for i in range(66000, 66300):
        genes[i] = core + genes[i][:12]
    bases, rec_off = po.concat_records(genes)
    k, bf_bits, c = 15, 1 << 31, 0.5
    ref = po.Index(bases, rec_off, k, bf_bits, wide=True)
    texts = [genes[i] for i in rng.integers(0, 70000, 2000)]
    texts += [genes[65536 + i] for i in range(0, 3000, 7)] + [genes[i][:30] for i in range(0, 3000, 7)]
    texts += [core[i:i + 30] for i in range(10)] + [core] * 30 + [b"", b"N" * 30, genes[65535], genes[65534], genes[69999]]
    seq, off = to_soa(texts)
    want = classes_of(*ref.analyze(seq, off, c)[1:])
    assert tuple(range(66000, 66300)) in want and any(len(t) == 2 and t[0] >= 65536 or t[-1] >= 65536 for t in want)
    with _shark(k=k, c=c, bf_bits=bf_bits, max_reads_per_chunk=1000, wide_ids=True, eq_classes=True) as sh:
        sh.build_index(bases, rec_off)
        for packed in (False, True):
            sh.reset_gene_counts()
            sh.analyze(seq, off, packed=packed)
            assert_classes(sh, want, packed)


def many_classes(n_rec, n_seg, seed=11):
    """A reference in which each of n_seg random 40-base segments is copied into a random subset of 2 ... 6 of n_rec
    records, and reads that are those segments (some twice, some reverse-complemented): one class per segment."""
    rng = np.random.default_rng(seed)
    parts = [[ACGT[rng.integers(0, 4, 30)].tobytes()] for _ in range(n_rec)]
    segs = [ACGT[rng.integers(0, 4, 40)].tobytes() for _ in range(n_seg)]
    for s in segs:
        for r in rng.choice(n_rec, int(rng.integers(2, 7)), replace=False):
            parts[r].append(s + ACGT[rng.integers(0, 4, 3)].tobytes())
    genes = [b"".join(p) for p in parts]
    bases, rec_off = po.concat_records(genes)
    texts = [rc(s) if i % 3 == 0 else s for i, s in enumerate(segs)] + segs[: n_seg // 4]
    return bases, rec_off, texts


@pytest.fixture(scope="module")
def many():
    bases, rec_off, texts = many_classes(3000, 24000)
    seq, off = to_soa(texts)
    ref = po.Index(bases, rec_off, 21, 1 << 30)
    cnt0, ar0, ag0 = ref.analyze(seq, off, 0.8)
    return bases, rec_off, seq, off, classes_of(ar0, ag0)


def test_eq_many_classes_grow_and_leftovers(many):
    """Tens of thousands of classes over several chunks and both slots, from the initial 4096 slots: the table grows and
    the leftover pass runs (more launches than the same chunks without the class table), and nothing is lost or counted
    twice."""
    bases, rec_off, seq, off, want = many
    assert len(want) > 20000 and sum(1 for t in want if len(t) >= 2) > 20000
    launches = {}
    for eq in (False, True):
        with _shark(k=21, c=0.8, bf_bits=1 << 30, max_reads_per_chunk=4096, gene_counts=True, eq_classes=eq) as sh:
            sh.build_index(bases, rec_off)
            keep, ar, ag, stats, chunks = classify(sh, True, seq, off, None)
            assert len(chunks) >= 6
            launches[eq] = [ch["kernel_launches"] for ch in chunks]
            if eq:
                rows = assert_classes(sh, want)
                assert totals(rows) == (int(keep.sum()), len(ar))
    extra = [b - a for a, b in zip(launches[False], launches[True])]
    assert min(extra) >= 0 and sum(extra) >= 6, extra   # >= 3 growths, each with its rehash and a leftover pass


def test_eq_one_launch_brings_more_new_classes_than_slots():
    """One chunk of 160 000 reads over 40 000 classes: K8's first wave alone (about 4 700 resident warps, each starting
    on a new class) asks for more slots than the initial 4096.  Claims stop at the load limit, the table grows and the
    leftover pass places the rest: the table is the grouping of the chunk's own results."""
    bases, rec_off, texts = many_classes(6000, 40000, seed=13)
    texts = [texts[i] for i in np.random.default_rng(13).permutation(len(texts))] * 4
    seq, off = to_soa(texts[:160000])
    with _shark(k=21, c=0.8, bf_bits=1 << 30, max_reads_per_chunk=1 << 18, eq_classes=True) as sh, \
            _shark(k=21, c=0.8, bf_bits=1 << 30, max_reads_per_chunk=1 << 18, gene_counts=True) as base:
        for x in (sh, base):
            x.build_index(bases, rec_off)
        keep, ar, ag, stats, chunks = classify(sh, True, seq, off, None)
        assert len(chunks) == 1
        want = classes_of(ar, ag)
        assert sum(1 for t in want if len(t) >= 2) > 30000
        assert_classes(sh, want)
        ref_chunks = classify(base, True, seq, off, None)[4]
        assert chunks[0]["kernel_launches"] >= ref_chunks[0]["kernel_launches"] + 6   # >= 3 growths + leftover passes
        classify(sh, False, seq, off, None)
        assert_classes(sh, {t: 2 * c for t, c in want.items()})


def test_eq_two_threads_grow_while_the_other_submits(many):
    """One host thread submits and collects slot 0 while another does slot 1, from the initial table size: growth in one
    thread's collect races the other thread's K8 enqueues (the context mutex orders them).  The table is the sum of what
    both threads collected."""
    import threading
    from shark_b200 import capi
    bases, rec_off, seq, off, want = many
    o32 = off.astype(np.uint32)
    bounds = [(a, min(a + 2048, len(off) - 1)) for a in range(0, len(off) - 1, 2048)]
    with _shark(k=21, c=0.8, bf_bits=1 << 30, n_slots=2, max_reads_per_chunk=2048, eq_classes=True) as sh:
        sh.build_index(bases, rec_off)
        got, errors = [{}, {}], []

        def worker(slot):
            try:
                for a, b in bounds[slot::2]:
                    pin = capi.PinnedBuffer(int(off[b] - off[a]) + 64)
                    pin.u8[:int(off[b] - off[a])] = seq[int(off[a]):int(off[b])]
                    sh.submit(slot, pin.u8, None, (o32[a:b + 1] - o32[a]).astype(np.uint32), b - a)
                    r = sh.collect(slot)
                    for t, c in classes_of(r["read_idx"], r["gene_idx"]).items():
                        got[slot][t] = got[slot].get(t, 0) + c
                    del pin
            except Exception as e:   # reported by the main thread
                errors.append((slot, e))

        threads = [threading.Thread(target=worker, args=(i,)) for i in (0, 1)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        assert not errors, errors
        both = {t: got[0].get(t, 0) + got[1].get(t, 0) for t in set(got[0]) | set(got[1])}
        assert both == want
        assert_classes(sh, want)


@pytest.mark.parametrize("bits", [0, 1, 4])
def test_eq_equal_hashes(monkeypatch, bits):
    """With the list hash cut to 0, 1 or 4 bits, unequal lists share hashes: the table is the same."""
    bases, rec_off, texts = many_classes(600, 5000, seed=12)
    seq, off = to_soa(texts)
    ref = po.Index(bases, rec_off, 21, 1 << 28)
    want = classes_of(*ref.analyze(seq, off, 0.8)[1:])
    monkeypatch.setenv("SHK_EQ_HASH_BITS", str(bits))
    with _shark(k=21, c=0.8, bf_bits=1 << 28, n_slots=3, max_reads_per_chunk=1024, eq_classes=True) as sh:
        sh.build_index(bases, rec_off)
        sh.analyze(seq, off, packed=True)
        assert_classes(sh, want, bits)
        sh.analyze(seq, off)
        assert_classes(sh, {t: 2 * c for t, c in want.items()}, bits)


@pytest.mark.parametrize("path", ["extend", "bulk", "wide"])
def test_eq_tie_saturated_chunks(monkeypatch, path):
    """Chunks of 2-, 4- and 130-way ties overflow the tie pool (the chunk runs again) and the multi list (the scatter
    runs again): every read is in the table once."""
    k, Rc = 21, 2048
    R = SegRef(21)
    ref = po.Index(R.bases, R.rec_off, k, BF)
    rng = np.random.default_rng(3)
    sat = lambda: [rc(x) if rng.random() < 0.5 else x for x in (R.seg_piece(("s2", "s4", "w130")[i % 3], 60) for i in range(Rc))]
    free = [R.piece(int(g), 60) for g in rng.integers(0, N_PLAIN, 64)]
    sh, packed = open_path(monkeypatch, path, k=k, c=0.5, bf_bits=BF, max_reads_per_chunk=Rc, eq_classes=True)
    with sh:
        sh.build_index(R.bases, R.rec_off)
        out = classify(sh, packed, *to_soa(free), None)
        normal = out[4][0]["kernel_launches"]
        sh.reset_gene_counts()
        seq, off = to_soa(sat() + sat())
        out = classify(sh, packed, seq, off, None)
        assert out[4][0]["kernel_launches"] >= 2 * normal + 1
        cnt0, ar0, ag0 = ref.analyze(seq, off, 0.5)
        assert (cnt0 == 130).sum() > 1000
        assert_classes(sh, classes_of(ar0, ag0), path)


def test_eq_resident_analysis_adds_each_time():
    from shark_b200 import capi
    case = CASES[1]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    ref = po.Index(bases, rec_off, case["k"], case["bf_bits"])
    a, b = 100, 900
    want = classes_of(*ref.analyze(seq[int(off[a]):int(off[b])], off[a:b + 1] - off[a], case["c"])[1:])
    with _shark(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=1024, eq_classes=True) as sh:
        sh.build_index(bases, rec_off)
        codes, valid = capi.host_pack(seq[int(off[a]):int(off[b])])
        sh.upload_packed(0, codes, valid, (off[a:b + 1] - off[a]).astype(np.uint32), b - a)
        assert table(sh) == []
        for n in range(1, 4):
            sh.analyze_resident(0)
            sh.collect(0)
            assert_classes(sh, {t: n * c for t, c in want.items()}, n)


def test_eq_empty_on_every_route_to_a_ready_index(tmp_path):
    """Build, rebuild, load, replicate (adopt + copies + finalize), sharded build and the staged protocol's
    switch_mode(2) each start with an empty table; reset empties it; set_options between chunks changes what later
    chunks add."""
    from shark_b200.engine import Shark
    from test_functors import _staged_build
    case = CASES[0]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    ref = po.Index(bases, rec_off, case["k"], case["bf_bits"])
    want = classes_of(*ref.analyze(seq, off, case["c"])[1:])
    kw = dict(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=1024, eq_classes=True)
    with _shark(**kw) as sh:
        sh.build_index(bases, rec_off)
        sh.analyze(seq, off)
        assert_classes(sh, want)
        sh.save_index(tmp_path / "ix.bin")
        for route in ("load", "rebuild", "replicate"):
            if route == "load":
                sh.load_index(tmp_path / "ix.bin")
            elif route == "rebuild":
                sh.build_index(bases, rec_off)
            else:
                with _shark(**kw) as src:
                    src.build_index(bases, rec_off)
                    assert sh.lib.shk_index_replicate(src.ctx, sh.ctx) == 0
            assert table(sh) == [], route
            sh.analyze(seq, off)
            assert_classes(sh, want, route)
        sh.reset_gene_counts()
        assert table(sh) == []
        half = (len(off) - 1) // 2
        sh.analyze(seq[:int(off[half])], off[:half + 1])
        sh.set_options(c=0.0)
        sh.analyze(seq[int(off[half]):], off[half:] - off[half])
        w0 = classes_of(*ref.analyze(seq[:int(off[half])], off[:half + 1], case["c"])[1:])
        w1 = classes_of(*ref.analyze(seq[int(off[half]):], off[half:] - off[half], 0.0)[1:])
        assert_classes(sh, {t: w0.get(t, 0) + w1.get(t, 0) for t in set(w0) | set(w1)}, "set_options")
    with _shark(**kw) as a, _shark(**kw) as b:
        Shark.build_index_sharded([a, b], bases, rec_off)
        assert table(a) == [] and table(b) == []
    with _shark(**kw) as sh:
        _staged_build(sh, [bases[rec_off[i]:rec_off[i + 1]].tobytes() for i in range(len(rec_off) - 1)], case["k"])
        assert table(sh) == []
        sh.analyze(seq, off)
        assert dict(table(sh)) == want


def test_eq_two_contexts_sum_to_one():
    import torch
    from shark_b200.engine import Shark
    case = CASES[1]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    half = (len(off) - 1) // 2
    parts = [(seq[:int(off[half])], off[:half + 1]), (seq[int(off[half]):], off[half:] - off[half])]
    kw = dict(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=512, eq_classes=True)
    dev1 = 1 if torch.cuda.device_count() >= 2 else 0
    add = lambda x, y: {t: x.get(t, 0) + y.get(t, 0) for t in set(x) | set(y)}
    with _shark(**kw) as sh:
        sh.build_index(bases, rec_off)
        sh.analyze(seq, off)
        whole = dict(table(sh))
        assert sum(1 for t in whole if len(t) >= 2) >= 2
        with _shark(device=dev1, **kw) as dst:
            assert dst.lib.shk_index_replicate(sh.ctx, dst.ctx) == 0
            dst.info = sh.info
            sh.reset_gene_counts()
            sh.analyze(*parts[0])
            dst.analyze(*parts[1])
            assert add(dict(table(sh)), dict(table(dst))) == whole
    with _shark(**kw) as a, _shark(device=dev1, **kw) as b:
        Shark.build_index_sharded([a, b], bases, rec_off)
        for sh, p in zip((a, b), parts):
            sh.analyze(*p)
        assert add(dict(table(a)), dict(table(b))) == whole


def test_eq_state_and_capacity_errors():
    from shark_b200 import capi
    case = CASES[0]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    kw = dict(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=1024)
    n, m = C.c_uint64(), C.c_uint64()
    call = lambda sh, *a: sh.lib.shk_eq_classes(sh.ctx, C.byref(n), C.byref(m), *a)
    for flags in (dict(), dict(gene_counts=True)):   # without the flag
        with _shark(**kw, **flags) as sh:
            sh.build_index(bases, rec_off)
            assert call(sh, None, None, None, 0, 0) == -3
            assert b"SHK_F_EQ_CLASSES" in sh.lib.shk_last_error(sh.ctx)
    with _shark(eq_classes=True, **kw) as sh:
        assert call(sh, None, None, None, 0, 0) == -3   # no index
        sh.build_index(bases, rec_off)
        assert call(sh, None, None, None, 0, 0) == 0 and n.value == 0 and m.value == 0
        o1 = np.ones(1, np.uint64)
        assert call(sh, capi.ptr(o1), None, None, 0, 0) == 0 and o1[0] == 0   # an empty table needs no ids or counts
        sh.analyze(seq, off)
        assert call(sh, None, None, None, 0, 0) == 0 and n.value > 1 and m.value > n.value
        N, M = n.value, m.value
        o, ids, cnt = np.zeros(N + 1, np.uint64), np.zeros(M, np.uint32), np.zeros(N, np.uint64)
        P = capi.ptr
        assert call(sh, P(o), P(ids), P(cnt), N - 1, M) == -4
        assert call(sh, P(o), P(ids), P(cnt), N, M - 1) == -4
        assert (n.value, m.value) == (N, M)
        assert call(sh, P(o), None, P(cnt), N, M) == -1
        assert sh.lib.shk_eq_classes(sh.ctx, None, C.byref(m), None, None, None, 0, 0) == -1
        before = sh.lib.shk_d2h_bytes(sh.ctx)
        assert call(sh, P(o), P(ids), P(cnt), N, M) == 0 and o[-1] == M and cnt.sum() > 0
        assert sh.lib.shk_d2h_bytes(sh.ctx) > before
        o32 = off[:101].astype(np.uint32)
        pin = capi.PinnedBuffer(int(off[100]) + 64)
        pin.u8[:int(off[100])] = seq[:int(off[100])]
        sh.submit(1, pin.u8, None, o32, 100)
        assert call(sh, None, None, None, 0, 0) == -3   # slot 1 in flight
        assert b"uncollected" in sh.lib.shk_last_error(sh.ctx)
        sh.collect(1)
        assert call(sh, None, None, None, 0, 0) == 0


def test_default_path_untouched():
    """With gene_counts=True and no class flag, every chunk's results, counters and D2H bytes are those of a run without
    either flag, with K8's one launch more; with the class flag the results are still the same."""
    from shark_b200 import capi
    case = CASES[4]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    o32 = off.astype(np.uint32)
    chunks, pins = [], []
    for a in range(0, len(off) - 1, 700):
        b = min(a + 700, len(off) - 1)
        pins.append(capi.PinnedBuffer(int(off[b] - off[a]) + 64))
        pins[-1].u8[:int(off[b] - off[a])] = seq[int(off[a]):int(off[b])]
        chunks.append((pins[-1].u8, None, (o32[a:b + 1] - o32[a]).astype(np.uint32), b - a))
    out, d2h = {}, {}
    for arm in ("none", "counts", "eq"):
        with _shark(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=1024, compact=True, scores=True,
                    gene_counts=arm == "counts", eq_classes=arm == "eq") as sh:
            sh.build_index(bases, rec_off)
            out[arm] = sh.analyze_chunks(chunks)
            d2h[arm] = sh.lib.shk_d2h_bytes(sh.ctx)
    assert d2h["none"] == d2h["counts"]
    for r0, r1, r2 in zip(out["none"], out["counts"], out["eq"]):
        for r in (r1, r2):
            assert np.array_equal(r0["gene16"], r["gene16"]) and np.array_equal(r0["multi"], r["multi"])
            assert np.array_equal(r0["scores"], r["scores"])
            for key in ("n_probes", "n_hits", "n_multi", "n_kept", "n_assoc", "n_slow_reads", "n_extended", "n_table_loads"):
                assert r0[key] == r[key], key
        assert r1["kernel_launches"] == r0["kernel_launches"] + 1


# ---- the CLI ---------------------------------------------------------------------------------------------------
def cli_oracle_classes(ref_path, s1, s2, k, c, b, q, single):
    """The expected --eqclasses file: `<count> <legend[g] ...>` per class, in sorted order of the index tuples."""
    legend, seqs = st.load_reference(ref_path)
    bases, rec_off = po.concat_records(seqs)
    pairs, _ = st.load_sample(s1, s2)
    seq, qual, off = st.join_reads(pairs, q > 0)
    ref = po.Index(bases, rec_off, k, b << 33)
    want = classes_of(*ref.analyze(seq, off, c, qual=qual, min_quality=q, single=single)[1:])
    name = lambda g: legend[g] if g < len(legend) else b""
    return b"".join(b" ".join([b"%d" % want[t]] + [name(g) for g in t]) + b"\n" for t in sorted(want))


def _cli(tmp_path, ref, s1, s2, flags, extra=()):
    args = ["-r", ref, "-1", s1, "-o", "o1.fq", "--eqclasses", "o.eq"] + (["-2", s2, "-p", "o2.fq"] if s2 else [])
    ssv = run_cli(args + list(flags) + list(extra), tmp_path)
    rd = lambda f: open(os.path.join(str(tmp_path), f), "rb").read()
    return ssv, rd("o1.fq"), (rd("o2.fq") if s2 else None), rd("o.eq")


@pytest.mark.parametrize("scenario,case", [(s, c) for s, cs in sorted(edge_cases().items()) for c in sorted(cs)] +
                         [("example", c) for c in sorted(example_cases()["cases"])])
def test_cli_eqclasses_goldens(tmp_path, scenario, case):
    """The class file against the oracle's table rendered with the ssv's names; its associations add up to the ssv's
    lines; the ssv and FASTQ bytes are those of a run without the option."""
    if scenario == "example":
        info = example_cases()["cases"][case]
        f = stage_example(tmp_path)
        ref, s1, s2 = f["ENSG00000277117.fa"], f["sample_1.fq"], f["sample_2.fq"] if info["paired"] else None
    else:
        info = edge_cases()[scenario][case]
        f = stage_edge(tmp_path, scenario)
        ref, s1, s2 = f["ref.fa"], f["r1.fq"], f.get("r2.fq") if info["paired"] else None
    ssv, o1, o2, eq = _cli(tmp_path, ref, s1, s2, info["flags"])
    args = ["-r", ref, "-1", s1, "-o", "n1.fq"] + (["-2", s2, "-p", "n2.fq"] if s2 else [])
    assert run_cli(args + list(info["flags"]), tmp_path) == ssv
    assert open(os.path.join(str(tmp_path), "n1.fq"), "rb").read() == o1
    if s2:
        assert open(os.path.join(str(tmp_path), "n2.fq"), "rb").read() == o2
    kw = flags_to_kwargs(info["flags"])
    assert eq == cli_oracle_classes(ref, s1, s2, kw["k"], kw["c"], kw["b"], kw["q"], kw["single"])
    assert sum(int(x.split(b" ")[0]) * (len(x.split(b" ")) - 1) for x in eq.splitlines()) == ssv.count(b"\n")
    if kw["single"]:
        assert all(len(x.split(b" ")) == 2 for x in eq.splitlines())


def test_cli_eqclasses_options(tmp_path):
    """-s, --wide-ids, --counts together, small chunks and --gpus 2 (with two devices): the oracle's file each time and
    the ssv of a run without the option."""
    import torch
    f = stage_edge(tmp_path, "multi")
    base = ["-r", f["ref.fa"], "-1", f["r1.fq"], "-2", f["r2.fq"], "-c", "0.3", "-o", "x1.fq", "-p", "x2.fq"]
    for single in (False, True):
        want = cli_oracle_classes(f["ref.fa"], f["r1.fq"], f["r2.fq"], 17, 0.3, 1, 0, single)
        s = ["-s"] if single else []
        ssv0 = run_cli(base + s, tmp_path)
        variants = [[], ["--wide-ids"], ["--chunk-reads", "1000"], ["--counts", "x.counts"]]
        if torch.cuda.device_count() >= 2:
            variants += [["--gpus", "2", "--chunk-reads", "1000"], ["--gpus", "2", "--sharded-build", "--chunk-reads", "1000"]]
        for v in variants:
            assert run_cli(base + s + v + ["--eqclasses", "x.eq"], tmp_path) == ssv0, v
            assert open(os.path.join(str(tmp_path), "x.eq"), "rb").read() == want, (single, v)
        if not single:
            assert any(len(x.split(b" ")) > 2 for x in want.splitlines())   # the edge reference has ties
