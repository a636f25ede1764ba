"""GPU: per-gene read counts accumulated on the device (SHK_F_GENE_COUNTS, shk_gene_counts, the CLI's --counts).

The counts are checked against the oracle's per-read associations aggregated per gene: unique[g] counts the reported reads
whose only association is g, shared[g] the reported reads with g among two or more tied associations.  They are checked on
every submit path and kernel (text with extension automatic, on and off; packed through K6b and through K6 with
SHK_BULK=0; the split upload; wide ids), at several -c and with -s, through both recoveries of shk_reads_collect (tie-pool
overflow: the chunk runs again; multi-list growth: the scatter runs again), across chunks and slots, for repeated resident
analysis, on two contexts, and through the CLI."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import GOLDEN, ROOT, edge_cases, example_cases, flags_to_kwargs, gz_read, stage_edge, stage_example
from oracle import pyoracle as po
from oracle import shark_text as st
from test_gpu_constructed import BF, N_PLAIN, SegRef, families, open_path, classify
from test_gpu_bulk import rc
from test_gpu_parity import ACGT, CASES, rnd_genes, quirky_reference, to_soa
from test_gpu_scores import CASE_IDS, _case_inputs

pytestmark = pytest.mark.gpu

CLI = os.path.join(ROOT, "shark_b200", "shark-b200")


def _shark(**kw):
    from shark_b200.engine import Shark
    return Shark(**kw)


def oracle_counts(cnt, ar, ag, n_genes):
    """(unique, shared) uint64[n_genes] from per-read associations: cnt per read, (ar, ag) the association list."""
    multi = cnt[ar.astype(np.int64)] >= 2
    g = ag.astype(np.int64)
    return (np.bincount(g[~multi], minlength=n_genes).astype(np.uint64),
            np.bincount(g[multi], minlength=n_genes).astype(np.uint64))


def assert_counts(sh, want, what=""):
    u, s = sh.gene_counts()
    assert u.dtype == np.uint64 and s.dtype == np.uint64 and len(u) == len(s) == sh.info.n_genes, what
    bad = np.nonzero((u != want[0]) | (s != want[1]))[0]
    assert len(bad) == 0, (what, bad[:8], u[bad[:4]], want[0][bad[:4]], s[bad[:4]], want[1][bad[:4]])


def counts_of_run(ar, ag, n_reads, n_genes):
    """The same aggregation over a device run's own association list (what shk_reads_collect returned)."""
    cnt = np.bincount(ar.astype(np.int64), minlength=n_reads)
    return oracle_counts(cnt, ar, ag, n_genes)


@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_counts_parity(monkeypatch, case):
    """The parity cases through text (lookup, extend, auto), packed (K6b, and K6 with SHK_BULK=0) and the split upload."""
    bases, rec_off, seq, off, qual = _case_inputs(case)
    ref = po.Index(bases, rec_off, case["k"], case["bf_bits"])
    cnt0, ar0, ag0 = ref.analyze(seq, off, case["c"], qual=qual, min_quality=case["q"], single=case["single"])
    want = oracle_counts(cnt0, ar0, ag0, ref.n_genes)
    assert want[0].sum() + want[1].sum() == cnt0.sum() and (want[0].sum() > 500 or case["c"] == 1.0)
    kw = dict(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], min_quality=case["q"], single=case["single"],
              max_reads_per_chunk=1024, gene_counts=True)
    for path in ("lookup", "extend", "auto", "bulk", "k6_packed", "split"):
        sh, packed = open_path(monkeypatch, path, **kw)
        with sh:
            sh.build_index(bases, rec_off)
            assert_counts(sh, (want[0] * 0, want[1] * 0), (path, "fresh"))
            keep, ar, ag, stats = sh.analyze(seq, off, qual, packed=packed)
            assert np.array_equal(ar, ar0) and np.array_equal(ag, ag0), path
            assert_counts(sh, want, path)
            assert_counts(sh, counts_of_run(ar, ag, len(off) - 1, ref.n_genes), path)


@pytest.mark.parametrize("k,c,single,bf_bits", [(31, 0.6, False, 1 << 30), (11, 0.3, False, 1 << 22), (21, 0.5, True, 1 << 28)])
def test_counts_bulk_stress(monkeypatch, k, c, single, bf_bits):
    """The K6b stress reads (lengths 0 ... 1100 at every alignment of the packed stream), K6b and K6 (SHK_BULK=0)."""
    from test_gpu_bulk import stress_reads
    rng = np.random.default_rng(7000 + k)
    genes = quirky_reference(rng)
    genes += rnd_genes(rng, 20, 1500, 3000)
    genes[45] = genes[44][:700] + genes[45][700:]
    genes[47] = genes[46][300:1200] + genes[47][900:]
    bases, rec_off = po.concat_records(genes)
    texts = stress_reads(rng, [g.upper() for g in genes], 6000, k) + [b"", b"A", b"ACGT" * 8]
    seq, off = to_soa(texts)
    ref = po.Index(bases, rec_off, k, bf_bits)
    want = oracle_counts(*ref.analyze(seq, off, c, single=single), ref.n_genes)
    for bulk in ("1", "0"):
        monkeypatch.setenv("SHK_BULK", bulk)
        with _shark(k=k, c=c, bf_bits=bf_bits, single=single, max_reads_per_chunk=1500, extend=True, compact=True,
                    gene_counts=True) as sh:
            sh.build_index(bases, rec_off)
            sh.analyze(seq, off, None, packed=True)
            assert_counts(sh, want, bulk)


@pytest.mark.parametrize("path", ["auto", "bulk", "wide"])
def test_counts_long_reads_and_wide_reads(monkeypatch, path):
    """From the constructed families: reads of 1024 and 1025 bytes (K6m) and reads of 95 ... 130 genes (K6m / K6x), plus
    the reads inside 2 ... 5-id segments and 130-way ties, at several -c and with -s on one context (set_options +
    reset)."""
    k = 17
    R = SegRef(1000 + k)
    texts = [t for t, f, _ in families(R, k) if f.startswith(("len", "wide", "inside"))]
    texts += [R.seg_piece("w130", 60) for _ in range(20)]
    seq, off = to_soa(texts)
    ref = po.Index(R.bases, R.rec_off, k, BF)
    sh, packed = open_path(monkeypatch, path, k=k, c=0.2, bf_bits=BF, max_reads_per_chunk=256, gene_counts=True)
    with sh:
        sh.build_index(R.bases, R.rec_off)
        for c in (0.0, 0.2, 0.5, 0.8):
            for single in (False, True):
                cnt0, ar0, ag0 = ref.analyze(seq, off, c, single=single)
                want = oracle_counts(cnt0, ar0, ag0, ref.n_genes)
                if c == 0.2 and not single:
                    assert (cnt0 == 130).sum() >= 20 and (np.diff(off.astype(np.int64)) > 1024).sum() >= 12
                sh.reset_gene_counts()
                sh.set_options(c=c, single=single)
                keep, ar, ag, stats = sh.analyze(seq, off, packed=packed)
                assert stats["n_slow_reads"] > 0
                assert_counts(sh, want, (path, c, single))


def test_counts_wide_ids():
    """SHK_F_WIDE_IDS with 70 000 records: gene ids above 65 535, 300-way ties among them; every association travels
    through the multi list and is counted from rec / pool (the kernel's global-memory variant: n_genes > 6144)."""
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
    cnt0, ar0, ag0 = ref.analyze(seq, off, c)
    want = oracle_counts(cnt0, ar0, ag0, ref.n_genes)
    assert want[0][65536:].sum() > 400 and want[1][66000:66300].min() >= 40 and want[0][65534] >= 1
    with _shark(k=k, c=c, bf_bits=bf_bits, max_reads_per_chunk=1000, wide_ids=True, gene_counts=True) as sh:
        sh.build_index(bases, rec_off)
        assert sh.info.n_genes > 6144
        for packed in (False, True):
            sh.reset_gene_counts()
            sh.analyze(seq, off, packed=packed)
            assert_counts(sh, want, packed)


def test_counts_marker_collision():
    """65 536 records: single winners 0xFFFE and 0xFFFF travel through the multi list and are counted unique."""
    rng = np.random.default_rng(5)
    genes = [ACGT[rng.integers(0, 4, 40)].tobytes() for _ in range(65536)]
    bases, rec_off = po.concat_records(genes)
    texts = [genes[i] for i in (0, 1, 65533, 65534, 65535, 65534, 65535, 7)] + [b"N" * 40]
    seq, off = to_soa(texts)
    ref = po.Index(bases, rec_off, 15, 1 << 30)
    cnt0, ar0, ag0 = ref.analyze(seq, off, 0.6)
    want = oracle_counts(cnt0, ar0, ag0, ref.n_genes)
    assert want[0][65534] == 2 and want[0][65535] == 2 and want[1].sum() == 0
    with _shark(k=15, c=0.6, bf_bits=1 << 30, max_reads_per_chunk=1 << 10, compact=True, gene_counts=True) as sh:
        sh.build_index(bases, rec_off)
        r = sh.analyze_chunks([(seq, None, off.astype(np.uint32), len(texts))])[0]
        assert r["n_multi"] >= 4
        assert_counts(sh, want)


@pytest.mark.parametrize("path", ["extend", "bulk", "wide"])
def test_counts_tie_saturated_chunks(monkeypatch, path):
    """Chunks of 2-, 4- and 130-way ties overflow the tie pool (the chunk runs again: its first run must add nothing) and
    the multi list (the scatter runs again: counting is not repeated).  Every association is counted once."""
    k, Rc = 21, 2048
    R = SegRef(21)
    ref = po.Index(R.bases, R.rec_off, k, BF)
    rng = np.random.default_rng(3)
    sat = lambda: [rc(x) if rng.random() < 0.5 else x for x in (R.seg_piece(("s2", "s4", "w130")[i % 3], 60) for i in range(Rc))]
    free = [R.piece(int(g), 60) for g in rng.integers(0, N_PLAIN, 64)]
    sh, packed = open_path(monkeypatch, path, k=k, c=0.5, bf_bits=BF, max_reads_per_chunk=Rc, gene_counts=True)
    with sh:
        sh.build_index(R.bases, R.rec_off)
        out = classify(sh, packed, *to_soa(free), None)
        normal = out[4][0]["kernel_launches"]
        sh.reset_gene_counts()
        texts = sat() + sat()
        seq, off = to_soa(texts)
        out = classify(sh, packed, seq, off, None)
        assert [ch["kernel_launches"] for ch in out[4]][0] == 2 * normal + 1   # re-run + re-scatter on the fresh slot
        cnt0, ar0, ag0 = ref.analyze(seq, off, 0.5)
        want = oracle_counts(cnt0, ar0, ag0, ref.n_genes)
        assert (cnt0 == 130).sum() > 1000 and want[1].sum() == cnt0.sum()
        assert_counts(sh, want, path)


def test_counts_accumulate_across_chunks_and_slots_then_reset():
    """Many chunks round-robin over three slots add up to the whole sample; reset zeroes; a second pass adds again."""
    case = CASES[4]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    ref = po.Index(bases, rec_off, case["k"], case["bf_bits"])
    cnt0, ar0, ag0 = ref.analyze(seq, off, case["c"])
    want = oracle_counts(cnt0, ar0, ag0, ref.n_genes)
    half = (len(off) - 1) // 2
    wh = oracle_counts(*ref.analyze(seq[:int(off[half])], off[:half + 1], case["c"]), ref.n_genes)
    with _shark(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], n_slots=3, max_reads_per_chunk=100, gene_counts=True) as sh:
        sh.build_index(bases, rec_off)
        stats = sh.analyze(seq, off, packed=True)[3]
        assert stats["chunks"] >= 30
        assert_counts(sh, want)
        sh.analyze(seq, off)
        assert_counts(sh, (2 * want[0], 2 * want[1]))
        sh.reset_gene_counts()
        assert_counts(sh, (0 * want[0], 0 * want[1]))
        sh.analyze(seq[:int(off[half])], off[:half + 1])
        assert_counts(sh, wh)


def test_counts_resident_analysis_adds_each_time():
    """shk_reads_analyze_resident adds every time it runs: n analyses of one resident chunk count n times."""
    from shark_b200 import capi
    case = CASES[1]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    ref = po.Index(bases, rec_off, case["k"], case["bf_bits"])
    a, b = 100, 900
    cnt0, ar0, ag0 = ref.analyze(seq[int(off[a]):int(off[b])], off[a:b + 1] - off[a], case["c"])
    want = oracle_counts(cnt0, ar0, ag0, ref.n_genes)
    with _shark(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=1024, gene_counts=True) as sh:
        sh.build_index(bases, rec_off)
        codes, valid = capi.host_pack(seq[int(off[a]):int(off[b])])
        sh.upload_packed(0, codes, valid, (off[a:b + 1] - off[a]).astype(np.uint32), b - a)
        assert_counts(sh, (0 * want[0], 0 * want[1]))   # an upload runs no kernel
        for n in range(1, 4):
            sh.analyze_resident(0)
            sh.collect(0)
            assert_counts(sh, (n * want[0], n * want[1]), n)


def test_results_and_launches_with_the_flag():
    """gene16, multi, score records and every counter of every chunk are the same with and without the flag; each chunk
    has exactly one launch more; D2H bytes grow by the read-back only."""
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
    for flag in (False, True):
        with _shark(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=1024, compact=True, scores=True,
                    gene_counts=flag) as sh:
            sh.build_index(bases, rec_off)
            out[flag] = sh.analyze_chunks(chunks)
            d2h[flag] = sh.lib.shk_d2h_bytes(sh.ctx)
            if flag:
                sh.gene_counts()
                assert sh.lib.shk_d2h_bytes(sh.ctx) - d2h[flag] == 16 * sh.info.n_genes
                u = np.zeros(sh.info.n_genes, np.uint64)
                before = sh.lib.shk_d2h_bytes(sh.ctx)
                assert sh.lib.shk_gene_counts(sh.ctx, capi.ptr(u), None, sh.info.n_genes) == 0
                assert sh.lib.shk_d2h_bytes(sh.ctx) - before == 8 * sh.info.n_genes and u.sum() > 0
    assert d2h[False] == d2h[True]
    for r0, r1 in zip(out[False], out[True]):
        assert np.array_equal(r0["gene16"], r1["gene16"]) and np.array_equal(r0["multi"], r1["multi"])
        assert np.array_equal(r0["scores"], r1["scores"])
        for key in ("n_probes", "n_hits", "n_multi", "n_kept", "n_assoc", "n_slow_reads", "n_extended", "n_table_loads"):
            assert r0[key] == r1[key], key
        assert r1["kernel_launches"] == r0["kernel_launches"] + 1


def test_two_contexts_sum_to_one():
    """Half the reads on each of two contexts - a replicated index and a sharded build - sum to one context's counts."""
    import torch
    case = CASES[1]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    n = len(off) - 1
    half = n // 2
    parts = [(seq[:int(off[half])], off[:half + 1]), (seq[int(off[half]):], off[half:] - off[half])]
    kw = dict(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=512, gene_counts=True)
    dev1 = 1 if torch.cuda.device_count() >= 2 else 0
    with _shark(**kw) as sh:
        sh.build_index(bases, rec_off)
        sh.analyze(seq, off)
        whole = sh.gene_counts()
        assert whole[0].sum() > 1000
        with _shark(device=dev1, **kw) as dst:
            assert dst.lib.shk_index_replicate(sh.ctx, dst.ctx) == 0
            dst.info = sh.info
            assert_counts(dst, (0 * whole[0], 0 * whole[1]), "replica fresh")
            sh.reset_gene_counts()
            sh.analyze(*parts[0])
            dst.analyze(*parts[1])
            u0, s0 = sh.gene_counts()
            u1, s1 = dst.gene_counts()
            assert np.array_equal(u0 + u1, whole[0]) and np.array_equal(s0 + s1, whole[1])
    from shark_b200.engine import Shark
    with _shark(**kw) as a, _shark(device=dev1, **kw) as b:
        Shark.build_index_sharded([a, b], bases, rec_off)
        for sh, p in zip((a, b), parts):
            assert_counts(sh, (0 * whole[0], 0 * whole[1]), "sharded fresh")
            sh.analyze(*p)
        (u0, s0), (u1, s1) = a.gene_counts(), b.gene_counts()
        assert np.array_equal(u0 + u1, whole[0]) and np.array_equal(s0 + s1, whole[1])


def test_counts_zeroed_when_an_index_becomes_ready(tmp_path):
    """A rebuild and a load start the counts at zero."""
    case = CASES[0]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    with _shark(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=1024, gene_counts=True) as sh:
        sh.build_index(bases, rec_off)
        sh.analyze(seq, off)
        u, s = sh.gene_counts()
        assert u.sum() > 0
        sh.save_index(tmp_path / "ix.bin")
        sh.load_index(tmp_path / "ix.bin")
        assert_counts(sh, (0 * u, 0 * s), "load")
        sh.analyze(seq, off)
        assert_counts(sh, (u, s), "after load")
        sh.build_index(bases, rec_off)
        assert_counts(sh, (0 * u, 0 * s), "rebuild")


def test_counts_argument_and_state_errors():
    from shark_b200 import capi
    case = CASES[0]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    kw = dict(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=1024)
    u = np.zeros(1 << 12, np.uint64)
    with _shark(**kw) as sh:   # without the flag
        sh.build_index(bases, rec_off)
        n = sh.info.n_genes
        assert sh.lib.shk_gene_counts(sh.ctx, capi.ptr(u), capi.ptr(u), n) == -3
        assert sh.lib.shk_gene_counts_reset(sh.ctx) == -3
        launches = sh.lib.shk_kernel_launches(sh.ctx)
        stats = sh.analyze(seq, off)[3]
        assert sh.lib.shk_kernel_launches(sh.ctx) - launches == stats["kernel_launches"]
    with _shark(gene_counts=True, **kw) as sh:
        assert sh.lib.shk_gene_counts(sh.ctx, capi.ptr(u), capi.ptr(u), 0) == -3   # no index
        assert sh.lib.shk_gene_counts_reset(sh.ctx) == -3
        sh.build_index(bases, rec_off)
        n = sh.info.n_genes
        assert sh.lib.shk_gene_counts(sh.ctx, capi.ptr(u), capi.ptr(u), n + 1) == -1
        assert sh.lib.shk_gene_counts(sh.ctx, capi.ptr(u), capi.ptr(u), n - 1) == -1
        assert sh.lib.shk_gene_counts(sh.ctx, None, None, n) == 0
        o32 = off[:101].astype(np.uint32)
        pin = capi.PinnedBuffer(int(off[100]) + 64)
        pin.u8[:int(off[100])] = seq[:int(off[100])]
        sh.submit(1, pin.u8, None, o32, 100)
        assert sh.lib.shk_gene_counts(sh.ctx, capi.ptr(u), None, n) == -3   # slot 1 in flight
        assert sh.lib.shk_gene_counts_reset(sh.ctx) == -3
        assert b"uncollected" in sh.lib.shk_last_error(sh.ctx)
        sh.collect(1)
        assert sh.lib.shk_gene_counts(sh.ctx, capi.ptr(u), None, n) == 0 and u[:n].sum() > 0
        assert sh.lib.shk_gene_counts_reset(sh.ctx) == 0
        assert sh.lib.shk_gene_counts(sh.ctx, capi.ptr(u), None, n) == 0 and u[:n].sum() == 0


# ---- the CLI ---------------------------------------------------------------------------------------------------
def run_cli(args, cwd, env=None):
    p = subprocess.run([CLI] + args, cwd=str(cwd), stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       env=dict(os.environ, **(env or {})))
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stdout


def cli_oracle_counts(ref_path, s1, s2, k, c, b, q, single):
    """The expected counts file: `<legend[g]> <unique> <shared>` for every gene index g."""
    legend, seqs = st.load_reference(ref_path)
    bases, rec_off = po.concat_records(seqs)
    pairs, _ = st.load_sample(s1, s2)
    seq, qual, off = st.join_reads(pairs, q > 0)
    ref = po.Index(bases, rec_off, k, b << 33)
    cnt, ar, ag = ref.analyze(seq, off, c, qual=qual, min_quality=q, single=single)
    u, s = oracle_counts(cnt, ar, ag, ref.n_genes)
    return b"".join(b"%s %d %d\n" % (legend[g] if g < len(legend) else b"", u[g], s[g]) for g in range(ref.n_genes))


def _cli_case(tmp_path, ref, s1, s2, flags, extra=()):
    args = ["-r", ref, "-1", s1, "-o", "o1.fq", "--counts", "o.counts"] + (["-2", s2, "-p", "o2.fq"] if s2 else [])
    ssv = run_cli(args + list(flags) + list(extra), tmp_path)
    rd = lambda f: open(os.path.join(str(tmp_path), f), "rb").read()
    return ssv, rd("o1.fq"), (rd("o2.fq") if s2 else None), rd("o.counts")


@pytest.mark.parametrize("scenario,case", [(s, c) for s, cs in sorted(edge_cases().items()) for c in sorted(cs)] +
                         [("example", c) for c in sorted(example_cases()["cases"])])
def test_cli_counts_goldens(tmp_path, scenario, case):
    """The counts file against the oracle; the ssv and FASTQ bytes are the reference's goldens, as without --counts."""
    if scenario == "example":
        info = example_cases()["cases"][case]
        f = stage_example(tmp_path)
        ref, s1, s2 = f["ENSG00000277117.fa"], f["sample_1.fq"], f["sample_2.fq"] if info["paired"] else None
    else:
        info = edge_cases()[scenario][case]
        f = stage_edge(tmp_path, scenario)
        ref, s1, s2 = f["ref.fa"], f["r1.fq"], f.get("r2.fq") if info["paired"] else None
    ssv, o1, o2, counts = _cli_case(tmp_path, ref, s1, s2, info["flags"])
    if scenario == "example":
        from helpers import md5
        assert (md5(ssv), md5(o1)) == (info["ssv_md5"], info["o1_md5"])
        if s2:
            assert md5(o2) == info["o2_md5"]
    else:
        d = os.path.join(GOLDEN, "edge", scenario)
        assert ssv == gz_read(os.path.join(d, case + ".ssv.gz")) and o1 == gz_read(os.path.join(d, case + ".o1.fq.gz"))
        if s2:
            assert o2 == gz_read(os.path.join(d, case + ".o2.fq.gz"))
    kw = flags_to_kwargs(info["flags"])
    assert counts == cli_oracle_counts(ref, s1, s2, kw["k"], kw["c"], kw["b"], kw["q"], kw["single"])
    # unique + shared per name = the ssv's lines per name (names may repeat: compare per gene index through the legend)
    tot = sum(int(x.split(b" ")[-1]) + int(x.split(b" ")[-2]) for x in counts.splitlines())
    assert tot == ssv.count(b"\n")


def test_cli_counts_options(tmp_path):
    """--counts with gzip inputs, small chunks, SHK_ONE_PROCESS=1, --load-index, --wide-ids, --scores, and --gpus 2 /
    --sharded-build when two devices are visible: the same counts file, ssv and FASTQ each time, and the ssv and FASTQ of
    a run without --counts."""
    import torch
    d = os.path.join(GOLDEN, "example")
    f = stage_example(tmp_path)
    ssv0, o10, o20, c0 = _cli_case(tmp_path, f["ENSG00000277117.fa"], f["sample_1.fq"], f["sample_2.fq"], [], ["--save-index", "ix.bin"])
    assert c0.count(b"\n") >= 1 and sum(int(x.split(b" ")[1]) for x in c0.splitlines()) > 1000
    gz = ["-r", os.path.join(d, "ENSG00000277117.fa.gz"), "-1", os.path.join(d, "sample_1.fq.gz"), "-2", os.path.join(d, "sample_2.fq.gz")]
    variants = [(gz + ["--chunk-reads", "1000"], {}), (gz, {"SHK_ONE_PROCESS": "1"}), (gz + ["--load-index", "ix.bin"], {}),
                (gz + ["--wide-ids"], {}), (gz + ["--scores", "v.scores"], {})]
    if torch.cuda.device_count() >= 2:
        variants += [(gz + ["--gpus", "2", "--chunk-reads", "1000"], {}), (gz + ["--gpus", "2", "--sharded-build"], {})]
    rd = lambda p: open(os.path.join(str(tmp_path), p), "rb").read()
    for args, env in variants:
        ssv = run_cli(args + ["-o", "v1.fq", "-p", "v2.fq", "--counts", "v.counts"], tmp_path, env)
        assert ssv == ssv0 and rd("v1.fq") == o10 and rd("v2.fq") == o20, (args, env)
        assert rd("v.counts") == c0, (args, env)
    ssv = run_cli(gz + ["-o", "w1.fq", "-p", "w2.fq"], tmp_path)
    assert ssv == ssv0 and rd("w1.fq") == o10 and rd("w2.fq") == o20


def test_cli_counts_edge_scenarios_multi_gpu(tmp_path):
    """Several genes, ties and the index/name quirk (edge 'multi' reference) through --wide-ids and, when two devices are
    visible, --gpus 2 with and without --sharded-build: the oracle's counts file each time."""
    import torch
    f = stage_edge(tmp_path, "multi")
    want = cli_oracle_counts(f["ref.fa"], f["r1.fq"], f["r2.fq"], 17, 0.3, 1, 0, False)
    base = ["-r", f["ref.fa"], "-1", f["r1.fq"], "-2", f["r2.fq"], "-c", "0.3", "-o", "x1.fq", "-p", "x2.fq", "--counts", "x.counts"]
    ssv0 = run_cli(base[:-2], tmp_path)
    variants = [[], ["--wide-ids"], ["--chunk-reads", "1000"]]
    if torch.cuda.device_count() >= 2:
        variants += [["--gpus", "2", "--chunk-reads", "1000"], ["--gpus", "2", "--sharded-build", "--chunk-reads", "1000"]]
    for v in variants:
        ssv = run_cli(base + v, tmp_path)
        assert ssv == ssv0, v
        assert open(os.path.join(str(tmp_path), "x.counts"), "rb").read() == want, v
    assert any(int(x.split(b" ")[2]) > 0 for x in want.splitlines())   # the edge reference has ties
