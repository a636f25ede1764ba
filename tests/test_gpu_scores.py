"""GPU: per-read score records (SHK_F_SCORES).  Every field of every record against the oracle's per-read gene table
(pyoracle.Index.read_table on the -q-masked text), on every submit path and kernel; results with the flag identical to
those without; the rule "reported iff n_best > 0 and cov >= c * len and (not -s or n_best == 1), with n_best
associations" on every run; one run at c = 0 filtered by that rule equal to real runs at other (c, -s); the records'
lifetime; and the CLI's --scores file."""
import os
import subprocess

import numpy as np
import pytest

from helpers import GOLDEN, ROOT, edge_cases, example_cases, flags_to_kwargs, gz_read, stage_edge, stage_example
from oracle import pyoracle as po
from oracle import shark_text as st
from test_gpu_parity import ACGT, CASES, quals_for, quirky_reference, rnd_genes, sample_reads, to_soa

pytestmark = pytest.mark.gpu

CLI = os.path.join(ROOT, "shark_b200", "shark-b200")
VALID = np.zeros(256, bool)
VALID[np.frombuffer(b"ACGTacgt", np.uint8)] = True


def _shark(**kw):
    from shark_b200.engine import Shark
    return Shark(**kw)


def oracle_scores(ref, seq, off, qual=None, q=0, cap=4096):
    """uint32[n, 4]: {len, cov, hits, n_best} per read, from the oracle's per-gene table of the masked text."""
    n = len(off) - 1
    out = np.zeros((n, 4), np.uint32)
    for i in range(n):
        t = seq[int(off[i]):int(off[i + 1])]
        if q:
            t = po.mask(t, qual[int(off[i]):int(off[i + 1])], q)
        out[i, 0] = VALID[t].sum()
        g, cv, h = ref.read_table(t.tobytes(), cap)
        if len(g):
            mc = cv.max()
            mh = h[cv == mc].max()
            out[i, 1:] = (mc, mh, ((cv == mc) & (h == mh)).sum())
    return out


def rule(scores, c, single):
    keep = (scores[:, 3] > 0) & (scores[:, 1].astype(np.float64) >= np.float64(c) * scores[:, 0].astype(np.float64))
    if single:
        keep &= scores[:, 3] == 1
    return keep


def check_invariant(scores, ar, n, c, single):
    """Reported iff the rule holds, and then with exactly n_best associations."""
    cnt = np.bincount(ar.astype(np.int64), minlength=n)[:n]
    keep = rule(scores, c, single)
    assert np.array_equal(cnt > 0, keep)
    assert np.array_equal(cnt[keep], scores[keep, 3])


def _case_inputs(case):
    rng = np.random.default_rng(case["k"] * 7 + case["L"])
    genes = quirky_reference(rng)
    bases, rec_off = po.concat_records(genes)
    texts = sample_reads(rng, genes, 3000, case["L"], paired=case["paired"])
    texts += [b"", b"A", b"N" * 50, b"ACGT" * 10 + b"N" + b"ACGT" * 10, b"ACGTN" * 12, b"acgt" * 12 + b"n.-*" + b"ACGT" * 10]
    texts += [ACGT[rng.integers(0, 4, int(n))].tobytes() for n in rng.integers(1, 70, 64)]
    seq, off = to_soa(texts)
    qual = None
    if case["q"]:
        qual = quals_for(rng, texts)
        if case["paired"]:
            for i in range(3000):
                qual[int(off[i]) + case["L"]] = 0x1B
    return bases, rec_off, seq, off, qual


CASE_IDS = lambda c: "k%d_c%g_b%d_q%d_%s%s_L%d" % (c["k"], c["c"], c["bf_bits"], c["q"], "s" if c["single"] else "m",
                                                 "pe" if c["paired"] else "se", c["L"])


@pytest.mark.parametrize("extend", [None, True, False], ids=["auto", "extend", "lookup"])
@pytest.mark.parametrize("case", CASES, ids=CASE_IDS)
def test_scores_parity(case, extend):
    """Text, packed and split upload (share 0.5): records equal to the oracle's, results equal to a run without the
    flag, the rule on every run."""
    bases, rec_off, seq, off, qual = _case_inputs(case)
    n = len(off) - 1
    ref = po.Index(bases, rec_off, case["k"], case["bf_bits"])
    want = oracle_scores(ref, seq, off, qual, case["q"])
    cnt0, ar0, ag0 = ref.analyze(seq, off, case["c"], qual=qual, min_quality=case["q"], single=case["single"])
    kw = dict(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], min_quality=case["q"], single=case["single"],
              max_reads_per_chunk=1024, extend=extend)
    runs = {}
    with _shark(**kw) as sh:
        sh.build_index(bases, rec_off)
        base = {p: sh.analyze(seq, off, qual, packed=p) for p in (False, True)}
    with _shark(scores=True, **kw) as sh:
        sh.build_index(bases, rec_off)
        for p in (False, True):
            runs["packed" if p else "text"] = (base[p], sh.analyze(seq, off, qual, packed=p))
    with _shark(scores=True, host_pack=0.5, **kw) as sh:
        sh.build_index(bases, rec_off)
        runs["split"] = (base[False], sh.analyze(seq, off, qual))
    for name, ((k0, a0, g0, s0), (keep, ar, ag, stats)) in runs.items():
        assert stats["scores"].shape == (n, 4), name
        assert np.array_equal(stats["scores"], want), (name, np.nonzero((stats["scores"] != want).any(1))[0][:10])
        assert np.array_equal(keep, k0) and np.array_equal(ar, a0) and np.array_equal(ag, g0), name
        assert (stats["n_probes"], stats["n_hits"]) == (s0["n_probes"], s0["n_hits"]), name
        assert np.array_equal(ar, ar0) and np.array_equal(ag, ag0), name
        check_invariant(stats["scores"], ar, n, case["c"], case["single"])
    assert (want[:, 3] > 0).sum() > 1000 and (want[:, 3] > 1).sum() > 0


def test_compact_results_unchanged_by_the_flag():
    """gene16, multi, n_probes and n_hits of every chunk are the same with and without the flag (compact form)."""
    case = CASES[4]   # k = 5: many genes per read, ties, the warp-per-read kernels
    bases, rec_off, seq, off, qual = _case_inputs(case)
    from shark_b200 import capi
    o32 = off.astype(np.uint32)
    chunks, pins = [], []   # (the pinned buffers must outlive the runs)
    for a in range(0, len(off) - 1, 700):
        b = min(a + 700, len(off) - 1)
        pins.append(capi.PinnedBuffer(int(off[b] - off[a]) + 64))
        pins[-1].u8[:int(off[b] - off[a])] = seq[int(off[a]):int(off[b])]
        chunks.append((pins[-1].u8, None, (o32[a:b + 1] - o32[a]).astype(np.uint32), b - a))
    out = {}
    for flag in (False, True):
        with _shark(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=1024, compact=True, scores=flag) as sh:
            sh.build_index(bases, rec_off)
            out[flag] = sh.analyze_chunks(chunks)
    assert len(out[True]) == len(chunks)
    for r0, r1 in zip(out[False], out[True]):
        assert np.array_equal(r0["gene16"], r1["gene16"]) and np.array_equal(r0["multi"], r1["multi"])
        assert (r0["n_probes"], r0["n_hits"], r0["n_multi"], r0["n_kept"]) == (r1["n_probes"], r1["n_hits"], r1["n_multi"], r1["n_kept"])
        assert r0["scores"] is None and r1["scores"].shape == (r1["n_reads"], 4)
        assert (r1["multi"][:, 0] < r1["n_reads"]).all()


@pytest.mark.parametrize("k,c,single,bf_bits", [(31, 0.6, False, 1 << 30), (21, 0.5, True, 1 << 28), (11, 0.3, False, 1 << 22),
                                                 (25, 0.0, False, 1000003)])
def test_scores_bulk_stress(monkeypatch, k, c, single, bf_bits):
    """The K6b stress reads (lengths 0 ... 1100 at every alignment of the packed stream) through the bulk kernel and
    through analyze_reads_kernel (SHK_BULK=0)."""
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
    want = oracle_scores(ref, seq, off)
    cnt0, ar0, ag0 = ref.analyze(seq, off, c, single=single)
    for bulk in ("1", "0"):
        monkeypatch.setenv("SHK_BULK", bulk)
        with _shark(k=k, c=c, bf_bits=bf_bits, single=single, max_reads_per_chunk=1500, extend=True, compact=True, scores=True) as sh:
            sh.build_index(bases, rec_off)
            keep, ar, ag, stats = sh.analyze(seq, off, None, packed=True)
        assert np.array_equal(stats["scores"], want), bulk
        assert np.array_equal(ar, ar0) and np.array_equal(ag, ag0), bulk
        check_invariant(stats["scores"], ar, len(texts), c, single)
    assert (want[:, 0] > 1024).sum() > 20


def test_scores_long_reads_and_300_way_ties():
    """Reads longer than 1024 bases and lists of 300 genes: the warp-per-read kernels write the records."""
    rng = np.random.default_rng(99)
    core = ACGT[rng.integers(0, 4, 400)].tobytes()
    genes = [core + ACGT[rng.integers(0, 4, 300)].tobytes() for _ in range(300)]
    genes += rnd_genes(rng, 20, 2500, 3000)
    bases, rec_off = po.concat_records(genes)
    texts = []
    for i in range(200):
        texts.append(core[i:i + 120])
        texts.append(genes[300 + i % 20][:1500 + i])
        texts.append(genes[i][350:500])
    seq, off = to_soa(texts)
    for extend in (None, False):
        for k, c, single in ((17, 0.6, False), (17, 0.6, True), (25, 0.2, False)):
            ref = po.Index(bases, rec_off, k, 1 << 28)
            want = oracle_scores(ref, seq, off)
            with _shark(k=k, c=c, bf_bits=1 << 28, single=single, max_reads_per_chunk=256, max_bytes_per_chunk=1 << 20,
                        extend=extend, scores=True) as sh:
                sh.build_index(bases, rec_off)
                for packed in (False, True):
                    keep, ar, ag, stats = sh.analyze(seq, off, packed=packed)
                    assert stats["n_slow_reads"] >= 300
                    assert np.array_equal(stats["scores"], want), (extend, k, single, packed)
                    check_invariant(stats["scores"], ar, len(texts), c, single)
            assert (want[:, 3] == 300).sum() >= 100 and (want[:, 0] > 1024).sum() == 200


def test_scores_degenerate_reads():
    """Empty reads, all-N reads, reads with fewer than k valid bases or without k valid bases in a row: {len, 0, 0, 0}."""
    rng = np.random.default_rng(5)
    genes = rnd_genes(rng, 10)
    bases, rec_off = po.concat_records(genes)
    k = 17
    texts = [b"", b"N" * 40, b"ACG", genes[0][:16], b"ACGTNACGTNACGTNACGTNACGTN" * 4, b"acgtacgtacgtacgtN" * 3, b".-*" * 30,
             genes[1][:16] + b"N" + genes[1][17:33], genes[2][:200]]
    seq, off = to_soa(texts)
    ref = po.Index(bases, rec_off, k, 1 << 24)
    want = oracle_scores(ref, seq, off)
    assert want[:-1, 1:].sum() == 0 and want[-1, 3] == 1
    assert want[:, 0].tolist()[:8] == [0, 0, 3, 16, 80, 48, 0, 32]
    for extend in (None, True, False):
        with _shark(k=k, c=0.6, bf_bits=1 << 24, max_reads_per_chunk=64, extend=extend, scores=True) as sh:
            sh.build_index(bases, rec_off)
            for packed in (False, True):
                assert np.array_equal(sh.analyze(seq, off, packed=packed)[3]["scores"], want), (extend, packed)


def test_scores_wide_ids():
    """SHK_F_WIDE_IDS with the 70 000-record reference, against the widened oracle."""
    rng = np.random.default_rng(70)
    genes = [ACGT[rng.integers(0, 4, int(rng.integers(36, 60)))].tobytes() for _ in range(70000)]
    for i in range(0, 3000, 7):
        genes[65536 + i] = genes[i][:30] + genes[65536 + i][30:]
    core = ACGT[rng.integers(0, 4, 40)].tobytes()
    for i in range(66000, 66300):
        genes[i] = core + genes[i][:12]
    genes[100] = b"N" * 40
    bases, rec_off = po.concat_records(genes)
    k, bf_bits, c = 15, 1 << 31, 0.5
    ref = po.Index(bases, rec_off, k, bf_bits, wide=True)
    texts = [genes[i] for i in rng.integers(0, 70000, 2000)]
    texts += [genes[65536 + i] for i in range(0, 3000, 7)] + [genes[i][:30] for i in range(0, 3000, 7)]
    texts += [core[i:i + 30] for i in range(10)] + [core] * 30 + [b"", b"N" * 30, b"ACGTACGTAC"]
    seq, off = to_soa(texts)
    want = oracle_scores(ref, seq, off, cap=1 << 17)
    assert (want[:, 3] == 300).sum() >= 30 and (want[:, 3] == 2).sum() > 300
    with _shark(k=k, c=c, bf_bits=bf_bits, max_reads_per_chunk=1000, wide_ids=True, scores=True) as sh:
        sh.build_index(bases, rec_off)
        for packed in (False, True):
            keep, ar, ag, stats = sh.analyze(seq, off, packed=packed)
            assert np.array_equal(stats["scores"], want), packed
            check_invariant(stats["scores"], ar, len(texts), c, False)


@pytest.mark.parametrize("case", [CASES[0], CASES[1], CASES[2], CASES[4], CASES[5], CASES[6], CASES[11]], ids=CASE_IDS)
def test_classify_once_threshold_later(case):
    """One run at c = 0 without -s, filtered by the rule, equals real runs at (c', s) association for association."""
    bases, rec_off, seq, off, qual = _case_inputs(case)
    n = len(off) - 1
    with _shark(k=case["k"], c=0.0, bf_bits=case["bf_bits"], min_quality=case["q"], single=False, max_reads_per_chunk=1024,
                scores=True) as sh:
        sh.build_index(bases, rec_off)
        keep, ar, ag, stats = sh.analyze(seq, off, qual)
        sc = stats["scores"]
        check_invariant(sc, ar, n, 0.0, False)
        has = sc[:, 3] > 0
        ratios = np.unique(sc[has, 1].astype(np.float64) / sc[has, 0].astype(np.float64))
        bounds = [float(x) for x in ratios[np.linspace(0, len(ratios) - 1, 8).astype(int)] if 0 <= x <= 1]
        for c in [0.05, 0.3, 0.6, 0.75, 1.0] + bounds:
            for single in (False, True):
                sel = rule(sc, c, single)[ar.astype(np.int64)]
                sh.set_options(c=c, single=single)
                k2, ar2, ag2, st2 = sh.analyze(seq, off, qual)
                assert np.array_equal(ar[sel], ar2) and np.array_equal(ag[sel], ag2), (c, single)
                assert np.array_equal(st2["scores"], sc), (c, single)
                check_invariant(st2["scores"], ar2, n, c, single)


def test_scores_lifetime():
    """Many chunks through 2 slots; repeated analyze_resident gives the same records; SHK_E_STATE without the flag,
    before the first collect, after an upload and while a chunk is in flight."""
    from shark_b200 import capi
    import ctypes as C
    case = CASES[1]
    bases, rec_off, seq, off, qual = _case_inputs(case)
    ref = po.Index(bases, rec_off, case["k"], case["bf_bits"])
    want = oracle_scores(ref, seq, off)
    sp, nn = C.POINTER(capi.ReadScore)(), C.c_uint32()
    with _shark(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=100, scores=True) as sh:
        sh.build_index(bases, rec_off)
        state = lambda slot: sh.lib.shk_reads_scores(sh.ctx, slot, C.byref(sp), C.byref(nn))
        assert state(0) == -3 and state(1) == -3 and state(2) == -1
        keep, ar, ag, stats = sh.analyze(seq, off, packed=True)
        assert stats["chunks"] >= 30 and np.array_equal(stats["scores"], want)
        a, b = 100, 200
        o32 = (off[a:b + 1] - off[a]).astype(np.uint32)
        codes, valid = capi.host_pack(seq[int(off[a]):int(off[b])])
        sh.upload_packed(0, codes, valid, o32, b - a)
        assert state(0) == -3
        first = None
        for _ in range(3):
            sh.analyze_resident(0)
            assert state(0) == -3
            r = sh.collect(0)
            assert state(0) == 0 and nn.value == b - a
            assert np.array_equal(r["scores"], want[a:b])
            if first is not None:
                assert np.array_equal(r["scores"], first) and np.array_equal(r["gene16"], g16)
            first, g16 = r["scores"], r["gene16"]
    with _shark(k=case["k"], c=case["c"], bf_bits=case["bf_bits"], max_reads_per_chunk=100) as sh:
        sh.build_index(bases, rec_off)
        sh.analyze(seq[:int(off[50])], off[:51])
        assert sh.lib.shk_reads_scores(sh.ctx, 0, C.byref(sp), C.byref(nn)) == -3


# ---- the CLI ---------------------------------------------------------------------------------------------------
def run_cli(args, cwd, env=None):
    p = subprocess.run([CLI] + args, cwd=str(cwd), stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       env=dict(os.environ, **(env or {})))
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    return p.stdout


def parse_scores(data):
    out = []
    for ln in data.splitlines():
        name, *v = ln.rsplit(b" ", 4)
        out.append((name, tuple(int(x) for x in v)))
    return out


def pair_up(ssv, scores):
    """[(score line, its ssv lines)]: a scores line with n_best = m goes with the next m ssv lines, all of its name."""
    lines = ssv.splitlines(keepends=True)
    out, i = [], 0
    for name, v in scores:
        part = lines[i:i + v[3]]
        assert len(part) == v[3] and all(x.split(b" ")[0] == name for x in part), (name, v, part[:3])
        out.append(((name, v), part))
        i += v[3]
    assert i == len(lines)
    return out


def cli_oracle_scores(ref_path, s1, s2, k, c, b, q, single):
    """The oracle's records of the reads the reference reports, in read order."""
    legend, seqs = st.load_reference(ref_path)
    bases, rec_off = po.concat_records(seqs)
    pairs, _ = st.load_sample(s1, s2)
    seq, qual, off = st.join_reads(pairs, q > 0)
    ref = po.Index(bases, rec_off, k, b << 33)
    cnt, _, _ = ref.analyze(seq, off, c, qual=qual, min_quality=q, single=single)
    sc = oracle_scores(ref, seq, off, qual, q)
    return [tuple(int(x) for x in sc[i]) for i in np.nonzero(cnt)[0]]


def _cli_case(tmp_path, ref, s1, s2, flags, extra=()):
    args = ["-r", ref, "-1", s1, "-o", "o1.fq", "--scores", "o.scores"] + (["-2", s2, "-p", "o2.fq"] if s2 else [])
    ssv = run_cli(args + list(flags) + list(extra), tmp_path)
    rd = lambda f: open(os.path.join(str(tmp_path), f), "rb").read()
    return ssv, rd("o1.fq"), (rd("o2.fq") if s2 else None), rd("o.scores")


@pytest.mark.parametrize("scenario,case", [(s, c) for s, cs in sorted(edge_cases().items()) for c in sorted(cs)] +
                         [("example", c) for c in sorted(example_cases()["cases"])])
def test_cli_scores_goldens(tmp_path, scenario, case):
    if scenario == "example":
        info = example_cases()["cases"][case]
        f = stage_example(tmp_path)
        ref, s1, s2 = f["ENSG00000277117.fa"], f["sample_1.fq"], f["sample_2.fq"] if info["paired"] else None
    else:
        info = edge_cases()[scenario][case]
        f = stage_edge(tmp_path, scenario)
        ref, s1, s2 = f["ref.fa"], f["r1.fq"], f.get("r2.fq") if info["paired"] else None
    ssv, o1, o2, sc = _cli_case(tmp_path, ref, s1, s2, info["flags"])
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
    recs = parse_scores(sc)
    pair_up(ssv, recs)
    kw = flags_to_kwargs(info["flags"])
    assert [v for _, v in recs] == cli_oracle_scores(ref, s1, s2, kw["k"], kw["c"], kw["b"], kw["q"], kw["single"])


def _filtered_ssv(ssv, sc, c, single):
    out = []
    for (name, v), part in pair_up(ssv, parse_scores(sc)):
        if v[3] > 0 and float(v[1]) >= c * float(v[0]) and (not single or v[3] == 1):
            out += part
    return b"".join(out)


@pytest.mark.parametrize("scenario,runs", [("multi", [(0.6, False, "pe_default"), (1.0, False, "pe_c1")]),
                                           ("io", [(0.6, False, "pe"), (0.6, True, "pe_s")])])
def test_cli_threshold_later_equals_reference_goldens(tmp_path, scenario, runs):
    """One CLI run at -c 0 --scores, its ssv filtered with the rule, equals the reference's own goldens byte for byte."""
    f = stage_edge(tmp_path, scenario)
    ssv, _, _, sc = _cli_case(tmp_path, f["ref.fa"], f["r1.fq"], f["r2.fq"], ["-c", "0"])
    for c, single, golden in runs:
        want = gz_read(os.path.join(GOLDEN, "edge", scenario, golden + ".ssv.gz"))
        assert _filtered_ssv(ssv, sc, c, single) == want, (c, single, golden)


def test_cli_scores_options(tmp_path):
    """--scores with gzip inputs, small chunks, SHK_ONE_PROCESS=1, --save-index / --load-index, --wide-ids, and
    --gpus 2 / --sharded-build when two devices are visible: the same scores file and ssv each time."""
    import torch
    d = os.path.join(GOLDEN, "example")
    f = stage_example(tmp_path)
    ssv0, _, _, sc0 = _cli_case(tmp_path, f["ENSG00000277117.fa"], f["sample_1.fq"], f["sample_2.fq"], [], ["--save-index", "ix.bin"])
    assert sc0.count(b"\n") > 1000
    gz = ["-r", os.path.join(d, "ENSG00000277117.fa.gz"), "-1", os.path.join(d, "sample_1.fq.gz"), "-2", os.path.join(d, "sample_2.fq.gz")]
    variants = [(gz + ["--chunk-reads", "1000"], {}), (gz, {"SHK_ONE_PROCESS": "1"}),
                (gz + ["--load-index", "ix.bin"], {}), (gz + ["--wide-ids"], {})]
    if torch.cuda.device_count() >= 2:
        variants += [(gz + ["--gpus", "2", "--chunk-reads", "1000"], {}), (gz + ["--gpus", "2", "--sharded-build"], {})]
    for args, env in variants:
        ssv = run_cli(args + ["-o", "v1.fq", "-p", "v2.fq", "--scores", "v.scores"], tmp_path, env)
        assert ssv == ssv0, (args, env)
        assert open(os.path.join(str(tmp_path), "v.scores"), "rb").read() == sc0, (args, env)
