"""The reference's functor seam (SURVEY.md 8b, seam 2): KmerBuilder / BloomfilterFiller / class BF /
ReadAnalyzer re-implemented over the C ABI (include/shark_b200_functors.hpp, the staged shk_bf_* calls).

CPU: the header compiles stand-alone, and the hybrid executable fails loudly without a device.
GPU: every staged call against the oracle, the protocol end to end against the one-call build, and the
hybrid executable byte-for-byte against the reference's goldens.
The hybrid executable is the reference's own main.cpp built on the header (oracle/_ref/shark_hybrid) where that has
been built, and otherwise tests/host_tools/functor_main.cpp, a restatement of that driver on the same header."""
import os
import subprocess

import numpy as np
import pytest

from helpers import GOLDEN, ROOT, edge_cases, example_cases, gz_read, md5, stage_edge, stage_example

REF_HYBRID = os.path.join(ROOT, "oracle", "_ref", "shark_hybrid")
REF = os.path.join(ROOT, "oracle", "_ref", "shark")


@pytest.fixture(scope="module", autouse=True)
def _built():
    from shark_b200 import build
    build.build()
    from oracle import pyoracle
    pyoracle.build()


@pytest.fixture(scope="module")
def hybrid(tmp_path_factory):
    if os.path.exists(REF_HYBRID):
        return REF_HYBRID
    out = str(tmp_path_factory.mktemp("hybrid") / "functor_main")
    lib = os.path.join(ROOT, "shark_b200")
    subprocess.check_call(["g++", "-O2", "-std=c++14", "-Wall", "-I", os.path.join(ROOT, "include"), "-I",
                           os.path.join(ROOT, "tests", "host_tools"), os.path.join(ROOT, "tests", "host_tools", "functor_main.cpp"),
                           "-o", out, "-L", lib, "-lshark_b200", "-Wl,-rpath," + lib, "-Wl,-rpath-link,/usr/local/cuda/lib64",
                           "-lz", "-pthread"])
    return out


# ------------------------------------------------------------------------------------------- CPU
def test_functor_header_compiles_standalone(tmp_path):
    """No reference tree needed: the header carries the interface types itself (common.hpp:30-36)."""
    src = tmp_path / "t.cpp"
    src.write_text(
        '#include "shark_b200_functors.hpp"\n'
        "int use(BF* bf, const vector<string>& legend) {\n"
        "  KmerBuilder kb(17); BloomfilterFiller bff(bf);\n"
        "  auto* texts = new vector<pair<string,string>>(); texts->push_back({\"g\", \"ACGT\"});\n"
        "  bff(kb(texts)); bf->add_at(7); bool ok = bf->switch_mode(1);\n"
        "  vector<uint64_t> kmers{1, 2}; bf->add_to_kmer(kmers, 0); ok = bf->switch_mode(2) && ok;\n"
        "  auto it = bf->get_index(5); (void)it;\n"
        "  ReadAnalyzer ra(bf, legend, 17, 0.6, true); vector<elem_t> reads; ReadAnalyzer::output_t out;\n"
        "  ra(reads, out); return ok ? (int)out.size() : -1; }\n")
    subprocess.run(["g++", "-std=c++14", "-Wall", "-Werror", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)],
                   check=True)


def test_hybrid_fails_loudly_without_gpu(tmp_path, hybrid):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    f = stage_example(tmp_path)
    p = subprocess.run([hybrid, "-r", f["ENSG00000277117.fa"], "-1", f["sample_1.fq"]], cwd=str(tmp_path),
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    assert p.returncode == 1 and p.stdout == b"" and b"no CUDA device" in p.stderr


# ------------------------------------------------------------------------------------------- GPU
def _records(rng, n, lo=20, hi=400):
    """Random records with N runs, lower case, records shorter than k and an all-N record (Q1)."""
    recs = []
    for i in range(n):
        L = int(rng.integers(lo, hi))
        s = bytearray(rng.choice(np.frombuffer(b"ACGT", np.uint8), L).tobytes())
        if i % 4 == 1:
            p = int(rng.integers(0, L))
            s[p:p + int(rng.integers(1, 4))] = b"N" * min(3, L - p)
        if i % 7 == 2:
            s = bytearray(bytes(s).lower())
        if i % 11 == 5:
            s = bytearray(b"N" * 40)
        if i % 13 == 6:
            s = bytearray(b"ACGTA")
        if i % 5 == 3 and i > 0:  # shared segment with the previous record: multi-gene lists
            m = min(len(s), len(recs[i - 1]), 60)
            s[:m] = recs[i - 1][:m]
        recs.append(bytes(s))
    return recs


def _expected_hashes(recs, k):
    from oracle import pyoracle as po
    out = []
    for s in recs:
        if len(s) < k:
            continue
        e = po.enumerate_kmers(s, k)
        if e is None:
            continue
        out += [po.xxh64_u64(int(v)) for v in e[0]]
    return np.array(out, dtype=np.uint64)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 5, 17, 31])
def test_kmer_hashes_match_kmerbuilder(k):
    """shk_kmer_hashes == KmerBuilder::operator() (KmerBuilder.hpp:40-72), order included."""
    from oracle import pyoracle as po
    from shark_b200.engine import Shark
    rng = np.random.default_rng(100 + k)
    recs = _records(rng, 120)
    bases, off = po.concat_records(recs)
    with Shark(k=k, bf_bits=1 << 20, max_reads_per_chunk=64) as sh:
        got = sh.kmer_hashes(bases, off)
        assert np.array_equal(got, _expected_hashes(recs, k))
        # batches of 100 records (main.cpp:132) give the same stream
        parts = [sh.kmer_hashes(*po.concat_records(recs[i:i + 100])) for i in range(0, len(recs), 100)]
        assert np.array_equal(np.concatenate(parts), got)
        assert len(sh.kmer_hashes(np.zeros(0, np.uint8), np.zeros(1, np.uint64))) == 0


def _staged_build(sh, recs, k, batch=100):
    """main.cpp:128-193 with the library's staged calls; returns the final nidx."""
    from oracle import pyoracle as po
    for i in range(0, len(recs), batch):  # pass 1: FastaSplitter -> KmerBuilder -> BloomfilterFiller
        sh.add_at(sh.kmer_hashes(*po.concat_records(recs[i:i + batch])))
    sh.switch_mode(1)
    nidx = 0
    for s in recs:  # pass 2 (main.cpp:159-187), including the `continue` that skips ++nidx
        if len(s) >= k:
            e = po.enumerate_kmers(s, k)
            if e is None:
                continue
            sh.add_to_kmer(e[0], nidx)
        nidx += 1
    sh.switch_mode(2)
    return nidx


@pytest.mark.gpu
@pytest.mark.parametrize("k,bf_bits", [(17, 1 << 22), (5, 1 << 14), (31, 3 << 20), (11, 1000003), (21, 1 << 33)])
def test_staged_protocol_builds_the_same_index(k, bf_bits):
    """add_at / switch_mode / add_to_kmer / switch_mode == the oracle's class BF == shk_index_build."""
    from oracle import pyoracle as po
    from shark_b200.engine import Shark
    rng = np.random.default_rng(k * 7 + 1)
    recs = _records(rng, 150)
    bases, off = po.concat_records(recs)
    ora = po.Index(bases, off, k, bf_bits)
    with Shark(k=k, bf_bits=bf_bits, max_reads_per_chunk=4096) as sh:
        assert sh.mode() == 0
        nidx = _staged_build(sh, recs, k)
        assert sh.mode() == 2 and nidx == ora.n_genes
        assert (sh.info.n_set_bits, sh.info.tot_ids) == (ora.n_set, ora.tot_ids)
        assert sh.info.n_genes <= ora.n_genes  # class BF only sees the indices that own a k-mer; main.cpp counts nidx
        pos, coff, ids = sh.export_index()
        assert np.array_equal(pos, ora.pos) and np.array_equal(coff, ora.off) and np.array_equal(ids, ora.ids)
        # BF::get_index on the staged index
        kmers = np.concatenate([po.enumerate_kmers(s, k)[0] for s in recs[:20] if len(s) >= k and po.enumerate_kmers(s, k)]
                               + [rng.integers(0, 1 << 62, 500, dtype=np.uint64) & np.uint64((1 << (2 * k)) - 1)])
        r0, b0, l0 = ora.probe(kmers)
        r1, b1, l1 = sh.get_index(kmers)
        assert np.array_equal(r0, r1) and np.array_equal(b0, b1) and np.array_equal(l0, l1)
        # and the sample stage on top of it
        reads = []
        for i in range(400):
            s = recs[int(rng.integers(0, len(recs)))]
            if len(s) < 60:
                s = bytes(rng.choice(np.frombuffer(b"ACGT", np.uint8), 80).tobytes())
            a = int(rng.integers(0, len(s) - 50))
            reads.append(s[a:a + 50].upper())
        seq, roff = po.concat_records(reads)
        cnt0, ar0, ag0 = ora.analyze(seq, roff, 0.6)
        keep, ar, ag, _ = sh.analyze(seq, roff)
        assert np.array_equal(ar, ar0) and np.array_equal(ag, ag0) and np.array_equal(keep, (cnt0 > 0).astype(np.uint8))
    with Shark(k=k, bf_bits=bf_bits, max_reads_per_chunk=64) as one:
        one.build_index(bases, off)
        p2, o2, i2 = one.export_index()
        assert np.array_equal(pos, p2) and np.array_equal(coff, o2) and np.array_equal(ids, i2)
        assert one.mode() == 2


@pytest.mark.gpu
def test_staged_protocol_states_and_limits():
    """Mode rules of class BF (bloomfilter.h:61-63,112-184) and the documented limits."""
    from shark_b200 import capi
    from shark_b200.engine import Shark
    with Shark(k=9, bf_bits=1 << 16, max_reads_per_chunk=64) as sh:
        sh.add_to_kmer(np.array([1, 2, 3], np.uint64), 0)  # `if (_mode != 1) return;`
        with pytest.raises(capi.SharkError) as e:
            sh.switch_mode(2)  # 0 -> 2 does not exist (the reference returns false)
        assert e.value.code == -3
        sh.add_at(np.array([5, 5 + (1 << 16), 70000], np.uint64))  # p % size
        assert sh.switch_mode(1) == 2
        with pytest.raises(capi.SharkError) as e:
            sh.add_at(np.array([9], np.uint64))
        assert e.value.code == -3
        with pytest.raises(capi.SharkError) as e:
            sh.switch_mode(1)
        assert e.value.code == -3
        sh.add_to_kmer(np.array([1], np.uint64), 3)
        with pytest.raises(capi.SharkError) as e:
            sh.add_to_kmer(np.array([1], np.uint64), 2)  # indices must not decrease
        assert e.value.code == -3
        with pytest.raises(capi.SharkError) as e:
            sh.add_to_kmer(np.array([1], np.uint64), 65536)  # 16-bit ids, small_vector.hpp:46
        assert e.value.code == -5
        sh.set_options(k=9, c=0.5, single=True)
        assert sh.switch_mode(2) == 2 and sh.mode() == 2
        with pytest.raises(capi.SharkError) as e:
            sh.switch_mode(2)
        assert e.value.code == -3
        pos, coff, ids = sh.export_index()
        assert list(pos) == [5, 70000 % (1 << 16)]


def _run(exe, args, cwd):
    p = subprocess.run([exe] + args, cwd=str(cwd), stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    return p.returncode, p.stdout, p.stderr


def _hybrid_case(hybrid, tmp_path, ref, s1, s2, flags):
    args = ["-r", ref, "-1", s1, "-o", "o1.fq"] + (["-2", s2, "-p", "o2.fq"] if s2 else []) + list(flags)
    rc, out, err = _run(hybrid, args, tmp_path)
    assert rc == 0, err.decode()
    o1 = open(os.path.join(str(tmp_path), "o1.fq"), "rb").read()
    o2 = open(os.path.join(str(tmp_path), "o2.fq"), "rb").read() if s2 else None
    return out, o1, o2


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(example_cases()["cases"]))
def test_hybrid_example_goldens(tmp_path, hybrid, case):
    """The reference's main.cpp + our functors reproduce the reference's own truth files."""
    info = example_cases()["cases"][case]
    f = stage_example(tmp_path)
    ssv, o1, o2 = _hybrid_case(hybrid, tmp_path, f["ENSG00000277117.fa"], f["sample_1.fq"],
                               f["sample_2.fq"] if info["paired"] else None, info["flags"])
    assert (md5(ssv), md5(o1)) == (info["ssv_md5"], info["o1_md5"])
    if info["paired"]:
        assert md5(o2) == info["o2_md5"]


@pytest.mark.gpu
@pytest.mark.parametrize("scenario,case", [(s, c) for s, cs in sorted(edge_cases().items()) for c in sorted(cs)])
def test_hybrid_edge_goldens(tmp_path, hybrid, scenario, case):
    info = edge_cases()[scenario][case]
    f = stage_edge(tmp_path, scenario)
    ssv, o1, o2 = _hybrid_case(hybrid, tmp_path, f["ref.fa"], f["r1.fq"], f.get("r2.fq") if info["paired"] else None, info["flags"])
    d = os.path.join(GOLDEN, "edge", scenario)
    assert ssv == gz_read(os.path.join(d, case + ".ssv.gz"))
    assert o1 == gz_read(os.path.join(d, case + ".o1.fq.gz"))
    if info["paired"]:
        assert o2 == gz_read(os.path.join(d, case + ".o2.fq.gz"))


@pytest.mark.gpu
def test_hybrid_threads_against_live_reference(tmp_path):
    """-t 4: ReadAnalyzer::operator() is called concurrently (main.cpp:219-223); the set of output
    lines and of kept records equals the reference binary's (Q12: only the order may differ)."""
    if not (os.path.exists(REF_HYBRID) and os.path.exists(REF)):
        pytest.skip("compiled reference binaries did not travel")
    from shark_b200 import synth
    names, bases, rec_off = synth.make_reference(80, seed=5)
    synth.write_fasta(str(tmp_path / "ref.fa"), names, bases, rec_off)
    seq, qual, _ = synth.make_reads(bases, 80, 260000, 75, True, seed=13, varied_qual=True, want_qual=True)
    synth.write_fastq(str(tmp_path / "a_1.fq"), str(tmp_path / "a_2.fq"), seq, qual, 260000, 75, True)

    def records(path):
        b = open(str(tmp_path / path), "rb").read().split(b"\n")
        return sorted(b"\n".join(b[i:i + 4]) for i in range(0, len(b) - 1, 4))

    for flags in (["-k", "17", "-t", "4"], ["-k", "21", "-q", "20", "-s", "-t", "3"]):
        base = ["-r", "ref.fa", "-1", "a_1.fq", "-2", "a_2.fq"]
        rc, out, err = _run(REF_HYBRID, base + ["-o", "h1.fq", "-p", "h2.fq"] + flags, tmp_path)
        assert rc == 0, err.decode()
        rc0, out0, _ = _run(REF, base + ["-o", "r1.fq", "-p", "r2.fq"] + flags, tmp_path)
        assert rc0 == 0 and len(out0) > 1000
        assert sorted(out.split(b"\n")) == sorted(out0.split(b"\n"))
        assert records("h1.fq") == records("r1.fq") and records("h2.fq") == records("r2.fq")
