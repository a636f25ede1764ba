"""The shark-b200 command-line drop-in: argument handling (CPU) and byte-identical outputs against
the reference's fixtures / reference-binary goldens (GPU)."""
import os
import subprocess

import pytest

from helpers import GOLDEN, ROOT, edge_cases, example_cases, gz_read, md5, stage_edge, stage_example, stage_synth, synth_cases

CLI = os.path.join(ROOT, "shark_b200", "shark-b200")
REF = os.path.join(ROOT, "oracle", "_ref", "shark")


@pytest.fixture(scope="module", autouse=True)
def _built():
    from shark_b200 import build
    build.build()
    assert os.path.exists(CLI)


def run_cli(args, cwd, exe=CLI):
    p = subprocess.run([exe] + args, cwd=str(cwd), stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    return p.returncode, p.stdout, p.stderr


# ---- argument_parser.hpp:84-174 (no GPU needed: parsing happens before any device call) ----------
@pytest.mark.parametrize("args,msg", [
    (["-r", "x.fa", "-1", "y.fq", "-k", "0"], b"shark: k must be in the range [1, 31]."),
    (["-r", "x.fa", "-1", "y.fq", "-k", "32"], b"shark: k must be in the range [1, 31]."),
    (["-r", "x.fa", "-1", "y.fq", "-c", "1.5"], b"shark: c must be in the range [0, 1]."),
    (["-r", "x.fa", "-1", "y.fq", "-q", "-3"], b"shark: q must be a positive value."),
    (["-r", "x.fa", "-1", "y.fq", "-t", "0"], b"USAGE_MESSAGEshark: at least 1 thread is required."),
    (["-r", "x.fa"], b"shark : missing required files"),
    (["-1", "y.fq"], b"shark : missing required files"),
    (["-r", "x.fa", "-1", "y.fq", "-z"], b"shark : unknown argument"),
])
def test_argument_errors_match_reference(tmp_path, args, msg):
    rc, out, err = run_cli(args, tmp_path)
    assert rc == 1 and out == b"" and msg in err
    if os.path.exists(REF):  # same text and exit code as the reference binary
        rc0, out0, err0 = run_cli(args, tmp_path, exe=REF)
        assert (rc0, out0) == (rc, out)
        assert err0.replace(b"./shark", b"").split(b"invalid option")[0][-200:] == \
            err.replace(b"./shark", b"").split(b"invalid option")[0][-200:] or b"invalid option" in err0


def test_help_matches_reference(tmp_path):
    rc, out, err = run_cli(["-h"], tmp_path)
    assert rc == 0 and out == b"" and err.decode() == synth_cases()["help"]
    if os.path.exists(REF):
        assert run_cli(["-h"], tmp_path, exe=REF) == (rc, out, err)


def test_no_gpu_fails_loudly(tmp_path):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    f = stage_example(tmp_path)
    rc, out, err = run_cli(["-r", f["ENSG00000277117.fa"], "-1", f["sample_1.fq"]], tmp_path)
    assert rc == 1 and out == b"" and b"no CUDA device" in err


# ---- end to end on the GPU -------------------------------------------------------------------------
def _run_case(tmp_path, ref, s1, s2, flags, extra=()):
    args = ["-r", ref, "-1", s1, "-o", "o1.fq"]
    if s2:
        args += ["-2", s2, "-p", "o2.fq"]
    rc, out, err = run_cli(args + list(flags) + list(extra), tmp_path)
    assert rc == 0, err.decode()
    o1 = open(os.path.join(str(tmp_path), "o1.fq"), "rb").read()
    o2 = open(os.path.join(str(tmp_path), "o2.fq"), "rb").read() if s2 else None
    return out, o1, o2


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(example_cases()["cases"]))
def test_cli_example_goldens(tmp_path, case):
    info = example_cases()["cases"][case]
    f = stage_example(tmp_path)
    ssv, o1, o2 = _run_case(tmp_path, f["ENSG00000277117.fa"], f["sample_1.fq"], f["sample_2.fq"] if info["paired"] else None,
                            info["flags"])
    assert ssv.count(b"\n") == info["ssv_lines"]
    assert (md5(ssv), md5(o1)) == (info["ssv_md5"], info["o1_md5"])
    if info["paired"]:
        assert md5(o2) == info["o2_md5"]


@pytest.mark.gpu
@pytest.mark.parametrize("scenario,case", [(s, c) for s, cs in sorted(edge_cases().items()) for c in sorted(cs)])
def test_cli_edge_goldens(tmp_path, scenario, case):
    info = edge_cases()[scenario][case]
    f = stage_edge(tmp_path, scenario)
    ssv, o1, o2 = _run_case(tmp_path, f["ref.fa"], f["r1.fq"], f.get("r2.fq") if info["paired"] else None, info["flags"])
    d = os.path.join(GOLDEN, "edge", scenario)
    assert ssv == gz_read(os.path.join(d, case + ".ssv.gz"))
    assert o1 == gz_read(os.path.join(d, case + ".o1.fq.gz"))
    if info["paired"]:
        assert o2 == gz_read(os.path.join(d, case + ".o2.fq.gz"))


@pytest.mark.gpu
def test_cli_gz_inputs_small_chunks_and_default_outputs(tmp_path):
    """gzip inputs, --chunk-reads 50000 (one batch per chunk -> many chunks through both slots),
    default output names (argument_parser.hpp:168-173)."""
    d = os.path.join(GOLDEN, "example")
    info = example_cases()["cases"]["default"]
    args = ["-r", os.path.join(d, "ENSG00000277117.fa.gz"), "-1", os.path.join(d, "sample_1.fq.gz"),
            "-2", os.path.join(d, "sample_2.fq.gz"), "--chunk-reads", "50000"]
    rc, out, err = run_cli(args, tmp_path)
    assert rc == 0, err.decode()
    assert md5(out) == info["ssv_md5"]
    assert md5(open(os.path.join(str(tmp_path), "sharked_sample.1"), "rb").read()) == info["o1_md5"]
    assert md5(open(os.path.join(str(tmp_path), "sharked_sample.2"), "rb").read()) == info["o2_md5"]
    assert b"[shark/Sample completed] Time elapsed" in err


def _stage_synth_set(tmp_path, s):
    f = stage_synth(tmp_path, s["pairs"], s["read_len"], s["seed"])
    assert {k: md5(open(p, "rb").read()) for k, p in f.items()} == s["inputs_md5"], "shark_b200.synth generates other inputs"
    return f


def test_synth_inputs_are_the_ones_of_the_goldens(tmp_path):
    """tests/golden/synth holds what the reference printed for generated inputs: they must still be generated the same."""
    for s in ("pairs", "bgzf"):
        _stage_synth_set(tmp_path, synth_cases()[s])


@pytest.mark.gpu
def test_cli_against_live_reference_binary(tmp_path):
    """A fresh random input through the CLI: byte for byte what the reference binary printed and wrote for it
    (digests in tests/golden/synth), and what the binary itself does when oracle/_ref/shark is built."""
    s = synth_cases()["pairs"]
    _stage_synth_set(tmp_path, s)
    for info in s["cases"].values():
        flags = info["flags"]
        base = ["-r", "ref.fa", "-1", "a_1.fq", "-2", "a_2.fq"]
        rc, out, err = run_cli(base + ["-o", "m1.fq", "-p", "m2.fq"] + flags, tmp_path)
        assert rc == info["rc"] == 0, err.decode()
        assert out.count(b"\n") == info["ssv_lines"] and len(out) > 1000
        assert md5(out) == info["ssv_md5"]
        assert md5(open(str(tmp_path / "m1.fq"), "rb").read()) == info["o1_md5"]
        assert md5(open(str(tmp_path / "m2.fq"), "rb").read()) == info["o2_md5"]
        if not os.path.exists(REF):
            continue
        rc0, out0, err0 = run_cli(base + ["-o", "r1.fq", "-p", "r2.fq"] + flags, tmp_path, exe=REF)
        assert rc0 == 0
        assert out == out0
        for a, b in (("m1.fq", "r1.fq"), ("m2.fq", "r2.fq")):
            assert open(str(tmp_path / a), "rb").read() == open(str(tmp_path / b), "rb").read()


@pytest.mark.gpu
def test_cli_blocked_gzip_inputs_parallel_inflate(tmp_path):
    """Samples compressed as BGZF (bgzip): the CLI inflates the blocks in parallel (`-t 4` = four inflate threads per
    file + read-ahead, csrc/host/bgzf.hpp) and must print what it prints for the plain files - and what the reference
    prints when it reads the very same .gz files through gzread (digests in tests/golden/synth)."""
    import random
    from test_host_ingest import _bgzf
    s = synth_cases()["bgzf"]
    _stage_synth_set(tmp_path, s)
    rng = random.Random(3)
    for m in ("1", "2"):
        data = open(str(tmp_path / ("a_%s.fq" % m)), "rb").read()
        open(str(tmp_path / ("a_%s.fq.gz" % m)), "wb").write(b"".join(_bgzf(data, rng)))
    info = s["cases"]["k21_q20"]
    flags = info["flags"]
    rc, out, err = run_cli(["-r", "ref.fa", "-1", "a_1.fq", "-2", "a_2.fq", "-o", "p1.fq", "-p", "p2.fq"] + flags, tmp_path)
    assert rc == 0, err.decode()
    rc, outz, err = run_cli(["-r", "ref.fa", "-1", "a_1.fq.gz", "-2", "a_2.fq.gz", "-o", "z1.fq", "-p", "z2.fq", "-t", "4",
                             "--chunk-reads", "50000"] + flags, tmp_path)
    assert rc == 0, err.decode()
    assert outz == out and len(out) > 100000
    for a, b in (("z1.fq", "p1.fq"), ("z2.fq", "p2.fq")):
        assert open(str(tmp_path / a), "rb").read() == open(str(tmp_path / b), "rb").read()
    assert (md5(out), out.count(b"\n")) == (info["ssv_md5"], info["ssv_lines"])
    assert md5(open(str(tmp_path / "z1.fq"), "rb").read()) == info["o1_md5"]
    assert md5(open(str(tmp_path / "z2.fq"), "rb").read()) == info["o2_md5"]
    if os.path.exists(REF):
        rc0, out0, _ = run_cli(["-r", "ref.fa", "-1", "a_1.fq.gz", "-2", "a_2.fq.gz", "-o", "r1.fq", "-p", "r2.fq"] + flags,
                               tmp_path, exe=REF)
        assert rc0 == 0 and out0 == out
        assert open(str(tmp_path / "r1.fq"), "rb").read() == open(str(tmp_path / "z1.fq"), "rb").read()
