"""Per-read score records (SHK_F_SCORES, shk_reads_scores, the CLI's --scores), the parts that need no GPU: the flag
is accepted, the new call checks its arguments, the record layout, the option's argument handling, and the Writer's
scores stream over faked results (tests/host_tools/scores_writer.cpp)."""
import ctypes
import os
import random
import subprocess

import pytest

from helpers import ROOT

HOST = os.path.join(ROOT, "shark_b200", "csrc", "host")
TOOLS = os.path.join(ROOT, "tests", "host_tools")
CLI = os.path.join(ROOT, "shark_b200", "shark-b200")


@pytest.fixture(scope="module")
def lib():
    from shark_b200 import build, capi
    build.build()
    return capi.load()


@pytest.fixture(scope="module")
def tool(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("host") / "scores_writer")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-pthread", "-I", HOST, os.path.join(TOOLS, "scores_writer.cpp"),
                           "-o", out, "-lz"])
    return out


def test_read_score_is_16_bytes():
    from shark_b200 import capi
    assert ctypes.sizeof(capi.ReadScore) == 16
    assert [f[0] for f in capi.ReadScore._fields_] == ["len", "cov", "hits", "n_best"]
    assert capi.F_SCORES == 32


def test_create_accepts_the_flag(lib):
    """Without a device, a context with SHK_F_SCORES fails for the missing device, not for an unknown flag bit."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from shark_b200 import capi
    p = capi.Params(k=17, c=0.6, bf_bits=1 << 20, flags=capi.F_SCORES | capi.F_COMPACT_RESULTS)
    ctx = ctypes.c_void_p()
    assert lib.shk_create(ctypes.byref(p), ctypes.byref(ctx)) == -2
    assert b"unknown flag" not in lib.shk_last_error(None)
    p.flags = 64
    assert lib.shk_create(ctypes.byref(p), ctypes.byref(ctx)) == -1


def test_scores_call_checks_its_arguments(lib):
    from shark_b200 import capi
    sp, n = ctypes.POINTER(capi.ReadScore)(), ctypes.c_uint32()
    assert lib.shk_reads_scores(None, 0, ctypes.byref(sp), ctypes.byref(n)) == -1


def test_cli_scores_needs_a_file(lib, tmp_path):
    r = subprocess.run([CLI, "-r", "x.fa", "-1", "y.fq", "--scores"], cwd=str(tmp_path), capture_output=True)
    assert r.returncode != 0 and r.stdout == b""
    assert b"unknown argument" in r.stderr


# ---- the Writer's scores stream -------------------------------------------------------------------------------
def _write_fastq(path, rng, n, name_run=3):
    with open(path, "w") as f:
        for i in range(n):
            L = rng.randint(18, 40)
            f.write("@r%d%s\n%s\n+\n%s\n" % (i // name_run, " x" if i % 11 == 0 else "", "".join(rng.choice("ACGTN") for _ in range(L)),
                                           "".join(chr(rng.randint(33, 74)) for _ in range(L))))


def _expected_scores(path):
    """scores_writer's faked results: read i is dropped when i % 7 == 3, has 2 associations when i % 5 == 1, else 1; its
    record is {i % 1000 + 1, i % 997, i * 2654435761 mod 2^32, associations}.  One line per kept read, named by the
    ssv's first field (the name up to the first blank)."""
    from oracle import shark_text as st
    pairs, _ = st.load_sample(path, None)
    out = []
    for i, (a, _) in enumerate(pairs):
        if i % 7 == 3:
            continue
        n = 2 if i % 5 == 1 else 1
        out.append(b"%s %d %d %d %d\n" % (st._cstr(a[0]), i % 1000 + 1, i % 997, (i * 2654435761) & 0xFFFFFFFF, n))
    return b"".join(out)


def _pipe(tool, tmp_path, f1, chunk, max_bytes, env, scores):
    o1 = str(tmp_path / "o1.fq")
    sc = str(tmp_path / "o.scores")
    for p in (o1, sc):
        if os.path.exists(p):
            os.unlink(p)
    cmd = [tool, f1, "--chunk", str(chunk), "--bytes", str(max_bytes)] + (["--scores", sc] if scores else [])
    r = subprocess.run(cmd, capture_output=True, timeout=300, env=dict(os.environ, OUT1=o1, **env))
    assert r.returncode == 0, r.stderr.decode()[-500:]
    return r.stdout, open(o1, "rb").read(), (open(sc, "rb").read() if scores else None)


def test_writer_scores_stream(tool, tmp_path):
    """120 000 reads through chunk sizes that do and do not divide the 50 000-read batch, a byte bound, one and
    several threads, mapped and written outputs: the scores lines are those of the kept reads, in order, the same
    bytes either way, and the ssv and FASTQ bytes do not depend on the stream being on."""
    rng = random.Random(11)
    f1 = str(tmp_path / "a.fq")
    _write_fastq(f1, rng, 120000)
    want = _expected_scores(f1)
    assert want.count(b"\n") > 100000
    ssv0, o10, _ = _pipe(tool, tmp_path, f1, 1000000, 10 ** 9, {}, False)
    for chunk, max_bytes, env in ((1000000, 10 ** 9, {}), (30000, 10 ** 9, {"SHK_HOST_THREADS": "4", "SHK_OUT": "map"}),
                                  (50000, 10 ** 9, {"SHK_HOST_THREADS": "1", "SHK_OUT": "write"}),
                                  (17777, 700000, {"SHK_HOST_THREADS": "3", "SHK_OUT": "map", "PREFAULT": "1"}),
                                  (40000, 10 ** 9, {"SHK_NO_BULK": "1", "SHK_OUT": "write"})):
        ssv, o1, sc = _pipe(tool, tmp_path, f1, chunk, max_bytes, env, True)
        assert sc == want, (chunk, env)
        assert ssv == ssv0 and o1 == o10, (chunk, env)
        ssv, o1, _ = _pipe(tool, tmp_path, f1, chunk, max_bytes, env, False)
        assert ssv == ssv0 and o1 == o10, (chunk, env)
