"""Per-gene read counts (SHK_F_GENE_COUNTS, shk_gene_counts, the CLI's --counts), the parts that need no GPU: the flag
value and the exported symbols, the new calls' argument checks, the option's argument handling, and the help text."""
import ctypes
import os
import subprocess

import pytest

from helpers import ROOT

CLI = os.path.join(ROOT, "shark_b200", "shark-b200")


@pytest.fixture(scope="module")
def lib():
    from shark_b200 import build, capi
    build.build()
    return capi.load()


def test_flag_and_exports(lib):
    from shark_b200 import capi
    assert capi.F_GENE_COUNTS == 128
    assert {"shk_gene_counts", "shk_gene_counts_reset"} <= set(capi.EXPORTED)
    hdr = open(os.path.join(ROOT, "include", "shark_b200.h")).read()
    assert "#define SHK_F_GENE_COUNTS 128u" in hdr
    assert lib.shk_abi_version() == 5


def test_create_accepts_the_flag(lib):
    """Without a device, a context with SHK_F_GENE_COUNTS or SHK_F_SCORES fails for the missing device, not for an unknown
    flag bit; the unassigned bits (64, 256 and up) are still an argument error."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from shark_b200 import capi
    ctx = ctypes.c_void_p()
    for flags in (capi.F_GENE_COUNTS, capi.F_SCORES | capi.F_COMPACT_RESULTS, capi.F_GENE_COUNTS | capi.F_SCORES | capi.F_WIDE_IDS):
        p = capi.Params(k=17, c=0.6, bf_bits=1 << 20, flags=flags)
        assert lib.shk_create(ctypes.byref(p), ctypes.byref(ctx)) == -2, flags
        assert b"unknown flag" not in lib.shk_last_error(None), flags
    for flags in (64, 256, capi.F_GENE_COUNTS | 64, 1 << 31):
        p.flags = flags
        assert lib.shk_create(ctypes.byref(p), ctypes.byref(ctx)) == -1, flags
        assert b"unknown flag" in lib.shk_last_error(None), flags


def test_counts_calls_check_the_context(lib):
    u = (ctypes.c_uint64 * 4)()
    assert lib.shk_gene_counts(None, u, u, 4) == -1
    assert lib.shk_gene_counts(None, None, None, 0) == -1
    assert lib.shk_gene_counts_reset(None) == -1


def test_cli_counts_needs_a_file(lib, tmp_path):
    r = subprocess.run([CLI, "-r", "x.fa", "-1", "y.fq", "--counts"], cwd=str(tmp_path), capture_output=True)
    assert r.returncode != 0 and r.stdout == b""
    assert b"unknown argument" in r.stderr


def test_help_text_unchanged(lib, tmp_path):
    """--counts, like the other extensions, stays out of the reference's usage text."""
    from helpers import synth_cases
    r = subprocess.run([CLI, "-h"], cwd=str(tmp_path), capture_output=True)
    assert r.returncode == 0 and r.stdout == b""
    assert r.stderr.decode() == synth_cases()["help"]
    assert b"counts" not in r.stderr
