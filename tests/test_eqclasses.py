"""Reads per equivalence class (SHK_F_EQ_CLASSES, shk_eq_classes, the CLI's --eqclasses), the parts that need no GPU:
the flag value and the export, the flag check of shk_create, the new call's argument checks, the option's argument
handling, the help text, and the CLI's merge of per-GPU tables and its file format (tests/host_tools/eqclasses_tool.cpp)
against a restatement in Python."""
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
    out = str(tmp_path_factory.mktemp("host") / "eqclasses_tool")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-Wall", "-I", HOST, os.path.join(TOOLS, "eqclasses_tool.cpp"), "-o", out])
    return out


def test_flag_and_export(lib):
    from shark_b200 import capi
    assert capi.F_EQ_CLASSES == 512
    assert "shk_eq_classes" in capi.EXPORTED
    hdr = open(os.path.join(ROOT, "include", "shark_b200.h")).read()
    assert "#define SHK_F_EQ_CLASSES 512u" in hdr
    assert lib.shk_abi_version() == 5


def test_create_checks_the_flag(lib):
    """SHK_F_EQ_CLASSES without SHK_F_GENE_COUNTS is an argument error that names both flags, found before the device is
    looked for; with both flags a context fails only for the missing device."""
    from shark_b200 import capi
    ctx = ctypes.c_void_p()
    p = capi.Params(k=17, c=0.6, bf_bits=1 << 20, flags=capi.F_EQ_CLASSES)
    for flags in (capi.F_EQ_CLASSES, capi.F_EQ_CLASSES | capi.F_SCORES | capi.F_COMPACT_RESULTS):
        p.flags = flags
        assert lib.shk_create(ctypes.byref(p), ctypes.byref(ctx)) == -1, flags
        err = lib.shk_last_error(None)
        assert b"SHK_F_EQ_CLASSES" in err and b"SHK_F_GENE_COUNTS" in err, err
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    for flags in (capi.F_EQ_CLASSES | capi.F_GENE_COUNTS, capi.F_EQ_CLASSES | capi.F_GENE_COUNTS | capi.F_WIDE_IDS):
        p.flags = flags
        assert lib.shk_create(ctypes.byref(p), ctypes.byref(ctx)) == -2, flags
        assert b"unknown flag" not in lib.shk_last_error(None), flags


def test_eq_classes_checks_the_context(lib):
    n, m = ctypes.c_uint64(), ctypes.c_uint64()
    off, cnt = (ctypes.c_uint64 * 4)(), (ctypes.c_uint64 * 4)()
    ids = (ctypes.c_uint32 * 4)()
    assert lib.shk_eq_classes(None, ctypes.byref(n), ctypes.byref(m), None, None, None, 0, 0) == -1
    assert lib.shk_eq_classes(None, ctypes.byref(n), ctypes.byref(m), off, ids, cnt, 3, 4) == -1
    assert lib.shk_eq_classes(None, None, None, None, None, None, 0, 0) == -1


def test_cli_eqclasses_needs_a_file(lib, tmp_path):
    r = subprocess.run([CLI, "-r", "x.fa", "-1", "y.fq", "--eqclasses"], cwd=str(tmp_path), capture_output=True)
    assert r.returncode != 0 and r.stdout == b""
    assert b"unknown argument" in r.stderr


def test_help_text_unchanged(lib, tmp_path):
    """--eqclasses, like the other extensions, stays out of the reference's usage text."""
    from helpers import synth_cases
    r = subprocess.run([CLI, "-h"], cwd=str(tmp_path), capture_output=True)
    assert r.returncode == 0 and r.stdout == b""
    assert r.stderr.decode() == synth_cases()["help"]
    assert b"eqclasses" not in r.stderr


def _merge_and_format(tables, names):
    """What the CLI writes: equal lists summed over the tables, classes with count 0 left out, lexicographic order of the
    lists, `<count> <name_1> ... <name_n>` with the ssv's name of each index (empty past the legend)."""
    total = {}
    for t in tables:
        for ids, count in t:
            total[tuple(ids)] = total.get(tuple(ids), 0) + count
    lines = []
    for ids in sorted(total):
        if total[ids]:
            lines.append(" ".join([str(total[ids])] + [names[g] if g < len(names) else "" for g in ids]) + "\n")
    return "".join(lines)


def _tool_input(tables, names):
    out = ["%d" % len(names)] + list(names) + ["%d" % len(tables)]
    for t in tables:
        out.append("%d" % len(t))
        out += ["%d %d %s" % (c, len(ids), " ".join(map(str, ids))) for ids, c in t]
    return "\n".join(out) + "\n"


def _random_table(rng, n_genes, n_classes):
    classes = set()
    while len(classes) < n_classes:
        k = rng.choice([1, 1, 2, 2, 3, 5, 33])
        classes.add(tuple(sorted(rng.sample(range(n_genes), min(k, n_genes)))))
    return [(list(c), rng.choice([0, 1, 1, 2, 7, 1 << 40])) for c in sorted(classes)]


@pytest.mark.parametrize("seed", range(6))
def test_merge_and_format(tool, seed):
    rng = random.Random(seed)
    n_genes = rng.choice([3, 40, 300, 70000])
    names = ["g%d_%s" % (i, "x" * (i % 3)) for i in range(min(n_genes, 200))]
    if seed == 1:
        names[1] = ""  # an empty name stays an empty field
    tables = [_random_table(rng, n_genes, rng.choice([0, 1, 50, 400])) for _ in range(rng.choice([1, 2, 3, 8]))]
    if seed == 2:  # the same lists on every GPU
        tables = [tables[0]] * 4
    r = subprocess.run([tool], input=_tool_input(tables, names).encode(), capture_output=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout.decode() == _merge_and_format(tables, names)


def test_merge_orders_prefixes_first(tool):
    """A list sorts before every longer list it is a prefix of, as Python's tuples do: (1,) < (1, 2) < (1, 2, 3) < (2,)."""
    tables = [[([1, 2, 3], 1), ([2], 4)], [([1], 2), ([1, 2], 3), ([2], 1)]]
    r = subprocess.run([tool], input=_tool_input(tables, ["a", "b", "c", "d"]).encode(), capture_output=True)
    assert r.stdout.decode() == "2 b\n3 b c\n1 b c d\n5 c\n"
