#!/usr/bin/env python
"""Regenerates tests/golden/ by running the UNMODIFIED reference binary (oracle/_ref/shark,
built by oracle/Makefile from /root/reference) on

  example/   the reference's own fixture (example/ENSG00000277117.fa, sample_{1,2}.fq; inputs
             stored gzipped, the three truth files stored as md5 + gz) under the flag
             variants of SURVEY.md App. B.2, and
  edge/      small generated inputs, one scenario per quirk of SURVEY.md App. C, and
  synth/     the larger generated inputs of tests/test_cli.py, kept as digests of the outputs.

Run here (needs /root/reference); the outputs are committed so the GPU box needs neither.
    python tests/golden/make_golden.py
"""
import gzip
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "shark")
EX = "/root/reference/example"


def md5(b):
    return hashlib.md5(b).hexdigest()


def run_ref(ref, s1, s2, flags, cwd):
    cmd = [REF_BIN, "-r", ref, "-1", s1, "-o", "o1.fq"]
    if s2:
        cmd += ["-2", s2, "-p", "o2.fq"]
    cmd += flags
    p = subprocess.run(cmd, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    out = {"rc": p.returncode, "ssv": p.stdout}
    out["o1"] = open(os.path.join(cwd, "o1.fq"), "rb").read() if os.path.exists(os.path.join(cwd, "o1.fq")) else b""
    out["o2"] = open(os.path.join(cwd, "o2.fq"), "rb").read() if s2 and os.path.exists(os.path.join(cwd, "o2.fq")) else None
    for f in ("o1.fq", "o2.fq"):
        if os.path.exists(os.path.join(cwd, f)):
            os.remove(os.path.join(cwd, f))
    return out


def gz_write(path, data):
    with open(path, "wb") as f:
        f.write(gzip.compress(data, 9, mtime=0))


# ---------------------------------------------------------------------------------------
def make_example():
    d = os.path.join(HERE, "example")
    os.makedirs(d, exist_ok=True)
    for f in ("ENSG00000277117.fa", "sample_1.fq", "sample_2.fq", "ENSG00000277117.truth.ssv",
              "sharked.sample_1.truth.fq", "sharked.sample_2.truth.fq"):
        gz_write(os.path.join(d, f + ".gz"), open(os.path.join(EX, f), "rb").read())
    cases = {
        "default": ([], True),
        "single_end": ([], False),
        "k31_c0.9_s": (["-k", "31", "-c", "0.9", "-s"], True),
        "k31_b4": (["-k", "31", "-b", "4"], True),
        "k21_c0.3": (["-k", "21", "-c", "0.3"], True),
        "b3": (["-b", "3"], True),
        "k21_q20_s": (["-k", "21", "-q", "20", "-s"], True),
        "c0": (["-c", "0"], True),
        "c1": (["-c", "1"], True),
        "q41": (["-q", "41"], True),
        "q40": (["-q", "40"], True),
        "k5_c0.9": (["-k", "5", "-c", "0.9"], True),
        "k9": (["-k", "9"], True),
    }
    res = {}
    with tempfile.TemporaryDirectory() as tmp:
        for name, (flags, paired) in cases.items():
            o = run_ref(EX + "/ENSG00000277117.fa", EX + "/sample_1.fq", EX + "/sample_2.fq" if paired else None, flags, tmp)
            res[name] = {"flags": flags, "paired": paired, "rc": o["rc"], "ssv_lines": o["ssv"].count(b"\n"),
                         "ssv_md5": md5(o["ssv"]), "o1_md5": md5(o["o1"]), "o2_md5": md5(o["o2"]) if paired else None}
            print("example", name, res[name]["ssv_lines"], file=sys.stderr)
    truth = {f: md5(open(os.path.join(EX, f), "rb").read()) for f in
             ("ENSG00000277117.truth.ssv", "sharked.sample_1.truth.fq", "sharked.sample_2.truth.fq")}
    assert res["default"]["ssv_md5"] == truth["ENSG00000277117.truth.ssv"]
    assert res["default"]["o1_md5"] == truth["sharked.sample_1.truth.fq"]
    assert res["default"]["o2_md5"] == truth["sharked.sample_2.truth.fq"]
    json.dump({"truth_md5": truth, "cases": res}, open(os.path.join(d, "cases.json"), "w"), indent=1, sort_keys=True)


# ---------------------------------------------------------------------------------------
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
COMP = {65: 84, 67: 71, 71: 67, 84: 65, 78: 78}


def rnd_seq(rng, n):
    return ACGT[rng.integers(0, 4, n)].tobytes()


def revcomp(s):
    return bytes(COMP.get(c, c) for c in reversed(s))


def fasta(recs, width=60, crlf=False):
    nl = b"\r\n" if crlf else b"\n"
    out = []
    for name, seq in recs:
        out.append(b">" + name + nl)
        for i in range(0, len(seq), width):
            out.append(seq[i:i + width] + nl)
    return b"".join(out)


def fastq(recs, crlf=False):
    nl = b"\r\n" if crlf else b"\n"
    return b"".join(b"@" + n + nl + s + nl + b"+" + nl + q + nl for n, s, q in recs)


def scenario_multi(rng):
    """Multi-gene lists, exact ties, N handling, the nidx desync (Q1), a record shorter than
    k, lower case, name comments, background reads, reads with N, per-base qualities."""
    genes = []
    for i in range(14):
        genes.append([b"g%02d" % i, bytearray(rnd_seq(rng, int(rng.integers(400, 900))))])
    genes[3][1][100:400] = genes[2][1][50:350]          # shared segment -> 2-gene lists
    genes[5][1] = bytearray(genes[4][1])                  # exact duplicate -> perfect ties
    genes[6][1][200:203] = b"NNN"
    genes[6][1][420] = ord("n")
    genes[7] = [b"gS", bytearray(b"N" * 64)]             # len >= k, no valid window: Q1
    genes[8] = [b"gshort", bytearray(b"ACGTACG")]        # shorter than k: consumes an index
    genes[9][1] = bytearray(bytes(genes[9][1]).lower())
    genes[10][1][0:40] = b"A" * 40                        # low-complexity run shared with g11
    genes[11][1][300:340] = b"A" * 40
    genes[12][1] = bytearray(genes[4][1][:300]) + bytearray(rnd_seq(rng, 300))  # partial copy
    recs = [(bytes(n) + (b" some comment" if i % 3 == 0 else b""), bytes(s)) for i, (n, s) in enumerate(genes)]
    r1, r2 = [], []
    L = 100
    for i in range(600):
        u = rng.random()
        if u < 0.85:
            g = int(rng.integers(0, len(genes)))
            s = bytes(genes[g][1]).upper()
            if len(s) < L + 60:
                a, b = rnd_seq(rng, L), rnd_seq(rng, L)
            else:
                st = int(rng.integers(0, len(s) - L - 50))
                a = bytearray(s[st:st + L])
                b = bytearray(revcomp(s[st + 50:st + 50 + L]))
                for m in (a, b):
                    for j in range(L):
                        if rng.random() < 0.02:
                            m[j] = ACGT[rng.integers(0, 4)]
                        if rng.random() < 0.004:
                            m[j] = ord("N")
                if rng.random() < 0.5:
                    a, b = b, a
                a, b = bytes(a), bytes(b)
        else:
            a, b = rnd_seq(rng, L), rnd_seq(rng, L)
        qa = bytes(int(x) for x in np.where(rng.random(L) < 0.03, rng.integers(35, 53, L), rng.integers(60, 74, L)))
        qb = bytes(int(x) for x in np.where(rng.random(L) < 0.03, rng.integers(35, 53, L), rng.integers(60, 74, L)))
        r1.append((b"r%05d" % i + (b" 1:N:0" if i % 2 else b""), a, qa))
        r2.append((b"r%05d" % i + (b"/2" if i % 5 == 0 else b""), b, qb))
    cases = {
        "pe_default": (["-k", "17"], True),
        "se_default": ([], False),
        "pe_k31_c0.9_s": (["-k", "31", "-c", "0.9", "-s"], True),
        "pe_k5_c0.3": (["-k", "5", "-c", "0.3"], True),
        "pe_k7_s": (["-k", "7", "-s"], True),
        "pe_k21_q20": (["-k", "21", "-q", "20"], True),
        "se_k21_q25_s": (["-k", "21", "-q", "25", "-s"], False),
        "pe_c0": (["-c", "0"], True),
        "pe_c1": (["-c", "1"], True),
        "pe_k11_c0.7": (["-k", "11", "-c", "0.7"], True),
        "pe_k1": (["-k", "1", "-c", "1"], True),
        "se_k31_q95": (["-k", "31", "-q", "95"], False),   # `char mq` wraps: FastqSplitter.hpp:75
    }
    return fasta(recs), fastq(r1), fastq(r2), cases


def scenario_io(rng):
    """Parser/IO quirks: CRLF, multi-line FASTQ, duplicate adjacent names (Q6), mate-2 names
    (Q7), unpaired tail (Q8), junk before the first header, blank lines."""
    genes = [(b"ga", rnd_seq(rng, 500)), (b"gb\tdesc", rnd_seq(rng, 500)), (b"gc", rnd_seq(rng, 300))]
    r1, r2 = [], []
    for i in range(60):
        g = genes[i % 3][1]
        st = int(rng.integers(0, len(g) - 130))
        a, b = g[st:st + 80], revcomp(g[st + 40:st + 120])
        name = b"dup" if i in (10, 11, 12, 30, 31) else b"x%03d" % i
        r1.append((name, a, b"I" * 80))
        r2.append((name + b"_m2", b, b"H" * 80))
    fa = b"junk line before header\n" + fasta(genes, width=70, crlf=True)
    # multi-line FASTQ for the first few records, CRLF for file 2, blank line inside a record
    f1 = b"".join(b"@" + n + b"\n" + s[:40] + b"\n" + s[40:] + b"\n+" + n + b"\n" + q[:40] + b"\n" + q[40:] + b"\n"
                  for n, s, q in r1[:5]) + b"\n" + fastq(r1[5:])
    f1 += b"@tail_unpaired\nACGTACGTACGTACGTACGTACGTACGT\n+\nIIIIIIIIIIIIIIIIIIIIIIIIIIII\n"
    f2 = fastq(r2, crlf=True)
    cases = {"pe": (["-k", "17"], True), "se": (["-k", "13", "-c", "0.5"], False), "pe_s": (["-s"], True)}
    return fa, f1, f2, cases


def scenario_trunc(rng):
    """A record whose quality is shorter than its sequence ends the input (kseq -2)."""
    g = rnd_seq(rng, 400)
    recs = [(b"t%02d" % i, g[i * 5:i * 5 + 90], b"I" * 90) for i in range(20)]
    f1 = fastq(recs[:12]) + b"@bad\n" + g[:90] + b"\n+\n" + b"I" * 50 + b"\n" + fastq(recs[12:])
    return fasta([(b"gt", g)]), f1, None, {"se": ([], False)}


def make_edge():
    d = os.path.join(HERE, "edge")
    if os.path.isdir(d):
        shutil.rmtree(d)
    os.makedirs(d)
    rng = np.random.default_rng(20261017)
    index = {}
    for sname, fn in (("multi", scenario_multi), ("io", scenario_io), ("trunc", scenario_trunc)):
        fa, f1, f2, cases = fn(rng)
        sd = os.path.join(d, sname)
        os.makedirs(sd)
        gz_write(os.path.join(sd, "ref.fa.gz"), fa)
        gz_write(os.path.join(sd, "r1.fq.gz"), f1)
        if f2 is not None:
            gz_write(os.path.join(sd, "r2.fq.gz"), f2)
        index[sname] = {}
        with tempfile.TemporaryDirectory() as tmp:
            for p, b in (("ref.fa", fa), ("r1.fq", f1), ("r2.fq", f2)):
                if b is not None:
                    open(os.path.join(tmp, p), "wb").write(b)
            for cname, (flags, paired) in cases.items():
                o = run_ref("ref.fa", "r1.fq", "r2.fq" if paired else None, flags, tmp)
                gz_write(os.path.join(sd, cname + ".ssv.gz"), o["ssv"])
                gz_write(os.path.join(sd, cname + ".o1.fq.gz"), o["o1"])
                if paired:
                    gz_write(os.path.join(sd, cname + ".o2.fq.gz"), o["o2"])
                index[sname][cname] = {"flags": flags, "paired": paired, "rc": o["rc"],
                                       "ssv_lines": o["ssv"].count(b"\n"), "ssv_md5": md5(o["ssv"]),
                                       "o1_md5": md5(o["o1"]), "o2_md5": md5(o["o2"]) if paired else None}
                print("edge", sname, cname, index[sname][cname]["ssv_lines"], file=sys.stderr)
    json.dump(index, open(os.path.join(d, "cases.json"), "w"), indent=1, sort_keys=True)


# ---------------------------------------------------------------------------------------
SYNTH = {   # generated inputs of tests/test_cli.py: pairs, read length, seed of the reads, flag variants
    "pairs": (120000, 75, 11, {"k17": ["-k", "17"], "k21_q20_s": ["-k", "21", "-q", "20", "-s"],
                               "k31_c0.8_b2": ["-k", "31", "-c", "0.8", "-b", "2"]}),
    "bgzf": (150000, 100, 13, {"k21_q20": ["-k", "21", "-q", "20"]}),
}


def make_synth():
    """synth/cases.json: the reference's help text, and digests of what it prints and writes for generated inputs
    (tests/helpers.py stage_synth) too large to store."""
    sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
    from helpers import stage_synth
    d = os.path.join(HERE, "synth")
    os.makedirs(d, exist_ok=True)
    out = {"help": subprocess.run([REF_BIN, "-h"], stdout=subprocess.PIPE, stderr=subprocess.PIPE).stderr.decode()}
    for key, (n, read_len, seed, cases) in SYNTH.items():
        with tempfile.TemporaryDirectory() as tmp:
            files = stage_synth(tmp, n, read_len, seed)
            res = {}
            for name, flags in cases.items():
                o = run_ref("ref.fa", "a_1.fq", "a_2.fq", flags, tmp)
                res[name] = {"flags": flags, "rc": o["rc"], "ssv_lines": o["ssv"].count(b"\n"), "ssv_md5": md5(o["ssv"]),
                             "o1_md5": md5(o["o1"]), "o2_md5": md5(o["o2"])}
                print("synth", key, name, res[name]["ssv_lines"], file=sys.stderr)
            out[key] = {"pairs": n, "read_len": read_len, "seed": seed, "cases": res,
                        "inputs_md5": {f: md5(open(p, "rb").read()) for f, p in files.items()}}
    json.dump(out, open(os.path.join(d, "cases.json"), "w"), indent=1, sort_keys=True)


if __name__ == "__main__":
    assert os.path.exists(REF_BIN), "build the reference first: make -C oracle ref"
    make_example()
    make_edge()
    make_synth()
