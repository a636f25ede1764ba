"""Shared test helpers: golden-fixture access and small synthetic inputs."""
import gzip
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def md5(b):
    return hashlib.md5(b).hexdigest()


def gunzip_to(src_gz, dst):
    with gzip.open(src_gz, "rb") as f, open(dst, "wb") as g:
        g.write(f.read())
    return dst


def gz_read(path):
    with gzip.open(path, "rb") as f:
        return f.read()


def example_cases():
    return json.load(open(os.path.join(GOLDEN, "example", "cases.json")))


def edge_cases():
    return json.load(open(os.path.join(GOLDEN, "edge", "cases.json")))


def synth_cases():
    return json.load(open(os.path.join(GOLDEN, "synth", "cases.json")))


def stage_synth(tmpdir, n_pairs, read_len, seed):
    """ref.fa (60 generated genes) and a_1.fq / a_2.fq (n_pairs generated read pairs with varied qualities) in tmpdir;
    the same bytes on every machine, so that what the reference printed for them can be stored as digests."""
    from shark_b200 import synth
    names, bases, rec_off = synth.make_reference(60, seed=7)
    synth.write_fasta(os.path.join(str(tmpdir), "ref.fa"), names, bases, rec_off)
    seq, qual, _ = synth.make_reads(bases, 60, n_pairs, read_len, True, seed=seed, varied_qual=True, want_qual=True)
    synth.write_fastq(os.path.join(str(tmpdir), "a_1.fq"), os.path.join(str(tmpdir), "a_2.fq"), seq, qual, n_pairs,
                      read_len, True)
    return {f: os.path.join(str(tmpdir), f) for f in ("ref.fa", "a_1.fq", "a_2.fq")}


def flags_to_kwargs(flags):
    """['-k','31','-s'] -> dict(k=31, single=True, ...) (argument_parser.hpp:84-174 defaults)."""
    kw = dict(k=17, c=0.6, b=1, q=0, single=False)
    it = iter(flags)
    for f in it:
        if f == "-k":
            kw["k"] = int(next(it))
        elif f == "-c":
            kw["c"] = float(next(it))
        elif f == "-b":
            kw["b"] = int(next(it))
        elif f == "-q":
            kw["q"] = int(next(it)) & 0xFF
        elif f == "-s":
            kw["single"] = True
        else:
            raise ValueError(f)
    return kw


def stage_example(tmpdir):
    d = os.path.join(GOLDEN, "example")
    out = {}
    for f in ("ENSG00000277117.fa", "sample_1.fq", "sample_2.fq"):
        out[f] = gunzip_to(os.path.join(d, f + ".gz"), os.path.join(str(tmpdir), f))
    return out


def stage_edge(tmpdir, scenario):
    d = os.path.join(GOLDEN, "edge", scenario)
    out = {}
    for f in ("ref.fa", "r1.fq", "r2.fq"):
        if os.path.exists(os.path.join(d, f + ".gz")):
            out[f] = gunzip_to(os.path.join(d, f + ".gz"), os.path.join(str(tmpdir), f))
    return out


ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
