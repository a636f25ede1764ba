"""A/B of the per-read score records (SHK_F_SCORES) on C2 and C4, in one process on one GPU.

Variants, each a context of its own over the same index and the same resident reads:
  parent   the default path (no flag) of another build of libshark_b200.so (--parent-lib), e.g. the commit before
           the records existed: checks that the default path did not move
  off      the default path of this build
  on       this build with SHK_F_SCORES

For each workload and each resident form - packed (bulk kernel K6b) and text (thread-per-read kernel K6) - the
variants take turns, --reps rounds of one pass over the chunks each, after --warmup passes.  Per pass:
  fast_ms     CUDA events around the classification kernel that every read enters (K6b / K6), chunk by chunk (one
              chunk in flight at a time, so that nothing overlaps it)
  classify_ms the same for all classification kernels of a chunk (+ the warp-per-read kernels, the scan and the scatter)
  step_ms     device time of a whole pass with every chunk in flight (what bench.py's value leg times), results read back
  d2h_bytes   result bytes copied back per pass
Times are per 1 Mi fragments (reads, or pairs for paired workloads).  Results are checked equal between the
variants.  Then the CLI on C2's 20 M-read file, alternately without and with --scores: wall time from exec to exit,
and byte equality of the ssv and FASTQ outputs.

    python profiles/scripts/scores_ab.py --parent-lib PATH --out profiles/scores_ab_<tag>.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

import bench  # noqa: E402  (WORKLOADS, make_workload: the benchmark's own inputs)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def open_shark(lib_path, wl, n_chunks, W, scores):
    """A context of the given build of the library (a Shark keeps the handle it was created with).  A build from
    before the records existed lacks shk_reads_scores: the binding gets a placeholder for it."""
    import ctypes
    import types
    from shark_b200 import capi
    from shark_b200.engine import Shark

    class Tolerant(ctypes.CDLL):
        def __getattr__(self, name):
            try:
                return super().__getattr__(name)
            except AttributeError:
                if name != "shk_reads_scores":
                    raise
                f = types.SimpleNamespace(argtypes=None, restype=None)
                setattr(self, name, f)
                return f

    capi.LIB_PATH, capi._lib = lib_path, None
    plain, capi.C.CDLL = capi.C.CDLL, Tolerant
    try:
        capi.load()
    finally:
        capi.C.CDLL = plain
    return Shark(k=wl["k"], c=wl["c"], bf_bits=wl["b"] << 33, min_quality=wl["q"], single=wl["single"],
                 n_slots=max(n_chunks, 2), max_reads_per_chunk=bench.CHUNK_READS, max_bytes_per_chunk=bench.CHUNK_READS * W,
                 compact=True, scores=scores)


def one_pass(sh, n_chunks):
    """-> (fast_ms, classify_ms, results): chunk by chunk, one in flight at a time."""
    fast = cls = 0.0
    res = []
    for i in range(n_chunks):
        sh.analyze_resident(i)
        r = sh.collect(i)
        fast += r["probe_kernel_ms"]
        cls += r["analyze_ms"]
        res.append(r)
    return fast, cls, res


def step_pass(sh, n_chunks):
    """-> (device ms of a pass with all chunks in flight, D2H bytes)."""
    d0 = sh.d2h_bytes()
    sh.timer_start()
    for i in range(n_chunks):
        sh.analyze_resident(i)
    for i in range(n_chunks):
        sh.collect(i, copy=False)
    return sh.timer_stop(), sh.d2h_bytes() - d0


def same_results(a, b):
    return all(np.array_equal(x["gene16"], y["gene16"]) and np.array_equal(x["multi"], y["multi"]) and
               (x["n_probes"], x["n_hits"]) == (y["n_probes"], y["n_hits"]) for x, y in zip(a, b))


def stats(v):
    v = np.asarray(v, float)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()), "runs": [float(x) for x in v]}


def workload_ab(name, args, variants):
    wl = bench.WORKLOADS[name]
    n_reads = args.reads
    wd = bench.make_workload(wl, 0, n_reads, 8)
    n_chunks, W = len(wd["chunks"]), wd["W"]
    sharks = {}
    for tag, (lib, flag) in variants.items():
        sharks[tag] = open_shark(lib, wl, n_chunks, W, flag)
        sharks[tag].build_index(wd["bases"], wd["rec_off"])
    out = {"desc": wl["desc"], "fragments": n_reads, "chunks": n_chunks, "forms": {}}
    mi = n_reads / float(1 << 20)
    for form in ("packed", "text"):
        for sh in sharks.values():
            for i in range(n_chunks):
                if form == "packed":
                    sh.upload_packed(i, *wd["packed"][i])
                else:
                    sh.upload(i, *wd["chunks"][i])
        for sh in sharks.values():
            for _ in range(args.warmup):
                one_pass(sh, n_chunks)
                step_pass(sh, n_chunks)
        m = {tag: {"fast": [], "classify": [], "step": [], "d2h": []} for tag in sharks}
        ref_results = None
        order = list(sharks)
        for rep in range(args.reps):
            for tag in (order if rep % 2 == 0 else order[::-1]):   # alternate, and alternate the order too
                sh = sharks[tag]
                f, c, res = one_pass(sh, n_chunks)
                s, d = step_pass(sh, n_chunks)
                m[tag]["fast"].append(f / mi)
                m[tag]["classify"].append(c / mi)
                m[tag]["step"].append(s / mi)
                m[tag]["d2h"].append(d)
                if ref_results is None:
                    ref_results = res
                elif not same_results(ref_results, res):
                    raise SystemExit("%s %s: results differ between variants" % (name, form))
                if tag == "on":
                    assert all(r["scores"].shape == (r["n_reads"], 4) for r in res)
        out["forms"][form] = {
            "kernel": "analyze_bulk_kernel (K6b)" if form == "packed" else "analyze_reads_kernel (K6)",
            "variants": {tag: {"fast_kernel_ms_per_Mi": stats(v["fast"]), "classify_ms_per_Mi": stats(v["classify"]),
                               "step_ms_per_Mi": stats(v["step"]), "d2h_bytes_per_step": int(np.median(v["d2h"]))}
                         for tag, v in m.items()},
        }
        log("[scores_ab] %s %s: %s" % (name, form, {t: round(float(np.median(v["fast"])), 3) for t, v in m.items()}))
    for sh in sharks.values():
        sh.close()
    return out, wd


def cli_ab(wd, args):
    """C2's reads repeated under fresh names to args.cli_reads, the CLI without and with --scores, alternating."""
    from shark_b200 import synth
    wl = bench.WORKLOADS["c2"]
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    with tempfile.TemporaryDirectory(dir=base) as tmp:
        fa, f1 = os.path.join(tmp, "ref.fa"), os.path.join(tmp, "s_1.fq")
        synth.write_fasta(fa, wd["names"], wd["bases"], wd["rec_off"])
        done = 0
        while done < args.cli_reads:
            for s, q, _, n in wd["chunks"]:
                m = min(n, args.cli_reads - done)
                if m <= 0:
                    break
                synth.write_fastq_fast(f1, None, s, q, m, wl["L"], False, first_name=done, append=done > 0)
                done += m
        flags = ["-k", str(wl["k"]), "-c", str(wl["c"]), "-b", str(wl["b"])]
        walls = {"off": [], "on": []}
        outs = {}
        for rep in range(args.reps + 1):
            for tag in (("off", "on") if rep % 2 == 0 else ("on", "off")):
                time.sleep(1.5)   # the device process of the previous run finishes its tear-down on its own
                o1, ssv, sc = (os.path.join(tmp, "%s.%s" % (tag, x)) for x in ("o1.fq", "ssv", "scores"))
                cmd = [bench.CLI_BIN, "-r", fa, "-1", f1, "-o", o1] + flags + (["--scores", sc] if tag == "on" else [])
                t0 = time.perf_counter()
                with open(ssv, "wb") as fo:
                    p = subprocess.run(cmd, stdout=fo, stderr=subprocess.PIPE)
                secs = time.perf_counter() - t0
                if p.returncode != 0:
                    raise SystemExit("CLI failed: " + p.stderr.decode()[-500:])
                if rep:   # the first round warms the page cache and the driver
                    walls[tag].append(secs)
                outs[tag] = (ssv, o1, sc)
        same = all(open(outs["off"][i], "rb").read() == open(outs["on"][i], "rb").read() for i in (0, 1))
        sc_lines = sum(1 for _ in open(outs["on"][2], "rb"))
        kept = sum(1 for _ in open(outs["on"][0], "rb"))
        return {"reads": args.cli_reads, "input": "uncompressed single-end FASTQ in %s" % (base or "the temp directory"),
                "wall_s": {t: stats(v) for t, v in walls.items()}, "ssv_and_fastq_identical": same,
                "scores_lines": sc_lines, "ssv_lines": kept}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True, help="libshark_b200.so of the build to compare the default path with")
    ap.add_argument("--workloads", default="c2,c4")
    ap.add_argument("--reads", type=int, default=4 << 20, help="resident fragments per workload")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cli-reads", type=int, default=20_000_000)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    this_lib = os.path.join(ROOT, "shark_b200", "libshark_b200.so")
    variants = {"parent": (os.path.abspath(args.parent_lib), False), "off": (this_lib, False), "on": (this_lib, True)}
    result = {"card": card(), "torch_device": torch.cuda.get_device_name(0),
              "method": __doc__.split("\n\n")[1] + " " + __doc__.split("\n\n")[2], "workloads": {}}
    c2 = None
    for name in args.workloads.split(","):
        r, wd = workload_ab(name, args, variants)
        result["workloads"][name] = r
        if name == "c2":
            c2 = wd
    if c2 is not None and args.cli_reads:
        result["cli_c2"] = cli_ab(c2, args)
    result["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"out": args.out, "card": result["card"]}))


if __name__ == "__main__":
    main()
