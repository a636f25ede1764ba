"""A/B of the reads per equivalence class (SHK_F_EQ_CLASSES) on C2 and C4 and on a many-classes workload, in one
process on one GPU.

Variants, each a context of its own over the same index and the same resident reads:
  parent   the default path (no flag) of another build of libshark_b200.so (--parent-lib), e.g. the commit before
           the class table existed: checks that the default path did not move
  off      the default path of this build
  counts   this build with SHK_F_GENE_COUNTS only (K8 without the insert pass)
  eq       this build with SHK_F_EQ_CLASSES (K8 with the insert pass)

For each workload and each resident form - packed (bulk kernel K6b) and text (thread-per-read kernel K6) - the
variants take turns, --reps rounds of one pass over the chunks each, after --warmup passes.  Per pass:
  step_ms     device time of a whole pass with every chunk in flight (what bench.py's value leg times), results read back
  launches    kernel launches of the pass
Times are per 1 Mi fragments.  Results are checked equal between the variants, and the class table of the "eq" variant
against the grouping of its own result lists by read.  The insert pass's own time comes from separate passes under
torch.profiler (CUDA activities): the summed device time of K8 in "eq" minus that in "counts", plus the leftover and
rehash kernels.  The many-classes workload (segments copied into random subsets of 2 ... 6 records, one class per
segment) starts from the table's initial size: its growth and leftover launches are counted per pass.  Then the CLI on
C2's 20 M-read file, alternately without and with --eqclasses: wall time from exec to exit, byte equality of the ssv and
FASTQ outputs, and the class file's associations against the ssv's lines.

Last, bench.py (the default path) alternately from the parent checkout and from this one, with the card read before each run.

    python profiles/scripts/eqclasses_ab.py --parent-root PATH --out profiles/eqclasses_ab.json
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


NEW_CALLS = ("shk_gene_counts", "shk_gene_counts_reset", "shk_eq_classes")


def open_shark(lib_path, wl, n_chunks, W, flags):
    """A context of the given build of the library (a Shark keeps the handle it was created with).  A build from
    before the counts existed lacks their calls: the binding gets placeholders for them."""
    import ctypes
    import types
    from shark_b200 import capi
    from shark_b200.engine import Shark

    class Tolerant(ctypes.CDLL):
        def __getattr__(self, name):
            try:
                return super().__getattr__(name)
            except AttributeError:
                if name not in NEW_CALLS:
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
                 compact=True, **flags)


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


def run_classes(res):
    """{gene tuple: reads} that the result lists of one pass imply (compact form: gene16 + multi)."""
    from shark_b200 import capi
    out = {}
    for r in res:
        g = r["gene16"].astype(np.int64)
        for x, c in zip(*np.unique(g[(g != capi.GENE_NONE) & (g != capi.GENE_MULTI)], return_counts=True)):
            out[(int(x),)] = out.get((int(x),), 0) + int(c)
        m = r["multi"]
        if len(m):
            for grp in np.split(m[:, 1].astype(np.int64), np.flatnonzero(np.diff(m[:, 0].astype(np.int64))) + 1):
                t = tuple(int(x) for x in grp)
                out[t] = out.get(t, 0) + 1
    return out


def table(sh):
    o, ids, cnt = sh.eq_classes()
    return {tuple(int(x) for x in ids[o[i]:o[i + 1]]): int(cnt[i]) for i in range(len(cnt))}


def kernel_profile(sh, n_chunks, passes):
    """-> {kernel name: summed device ms} over `passes` chunk-by-chunk passes, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(passes):
            one_pass(sh, n_chunks)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t:
            out[e.key] = out.get(e.key, 0.0) + t / 1e3
    return out


def same_results(a, b):
    return all(np.array_equal(x["gene16"], y["gene16"]) and np.array_equal(x["multi"], y["multi"]) and
               (x["n_probes"], x["n_hits"]) == (y["n_probes"], y["n_hits"]) for x, y in zip(a, b))


def stats(v):
    v = np.asarray(v, float)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()), "runs": [float(x) for x in v]}


def many_classes_workload(n_rec=3000, n_seg=24000, seed=11):
    """One class per segment: n_seg random 40-base segments, each copied into 2 ... 6 of n_rec records; the reads are the
    segments (a third reverse-complemented) and a quarter of them again, in chunks of 4096."""
    from oracle import pyoracle as po
    rng = np.random.default_rng(seed)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    comp = bytes.maketrans(b"ACGT", b"TGCA")
    parts = [[acgt[rng.integers(0, 4, 30)].tobytes()] for _ in range(n_rec)]
    segs = [acgt[rng.integers(0, 4, 40)].tobytes() for _ in range(n_seg)]
    for x in segs:
        for r in rng.choice(n_rec, int(rng.integers(2, 7)), replace=False):
            parts[r].append(x + acgt[rng.integers(0, 4, 3)].tobytes())
    bases, rec_off = po.concat_records([b"".join(p) for p in parts])
    texts = [x.translate(comp)[::-1] if i % 3 == 0 else x for i, x in enumerate(segs)] + segs[: n_seg // 4]
    chunks = []
    for a in range(0, len(texts), 4096):
        t = texts[a:a + 4096]
        off = np.zeros(len(t) + 1, np.uint32)
        off[1:] = np.cumsum([len(x) for x in t])
        chunks.append((np.frombuffer(b"".join(t), np.uint8).copy(), None, off, len(t)))
    return {"bases": bases, "rec_off": rec_off, "chunks": chunks, "W": 48, "fragments": len(texts)}


def workload_ab(name, args, variants):
    if name == "many":
        wl = dict(k=21, c=0.8, b=1, q=0, single=False, desc="many classes: 24000 segments in 2 ... 6 of 3000 records")
        wd = many_classes_workload()
        n_reads = wd["fragments"]
    else:
        wl = bench.WORKLOADS[name]
        n_reads = args.reads
        wd = bench.make_workload(wl, 0, n_reads, 8)
    n_chunks, W = len(wd["chunks"]), wd["W"]
    sharks = {}
    for tag, (lib, flags) in variants.items():
        sharks[tag] = open_shark(lib, wl, n_chunks, W, flags)
        sharks[tag].build_index(wd["bases"], wd["rec_off"])
    out = {"desc": wl["desc"], "fragments": n_reads, "chunks": n_chunks, "n_genes": sharks["eq"].info.n_genes, "forms": {}}
    mi = n_reads / float(1 << 20)
    from shark_b200 import capi
    for form in ("packed", "text"):
        if name == "many":   # the class table back at its initial size
            sharks["eq"].build_index(wd["bases"], wd["rec_off"])
        for sh in sharks.values():
            for i in range(n_chunks):
                if form == "packed":
                    s_, _, o_, n_ = wd["chunks"][i] if name == "many" else (None, None, None, None)
                    sh.upload_packed(i, *(wd["packed"][i] if name != "many" else (*capi.host_pack(s_), o_, n_)))
                else:
                    sh.upload(i, *wd["chunks"][i])
        eq = sharks["eq"]
        if name == "many":   # from the initial size: the growth and leftover launches of one pass
            f, c, res = one_pass(eq, n_chunks)
            f, c, base = one_pass(sharks["counts"], n_chunks)
            got = table(eq)
            if got != run_classes(res):
                raise SystemExit("%s %s: the class table differs from the result lists" % (name, form))
            out["forms"].setdefault(form, {})["first_pass_from_initial_size"] = {
                "classes": len(got), "multi_gene_classes": sum(1 for t in got if len(t) >= 2),
                "extra_launches_per_chunk": [r["kernel_launches"] - b["kernel_launches"] for r, b in zip(res, base)]}
        for sh in sharks.values():
            for _ in range(args.warmup):
                one_pass(sh, n_chunks)
                step_pass(sh, n_chunks)
        m = {tag: {"step": [], "launches": []} for tag in sharks}
        ref_results = None
        order = list(sharks)
        for rep in range(args.reps):
            for tag in (order if rep % 2 == 0 else order[::-1]):   # alternate, and alternate the order too
                sh = sharks[tag]
                f, c, res = one_pass(sh, n_chunks)
                l0 = sh.lib.shk_kernel_launches(sh.ctx)
                s, d = step_pass(sh, n_chunks)
                m[tag]["step"].append(s / mi)
                m[tag]["launches"].append(sh.lib.shk_kernel_launches(sh.ctx) - l0)
                if ref_results is None:
                    ref_results = res
                elif not same_results(ref_results, res):
                    raise SystemExit("%s %s: results differ between variants" % (name, form))
                if tag == "eq" and rep == 0:   # the table of exactly one pass equals what its result lists imply
                    sh.reset_gene_counts()
                    f, c, res = one_pass(sh, n_chunks)
                    if table(sh) != run_classes(res):
                        raise SystemExit("%s %s: the class table differs from the result lists" % (name, form))
        d0 = eq.d2h_bytes()
        n_classes = len(table(eq))
        readback = eq.d2h_bytes() - d0
        prof = {tag: kernel_profile(sharks[tag], n_chunks, 3) for tag in ("counts", "eq")}
        k8 = {tag: sum(v for k, v in p.items() if "gene_counts_kernel" in k) for tag, p in prof.items()}
        extra = sum(v for k, v in prof["eq"].items() if "eq_leftover_kernel" in k or "eq_rehash_kernel" in k)
        cls = sum(v for k, v in prof["eq"].items() if "analyze_" in k)
        insert = k8["eq"] - k8["counts"] + extra
        out["forms"].setdefault(form, {}).update({
            "kernel": "analyze_bulk_kernel (K6b)" if form == "packed" else "analyze_reads_kernel (K6)",
            "k8_with_insert_ms_per_Mi": k8["eq"] / 3 / mi,
            "k8_without_insert_ms_per_Mi": k8["counts"] / 3 / mi,
            "leftover_and_rehash_ms_per_Mi": extra / 3 / mi,
            "insert_pass_ms_per_Mi": insert / 3 / mi,
            "classification_kernels_ms_per_Mi": cls / 3 / mi,
            "insert_share_of_classification": insert / cls if cls else None,
            "classes_after_all_passes": n_classes,
            "table_readback_bytes": readback,
            "variants": {tag: {"step_ms_per_Mi": stats(v["step"]), "launches_per_step": int(np.median(v["launches"]))}
                         for tag, v in m.items()},
        })
        log("[eqclasses_ab] %s %s: step %s, insert %.4f ms/Mi (%.2f %% of the classification kernels)" % (
            name, form, {t: round(float(np.median(v["step"])), 3) for t, v in m.items()}, insert / 3 / mi,
            100.0 * insert / cls if cls else float("nan")))
    for sh in sharks.values():
        sh.close()
    return out, wd


def cli_ab(wd, args):
    """C2's reads repeated under fresh names to args.cli_reads, the CLI without and with --eqclasses, alternating."""
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
                o1, ssv, sc = (os.path.join(tmp, "%s.%s" % (tag, x)) for x in ("o1.fq", "ssv", "eq"))
                cmd = [bench.CLI_BIN, "-r", fa, "-1", f1, "-o", o1] + flags + (["--eqclasses", sc] if tag == "on" else [])
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
        lines = open(outs["on"][2], "rb").read().splitlines()
        counted = sum(int(x.split(b" ")[0]) * (len(x.split(b" ")) - 1) for x in lines)
        ssv_lines = sum(1 for _ in open(outs["on"][0], "rb"))
        return {"reads": args.cli_reads, "input": "uncompressed single-end FASTQ in %s" % (base or "the temp directory"),
                "wall_s": {t: stats(v) for t, v in walls.items()}, "ssv_and_fastq_identical": same,
                "classes": len(lines), "class_associations": counted, "ssv_lines": ssv_lines,
                "classes_match_ssv": counted == ssv_lines}


def bench_ab(args):
    """bench.py --gpus 1 --steps 5 --warmup 2 (the default path), alternately from the parent tree and from this one, each
    with the card read right before it: the headline value, and C2's."""
    runs = []
    for rep in range(args.bench_reps):
        for tag, root in (("parent", os.path.abspath(args.parent_root)), ("this", ROOT)):
            c = card()
            p = subprocess.run([sys.executable, "bench.py", "--gpus", "1", "--steps", "5", "--warmup", "2"], cwd=root,
                               capture_output=True, text=True)
            if p.returncode != 0:
                raise SystemExit("bench.py failed in %s: %s" % (root, p.stderr[-500:]))
            d = json.loads(p.stdout.strip().splitlines()[-1])
            runs.append({"tree": tag, "card": c, "value": d["value"], "unit": d["unit"],
                         "c2_value": d.get("workloads", {}).get("c2", {}).get("value")})
            log("[eqclasses_ab] bench %s: %.1f M %s" % (tag, d["value"] / 1e6, d["unit"]))
    return {"command": "bench.py --gpus 1 --steps 5 --warmup 2", "runs": runs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-root", required=True, help="a built checkout of the commit to compare the default path with")
    ap.add_argument("--bench-reps", type=int, default=2, help="alternating bench.py runs per tree (0: none)")
    ap.add_argument("--workloads", default="c2,c4,many")
    ap.add_argument("--reads", type=int, default=4 << 20, help="resident fragments per workload")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--cli-reads", type=int, default=20_000_000)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    this_lib = os.path.join(ROOT, "shark_b200", "libshark_b200.so")
    parent_lib = os.path.join(os.path.abspath(args.parent_root), "shark_b200", "libshark_b200.so")
    variants = {"parent": (parent_lib, {}), "off": (this_lib, {}), "counts": (this_lib, {"gene_counts": True}),
                "eq": (this_lib, {"eq_classes": True})}
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
    if args.bench_reps:
        result["bench"] = bench_ab(args)
    result["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"out": args.out, "card": result["card"]}))


if __name__ == "__main__":
    main()
