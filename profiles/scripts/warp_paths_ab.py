"""A/B of the warp-per-read kernels K6m (analyze_mid_kernel) and K6x (analyze_slow_kernel), in one process on one GPU.

bench.py does not time these kernels: its reads almost never leave the fast kernels.  Here every chunk is made of reads
that the fast kernels hand on, over a reference with segments copied into exactly m records:
  mid     150-base reads inside segments shared by 5, 16, 32, 64 or 90 records (K6m settles them: at most kMidMaxGenes
          genes), and one read in four 1500 bases long, three 500-base pieces of three records (longer than 1024 bytes)
  exact   150-base reads inside segments shared by 130 records (K6m hands them on, K6x settles them)
  wide    SHK_F_WIDE_IDS: 150-base reads of single records; every read goes through K6m
Each chunk is resident in HBM (text), once in each of --passes slots.  Variants are contexts of two builds of
libshark_b200.so over the same index: `parent` (--parent-lib) and `this` (--this-lib, default the build in the tree).
After --warmup passes, --reps rounds alternate the variants (and their order); per round and variant the device
stopwatch (shk_device_timer_*, all slot streams) covers one shk_reads_analyze_resident per slot, i.e. the classification
kernels of --passes chunks, and the results are collected after the window.  A pass also runs the fast kernel that hands
the reads on and the scan and scatter; their code is the same in both builds.  Results (gene16, multi, n_probes, n_hits,
n_slow_reads) must be equal between the variants.

    python profiles/scripts/warp_paths_ab.py --parent-lib PATH --out DIR/warp_paths_ab.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

K, C, BF_BITS = 31, 0.6, 1 << 33
ACGT = np.frombuffer(b"ACGT", np.uint8)
COMP = np.zeros(256, np.uint8)
COMP[list(b"ACGT")] = list(b"TGCA")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def make_reference(rng, n_rec=200, priv=3000, seg_len=1000, mults=(5, 16, 32, 64, 90, 130), per_mult=4):
    """Records = a private block each, then copies of the segments assigned to them.  -> bases, rec_off, private block
    offsets, {m: [segment arrays]}"""
    parts = [[rng.integers(0, 4, priv, dtype=np.uint8)] for _ in range(n_rec)]
    segs = {}
    for m in mults:
        segs[m] = []
        for _ in range(per_mult):
            s = rng.integers(0, 4, seg_len, dtype=np.uint8)
            segs[m].append(ACGT[s])
            for r in rng.choice(n_rec, m, replace=False):
                parts[r].append(s)
    recs = [ACGT[np.concatenate(p)] for p in parts]
    rec_off = np.zeros(n_rec + 1, np.uint64)
    rec_off[1:] = np.cumsum([len(r) for r in recs])
    return np.concatenate(recs), rec_off, segs


def strand(rng, s):
    return COMP[s[::-1]] if rng.integers(2) else s


def chunk(reads):
    off = np.zeros(len(reads) + 1, np.uint32)
    off[1:] = np.cumsum([len(r) for r in reads])
    return np.concatenate(reads), off


def make_chunks(rng, bases, rec_off, segs, n_mid, n_exact, n_wide):
    def piece(m, L):
        s = segs[m][rng.integers(len(segs[m]))]
        o = rng.integers(0, len(s) - L + 1)
        return strand(rng, s[o:o + L])

    def private(L):
        r = rng.integers(len(rec_off) - 1)
        o = int(rec_off[r]) + int(rng.integers(0, 3000 - L + 1))
        return bases[o:o + L]

    mid = []
    for i in range(n_mid):
        if i % 4 == 3:
            mid.append(strand(rng, np.concatenate([private(500) for _ in range(3)])))
        else:
            mid.append(piece((5, 16, 32, 64, 90)[rng.integers(5)], 150))
    exact = [piece(130, 150) for _ in range(n_exact)]
    wide = [strand(rng, private(150)) for _ in range(n_wide)]
    return {"mid": chunk(mid), "exact": chunk(exact), "wide": chunk(wide)}


def open_shark(lib_path, wide, n_slots, max_reads, max_bytes):
    from shark_b200 import capi
    from shark_b200.engine import Shark
    capi.LIB_PATH, capi._lib = lib_path, None
    capi.load()
    return Shark(k=K, c=C, bf_bits=BF_BITS, n_slots=n_slots, max_reads_per_chunk=max_reads, max_bytes_per_chunk=max_bytes,
                 compact=True, wide_ids=wide)


def timed_passes(sh, n_slots):
    """-> (device ms of the kernels of one chunk per slot, the results), collected after the timed window."""
    sh.timer_start()
    for s in range(n_slots):
        sh.analyze_resident(s)
    ms = sh.timer_stop()
    return ms, [sh.collect(s) for s in range(n_slots)]


def same(x, y):
    return (np.array_equal(x["gene16"], y["gene16"]) and np.array_equal(x["multi"], y["multi"]) and
            (x["n_probes"], x["n_hits"], x["n_slow_reads"]) == (y["n_probes"], y["n_hits"], y["n_slow_reads"]))


def stats(v):
    v = np.asarray(v, float)
    return {"median": float(np.median(v)), "min": float(v.min()), "max": float(v.max()),
            "spread_pct": float(100.0 * (v.max() - v.min()) / np.median(v)), "runs": [float(x) for x in v]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True, help="libshark_b200.so of the build to compare with")
    ap.add_argument("--mid-reads", type=int, default=65536)
    ap.add_argument("--exact-reads", type=int, default=16384)
    ap.add_argument("--wide-reads", type=int, default=262144)
    ap.add_argument("--passes", type=int, default=5, help="chunks (one per slot) per timed window")
    ap.add_argument("--this-lib", default=os.path.join(ROOT, "shark_b200", "libshark_b200.so"))
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--out", required=True)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    rng = np.random.default_rng(args.seed)
    bases, rec_off, segs = make_reference(rng)
    chunks = make_chunks(rng, bases, rec_off, segs, args.mid_reads, args.exact_reads, args.wide_reads)
    max_reads = max(len(off) - 1 for _, off in chunks.values())
    max_bytes = max(len(seq) for seq, _ in chunks.values())
    libs = {"parent": os.path.abspath(args.parent_lib), "this": os.path.abspath(args.this_lib)}
    result = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "method": __doc__.split("\n\n")[1],
              "k": K, "c": C, "bf_bits": BF_BITS, "chunks": {}}
    for name, (seq, off) in chunks.items():
        n = len(off) - 1
        sharks = {tag: open_shark(lib, name == "wide", args.passes, max_reads, max_bytes) for tag, lib in libs.items()}
        for sh in sharks.values():
            sh.build_index(bases, rec_off)
            for s in range(args.passes):
                sh.upload(s, seq, None, off, n)
        ref = None
        for tag, sh in sharks.items():
            for _ in range(args.warmup):
                _, rs = timed_passes(sh, args.passes)
            ref = ref or rs[0]
            if not all(same(ref, r) for r in rs):
                raise SystemExit("%s: results differ between variants" % name)
        times = {tag: [] for tag in sharks}
        order = list(sharks)
        for rep in range(args.reps):
            for tag in (order if rep % 2 == 0 else order[::-1]):
                ms, rs = timed_passes(sharks[tag], args.passes)
                times[tag].append(ms / args.passes)
                if not all(same(ref, r) for r in rs):
                    raise SystemExit("%s: results differ between variants" % name)
        result["chunks"][name] = {
            "reads": n, "bases": int(off[-1]), "n_slow_reads": int(ref["n_slow_reads"]), "n_kept": int(ref["n_kept"]),
            "n_multi": int(ref["n_multi"]), "n_probes": int(ref["n_probes"]),
            "ms_per_pass": {tag: stats(v) for tag, v in times.items()},
            "this_over_parent": float(np.median(times["this"]) / np.median(times["parent"]))}
        print("[warp_paths_ab] %s: %d reads, %d handed on; ms per pass: parent %.3f, this %.3f" % (
            name, n, ref["n_slow_reads"], np.median(times["parent"]), np.median(times["this"])), file=sys.stderr)
        for sh in sharks.values():
            sh.close()
    result["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"out": args.out, "card": result["card"]}))


if __name__ == "__main__":
    main()
