#!/usr/bin/env python
"""bench.py - reads/s of Shark's k-mer Bloom-filter hot path on B200 (see DESIGN.md, Measurement).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workloads c4,c3,c2] [--dump-outputs DIR]

A step = one pass of the hot path over this rank's whole batch of synthetic reads.
  N = 1   the default run measures C4 (headline: the largest single-GPU configuration of BASELINE.json - 20 k genes,
          k=31, 4 GiB filter, paired 150 bp), then C3 and C2; every workload has its own record under "workloads"
          (value / e2e / roofline / probe / cpu_baseline with parity on the sample), the top-level keys are C4's.
  N > 1   (torchrun, one process per GPU) the workload is C5: C4's index and flags, the read stream sharded by
          rank (weak scaling: every rank gets its own slice of the same size), index built on rank 0 and
          replicated with an NCCL broadcast AND built again by the sharded P2P OR-merge mode (both must be
          identical); every rank checks its own results against the reference binary on a sample of its shard.
Per workload:
  value   fragments/s (reads for single-end, pairs for paired-end workloads) with the reads already resident in
          HBM when the timed region starts: kernels + result read-back, CUDA events over all slot streams
  e2e     the same through the public API (Shark.analyze_chunks -> shk_reads_submit/collect) from pinned HOST
          buffers of read TEXT, H2D and D2H inside the timed region; split upload (SHK_F_HOST_PACK): part of every
          chunk crosses the link as text while the host cores pack the rest to 3 bits per base (inside the timed
          region; time = max(device stopwatch, host clock)).  e2e_plain (text only) and e2e_packed (host buffers
          that already hold the packed form the CLI's batcher emits, shk_reads_submit_packed) ride along.
  roofline  the dominant kernel (analyze_reads_kernel): 32 B x (k-mer windows probed) / its CUDA-event time,
          against the measured HBM copy rate in MEASURED_PEAKS.json (and the measured random-sector ceiling)
  cpu_baseline  the unmodified reference (oracle/_ref/shark -t <cores>) on a bounded sample of the same reads, on
          this box's host cores, with sorted-ssv equality against our output on the same sample
  cli     (C2 only) the process seam: both command-line programs on the same FASTQ files
--impl reference: the reference's own CPU implementation on the same config (headline workload), one process fed
through named pipes so that every step is one pass of a bounded sample in steady state.
"""
import argparse
import fcntl
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # genes, reads per GPU, read length, paired, k, -b, -q, -s, -c, reads of the CPU sample
    "c2": dict(genes=1000, reads=10_000_000, L=100, paired=False, k=17, b=1, q=0, single=False, c=0.6, cpu_sample=2_000_000,
               desc="C2: SYN(1000 genes x 3 kbp), 10M single-end 100 bp reads, k=17, c=0.6, 1 GiB Bloom filter"),
    "c3": dict(genes=5000, reads=8_000_000, L=150, paired=True, k=21, b=1, q=20, single=True, c=0.6, cpu_sample=500_000,
               desc="C3 (8M-pair slice of 50M): SYN(5000 genes), paired 150 bp, k=21, -q 20, -s, 1 GiB Bloom filter"),
    "c4": dict(genes=20000, reads=8_000_000, L=150, paired=True, k=31, b=4, q=0, single=False, c=0.6, cpu_sample=500_000,
               desc="C4 (8M-pair slice of 100M): SYN(20000 genes ~60 Mbp), paired 150 bp, k=31, 4 GiB Bloom filter"),
    "c5": dict(genes=20000, reads=8_000_000, L=150, paired=True, k=31, b=4, q=0, single=False, c=0.6, cpu_sample=500_000,
               desc="C5 (8M-pair slice per GPU of 200M): C4's reference and flags, paired 150 bp, reads sharded by rank, "
                    "index replicated (NCCL broadcast; also built by the sharded P2P OR-merge mode)"),
}
CHUNK_READS = 1 << 20
DUMP_BYTES = 64_000_000   # --dump-outputs: all files together
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "shark")
CLI_BIN = os.path.join(ROOT, "shark_b200", "shark-b200")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def unit_of(wl):
    return "pairs/s" if wl["paired"] else "reads/s"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_source_hash():
    """Hash of the sources the classification kernels are compiled from: keys profiles/traffic.json, so that a
    dram-bytes figure captured with ncu is only reported for the kernels it was captured from."""
    import hashlib
    h = hashlib.sha1()
    for f in ("shk_reads.cu", "shk_reads.cuh", "shk_bulk.cu", "shk_device.cuh", "shk_internal.h"):
        h.update(open(os.path.join(ROOT, "shark_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:12]


def traffic_for(name):
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(tp)).get(name)
    except Exception:
        return None, "no ncu capture on file"
    if not t:
        return None, "no ncu capture on file for this workload"
    if t.get("kernel_source_hash") != kernel_source_hash():
        return None, "the ncu capture on file is of other kernel sources (%s): not reported" % t.get("kernel_source_hash")
    return t.get("dram_bytes_per_launch"), t.get("source")


def dump_outputs(outdir, prefix, outputs, budget):
    """Writes what one step of the value leg returned, expanded as a caller of the API receives it (Shark.expand: per
    read the gene16 code, 0xFFFF none and 0xFFFE several, and the (read, gene) associations), as three arrays over the
    rank's reads:
      <prefix>_read.npy   float64[m]     indices of the reads written (all reads, or a fixed seeded sample when all of
                                         them would not fit in `budget` bytes)
      <prefix>_gene.npy   float32[m]     gene16 of those reads
      <prefix>_assoc.npy  float64[r, 2]  (read, gene) associations of those reads, by read then gene"""
    from shark_b200.engine import Shark
    gene, assoc, first = [], [], 0
    for g, m in outputs:
        ridx, gidx, _ = Shark.expand({"gene16": g, "multi": m})
        gene.append(g)
        assoc.append(np.stack([ridx.astype(np.int64) + first, gidx.astype(np.int64)], 1))
        first += len(g)
    gene, assoc = np.concatenate(gene), np.concatenate(assoc)
    n = len(gene)
    m = min(n, (budget - 1024) // 24)   # 12 bytes per read written; at least as much is left for the associations
    reads = np.arange(n) if m == n else np.sort(np.random.default_rng(0).choice(n, m, replace=False))
    rows = assoc[np.isin(assoc[:, 0], reads)][: (budget - 1024 - 12 * m) // 16]
    os.makedirs(outdir, exist_ok=True)
    for key, a in (("read", reads.astype(np.float64)), ("gene", gene[reads].astype(np.float32)),
                   ("assoc", rows.astype(np.float64))):
        np.save(os.path.join(outdir, "%s_%s.npy" % (prefix, key)), a)


def probe_kmers(bases, k, n, seed=7):
    """n canonical k-mers for the stand-alone probe kernel (BF::get_index): half are windows of the
    reference (hits), half are random (misses, up to the filter's false-positive rate)."""
    rng = np.random.default_rng(seed)
    code = np.full(256, 4, np.uint8)
    for i, ch in enumerate(b"ACGT"):
        code[ch] = code[ch | 0x20] = i
    c = code[np.asarray(bases[: min(len(bases), 4_000_000)])].astype(np.uint64)
    m = len(c) - k + 1
    fwd = np.zeros(m, np.uint64)
    rc = np.zeros(m, np.uint64)
    bad = np.zeros(m, bool)
    for j in range(k):
        cj = c[j:j + m]
        bad |= cj > 3
        fwd = (fwd << np.uint64(2)) | (cj & np.uint64(3))
        rc |= (np.uint64(3) - (cj & np.uint64(3))) << np.uint64(2 * j)
    canon = np.minimum(fwd, rc)[~bad]
    hits = canon[rng.integers(0, len(canon), n // 2)]
    miss = rng.integers(0, 1 << 62, n - n // 2, dtype=np.uint64) & np.uint64((1 << (2 * k)) - 1)
    out = np.concatenate([hits, miss])
    rng.shuffle(out)
    return out


def generate_reads(wl, bases, first, n_reads, out_seq, out_qual, threads):
    """Fills the pinned text (and quality) buffers block by block; blocks are pure functions of (seed, block
    index), so they are generated by a few threads at once (numpy releases the GIL in its inner loops)."""
    from concurrent.futures import ThreadPoolExecutor
    from shark_b200 import synth
    W = 2 * wl["L"] + 1 if wl["paired"] else wl["L"]
    want_q = wl["q"] > 0
    blocks = [(b, min(synth.BLOCK, n_reads - b * synth.BLOCK)) for b in range((n_reads + synth.BLOCK - 1) // synth.BLOCK)]

    def one(job):
        b, m = job
        t, q = synth.make_read_block(bases, wl["genes"], 3000, first // synth.BLOCK + b, synth.BLOCK, wl["L"], wl["paired"],
                                     2, want_q, want_q)
        a = b * synth.BLOCK
        out_seq[a * W:(a + m) * W] = t[:m].reshape(-1)
        if want_q:
            out_qual[a * W:(a + m) * W] = q[:m].reshape(-1)

    with ThreadPoolExecutor(max(1, min(threads, len(blocks)))) as ex:
        list(ex.map(one, blocks))


def make_workload(wl, rank, n_reads, gen_threads):
    """-> dict with the reference, pinned chunk lists in text and in packed form, keepalive buffers."""
    from shark_b200 import capi, synth
    names, bases, rec_off = synth.make_reference(wl["genes"], seed=1)
    W = 2 * wl["L"] + 1 if wl["paired"] else wl["L"]
    want_q = wl["q"] > 0
    blocks_per_rank = (wl["reads"] + synth.BLOCK - 1) // synth.BLOCK
    first = rank * blocks_per_rank * synth.BLOCK
    pin_seq = capi.PinnedBuffer(n_reads * W + 64)
    pin_qual = capi.PinnedBuffer(n_reads * W + 64) if want_q else None
    t0 = time.time()
    generate_reads(wl, bases, first, n_reads, pin_seq.u8, pin_qual.u8 if want_q else None, gen_threads)
    log("[bench] rank %d generated %d reads in %.1fs (%d threads)" % (rank, n_reads, time.time() - t0, gen_threads))
    pin_off = capi.PinnedBuffer((CHUNK_READS + 1) * 4)
    off32 = pin_off.view(np.uint32, CHUNK_READS + 1)
    off32[:] = np.arange(CHUNK_READS + 1, dtype=np.uint32) * np.uint32(W)
    chunks, packed, keep = [], [], [pin_seq, pin_qual, pin_off]
    t0 = time.time()
    for a in range(0, n_reads, CHUNK_READS):
        n = min(CHUNK_READS, n_reads - a)
        s = pin_seq.u8[a * W:(a + n) * W]
        q = pin_qual.u8[a * W:(a + n) * W] if want_q else None
        chunks.append((s, q, off32[:n + 1], n))
        # the same chunk in the packed form of shk_host_pack (what the CLI's batcher hands to shk_reads_submit_packed)
        g = (n * W + 31) // 32
        pc, pv = capi.PinnedBuffer(g * 8 + 64), capi.PinnedBuffer(g * 4 + 64)
        codes, valid = pc.view(np.uint64, g), pv.view(np.uint32, g)
        rc = capi.load().shk_host_pack(capi.ptr(s), capi.ptr(q) if want_q else None, wl["q"], n * W, capi.ptr(codes),
                                       capi.ptr(valid), 1)
        if rc:
            raise SystemExit("shk_host_pack failed")
        packed.append((codes, valid, off32[:n + 1], n))
        keep += [pc, pv]
    log("[bench] rank %d packed copies of the chunks in %.1fs" % (rank, time.time() - t0))
    return dict(names=names, bases=bases, rec_off=rec_off, chunks=chunks, packed=packed, keep=keep, W=W, first=first)


# ---------------------------------------------------------------------------------------------------------
# The reference's own CPU path: oracle/_ref/shark (the unmodified program) fed through named pipes.
# ---------------------------------------------------------------------------------------------------------
def reference_stream(wl, seq, qual, sample, workdir, threads, warm, timed, keep_ssv):
    """One run of oracle/_ref/shark -t threads whose sample files are named pipes: this process writes the
    FASTQ text of the first `sample` reads (warm + timed) times back to back.  A pass ends when its last byte
    has been accepted by the pipe, i.e. consumed by the reference up to the pipe's capacity; in steady state
    the time between two such points is the reference's time for one pass of the sample (index build and
    start-up are outside, every thread stays busy - the reference hands out batches of 50 000 reads,
    main.cpp:215).  -> (list of seconds per timed pass, path of the ssv or None)."""
    from shark_b200 import synth
    fa = os.path.join(workdir, "ref.fa")
    if not os.path.exists(fa):
        names, bases, rec_off = synth.make_reference(wl["genes"], seed=1)
        synth.write_fasta(fa, names, bases, rec_off)
    b1, b2 = synth.fastq_bytes(seq, qual, sample, wl["L"], wl["paired"])
    fifos = [os.path.join(workdir, "s_1.fq")] + ([os.path.join(workdir, "s_2.fq")] if wl["paired"] else [])
    for f in fifos:
        if os.path.exists(f):
            os.unlink(f)
        os.mkfifo(f)
    # our own read ends keep the pipes alive across the reference's open/close of every input at start-up
    # (main.cpp:88-106); they never read
    guards = [os.open(f, os.O_RDONLY | os.O_NONBLOCK) for f in fifos]
    cmd = [REF_BIN, "-r", fa, "-1", fifos[0], "-o", "/dev/null", "-k", str(wl["k"]), "-c", str(wl["c"]), "-b", str(wl["b"]),
           "-t", str(threads)]
    if wl["paired"]:
        cmd += ["-2", fifos[1], "-p", "/dev/null"]
    if wl["q"]:
        cmd += ["-q", str(wl["q"])]
    if wl["single"]:
        cmd += ["-s"]
    ssv = os.path.join(workdir, "ref.ssv") if keep_ssv else None
    fo = open(ssv, "wb") if keep_ssv else open(os.devnull, "wb")
    proc = subprocess.Popen(cmd, stdout=fo, stderr=subprocess.PIPE)
    marks, stage = [], {}

    def watch_stderr():  # the sample stage starts right after this stamp (main.cpp:194-199)
        for ln in proc.stderr:
            if b"Second switch performed" in ln and "t" not in stage:
                stage["t"] = time.perf_counter()

    def feed(path, data, record):
        fd = os.open(path, os.O_WRONLY)
        try:
            fcntl.fcntl(fd, 1031, 1 << 20)  # F_SETPIPE_SZ
        except OSError:
            pass
        mv = memoryview(data)
        try:
            for _ in range(warm + timed):
                o = 0
                while o < len(mv):
                    o += os.write(fd, mv[o:o + (1 << 20)])
                if record:
                    marks.append(time.perf_counter())
        except BrokenPipeError:
            pass
        finally:
            os.close(fd)

    ths = [threading.Thread(target=feed, args=(fifos[0], b1, True)), threading.Thread(target=watch_stderr)]
    if wl["paired"]:
        ths.append(threading.Thread(target=feed, args=(fifos[1], b2, False)))
    t_start = time.perf_counter()
    for t in ths:
        t.start()
    rc = proc.wait()
    t_exit = time.perf_counter()
    for g in guards:  # a reference that died early leaves the feeders blocked on a full pipe: this unblocks them
        os.close(g)
    for t in ths:
        t.join()
    fo.close()
    if rc != 0 or len(marks) != warm + timed:
        raise RuntimeError("reference run failed (rc %s, %d of %d passes)" % (rc, len(marks), warm + timed))
    edges = [stage.get("t", t_start)] + marks
    if warm == 0:
        # no warm-up pass: the timed passes run from the start of the sample stage (nothing in flight) to the end of
        # the process (nothing in flight); with warm-up passes both ends are "last byte consumed" in steady state
        edges[-1] = t_exit
    per_pass = [edges[i + 1] - edges[i] for i in range(warm + timed)]
    return per_pass[warm:], ssv


def reference_sample_reads(wl, n):
    """The first n reads of the workload's stream (what rank 0 holds) as text (+ qualities)."""
    from shark_b200 import synth
    names, bases, rec_off = synth.make_reference(wl["genes"], seed=1)
    want_q = wl["q"] > 0
    seq, qual, _ = synth.make_reads(bases, wl["genes"], n, wl["L"], wl["paired"], seed=2, varied_qual=want_q, want_qual=want_q)
    return seq, qual


def our_lines(sh, wd, first_name, n):
    """ssv lines of the first n reads of this rank's chunks, through the public API."""
    W, names = wd["W"], wd["names"]
    pref, left = [], n
    for c0 in wd["chunks"]:
        if left <= 0:
            break
        m = min(left, c0[3])
        pref.append((c0[0][: m * W], None if c0[1] is None else c0[1][: m * W], c0[2][: m + 1], m))
        left -= m
    ours, base = [], first_name
    for res, c0 in zip(sh.analyze_chunks(pref), pref):
        ridx, gidx, _ = sh.expand(res)
        ours += [b"r%09d %s" % (base + int(a), names[int(g)]) for a, g in zip(ridx, gidx)]
        base += c0[3]
    return ours


def cpu_baseline_leg(wl, sh, wd, cores, sample, passes=(1, 2)):
    """cpu_baseline of one workload: the reference on the first `sample` reads, streamed (1 warm-up pass + 2
    timed), and parity of the sorted ssv against our output for the same reads."""
    if not os.path.exists(REF_BIN):
        return {"value": None, "unit": unit_of(wl), "cores": cores, "kind": "reference", "sample": "oracle/_ref/shark is not built"}
    W = wd["W"]
    seq = wd["keep"][0].u8[: sample * W]          # the chunks are views of one buffer
    qual = wd["keep"][1].u8[: sample * W] if wl["q"] else None
    with tempfile.TemporaryDirectory() as tmp:
        t0 = time.perf_counter()
        per_pass, ssv = reference_stream(wl, seq, qual, sample, tmp, cores, passes[0], passes[1], True)
        whole = time.perf_counter() - t0
        t = float(np.mean(per_pass))
        ref_lines = sorted(ln for ln in open(ssv, "rb").read().split(b"\n") if ln)
    ours = sorted(our_lines(sh, wd, wd["first"], sample) * (passes[0] + passes[1]))
    return {"value": sample / t, "unit": unit_of(wl), "cores": cores, "kind": "reference",
            "sample": "first %d %s of the workload streamed %d+%d times through oracle/_ref/shark -t %d (named pipes, "
                      "steady state: %.2fs per pass; whole run with index build %.1fs)"
                      % (sample, "pairs" if wl["paired"] else "reads", passes[0], passes[1], cores, t, whole),
            "parity_on_sample": bool(ours == ref_lines), "ssv_lines": len(ref_lines) // (passes[0] + passes[1])}


def cli_leg(wl, wd, cores, n_total):
    """The process seam (main.cpp:83-240): shark-b200 and oracle/_ref/shark -t <cores> on the same FASTQ files
    in /dev/shm; wall times, reads/s and byte equality of sorted ssv and of the kept FASTQ records."""
    from shark_b200 import synth
    if not (os.path.exists(REF_BIN) and os.path.exists(CLI_BIN)):
        return {"unavailable": "oracle/_ref/shark or shark_b200/shark-b200 is not built"}
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    out = {"reads": n_total, "files": "uncompressed FASTQ in %s" % (base or "the temp directory")}
    with tempfile.TemporaryDirectory(dir=base) as tmp:
        fa = os.path.join(tmp, "ref.fa")
        synth.write_fasta(fa, wd["names"], wd["bases"], wd["rec_off"])
        f1, f2 = os.path.join(tmp, "s_1.fq"), os.path.join(tmp, "s_2.fq")
        W, done, t0 = wd["W"], 0, time.perf_counter()
        while done < n_total:  # the rank's chunks, repeated under fresh names until n_total reads are written
            for s, q, _, n in wd["chunks"]:
                m = min(n, n_total - done)
                if m <= 0:
                    break
                synth.write_fastq_fast(f1, f2, s, q, m, wl["L"], wl["paired"], first_name=done, append=done > 0)
                done += m
        out["input_bytes"] = os.path.getsize(f1) + (os.path.getsize(f2) if wl["paired"] else 0)
        log("[bench/cli] wrote %d reads (%.1f GB of FASTQ) in %.1fs" % (n_total, out["input_bytes"] / 1e9, time.perf_counter() - t0))
        flags = ["-k", str(wl["k"]), "-c", str(wl["c"]), "-b", str(wl["b"])]
        if wl["q"]:
            flags += ["-q", str(wl["q"])]
        if wl["single"]:
            flags += ["-s"]

        def run(binary, tag, extra, env=None):
            o1, o2, ssv = (os.path.join(tmp, "%s.%s" % (tag, x)) for x in ("o1.fq", "o2.fq", "ssv"))
            cmd = [binary, "-r", fa, "-1", f1, "-o", o1] + flags + extra
            if wl["paired"]:
                cmd += ["-2", f2, "-p", o2]
            t0 = time.perf_counter()
            with open(ssv, "wb") as fo:
                p = subprocess.run(cmd, stdout=fo, stderr=subprocess.PIPE, env=env)
            secs = time.perf_counter() - t0
            if p.returncode != 0:
                raise RuntimeError("%s failed: %s" % (tag, p.stderr.decode()[-500:]))
            return secs, ssv, o1, o2, p.stderr.decode()

        env = dict(os.environ, SHK_TIMING="1")
        ours_runs = []
        for _ in range(3):
            time.sleep(1.5)  # the device process of the previous run finishes its tear-down on its own (detached)
            ours_runs.append(run(CLI_BIN, "ours", ["-t", str(cores)], env))
        ours = ours_runs[0]
        ours2 = min(ours_runs[1:], key=lambda r: r[0])   # page cache and driver state warm
        ref = run(REF_BIN, "ref", ["-t", str(cores)])
        stamps = {}
        for ln in ours2[4].splitlines():
            if ln.startswith("[shark-b200/timing]"):
                parts = ln[len("[shark-b200/timing]"):].rsplit(None, 2)
                try:
                    stamps[parts[0].strip()] = float(parts[1])
                except (ValueError, IndexError):
                    pass

        def sorted_equal(a, b):
            ra = subprocess.run(["sort", a], stdout=subprocess.PIPE, env=dict(os.environ, LC_ALL="C")).stdout
            rb = subprocess.run(["sort", b], stdout=subprocess.PIPE, env=dict(os.environ, LC_ALL="C")).stdout
            return ra == rb and len(ra) > 0

        def fastq_equal(a, b):
            # records keyed by name: 4-line records -> one line each, sorted
            def key(path):
                p1 = subprocess.Popen(["paste", "-", "-", "-", "-"], stdin=open(path, "rb"), stdout=subprocess.PIPE)
                o = subprocess.run(["sort"], stdin=p1.stdout, stdout=subprocess.PIPE, env=dict(os.environ, LC_ALL="C")).stdout
                p1.wait()
                return o
            ka, kb = key(a), key(b)
            return ka == kb and len(ka) > 0

        steady = None
        if "output written" in stamps and "index ready" in stamps:
            # reads/s of the sample stage once the index exists and the pipeline runs (start-up excluded)
            span = stamps["output written"] - stamps["index ready"]
            steady = n_total / (span * 1e-3) if span > 0 else None
        out.update({
            "ours": {"wall_s": min(ours[0], ours2[0]), "wall_s_runs": [r[0] for r in ours_runs],
                     "fragments_per_s": n_total / min(ours[0], ours2[0]),
                     "after_device_start_fragments_per_s": steady, "stamps_ms": stamps,
                     "note": "wall = the process the user starts, from exec to exit (outputs complete); device start-up "
                             "(`contexts created`) is inside it; after_device_start = reads / (output written - index ready)"},
            "reference": {"wall_s": ref[0], "fragments_per_s": n_total / ref[0], "threads": cores},
            "speedup_wall": ref[0] / min(ours[0], ours2[0]),
            "ssv_sorted_equal": sorted_equal(ours2[1], ref[1]),
            "out1_records_equal": fastq_equal(ours2[2], ref[2]),
            "out2_records_equal": fastq_equal(ours2[3], ref[3]) if wl["paired"] else None,
            "ssv_lines": sum(1 for _ in open(ref[1], "rb")),
        })
    return out


def base_config(name, wl, n_reads, world, upload):
    W = 2 * wl["L"] + 1 if wl["paired"] else wl["L"]
    return {"workload": wl["desc"], "name": name, "reads_per_gpu": n_reads, "read_len": wl["L"], "paired": wl["paired"],
            "k": wl["k"], "bf_gib": wl["b"], "min_quality": wl["q"], "single": wl["single"], "c": wl["c"],
            "chunk_reads": CHUNK_READS, "fragment": "read pair" if wl["paired"] else "read",
            "sharding": "reads sharded by rank, index replicated (NCCL broadcast)" if world > 1 else "single GPU",
            "upload": ("e2e: plain text over PCIe" if upload == "plain" else
                       "e2e: split upload through shk_reads_submit (SHK_F_HOST_PACK): text in pinned host memory, part of "
                       "every chunk packed to 3 bits/base by the host cores inside the timed region, share = %s"
                       % ("auto-balanced" if upload == "split" else upload)),
            "l2": "inputs larger than L2: every step streams %d MB of reads and probes a %.1f GB filter at random"
                  % (n_reads * W // 1_000_000, wl["b"] * 8 / 7 * 1.0737)}


# ---------------------------------------------------------------------------------------------------------
# our arm, one workload
# ---------------------------------------------------------------------------------------------------------
def run_workload(name, args, rank, world, local_rank, cores, dist, torch):
    from shark_b200.engine import Shark
    wl = WORKLOADS[name]
    n_reads = args.reads or wl["reads"]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    wd = make_workload(wl, rank, n_reads, max(1, min(8, cores)))
    chunks, packed, W = wd["chunks"], wd["packed"], wd["W"]
    n_chunks = len(chunks)
    sh = Shark(k=wl["k"], c=wl["c"], bf_bits=wl["b"] << 33, min_quality=wl["q"], single=wl["single"], device=local_rank,
               n_slots=max(n_chunks, 2), max_reads_per_chunk=CHUNK_READS, max_bytes_per_chunk=CHUNK_READS * W,
               extend={"auto": None, "on": True, "off": False}[args.extend], compact=True)
    # ---- index: build on rank 0, replicate over NVLink; N > 1 also runs the sharded build and compares
    bcast_ms = 0.0
    index_mode = args.index or ("both" if world > 1 else "single")
    index_extra = {"mode": "single GPU" if world == 1 else index_mode}
    if world == 1 or index_mode in ("broadcast", "both"):
        if rank == 0:
            info = sh.build_index(wd["bases"], wd["rec_off"])
            log("[bench] %s index: %d genes, %d set bits, %d ids, %.2f ms on device (%.1f ms wall)" %
                (name, info.n_genes, info.n_set_bits, info.tot_ids, info.build_ms, info.build_wall_ms))
        if world > 1:
            from shark_b200 import dist_index
            bcast_ms = dist_index.broadcast_index(sh, src=0)
    if world > 1 and index_mode in ("sharded", "both"):
        from shark_b200 import dist_index
        before = sh.export_index() if index_mode == "both" else None
        b_info = sh.info
        barrier()
        s_info, s_secs = dist_index.build_index_sharded(sh, wd["bases"], wd["rec_off"])
        index_extra.update({"sharded_wall_ms": s_secs * 1e3, "sharded_device_ms": s_info.build_ms, "n_shards": s_info.n_shards,
                            "sharded_steps_wall_ms": getattr(dist_index.build_index_sharded, "last_steps_ms", None)})
        if before is not None:
            after = sh.export_index()
            same = all(np.array_equal(a, b) for a, b in zip(before, after)) and \
                (b_info.n_genes, b_info.n_set_bits, b_info.tot_ids) == (s_info.n_genes, s_info.n_set_bits, s_info.tot_ids)
            flag = torch.tensor([1.0 if same else 0.0], dtype=torch.float64, device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            index_extra["sharded_equals_broadcast"] = bool(flag.item() == 1.0)
            index_extra["sharded_equals_broadcast_checked_on"] = "every rank (exported set bits, CSR offsets and ids)"
            del before, after
        log("[bench] rank %d sharded index build: %.1f ms wall, %.2f ms on device" % (rank, s_secs * 1e3, s_info.build_ms))
    info = sh.info
    launches0 = sh.kernel_launches()

    # random-sector ceiling (kernel B0) for the secondary roofline denominator
    rs_ms = sh.random_sector_bench(1 << 28)
    rs_gbs = (1 << 28) * 32 / rs_ms / 1e6
    # stand-alone probe kernel (K5 = BF::get_index: filter word -> sector rank -> entry) on 2^25 canonical k-mers,
    # half hits / half misses: the "BF probe GB/s vs the random-sector roofline" half of the metric
    pk = probe_kmers(wd["bases"], wl["k"], 1 << 25)
    pb_ms, pb_hits = sh.probe_bench(pk, reps=4)
    pb_gbs = len(pk) * 32 / pb_ms / 1e6
    probe = {"kernel": "probe_bench_kernel (hash -> filter word -> sector + rank -> entry)", "probes": len(pk),
             "ms": pb_ms, "gprobes_per_s": len(pk) / pb_ms / 1e6, "achieved_gbs_32B_per_probe": pb_gbs,
             "random_sector_ceiling_gbs": rs_gbs, "frac_of_random_sector_ceiling": pb_gbs / rs_gbs if rs_gbs else None,
             "hit_fraction": pb_hits / len(pk)}
    del pk

    # ---- device-resident: upload once, then time K passes of the kernels + result read-back
    def resident_leg(form):
        for i in range(n_chunks):
            if form == "packed":
                sh.upload_packed(i, *packed[i])
            else:
                sh.upload(i, *chunks[i])

        def step():
            for i in range(n_chunks):
                sh.analyze_resident(i)
            return [sh.collect(i, copy=False) for i in range(n_chunks)]

        for _ in range(args.warmup):
            step()
        barrier()
        l0 = sh.kernel_launches()
        t0 = time.perf_counter()
        sh.timer_start()  # device stopwatch (CUDA events over all slot streams); the host clock is the cross-check
        tot = dict(n_probes=0, n_hits=0, n_assoc=0, n_slow_reads=0, n_extended=0, n_table_loads=0, n_multi=0, n_kept=0)
        for _ in range(args.steps):
            last = step()
            for r in last:
                for key in tot:
                    tot[key] += r[key]
        t_dev = sh.timer_stop() * 1e-3
        barrier()
        t_wall = time.perf_counter() - t0
        launches = sh.kernel_launches() - l0
        # the last timed step's results, copied before the roofline pass below overwrites the slots' result buffers
        outputs = [(r["gene16"].copy(), r["multi"].copy()) for r in last] if args.dump_outputs else None
        # roofline pass: the same launches one at a time (no overlap between the slots' streams), so that the
        # CUDA-event time of analyze_reads_kernel is the time of that kernel alone
        probe_ms = 0.0
        for _ in range(args.steps):
            for i in range(n_chunks):
                sh.analyze_resident(i)
                probe_ms += sh.collect(i, copy=False)["probe_kernel_ms"]
        return dict(t_dev=t_dev, t_wall=t_wall, launches=launches, probe_ms=probe_ms, outputs=outputs, **tot)

    sampler = ClockSampler(local_rank)
    sampler.start()
    res_text = resident_leg("text")
    res_packed = resident_leg("packed")

    # ---- end to end through the public API: pinned host chunks -> H2D -> kernels -> D2H
    sh.n_slots = max(2, min(args.e2e_slots, n_chunks))  # slots reused round-robin by analyze_chunks
    leg_stats = {}

    def e2e_leg(mode):
        # K steps = K passes over the rank's chunks as ONE stream through the slots (a step boundary does not drain
        # the pipeline: a sample is a stream of chunks, not a sequence of separately flushed batches)
        kms = [0.0, 0]

        def seen(r):  # device time of the classification kernels of this chunk, while the copies of the next ones run
            kms[0] += r["analyze_ms"]
            kms[1] += 1

        if mode == "packed":
            sh.set_upload_mode(False)
            run = lambda k: sh.analyze_chunks(packed * k, copy=False, on_result=seen, packed=True)  # noqa: E731
        else:
            sh.set_upload_mode(False if mode == "plain" else (True if mode == "split" else float(mode)))
            run = lambda k: sh.analyze_chunks(chunks * k, copy=False, on_result=seen)  # noqa: E731
        if args.warmup:
            run(args.warmup)
        barrier()
        h0, dd0 = sh.h2d_bytes(), sh.d2h_bytes()
        t0 = time.perf_counter()
        sh.timer_start()
        kms[0], kms[1] = 0.0, 0
        run(args.steps)
        t_dev = sh.timer_stop() * 1e-3
        # the split upload packs on the host BEFORE a chunk's first device operation: the device stopwatch would
        # miss the packing of the first chunk, the host clock around the same region does not
        barrier()
        t_wall = time.perf_counter() - t0
        leg_stats[mode] = sh.upload_stats()
        t = max(t_dev, t_wall) if mode not in ("plain", "packed") else t_dev
        return dict(t=t, t_dev=t_dev, t_wall=t_wall, h2d=(sh.h2d_bytes() - h0) // max(args.steps, 1),
                    d2h=(sh.d2h_bytes() - dd0) // max(args.steps, 1), kernels_ms_per_chunk=kms[0] / max(kms[1], 1))

    legs = {}
    for mode in ("plain", "packed", args.upload):
        if mode not in legs:
            legs[mode] = e2e_leg(mode)
    clocks = sampler.stop()

    # ---- max over ranks (device times; the wall-clock figures ride along as a cross-check)
    keys = [res_text["t_dev"], res_packed["t_dev"], res_text["probe_ms"], res_packed["probe_ms"], res_text["t_wall"],
            legs[args.upload]["t"], legs["plain"]["t"], legs["packed"]["t"], legs[args.upload]["t_wall"]]
    times = torch.tensor(keys, dtype=torch.float64, device="cuda")
    sums = torch.tensor([float(res_text["n_probes"]), float(res_text["n_hits"]), float(res_text["n_assoc"]),
                         float(legs[args.upload]["h2d"]), float(legs[args.upload]["d2h"]),
                         float(res_packed["n_assoc"]), float(res_packed["n_probes"])], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    (t_text, t_packed, pm_text, pm_packed, t_text_wall, t_e2e, t_plain, t_e2e_packed, t_e2e_wall) = times.tolist()
    total = n_reads * world * args.steps
    forms_agree = res_text["n_assoc"] == res_packed["n_assoc"] and res_text["n_probes"] == res_packed["n_probes"]

    peak, peak_src = measured_peaks()

    def roofline_of(res, probe_ms_max, form):
        launches = args.steps * n_chunks
        ppl = res["n_probes"] / max(launches, 1)
        ms = probe_ms_max / max(launches, 1)
        achieved = 32.0 * ppl / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        traffic, traffic_src = traffic_for(name + "_" + form)
        # packed reads over the extension structures are classified by the bulk kernel (shk_bulk.cu) unless SHK_BULK=0;
        # the thread-per-read kernel extends only over a DRAM-sized table (info.plain_front: slots-only copy in L2)
        bulk = form == "packed" and info.extend and os.environ.get("SHK_BULK", "1")[:1] != "0"
        ext_k6 = bool(info.extend) and not info.plain_front
        uses_ext = bulk or ext_k6
        kname = "analyze_bulk_kernel (packed reads, diagonals + shared lookups)" if bulk else \
            "analyze_reads_kernel<%s%s>" % ("PACKED" if form == "packed" else "TEXT", ", EXT" if ext_k6 else "")
        return {"bound": "hbm", "kernel": kname,
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src, "algorithmic_bytes_per_launch": 32.0 * ppl,
                "probes_per_launch": ppl, "kernel_ms_per_launch": ms, "launches_per_step": n_chunks,
                "hit_fraction": res["n_hits"] / max(res["n_probes"], 1), "extend": bool(uses_ext),
                "extended_fraction": res["n_extended"] / max(res["n_probes"], 1),
                "table_loads_per_probe": (res["n_table_loads"] / max(res["n_probes"], 1)) if uses_ext else 1.0,
                "random_sector_ceiling_gbs": rs_gbs, "frac_of_random_sector_ceiling": achieved / rs_gbs if rs_gbs else None,
                "limiter": ("instruction issue (hash + coarse filter of the windows that are not copied from the window before) "
                            "and L2/DRAM latency at 24 warps per SM; DRAM traffic is below the algorithmic bytes because "
                            "most windows need no table access at all (DESIGN.md 3, 5)") if bulk else
                           ("integer ALU pipe (hashing); DRAM traffic is below the algorithmic bytes because the exact "
                            "front table / extension structures answer most probes from L2 (DESIGN.md 3, 5)")}

    value_form = args.value_form
    t_value = t_packed if value_form == "packed" else t_text
    res_v = res_packed if value_form == "packed" else res_text
    roofline = roofline_of(res_v, pm_packed if value_form == "packed" else pm_text, value_form)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, name if world == 1 else "%s_rank%d" % (name, rank), res_v["outputs"], args.dump_bytes)

    # ---- parity
    cpu_baseline, parity_ranks = None, None
    if not args.no_cpu_baseline:
        if world == 1:
            cpu_baseline = cpu_baseline_leg(wl, sh, wd, cores, min(args.cpu_sample or wl["cpu_sample"], n_reads))
        else:
            # every rank checks the first reads of ITS shard, on ITS replica of the index, against the reference binary
            ok = rank_parity(wl, sh, wd, args.rank_sample)
            flag = torch.tensor([1.0 if ok else 0.0], dtype=torch.float64, device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.SUM)
            parity_ranks = {"ranks_ok": int(flag.item()), "ranks": world, "sample_per_rank": args.rank_sample,
                            "how": "sorted ssv of the first reads of each rank's own shard, computed on that rank's GPU, "
                                   "against oracle/_ref/shark on the same reads"}
    cli = None
    if world == 1 and name == "c2" and not args.no_cli:
        try:
            cli = cli_leg(wl, wd, cores, args.cli_reads)
        except Exception as e:  # the process seam is reported, never fatal for the kernel numbers
            cli = {"error": str(e)[-400:]}

    h2d_step, d2h_step = sums.tolist()[3] / world, sums.tolist()[4] / world
    u = unit_of(wl)
    # aggregate host-to-device rate of every e2e leg: beyond one GPU per host they converge on the host's ceiling
    agg = {"text_split": h2d_step * world / (t_e2e / args.steps) / 1e9,
           "text_plain": legs["plain"]["h2d"] * world / (t_plain / args.steps) / 1e9,
           "packed": legs["packed"]["h2d"] * world / (t_e2e_packed / args.steps) / 1e9}
    host_limit = {"h2d_gbs_all_gpus_by_leg": agg, "max_gbs": max(agg.values()), "ranks_on_host": world, "cores_per_rank": cores,
                  "note": "every e2e leg moves its bytes out of ONE host's memory: past one GPU the legs converge on the same "
                          "aggregate rate whatever the form of the reads - the host's ceiling, not the GPUs' and not NVLink's; "
                          "fewer bytes per read (packed: 0.375 B per base) is what moves more reads through it"}
    rec = {
        "metric": "reads/sec", "value": total / t_value, "unit": u, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": t_value / args.steps * 1e3,
        "timing": "CUDA events over all slot streams (shk_device_timer_*), max over ranks",
        "wall_ms_per_step": t_text_wall / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": dict(base_config(name, wl, n_reads, world, args.upload), resident_form=value_form),
        "value_by_form": {"text": total / t_text, "packed": total / t_packed, "unit": u, "forms_agree": bool(forms_agree),
                          "note": "reads resident in HBM as text (1 byte per base, + qualities with -q) or in the packed form "
                                  "(0.375 bytes per base, masking folded in); identical results"},
        "mates_per_s": total * (2 if wl["paired"] else 1) / t_value,
        "e2e": {"value": total / t_e2e, "unit": u, "h2d_bytes_per_step": int(h2d_step), "d2h_bytes_per_step": int(d2h_step),
                "upload": args.upload, "slots": sh.n_slots, "packed_share": leg_stats[args.upload][0],
                "pack_gbases_per_s": leg_stats[args.upload][1], "ms_per_step": t_e2e / args.steps * 1e3,
                "wall_ms_per_step": t_e2e_wall / args.steps * 1e3, "pack": "%s, %d threads" % capi_pack_info(),
                "kernels_ms_per_chunk_while_copying": legs[args.upload]["kernels_ms_per_chunk"],
                "h2d_gbs_per_gpu": h2d_step / (t_e2e / args.steps) / 1e9, "d2h_gbs_per_gpu": d2h_step / (t_e2e / args.steps) / 1e9,
                "h2d_gbs_all_gpus": h2d_step * world / (t_e2e / args.steps) / 1e9,
                "input": "read text (and qualities with -q) in pinned host memory"},
        "e2e_plain": {"value": total / t_plain, "unit": u, "h2d_bytes_per_step": int(legs["plain"]["h2d"]),
                      "ms_per_step": t_plain / args.steps * 1e3, "input": "read text in pinned host memory, no host packing"},
        "e2e_packed": {"value": total / t_e2e_packed, "unit": u, "h2d_bytes_per_step": int(legs["packed"]["h2d"]),
                       "d2h_bytes_per_step": int(legs["packed"]["d2h"]), "ms_per_step": t_e2e_packed / args.steps * 1e3,
                       "kernels_ms_per_chunk_while_copying": legs["packed"]["kernels_ms_per_chunk"],
                       "input": "pinned host buffers already in the packed form the CLI's batcher emits (packing NOT in "
                                "the timed region): shk_reads_submit_packed"},
        "host_limit": host_limit,
        "gpu_launches": int(res_v["launches"]), "roofline": roofline,
        "roofline_text": roofline_of(res_text, pm_text, "text") if value_form == "packed" else None,
        "probe": probe, "cpu_baseline": cpu_baseline, "parity_ranks": parity_ranks, "cli": cli, "clocks": clocks,
        "index": {"n_genes": info.n_genes, "n_set_bits": info.n_set_bits, "tot_ids": info.tot_ids,
                  "build_ms": info.build_ms, "build_wall_ms": info.build_wall_ms, "broadcast_ms": bcast_ms,
                  "device_bytes": info.device_bytes, **index_extra},
        "associations_per_step": sums.tolist()[2] / args.steps / world, "slow_reads_per_step": res_v["n_slow_reads"] / args.steps,
        "multi_entries_per_step": res_v["n_multi"] / args.steps, "kept_per_step": res_v["n_kept"] / args.steps,
    }
    sh.close()
    for b in wd["keep"]:
        if b is not None:
            b.free()
    return rec


def rank_parity(wl, sh, wd, sample):
    if not os.path.exists(REF_BIN):
        return False
    W = wd["W"]
    c0 = wd["chunks"][0]
    sample = min(sample, c0[3])
    seq = np.array(c0[0][: sample * W])
    qual = np.array(c0[1][: sample * W]) if wl["q"] else None
    cores = len(os.sched_getaffinity(0))
    with tempfile.TemporaryDirectory() as tmp:
        _, ssv = reference_stream(wl, seq, qual, sample, tmp, max(1, min(4, cores)), 0, 1, True)
        ref_lines = sorted(ln for ln in open(ssv, "rb").read().split(b"\n") if ln)
    # the reference names its reads from r000000000; ours carry the shard's first read index: compare with local names
    ours = sorted(our_lines(sh, wd, 0, sample))
    return bool(ours == ref_lines and len(ours) > 0)


def capi_pack_info():
    from shark_b200 import capi
    return capi.host_pack_info()


def pin_rank_cores(local_rank, local_world):
    """N ranks on one host: every rank keeps to its own slice of the cores this job may use (its submitting
    thread and its pack threads then never migrate onto another rank's cores)."""
    if local_world <= 1 or os.environ.get("SHK_BENCH_PIN", "1") == "0" or not hasattr(os, "sched_setaffinity"):
        return None
    cpus = sorted(os.sched_getaffinity(0))
    per = len(cpus) // local_world
    if per < 1:
        return None
    mine = cpus[local_rank * per:(local_rank + 1) * per]
    try:
        os.sched_setaffinity(0, mine)
    except OSError:
        return None
    return mine


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workloads", "--workload", default="", help="comma-separated subset of c2,c3,c4,c5; the first is the "
                    "headline (default: c4,c3,c2 on one GPU, c5 under torchrun)")
    ap.add_argument("--reads", type=int, default=0, help="override reads per GPU (testing)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="reads per pass given to the CPU reference (0 = per workload)")
    ap.add_argument("--rank-sample", type=int, default=20000, help="N > 1: reads of every rank's shard checked against the reference")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cli", action="store_true")
    ap.add_argument("--cli-reads", type=int, default=20_000_000)
    ap.add_argument("--extend", default="auto", choices=["auto", "on", "off"],
                    help="anchor-and-extend: automatic (on for DRAM-sized front tables), or forced (A/B runs)")
    ap.add_argument("--upload", default="split",
                    help="how the headline e2e moves the reads: 'plain' (text over PCIe), 'split' (part of every chunk packed to "
                         "3 bits per base by the host cores while the rest is in flight, auto-balanced) or a fixed packed share "
                         "in (0, 1]")
    ap.add_argument("--value-form", default="packed", choices=["text", "packed"],
                    help="form in which the reads are resident in HBM for `value` (both are measured: value_by_form)")
    ap.add_argument("--e2e-slots", type=int, default=5, help="chunks in flight in the e2e legs")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last one returned for every workload as DIR/<workload>_"
                         "{read,gene,assoc}.npy (float, at most 64 MB in all), so that two builds can be compared")
    ap.add_argument("--index", default="", choices=["", "broadcast", "sharded", "both"],
                    help="N > 1: build on rank 0 + NCCL broadcast, the sharded P2P OR-merge build, or both (default) with an "
                         "equality check on every rank")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    names = [w for w in args.workloads.split(",") if w] or (["c5"] if world > 1 else ["c4", "c3", "c2"])
    for w in names:
        if w not in WORKLOADS:
            raise SystemExit("unknown workload %r" % w)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what this project computes; the reference arm computes nothing of ours")
    args.dump_bytes = DUMP_BYTES // (len(names) * world)   # every workload and rank gets an equal share
    head = WORKLOADS[names[0]]

    # ---------------------------------------------------------------- reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
        n_reads = args.reads or head["reads"]
        sample = min(args.cpu_sample or head["cpu_sample"], n_reads)
        if not os.path.exists(REF_BIN):
            print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/shark is not built"}))
            return 0
        seq, qual = reference_sample_reads(head, sample)
        with tempfile.TemporaryDirectory() as tmp:
            t0 = time.perf_counter()
            per_pass, _ = reference_stream(head, seq, qual, sample, tmp, cores, args.warmup, args.steps, False)
            whole = time.perf_counter() - t0
        t = float(np.mean(per_pass))
        v = sample / t
        u = unit_of(head)
        log("[bench/reference] %d passes of %d: %.2fs per pass (whole run %.1fs)" % (args.steps, sample, t, whole))
        sample_desc = ("first %d %s of the workload per step, streamed through one oracle/_ref/shark -t %d process over named "
                       "pipes (steady state; index build outside the timed steps; whole run %.1fs)"
                       % (sample, "pairs" if head["paired"] else "reads", cores, whole))
        print(json.dumps({
            "impl": "reference", "metric": "reads/sec", "value": v, "unit": u, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": dict(base_config(names[0], head, n_reads, world, args.upload), resident_form=args.value_form),
            "cpu_baseline": {"value": v, "unit": u, "cores": cores, "kind": "reference", "sample": sample_desc},
            "e2e": {"value": v, "unit": u, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        return 0

    # ---------------------------------------------------------------- our arm
    # libraries (NCCL's version banner, ...) may write to fd 1: keep the real stdout for the ONE
    # JSON line and send everything else to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    pinned = pin_rank_cores(local_rank, local_world)
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    os.environ.setdefault("SHK_PACK_THREADS", str(max(1, min(32, cores))))
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    records = {}
    for w in names:
        t0 = time.time()
        records[w] = run_workload(w, args, rank, world, local_rank, cores, dist, torch)
        log("[bench] rank %d workload %s done in %.1fs" % (rank, w, time.time() - t0))
    if rank == 0:
        out = dict(records[names[0]])
        out["host"] = {"cores_per_rank": cores, "ranks_on_host": local_world,
                       "rank_core_slice": ("cpus %d-%d" % (pinned[0], pinned[-1])) if pinned else "not pinned"}
        out["workloads"] = {w: records[w] for w in names}
        real_stdout.write(json.dumps(out) + "\n")
        real_stdout.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
