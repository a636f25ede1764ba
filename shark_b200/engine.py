"""Host-side mirror of the reference's hot-path interface on top of the C ABI.

`Shark` owns one context (= one GPU).  Its methods follow the reference's stages:
  build_index   = pass 1 + BF::switch_mode(1) + pass 2 + BF::switch_mode(2)   (main.cpp:128-193)
  get_index     = BF::get_index                                               (bloomfilter.h:78-102)
  analyze       = FastqSplitter masking + ReadAnalyzer::operator()            (ReadAnalyzer.hpp:39-110)
All compute happens in libshark_b200.so; nothing here touches oracle/.
"""
import ctypes as C

import numpy as np

from . import capi


class Shark:
    def __init__(self, k=17, c=0.6, bf_bits=1 << 33, min_quality=0, single=False, device=0, n_slots=2,
                 max_reads_per_chunk=1 << 20, max_bytes_per_chunk=0, extend=None, host_pack=False, compact=False,
                 wide_ids=False, scores=False):
        """extend: None = automatic (anchor-and-extend when the front table is DRAM-sized), True /
        False = force it on / off (results are identical; tests run both).  compact: results stay in the
        compact form (gene16 / multi), shk_reads_collect does no per-read host work.  scores: every result also
        carries the per-read score records {len, cov, hits, n_best} (SHK_F_SCORES, include/shark_b200.h)."""
        self.lib = capi.load()
        flags = 0 if extend is None else (capi.F_EXTEND_ON if extend else capi.F_EXTEND_OFF)
        if compact:
            flags |= capi.F_COMPACT_RESULTS
        if wide_ids:  # SURVEY.md 8f.4: 32-bit gene ids (more than 65536 reference records), an opt-in extension
            flags |= capi.F_WIDE_IDS
        if scores:
            flags |= capi.F_SCORES
        self.compact = bool(compact)
        self.scores = bool(scores)
        self.wide_ids = bool(wide_ids)
        permille = 0
        if host_pack:  # split upload: part of every chunk is packed to 3 bits per base by the host cores
            flags |= capi.F_HOST_PACK
            if host_pack is not True:  # a number in (0, 1]: fixed share instead of the automatic balance
                permille = max(1, min(1000, int(round(float(host_pack) * 1000))))
        self.params = capi.Params(k=k, c=c, bf_bits=bf_bits, min_quality=min_quality, single=int(bool(single)),
                                  device=device, n_slots=n_slots, max_reads_per_chunk=max_reads_per_chunk,
                                  max_bytes_per_chunk=max_bytes_per_chunk, flags=flags,
                                  host_pack_permille=permille)
        self.ctx = C.c_void_p()
        rc = self.lib.shk_create(C.byref(self.params), C.byref(self.ctx))
        if rc:
            raise capi.SharkError(rc, self.lib.shk_last_error(None).decode())
        self.k, self.c, self.bf_bits = k, c, bf_bits
        self.min_quality, self.single = min_quality, bool(single)
        self.n_slots = n_slots
        self.max_reads = max_reads_per_chunk
        self.max_bytes = max_bytes_per_chunk or 320 * max_reads_per_chunk
        self.info = None
        self._staging = {}

    # -- lifetime ---------------------------------------------------------------------------
    def close(self):
        if getattr(self, "ctx", None):
            self.lib.shk_destroy(self.ctx)
            self.ctx = None
        for _, bufs in getattr(self, "_staging", {}).values():
            for b in bufs:
                if b is not None:
                    b.free()
        self._staging = {}

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc):
        if rc:
            raise capi.SharkError(rc, self.lib.shk_last_error(self.ctx).decode())

    # -- index ------------------------------------------------------------------------------
    def build_index(self, bases, rec_off):
        """bases: uint8 concatenated record sequences as parsed; rec_off: uint64[n_records+1]."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
        info = capi.IndexInfo()
        self._check(self.lib.shk_index_build(self.ctx, capi.ptr(bases) if len(bases) else None, capi.ptr(rec_off),
                                             len(rec_off) - 1, C.byref(info)))
        self.info = info
        return info

    # -- sharded build (SURVEY.md 8e second mode): per-GPU gene shards + P2P OR-merge ---------
    def shard_begin(self, bases, rec_off, shard, n_shards):
        """Pass 1 over this context's shard of the records -> capi.ShardMem (exchange it with the peers)."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
        mem = capi.ShardMem()
        self._check(self.lib.shk_shard_begin(self.ctx, capi.ptr(bases) if len(bases) else None, capi.ptr(rec_off),
                                             len(rec_off) - 1, shard, n_shards, C.byref(mem)))
        return mem

    def shard_open(self, peer):
        opened = capi.ShardMem()
        self._check(self.lib.shk_shard_open(self.ctx, C.byref(peer), C.byref(opened)))
        return opened

    def shard_close(self, opened):
        self._check(self.lib.shk_shard_close(self.ctx, C.byref(opened)))

    def shard_merge(self, phase, all_mem):
        self._check(self.lib.shk_shard_merge(self.ctx, phase, all_mem))

    def shard_rank(self):
        self._check(self.lib.shk_shard_rank(self.ctx))

    def shard_finish(self, all_mem):
        info = capi.IndexInfo()
        self._check(self.lib.shk_shard_finish(self.ctx, all_mem, C.byref(info)))
        self.info = info
        return info

    def shard_end(self):
        self._check(self.lib.shk_shard_end(self.ctx))

    @staticmethod
    def build_index_sharded(sharks, bases, rec_off):
        """The whole sharded protocol for several contexts of this process (shk_index_build_sharded)."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
        arr = (C.c_void_p * len(sharks))(*[s.ctx for s in sharks])
        info = capi.IndexInfo()
        rc = sharks[0].lib.shk_index_build_sharded(arr, len(sharks), capi.ptr(bases) if len(bases) else None,
                                                   capi.ptr(rec_off), len(rec_off) - 1, C.byref(info))
        sharks[0]._check(rc)
        for s in sharks:
            i = capi.IndexInfo()
            s._check(s.lib.shk_index_info_get(s.ctx, C.byref(i)))
            s.info = i
        return info

    # -- index serialisation ------------------------------------------------------------------
    def save_index(self, path):
        self._check(self.lib.shk_index_save(self.ctx, str(path).encode()))

    def load_index(self, path):
        info = capi.IndexInfo()
        self._check(self.lib.shk_index_load(self.ctx, str(path).encode(), C.byref(info)))
        self.info = info
        return info

    # -- staged build: the reference's functor protocol (KmerBuilder / BloomfilterFiller / class BF) --
    def kmer_hashes(self, bases, rec_off):
        """KmerBuilder::operator() (KmerBuilder.hpp:40-72) -> uint64 hashes of all canonical k-mers."""
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        rec_off = np.ascontiguousarray(rec_off, dtype=np.uint64)
        out = np.zeros(max(len(bases), 1), np.uint64)
        n = C.c_uint64()
        self._check(self.lib.shk_kmer_hashes(self.ctx, capi.ptr(bases) if len(bases) else None, capi.ptr(rec_off),
                                             len(rec_off) - 1, capi.ptr(out), len(bases), C.byref(n)))
        return out[: n.value].copy()

    def add_at(self, positions):
        """BloomfilterFiller::operator() / BF::add_at (bloomfilter.h:57-59) for a batch."""
        positions = np.ascontiguousarray(positions, dtype=np.uint64)
        self._check(self.lib.shk_bf_add_at(self.ctx, capi.ptr(positions) if len(positions) else None, len(positions)))

    def switch_mode(self, new_mode):
        """BF::switch_mode (bloomfilter.h:112-184) -> number of set bits."""
        n = C.c_uint64()
        self._check(self.lib.shk_bf_switch_mode(self.ctx, new_mode, C.byref(n)))
        if new_mode == 2:
            info = capi.IndexInfo()
            self._check(self.lib.shk_index_info_get(self.ctx, C.byref(info)))
            self.info = info
        return n.value

    def add_to_kmer(self, kmers, input_idx):
        """BF::add_to_kmer (bloomfilter.h:61-75)."""
        kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
        self._check(self.lib.shk_bf_add_to_kmer(self.ctx, capi.ptr(kmers) if len(kmers) else None, len(kmers), input_idx))

    def mode(self):
        return self.lib.shk_bf_mode(self.ctx)

    def set_options(self, k=None, c=None, min_quality=None, single=None):
        k = self.k if k is None else k
        c = self.c if c is None else c
        q = self.min_quality if min_quality is None else min_quality
        s = self.single if single is None else bool(single)
        self._check(self.lib.shk_set_options(self.ctx, k, c, q, int(s)))
        self.k, self.c, self.min_quality, self.single = k, c, q, s

    def export_index(self, wide=None):
        """-> (set_bit_pos uint64[n_set], offsets uint32[n_set+1], ids uint16[tot_ids]); ids uint32 through
        shk_index_export_wide when wide (default: what the index holds)"""
        n, t = self.info.n_set_bits, self.info.tot_ids
        wide = (self.info.id_bits == 32) if wide is None else wide
        pos = np.zeros(n, np.uint64)
        off = np.zeros(n + 1, np.uint32)
        ids = np.zeros(t, np.uint32 if wide else np.uint16)
        fn = self.lib.shk_index_export_wide if wide else self.lib.shk_index_export
        self._check(fn(self.ctx, capi.ptr(pos) if n else None, capi.ptr(off), capi.ptr(ids) if t else None))
        return pos, off, ids

    def index_views(self):
        v = capi.IndexViews()
        self._check(self.lib.shk_index_views_get(self.ctx, C.byref(v)))
        return v

    def adopt_index(self, info):
        self._check(self.lib.shk_index_adopt(self.ctx, C.byref(info)))
        self.info = info

    def finalize_index(self):
        self._check(self.lib.shk_index_finalize(self.ctx))

    def get_index(self, kmers):
        """BF::get_index for canonical k-mers -> (rank int64 (-1 = miss), begin uint32, len uint32)."""
        kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
        n = len(kmers)
        rank = np.zeros(n, np.int64)
        begin = np.zeros(n, np.uint32)
        ln = np.zeros(n, np.uint32)
        if n:
            self._check(self.lib.shk_probe(self.ctx, capi.ptr(kmers), n, capi.ptr(rank), capi.ptr(begin), capi.ptr(ln)))
        return rank, begin, ln

    def probe_bench(self, kmers, reps=3):
        kmers = np.ascontiguousarray(kmers, dtype=np.uint64)
        ms, hits = C.c_float(), C.c_uint64()
        self._check(self.lib.shk_probe_bench(self.ctx, capi.ptr(kmers), len(kmers), reps, C.byref(ms), C.byref(hits)))
        return ms.value, hits.value

    def random_sector_bench(self, n_loads, span_bytes=0, seed=1):
        ms = C.c_float()
        self._check(self.lib.shk_random_sector_bench(self.ctx, n_loads, span_bytes, seed, C.byref(ms)))
        return ms.value

    # -- reads ------------------------------------------------------------------------------
    def submit(self, slot, seq, qual, off32, n_reads):
        self._check(self.lib.shk_reads_submit(self.ctx, slot, capi.ptr(seq), capi.ptr(qual) if qual is not None else None,
                                              capi.ptr(off32), n_reads))

    def submit_packed(self, slot, codes, valid, off32, n_reads):
        """The chunk in the packed form of capi.host_pack (masking already applied)."""
        self._check(self.lib.shk_reads_submit_packed(self.ctx, slot, capi.ptr(codes), capi.ptr(valid), capi.ptr(off32), n_reads))

    def upload_packed(self, slot, codes, valid, off32, n_reads):
        self._check(self.lib.shk_reads_upload_packed(self.ctx, slot, capi.ptr(codes), capi.ptr(valid), capi.ptr(off32), n_reads))

    def upload(self, slot, seq, qual, off32, n_reads):
        self._check(self.lib.shk_reads_upload(self.ctx, slot, capi.ptr(seq), capi.ptr(qual) if qual is not None else None,
                                              capi.ptr(off32), n_reads))

    def analyze_resident(self, slot):
        self._check(self.lib.shk_reads_analyze_resident(self.ctx, slot))

    def collect(self, slot, copy=True):
        """-> dict(read_idx, gene_idx, keep, gene16, multi, n_probes, n_hits, analyze_ms, ...); with compact=True
        the expanded arrays (read_idx, gene_idx, keep) are None; with scores=True, scores = uint32[n_reads, 4]
        (len, cov, hits, n_best per read)."""
        res = capi.ChunkResult()
        self._check(self.lib.shk_reads_collect(self.ctx, slot, C.byref(res)))
        n = res.n_assoc
        gene16 = np.ctypeslib.as_array(res.gene16, shape=(max(res.n_reads, 1),))[: res.n_reads]
        if res.n_multi:
            multi = np.ctypeslib.as_array(C.cast(res.multi, C.POINTER(C.c_uint32)), shape=(res.n_multi, 2))
        else:
            multi = np.zeros((0, 2), np.uint32)
        if copy:
            gene16, multi = gene16.copy(), multi.copy()
        a = keep = None
        if not self.compact:
            if n:
                a = np.ctypeslib.as_array(C.cast(res.assoc, C.POINTER(C.c_uint32)), shape=(n, 2))
            else:
                a = np.zeros((0, 2), np.uint32)
            keep = np.ctypeslib.as_array(res.keep, shape=(max(res.n_reads, 1),))[: res.n_reads]
            if copy:
                a, keep = a.copy(), keep.copy()
        scores = None
        if self.scores:
            sp, ns = C.POINTER(capi.ReadScore)(), C.c_uint32()
            self._check(self.lib.shk_reads_scores(self.ctx, slot, C.byref(sp), C.byref(ns)))
            if ns.value:
                scores = np.ctypeslib.as_array(C.cast(sp, C.POINTER(C.c_uint32)), shape=(ns.value, 4))
                if copy:
                    scores = scores.copy()
            else:
                scores = np.zeros((0, 4), np.uint32)
        return dict(read_idx=None if a is None else a[:, 0], gene_idx=None if a is None else a[:, 1], keep=keep, scores=scores,
                    gene16=gene16, multi=multi, n_multi=int(res.n_multi), n_kept=int(res.n_kept),
                    n_assoc=int(n), n_reads=res.n_reads,
                    n_slow_reads=res.n_slow_reads, n_probes=res.n_probes, n_hits=res.n_hits,
                    analyze_ms=res.analyze_ms, total_ms=res.total_ms, kernel_launches=res.kernel_launches,
                    probe_kernel_ms=res.probe_kernel_ms, n_extended=res.n_extended, n_table_loads=res.n_table_loads)

    @staticmethod
    def expand(result):
        """Compact result dict -> (read_idx uint32[n_assoc], gene_idx uint32[n_assoc], keep uint8[n_reads]),
        vectorised (what shk_result_expand does in C)."""
        g = result["gene16"].astype(np.uint32)
        keep = (g != capi.GENE_NONE).astype(np.uint8)
        single = np.nonzero(g < capi.GENE_MULTI)[0].astype(np.uint32)
        multi = result["multi"]
        ridx = np.concatenate([single, multi[:, 0]])
        gidx = np.concatenate([g[single], multi[:, 1]])
        order = np.lexsort((gidx, ridx))
        return ridx[order], gidx[order], keep

    def timer_start(self):
        """Device stopwatch (CUDA events) over all slot streams of this context."""
        self._check(self.lib.shk_device_timer_start(self.ctx))

    def timer_stop(self):
        """-> device milliseconds since timer_start, after everything enqueued in between has finished."""
        ms = C.c_float()
        self._check(self.lib.shk_device_timer_stop(self.ctx, C.byref(ms)))
        return ms.value

    def set_upload_mode(self, host_pack):
        """False = plain text upload; True = split upload, balanced automatically; a number in (0, 1] = fixed share."""
        auto = host_pack is None or isinstance(host_pack, bool)   # (1.0 == True in Python: test the type)
        permille = 0 if auto else max(1, min(1000, int(round(float(host_pack) * 1000))))
        self._check(self.lib.shk_set_upload_mode(self.ctx, int(bool(host_pack)), permille))

    def upload_stats(self):
        """-> (share of a chunk the host packs, last packing rate in Gbases/s)"""
        a, b = C.c_double(), C.c_double()
        self._check(self.lib.shk_upload_stats(self.ctx, C.byref(a), C.byref(b)))
        return a.value, b.value

    def h2d_bytes(self):
        return int(self.lib.shk_h2d_bytes(self.ctx))

    def d2h_bytes(self):
        return int(self.lib.shk_d2h_bytes(self.ctx))

    def kernel_launches(self):
        return int(self.lib.shk_kernel_launches(self.ctx))

    def _stage(self, slot, nbytes_seq, n_reads, with_qual):
        key = slot
        need = (nbytes_seq, n_reads, with_qual)
        cur = self._staging.get(key)
        if cur is None or cur[0][0] < nbytes_seq or cur[0][1] < n_reads or (with_qual and not cur[0][2]):
            if cur is not None:
                for b in cur[1]:
                    if b is not None:
                        b.free()
            cap_b = max(nbytes_seq, 1 << 16)
            cap_r = max(n_reads, 1 << 10)
            bufs = (capi.PinnedBuffer(cap_b), capi.PinnedBuffer(cap_b) if with_qual else None,
                    capi.PinnedBuffer((cap_r + 1) * 4))
            cur = ((cap_b, cap_r, with_qual), bufs)
            self._staging[key] = cur
        return cur[1]

    def plan_chunks(self, off):
        """Splits reads [0, n) into chunks that fit a slot -> list of (first, last) read indices."""
        off = np.asarray(off)
        n = len(off) - 1
        chunks, i = [], 0
        while i < n:
            j = min(i + self.max_reads, n)
            if int(off[j]) - int(off[i]) > self.max_bytes:
                j = int(np.searchsorted(off, int(off[i]) + self.max_bytes, side="right")) - 1
                if j <= i:
                    raise capi.SharkError(-4, "read %d alone exceeds max_bytes_per_chunk" % i)
            chunks.append((i, j))
            i = j
        return chunks

    def analyze(self, seq, off, qual=None, packed=False):
        """Classifies reads given as SoA (seq uint8, off uint64/uint32 [n+1], qual uint8|None):
        chunks them, streams the chunks through the slots (pinned staging, double buffered) and
        returns (keep uint8[n], assoc_read uint64[m], assoc_gene uint32[m], stats); with scores=True
        stats["scores"] = uint32[n, 4].  packed=True: every
        chunk is reduced to codes + validity bits with shk_host_pack first and goes through
        shk_reads_submit_packed (what the CLI's batcher does)."""
        seq = np.ascontiguousarray(seq, dtype=np.uint8)
        off = np.ascontiguousarray(off)
        n = len(off) - 1
        with_qual = (self.min_quality & 0xFF) != 0
        if with_qual and qual is None:
            raise capi.SharkError(-1, "min_quality != 0 needs qualities")
        keep = np.zeros(n, np.uint8)
        out_r, out_g, out_s = [], [], []
        stats = dict(n_probes=0, n_hits=0, analyze_ms=0.0, probe_kernel_ms=0.0, n_slow_reads=0, kernel_launches=0, chunks=0,
                     n_extended=0, n_table_loads=0)
        chunks = self.plan_chunks(off) if n else []
        pending = []

        def drain():
            slot, first = pending.pop(0)
            r = self.collect(slot)
            if self.compact:
                r["read_idx"], r["gene_idx"], r["keep"] = self.expand(r)
                assert len(r["read_idx"]) == r["n_assoc"] and int(r["keep"].sum()) == r["n_kept"]
            keep[first:first + r["n_reads"]] = r["keep"]
            out_r.append(r["read_idx"].astype(np.uint64) + np.uint64(first))
            out_g.append(r["gene_idx"])
            if self.scores:
                out_s.append(r["scores"])
            for key in ("n_probes", "n_hits", "analyze_ms", "probe_kernel_ms", "n_slow_reads", "kernel_launches",
                        "n_extended", "n_table_loads"):
                stats[key] += r[key]
            stats["chunks"] += 1

        for ci, (a, b) in enumerate(chunks):
            slot = ci % self.n_slots
            if len(pending) == self.n_slots:
                drain()
            base = int(off[a])
            nb = int(off[b]) - base
            s_seq, s_qual, s_off = self._stage(slot, nb, b - a, with_qual)
            o32 = s_off.view(np.uint32, b - a + 1)
            o32[:] = (off[a:b + 1] - off[a]).astype(np.uint32)
            if packed:
                codes, valid = capi.host_pack(seq[base:base + nb], qual[base:base + nb] if with_qual else None,
                                              self.min_quality)
                g = len(codes)
                s_seq.u8[:g * 8] = codes.view(np.uint8)      # the staging buffers are pinned: reuse them
                pv = s_seq.u8[((g * 8 + 63) // 64) * 64:][:g * 4]
                pv[:] = valid.view(np.uint8)
                self.submit_packed(slot, s_seq.u8[:g * 8].view(np.uint64) if g else s_seq.u8[:0].view(np.uint64),
                                   pv.view(np.uint32), o32, b - a)
            else:
                s_seq.u8[:nb] = seq[base:base + nb]
                if with_qual:
                    s_qual.u8[:nb] = qual[base:base + nb]
                self.submit(slot, s_seq.u8, s_qual.u8 if with_qual else None, o32, b - a)
            pending.append((slot, a))
        while pending:
            drain()
        ar = np.concatenate(out_r) if out_r else np.zeros(0, np.uint64)
        ag = np.concatenate(out_g) if out_g else np.zeros(0, np.uint32)
        if self.scores:  # per read {len, cov, hits, n_best}, in read order
            stats["scores"] = np.concatenate(out_s) if out_s else np.zeros((0, 4), np.uint32)
        return keep, ar, ag, stats

    def analyze_chunks(self, chunks, copy=True, on_result=None, packed=False):
        """Streams pre-chunked host inputs through the slots, double buffered: chunk i+1 is
        submitted (H2D + kernels enqueued) before chunk i is collected.  `chunks` is a sequence
        of (seq uint8, qual uint8|None, off32 uint32[n+1], n_reads) whose arrays should live in
        pinned memory (capi.PinnedBuffer) so that the copies are asynchronous - this is what the
        FASTQ batcher of the host side produces.  packed=True: the chunks are (codes uint64, valid uint32,
        off32, n_reads) in the packed form and go through shk_reads_submit_packed.  Returns the per-chunk
        result dicts in order (or feeds them to on_result)."""
        results, pending = [], []

        def drain():
            slot = pending.pop(0)
            r = self.collect(slot, copy=copy)
            if on_result is not None:
                on_result(r)
            else:
                results.append(r)

        for ci, (seq, qual, off32, n_reads) in enumerate(chunks):
            slot = ci % self.n_slots
            if len(pending) == self.n_slots:
                drain()
            if packed:
                self.submit_packed(slot, seq, qual, off32, n_reads)
            else:
                self.submit(slot, seq, qual, off32, n_reads)
            pending.append(slot)
        while pending:
            drain()
        return results
