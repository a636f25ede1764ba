"""ctypes binding of libshark_b200.so (include/shark_b200.h).

This is the only way Python reaches the product: every compute call goes through the C ABI into
the CUDA kernels.  There is no CPU fallback; a missing library or device raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# SHK_LIB: tuning builds (shark_b200/build.py --variant); the product is libshark_b200.so
LIB_PATH = os.environ.get("SHK_LIB") or os.path.join(_HERE, "libshark_b200.so")

SHK_OK = 0
STATUS = {0: "SHK_OK", -1: "SHK_E_ARG", -2: "SHK_E_CUDA", -3: "SHK_E_STATE", -4: "SHK_E_CAPACITY", -5: "SHK_E_LIMIT",
          -6: "SHK_E_NOMEM"}

EXPORTED = [
    "shk_abi_version", "shk_create", "shk_destroy", "shk_last_error", "shk_index_build", "shk_index_info_get",
    "shk_index_export", "shk_index_views_get", "shk_index_adopt", "shk_index_finalize", "shk_index_replicate", "shk_probe", "shk_probe_bench",
    "shk_random_sector_bench", "shk_alloc_pinned", "shk_free_pinned", "shk_reads_submit", "shk_reads_collect",
    "shk_reads_upload", "shk_reads_analyze_resident", "shk_kernel_launches", "shk_device_timer_start",
    "shk_device_timer_stop", "shk_kmer_hashes", "shk_bf_add_at", "shk_bf_switch_mode", "shk_bf_add_to_kmer", "shk_bf_mode",
    "shk_set_options", "shk_shard_begin", "shk_shard_open", "shk_shard_close", "shk_shard_merge", "shk_shard_rank",
    "shk_shard_finish", "shk_shard_end", "shk_shard_cuts", "shk_index_build_sharded", "shk_index_save", "shk_index_load",
    "shk_host_pack", "shk_host_pack_info", "shk_h2d_bytes", "shk_d2h_bytes", "shk_set_upload_mode", "shk_upload_stats",
    "shk_reads_submit_packed", "shk_reads_upload_packed", "shk_result_expand", "shk_index_export_wide", "shk_reads_scores",
]


class SharkError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("%s: %s" % (STATUS.get(code, code), msg))
        self.code = code


class Params(C.Structure):
    _fields_ = [("k", C.c_uint32), ("c", C.c_double), ("bf_bits", C.c_uint64), ("min_quality", C.c_int32),
                ("single", C.c_int32), ("device", C.c_int32), ("n_slots", C.c_uint32),
                ("max_reads_per_chunk", C.c_uint32), ("max_bytes_per_chunk", C.c_uint64), ("flags", C.c_uint32),
                ("host_pack_permille", C.c_uint32), ("reserved", C.c_uint32 * 6)]


F_EXTEND_ON, F_EXTEND_OFF, F_HOST_PACK, F_COMPACT_RESULTS, F_WIDE_IDS, F_SCORES = 1, 2, 4, 8, 16, 32
GENE_NONE, GENE_MULTI = 0xFFFF, 0xFFFE


class IndexInfo(C.Structure):
    _fields_ = [("n_records", C.c_uint32), ("n_genes", C.c_uint32), ("n_set_bits", C.c_uint64), ("tot_ids", C.c_uint64),
                ("n_windows", C.c_uint64), ("bf_bits", C.c_uint64), ("device_bytes", C.c_uint64), ("build_ms", C.c_float),
                ("front_shift", C.c_uint32), ("front_entries", C.c_uint64), ("ref_bases", C.c_uint64),
                ("extend", C.c_uint32), ("coarse_shift", C.c_uint32), ("build_wall_ms", C.c_float),
                ("n_shards", C.c_uint32), ("id_bits", C.c_uint32), ("plain_front", C.c_uint32)]


class ShardMem(C.Structure):
    """shk_shard_mem: one context's buffers in the sharded index build."""
    _fields_ = [("dev_ptr", C.c_void_p * 3), ("ipc_handle", (C.c_uint8 * 64) * 3), ("pid", C.c_int64),
                ("device", C.c_int32), ("shard", C.c_uint32), ("ipc_ok", C.c_uint32), ("reserved", C.c_uint32)]


class IndexViews(C.Structure):
    _fields_ = [("dev_ptr", C.c_void_p * 8), ("bytes", C.c_uint64 * 8), ("info", IndexInfo)]


class Assoc(C.Structure):
    _fields_ = [("read_idx", C.c_uint32), ("gene_idx", C.c_uint32)]


class ReadScore(C.Structure):
    """shk_read_score: a read is reported iff n_best > 0 and cov >= c * len (IEEE double) and (not -s or n_best == 1)."""
    _fields_ = [("len", C.c_uint32), ("cov", C.c_uint32), ("hits", C.c_uint32), ("n_best", C.c_uint32)]


class ChunkResult(C.Structure):
    _fields_ = [("n_assoc", C.c_uint64), ("assoc", C.POINTER(Assoc)), ("keep", C.POINTER(C.c_uint8)),
                ("n_reads", C.c_uint32), ("n_slow_reads", C.c_uint32), ("n_probes", C.c_uint64), ("n_hits", C.c_uint64),
                ("analyze_ms", C.c_float), ("total_ms", C.c_float), ("kernel_launches", C.c_uint32),
                ("probe_kernel_ms", C.c_float), ("n_extended", C.c_uint64), ("n_table_loads", C.c_uint64),
                ("gene16", C.POINTER(C.c_uint16)), ("multi", C.POINTER(Assoc)), ("n_multi", C.c_uint64),
                ("n_kept", C.c_uint64)]


_lib = None


def load():
    """Loads the in-tree shared library (build it with `python shark_b200/build.py`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SharkError(-2, "libshark_b200.so is not built (python shark_b200/build.py); there is no fallback")
    L = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    L.shk_abi_version.restype = C.c_int
    L.shk_create.argtypes = [C.POINTER(Params), C.POINTER(vp)]
    L.shk_destroy.argtypes = [vp]
    L.shk_destroy.restype = None
    L.shk_last_error.argtypes = [vp]
    L.shk_last_error.restype = C.c_char_p
    L.shk_index_build.argtypes = [vp, vp, vp, C.c_uint32, C.POINTER(IndexInfo)]
    L.shk_index_info_get.argtypes = [vp, C.POINTER(IndexInfo)]
    L.shk_index_export.argtypes = [vp, vp, vp, vp]
    L.shk_index_export_wide.argtypes = [vp, vp, vp, vp]
    L.shk_index_views_get.argtypes = [vp, C.POINTER(IndexViews)]
    L.shk_index_adopt.argtypes = [vp, C.POINTER(IndexInfo)]
    L.shk_index_finalize.argtypes = [vp]
    L.shk_index_replicate.argtypes = [vp, vp]
    L.shk_probe.argtypes = [vp, vp, C.c_uint64, vp, vp, vp]
    L.shk_probe_bench.argtypes = [vp, vp, C.c_uint64, C.c_uint32, C.POINTER(C.c_float), C.POINTER(C.c_uint64)]
    L.shk_random_sector_bench.argtypes = [vp, C.c_uint64, C.c_uint64, C.c_uint64, C.POINTER(C.c_float)]
    L.shk_alloc_pinned.argtypes = [C.POINTER(vp), C.c_size_t]
    L.shk_free_pinned.argtypes = [vp]
    L.shk_reads_submit.argtypes = [vp, C.c_uint32, vp, vp, vp, C.c_uint32]
    L.shk_reads_collect.argtypes = [vp, C.c_uint32, C.POINTER(ChunkResult)]
    L.shk_reads_submit_packed.argtypes = [vp, C.c_uint32, vp, vp, vp, C.c_uint32]
    L.shk_reads_upload_packed.argtypes = [vp, C.c_uint32, vp, vp, vp, C.c_uint32]
    L.shk_result_expand.argtypes = [C.POINTER(ChunkResult), vp, vp]
    L.shk_reads_scores.argtypes = [vp, C.c_uint32, C.POINTER(C.POINTER(ReadScore)), C.POINTER(C.c_uint32)]
    L.shk_reads_upload.argtypes = [vp, C.c_uint32, vp, vp, vp, C.c_uint32]
    L.shk_reads_analyze_resident.argtypes = [vp, C.c_uint32]
    L.shk_device_timer_start.argtypes = [vp]
    L.shk_device_timer_stop.argtypes = [vp, C.POINTER(C.c_float)]
    L.shk_kernel_launches.argtypes = [vp]
    L.shk_kmer_hashes.argtypes = [vp, vp, vp, C.c_uint32, vp, C.c_uint64, C.POINTER(C.c_uint64)]
    L.shk_bf_add_at.argtypes = [vp, vp, C.c_uint64]
    L.shk_bf_switch_mode.argtypes = [vp, C.c_int, C.POINTER(C.c_uint64)]
    L.shk_bf_add_to_kmer.argtypes = [vp, vp, C.c_uint64, C.c_int32]
    L.shk_bf_mode.argtypes = [vp]
    L.shk_set_options.argtypes = [vp, C.c_uint32, C.c_double, C.c_int32, C.c_int32]
    L.shk_shard_begin.argtypes = [vp, vp, vp, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(ShardMem)]
    L.shk_shard_open.argtypes = [vp, C.POINTER(ShardMem), C.POINTER(ShardMem)]
    L.shk_shard_close.argtypes = [vp, C.POINTER(ShardMem)]
    L.shk_shard_merge.argtypes = [vp, C.c_int, C.POINTER(ShardMem)]
    L.shk_shard_rank.argtypes = [vp]
    L.shk_shard_finish.argtypes = [vp, C.POINTER(ShardMem), C.POINTER(IndexInfo)]
    L.shk_shard_end.argtypes = [vp]
    L.shk_shard_cuts.argtypes = [vp, C.c_uint32, C.c_uint32, vp]
    L.shk_index_build_sharded.argtypes = [C.POINTER(vp), C.c_uint32, vp, vp, C.c_uint32, C.POINTER(IndexInfo)]
    L.shk_index_save.argtypes = [vp, C.c_char_p]
    L.shk_index_load.argtypes = [vp, C.c_char_p, C.POINTER(IndexInfo)]
    L.shk_host_pack.argtypes = [vp, vp, C.c_int32, C.c_uint64, vp, vp, C.c_int32]
    L.shk_host_pack_info.argtypes = [C.POINTER(C.c_int32)]
    L.shk_host_pack_info.restype = C.c_char_p
    L.shk_set_upload_mode.argtypes = [vp, C.c_uint32, C.c_uint32]
    L.shk_upload_stats.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.shk_h2d_bytes.argtypes = [vp]
    L.shk_h2d_bytes.restype = C.c_uint64
    L.shk_d2h_bytes.argtypes = [vp]
    L.shk_d2h_bytes.restype = C.c_uint64
    L.shk_kernel_launches.restype = C.c_uint64
    for name in EXPORTED:
        f = getattr(L, name)
        if name in ("shk_host_pack_info", "shk_h2d_bytes", "shk_d2h_bytes", "shk_kernel_launches", "shk_last_error", "shk_destroy"):
            continue
        if f.restype is C.c_int or name in ("shk_create",):
            f.restype = C.c_int
    _lib = L
    return L


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class PinnedBuffer:
    """Host staging memory from shk_alloc_pinned, viewed as a numpy array."""

    def __init__(self, nbytes):
        self._p = C.c_void_p()
        rc = load().shk_alloc_pinned(C.byref(self._p), nbytes)
        if rc:
            raise SharkError(rc, load().shk_last_error(None).decode())
        self.nbytes = nbytes
        self.u8 = np.ctypeslib.as_array(C.cast(self._p, C.POINTER(C.c_uint8)), shape=(max(nbytes, 1),))[:nbytes]

    def view(self, dtype, count=None):
        a = self.u8.view(dtype)
        return a if count is None else a[:count]

    def free(self):
        if self._p:
            load().shk_free_pinned(self._p)
            self._p = C.c_void_p()
            self.u8 = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def host_pack(seq, qual=None, min_quality=0, parallel=False):
    """shk_host_pack: (codes uint64[ceil(n/32)], valid uint32[ceil(n/32)]) of a text buffer.  Pure host code."""
    seq = np.ascontiguousarray(seq, dtype=np.uint8)
    n = len(seq)
    g = (n + 31) // 32
    codes = np.zeros(max(g, 1), np.uint64)
    valid = np.zeros(max(g, 1), np.uint32)
    if qual is not None:
        qual = np.ascontiguousarray(qual, dtype=np.uint8)
    rc = load().shk_host_pack(ptr(seq) if n else None, ptr(qual) if qual is not None and n else None, min_quality, n,
                              ptr(codes), ptr(valid), int(parallel))
    if rc:
        raise SharkError(rc, load().shk_last_error(None).decode())
    return codes[:g], valid[:g]


def host_pack_info():
    n = C.c_int32()
    isa = load().shk_host_pack_info(C.byref(n)).decode()
    return isa, n.value
