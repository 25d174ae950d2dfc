"""ctypes binding of libhetmers_b200.so (include/hetmers_b200.h).  The library is built in-tree by
`make lib` / `__graft_entry__.build()`; if it is missing this module raises -- there is no CPU or
PyTorch fallback for the hetmers path."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HETMERS_LIB") or os.path.join(HERE, "lib", "libhetmers_b200.so")   # (override: tuning builds)
BIN_PATH = os.path.join(HERE, "bin", "hetmers")

SMAX, FMAX = 1000, 500
PLOT_W = FMAX + 1
PLOT_CELLS = (SMAX + 1) * (FMAX + 1)

# every symbol include/hetmers_b200.h declares (tests check the .so exports all of them)
ABI_SYMBOLS = [
    "hm_last_error", "hm_abi_version", "hm_device_count", "hm_device_info",
    "hm_k_unpack_records", "hm_k_build_bucket_index", "hm_k_pass1_degree", "hm_k_pass2_plot",
    "hm_k_min_count", "hm_k_find_keys", "hm_pick_bucket_bits", "hm_k_pass2_extract", "hm_scan_extract", "hm_scan_extract_path", "hm_pass2_scratch_bytes",
    "hm_k_build_filter", "hm_filter_words", "hm_pick_filter_bits",
    "hm_dev_alloc", "hm_dev_free", "hm_ipc_export", "hm_ipc_open", "hm_ipc_close", "hm_p2p_native_atomics",
    "hm_scan_create", "hm_prewarm", "hm_set_io_threads", "hm_scan_destroy", "hm_scan_examine", "hm_scan_condition", "hm_scan_run", "hm_hetmers_host",
    "hm_scan_run_path", "hm_scan_is_symmetric", "hm_symm_plan", "hm_symm_seeds", "hm_k_symm_fingerprint", "hm_k_symm_runscan", "hm_k_symm_runs", "hm_k_symm_resolve",
    "hm_symm_status", "hm_symm_align_cut",
    "hm_scan_download", "hm_scan_create_sharded", "hm_scan_shard_info", "hm_shard_cuts", "hm_plan_placement", "hm_device_free_bytes",
    "hm_table_open", "hm_table_close", "hm_table_view", "hm_write_smu",
]


class HostTable(C.Structure):
    _fields_ = [("kmer", C.c_int32), ("ibyte", C.c_int32), ("nparts", C.c_int32), ("minval", C.c_int32),
                ("nels", C.c_int64), ("index", C.POINTER(C.c_int64)), ("part_nels", C.POINTER(C.c_int64)),
                ("part_rec", C.POINTER(C.c_void_p)), ("part_fd", C.POINTER(C.c_int32)),
                ("part_fd_off", C.POINTER(C.c_int64))]


MAX_SHARDS = 16


class Shards(C.Structure):
    """hm_shards: shard offsets + every owner's full-length incidence array as seen from this GPU"""
    _fields_ = [("n_shards", C.c_int32), ("self_", C.c_int32), ("off", C.c_int64 * (MAX_SHARDS + 1)),
                ("deg", C.c_void_p * MAX_SHARDS), ("scratch", C.c_void_p), ("scratch_bytes", C.c_int64)]


class SymmLayout(C.Structure):
    """hm_symm_layout: work area of the strand-symmetric scan"""
    _fields_ = [("bytes", C.c_int64), ("off_header", C.c_int64), ("off_bloom", C.c_int64), ("seg_words", C.c_int64),
                ("off_cand_key", C.c_int64), ("off_cand_lo", C.c_int64), ("off_cand_meta", C.c_int64),
                ("cand_cap", C.c_int64), ("range", C.c_int64), ("off_runs", C.c_int64), ("runs_cap", C.c_int64),
                ("n_seg", C.c_int32), ("pad", C.c_int32)]


class SymmShards(C.Structure):
    """hm_symm_shards: run-aligned shard cuts + the first key of every shard"""
    _fields_ = [("n_seg", C.c_int32), ("self_", C.c_int32), ("off", C.c_int64 * (MAX_SHARDS + 1)),
                ("first_key", C.c_uint64 * MAX_SHARDS)]


SYMM_ASYMMETRIC, SYMM_OVERFLOW = 1, 2
PLACE_NOFIT, PLACE_REPLICA, PLACE_SHARDED = 0, 1, 2
EINVAL, EUNSUPPORTED = -1, -6


class PairRec(C.Structure):
    """hm_pair_rec: one line of extract_kmer_pairs' output"""
    _fields_ = [("key_hi", C.c_uint64), ("key_lo", C.c_uint64), ("smudge", C.c_uint32),
                ("pos", C.c_uint8), ("alt", C.c_uint8), ("pad", C.c_uint16)]


class ExtractStats(C.Structure):
    """hm_extract_stats: route, slices and times of one extraction"""
    _fields_ = [("path", C.c_int32), ("slices", C.c_int32), ("n_records", C.c_int64),
                ("ms_kernel", C.c_double), ("ms_copy", C.c_double), ("ms_sort", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class ScanStats(C.Structure):
    _fields_ = [("nels", C.c_int64), ("n_gpus", C.c_int32), ("bucket_bits", C.c_int32),
                ("filter_bits", C.c_int32), ("path", C.c_int32),
                ("ms_h2d_unpack", C.c_double), ("ms_pass1", C.c_double), ("ms_pass2", C.c_double),
                ("ms_scan", C.c_double), ("ms_total", C.c_double), ("kernel_launches", C.c_int64),
                ("ms_alloc", C.c_double), ("ms_records", C.c_double), ("ms_index", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class HetmersError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libhetmers_b200 error {code}: {msg}")
        self.code = code


_lib = None


def lib():
    """Load the shared library once; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `make lib` (or __graft_entry__.build()); "
                          "the hetmers path has no CPU / PyTorch fallback")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int, C.c_int64
    L.hm_last_error.restype = C.c_char_p
    L.hm_device_info.argtypes = [i32, C.c_char_p, i32, C.POINTER(i32), C.POINTER(i64)]
    L.hm_k_unpack_records.argtypes = [vp, i64, i64, vp, i32, i32, vp, vp, vp, vp]
    L.hm_k_build_bucket_index.argtypes = [vp, i64, i32, vp, i32, vp]
    L.hm_k_pass1_degree.argtypes = [vp, vp, vp, i64, vp, i32, i32, vp, i32, i32, i64, i64, vp, vp, C.POINTER(Shards), vp]
    L.hm_dev_alloc.argtypes = [i64, C.POINTER(vp)]
    L.hm_dev_free.argtypes = [vp]
    L.hm_ipc_export.argtypes = [vp, C.c_char_p]
    L.hm_ipc_open.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.hm_ipc_close.argtypes = [vp]
    L.hm_p2p_native_atomics.argtypes = [i32, i32]
    L.hm_k_build_filter.argtypes = [vp, i64, i32, vp, vp]
    L.hm_filter_words.argtypes = [i32]
    L.hm_filter_words.restype = i64
    L.hm_pick_filter_bits.argtypes = [i64]
    L.hm_k_pass2_plot.argtypes = [vp, vp, vp, i32, i64, i64, vp, C.POINTER(Shards), vp]
    L.hm_k_min_count.argtypes = [vp, i64, i64, vp, vp]
    L.hm_k_find_keys.argtypes = [vp, vp, i64, vp, i32, i32, vp, vp, i64, vp, vp]
    L.hm_pick_bucket_bits.argtypes = [i64]
    L.hm_pass2_scratch_bytes.argtypes = [i64, i32]
    L.hm_pass2_scratch_bytes.restype = i64
    L.hm_symm_plan.argtypes = [i64, i64, i32, i32, C.POINTER(SymmLayout)]
    L.hm_symm_seeds.argtypes = [C.POINTER(C.c_uint64)]
    L.hm_symm_seeds.restype = None
    L.hm_k_symm_fingerprint.argtypes = [vp, vp, vp, i64, i64, i32, C.POINTER(C.c_uint64), vp, vp]
    L.hm_k_symm_runscan.argtypes = [vp, vp, vp, i64, vp, i32, i32, i32, i64, i64, vp, C.POINTER(SymmLayout),
                                    C.POINTER(SymmShards), vp]
    L.hm_k_symm_runs.argtypes = [vp, vp, vp, i64, vp, i32, i32, i32, i64, i64, vp, C.POINTER(SymmLayout),
                                 C.POINTER(SymmShards), vp]
    L.hm_k_symm_resolve.argtypes = [vp, vp, vp, i64, vp, i32, i32, i32, vp, C.POINTER(SymmLayout),
                                    C.POINTER(SymmShards), vp, vp]
    L.hm_symm_status.argtypes = [vp, C.POINTER(SymmLayout), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), vp]
    L.hm_symm_align_cut.argtypes = [vp, i64, i32, i64, C.POINTER(i64)]
    L.hm_scan_create.argtypes = [C.POINTER(HostTable), C.POINTER(i32), i32, C.POINTER(vp)]
    L.hm_scan_destroy.argtypes = [vp]
    L.hm_scan_destroy.restype = None
    L.hm_scan_examine.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(i32)]
    L.hm_scan_condition.argtypes = [vp, i32, i32, i32, C.POINTER(i64)]
    L.hm_scan_run.argtypes = [vp, vp, C.POINTER(ScanStats)]
    L.hm_scan_run_path.argtypes = [vp, i32, vp, C.POINTER(ScanStats)]
    L.hm_scan_is_symmetric.argtypes = [vp]
    L.hm_scan_extract.argtypes = [vp, vp, C.POINTER(C.POINTER(PairRec)), C.POINTER(i64)]
    L.hm_scan_extract_path.argtypes = [vp, i32, vp, C.POINTER(C.POINTER(PairRec)), C.POINTER(i64),
                                       C.POINTER(ExtractStats)]
    L.hm_hetmers_host.argtypes = [C.POINTER(HostTable), C.POINTER(i32), i32, vp, C.POINTER(ScanStats)]
    L.hm_scan_download.argtypes = [vp, vp, vp, vp, vp]
    L.hm_scan_create_sharded.argtypes = [C.POINTER(HostTable), C.POINTER(i32), i32, C.POINTER(vp)]
    L.hm_scan_shard_info.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]
    L.hm_shard_cuts.argtypes = [vp, vp, vp, i64, i32, i32, i32, i32, C.POINTER(C.c_uint64)]
    L.hm_device_free_bytes.argtypes = [i32, C.POINTER(i64)]
    L.hm_plan_placement.argtypes = [i32, i64, i32, i32, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]
    L.hm_table_open.argtypes = [C.c_char_p, C.POINTER(vp)]
    L.hm_table_close.argtypes = [vp]
    L.hm_table_close.restype = None
    L.hm_table_view.argtypes = [vp]
    L.hm_table_view.restype = C.POINTER(HostTable)
    L.hm_write_smu.argtypes = [C.c_char_p, vp]
    _lib = L
    return L


def check(rc: int):
    if rc != 0:
        raise HetmersError(rc, lib().hm_last_error().decode(errors="replace"))


def plan_placement(kmer: int, nels: int, free_bytes, do_symm: bool = False):
    """-> (PLACE_*, bytes per device of a replica, bytes per device of a shard) for a table of nels
    entries on len(free_bytes) devices (hm_plan_placement)"""
    fb = (C.c_int64 * len(free_bytes))(*[int(x) for x in free_bytes])
    rep, shd = C.c_int64(), C.c_int64()
    r = lib().hm_plan_placement(kmer, nels, int(do_symm), len(free_bytes), fb, C.byref(rep), C.byref(shd))
    if r < 0:
        check(r)
    return r, rep.value, shd.value


def shard_cuts(hi, lo, cnt, kmer: int, n_shards: int, min_count: int = 0, add_rc: bool = False):
    """cut keys of n_shards run-aligned key ranges from a sample of records (hm_shard_cuts): uint64[n_shards]"""
    import numpy as np
    hi = np.ascontiguousarray(hi, dtype=np.uint64)
    lo = None if lo is None else np.ascontiguousarray(lo, dtype=np.uint64)
    cnt = None if cnt is None else np.ascontiguousarray(cnt, dtype=np.uint16)
    out = (C.c_uint64 * n_shards)()
    check(lib().hm_shard_cuts(hi.ctypes.data, None if lo is None else lo.ctypes.data,
                              None if cnt is None else cnt.ctypes.data, hi.size, kmer, min_count, int(add_rc),
                              n_shards, out))
    return np.array(out[:], dtype=np.uint64)
