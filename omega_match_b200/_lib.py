"""Loader and ctypes signatures for libomega_match.so (the B200 build).

The library is the product; there is no Python or CPU matching path behind it.  If the
shared object is missing (or `OMEGA_MATCH_LIB_PATH`, the reference binding's override --
bindings/python/omega_match/omega_match.py:409-420 -- points nowhere) importing fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG_DIR = Path(__file__).resolve().parent
DEFAULT_LIB = PKG_DIR / "lib" / "libomega_match.so"


class PatternStoreStatsC(C.Structure):  # include/olm_b200.h, [ref list_matcher.h:32-40]
    _fields_ = [("total_input_bytes", C.c_uint64), ("total_stored_bytes", C.c_uint64),
                ("stored_pattern_count", C.c_uint32), ("short_pattern_count", C.c_uint32),
                ("duplicate_patterns", C.c_uint32), ("smallest_pattern_length", C.c_uint32),
                ("largest_pattern_length", C.c_uint32)]


class MatchStatsC(C.Structure):  # [ref list_matcher.h:43-49]
    _fields_ = [("total_hits", C.c_uint64), ("total_misses", C.c_uint64), ("total_filtered", C.c_uint64),
                ("total_attempts", C.c_uint64), ("total_comparisons", C.c_uint64)]


class MatchResultC(C.Structure):  # [ref list_matcher.h:19-23]
    _fields_ = [("offset", C.c_size_t), ("len", C.c_uint32), ("match", C.c_void_p)]


class MatchResultsC(C.Structure):  # [ref list_matcher.h:26-29]
    _fields_ = [("count", C.c_size_t), ("matches", C.POINTER(MatchResultC))]


class CudaResultsC(C.Structure):
    _fields_ = [("count", C.c_uint64), ("records", C.c_void_p), ("device", C.c_int)]


class CudaTimingC(C.Structure):
    _fields_ = [("total_ms", C.c_float), ("transform_ms", C.c_float), ("scan_ms", C.c_float),
                ("filter_ms", C.c_float), ("h2d_ms", C.c_float), ("d2h_ms", C.c_float),
                ("scan_launches", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("matches_before_filter", C.c_uint64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class ShardC(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("own_begin", "own_end", "slice_begin", "slice_end")]


class NewlineFactsC(C.Structure):  # olm_newline_facts_t
    _fields_ = [(n, C.c_uint64) for n in ("newlines", "first", "last")]


class LineOriginC(C.Structure):  # olm_line_origin_t
    _fields_ = [(n, C.c_uint64) for n in ("line", "begin", "next_newline")]


class StreamStateC(C.Structure):  # olm_cuda_stream_state_t
    _fields_ = [("received", C.c_uint64), ("settled", C.c_uint64), ("finished", C.c_int)]


class StoreInfoC(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in ("flags", "smallest", "largest", "stored_patterns", "table_size",
                                         "occupied_buckets", "len1", "len2", "len3", "len4")] + [
        ("store_bytes", C.c_uint64), ("file_bytes", C.c_uint64)] + [
        (n, C.c_uint32) for n in ("gram_keys", "key_buckets", "g4_bits", "class_run", "class_and_mask",
                                  "class_ranges")] + [("class_lo", C.c_uint32 * 2), ("class_hi", C.c_uint32 * 2), ("key_bytes", C.c_uint32),
                                  ("coop", C.c_uint32)]

    def as_dict(self):
        d = {}
        for n, _ in self._fields_:
            v = getattr(self, n)
            d[n] = list(v) if hasattr(v, "__len__") else int(v)
        return d


# Every symbol include/olm_b200.h declares: (name, restype, argtypes)
_vp, _cp, _ci = C.c_void_p, C.c_char_p, C.c_int
_flags7 = [_ci] * 7
ABI = [
    # part 1: the reference's 22 entry points
    ("omega_list_matcher_match", C.POINTER(MatchResultsC), [_vp, _vp, C.c_size_t] + _flags7),
    ("omega_match_results_destroy", None, [C.POINTER(MatchResultsC)]),
    ("omega_list_matcher_create", _vp, [_cp, _ci, _ci, _ci, C.POINTER(PatternStoreStatsC)]),
    ("omega_list_matcher_create_from_buffer", _vp, [_cp, _cp, C.c_uint64, _ci, _ci, _ci, C.POINTER(PatternStoreStatsC)]),
    ("omega_list_matcher_add_stats", _ci, [_vp, C.POINTER(MatchStatsC)]),
    ("omega_list_matcher_destroy", _ci, [_vp]),
    ("omega_list_matcher_emit_header_info", _ci, [_vp, _vp]),
    ("omega_matcher_set_num_threads", _ci, [_vp, _ci]),
    ("omega_matcher_get_num_threads", _ci, [_vp]),
    ("omega_matcher_set_chunk_size", _ci, [_vp, _ci]),
    ("omega_matcher_get_chunk_size", _ci, [_vp]),
    ("omega_list_matcher_compiler_create", _vp, [_cp, _ci, _ci, _ci]),
    ("omega_list_matcher_compiler_add_pattern", _ci, [_vp, _cp, C.c_uint32]),
    ("omega_list_matcher_compiler_get_pattern_store_stats", C.POINTER(PatternStoreStatsC), [_vp]),
    ("omega_list_matcher_compiler_destroy", _ci, [_vp]),
    ("omega_list_matcher_compile_patterns", _ci, [_cp, _cp, C.c_uint64, _ci, _ci, _ci, C.POINTER(PatternStoreStatsC)]),
    ("omega_list_matcher_compile_patterns_filename", _ci, [_cp, _cp, _ci, _ci, _ci, C.POINTER(PatternStoreStatsC)]),
    ("omega_list_matcher_is_compiled", _ci, [_cp]),
    ("omega_matcher_map_file", _vp, [_vp, C.POINTER(C.c_size_t), _ci]),
    ("omega_matcher_map_filename", _vp, [_cp, C.POINTER(C.c_size_t), _ci]),
    ("omega_matcher_unmap_file", _ci, [_vp, C.c_size_t]),
    ("omega_match_version", _cp, []),
    # part 2: B200 extensions
    ("olm_cuda_device_count", _ci, []),
    ("olm_cuda_set_default_device", _ci, [_ci]),
    ("olm_cuda_matcher_device", _ci, [_vp]),
    ("olm_cuda_match_device", _ci, [_vp, _vp, C.c_size_t, _vp] + _flags7 + [C.POINTER(CudaResultsC)]),
    ("olm_cuda_match_shard", _ci, [_vp, _vp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, _vp]
     + [_ci] * 6 + [C.POINTER(CudaResultsC)]),
    ("olm_cuda_match_shard_host", _ci, [_vp, _vp, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, _vp]
     + [_ci] * 6 + [C.POINTER(CudaResultsC)]),
    ("olm_cuda_matcher_create_multi", _vp, [_cp, C.POINTER(_ci), _ci]),
    ("olm_cuda_matcher_device_count", _ci, [_vp]),
    ("olm_shard_plan", _ci, [C.c_uint32, _ci, C.c_uint64, _ci, _ci, C.POINTER(ShardC)]),
    ("olm_cuda_shard_plan", _ci, [_vp, C.c_uint64, _ci, _ci, C.POINTER(ShardC)]),
    ("olm_cuda_comm_unique_id", _ci, [_vp, C.c_size_t]),
    ("olm_cuda_comm_create", _vp, [_vp, _vp, _ci, _ci]),
    ("olm_cuda_comm_destroy", _ci, [_vp]),
    ("olm_cuda_gather_records", _ci, [_vp, _vp, C.c_uint64, _ci, _ci, C.POINTER(CudaResultsC)]),
    ("olm_cuda_no_overlap", C.c_int64, [_vp, _vp, C.c_uint64]),
    ("olm_cuda_sort_records", _ci, [_vp, _vp, C.c_uint64]),
    ("olm_cuda_format_records", _ci, [_vp, _vp, C.c_uint64, _vp, C.c_uint64, C.POINTER(_vp), C.POINTER(C.c_uint64)]),
    ("olm_cuda_last_timing", _ci, [_vp, C.POINTER(CudaTimingC)]),
    ("olm_cuda_set_exact_stats", _ci, [_vp, _ci]),
    ("olm_cuda_set_pattern_ids", _ci, [_vp, _ci]),
    ("olm_pattern_count", C.c_int64, [_vp]),
    ("olm_pattern_bytes", _ci, [_vp, C.c_uint64, C.POINTER(C.c_void_p), C.POINTER(C.c_uint32)]),
    ("olm_cuda_count_patterns", _ci, [_vp, _vp, C.c_size_t] + _flags7 + [_vp, C.POINTER(C.c_uint64)]),
    ("olm_cuda_count_patterns_device", _ci, [_vp, _vp, C.c_size_t] + _flags7 + [_vp, C.POINTER(C.c_uint64)]),
    ("olm_cuda_count_records", _ci, [_vp, _vp, C.c_uint64, _vp]),
    ("olm_cuda_match_lines", _ci, [_vp, _vp, C.c_size_t] + _flags7 + [C.POINTER(C.POINTER(MatchResultsC)), C.POINTER(_vp)]),
    ("olm_cuda_matching_lines", _ci, [_vp, _vp, C.c_size_t] + _flags7
     + [C.POINTER(_vp), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    ("olm_lines_free", None, [_vp]),
    ("olm_cuda_line_positions", _ci, [_vp, _vp, C.c_uint64, _vp, C.c_uint64, C.c_uint64, C.POINTER(LineOriginC), _vp]),
    ("olm_cuda_newline_facts", _ci, [_vp, _vp, C.c_uint64, C.POINTER(NewlineFactsC)]),
    ("olm_cuda_matching_lines_device", _ci, [_vp, _vp, C.c_uint64, C.POINTER(_vp), C.POINTER(C.c_uint64)]),
    ("olm_cuda_stream_open", _vp, [_vp] + _flags7 + [_vp]),
    ("olm_cuda_stream_push", _ci, [_vp, _vp, C.c_size_t, _ci, C.POINTER(C.POINTER(MatchResultsC))]),
    ("olm_cuda_stream_push_device", _ci, [_vp, _vp, C.c_size_t, _ci, C.POINTER(CudaResultsC)]),
    ("olm_cuda_stream_count", _ci, [_vp, _vp, C.c_size_t, _ci, _vp, C.POINTER(C.c_uint64)]),
    ("olm_cuda_stream_state", _ci, [_vp, C.POINTER(StreamStateC)]),
    ("olm_cuda_stream_close", _ci, [_vp]),
    ("olm_cuda_host_alloc", _vp, [C.c_size_t]),
    ("olm_cuda_host_free", None, [_vp]),
    ("olm_store_inspect", _ci, [_cp, C.POINTER(StoreInfoC)]),
]

_lib = None
_lib_path = None


def library_path() -> Path:
    override = os.getenv("OMEGA_MATCH_LIB_PATH")
    return Path(override) if override else DEFAULT_LIB


def load():
    """dlopen the library once and attach the signatures.  Raises if it is not there."""
    global _lib, _lib_path
    if _lib is None:
        path = library_path()
        if not path.is_file():
            raise RuntimeError(
                f"native library not found: {path}. Build it with `make -C omega_match_b200/csrc` "
                "(or __graft_entry__.build()); there is no fallback implementation.")
        lib = C.CDLL(str(path))
        for name, res, args in ABI:
            fn = getattr(lib, name)  # AttributeError here = the .so does not export the ABI
            fn.restype = res
            fn.argtypes = args
        _lib, _lib_path = lib, path
    return _lib
