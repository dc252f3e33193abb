"""Host-side mirror of the reference's Python binding, on top of the B200 library.

Same class and method names, arguments and error behaviour as
bindings/python/omega_match/omega_match.py (Compiler :486-608, Matcher :611-727,
dataclasses :294-320), so code and tests written for the reference read the same here.
The reference binding itself also works unchanged: point OMEGA_MATCH_LIB_PATH at
omega_match_b200/lib/libomega_match.so (see INTEGRATION.md).

Additions (not in the reference): `Matcher.match_arrays` (numpy result without per-match
Python objects), `Matcher.match_device` / `match_shard` (device-resident haystack and
results), `Matcher.last_timing`, pattern ids (`Matcher.match_ids`, `set_pattern_ids`,
`pattern_count`, `pattern`), pattern counts (`Matcher.pattern_counts`, `pattern_counts_device`,
`count_records_device`), lines (`Matcher.match_lines`, `matching_lines`, `line_positions_device`,
`newline_facts_device`, `matching_lines_device`).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional

import numpy as np

from . import _lib
from ._lib import (CudaResultsC, CudaTimingC, MatchStatsC, PatternStoreStatsC)

# (offset, len) pairs as tests and benches consume them
MATCH_DTYPE = np.dtype([("offset", "<u8"), ("len", "<u4"), ("_pad", "<u4")])
# match_ids(): the same 16 bytes, the pad holding the pattern id (include/olm_b200.h)
MATCH_IDS_DTYPE = np.dtype([("offset", "<u8"), ("len", "<u4"), ("pattern_id", "<u4")])
# match_lines(): a record with the line it lies on (include/olm_b200.h "lines"); pattern_id is there
# only while pattern ids are on
LINE_MATCH_DTYPE = np.dtype([("offset", "<u8"), ("len", "<u4"), ("line", "<u8"), ("line_begin", "<u8"),
                             ("line_end", "<u8")])
LINE_MATCH_IDS_DTYPE = np.dtype([("offset", "<u8"), ("len", "<u4"), ("pattern_id", "<u4"), ("line", "<u8"),
                                 ("line_begin", "<u8"), ("line_end", "<u8")])
# olm_line_pos_t (per record) and olm_line_t (per matching line)
LINE_POS_DTYPE = np.dtype([("line", "<u8"), ("begin", "<u8"), ("end", "<u8")])
LINE_DTYPE = np.dtype([("line", "<u8"), ("begin", "<u8"), ("end", "<u8"), ("records", "<u8")])
# omega_match_result_t as the library writes it (24 bytes)
RECORD_DTYPE = np.dtype([("offset", "<u8"), ("len", "<u4"), ("_pad", "<u4"), ("match", "<u8")])

FLAG_NAMES = ("no_overlap", "longest_only", "word_boundary", "word_prefix", "word_suffix",
              "line_start", "line_end")


@dataclass
class PatternStoreStats:
    total_input_bytes: int
    total_stored_bytes: int
    stored_pattern_count: int
    short_pattern_count: int
    duplicate_patterns: int
    smallest_pattern_length: int
    largest_pattern_length: int


@dataclass
class MatchStats:
    total_hits: int
    total_misses: int
    total_filtered: int
    total_attempts: int
    total_comparisons: int


@dataclass
class MatchResult:
    offset: int
    match: bytes

    @property
    def length(self) -> int:
        return len(self.match)


def get_version() -> str:
    v = _lib.load().omega_match_version()
    if not v:
        raise RuntimeError("Failed to get native library version")
    return v.decode("utf-8")


def get_library_info() -> Dict[str, str]:
    _lib.load()
    return {"path": str(_lib._lib_path), "variant": "linux-x64-b200-sm_100a", "optimization": "CUDA",
            "platform": "linux-x86_64"}


def _stats_from(c) -> PatternStoreStats:
    return PatternStoreStats(**{k: int(getattr(c, k)) for k in PatternStoreStats.__annotations__})


def _flag_ints(kw) -> List[int]:
    bad = set(kw) - set(FLAG_NAMES)
    if bad:
        raise TypeError(f"unexpected match options: {sorted(bad)}")
    return [int(bool(kw.get(n, False))) for n in FLAG_NAMES]


def _host_haystack(haystack):
    """(object that keeps the bytes alive, address, size) of a bytes-like or numpy haystack."""
    if isinstance(haystack, np.ndarray):
        hay = np.ascontiguousarray(haystack, dtype=np.uint8)
        return hay, hay.ctypes.data, hay.size
    hay = (C.c_char * len(haystack)).from_buffer_copy(haystack) if len(haystack) else None
    return hay, (C.addressof(hay) if hay is not None else None), len(haystack)


class Compiler:
    def __init__(self, compiled_file: str, case_insensitive: bool = False, ignore_punctuation: bool = False,
                 elide_whitespace: bool = False) -> None:
        self._lib = _lib.load()
        self._compiler = self._lib.omega_list_matcher_compiler_create(
            compiled_file.encode("utf-8"), int(case_insensitive), int(ignore_punctuation), int(elide_whitespace))
        if not self._compiler:
            raise RuntimeError("Failed to create compiler")

    def __enter__(self):
        return self

    def __exit__(self, *_exc) -> None:
        self.destroy()

    def __del__(self):
        self.destroy()

    def add_pattern(self, pattern: bytes) -> None:
        if not isinstance(pattern, (bytes, bytearray)):
            raise TypeError("Pattern must be bytes")
        if self._lib.omega_list_matcher_compiler_add_pattern(self._compiler, bytes(pattern), len(pattern)) != 0:
            raise ValueError("Failed to add pattern")

    def get_stats(self) -> PatternStoreStats:
        p = self._lib.omega_list_matcher_compiler_get_pattern_store_stats(self._compiler)
        if not p:
            raise RuntimeError("Failed to retrieve stats")
        return _stats_from(p.contents)

    def destroy(self) -> None:
        if getattr(self, "_compiler", None):
            self._lib.omega_list_matcher_compiler_destroy(self._compiler)
            self._compiler = None

    @staticmethod
    def compile_from_filename(compiled_file: str, patterns_file: str, case_insensitive: bool = False,
                              ignore_punctuation: bool = False, elide_whitespace: bool = False) -> PatternStoreStats:
        st = PatternStoreStatsC()
        if _lib.load().omega_list_matcher_compile_patterns_filename(
                compiled_file.encode("utf-8"), patterns_file.encode("utf-8"), int(case_insensitive),
                int(ignore_punctuation), int(elide_whitespace), C.byref(st)) != 0:
            raise RuntimeError("Compilation failed")
        return _stats_from(st)

    @staticmethod
    def compile_from_buffer(compiled_file: str, patterns_buf: bytes, case_insensitive: bool = False,
                            ignore_punctuation: bool = False, elide_whitespace: bool = False) -> PatternStoreStats:
        st = PatternStoreStatsC()
        if _lib.load().omega_list_matcher_compile_patterns(
                compiled_file.encode("utf-8"), bytes(patterns_buf), len(patterns_buf), int(case_insensitive),
                int(ignore_punctuation), int(elide_whitespace), C.byref(st)) != 0:
            raise RuntimeError("Compilation failed")
        return _stats_from(st)


class Matcher:
    _matcher = None
    _pattern_ids = False

    def __init__(self, compiled_or_patterns_file: str, case_insensitive: bool = False,
                 ignore_punctuation: bool = False, elide_whitespace: bool = False,
                 device: Optional[int] = None, devices: Optional[List[int]] = None) -> None:
        """`devices` (B200 extension): several GPUs in this process -- match() shards every haystack by
        byte range over them (include/olm_b200.h olm_cuda_matcher_create_multi; compiled stores only)."""
        self._lib = _lib.load()
        self._comm = None
        if device is not None:
            self._lib.olm_cuda_set_default_device(int(device))
        st = PatternStoreStatsC()
        if devices is not None:
            arr = (C.c_int * len(devices))(*devices)
            m = self._lib.olm_cuda_matcher_create_multi(compiled_or_patterns_file.encode("utf-8"), arr, len(devices))
        else:
            m = self._lib.omega_list_matcher_create(compiled_or_patterns_file.encode("utf-8"), int(case_insensitive),
                                                    int(ignore_punctuation), int(elide_whitespace), C.byref(st))
        if not m:
            raise RuntimeError("Failed to create matcher")
        self._matcher = m
        self._match_stats = MatchStatsC()
        if self._lib.omega_list_matcher_add_stats(self._matcher, C.byref(self._match_stats)) != 0:
            raise RuntimeError("Failed to attach stats to matcher")

    def __enter__(self):
        return self

    def __exit__(self, *_exc) -> None:
        self.destroy()

    def __del__(self):
        self.destroy()

    # -- reference API ---------------------------------------------------------------------
    def match(self, haystack: bytes, no_overlap: bool = False, longest_only: bool = False,
              word_boundary: bool = False, word_prefix: bool = False, word_suffix: bool = False,
              line_start: bool = False, line_end: bool = False) -> List[MatchResult]:
        if not isinstance(haystack, (bytes, bytearray)):
            raise TypeError("haystack must be bytes or bytearray")
        rec = self._match_records(haystack, no_overlap=no_overlap, longest_only=longest_only,
                                  word_boundary=word_boundary, word_prefix=word_prefix,
                                  word_suffix=word_suffix, line_start=line_start, line_end=line_end)
        mv = memoryview(haystack)
        return [MatchResult(offset=int(o), match=bytes(mv[int(o):int(o) + int(n)]))
                for o, n in zip(rec["offset"], rec["len"])]

    def get_match_stats(self) -> MatchStats:
        return MatchStats(**{k: int(getattr(self._match_stats, k)) for k in MatchStats.__annotations__})

    def set_exact_stats(self, on: bool = True) -> None:
        """B200 extension: make get_match_stats() equal the reference's counters exactly (one extra
        kernel per call, include/olm_b200.h olm_cuda_set_exact_stats)."""
        if self._lib.olm_cuda_set_exact_stats(self._matcher, int(bool(on))) != 0:
            raise RuntimeError("Failed to switch exact statistics")

    def reset_match_stats(self) -> None:
        for k in MatchStats.__annotations__:
            setattr(self._match_stats, k, 0)

    def set_threads(self, threads: int) -> None:
        if self._lib.omega_matcher_set_num_threads(self._matcher, threads) != 0:
            raise ValueError(f"Invalid thread count: {threads}")

    def get_threads(self) -> int:
        return self._lib.omega_matcher_get_num_threads(self._matcher)

    def set_chunk_size(self, chunk: int) -> None:
        if self._lib.omega_matcher_set_chunk_size(self._matcher, chunk) != 0:
            raise ValueError(f"Invalid chunk size: {chunk}")

    def get_chunk_size(self) -> int:
        return self._lib.omega_matcher_get_chunk_size(self._matcher)

    def destroy(self) -> None:
        if getattr(self, "_comm", None):
            self._lib.olm_cuda_comm_destroy(self._comm)
            self._comm = None
        if getattr(self, "_matcher", None):
            self._lib.omega_list_matcher_destroy(self._matcher)
            self._matcher = None

    # -- additions -------------------------------------------------------------------------
    def _match_records(self, haystack, **kw) -> np.ndarray:
        """omega_list_matcher_match() on a host buffer -> copy of the 24-byte records."""
        hay, ptr, n = _host_haystack(haystack)
        res = self._lib.omega_list_matcher_match(self._matcher, ptr, n, *_flag_ints(kw))
        if not res:
            raise RuntimeError("omega_list_matcher_match failed (CUDA error, see stderr)")
        cnt = res.contents.count
        out = np.zeros(cnt, dtype=RECORD_DTYPE)
        if cnt:
            C.memmove(out.ctypes.data, res.contents.matches, cnt * RECORD_DTYPE.itemsize)
            if not (out["match"] == out["offset"] + np.uint64(ptr)).all():
                raise RuntimeError("result.match does not alias haystack + offset")
        self._lib.omega_match_results_destroy(res)
        return out

    def match_arrays(self, haystack, **kw) -> np.ndarray:
        """Like match(), but returns a structured array (offset, len) in result order."""
        rec = self._match_records(haystack, **kw)
        out = np.zeros(rec.size, dtype=MATCH_DTYPE)
        out["offset"] = rec["offset"]
        out["len"] = rec["len"]
        return out

    # -- pattern ids (include/olm_b200.h) ------------------------------------------------------
    def set_pattern_ids(self, on: bool = True) -> None:
        """While on, every match call writes the id of each record's pattern into the record's pad
        word (RECORD_DTYPE `_pad`): match_device / match_shard / match_shard_host records carry ids.
        Switching on the first time builds the catalogue and uploads its lookup table."""
        if self._lib.olm_cuda_set_pattern_ids(self._matcher, int(bool(on))) != 0:
            raise RuntimeError("olm_cuda_set_pattern_ids failed (malformed store? see stderr)")
        self._pattern_ids = bool(on)

    @property
    def pattern_count(self) -> int:
        """Number of distinct normalised patterns of the store: ids are 0 .. pattern_count - 1."""
        n = self._lib.olm_pattern_count(self._matcher)
        if n < 0:
            raise RuntimeError("olm_pattern_count failed (malformed store? see stderr)")
        return int(n)

    def pattern(self, pattern_id: int) -> bytes:
        """The stored (normalised) bytes of a pattern id."""
        p, n = C.c_void_p(), C.c_uint32()
        if pattern_id < 0 or self._lib.olm_pattern_bytes(self._matcher, pattern_id, C.byref(p), C.byref(n)) != 0:
            raise IndexError(f"pattern id {pattern_id} out of range")
        return C.string_at(p.value, n.value) if n.value else b""

    def match_ids(self, haystack, **kw) -> np.ndarray:
        """Like match_arrays(), with the id of each match's pattern: MATCH_IDS_DTYPE (offset, len,
        pattern_id) in result order.  Ids are switched on for this call only."""
        was = self._pattern_ids
        self.set_pattern_ids(True)
        try:
            rec = self._match_records(haystack, **kw)
        finally:
            if not was:
                self.set_pattern_ids(False)
        out = np.zeros(rec.size, dtype=MATCH_IDS_DTYPE)
        out["offset"] = rec["offset"]
        out["len"] = rec["len"]
        out["pattern_id"] = rec["_pad"]
        return out

    # -- pattern counts (include/olm_b200.h) ---------------------------------------------------
    def pattern_counts(self, haystack, **kw) -> np.ndarray:
        """How often each pattern occurs in a host haystack: uint64 array of pattern_count entries,
        counts[id] = the records of pattern id that match() with the same options would return.
        Only the counts leave the GPU; the ids setting is left as it is."""
        hay, ptr, n = _host_haystack(haystack)
        counts = np.zeros(self.pattern_count, dtype=np.uint64)
        total = C.c_uint64()
        if self._lib.olm_cuda_count_patterns(self._matcher, ptr, n, *_flag_ints(kw), counts.ctypes.data,
                                             C.byref(total)) != 0:
            raise RuntimeError("olm_cuda_count_patterns failed (see stderr)")
        return counts

    def pattern_counts_device(self, dev_ptr: int, size: int, counts_ptr: int, **kw) -> int:
        """Device haystack (as match_device) -> counts ADDED into pattern_count uint64 words of device
        memory at counts_ptr; returns the number of records counted."""
        total = C.c_uint64()
        if self._lib.olm_cuda_count_patterns_device(self._matcher, dev_ptr, size, *_flag_ints(kw), counts_ptr,
                                                    C.byref(total)) != 0:
            raise RuntimeError("olm_cuda_count_patterns_device failed (see stderr)")
        return int(total.value)

    def count_records_device(self, records_ptr: int, count: int, counts_ptr: int) -> None:
        """Device records whose pad words hold ids (made with set_pattern_ids(True)) -> counts ADDED
        into pattern_count uint64 words of device memory at counts_ptr."""
        if self._lib.olm_cuda_count_records(self._matcher, records_ptr, count, counts_ptr) != 0:
            raise RuntimeError("olm_cuda_count_records failed (id out of range? see stderr)")

    # -- lines (include/olm_b200.h "lines") ----------------------------------------------------
    def match_lines(self, haystack, **kw) -> np.ndarray:
        """Like match_arrays(), with the line of every match: LINE_MATCH_DTYPE (offset, len, line,
        line_begin, line_end) in result order; with pattern ids on, LINE_MATCH_IDS_DTYPE, which adds
        pattern_id.  line is 0-based (grep -n prints line + 1); the line's bytes are
        haystack[line_begin:line_end], without its '\n'."""
        hay, ptr, n = _host_haystack(haystack)
        res, pos = C.POINTER(_lib.MatchResultsC)(), C.c_void_p()
        if self._lib.olm_cuda_match_lines(self._matcher, ptr, n, *_flag_ints(kw), C.byref(res), C.byref(pos)) != 0:
            raise RuntimeError("olm_cuda_match_lines failed (see stderr)")
        try:
            cnt = res.contents.count
            rec = np.zeros(cnt, dtype=RECORD_DTYPE)
            lp = np.zeros(cnt, dtype=LINE_POS_DTYPE)
            if cnt:
                C.memmove(rec.ctypes.data, res.contents.matches, cnt * RECORD_DTYPE.itemsize)
                C.memmove(lp.ctypes.data, pos.value, cnt * LINE_POS_DTYPE.itemsize)
        finally:
            self._lib.omega_match_results_destroy(res)
            self._lib.olm_lines_free(pos)
        out = np.zeros(cnt, dtype=LINE_MATCH_IDS_DTYPE if self._pattern_ids else LINE_MATCH_DTYPE)
        out["offset"] = rec["offset"]
        out["len"] = rec["len"]
        if self._pattern_ids:
            out["pattern_id"] = rec["_pad"]
        out["line"], out["line_begin"], out["line_end"] = lp["line"], lp["begin"], lp["end"]
        return out

    def matching_lines(self, haystack, **kw) -> np.ndarray:
        """The distinct lines that hold a match, in order: LINE_DTYPE (line, begin, end, records), records
        = the matches match() with the same options returns on that line.  len() is grep -c.  Only the
        lines leave the GPU."""
        hay, ptr, n = _host_haystack(haystack)
        lines, n_lines, total = C.c_void_p(), C.c_uint64(), C.c_uint64()
        if self._lib.olm_cuda_matching_lines(self._matcher, ptr, n, *_flag_ints(kw), C.byref(lines), C.byref(n_lines),
                                             C.byref(total)) != 0:
            raise RuntimeError("olm_cuda_matching_lines failed (see stderr)")
        out = np.zeros(n_lines.value, dtype=LINE_DTYPE)
        if n_lines.value:
            C.memmove(out.ctypes.data, lines.value, n_lines.value * LINE_DTYPE.itemsize)
        self._lib.olm_lines_free(lines)
        return out

    def line_positions_device(self, records_ptr: int, count: int, bytes_ptr: int, bytes_begin: int, bytes_len: int,
                              positions_ptr: int, origin=None) -> None:
        """Device records (offsets in [bytes_begin, bytes_begin + bytes_len)) -> one olm_line_pos_t (3
        uint64: line, begin, end) per record at positions_ptr.  bytes_ptr holds those bytes; `origin` =
        (line, begin, next_newline) of what lies outside them (sharding.line_origins), None for a whole
        haystack (bytes_begin 0)."""
        o = C.byref(_lib.LineOriginC(*origin)) if origin is not None else None
        if self._lib.olm_cuda_line_positions(self._matcher, records_ptr, count, bytes_ptr, bytes_begin, bytes_len, o,
                                             positions_ptr) != 0:
            raise RuntimeError("olm_cuda_line_positions failed (see stderr)")

    def newline_facts_device(self, bytes_ptr: int, size: int):
        """(newlines, first, last) of the device bytes [0, size), positions relative to them; first and
        last are None without a '\n'."""
        f = _lib.NewlineFactsC()
        if self._lib.olm_cuda_newline_facts(self._matcher, bytes_ptr, size, C.byref(f)) != 0:
            raise RuntimeError("olm_cuda_newline_facts failed (see stderr)")
        none = (1 << 64) - 1
        return (int(f.newlines), None if f.first == none else int(f.first), None if f.last == none else int(f.last))

    def matching_lines_device(self, positions_ptr: int, count: int):
        """Device positions (record order) -> (n_lines, device pointer of n_lines olm_line_t: 4 uint64
        line, begin, end, records), valid until the next call."""
        p, n = C.c_void_p(), C.c_uint64()
        if self._lib.olm_cuda_matching_lines_device(self._matcher, positions_ptr, count, C.byref(p), C.byref(n)) != 0:
            raise RuntimeError("olm_cuda_matching_lines_device failed (see stderr)")
        return int(n.value), int(p.value or 0)

    def stream(self, match_ptr_base: int = 0, **kw) -> "MatchStream":
        """A stream over one haystack that arrives in pieces (include/olm_b200.h "Streams"): the records
        of all pushes, in push order, are those of one match over the concatenation, with offsets
        counted from the stream's first byte."""
        return MatchStream(self, match_ptr_base, **kw)

    def match_device(self, dev_ptr: int, size: int, match_ptr_base: Optional[int] = None, **kw):
        """Haystack already in HBM (16-byte aligned device pointer).  Returns (count, device
        pointer of the 24-byte records); the records stay valid until the next call.  With
        set_pattern_ids(True) their pad words hold the pattern ids."""
        res = CudaResultsC()
        base = dev_ptr if match_ptr_base is None else match_ptr_base
        if self._lib.olm_cuda_match_device(self._matcher, dev_ptr, size, base, *_flag_ints(kw), C.byref(res)) != 0:
            raise RuntimeError("olm_cuda_match_device failed (see stderr)")
        return int(res.count), int(res.records or 0)

    def match_shard(self, dev_ptr: int, slice_begin: int, slice_len: int, own_begin: int, own_end: int,
                    global_size: int, match_ptr_base: int = 0, **kw):
        """One byte-range shard of a larger haystack (SURVEY 8e); no_overlap is not applied.  With
        set_pattern_ids(True) the records' pad words hold the pattern ids."""
        if kw.get("no_overlap"):
            raise ValueError("no_overlap crosses shards: apply Matcher.no_overlap_device on the gathered records")
        f = _flag_ints(kw)[1:]
        res = CudaResultsC()
        if self._lib.olm_cuda_match_shard(self._matcher, dev_ptr, slice_begin, slice_len, own_begin, own_end,
                                          global_size, match_ptr_base, *f, C.byref(res)) != 0:
            raise RuntimeError("olm_cuda_match_shard failed (see stderr)")
        return int(res.count), int(res.records or 0)

    def match_shard_host(self, host_ptr: int, slice_begin: int, slice_len: int, own_begin: int, own_end: int,
                         global_size: int, match_ptr_base: int = 0, **kw):
        """match_shard() for a slice in host memory: segmented H2D overlapped with the scan; the
        records stay on the device (include/olm_b200.h olm_cuda_match_shard_host).  With
        set_pattern_ids(True) their pad words hold the pattern ids."""
        if kw.get("no_overlap"):
            raise ValueError("no_overlap crosses shards: apply Matcher.no_overlap_device on the gathered records")
        f = _flag_ints(kw)[1:]
        res = CudaResultsC()
        if self._lib.olm_cuda_match_shard_host(self._matcher, host_ptr, slice_begin, slice_len, own_begin, own_end,
                                               global_size, match_ptr_base, *f, C.byref(res)) != 0:
            raise RuntimeError("olm_cuda_match_shard_host failed (see stderr)")
        return int(res.count), int(res.records or 0)

    # -- one process per GPU: the library's own NCCL gather (include/olm_b200.h) ---------------
    @staticmethod
    def comm_unique_id() -> bytes:
        """Rank 0: the 128-byte id every rank of the job passes to comm_init()."""
        buf = C.create_string_buffer(128)
        if _lib.load().olm_cuda_comm_unique_id(buf, 128) != 0:
            raise RuntimeError("olm_cuda_comm_unique_id failed (NCCL not loadable?)")
        return buf.raw

    def comm_init(self, unique_id: bytes, rank: int, world: int) -> None:
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._comm = self._lib.olm_cuda_comm_create(self._matcher, buf, rank, world)
        if not self._comm:
            raise RuntimeError("olm_cuda_comm_create failed")

    def gather_records(self, records_ptr: int, count: int, root: int = 0, no_overlap: bool = False):
        """Collective: the ranks' sorted records -> (count, device pointer) of the whole on `root`
        ((0, 0) on the other ranks)."""
        res = CudaResultsC()
        if self._lib.olm_cuda_gather_records(self._comm, records_ptr, count, root, int(no_overlap), C.byref(res)) != 0:
            raise RuntimeError("olm_cuda_gather_records failed (see stderr)")
        return int(res.count), int(res.records or 0)

    def shard_plan(self, global_size: int, world: int, rank: int):
        sh = _lib.ShardC()
        if self._lib.olm_cuda_shard_plan(self._matcher, global_size, world, rank, C.byref(sh)) != 0:
            raise RuntimeError("olm_cuda_shard_plan failed")
        return sh.own_begin, sh.own_end, sh.slice_begin, sh.slice_end

    @property
    def device_count(self) -> int:
        return self._lib.olm_cuda_matcher_device_count(self._matcher)

    def no_overlap_device(self, records_ptr: int, count: int) -> int:
        n = self._lib.olm_cuda_no_overlap(self._matcher, records_ptr, count)
        if n < 0:
            raise RuntimeError("olm_cuda_no_overlap failed")
        return int(n)

    def format_records_device(self, records_ptr: int, count: int, haystack_ptr: int, offset0: int = 0):
        """The CLI's listing ("offset:bytes\\n" per record, main.c:89-133) formatted on the GPU ->
        (device pointer of the text, its length)."""
        text, n = C.c_void_p(), C.c_uint64()
        if self._lib.olm_cuda_format_records(self._matcher, records_ptr, count, haystack_ptr, offset0,
                                             C.byref(text), C.byref(n)) != 0:
            raise RuntimeError("olm_cuda_format_records failed")
        return int(text.value or 0), int(n.value)

    def sort_records_device(self, records_ptr: int, count: int) -> None:
        if self._lib.olm_cuda_sort_records(self._matcher, records_ptr, count) != 0:
            raise RuntimeError("olm_cuda_sort_records failed")

    def last_timing(self) -> dict:
        t = CudaTimingC()
        if self._lib.olm_cuda_last_timing(self._matcher, C.byref(t)) != 0:
            raise RuntimeError("olm_cuda_last_timing failed")
        return t.as_dict()

    @property
    def device(self) -> int:
        return self._lib.olm_cuda_matcher_device(self._matcher)


class MatchStream:
    """Consecutive pieces of one haystack pushed into a Matcher (Matcher.stream()).  A context manager;
    it keeps its Matcher alive and must be closed before the Matcher is destroyed."""

    def __init__(self, matcher: Matcher, match_ptr_base: int = 0, **kw) -> None:
        self._matcher = matcher
        self._lib = matcher._lib
        self._s = self._lib.olm_cuda_stream_open(matcher._matcher, *_flag_ints(kw), match_ptr_base)
        if not self._s:
            raise RuntimeError("olm_cuda_stream_open failed")

    def __enter__(self):
        return self

    def __exit__(self, *_exc) -> None:
        self.close()

    def __del__(self):
        self.close()

    def close(self) -> None:
        if getattr(self, "_s", None):
            self._lib.olm_cuda_stream_close(self._s)
            self._s = None

    def _state(self):
        st = _lib.StreamStateC()
        if not self._s or self._lib.olm_cuda_stream_state(self._s, C.byref(st)) != 0:
            raise RuntimeError("the stream is closed")
        return st

    @property
    def received(self) -> int:
        return int(self._state().received)

    @property
    def settled(self) -> int:
        return int(self._state().settled)

    def push(self, data, last: bool = False) -> np.ndarray:
        """Host bytes (bytes, memoryview or uint8 array) -> the records this push settled: MATCH_DTYPE,
        or MATCH_IDS_DTYPE while pattern ids are on."""
        hay, ptr, n = _host_haystack(data)
        res = C.POINTER(_lib.MatchResultsC)()
        if not self._s or self._lib.olm_cuda_stream_push(self._s, ptr, n, int(bool(last)), C.byref(res)) != 0:
            raise RuntimeError("olm_cuda_stream_push failed (see stderr)")
        cnt = res.contents.count
        rec = np.zeros(cnt, dtype=RECORD_DTYPE)
        if cnt:
            C.memmove(rec.ctypes.data, res.contents.matches, cnt * RECORD_DTYPE.itemsize)
        self._lib.omega_match_results_destroy(res)
        ids = self._matcher._pattern_ids
        out = np.zeros(cnt, dtype=MATCH_IDS_DTYPE if ids else MATCH_DTYPE)
        out["offset"] = rec["offset"]
        out["len"] = rec["len"]
        if ids:
            out["pattern_id"] = rec["_pad"]
        return out

    def push_device(self, dev_ptr: int, size: int, last: bool = False):
        """Device bytes (the contract of Matcher.match_device) -> (device pointer of the settled
        24-byte records, their count); valid until the next call on the matcher."""
        res = CudaResultsC()
        if not self._s or self._lib.olm_cuda_stream_push_device(self._s, dev_ptr, size, int(bool(last)),
                                                                C.byref(res)) != 0:
            raise RuntimeError("olm_cuda_stream_push_device failed (see stderr)")
        return int(res.records or 0), int(res.count)

    def count(self, data, counts: np.ndarray, last: bool = False) -> int:
        """Host bytes -> counts[id] += the settled records of pattern id (counts: uint64 array of
        pattern_count entries); returns their number."""
        if not (isinstance(counts, np.ndarray) and counts.dtype == np.uint64 and counts.flags.c_contiguous
                and counts.size >= self._matcher.pattern_count):
            raise ValueError("counts must be a contiguous uint64 array of pattern_count entries")
        hay, ptr, n = _host_haystack(data)
        total = C.c_uint64()
        if not self._s or self._lib.olm_cuda_stream_count(self._s, ptr, n, int(bool(last)), counts.ctypes.data,
                                                          C.byref(total)) != 0:
            raise RuntimeError("olm_cuda_stream_count failed (see stderr)")
        return int(total.value)
