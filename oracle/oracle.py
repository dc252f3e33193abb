"""oracle/oracle.py -- ctypes front ends for the CPU checkers.  TEST INFRASTRUCTURE ONLY.

Two checkers live here; neither is ever imported by the shipped package
(`omega_match_b200`), only by tests/, __graft_entry__.smoke() and bench.py's CPU legs:

* `Oracle`  -- oracle/olm_oracle.c, the plain-C restatement (travels as source, is compiled
               by `make -C oracle port` / __graft_entry__.build()).
* `RefLib`  -- oracle/_ref/libomega_match_ref.so, the UNMODIFIED reference compiled from
               /root/reference by `make -C oracle ref` (prebuilt binary travels to the GPU
               box; nothing here reads /root/reference at run time).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
PORT_SO = HERE / "_build" / "libolm_oracle.so"
REF_SO = HERE / "_ref" / "libomega_match_ref.so"

MATCH_DTYPE = np.dtype([("offset", "<u8"), ("len", "<u4"), ("_pad", "<u4")])
FLAG_NAMES = ("no_overlap", "longest_only", "word_boundary", "word_prefix", "word_suffix",
              "line_start", "line_end")


def build_port(force: bool = False) -> Path:
    src = HERE / "olm_oracle.c"
    if force or not PORT_SO.exists() or PORT_SO.stat().st_mtime < src.stat().st_mtime:
        subprocess.check_call(["make", "-C", str(HERE), "port"], stdout=subprocess.DEVNULL)
    return PORT_SO


def ref_available() -> bool:
    return REF_SO.exists()


class _Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("hits", "misses", "filtered", "attempts", "comparisons")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


def _flags(kw):
    bad = set(kw) - set(FLAG_NAMES)
    if bad:
        raise TypeError(f"unknown match flags {bad}")
    return [int(bool(kw.get(n, False))) for n in FLAG_NAMES]


class Oracle:
    """The C restatement (oracle/olm_oracle.c)."""

    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            L = C.CDLL(str(build_port()))
            L.olm_oracle_from_patterns.restype = C.c_void_p
            L.olm_oracle_from_patterns.argtypes = [C.c_char_p, C.c_size_t, C.c_int, C.c_int, C.c_int]
            L.olm_oracle_from_olm.restype = C.c_void_p
            L.olm_oracle_from_olm.argtypes = [C.c_char_p, C.c_size_t]
            L.olm_oracle_free.argtypes = [C.c_void_p]
            for fn in ("flags", "smallest", "largest", "long_count", "table_size"):
                f = getattr(L, "olm_oracle_" + fn)
                f.restype = C.c_uint32
                f.argtypes = [C.c_void_p]
            L.olm_oracle_short_count.restype = C.c_uint32
            L.olm_oracle_short_count.argtypes = [C.c_void_p, C.c_int]
            L.olm_oracle_pattern_digest.restype = C.c_uint64
            L.olm_oracle_pattern_digest.argtypes = [C.c_void_p]
            L.olm_oracle_match.restype = C.c_int64
            L.olm_oracle_match.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t] + [C.c_int] * 7 + [
                C.c_uint8, C.POINTER(C.c_void_p), C.POINTER(_Stats)]
            L.olm_oracle_free_matches.argtypes = [C.c_void_p]
            L.olm_oracle_transform.restype = C.c_uint32
            L.olm_oracle_transform.argtypes = [C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_uint32,
                                               C.c_void_p, C.c_void_p]
            L.olm_oracle_stream_digest.restype = C.c_uint64
            L.olm_oracle_stream_digest.argtypes = [C.c_void_p, C.c_size_t]
            cls._lib = L
        return cls._lib

    def __init__(self, handle):
        if not handle:
            raise ValueError("oracle: could not build pattern set")
        self._h = handle
        self.stats = _Stats()

    @classmethod
    def from_patterns(cls, patterns, case_insensitive=False, ignore_punctuation=False,
                      elide_whitespace=False):
        buf = patterns if isinstance(patterns, (bytes, bytearray)) else b"\n".join(patterns)
        buf = bytes(buf)
        return cls(cls.lib().olm_oracle_from_patterns(buf, len(buf), int(case_insensitive),
                                                      int(ignore_punctuation), int(elide_whitespace)))

    @classmethod
    def from_olm(cls, path_or_bytes):
        data = path_or_bytes if isinstance(path_or_bytes, (bytes, bytearray)) else Path(path_or_bytes).read_bytes()
        return cls(cls.lib().olm_oracle_from_olm(bytes(data), len(data)))

    def __del__(self):
        if getattr(self, "_h", None):
            self.lib().olm_oracle_free(self._h)
            self._h = None

    def info(self):
        L = self.lib()
        return dict(flags=L.olm_oracle_flags(self._h), smallest=L.olm_oracle_smallest(self._h),
                    largest=L.olm_oracle_largest(self._h), long=L.olm_oracle_long_count(self._h),
                    table_size=L.olm_oracle_table_size(self._h),
                    short=[L.olm_oracle_short_count(self._h, i) for i in (1, 2, 3, 4)],
                    digest=L.olm_oracle_pattern_digest(self._h))

    def match(self, haystack, tail_byte=0, **kw) -> np.ndarray:
        """-> structured array (offset,len) in the reference's final order."""
        L = self.lib()
        hay = np.frombuffer(haystack, dtype=np.uint8) if not isinstance(haystack, np.ndarray) else haystack
        hay = np.ascontiguousarray(hay, dtype=np.uint8)
        out = C.c_void_p()
        n = L.olm_oracle_match(self._h, hay.ctypes.data, hay.size, *_flags(kw), tail_byte,
                               C.byref(out), C.byref(self.stats))
        if n == 0:
            if out.value:
                L.olm_oracle_free_matches(out)
            return np.zeros(0, dtype=MATCH_DTYPE)
        arr = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_uint8)), shape=(n * 16,)).view(MATCH_DTYPE).copy()
        L.olm_oracle_free_matches(out)
        return arr

    @classmethod
    def transform(cls, src: bytes, case_insensitive=False, ignore_punctuation=False, elide_whitespace=False):
        out = np.zeros(max(len(src), 1), dtype=np.uint8)
        mp = np.zeros(max(len(src), 1), dtype=np.uint32)
        n = cls.lib().olm_oracle_transform(int(case_insensitive), int(ignore_punctuation), int(elide_whitespace),
                                           bytes(src), len(src), out.ctypes.data, mp.ctypes.data)
        return out[:n].tobytes(), mp[:n].copy()

    @classmethod
    def stream_digest(cls, matches: np.ndarray) -> int:
        m = np.ascontiguousarray(matches, dtype=MATCH_DTYPE)
        return int(cls.lib().olm_oracle_stream_digest(m.ctypes.data, m.size))


# ---------------------------------------------------------------------------------------------
# The unmodified reference library, through its own C API (omega/list_matcher.h).


class _RefResult(C.Structure):
    _fields_ = [("offset", C.c_size_t), ("len", C.c_uint32), ("match", C.c_void_p)]


class _RefResults(C.Structure):
    _fields_ = [("count", C.c_size_t), ("matches", C.POINTER(_RefResult))]


class PatternStoreStats(C.Structure):
    _fields_ = [("total_input_bytes", C.c_uint64), ("total_stored_bytes", C.c_uint64),
                ("stored_pattern_count", C.c_uint32), ("short_pattern_count", C.c_uint32),
                ("duplicate_patterns", C.c_uint32), ("smallest_pattern_length", C.c_uint32),
                ("largest_pattern_length", C.c_uint32)]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


REF_RESULT_DTYPE = np.dtype([("offset", "<u8"), ("len", "<u4"), ("_pad", "<u4"), ("match", "<u8")])


def bind_list_matcher_api(L):
    """Attach ctypes signatures of omega/list_matcher.h to a loaded library."""
    vp, cp, ci = C.c_void_p, C.c_char_p, C.c_int
    L.omega_list_matcher_compile_patterns.restype = ci
    L.omega_list_matcher_compile_patterns.argtypes = [cp, cp, C.c_uint64, ci, ci, ci, C.POINTER(PatternStoreStats)]
    L.omega_list_matcher_compile_patterns_filename.restype = ci
    L.omega_list_matcher_compile_patterns_filename.argtypes = [cp, cp, ci, ci, ci, C.POINTER(PatternStoreStats)]
    L.omega_list_matcher_create.restype = vp
    L.omega_list_matcher_create.argtypes = [cp, ci, ci, ci, C.POINTER(PatternStoreStats)]
    L.omega_list_matcher_destroy.restype = ci
    L.omega_list_matcher_destroy.argtypes = [vp]
    L.omega_list_matcher_add_stats.restype = ci
    L.omega_list_matcher_add_stats.argtypes = [vp, C.POINTER(_Stats)]
    L.omega_list_matcher_match.restype = C.POINTER(_RefResults)
    L.omega_list_matcher_match.argtypes = [vp, vp, C.c_size_t] + [ci] * 7
    L.omega_match_results_destroy.restype = None
    L.omega_match_results_destroy.argtypes = [C.POINTER(_RefResults)]
    L.omega_matcher_set_num_threads.restype = ci
    L.omega_matcher_set_num_threads.argtypes = [vp, ci]
    L.omega_matcher_get_num_threads.restype = ci
    L.omega_matcher_get_num_threads.argtypes = [vp]
    L.omega_matcher_set_chunk_size.restype = ci
    L.omega_matcher_set_chunk_size.argtypes = [vp, ci]
    L.omega_matcher_get_chunk_size.restype = ci
    L.omega_matcher_get_chunk_size.argtypes = [vp]
    L.omega_match_version.restype = cp
    L.omega_match_version.argtypes = []
    L.omega_list_matcher_is_compiled.restype = ci
    L.omega_list_matcher_is_compiled.argtypes = [cp]
    return L


class RefLib:
    """The reference's own library, unmodified (oracle/_ref)."""

    _lib = None

    @classmethod
    def lib(cls):
        if cls._lib is None:
            if not REF_SO.exists():
                raise FileNotFoundError(f"{REF_SO} missing: run `make -C oracle ref REF=<reference checkout>`")
            cls._lib = bind_list_matcher_api(C.CDLL(str(REF_SO)))
        return cls._lib

    @classmethod
    def compile(cls, out_path, patterns, case_insensitive=False, ignore_punctuation=False, elide_whitespace=False):
        buf = patterns if isinstance(patterns, (bytes, bytearray)) else b"\n".join(patterns)
        st = PatternStoreStats()
        rc = cls.lib().omega_list_matcher_compile_patterns(os.fsencode(str(out_path)), bytes(buf), len(buf),
                                                           int(case_insensitive), int(ignore_punctuation),
                                                           int(elide_whitespace), C.byref(st))
        if rc != 0:
            raise RuntimeError("reference compile failed")
        return st.as_dict()

    def __init__(self, olm_path, threads=0):
        L = self.lib()
        self._m = L.omega_list_matcher_create(os.fsencode(str(olm_path)), 0, 0, 0, None)
        if not self._m:
            raise RuntimeError("reference create failed")
        self.stats = _Stats()
        L.omega_list_matcher_add_stats(self._m, C.byref(self.stats))
        if threads:
            L.omega_matcher_set_num_threads(self._m, threads)

    def threads(self):
        return self.lib().omega_matcher_get_num_threads(self._m)

    def close(self):
        if getattr(self, "_m", None):
            self.lib().omega_list_matcher_destroy(self._m)
            self._m = None

    __del__ = close

    def match(self, haystack, **kw) -> np.ndarray:
        """-> structured array (offset,len).  The haystack is copied into a buffer that is
        followed by a NUL byte, so the reference's one-past-the-end reads are defined."""
        L = self.lib()
        n = len(haystack)
        buf = np.zeros(n + 64, dtype=np.uint8)
        buf[:n] = np.frombuffer(haystack, dtype=np.uint8) if not isinstance(haystack, np.ndarray) else haystack
        res = L.omega_list_matcher_match(self._m, buf.ctypes.data, n, *_flags(kw))
        cnt = res.contents.count
        out = np.zeros(cnt, dtype=MATCH_DTYPE)
        if cnt:
            raw = np.ctypeslib.as_array(C.cast(res.contents.matches, C.POINTER(C.c_uint8)), shape=(cnt * 24,))
            rec = raw.view(REF_RESULT_DTYPE)
            out["offset"] = rec["offset"]
            out["len"] = rec["len"]
        L.omega_match_results_destroy(res)
        return out

    def match_timed(self, buf: np.ndarray, n: int, **kw):
        """Time only omega_list_matcher_match() (BASELINE.md section 3).  -> (count, seconds)."""
        import time
        L = self.lib()
        t0 = time.perf_counter()
        res = L.omega_list_matcher_match(self._m, buf.ctypes.data, n, *_flags(kw))
        dt = time.perf_counter() - t0
        cnt = res.contents.count
        L.omega_match_results_destroy(res)
        return cnt, dt
