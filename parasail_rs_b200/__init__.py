"""parasail_rs_b200 -- host-side mirror of parasail-rs's API over the B200 C ABI.

Rust cannot be compiled in this environment, so the reference's safe wrapper
(`Aligner::new()...build()`, `align(Some(query), reference)`, `Profile::new`, `Matrix`, the
`Alignment` getters) is mirrored here in Python with the same names, argument meaning and error
behaviour, calling exactly the C symbols the Rust crate binds (include/parasail_b200.h).  The
parity tests therefore read like [REF tests/test_parasail.rs].  Two entry points are new (north
star): `Aligner.align_batch` (many pairs) and `Aligner.scan` (one profile vs a resident Database), with
`Aligner.search` / `Aligner.align_subjects` for the alignments of a scan's hits.

All alignment work runs in hand-written CUDA (csrc/); nothing here computes a score on the CPU.
"""
import ctypes as C
import os

import numpy as np

from . import _lib
from ._lib import CBatch, CMatrix, CResult, FUNCTION_T, PFUNCTION_T, last_error, lib

__all__ = ["Aligner", "AlignerBuilder", "Alignment", "Matrix", "Profile", "ProfileBuilder", "Database", "BoxDatabase", "BatchResult",
           "Traceback", "TraceFlags", "Error", "Panic"]


# ---- errors: one class per variant of the reference's error enums ------------------------------
class Error(Exception):
    """umbrella error [REF src/error.rs:4-17]"""


class Panic(RuntimeError):
    """conditions on which the reference panics (programmer errors) [REF src/aligner/mod.rs:353-358, 403-406]"""


class InteriorNulByte(Error): pass      # [REF src/aligner/error.rs:5-12]
class NoBandwidth(Error): pass
class QueryIsEmpty(Error): pass         # [REF src/profile/error.rs:6-16]
class NullProfile(Error): pass
class ProfileFnLookupFailed(Error): pass
class FailedLookup(Error): pass         # [REF src/matrix/error.rs:7-16]
class FileNotFound(Error): pass
class NullMatrix(Error): pass
class NotSquare(Error): pass
class NotBuiltIn(Error): pass
class InvalidIndex(Error): pass
class NoStats(Error): pass              # [REF src/alignment/error.rs:6-16]
class NoTable(Error): pass
class NoStatsTable(Error): pass
class NoRowCol(Error): pass
class NoTrace(Error): pass
class DeviceError(Error):
    """the GPU path failed (no device, CUDA error); there is no CPU fallback"""


def _bytes(x, what="sequence"):
    if isinstance(x, str):
        x = x.encode()
    if isinstance(x, np.ndarray):
        x = x.astype(np.uint8).tobytes()
    x = bytes(x)
    if b"\0" in x:
        raise InteriorNulByte(f"{what} contains an interior NUL byte")  # CString::new failure
    return x


class TraceFlags:
    """bit values of a trace-table cell [REF src/alignment/table.rs:127-142]"""
    ZERO, INS, DEL, DIAG, DIAG_E, INS_E, DIAG_F, DEL_F = 0, 1, 2, 4, 8, 16, 32, 64
    ALL = 127


# ---- Matrix [REF src/matrix/mod.rs:25-307] ------------------------------------------------------
class Matrix:
    def __init__(self, inner, builtin):
        self.inner = inner
        self.builtin = builtin

    @staticmethod
    def create(alphabet, match_score, mismatch_score):
        if not (match_score >= 0 and mismatch_score <= 0):
            raise Panic("Match score should be a positive integer and mismatch score should be a negative integer.")
        alphabet = _bytes(alphabet, "alphabet")
        if not alphabet:
            raise Panic("Alphabet should not be empty.")
        return Matrix(lib().parasail_matrix_create(alphabet, match_score, mismatch_score), False)

    @staticmethod
    def from_name(matrix_name):
        """`Matrix::from` [REF src/matrix/mod.rs:57-73]"""
        if not matrix_name:
            raise Panic("Matrix name should not be empty.")
        m = lib().parasail_matrix_lookup(_bytes(matrix_name, "matrix name"))
        if not m:
            raise FailedLookup(matrix_name)
        return Matrix(m, True)

    @staticmethod
    def from_file(path):
        if not os.path.exists(path):
            raise FileNotFound(path)
        m = lib().parasail_matrix_from_file(_bytes(path, "path"))
        if not m:
            raise NullMatrix()
        return Matrix(m, False)

    @staticmethod
    def create_pssm(alphabet, values, rows):
        arr = (C.c_int * len(values))(*values)
        m = lib().parasail_matrix_pssm_create(_bytes(alphabet, "alphabet"), arr, rows)
        if not m:
            raise NullMatrix()
        return Matrix(m, False)

    def to_pssm(self, pssm_query):
        q = _bytes(pssm_query, "pssm query")
        if not q:
            raise Panic("PSSM query sequence should not be empty.")
        if self.inner.contents.type != 0:
            raise NotSquare()
        m = lib().parasail_matrix_convert_square_to_pssm(self.inner, q, len(q))
        if not m:
            raise NullMatrix()
        return Matrix(m, False)

    def set_value(self, row, col, value):
        if self.builtin:
            raise NotBuiltIn()  # sic: the reference's name for "cannot edit a built-in" (SURVEY Q7)
        size = self.inner.contents.size - 2
        if size < 0:
            raise NullMatrix()
        if row < 0 or row > size or col < 0 or col > size:
            raise InvalidIndex(row, col)
        lib().parasail_matrix_set_value(self.inner, row, col, value)

    @staticmethod
    def default():
        return Matrix.create(b"ACGTA", 1, -1)  # [REF src/matrix/mod.rs:246-250]

    def clone(self):
        return Matrix(lib().parasail_matrix_copy(self.inner), False)

    # fields the Rust side reads directly
    @property
    def size(self): return self.inner.contents.size
    @property
    def length(self): return self.inner.contents.length
    @property
    def type_(self): return self.inner.contents.type

    def values(self):
        c = self.inner.contents
        return np.ctypeslib.as_array(c.matrix, shape=(c.length, c.size)).copy()

    def mapper(self):
        return np.ctypeslib.as_array(self.inner.contents.mapper, shape=(256,)).copy()

    def __str__(self):
        return "\n".join(" ".join(str(v) for v in row) + " " for row in self.values()) + "\n"

    def __del__(self):
        try:
            if not self.builtin and self.inner:
                lib().parasail_matrix_free(self.inner)
        except Exception:
            pass


# ---- Profile [REF src/profile/mod.rs:42-395] -----------------------------------------------------
_ISA = {"Best": "", "SSE2": "_sse_128", "SSE41": "_sse_128", "AVX2": "_avx_256", "AltiVec": "_altivec_128",
        "Neon": "_neon_128"}
_WIDTH = {"Sat": "sat", "Bit8": "8", "Bit16": "16", "Bit32": "32", "Bit64": "64", 8: "8", 16: "16", 32: "32", 64: "64"}


class Profile:
    def __init__(self, inner, use_stats, query_len):
        self.inner = inner
        self.use_stats = use_stats
        self.query_len = query_len

    @staticmethod
    def new(query, with_stats, matrix):
        q = _bytes(query, "query") if len(query) else b""
        if not q:
            raise QueryIsEmpty()
        fn = lib().parasail_profile_create_stats_sat if with_stats else lib().parasail_profile_create_sat
        p = fn(q, len(q), matrix.inner)
        if not p:
            raise NullProfile()
        return Profile(p, bool(with_stats), len(q))

    @staticmethod
    def new_ssw(query_bytes, matrix, score_size):
        """[REF src/profile/mod.rs:337-358]"""
        if len(query_bytes) == 0:
            raise Panic("Query sequence has length 0.")
        q = _bytes(query_bytes, "query")
        p = lib().parasail_ssw_init(q, len(q), matrix.inner, int(score_size))
        if not p:
            raise NullProfile()
        return Profile(p, True, len(q))

    @staticmethod
    def builder(query, matrix):
        return ProfileBuilder(query, matrix)

    @staticmethod
    def default():
        return Profile(None, False, 0)

    def is_null(self):
        return not self.inner

    def __del__(self):
        try:
            if self.inner:
                lib().parasail_profile_free(self.inner)
        except Exception:
            pass


class ProfileBuilder:
    def __init__(self, query, matrix):
        self._query, self._matrix = query, matrix
        self._stats, self._width, self._isa = False, "Sat", "Best"

    def use_stats(self, flag=True):
        self._stats = bool(flag); return self

    def solution_width(self, width):
        self._width = width; return self

    def instruction_set(self, isa):
        self._isa = isa; return self

    def build(self):
        q = _bytes(self._query, "query") if len(self._query) else b""
        if not q:
            raise QueryIsEmpty()
        name = f"parasail_profile_create{'_stats' if self._stats else ''}{_ISA[self._isa]}_{_WIDTH[self._width]}"
        fn = getattr(lib(), name, None)
        if fn is None:
            raise ProfileFnLookupFailed(name)
        p = fn(q, len(q), self._matrix.inner)
        if not p:
            raise NullProfile()
        return Profile(p, self._stats, len(q))


# ---- Alignment [REF src/alignment/mod.rs:54-504] -------------------------------------------------
class Traceback:
    def __init__(self, query, comparison, reference):
        self.query, self.comparison, self.reference = query, comparison, reference


class Alignment:
    def __init__(self, inner, matrix, query_len, ref_len):
        self.inner, self.matrix, self.query_len, self.ref_len = inner, matrix, query_len, ref_len

    def _get(self, name):
        return getattr(lib(), f"parasail_result_get_{name}")(self.inner)

    def _is(self, name):
        return getattr(lib(), f"parasail_result_is_{name}")(self.inner) != 0

    def get_score(self): return self._get("score")
    def get_end_query(self): return self._get("end_query")
    def get_end_ref(self): return self._get("end_ref")

    def get_matches(self):
        if not self.is_stats():
            raise NoStats("get_matches()")
        return self._get("matches")

    def get_similar(self):
        return self._get("similar")  # the reference does not guard this one (SURVEY Q8)

    def get_length(self):
        if not self.is_stats():
            raise NoStats("get_length()")
        return self._get("length")

    def _array(self, name, n, shape=None):
        p = self._get(name)
        if not p:
            raise DeviceError(f"{name}: not produced ({last_error()})")
        a = np.ctypeslib.as_array(p, shape=(n,)).copy()
        return a.reshape(shape) if shape else a

    def _table(self, name, need_stats):
        if need_stats:
            if not self.is_stats_table():
                raise NoStatsTable(f"get_{name}()")
        elif not (self.is_table() or self.is_stats_table()):
            raise NoTable(f"get_{name}()")
        return self._array(name, self.query_len * self.ref_len, (self.query_len, self.ref_len))

    def get_score_table(self): return self._table("score_table", False)
    def get_matches_table(self): return self._table("matches_table", True)
    def get_similar_table(self): return self._table("similar_table", True)
    def get_length_table(self): return self._table("length_table", True)

    def _rowcol(self, name, need_stats, n):
        if need_stats:
            if not self.is_stats_rowcol():
                raise NoRowCol(f"get_{name}()")
        elif not (self.is_rowcol() or self.is_stats_rowcol()):
            raise NoRowCol(f"get_{name}()")
        return self._array(name, n)

    def get_score_row(self): return self._rowcol("score_row", False, self.ref_len)
    def get_matches_row(self): return self._rowcol("matches_row", True, self.ref_len)
    def get_similar_row(self): return self._rowcol("similar_row", True, self.ref_len)
    def get_length_row(self): return self._rowcol("length_row", True, self.ref_len)
    def get_score_col(self): return self._rowcol("score_col", False, self.query_len)
    def get_matches_col(self): return self._rowcol("matches_col", True, self.query_len)
    def get_similar_col(self): return self._rowcol("similar_col", True, self.query_len)
    def get_length_col(self): return self._rowcol("length_col", True, self.query_len)

    def get_trace_table(self):
        if not self.is_trace():
            raise NoTrace("get_trace_table()")
        p = lib().parasail_result_get_trace_table(self.inner)
        if not p:
            raise DeviceError(f"trace table not produced ({last_error()})")
        raw = C.cast(p, C.POINTER(C.c_int8))
        return np.ctypeslib.as_array(raw, shape=(self.query_len * self.ref_len,)).copy().reshape(self.query_len, self.ref_len)

    def get_traceback_strings(self, query, reference):
        if not self.is_trace():
            raise NoTrace("get_traceback_strings()")
        q, r = _bytes(query), _bytes(reference)
        tb = lib().parasail_result_get_traceback(self.inner, q, len(q), r, len(r), self.matrix.inner, b"|", b" ", b" ")
        if not tb:
            raise DeviceError(last_error())
        t = tb.contents
        out = Traceback(C.string_at(t.query).decode(), C.string_at(t.comp).decode(), C.string_at(t.ref).decode())
        lib().parasail_traceback_free(tb)
        return out

    def print_traceback(self, query, reference):
        if self.is_trace():
            q, r = _bytes(query), _bytes(reference)
            lib().parasail_traceback_generic(q, len(q), r, len(r), b"Query:", b"Target:", self.matrix.inner, self.inner,
                                             b"|", b" ", b" ", 80, 7, 1)
        else:
            print("Alignment string is not available without traceback enabled. Consider using the `use_trace` "
                  "method on AlignerBuilder.")

    def get_cigar(self, query, reference):
        if not self.is_trace():
            raise NoTrace("get_cigar()")
        q, r = _bytes(query), _bytes(reference)
        c = lib().parasail_result_get_cigar(self.inner, q, len(q), r, len(r), self.matrix.inner)
        if not c:
            raise DeviceError(last_error())
        s = lib().parasail_cigar_decode(c)
        text = C.string_at(s).decode()
        self.cigar_beg = (c.contents.beg_query, c.contents.beg_ref)
        C.CDLL(None).free(C.c_void_p(s))  # malloc'd, adopted by the caller like CString::from_raw
        lib().parasail_cigar_free(c)
        return text

    def is_global(self): return self._is("nw")
    def is_semi_global(self): return self._is("sg")
    def is_local(self): return self._is("sw")
    def is_saturated(self): return self._is("saturated")
    def is_banded(self): return self._is("banded")
    def is_scan(self): return self._is("scan")
    def is_striped(self): return self._is("striped")
    def is_diag(self): return self._is("diag")
    def is_blocked(self): return self._is("blocked")
    def is_stats(self): return self._is("stats")
    def is_stats_table(self): return self._is("stats_table")
    def is_table(self): return self._is("table")
    def is_rowcol(self): return self._is("rowcol")
    def is_stats_rowcol(self): return self._is("stats_rowcol")
    def is_trace(self): return self._is("trace")

    def __del__(self):
        try:
            if self.inner:
                lib().parasail_result_free(self.inner)
        except Exception:
            pass


# ---- batched results (north star; no reference counterpart) ---------------------------------------
class BatchResult:
    """struct-of-arrays view over a psb_batch_t (pinned host memory owned by the library)"""

    def __init__(self, ptr):
        self._ptr = ptr
        b = ptr.contents
        self.n = int(b.n)
        self.flag = int(b.flag)
        self.cells = float(b.cells)
        self.n_retried = int(b.n_retried)

        def arr(p, n=self.n):
            return np.ctypeslib.as_array(p, shape=(n,)) if p else None
        self.score, self.end_query, self.end_ref = arr(b.score), arr(b.end_query), arr(b.end_ref)
        self.matches, self.similar, self.length = arr(b.matches), arr(b.similar), arr(b.length)
        self.beg_query, self.beg_ref = arr(b.beg_query), arr(b.beg_ref)
        self.saturated = arr(b.saturated)
        self.cigar_off = arr(b.cigar_off, self.n + 1)
        self.cigar_ops = arr(b.cigar_ops, int(self.cigar_off[-1])) if self.cigar_off is not None and self.cigar_off[-1] > 0 else (
            np.zeros(0, dtype=np.uint32) if self.cigar_off is not None else None)

    def cigar(self, i):
        ops = self.cigar_ops[self.cigar_off[i]: self.cigar_off[i + 1]]
        return "".join(f"{int(o) >> 4}{'MIDNSHP=X'[int(o) & 15]}" for o in ops)

    def topk(self, k):
        idx = np.zeros(k, dtype=np.int64)
        sc = np.zeros(k, dtype=np.int32)
        m = lib().psb_batch_topk(self._ptr, k, idx.ctypes.data_as(C.c_void_p), sc.ctypes.data_as(C.c_void_p))
        if m < 0:
            raise DeviceError(last_error())
        return idx[:m], sc[:m]

    def __del__(self):
        try:
            lib().psb_batch_free(self._ptr)
        except Exception:
            pass


def _concat(seqs):
    if isinstance(seqs, tuple) and len(seqs) == 2 and isinstance(seqs[0], np.ndarray):
        cat, off = seqs
        return np.ascontiguousarray(cat, dtype=np.uint8), np.ascontiguousarray(off, dtype=np.int64)
    arrs = [np.frombuffer(_bytes(s), dtype=np.uint8) if not isinstance(s, np.ndarray) else s.astype(np.uint8) for s in seqs]
    off = np.zeros(len(arrs) + 1, dtype=np.int64)
    off[1:] = np.cumsum([len(a) for a in arrs])
    cat = np.concatenate(arrs) if arrs else np.zeros(0, dtype=np.uint8)
    return np.ascontiguousarray(cat), off


class Database:
    """a subject database resident on the current GPU, bit-packed and length-sorted on the device"""

    def __init__(self, subjects, matrix, _inner=None):
        self._keep = matrix
        if _inner is None:
            cat, off = _concat(subjects)
            _inner = lib().psb_db_create(cat.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p), len(off) - 1, matrix.inner)
        self.inner = _inner
        if not self.inner:
            raise DeviceError(last_error())
        self.n = int(lib().psb_db_count(self.inner))
        self.residues = int(lib().psb_db_residues(self.inner))
        self.device_bytes = int(lib().psb_db_device_bytes(self.inner))
        self.bits = int(lib().psb_db_bits(self.inner))

    @staticmethod
    def from_fasta(path, matrix):
        """FASTA file -> resident packed database (psb_db_from_fasta)"""
        return Database(None, matrix, _inner=lib().psb_db_from_fasta(str(path).encode(), matrix.inner) or 0)

    @staticmethod
    def load(path, matrix):
        """a database saved with save(): no sorting or packing, one upload (psb_db_load)"""
        return Database(None, matrix, _inner=lib().psb_db_load(str(path).encode(), matrix.inner) or 0)

    def save(self, path):
        rc = lib().psb_db_save(self.inner, str(path).encode())
        if rc != 0:
            raise Error(f"psb_db_save failed ({rc}): {last_error()}")

    def subject(self, i):
        """subject `i` (caller order) read back out of the packed store (psb_db_subject), as the letters of the
        matrix's alphabet: code c comes back as alphabet[c].  Lowercase input therefore comes back as the
        alphabet's letter, and a residue the alphabet does not know as its wildcard (`*` for Matrix.create)."""
        n = int(lib().psb_db_subject(self.inner, int(i), None, 0))
        if n < 0:
            raise DeviceError(f"psb_db_subject failed ({n}): {last_error()}")
        codes = np.zeros(n, dtype=np.uint8)
        rc = int(lib().psb_db_subject(self.inner, int(i), codes.ctypes.data_as(C.c_void_p), n))
        if rc < 0:
            raise DeviceError(f"psb_db_subject failed ({rc}): {last_error()}")
        alphabet = np.frombuffer(self._keep.inner.contents.alphabet, dtype=np.uint8)
        return alphabet[codes].tobytes()

    def __del__(self):
        try:
            if self.inner:
                lib().psb_db_free(self.inner)
        except Exception:
            pass


class BoxDatabase:
    """a subject database sharded over the GPUs of this box, driven from this process (psb_box_db_create): contiguous
    caller-id ranges of equal residue count, shard s resident on devices[s] (devices may repeat; None: one shard per
    visible GPU).  Aligner.scan, align_subjects, search and search_many take it in place of a Database and return
    the same rows."""

    def __init__(self, subjects, matrix, devices=None):
        self._keep = matrix
        self.inner = None
        cat, off = _concat(subjects)
        devs = None if devices is None else (C.c_int * max(len(devices), 1))(*devices)
        self.inner = lib().psb_box_db_create(cat.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p), len(off) - 1,
                                             matrix.inner, devs, 0 if devices is None else len(devices))
        if not self.inner:
            raise DeviceError(last_error())
        self.n = int(lib().psb_box_db_count(self.inner))
        self.residues = int(off[-1] - off[0])
        S = int(lib().psb_box_db_shards(self.inner, None, None))
        first = np.zeros(S + 1, dtype=np.int64)
        dev = np.zeros(S, dtype=np.int32)
        lib().psb_box_db_shards(self.inner, first.ctypes.data_as(C.c_void_p), dev.ctypes.data_as(C.c_void_p))
        self.shards = [(int(first[s]), int(first[s + 1]), int(dev[s])) for s in range(S)]

    def subject(self, i):
        """subject `i` (caller order), as Database.subject"""
        n = int(lib().psb_box_db_subject(self.inner, int(i), None, 0))
        if n < 0:
            raise DeviceError(f"psb_box_db_subject failed ({n}): {last_error()}")
        codes = np.zeros(n, dtype=np.uint8)
        rc = int(lib().psb_box_db_subject(self.inner, int(i), codes.ctypes.data_as(C.c_void_p), n))
        if rc < 0:
            raise DeviceError(f"psb_box_db_subject failed ({rc}): {last_error()}")
        alphabet = np.frombuffer(self._keep.inner.contents.alphabet, dtype=np.uint8)
        return alphabet[codes].tobytes()

    def __del__(self):
        try:
            if self.inner:
                lib().psb_box_db_free(self.inner)
        except Exception:
            pass


def _on(database, single, box):
    """the C entry point for a Database or a BoxDatabase"""
    name = box if isinstance(database, BoxDatabase) else single
    return name, getattr(lib(), name)


# ---- Aligner [REF src/aligner/mod.rs:67-535] -----------------------------------------------------
class AlignerBuilder:
    def __init__(self):
        # defaults [REF src/aligner/mod.rs:86-104]
        self._mode = "nw"
        self._solution_width = "sat"
        self._matrix = Matrix.default()
        self._gap_open = 0
        self._gap_extend = 0
        self._profile = Profile.default()
        self._allow_query_gaps = []
        self._allow_ref_gaps = []
        self._vec_strategy = "_striped"
        self._use_stats = ""
        self._use_table = ""
        self._use_trace = ""
        self._bandwidth = None

    def global_(self): self._mode = "nw"; return self
    def semi_global(self): self._mode = "sg"; return self
    def local(self): self._mode = "sw"; return self
    def solution_width(self, w): self._solution_width = str(w); return self
    def matrix(self, m): self._matrix = m; return self
    def gap_open(self, v): self._gap_open = v; return self
    def gap_extend(self, v): self._gap_extend = v; return self
    def profile(self, p): self._profile = p; return self
    def allow_query_gaps(self, gaps): self._allow_query_gaps = list(gaps); return self
    def allow_ref_gaps(self, gaps): self._allow_ref_gaps = list(gaps); return self
    def striped(self): self._vec_strategy = "_striped"; return self
    def scan(self): self._vec_strategy = "_scan"; return self
    def diag(self): self._vec_strategy = "_diag"; return self
    def bandwidth(self, b): self._bandwidth = b; return self

    def use_stats(self):
        self._use_stats = "_stats"
        self._use_trace = ""  # stats and traceback are exclusive [REF src/aligner/mod.rs:213-223]
        return self

    def use_table(self):
        self._use_table = "_table"
        self._use_trace = ""
        return self

    def use_last_rowcol(self):
        self._use_table = "_rowcol"
        return self

    def use_trace(self):
        self._use_trace = "_trace"
        self._use_table = ""
        self._use_stats = ""
        return self

    @staticmethod
    def _allowed(prefix, gaps):
        if "prefix" in gaps and "suffix" in gaps:
            return f"_{prefix}x"
        if "prefix" in gaps:
            return f"_{prefix}b"
        if "suffix" in gaps:
            return f"_{prefix}e"
        return ""

    def get_parasail_fn_name(self):
        """[REF src/aligner/mod.rs:289-331]"""
        sg = ""
        if self._mode == "sg":
            sg = self._allowed("q", self._allow_query_gaps) + self._allowed("d", self._allow_ref_gaps)
            if sg == "_qx_dx":
                sg = ""
        if self._profile.is_null():
            profile, stats = "", self._use_stats
        else:
            if self._vec_strategy not in ("_striped", "_scan"):
                raise Panic("Vectorization strategy must be striped or scan for alignment with a profile.")
            profile = "_profile"
            stats = "_stats" if self._profile.use_stats else ""
        return f"{self._mode}{sg}{self._use_trace}{stats}{self._use_table}{self._vec_strategy}{profile}_{self._solution_width}"

    def build(self):
        name = self.get_parasail_fn_name()
        if self._profile.is_null():
            fn = lib().parasail_lookup_function(name.encode())
        else:
            fn = lib().parasail_lookup_pfunction(name.encode())
        if not fn:
            raise Panic(f"Parasail function: {name}, not found.")
        return Aligner(name, fn, self._matrix, self._gap_open, self._gap_extend, self._profile, self._vec_strategy,
                       self._bandwidth)


class SSWResult:
    """[REF src/alignment/mod.rs:506-551] field reads on parasail_result_ssw_t, freed on drop"""

    def __init__(self, inner):
        self.inner = inner

    def score(self): return int(self.inner.contents.score1)
    def ref_start(self): return int(self.inner.contents.ref_begin1)
    def ref_end(self): return int(self.inner.contents.ref_end1)
    def query_start(self): return int(self.inner.contents.read_begin1)
    def query_end(self): return int(self.inner.contents.read_end1)
    def cigar_len(self): return int(self.inner.contents.cigarLen)

    def cigar(self):
        n = self.cigar_len()
        return np.ctypeslib.as_array(self.inner.contents.cigar, shape=(n,)).copy() if n else np.zeros(0, dtype=np.uint32)

    def __del__(self):
        try:
            if self.inner:
                lib().parasail_result_ssw_free(self.inner)
                self.inner = None
        except Exception:
            pass


class Aligner:
    def __init__(self, fn_name, fn_ptr, matrix, gap_open, gap_extend, profile, vec_strategy, bandwidth):
        self.fn_name = fn_name
        self._fn = (PFUNCTION_T if not profile.is_null() else FUNCTION_T)(fn_ptr)
        self.matrix, self.gap_open, self.gap_extend = matrix, gap_open, gap_extend
        self._profile, self.vec_strategy, self._bandwidth = profile, vec_strategy, bandwidth

    @staticmethod
    def new():
        return AlignerBuilder()

    def align(self, query, reference):
        """[REF src/aligner/mod.rs:397-452]"""
        r = _bytes(reference, "reference")
        if self._profile.is_null():
            if query is None:
                raise Panic("Query sequence is required for alignment without a profile.")
            q = _bytes(query, "query")
            res = self._fn(q, len(q), r, len(r), self.gap_open, self.gap_extend, self.matrix.inner)
            return Alignment(res, self.matrix, len(q), len(r))
        res = self._fn(self._profile.inner, r, len(r), self.gap_open, self.gap_extend)
        return Alignment(res, self.matrix, self._profile.query_len, len(r))

    def banded_nw(self, query, reference):
        q, r = _bytes(query, "query"), _bytes(reference, "reference")
        if self._bandwidth is None:
            raise NoBandwidth()
        res = lib().parasail_nw_banded(q, len(q), r, len(r), self.gap_open, self.gap_extend, self._bandwidth, self.matrix.inner)
        return Alignment(res, self.matrix, len(q), len(r))

    def ssw(self, query, reference):
        """Striped-Smith-Waterman-compatible local alignment [REF src/aligner/mod.rs:491-529]"""
        r = _bytes(reference, "reference")
        if query is None:
            raise Panic("Query sequence is required for SSW alignment for now.")
        q = _bytes(query, "query")
        res = lib().parasail_ssw(q, len(q), r, len(r), self.gap_open, self.gap_extend, self.matrix.inner)
        return SSWResult(res)

    # ---- new batched entry points ------------------------------------------------------------
    def align_batch(self, queries, references):
        """many independent pairs in one call (psb_align_pairs); sequences as lists of bytes/arrays or
        (concatenated uint8 array, int64 offsets) tuples"""
        if not self._profile.is_null():
            raise Panic("align_batch takes explicit queries; use scan() with a profile")
        qc, qo = _concat(queries)
        rc, ro = _concat(references)
        if len(qo) != len(ro):
            raise Panic("align_batch: queries and references differ in count")
        out = C.POINTER(CBatch)()
        rc_ = lib().psb_align_pairs(self.fn_name.encode(), self.matrix.inner, self.gap_open, self.gap_extend,
                                    qc.ctypes.data_as(C.c_void_p), qo.ctypes.data_as(C.c_void_p),
                                    rc.ctypes.data_as(C.c_void_p), ro.ctypes.data_as(C.c_void_p), len(ro) - 1, C.byref(out))
        if rc_ != 0:
            raise DeviceError(f"psb_align_pairs failed ({rc_}): {last_error()}")
        return BatchResult(out)

    def banded_nw_batch(self, queries, references):
        """banded global alignment of many pairs (psb_align_pairs_banded) with the aligner's bandwidth(k): only the
        band of each pair is filled.  Inputs as align_batch; use_trace() / use_stats() select the outputs."""
        if not self._profile.is_null():
            raise Panic("banded_nw_batch takes explicit queries, not a profile")
        if not self.fn_name.startswith("nw"):
            raise Panic(f"banded_nw_batch is global alignment only, not {self.fn_name}")
        if self._bandwidth is None:
            raise NoBandwidth()
        qc, qo = _concat(queries)
        rc, ro = _concat(references)
        if len(qo) != len(ro):
            raise Panic("banded_nw_batch: queries and references differ in count")
        out = C.POINTER(CBatch)()
        rc_ = lib().psb_align_pairs_banded(self.fn_name.encode(), self.matrix.inner, self.gap_open, self.gap_extend,
                                           self._bandwidth, qc.ctypes.data_as(C.c_void_p), qo.ctypes.data_as(C.c_void_p),
                                           rc.ctypes.data_as(C.c_void_p), ro.ctypes.data_as(C.c_void_p), len(ro) - 1,
                                           C.byref(out))
        if rc_ != 0:
            raise DeviceError(f"psb_align_pairs_banded failed ({rc_}): {last_error()}")
        return BatchResult(out)

    def scan(self, database):
        """the aligner's resident profile against a resident Database or BoxDatabase (psb_scan, psb_box_scan)"""
        if self._profile.is_null():
            raise Panic("scan() needs an aligner built with .profile(...)")
        out = C.POINTER(CBatch)()
        name, fn = _on(database, "psb_scan", "psb_box_scan")
        rc_ = fn(self.fn_name.encode(), self._profile.inner, self.gap_open, self.gap_extend, database.inner, C.byref(out))
        if rc_ != 0:
            raise DeviceError(f"{name} failed ({rc_}): {last_error()}")
        return BatchResult(out)

    def align_subjects(self, database, ids=None):
        """the aligner's profile against selected subjects of a resident Database or BoxDatabase (psb_db_align,
        psb_box_align): row i belongs to
        ids[i] (caller-order ids, any order, repeats allowed); ids=None aligns every subject.  With use_trace()
        the rows carry CIGARs and begin coordinates, with a stats profile matches/similar/length."""
        if self._profile.is_null():
            raise Panic("align_subjects() needs an aligner built with .profile(...)")
        if ids is None:
            ptr, n = None, database.n
        else:
            ids = np.ascontiguousarray(ids, dtype=np.int64)
            ptr, n = ids.ctypes.data_as(C.c_void_p), len(ids)
        out = C.POINTER(CBatch)()
        name, fn = _on(database, "psb_db_align", "psb_box_align")
        rc_ = fn(self.fn_name.encode(), self._profile.inner, self.gap_open, self.gap_extend, database.inner, ptr, n, C.byref(out))
        if rc_ != 0:
            raise DeviceError(f"{name} failed ({rc_}): {last_error()}")
        return BatchResult(out)

    def search(self, database, k):
        """scan the whole Database score-only, keep the k best subjects (ties by smaller id) and align those with this
        aligner's own function: returns (ids, BatchResult) with row i belonging to ids[i].  The one-query case of
        search_many."""
        if self._profile.is_null():
            raise Panic("search() needs an aligner built with .profile(...)")
        ids, hits = self.search_many(database, [self._profile], k)
        return ids[0], hits

    def search_many(self, database, profiles, k):
        """search() for several query Profiles in one call (psb_db_search, or psb_box_search for a BoxDatabase, whose
        rows are the same), with this aligner's function name, gaps
        and width: each query's scan, and the choice of its k best subjects, run on the GPU; one alignment pass then
        serves the hits of every query.  Returns (ids, BatchResult): ids has shape (len(profiles), kk) with
        kk = min(k, database.n), and row q * kk + r of the batch belongs to ids[q, r]."""
        if self._profile.is_null():
            raise Panic("search_many() needs an aligner built with .profile(...)")
        profiles = list(profiles)
        nq = len(profiles)
        kk = min(int(k), database.n) if nq and k > 0 else 0
        ptrs = (C.c_void_p * max(nq, 1))(*[p.inner for p in profiles])
        ids = np.zeros((nq, kk), dtype=np.int64)
        out = C.POINTER(CBatch)()
        name, fn = _on(database, "psb_db_search", "psb_box_search")
        rc_ = fn(self.fn_name.encode(), ptrs, nq, self.gap_open, self.gap_extend, database.inner, int(k), ids.ctypes.data_as(C.c_void_p),
                 C.byref(out))
        if rc_ != 0:
            raise DeviceError(f"{name} failed ({rc_}): {last_error()}")
        return ids, BatchResult(out)


def _scan_host(self, subjects):
    """the aligner's profile against a database held in HOST memory (psb_scan_host): upload,
    device-side packing and scan are pipelined inside the call; nothing stays resident"""
    if self._profile.is_null():
        raise Panic("scan_host() needs an aligner built with .profile(...)")
    cat, off = _concat(subjects)
    out = C.POINTER(CBatch)()
    rc_ = lib().psb_scan_host(self.fn_name.encode(), self._profile.inner, self.gap_open, self.gap_extend,
                              cat.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p), len(off) - 1, C.byref(out))
    if rc_ != 0:
        raise DeviceError(f"psb_scan_host failed ({rc_}): {last_error()}")
    return BatchResult(out)


Aligner.scan_host = _scan_host


def _scan_box(self, subjects, n_gpus=0):
    """the aligner's profile against a host database over n_gpus devices of this box from ONE process
    (psb_scan_box): contiguous residue-balanced ranges, one worker thread per device, caller-order results"""
    if self._profile.is_null():
        raise Panic("scan_box() needs an aligner built with .profile(...)")
    cat, off = _concat(subjects)
    out = C.POINTER(CBatch)()
    rc_ = lib().psb_scan_box(self.fn_name.encode(), self._profile.inner, self.gap_open, self.gap_extend,
                             cat.ctypes.data_as(C.c_void_p), off.ctypes.data_as(C.c_void_p), len(off) - 1, int(n_gpus), C.byref(out))
    if rc_ != 0:
        raise DeviceError(f"psb_scan_box failed ({rc_}): {last_error()}")
    return BatchResult(out)


Aligner.scan_box = _scan_box


def read_fasta(path):
    """FASTA file -> (residues uint8 array, int64 offsets, list of header lines) (psb_fasta_read)"""
    fa = lib().psb_fasta_read(str(path).encode())
    if not fa:
        raise Error(last_error())
    try:
        n = int(lib().psb_fasta_count(fa))
        off = np.ctypeslib.as_array(lib().psb_fasta_offsets(fa), shape=(n + 1,)).copy()
        cat = np.ctypeslib.as_array(lib().psb_fasta_residues(fa), shape=(int(off[-1]),)).copy() if off[-1] else np.zeros(0, dtype=np.uint8)
        names = []
        ln = C.c_int()
        for i in range(n):
            ptr = lib().psb_fasta_name(fa, i, C.byref(ln))
            names.append(C.string_at(ptr, ln.value).decode(errors="replace") if ptr and ln.value else "")
        return cat, off, names
    finally:
        lib().psb_fasta_free(fa)


def shard_plan(offsets, n_shards):
    """residue-balanced assignment of subjects to GPUs (psb_shard_plan)"""
    off = np.ascontiguousarray(offsets, dtype=np.int64)
    out = np.zeros(len(off) - 1, dtype=np.int32)
    rc = lib().psb_shard_plan(off.ctypes.data_as(C.c_void_p), len(off) - 1, n_shards, out.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise Error(last_error())
    return out


def trim():
    """give back the memory the library keeps between calls on this thread's device (psb_trim)"""
    if lib().psb_trim() != 0:
        raise Error(last_error())


def host_scan_plan(total, upload_ms_per_byte, scan_ms_per_byte):
    """piece sizes (bytes) psb_scan_host / psb_scan_box would use for `total` residues at the given rates"""
    out = np.zeros(256, dtype=np.int64)
    k = lib().psb_host_scan_plan(int(total), float(upload_ms_per_byte), float(scan_ms_per_byte), out.ctypes.data_as(C.c_void_p), len(out))
    if k < 0:
        raise Error(last_error())
    return out[:min(k, len(out))].tolist()


def kernel_ms():
    return float(lib().psb_last_kernel_ms())


def launches():
    return int(lib().psb_last_launches())
