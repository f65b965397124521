"""ctypes loader for libparasail_b200.so (the C ABI in include/parasail_b200.h).

The library is built in-tree by parasail_rs_b200.build.build_library() (nvcc, sm_100a).  There is
no Python or CPU fallback: if the shared object is missing this module raises, and every
alignment call raises when no CUDA device is usable.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# PSB_LIB_PATH selects another build of the same library (kernel tuning experiments)
LIB_PATH = os.environ.get("PSB_LIB_PATH") or os.path.join(HERE, "libparasail_b200.so")


class CMatrix(C.Structure):
    # field order = upstream parasail_matrix_t (SURVEY Appendix C); Rust reads type/size/length/matrix
    _fields_ = [("name", C.c_char_p), ("matrix", C.POINTER(C.c_int)), ("mapper", C.POINTER(C.c_int)),
                ("size", C.c_int), ("max", C.c_int), ("min", C.c_int), ("user_matrix", C.POINTER(C.c_int)),
                ("type", C.c_int), ("length", C.c_int), ("alphabet", C.c_char_p), ("query", C.c_char_p)]


class CResult(C.Structure):
    _fields_ = [("score", C.c_int), ("end_query", C.c_int), ("end_ref", C.c_int), ("flag", C.c_int),
                ("extra", C.c_void_p)]


class CCigar(C.Structure):
    _fields_ = [("seq", C.POINTER(C.c_uint32)), ("len", C.c_int), ("beg_query", C.c_int), ("beg_ref", C.c_int)]


class CResultSSW(C.Structure):
    """parasail_result_ssw_t [REF src/alignment/mod.rs:507-551 reads these fields directly]"""
    _fields_ = [("score1", C.c_uint16), ("ref_begin1", C.c_int32), ("ref_end1", C.c_int32), ("read_begin1", C.c_int32),
                ("read_end1", C.c_int32), ("cigar", C.POINTER(C.c_uint32)), ("cigarLen", C.c_int32)]


class CTraceback(C.Structure):
    _fields_ = [("query", C.c_void_p), ("comp", C.c_void_p), ("ref", C.c_void_p)]


class CBatch(C.Structure):
    _fields_ = [("n", C.c_int64), ("flag", C.c_int), ("score", C.POINTER(C.c_int)), ("end_query", C.POINTER(C.c_int)),
                ("end_ref", C.POINTER(C.c_int)), ("matches", C.POINTER(C.c_int)), ("similar", C.POINTER(C.c_int)),
                ("length", C.POINTER(C.c_int)), ("cigar_off", C.POINTER(C.c_int64)), ("cigar_ops", C.POINTER(C.c_uint32)),
                ("beg_query", C.POINTER(C.c_int)), ("beg_ref", C.POINTER(C.c_int)), ("saturated", C.POINTER(C.c_uint8)),
                ("n_retried", C.c_int64), ("cells", C.c_double), ("impl", C.c_void_p)]


FUNCTION_T = C.CFUNCTYPE(C.POINTER(CResult), C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int,
                         C.POINTER(CMatrix))
PFUNCTION_T = C.CFUNCTYPE(C.POINTER(CResult), C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int)

RESULT_INT_GETTERS = ["score", "end_query", "end_ref", "matches", "similar", "length"]
RESULT_ARRAY_GETTERS = [f"{a}_{b}" for b in ("table", "row", "col") for a in ("score", "matches", "similar", "length")]
RESULT_PREDICATES = ["nw", "sg", "sw", "saturated", "banded", "scan", "striped", "diag", "blocked", "stats",
                     "stats_table", "stats_rowcol", "table", "rowcol", "trace"]
PROFILE_CREATORS = [f"parasail_profile_create{st}{isa}_{w}" for st in ("", "_stats")
                    for isa in ("", "_sse_128", "_avx_256", "_neon_128", "_altivec_128")
                    for w in ("8", "16", "32", "64", "sat")]

# every symbol include/parasail_b200.h declares (checked by tests/test_abi_symbols.py)
ALL_SYMBOLS = (
    ["parasail_lookup_function", "parasail_lookup_pfunction", "parasail_matrix_create", "parasail_matrix_lookup",
     "parasail_matrix_from_file", "parasail_matrix_pssm_create", "parasail_matrix_copy",
     "parasail_matrix_convert_square_to_pssm", "parasail_matrix_set_value", "parasail_matrix_free",
     "parasail_profile_free", "parasail_result_free", "parasail_result_get_trace_table", "parasail_result_get_cigar",
     "parasail_cigar_decode", "parasail_cigar_free", "parasail_result_get_traceback", "parasail_traceback_free",
     "parasail_traceback_generic", "parasail_nw_banded", "parasail_ssw", "parasail_ssw_init", "parasail_result_ssw_free",
     "psb_last_error", "psb_device_count", "psb_set_device", "psb_set_stream", "psb_synchronize", "psb_batch_free",
     "psb_align_pairs", "psb_align_pairs_banded", "psb_db_create", "psb_db_count", "psb_db_residues", "psb_db_device_bytes", "psb_db_free",
     "psb_scan", "psb_db_align", "psb_db_search", "psb_db_subject", "psb_scan_host", "psb_box_db_create", "psb_box_db_count",
     "psb_box_db_shards", "psb_box_db_subject", "psb_box_db_free", "psb_box_scan", "psb_box_align", "psb_box_search", "psb_batch_topk", "psb_shard_plan", "psb_last_kernel_ms", "psb_last_launches", "psb_version"]
    + PROFILE_CREATORS
    + [f"parasail_result_get_{g}" for g in RESULT_INT_GETTERS + RESULT_ARRAY_GETTERS]
    + [f"parasail_result_is_{p}" for p in RESULT_PREDICATES])

_lib = None


def lib():
    """The loaded library.  Raises (never falls back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(nvcc, sm_100a). parasail_rs_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    L.parasail_lookup_function.restype = C.c_void_p
    L.parasail_lookup_function.argtypes = [C.c_char_p]
    L.parasail_lookup_pfunction.restype = C.c_void_p
    L.parasail_lookup_pfunction.argtypes = [C.c_char_p]
    L.parasail_matrix_create.restype = C.POINTER(CMatrix)
    L.parasail_matrix_create.argtypes = [C.c_char_p, C.c_int, C.c_int]
    L.parasail_matrix_lookup.restype = C.POINTER(CMatrix)
    L.parasail_matrix_lookup.argtypes = [C.c_char_p]
    L.parasail_matrix_from_file.restype = C.POINTER(CMatrix)
    L.parasail_matrix_from_file.argtypes = [C.c_char_p]
    L.parasail_matrix_pssm_create.restype = C.POINTER(CMatrix)
    L.parasail_matrix_pssm_create.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.c_int]
    L.parasail_matrix_copy.restype = C.POINTER(CMatrix)
    L.parasail_matrix_copy.argtypes = [C.POINTER(CMatrix)]
    L.parasail_matrix_convert_square_to_pssm.restype = C.POINTER(CMatrix)
    L.parasail_matrix_convert_square_to_pssm.argtypes = [C.POINTER(CMatrix), C.c_char_p, C.c_int]
    L.parasail_matrix_set_value.restype = None
    L.parasail_matrix_set_value.argtypes = [C.POINTER(CMatrix), C.c_int, C.c_int, C.c_int]
    L.parasail_matrix_free.restype = None
    L.parasail_matrix_free.argtypes = [C.POINTER(CMatrix)]
    for name in PROFILE_CREATORS:
        f = getattr(L, name)
        f.restype = C.c_void_p
        f.argtypes = [C.c_char_p, C.c_int, C.POINTER(CMatrix)]
    L.parasail_profile_free.restype = None
    L.parasail_profile_free.argtypes = [C.c_void_p]
    L.parasail_result_free.restype = None
    L.parasail_result_free.argtypes = [C.POINTER(CResult)]
    for g in RESULT_INT_GETTERS:
        f = getattr(L, f"parasail_result_get_{g}")
        f.restype = C.c_int
        f.argtypes = [C.POINTER(CResult)]
    for g in RESULT_ARRAY_GETTERS + ["trace_table"]:
        f = getattr(L, f"parasail_result_get_{g}")
        f.restype = C.POINTER(C.c_int)
        f.argtypes = [C.POINTER(CResult)]
    for p in RESULT_PREDICATES:
        f = getattr(L, f"parasail_result_is_{p}")
        f.restype = C.c_int
        f.argtypes = [C.POINTER(CResult)]
    L.parasail_result_get_cigar.restype = C.POINTER(CCigar)
    L.parasail_result_get_cigar.argtypes = [C.POINTER(CResult), C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.POINTER(CMatrix)]
    L.parasail_cigar_decode.restype = C.c_void_p
    L.parasail_cigar_decode.argtypes = [C.POINTER(CCigar)]
    L.parasail_cigar_free.restype = None
    L.parasail_cigar_free.argtypes = [C.POINTER(CCigar)]
    L.parasail_result_get_traceback.restype = C.POINTER(CTraceback)
    L.parasail_result_get_traceback.argtypes = [C.POINTER(CResult), C.c_char_p, C.c_int, C.c_char_p, C.c_int,
                                                C.POINTER(CMatrix), C.c_char, C.c_char, C.c_char]
    L.parasail_traceback_free.restype = None
    L.parasail_traceback_free.argtypes = [C.POINTER(CTraceback)]
    L.parasail_traceback_generic.restype = None
    L.parasail_traceback_generic.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_char_p,
                                             C.POINTER(CMatrix), C.POINTER(CResult), C.c_char, C.c_char, C.c_char,
                                             C.c_int, C.c_int, C.c_int]
    L.parasail_nw_banded.restype = C.POINTER(CResult)
    L.parasail_nw_banded.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(CMatrix)]
    L.parasail_ssw.restype = C.POINTER(CResultSSW)
    L.parasail_ssw.argtypes = [C.c_char_p, C.c_int, C.c_char_p, C.c_int, C.c_int, C.c_int, C.POINTER(CMatrix)]
    L.parasail_ssw_init.restype = C.c_void_p
    L.parasail_ssw_init.argtypes = [C.c_char_p, C.c_int, C.POINTER(CMatrix), C.c_int8]
    L.parasail_result_ssw_free.restype = None
    L.parasail_result_ssw_free.argtypes = [C.POINTER(CResultSSW)]
    L.psb_last_error.restype = C.c_char_p
    L.psb_version.restype = C.c_char_p
    L.psb_device_count.restype = C.c_int
    L.psb_set_device.argtypes = [C.c_int]
    L.psb_set_stream.argtypes = [C.c_void_p]
    L.psb_batch_free.restype = None
    L.psb_batch_free.argtypes = [C.POINTER(CBatch)]
    L.psb_align_pairs.restype = C.c_int
    L.psb_align_pairs.argtypes = [C.c_char_p, C.POINTER(CMatrix), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_int64, C.POINTER(C.POINTER(CBatch))]
    L.psb_align_pairs_banded.restype = C.c_int
    L.psb_align_pairs_banded.argtypes = [C.c_char_p, C.POINTER(CMatrix), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.POINTER(CBatch))]
    L.psb_db_create.restype = C.c_void_p
    L.psb_db_create.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(CMatrix)]
    L.psb_db_count.restype = C.c_int64
    L.psb_db_count.argtypes = [C.c_void_p]
    L.psb_db_residues.restype = C.c_int64
    L.psb_db_residues.argtypes = [C.c_void_p]
    L.psb_db_device_bytes.restype = C.c_int64
    L.psb_db_device_bytes.argtypes = [C.c_void_p]
    L.psb_db_free.restype = None
    L.psb_db_free.argtypes = [C.c_void_p]
    L.psb_db_bits.restype = C.c_int
    L.psb_db_bits.argtypes = [C.c_void_p]
    L.psb_fasta_read.restype = C.c_void_p
    L.psb_fasta_read.argtypes = [C.c_char_p]
    L.psb_fasta_count.restype = C.c_int64
    L.psb_fasta_count.argtypes = [C.c_void_p]
    L.psb_fasta_residues.restype = C.POINTER(C.c_uint8)
    L.psb_fasta_residues.argtypes = [C.c_void_p]
    L.psb_fasta_offsets.restype = C.POINTER(C.c_int64)
    L.psb_fasta_offsets.argtypes = [C.c_void_p]
    L.psb_fasta_name.restype = C.c_void_p
    L.psb_fasta_name.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_int)]
    L.psb_fasta_free.restype = None
    L.psb_fasta_free.argtypes = [C.c_void_p]
    L.psb_db_from_fasta.restype = C.c_void_p
    L.psb_db_from_fasta.argtypes = [C.c_char_p, C.POINTER(CMatrix)]
    L.psb_db_save.restype = C.c_int
    L.psb_db_save.argtypes = [C.c_void_p, C.c_char_p]
    L.psb_db_load.restype = C.c_void_p
    L.psb_db_load.argtypes = [C.c_char_p, C.POINTER(CMatrix)]
    L.psb_scan.restype = C.c_int
    L.psb_scan.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.POINTER(CBatch))]
    L.psb_db_align.restype = C.c_int
    L.psb_db_align.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                               C.POINTER(C.POINTER(CBatch))]
    L.psb_db_search.restype = C.c_int
    L.psb_db_search.argtypes = [C.c_char_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                C.POINTER(C.POINTER(CBatch))]
    L.psb_db_subject.restype = C.c_int64
    L.psb_db_subject.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]
    L.psb_scan_host.restype = C.c_int
    L.psb_scan_host.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                                C.POINTER(C.POINTER(CBatch))]
    L.psb_scan_box.restype = C.c_int
    L.psb_scan_box.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_int,
                               C.POINTER(C.POINTER(CBatch))]
    L.psb_box_db_create.restype = C.c_void_p
    L.psb_box_db_create.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(CMatrix), C.c_void_p, C.c_int]
    L.psb_box_db_count.restype = C.c_int64
    L.psb_box_db_count.argtypes = [C.c_void_p]
    L.psb_box_db_shards.restype = C.c_int
    L.psb_box_db_shards.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.psb_box_db_subject.restype = C.c_int64
    L.psb_box_db_subject.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64]
    L.psb_box_db_free.restype = None
    L.psb_box_db_free.argtypes = [C.c_void_p]
    L.psb_box_scan.restype = C.c_int
    L.psb_box_scan.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.POINTER(CBatch))]
    L.psb_box_align.restype = C.c_int
    L.psb_box_align.argtypes = [C.c_char_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64,
                                C.POINTER(C.POINTER(CBatch))]
    L.psb_box_search.restype = C.c_int
    L.psb_box_search.argtypes = [C.c_char_p, C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                 C.POINTER(C.POINTER(CBatch))]
    L.psb_batch_topk.restype = C.c_int
    L.psb_batch_topk.argtypes = [C.POINTER(CBatch), C.c_int, C.c_void_p, C.c_void_p]
    L.psb_shard_plan.restype = C.c_int
    L.psb_shard_plan.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p]
    L.psb_trim.restype = C.c_int
    L.psb_trim.argtypes = []
    L.psb_host_scan_plan.restype = C.c_int
    L.psb_host_scan_plan.argtypes = [C.c_int64, C.c_double, C.c_double, C.c_void_p, C.c_int]
    L.psb_last_kernel_ms.restype = C.c_double
    L.psb_last_launches.restype = C.c_int
    _lib = L
    return L


def last_error() -> str:
    return lib().psb_last_error().decode(errors="replace")
