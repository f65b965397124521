"""Banded nw through the CPU oracle for many pairs: oracle.align_batch with the band half-width `band` set in the
oracle's config, as oracle.align(..., band=k) does for one pair."""
import ctypes as C

import numpy as np

from oracle import oracle as orc


def align_batch(qcat, qoff, rcat, roff, mat, open, gap, band, stats=False, cigar=False, threads=0):
    """n pairs of banded nw (band half-width `band` > 0; 0 = the full table).  Returns the dict oracle.align_batch
    returns: int32 arrays score / end_query / end_ref / matches / similar / length / beg_query / beg_ref and, with
    cigar, the CIGAR CSR (cigar_off, cigar_ops)."""
    qcat = np.ascontiguousarray(np.frombuffer(bytes(qcat), dtype=np.uint8) if not isinstance(qcat, np.ndarray) else qcat, dtype=np.uint8)
    rcat = np.ascontiguousarray(np.frombuffer(bytes(rcat), dtype=np.uint8) if not isinstance(rcat, np.ndarray) else rcat, dtype=np.uint8)
    qoff = np.ascontiguousarray(qoff, dtype=np.int64)
    roff = np.ascontiguousarray(roff, dtype=np.int64)
    n = len(roff) - 1
    cfg = orc.Config(orc.NW, 1, 1, 1, 1, open, gap, band)
    orc.set_threads(threads)
    res = {k: np.zeros(n, dtype=np.int32) for k in ("score", "end_query", "end_ref", "matches", "similar", "length",
                                                     "beg_query", "beg_ref")}
    cap = int(qoff[-1] - qoff[0] + roff[-1] - roff[0]) + 8 if cigar else 0
    cig_ops = np.zeros(max(cap, 1), dtype=np.uint32)
    cig_off = np.zeros(n + 1, dtype=np.int64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = orc.lib().psbo_align_batch(p(qcat), p(qoff), p(rcat), p(roff), C.c_int64(n), C.c_int(0), C.byref(cfg),
                                    C.byref(mat.c), p(res["score"]), p(res["end_query"]), p(res["end_ref"]),
                                    p(res["matches"]) if stats else None, p(res["similar"]) if stats else None,
                                    p(res["length"]) if stats else None, C.c_int(int(cigar)), p(cig_ops),
                                    C.c_int64(cap), p(cig_off), p(res["beg_query"]), p(res["beg_ref"]))
    if rc != 0:
        raise RuntimeError("oracle batch failed")
    if cigar:
        res["cigar_off"] = cig_off
        res["cigar_ops"] = cig_ops[: cig_off[-1]].copy()
    return res
