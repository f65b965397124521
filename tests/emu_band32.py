"""Builds and drives tests/emu/band32_kernels.cpp: the band kernel (csrc/kern_band32.cuh) and walk_band_kernel
compiled with -DPSB_EMULATE so that their warp programs run on CPU threads (test-only, never shipped).  The library
is built once per process in a temporary directory."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "emu", "band32_kernels.cpp")
_lib = None
_tmp = None


def lib():
    global _lib, _tmp
    if _lib is None:
        _tmp = tempfile.TemporaryDirectory(prefix="psb_emu_band32_")
        out = os.path.join(_tmp.name, "libpsb_emu_band32.so")
        subprocess.run(["g++", "-std=c++20", "-O1", "-shared", "-fPIC", "-pthread", "-o", out, SRC], check=True)
        _lib = C.CDLL(out)
    return _lib


class Band32Params(C.Structure):
    _fields_ = [("q", C.c_void_p), ("q_off", C.c_void_p), ("r", C.c_void_p), ("r_off", C.c_void_p),
                ("order", C.c_void_p), ("n", C.c_int), ("shared_query", C.c_int), ("matrix", C.c_void_p),
                ("size", C.c_int), ("is_pssm", C.c_int), ("open", C.c_int), ("gap", C.c_int), ("k", C.c_int),
                ("score", C.c_void_p), ("end_query", C.c_void_p), ("end_ref", C.c_void_p),
                ("matches", C.c_void_p), ("similar", C.c_void_p), ("length", C.c_void_p),
                ("trace", C.c_void_p), ("trace_off", C.c_void_p), ("counter", C.c_void_p), ("rr", C.c_int)]


def band_geom(lq, lr, k):
    """(lo, hi, W) of the band of a pair (oracle rule band_rule = 0)"""
    d = lr - lq
    lo, hi = -k + min(d, 0), k + max(d, 0)
    return lo, hi, hi - lo + 1


def band32(qs, rs, mat, k, open, gap, R, stats=False, trace=False, rr=0, nblocks=1):
    """Run the emulated band kernel (csrc/kern_band32.cuh) on pairs of raw residues.  R: offsets per lane of a
    register variant (2, 4, 8, 16), or 0 for the shared-memory variant with `rr` offsets per lane.  With trace:
    'trace' holds each pair's band-layout block (lq x W bytes) and the emulated walk's 'cigar_ops' (forward order),
    'beg_query', 'beg_ref'."""
    assert lib().emu_sizeof_band32() == C.sizeof(Band32Params)
    mapper = mat.mapper.astype(np.uint8)
    qm = [mapper[np.asarray(q, dtype=np.uint8)] for q in qs]
    rm = [mapper[np.asarray(r, dtype=np.uint8)] for r in rs]
    n = len(rm)
    qcat = np.ascontiguousarray(np.concatenate(qm)).astype(np.uint8)
    qoff = np.zeros(n + 1, dtype=np.int64); qoff[1:] = np.cumsum([len(x) for x in qm])
    rcat = np.ascontiguousarray(np.concatenate(rm)).astype(np.uint8)
    roff = np.zeros(n + 1, dtype=np.int64); roff[1:] = np.cumsum([len(x) for x in rm])
    matrix = np.ascontiguousarray(mat.table, dtype=np.int32)
    outs = {name: np.full(n, -777, dtype=np.int32) for name in ("score", "end_query", "end_ref", "matches", "similar",
                                                                 "length", "nops", "beg_query", "beg_ref")}
    geo = [band_geom(len(qm[i]), len(rm[i]), k) for i in range(n)]
    trace_off = np.zeros(n + 1, dtype=np.int64)
    trace_off[1:] = np.cumsum([len(qm[i]) * geo[i][2] for i in range(n)])
    blob = np.full(int(trace_off[-1]) + 16, 0xee, dtype=np.uint8)
    rev_off = np.zeros(n + 1, dtype=np.int64); rev_off[1:] = np.cumsum([len(a) + len(b) + 2 for a, b in zip(qm, rm)])
    rev = np.zeros(int(rev_off[-1]) + 4, dtype=np.uint32)
    counter = np.zeros(1, dtype=np.int32)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    p = Band32Params(ptr(qcat), ptr(qoff), ptr(rcat), ptr(roff), None, n, 0, ptr(matrix), mat.size, int(mat.is_pssm),
                     open, gap, k, ptr(outs["score"]), ptr(outs["end_query"]), ptr(outs["end_ref"]), ptr(outs["matches"]),
                     ptr(outs["similar"]), ptr(outs["length"]), ptr(blob), ptr(trace_off), ptr(counter), rr)
    rc = lib().emu_band32(R, int(stats), int(trace), C.byref(p), nblocks, ptr(rev), ptr(rev_off), ptr(outs["nops"]),
                          ptr(outs["beg_query"]), ptr(outs["beg_ref"]))
    assert rc == 0, rc
    if trace:
        outs["trace"] = [blob[trace_off[i]: trace_off[i + 1]].reshape(len(qm[i]), geo[i][2]) for i in range(n)]
        outs["cigar_ops"] = [rev[rev_off[i]: rev_off[i] + outs["nops"][i]][::-1].copy() for i in range(n)]
    return outs
