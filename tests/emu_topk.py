"""Builds and drives tests/emu/topk_kernels.cpp: the selection kernels (csrc/kern_topk.cuh) compiled with -DPSB_EMULATE
so that their warp programs run on CPU threads (test-only, never shipped).  The library is built once per process in a
temporary directory."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "emu", "topk_kernels.cpp")
_lib = None
_tmp = None


def lib():
    global _lib, _tmp
    if _lib is None:
        _tmp = tempfile.TemporaryDirectory(prefix="psb_emu_topk_")
        out = os.path.join(_tmp.name, "libpsb_emu_topk.so")
        subprocess.run(["g++", "-std=c++20", "-O1", "-shared", "-fPIC", "-pthread", "-o", out, SRC], check=True)
        _lib = C.CDLL(out)
    return _lib


def topk(score, kk, nblocks=1, nwarps=1):
    """Run the emulated selection over one query's scores in caller order.  Returns the kk rows (ids, scores) in the
    kernel's order; end_query / end_ref are carried as id + 1 and id + 2 to check the gather."""
    score = np.ascontiguousarray(score, dtype=np.int32)
    n = len(score)
    eq = np.arange(1, n + 1, dtype=np.int32)
    er = np.arange(2, n + 2, dtype=np.int32)
    outs = [np.full(kk, -777, dtype=np.int32) for _ in range(4)]
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = lib().emu_topk(ptr(score), ptr(eq), ptr(er), C.c_longlong(n), kk, nblocks, nwarps, *(ptr(o) for o in outs))
    assert rc == 0, rc
    ids, sc, oeq, oer = outs
    assert np.array_equal(oeq, ids + 1) and np.array_equal(oer, ids + 2)
    return ids, sc
