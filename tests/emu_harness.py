"""Builds and drives tests/emu/emu_kernels.cpp: the product's kernel sources compiled with
-DPSB_EMULATE so that warp programs run on CPU threads (test-only, never shipped)."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "emu", "emu_kernels.cpp")
OUT = os.path.join(ROOT, "tests", "emu", "libpsb_emu.so")
_lib = None


def lib():
    global _lib
    if _lib is None:
        deps = [SRC] + [os.path.join(ROOT, "parasail_rs_b200", "csrc", f)
                        for f in os.listdir(os.path.join(ROOT, "parasail_rs_b200", "csrc")) if f.endswith((".cuh", ".h"))]
        if not os.path.exists(OUT) or any(os.path.getmtime(d) > os.path.getmtime(OUT) for d in deps):
            subprocess.run(["g++", "-std=c++20", "-O1", "-shared", "-fPIC", "-pthread", "-o", OUT, SRC], check=True)
        _lib = C.CDLL(OUT)
    return _lib


class Gotoh32Params(C.Structure):
    _fields_ = [("q", C.c_void_p), ("q_off", C.c_void_p), ("r", C.c_void_p), ("r_off", C.c_void_p),
                ("order", C.c_void_p), ("n", C.c_int), ("shared_query", C.c_int), ("matrix", C.c_void_p),
                ("size", C.c_int), ("is_pssm", C.c_int), ("open", C.c_int), ("gap", C.c_int),
                ("mode", C.c_int), ("s1_beg", C.c_int), ("s1_end", C.c_int), ("s2_beg", C.c_int),
                ("s2_end", C.c_int), ("score", C.c_void_p), ("end_query", C.c_void_p), ("end_ref", C.c_void_p),
                ("matches", C.c_void_p), ("similar", C.c_void_p), ("length", C.c_void_p), ("bnd", C.c_void_p),
                ("bnd_stride", C.c_longlong), ("trace", C.c_void_p), ("trace_off", C.c_void_p),
                ("counter", C.c_void_p), ("out_map", C.c_void_p), ("tabH", C.c_void_p), ("tabM", C.c_void_p),
                ("tabS", C.c_void_p), ("tabL", C.c_void_p), ("tab_off", C.c_void_p), ("r_words", C.c_void_p),
                ("r_word_off", C.c_void_p), ("r_len", C.c_void_p), ("r_bits", C.c_int), ("n_dev", C.c_void_p),
                ("banded", C.c_int), ("band_lo", C.c_int), ("band_hi", C.c_int)]


def trace_to_rowmajor(blob, off, K, lq, lr, dtype=np.int8):
    """kernel trace / table layout [strip][step][lane][K] -> row-major lq x lr cells"""
    nsteps = lr + 31
    out = np.zeros((lq, lr), dtype=dtype)
    i = np.arange(lq)
    strip, rem = i // (32 * K), i % (32 * K)
    t, k = rem // K, rem % K
    for j in range(lr):
        s = j + t
        idx = off + ((strip * nsteps + s) * 32 + t) * K + k
        out[:, j] = blob[idx].astype(dtype)
    return out


TABLE_PLANES = ("score_table", "matches_table", "similar_table", "length_table")


def gotoh32(qs, rs, mat, K, mode, open, gap, flags=(1, 1, 1, 1), stats=False, trace=False, wide=False,
            shared_query=False, nblocks=1, profile=False, packed_bits=0, table=False):
    """Run the emulated general kernel on pairs (lists of uint8 arrays of raw residues).
    table: the TABLE instantiation (statistics with the wide word, as the device runs it); the four int32 planes
    come back row-major as outs[plane name][pair]."""
    assert lib().emu_sizeof_params() == C.sizeof(Gotoh32Params)
    if table:
        assert not trace and not profile and not packed_bits
        stats = wide = True
    mapper = mat.mapper.astype(np.uint8)
    qm = [mapper[np.asarray(q, dtype=np.uint8)] for q in qs]
    rm = [mapper[np.asarray(r, dtype=np.uint8)] for r in rs]
    n = len(rm)
    qcat = np.concatenate(qm).astype(np.uint8)
    qoff = np.zeros(len(qm) + 1, dtype=np.int64); qoff[1:] = np.cumsum([len(x) for x in qm])
    rcat = np.concatenate(rm).astype(np.uint8)
    roff = np.zeros(n + 1, dtype=np.int64); roff[1:] = np.cumsum([len(x) for x in rm])
    matrix = np.ascontiguousarray(mat.table, dtype=np.int32)
    outs = {k: np.full(n, -777, dtype=np.int32) for k in ("score", "end_query", "end_ref", "matches", "similar", "length")}
    maxlr = int(max(len(x) for x in rm))
    per_col = 2 + (2 * (2 if wide else 1) if stats else 0)
    bnd = np.zeros(nblocks * per_col * maxlr + 16, dtype=np.int32)
    counter = np.zeros(1, dtype=np.int32)
    trace_off = np.zeros(n, dtype=np.int64)
    tot = 0
    for p in range(n):
        lq = len(qm[0]) if shared_query else len(qm[p])
        nstrips = (lq + 32 * K - 1) // (32 * K)
        trace_off[p] = tot
        tot += ((nstrips * (len(rm[p]) + 31) * 32 * K + 15) // 16) * 16
    blob = np.zeros(tot if trace else 16, dtype=np.uint8)
    # (cells the kernel never writes keep a sentinel that no table value takes)
    planes = [np.full(tot, -0x7fff0000, dtype=np.int32) for _ in TABLE_PLANES] if table else []
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    p = Gotoh32Params(ptr(qcat), ptr(qoff), ptr(rcat), ptr(roff), None, n, int(shared_query), ptr(matrix),
                      mat.size, int(mat.is_pssm), open, gap, mode, flags[0], flags[1], flags[2], flags[3],
                      ptr(outs["score"]), ptr(outs["end_query"]), ptr(outs["end_ref"]), ptr(outs["matches"]),
                      ptr(outs["similar"]), ptr(outs["length"]), ptr(bnd), per_col * maxlr, ptr(blob),
                      ptr(trace_off), ptr(counter), None, None, None, None, None, None, None, None, None, 0, None, 0, 0, 0)
    if table:
        p.tabH, p.tabM, p.tabS, p.tabL = (ptr(x).value for x in planes)
        p.tab_off = ptr(trace_off).value
    if packed_bits:
        # subjects from the bit-packed store, in the store's (length-sorted) order; work count from memory
        words, word_off, lens, perm = pack_db(rm, packed_bits)
        ndev = np.array([n], dtype=np.int32)
        p.r_words, p.r_word_off, p.r_len, p.r_bits = ptr(words).value, ptr(word_off).value, ptr(lens).value, packed_bits
        p.out_map, p.n_dev = ptr(perm).value, ptr(ndev).value
        p.n = n + 5   # the bound is not the count
        keep_alive = (words, word_off, lens, perm, ndev)
    lib().emu_gotoh32_use_profile(int(profile))
    rc = lib().emu_gotoh32(K, int(stats), int(trace), int(wide), C.byref(p), nblocks)
    lib().emu_gotoh32_use_profile(0)
    assert rc == 0
    lq_of = lambda i: len(qm[0]) if shared_query else len(qm[i])
    if trace:
        outs["trace"] = [trace_to_rowmajor(blob, int(trace_off[i]), K, lq_of(i), len(rm[i])) for i in range(n)]
    for name, plane in zip(TABLE_PLANES, planes):
        outs[name] = [trace_to_rowmajor(plane, int(trace_off[i]), K, lq_of(i), len(rm[i]), np.int32) for i in range(n)]
    return outs


class Sw16Params(C.Structure):
    _fields_ = [("prof", C.c_void_p), ("nletters", C.c_int), ("lq", C.c_int), ("open", C.c_int), ("gap", C.c_int),
                ("max_score", C.c_int), ("words", C.c_void_p), ("word_off", C.c_void_p), ("len", C.c_void_p),
                ("bits", C.c_int), ("n", C.c_longlong), ("out_map", C.c_void_p), ("score", C.c_void_p),
                ("end_query", C.c_void_p), ("end_ref", C.c_void_p), ("retry", C.c_void_p),
                ("retry_count", C.c_void_p), ("sid_base", C.c_int), ("counter", C.c_void_p),
                ("res_off", C.c_void_p), ("bnd_in", C.c_void_p), ("bnd_out", C.c_void_p), ("row0", C.c_int), ("merge", C.c_int),
                ("mul_one", C.c_uint), ("mul_64k", C.c_uint)]


def pack_db(subjects_mapped, bits):
    """host mirror of pack_db_kernel: sorted by length (descending, stable), rpw residues per word"""
    rpw = {2: 16, 3: 10}.get(bits, 6)
    n = len(subjects_mapped)
    perm = sorted(range(n), key=lambda i: -len(subjects_mapped[i]))
    word_off = np.zeros(n + 1, dtype=np.int64)
    lens = np.zeros(n, dtype=np.int32)
    words = []
    for s, i in enumerate(perm):
        seq = subjects_mapped[i]
        lens[s] = len(seq)
        nw = (len(seq) + rpw - 1) // rpw
        for w in range(nw):
            v = 0
            for t in range(rpw):
                idx = w * rpw + t
                if idx < len(seq):
                    v |= int(seq[idx]) << (bits * t)
            words.append(v)
        word_off[s + 1] = word_off[s] + nw
    return np.array(words + [0], dtype=np.uint32), word_off, lens, np.array(perm, dtype=np.int32)


def sw16(query, subjects, mat, open, gap, bits=5, nblocks=1, ranges=None, raw=False):
    """Run the emulated packed scan kernel: one query vs subjects.  Returns (outs, retry list): the caller ids of
    the re-run list, sorted, one entry per push (a subject pushed twice is listed twice).
    ranges: launches over sorted positions [(first, count), ...] as the engine's head and main launches
    (sw16_subjects: pointers offset by `first`, sid_base = first); default one launch over everything.
    raw: the re-run list as pushed instead (sorted positions, push order)."""
    assert lib().emu_sizeof_sw16() == C.sizeof(Sw16Params)
    mapper = mat.mapper.astype(np.uint8)
    qm = np.ascontiguousarray(mapper[np.asarray(query, dtype=np.uint8)])
    sm = [mapper[np.asarray(s, dtype=np.uint8)] for s in subjects]
    table = np.ascontiguousarray(mat.table, dtype=np.int32)
    prof = np.zeros(33 * 2048, dtype=np.int8)
    K, mx, ch = C.c_int(), C.c_int(), C.c_int()
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    nb = lib().emu_sw16_build(ptr(qm), len(qm), ptr(table), mat.size, open, ptr(prof), prof.size, C.byref(K), C.byref(mx),
                              C.byref(ch))
    assert nb > 0, nb
    words, word_off, lens, perm = pack_db(sm, bits)
    n = len(sm)
    outs = {k: np.full(n, -777, dtype=np.int32) for k in ("score", "end_query", "end_ref")}
    retry = np.full(n + 2, -1, dtype=np.int32)
    retry_count = np.zeros(1, dtype=np.int32)
    at = lambda a, first: C.c_void_p(a.ctypes.data + first * a.itemsize)
    for first, count in ranges if ranges is not None else [(0, n)]:
        counter = np.zeros(1, dtype=np.int32)
        p = Sw16Params(ptr(prof), mat.size + 1, len(qm), open, gap, mx.value, ptr(words), at(word_off, first), at(lens, first), bits,
                       count, at(perm, first), ptr(outs["score"]), ptr(outs["end_query"]), ptr(outs["end_ref"]), ptr(retry),
                       ptr(retry_count), first, ptr(counter), None, None, None, 0, 0, 1, 65536)
        rc = lib().emu_sw16(K.value, C.byref(p), nblocks)
        assert rc == 0, (rc, K.value)
    pushed = [int(i) for i in retry[: retry_count[0]]]
    return outs, pushed if raw else sorted(int(perm[i]) for i in pushed)


class Wave32Params(C.Structure):
    _fields_ = [("q", C.c_void_p), ("r", C.c_void_p), ("Lq", C.c_int), ("Lr", C.c_int), ("matrix", C.c_void_p),
                ("size", C.c_int), ("open", C.c_int), ("gap", C.c_int), ("mode", C.c_int), ("s1_beg", C.c_int),
                ("s1_end", C.c_int), ("s2_beg", C.c_int), ("s2_end", C.c_int), ("bnd", C.c_void_p),
                ("progress", C.c_void_p), ("next_strip", C.c_void_p), ("cand", C.c_void_p), ("multi_n", C.c_int),
                ("r_off", C.c_void_p), ("trace_h", C.c_void_p), ("trace_bits", C.c_void_p)]


class WaveReduceParams(C.Structure):
    _fields_ = [("cand", C.c_void_p), ("nstrips", C.c_int), ("mode", C.c_int), ("s1_end", C.c_int), ("s2_end", C.c_int),
                ("Lr", C.c_int), ("score", C.c_void_p), ("end_query", C.c_void_p), ("end_ref", C.c_void_p),
                ("multi_n", C.c_int), ("r_off", C.c_void_p), ("out_map", C.c_void_p), ("first_id", C.c_int)]


def wave32(q, r, mat, K, mode, open, gap, flags=(1, 1, 1, 1), nblocks=1, v2=False):
    """Run the emulated long-pair wavefront kernel on one pair; returns (score, end_query, end_ref).
    v2: False/True select generation 1/2; the integer 2 selects generation 3 (column-blocked, local only)."""
    lib().emu_wave32_use_v2(int(v2))
    assert lib().emu_sizeof_wave32() == C.sizeof(Wave32Params) and lib().emu_sizeof_wavereduce() == C.sizeof(WaveReduceParams)
    mapper = mat.mapper.astype(np.uint8)
    qm = np.ascontiguousarray(mapper[np.asarray(q, dtype=np.uint8)])
    rm = np.ascontiguousarray(mapper[np.asarray(r, dtype=np.uint8)])
    table = np.ascontiguousarray(mat.table, dtype=np.int32)
    nstrips = (len(qm) + 32 * K - 1) // (32 * K)
    bnd = np.zeros(nstrips * 2 * len(rm) + 16, dtype=np.int32)
    progress = np.zeros(nstrips + 1, dtype=np.int32)
    nxt = np.zeros(1, dtype=np.int32)
    cand = np.zeros(nstrips * 8 + 8, dtype=np.int32)
    out = np.zeros(3, dtype=np.int32)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    p = Wave32Params(ptr(qm), ptr(rm), len(qm), len(rm), ptr(table), mat.size, open, gap, mode, flags[0], flags[1], flags[2],
                     flags[3], ptr(bnd), ptr(progress), ptr(nxt), ptr(cand), 0, None, None, None)
    rp = WaveReduceParams(ptr(cand), nstrips, mode, flags[1], flags[3], len(rm), out.ctypes.data, out.ctypes.data + 4,
                          out.ctypes.data + 8, 0, None, None, 0)
    rc = lib().emu_wave32(K, C.byref(p), C.byref(rp), nblocks)
    assert rc == 0
    return int(out[0]), int(out[1]), int(out[2])


def wave32_multi(q, subjects, mat, K, mode, open, gap, flags=(1, 1, 1, 1), nblocks=1, v2=False):
    """Multi-pair form of the wavefront kernel: one query vs several subjects in one launch."""
    lib().emu_wave32_use_v2(int(v2))
    mapper = mat.mapper.astype(np.uint8)
    qm = np.ascontiguousarray(mapper[np.asarray(q, dtype=np.uint8)])
    sm = [mapper[np.asarray(s, dtype=np.uint8)] for s in subjects]
    rcat = np.ascontiguousarray(np.concatenate(sm))
    roff = np.zeros(len(sm) + 1, dtype=np.int64); roff[1:] = np.cumsum([len(x) for x in sm])
    table = np.ascontiguousarray(mat.table, dtype=np.int32)
    n = len(sm)
    nstrips = (len(qm) + 32 * K - 1) // (32 * K)
    bnd = np.zeros(nstrips * 2 * int(roff[-1]) + 16, dtype=np.int32)
    progress = np.zeros(n * nstrips + 1, dtype=np.int32)
    nxt = np.zeros(1, dtype=np.int32)
    cand = np.zeros(n * nstrips * 8 + 8, dtype=np.int32)
    outs = [np.full(n, -777, dtype=np.int32) for _ in range(3)]
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    p = Wave32Params(ptr(qm), ptr(rcat), len(qm), 0, ptr(table), mat.size, open, gap, mode, flags[0], flags[1], flags[2],
                     flags[3], ptr(bnd), ptr(progress), ptr(nxt), ptr(cand), n, ptr(roff), None, None)
    rp = WaveReduceParams(ptr(cand), nstrips, mode, flags[1], flags[3], 0, ptr(outs[0]), ptr(outs[1]), ptr(outs[2]), n,
                          ptr(roff), None, 0)
    rc = lib().emu_wave32(K, C.byref(p), C.byref(rp), nblocks)
    assert rc == 0
    return outs


def wave32_trace(q, r, mat, mode, open, gap, flags=(1, 1, 1, 1), what=1, nblocks=1):
    """Long pair with traceback (what=1) or statistics (what=2): the TRACE instantiation of the column-blocked
    wavefront kernel followed by walk32_kernel.  Returns a dict like the oracle's (cigar_ops in forward order)."""
    mapper = mat.mapper.astype(np.uint8)
    qm = np.ascontiguousarray(mapper[np.asarray(q, dtype=np.uint8)])
    rm = np.ascontiguousarray(mapper[np.asarray(r, dtype=np.uint8)])
    table = np.ascontiguousarray(mat.table, dtype=np.int32)
    out = np.full(8, -777, dtype=np.int32)
    rev = np.zeros(len(qm) + len(rm) + 4, dtype=np.uint32)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = lib().emu_wave32_trace(ptr(qm), len(qm), ptr(rm), len(rm), ptr(table), mat.size, open, gap, mode, flags[0], flags[1],
                                flags[2], flags[3], what, nblocks, ptr(out), ptr(rev))
    assert rc == 0, rc
    res = {"score": int(out[0]), "end_query": int(out[1]), "end_ref": int(out[2])}
    if what == 1:
        res.update(cigar_ops=rev[: out[3]][::-1].copy(), beg_query=int(out[4]), beg_ref=int(out[5]))
    else:
        res.update(matches=int(out[3]), similar=int(out[4]), length=int(out[5]))
    return res


def pairs16(qs, rs, mat, G, K, mode, open, gap, flags=(1, 1, 1, 1), what=0, nblocks=1):
    """Run the emulated packed 16-bit many-pairs kernel (csrc/kern_pairs16.cuh), two pairs per word in the
    given order.  what: 0 score only, 1 trace + CIGAR walk, 2 trace + statistics walk.  Returns a dict of
    arrays (plus 'cigar_ops' lists in forward order and beg_query / beg_ref for what == 1), or None when
    the class / 16-bit bound does not admit the batch."""
    mapper = mat.mapper.astype(np.uint8)
    qm = [mapper[np.asarray(q, dtype=np.uint8)] for q in qs]
    rm = [mapper[np.asarray(r, dtype=np.uint8)] for r in rs]
    n = len(qm)
    qcat = np.ascontiguousarray(np.concatenate(qm)); rcat = np.ascontiguousarray(np.concatenate(rm))
    qoff = np.zeros(n + 1, dtype=np.int64); qoff[1:] = np.cumsum([len(x) for x in qm])
    roff = np.zeros(n + 1, dtype=np.int64); roff[1:] = np.cumsum([len(x) for x in rm])
    table = np.ascontiguousarray(mat.table, dtype=np.int32)
    outs = {k: np.full(n, -777, dtype=np.int32) for k in ("score", "end_query", "end_ref", "matches", "similar", "length",
                                                          "nops", "beg_query", "beg_ref")}
    rev_off = np.zeros(n + 1, dtype=np.int64); rev_off[1:] = np.cumsum([len(a) + len(b) + 2 for a, b in zip(qm, rm)])
    rev = np.zeros(int(rev_off[-1]) + 4, dtype=np.uint32)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = lib().emu_pairs16(G, K, mode, flags[0], flags[1], flags[2], flags[3], what, n, ptr(qcat), ptr(qoff), ptr(rcat),
                           ptr(roff), ptr(table), mat.size, int(table.min()), int(table.max()), open, gap, nblocks,
                           ptr(outs["score"]), ptr(outs["end_query"]), ptr(outs["end_ref"]), ptr(outs["matches"]),
                           ptr(outs["similar"]), ptr(outs["length"]), ptr(rev), ptr(rev_off), ptr(outs["nops"]),
                           ptr(outs["beg_query"]), ptr(outs["beg_ref"]))
    if rc == -2:
        return None
    assert rc == 0, rc
    if what == 1:
        outs["cigar_ops"] = [rev[rev_off[i]: rev_off[i] + outs["nops"][i]][::-1].copy() for i in range(n)]
    return outs


def sw16_strips(query, subjects, mat, open, gap, rows_per_strip, bits=5, nblocks=1):
    """The strip-wise scan of a long query (STRIP instantiations of csrc/kern_sw16.cuh, host loop as in
    engine.cu): one sweep of the database per strip of `rows_per_strip` query rows.  Returns (outs, retry): the
    caller ids of the re-run list, sorted, one entry per push."""
    mapper = mat.mapper.astype(np.uint8)
    qm = np.ascontiguousarray(mapper[np.asarray(query, dtype=np.uint8)])
    sm = [mapper[np.asarray(s, dtype=np.uint8)] for s in subjects]
    table = np.ascontiguousarray(mat.table, dtype=np.int32)
    words, word_off, lens, perm = pack_db(sm, bits)
    n = len(sm)
    outs = {k: np.full(n, -777, dtype=np.int32) for k in ("score", "end_query", "end_ref")}
    nst = (len(qm) + rows_per_strip - 1) // rows_per_strip
    retry = np.full(n * nst + 2, -1, dtype=np.int32)
    retry_count = np.zeros(1, dtype=np.int32)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    rc = lib().emu_sw16_strips(ptr(qm), len(qm), ptr(table), mat.size, open, gap, rows_per_strip, ptr(words), ptr(word_off), ptr(lens),
                               bits, C.c_longlong(n), ptr(perm), ptr(outs["score"]), ptr(outs["end_query"]), ptr(outs["end_ref"]),
                               ptr(retry), ptr(retry_count), nblocks)
    assert rc == 0, rc
    return outs, sorted(int(perm[i]) for i in retry[: retry_count[0]])
