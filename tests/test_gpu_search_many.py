"""Many query profiles against a resident database in one call (psb_db_search, Aligner.search_many): every query's
rows against a loop of psb_scan + lexsort + psb_db_align per query, a sample against the CPU oracle, and the error
cases of the C ABI."""
import ctypes as C
import threading

import numpy as np
import pytest

import psb_data

pytestmark = pytest.mark.gpu

KEYS3 = ("score", "end_query", "end_ref", "saturated")
STATS = ("matches", "similar", "length")
MODES = {"local": 2, "global_": 0, "semi_global": 1}
PSB_EINVAL, PSB_EUNSUPPORTED = -1, -5


@pytest.fixture(scope="module")
def ps():
    import __graft_entry__ as g
    g.build()
    import parasail_rs_b200 as ps
    return ps


@pytest.fixture(scope="module")
def b62(ps):
    return ps.Matrix.from_name("blosum62")


@pytest.fixture(scope="module")
def mixed(ps, b62):
    """12 queries of 30 to 1 200 residues (one and several strips of the packed scan) and one of 6 401 (the 32-bit
    scan), against 500 proteins with segments of several queries planted"""
    lens = [30, 64, 100, 180, 250, 333, 400, 401, 640, 800, 1000, 1200, 6401]
    queries = [psb_data.random_seq(3100, i, n) for i, n in enumerate(lens)]
    cat, off = psb_data.protein_db(3101, 3102, 500, query=queries[6], planted_frac=0.03)
    subs = [cat[off[i]:off[i + 1]].copy() for i in range(500)]
    for j, q in enumerate(queries):
        s = 7 + 37 * j
        subs[s] = np.concatenate([subs[s][:20], psb_data.mutate(q[: min(len(q), 300)], 3103, j, 0.1, 0.02)])
    cat, off = psb_data.concat(subs)
    return queries, cat, off, ps.Database((cat, off), b62)


def aligner(ps, mode, prof, o=10, e=1, out="", width=None, flags=None):
    b = getattr(ps.Aligner.new(), mode)().gap_open(o).gap_extend(e).profile(prof)
    if flags is not None:
        b = b.allow_query_gaps([g for g, f in (("prefix", flags[0]), ("suffix", flags[1])) if f])
        b = b.allow_ref_gaps([g for g, f in (("prefix", flags[2]), ("suffix", flags[3])) if f])
    if width is not None:
        b = b.solution_width(width)
    return b.use_trace().build() if out == "trace" else b.build()


def c_call(ps, fn, *args):
    out = C.POINTER(ps.CBatch)()
    rc = getattr(ps._lib.lib(), fn)(*args, C.byref(out))
    assert rc == 0, (fn, rc, ps._lib.last_error())
    return ps.BatchResult(out)


def reference(ps, name, profs, db, k, o, e):
    """the per-query composition: psb_scan (score-only name), lexsort, psb_db_align; per query (ids, rows, scan)"""
    score_only = name.replace("_trace", "").replace("_stats", "")
    res = []
    for p in profs:
        scan = c_call(ps, "psb_scan", score_only.encode(), p.inner, o, e, db.inner)
        ids = np.lexsort((np.arange(scan.n), -scan.score.astype(np.int64)))[: min(k, db.n)]
        if "_trace" in name or "_stats" in name:
            arr = np.ascontiguousarray(ids, dtype=np.int64)
            rows = c_call(ps, "psb_db_align", name.encode(), p.inner, o, e, db.inner, arr.ctypes.data_as(C.c_void_p), len(arr))
        else:
            rows = None
        res.append((ids, rows, scan))
    return res


def assert_matches_reference(got_ids, got, ref, name, tag):
    kk = got_ids.shape[1]
    assert got.n == len(ref) * kk, tag
    assert got.n_retried == sum(r[2].n_retried for r in ref), tag
    for q, (ids, rows, scan) in enumerate(ref):
        assert np.array_equal(got_ids[q], ids), (tag, q)
        sl = slice(q * kk, (q + 1) * kk)
        src = {k: getattr(scan, k)[ids] for k in KEYS3} if rows is None else {k: getattr(rows, k) for k in KEYS3}
        if rows is not None and "_stats" in name:
            src.update({k: getattr(rows, k) for k in STATS})
        if rows is not None and "_trace" in name:
            src.update({k: getattr(rows, k) for k in ("beg_query", "beg_ref")})
        for k, x in src.items():
            assert np.array_equal(getattr(got, k)[sl], x), (tag, q, k)
        if rows is not None and "_trace" in name:
            for r in range(kk):
                assert got.cigar(q * kk + r) == rows.cigar(r), (tag, q, r)


def oracle_rows(oracle, omat, query, cat, off, ids, mode, o, e, flags=(1, 1, 1, 1), **kw):
    rc, ro = psb_data.concat([cat[off[i]:off[i + 1]] for i in ids])
    return oracle.align_batch(query, np.array([0, len(query)]), rc, ro, omat, mode=mode, open=o, gap=e, s1_beg=flags[0],
                              s1_end=flags[1], s2_beg=flags[2], s2_end=flags[3], shared_query=True, threads=0, **kw)


@pytest.mark.parametrize("mode,flags", [("local", None), ("global_", None), ("semi_global", None), ("semi_global", (1, 0, 0, 1))])
def test_many_queries_against_per_query_loop(ps, oracle, blosum62, b62, mixed, mode, flags):
    queries, cat, off, db = mixed
    for out in ("trace", "stats", ""):
        profs = [ps.Profile.new(q, out == "stats", b62) for q in queries]
        a = aligner(ps, mode, profs[0], out=out, flags=flags)
        for k in (1, 50, db.n + 7):
            ids, got = a.search_many(db, profs, k)
            kk = min(k, db.n)
            assert ids.shape == (len(queries), kk)
            ref = reference(ps, a.fn_name, profs, db, k, 10, 1)
            assert_matches_reference(ids, got, ref, a.fn_name, f"{a.fn_name} k={k}")
            assert got.cells >= sum(len(q) for q in queries) * float(off[-1])
        if out:
            # a sample against the CPU oracle: the 400-aa query's first 20 rows, and the 6 401-aa query's first 3
            for q, m in ((6, 20), (12, 3)):
                rows = ids[q, :m]
                exp = oracle_rows(oracle, blosum62, queries[q], cat, off, rows, MODES[mode], 10, 1, flags or (1, 1, 1, 1),
                                  cigar=out == "trace", stats=out == "stats")
                sl = slice(q * ids.shape[1], q * ids.shape[1] + m)
                for key in ("score", "end_query", "end_ref") + (STATS if out == "stats" else ("beg_query", "beg_ref")):
                    assert np.array_equal(getattr(got, key)[sl], exp[key]), (mode, out, q, key)


def test_ties_at_the_threshold_go_to_the_smallest_ids(ps, b62):
    query = psb_data.random_seq(3200, 0, 200)
    filler = psb_data.random_seq(3200, 1, 60)
    rng = np.random.default_rng(3201)
    subs = [filler.copy() for _ in range(6000)]   # thousands of equal scores
    better = rng.choice(6000, 40, replace=False)
    for j, s in enumerate(better):
        subs[s] = np.concatenate([filler[:10], psb_data.mutate(query[: 40 + 3 * j], 3202, j, 0.1, 0.0)])
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), b62)
    profs = [ps.Profile.new(query, False, b62), ps.Profile.new(psb_data.random_seq(3203, 0, 90), False, b62)]
    for out in ("", "trace"):
        a = aligner(ps, "local", profs[0], out=out)
        ids, got = a.search_many(db, profs, 1000)
        assert_matches_reference(ids, got, reference(ps, a.fn_name, profs, db, 1000, 10, 1), a.fn_name, f"ties {out}")
        # the tied fillers taken are the smallest ids among them, in increasing order
        tied = np.setdiff1d(np.arange(6000), better)
        rest = [int(i) for i in ids[0] if i not in set(better.tolist())]
        assert len(rest) >= 900 and rest == tied[:len(rest)].tolist()


def test_routed_and_re_run_subjects(ps):
    m = ps.Matrix.create(b"ACGT", 100, -90)
    q = psb_data.random_seq(3300, 0, 400, protein=False)
    subs = [psb_data.random_seq(3301, i, 80 + 5 * i, protein=False) for i in range(60)]
    subs[9] = q.copy()                                          # 40 000: beyond the 16-bit range, re-run at 32 bit
    subs[31] = np.concatenate([psb_data.random_seq(3302, 0, 40000, protein=False), q[:300],
                               psb_data.random_seq(3302, 1, 30000, protein=False)])   # routed: over 65 535 residues
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), m)
    profs = [ps.Profile.new(q, False, m), ps.Profile.new(q[50:350].copy(), False, m)]
    for out in ("", "trace"):
        a = aligner(ps, "local", profs[0], 5, 2, out=out)
        ids, got = a.search_many(db, profs, 5)
        ref = reference(ps, a.fn_name, profs, db, 5, 5, 2)
        assert_matches_reference(ids, got, ref, a.fn_name, f"routed {out}")
        assert got.n_retried >= 2 * 1 + 1   # the routed subject in both scans, the full copy re-run at least once
        assert ids[0, 0] == 9 and 31 in ids[0].tolist() and {9, 31} <= set(ids[1].tolist())


def test_explicit_16_bit_width(ps):
    m = ps.Matrix.create(b"ACGT", 100, -90)
    q = psb_data.random_seq(3310, 0, 400, protein=False)
    subs = [psb_data.random_seq(3311, i, 100 + 7 * i, protein=False) for i in range(40)]
    subs[5] = q.copy()
    subs[11] = np.concatenate([subs[11][:50], q[20:390]])
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), m)
    profs = [ps.Profile.new(q, False, m), ps.Profile.new(q[:200].copy(), False, m)]
    # a saturated result reads 0 before the selection (as psb_scan returns it), so it is among the hits only when k
    # takes most of the database
    for mode in ("local", "global_"):
        for out in ("", "trace"):
            a = aligner(ps, mode, profs[0], 5, 2, out=out, width=16)
            for k in (12, 40):
                ids, got = a.search_many(db, profs, k)
                assert_matches_reference(ids, got, reference(ps, a.fn_name, profs, db, k, 5, 2), a.fn_name, f"16 bit {mode} {out} k={k}")
                if mode == "local" and k == 40:
                    assert got.saturated[list(ids[0]).index(5)] == 1   # the query's own copy: 40 000 at 16 bit


def test_all_negative_global(ps):
    m = ps.Matrix.create(b"ACGT", 1, -4)
    subs = [psb_data.random_seq(3400, i, 200 + 11 * i, protein=False) for i in range(300)]
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), m)
    profs = [ps.Profile.new(psb_data.random_seq(3401, j, 150 + 50 * j, protein=False), False, m) for j in range(3)]
    for out in ("", "trace"):
        a = aligner(ps, "global_", profs[0], 6, 2, out=out)
        ids, got = a.search_many(db, profs, 40)
        assert (got.score < 0).all()
        assert_matches_reference(ids, got, reference(ps, a.fn_name, profs, db, 40, 6, 2), a.fn_name, f"negative {out}")


def test_mixed_matrices_take_separate_passes(ps, b62, mixed):
    queries, cat, off, db = mixed
    edited = b62.clone()
    edited.set_value(0, 0, 9)
    pssm = b62.to_pssm(bytes(queries[3]))
    profs = [ps.Profile.new(queries[6], False, b62), ps.Profile.new(queries[4], False, edited), ps.Profile.new(queries[3], False, pssm),
             ps.Profile.new(queries[8], False, b62), ps.Profile.new(queries[5], False, edited)]
    for mode in ("local", "semi_global"):
        a = aligner(ps, mode, profs[0], out="trace")
        ids, got = a.search_many(db, profs, 30)
        assert_matches_reference(ids, got, reference(ps, a.fn_name, profs, db, 30, 10, 1), a.fn_name, f"mixed {mode}")


def test_single_query_search_is_one_query_search_many(ps, b62, mixed):
    queries, cat, off, db = mixed
    prof = ps.Profile.new(queries[6], False, b62)
    a = aligner(ps, "local", prof, out="trace")
    ids, hits = a.search(db, 25)
    ids2, many = a.search_many(db, [prof], 25)
    assert ids.shape == (25,) and np.array_equal(ids, ids2[0])
    for k in KEYS3 + ("beg_query", "beg_ref", "cigar_off", "cigar_ops"):
        assert np.array_equal(getattr(hits, k), getattr(many, k)), k


def test_counters_cover_the_whole_call(ps, b62, mixed):
    queries, cat, off, db = mixed
    profs = [ps.Profile.new(q, False, b62) for q in queries[:6]]
    a = aligner(ps, "local", profs[0], out="trace")
    a.search_many(db, profs, 50)   # warm
    scan_ms, scan_launches = 0.0, 0
    for p in profs:
        c_call(ps, "psb_scan", b"sw_striped_profile_sat", p.inner, 10, 1, db.inner)
        scan_ms += ps.kernel_ms(); scan_launches += ps.launches()
    ids, got = a.search_many(db, profs, 50)
    ms, launches = ps.kernel_ms(), ps.launches()
    arr = np.ascontiguousarray(ids[0])
    c_call(ps, "psb_db_align", a.fn_name.encode(), profs[0].inner, 10, 1, db.inner, arr.ctypes.data_as(C.c_void_p), len(arr))
    # every scan, 12 selection launches per query, and at least one pairs pass
    assert launches >= scan_launches + 12 * len(profs) + ps.launches()
    assert ms >= 0.5 * scan_ms and ms > 0


def test_two_threads_same_database(ps, b62, mixed):
    queries, cat, off, db = mixed
    profs = [ps.Profile.new(q, False, b62) for q in queries[:8]]
    a = aligner(ps, "semi_global", profs[0], out="trace")
    go = threading.Barrier(2)
    outs, errors = [None, None], []

    def work(t):
        try:
            go.wait()
            outs[t] = a.search_many(db, profs, 40)
        except Exception as ex:  # noqa: BLE001
            errors.append(repr(ex))
    th = [threading.Thread(target=work, args=(t,)) for t in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errors, errors
    single = a.search_many(db, profs, 40)
    for t in range(2):
        assert np.array_equal(outs[t][0], single[0])
        for k in KEYS3 + ("beg_query", "beg_ref", "cigar_off", "cigar_ops"):
            assert np.array_equal(getattr(outs[t][1], k), getattr(single[1], k)), (t, k)


def test_errors(ps, b62, mixed):
    queries, cat, off, db = mixed
    L = ps._lib.lib()
    prof = ps.Profile.new(queries[2], False, b62)
    dna_prof = ps.Profile.new(b"ACGTACGT", False, ps.Matrix.create(b"ACGT", 2, -3))

    def call(name, profs, nq=None, k=5, ids=True, out=True, database=db):
        arr = (C.c_void_p * max(len(profs), 1))(*[p.inner if p is not None else None for p in profs])
        nq = len(profs) if nq is None else nq
        idbuf = np.zeros(max(nq, 1) * max(min(k, db.n), 1), dtype=np.int64)
        o = C.POINTER(ps.CBatch)()
        rc = L.psb_db_search(name, arr if profs is not None else None, nq, 10, 1, database.inner if database is not None else None, k,
                             idbuf.ctypes.data_as(C.c_void_p) if ids else None, C.byref(o) if out else None)
        if rc == 0:
            L.psb_batch_free(o)
        return rc

    name = b"sw_trace_striped_profile_sat"
    assert call(name, [prof, prof]) == 0
    assert call(b"sw_trace_striped_sat", [prof]) == PSB_EINVAL            # not a profile name
    assert call(b"not_a_function", [prof]) == PSB_EINVAL
    assert call(name, [prof], nq=0) == PSB_EINVAL
    assert call(name, [prof], k=0) == PSB_EINVAL
    assert call(name, [prof], k=-3) == PSB_EINVAL
    assert call(name, [prof], ids=False) == PSB_EINVAL
    assert call(name, [prof], out=False) == PSB_EINVAL
    assert call(name, [prof], database=None) == PSB_EINVAL
    assert call(name, [prof, None, prof]) == PSB_EINVAL and "profiles[1]" in ps._lib.last_error()
    assert call(name, [prof, prof, dna_prof]) == PSB_EINVAL and "profiles[2]" in ps._lib.last_error()
    assert call(b"sw_table_striped_profile_sat", [prof]) == PSB_EUNSUPPORTED
    assert call(b"sw_rowcol_striped_profile_sat", [prof]) == PSB_EUNSUPPORTED
    # more than 2^31 - 1 rows: refused before any device work (the id buffer is never touched)
    big = np.zeros(1, dtype=np.int64)
    arr = (C.c_void_p * 1)(prof.inner)
    o = C.POINTER(ps.CBatch)()
    assert L.psb_db_search(name, arr, (2**31) // min(400, db.n) + 1, 10, 1, db.inner, 400, big.ctypes.data_as(C.c_void_p), C.byref(o)) == PSB_EUNSUPPORTED
    with pytest.raises(ps.Panic):
        ps.Aligner.new().local().matrix(b62).use_trace().build().search_many(db, [prof], 10)
