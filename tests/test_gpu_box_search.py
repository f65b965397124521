"""A resident database sharded over the devices of the box (BoxDatabase; psb_box_db_create, psb_box_scan,
psb_box_align, psb_box_search): every row against the same call on a single-device Database built from the same
arrays.  Repeated devices put several shards on one GPU, so every case but the multi-device one runs on a machine with
one GPU."""
import ctypes as C
import threading

import numpy as np
import pytest

import psb_data

KEYS3 = ("score", "end_query", "end_ref", "saturated")
STATS = ("matches", "similar", "length")
TRACE = ("beg_query", "beg_ref", "cigar_off", "cigar_ops")
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
    """the queries and database of test_gpu_search_many's `mixed` shape (12 queries of 30 to 1 200 residues and one of
    6 401, 400 proteins with segments of several queries planted), with a 72 000-residue subject first: a third of the
    residues, so with three or five shards it is a shard of its own (and a routed subject)"""
    lens = [30, 64, 100, 180, 250, 333, 400, 401, 640, 800, 1000, 1200, 6401]
    queries = [psb_data.random_seq(3100, i, n) for i, n in enumerate(lens)]
    cat, off = psb_data.protein_db(3101, 3102, 400, query=queries[6], planted_frac=0.03)
    subs = [cat[off[i]:off[i + 1]].copy() for i in range(400)]
    for j, q in enumerate(queries):
        s = 7 + 29 * j
        subs[s] = np.concatenate([subs[s][:20], psb_data.mutate(q[: min(len(q), 300)], 3103, j, 0.1, 0.02)])
    subs.insert(0, np.concatenate([psb_data.random_seq(3104, 0, 50000), queries[9], psb_data.random_seq(3104, 1, 22000 - len(queries[9]))]))
    cat, off = psb_data.concat(subs)
    return queries, cat, off, ps.Database((cat, off), b62)


@pytest.fixture(scope="module")
def boxes(ps, b62, mixed):
    queries, cat, off, db = mixed
    return {s: ps.BoxDatabase((cat, off), b62, devices=[0] * s) for s in (3, 5)}


@pytest.fixture(scope="module")
def dna(ps):
    """DNA subjects around one over 65 535 residues (routed) at the end of a middle shard, with copies of the query
    (16-bit re-runs) beside it in the same shard and the next; five shards leave one subject alone"""
    m = ps.Matrix.create(b"ACGT", 100, -90)
    q = psb_data.random_seq(3500, 0, 400, protein=False)
    subs = [psb_data.random_seq(3501, i, 80 + (i * 37) % 300, protein=False) for i in range(300)]
    subs[250] = np.concatenate([psb_data.random_seq(3502, 0, 40000, protein=False), q[:300], psb_data.random_seq(3502, 1, 30000, protein=False)])
    for i in (5, 248, 249, 252, 290):
        subs[i] = np.concatenate([subs[i][:30], q])
    cat, off = psb_data.concat(subs)
    return m, q, cat, off, ps.Database((cat, off), m)


def aligner(ps, mode, prof, o=10, e=1, out="", width=None, flags=None):
    b = getattr(ps.Aligner.new(), mode)().gap_open(o).gap_extend(e).profile(prof)
    if flags is not None:
        b = b.allow_query_gaps([g for g, f in (("prefix", flags[0]), ("suffix", flags[1])) if f])
        b = b.allow_ref_gaps([g for g, f in (("prefix", flags[2]), ("suffix", flags[3])) if f])
    if width is not None:
        b = b.solution_width(width)
    return b.use_trace().build() if out == "trace" else b.build()


def assert_same_rows(got, exp, tag, retried=False):
    """every field of two batches; n_retried only when asked (it depends on the cut)"""
    assert got.n == exp.n and got.flag == exp.flag and got.cells == exp.cells, tag
    if retried:
        assert got.n_retried == exp.n_retried, tag
    for k in KEYS3 + STATS + TRACE:
        a, b = getattr(got, k), getattr(exp, k)
        assert (a is None) == (b is None), (tag, k)
        if a is not None:
            assert np.array_equal(a, b), (tag, k, np.flatnonzero(a != b)[:5] if a.shape == b.shape else (a.shape, b.shape))


def assert_same_search(box, db, a, profs, k, tag):
    ids, got = a.search_many(box, profs, k)
    ids_ref, exp = a.search_many(db, profs, k)
    assert ids.shape == ids_ref.shape == (len(profs), min(k, db.n)), tag
    assert np.array_equal(ids, ids_ref), tag
    assert_same_rows(got, exp, tag)
    return ids, got


@pytest.mark.gpu
@pytest.mark.parametrize("mode,flags", [("local", None), ("global_", None), ("semi_global", None), ("semi_global", (1, 0, 0, 1))])
def test_search_equals_single_device(ps, b62, mixed, boxes, mode, flags):
    queries, cat, off, db = mixed
    for S, box in boxes.items():
        assert len(box.shards) == S and box.shards[0][:2] == (0, 1)   # the long subject is a shard of its own
        for out in ("trace", "stats", ""):
            profs = [ps.Profile.new(q, out == "stats", b62) for q in queries]
            a = aligner(ps, mode, profs[0], out=out, flags=flags)
            for k in (1, 50, db.n + 7):   # 50 is more than the first shard holds
                assert_same_search(box, db, a, profs, k, f"{S} shards {a.fn_name} k={k}")


@pytest.mark.gpu
def test_routed_and_re_run_subjects(ps, dna):
    m, q, cat, off, db = dna
    profs = [ps.Profile.new(q, False, m), ps.Profile.new(q[50:350].copy(), False, m)]
    for S in (3, 5):
        box = ps.BoxDatabase((cat, off), m, devices=[0] * S)
        middle = [s for s, (f, e, d) in enumerate(box.shards) if f <= 250 < e][0]
        assert 0 < middle < len(box.shards) - 1
        assert S == 3 or any(e - f == 1 for f, e, d in box.shards)
        for out in ("", "trace"):
            a = aligner(ps, "local", profs[0], 5, 2, out=out)
            for k in (1, 8, db.n + 7):
                ids, got = assert_same_search(box, db, a, profs, k, f"{S} shards routed {out} k={k}")
            assert got.n_retried >= 2 + 5   # the routed subject in both scans, every copy of the query at least once
            assert {5, 248, 249, 250, 252, 290} <= set(ids[0][:6].tolist())


@pytest.mark.gpu
def test_ties_across_shards_go_to_the_smallest_ids(ps, b62):
    query = psb_data.random_seq(3200, 0, 200)
    filler = psb_data.random_seq(3200, 1, 60)
    rng = np.random.default_rng(3201)
    subs = [filler.copy() for _ in range(6000)]   # one tie group over every shard boundary
    better = rng.choice(6000, 40, replace=False)
    for j, s in enumerate(better):
        subs[s] = np.concatenate([filler[:10], psb_data.mutate(query[: 40 + 3 * j], 3202, j, 0.1, 0.0)])
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), b62)
    box = ps.BoxDatabase((cat, off), b62, devices=[0] * 4)
    assert len(box.shards) == 4
    profs = [ps.Profile.new(query, False, b62), ps.Profile.new(psb_data.random_seq(3203, 0, 90), False, b62)]
    tied = np.setdiff1d(np.arange(6000), better)
    for out in ("", "trace"):
        a = aligner(ps, "local", profs[0], out=out)
        for k in (1000, 2500):   # the tie group is cut inside the first shard, and past it
            ids, got = assert_same_search(box, db, a, profs, k, f"ties {out} k={k}")
            rest = [int(i) for i in ids[0] if i not in set(better.tolist())]
            assert len(rest) >= k - 40 and rest == tied[:len(rest)].tolist()


@pytest.mark.gpu
@pytest.mark.parametrize("width", [8, 16])
def test_explicit_widths_flag_the_same_rows(ps, dna, width):
    m, q, cat, off, db = dna
    box = ps.BoxDatabase((cat, off), m, devices=[0] * 3)
    profs = [ps.Profile.new(q, False, m), ps.Profile.new(q[:200].copy(), False, m)]
    for mode in ("local", "global_"):
        for out in ("", "trace"):
            a = aligner(ps, mode, profs[0], 5, 2, out=out, width=width)
            for k in (12, db.n):
                ids, got = assert_same_search(box, db, a, profs, k, f"{width} bit {mode} {out} k={k}")
                if k == db.n:
                    assert got.saturated.any()


@pytest.mark.gpu
def test_scan_equals_single_device(ps, b62, mixed, boxes, dna):
    queries, cat, off, db = mixed
    for S, box in boxes.items():
        for stats in (False, True):
            for q in (queries[6], queries[12]):
                prof = ps.Profile.new(q, stats, b62)
                for mode in ("local", "semi_global"):
                    a = aligner(ps, mode, prof)
                    assert_same_rows(a.scan(box), a.scan(db), f"{S} shards {a.fn_name}", retried=True)
    m, q, cat, off, db = dna
    box = ps.BoxDatabase((cat, off), m, devices=[0] * 3)
    for width in (None, 16):
        a = aligner(ps, "local", ps.Profile.new(q, False, m), 5, 2, width=width)
        got, exp = a.scan(box), a.scan(db)
        assert_same_rows(got, exp, f"dna {a.fn_name}")
        if width is None:
            assert got.n_retried >= 6 and exp.n_retried >= 6   # the routed subject and every copy of the query


@pytest.mark.gpu
def test_align_equals_single_device(ps, b62, mixed, boxes):
    queries, cat, off, db = mixed
    rng = np.random.default_rng(3600)
    for S, box in boxes.items():
        ids = np.concatenate([rng.integers(0, db.n, 300), [db.n - 1, 0, 0, 5, db.n - 1]]) [rng.permutation(305)]
        for f, e, d in box.shards:   # every shard's first and last id, out of order
            ids = np.concatenate([[e - 1], ids, [f]])
        for stats, out in ((False, "trace"), (True, "")):
            prof = ps.Profile.new(queries[4], stats, b62)
            for mode in ("local", "global_"):
                a = aligner(ps, mode, prof, out=out)
                assert_same_rows(a.align_subjects(box, ids), a.align_subjects(db, ids), f"{S} shards {a.fn_name}")
                assert_same_rows(a.align_subjects(box), a.align_subjects(db), f"{S} shards {a.fn_name} all")
                one = np.array([box.shards[-1][0] + 1] * 3)   # every row on one shard
                assert_same_rows(a.align_subjects(box, one), a.align_subjects(db, one), f"{S} shards {a.fn_name} one shard")


@pytest.mark.gpu
def test_subjects_at_shard_edges(ps, mixed, boxes):
    queries, cat, off, db = mixed
    for S, box in boxes.items():
        assert box.n == db.n and box.residues == db.residues
        assert box.shards[0][0] == 0 and box.shards[-1][1] == db.n
        assert all(box.shards[s][1] == box.shards[s + 1][0] for s in range(S - 1))
        for f, e, d in box.shards:
            assert d == 0
            for i in (f, e - 1):
                assert box.subject(i) == db.subject(i), (S, i)


@pytest.mark.gpu
def test_two_threads_same_box(ps, b62, mixed, boxes):
    queries, cat, off, db = mixed
    box = boxes[3]
    profs = [ps.Profile.new(q, False, b62) for q in queries[:8]]
    a = aligner(ps, "semi_global", profs[0], out="trace")
    scan = aligner(ps, "semi_global", profs[0])
    go = threading.Barrier(2)
    outs, errors = [None, None], []

    def work(t):
        try:
            go.wait()
            outs[t] = a.search_many(box, profs, 40) if t == 0 else (a.search_many(box, profs[::-1], 25), scan.scan(box))
        except Exception as ex:  # noqa: BLE001
            errors.append(repr(ex))
    th = [threading.Thread(target=work, args=(t,)) for t in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errors, errors
    single = a.search_many(box, profs, 40)
    assert np.array_equal(outs[0][0], single[0])
    assert_same_rows(outs[0][1], single[1], "thread 0")
    single = a.search_many(box, profs[::-1], 25)
    assert np.array_equal(outs[1][0][0], single[0])
    assert_same_rows(outs[1][0][1], single[1], "thread 1")
    assert_same_rows(outs[1][1], scan.scan(box), "thread 1 scan", retried=True)


@pytest.mark.gpu
def test_errors(ps, b62, mixed, boxes):
    queries, cat, off, db = mixed
    box = boxes[3]
    L = ps._lib.lib()
    err = ps._lib.last_error
    prof = ps.Profile.new(queries[2], False, b62)
    dna_prof = ps.Profile.new(b"ACGTACGT", False, ps.Matrix.create(b"ACGT", 2, -3))
    name = b"sw_trace_striped_profile_sat"
    a = aligner(ps, "local", prof, out="trace")
    a.search_many(box, [prof], 5)
    launches = ps.launches()

    def search(name, profs, nq=None, k=5, ids=True, out=True, database=box):
        arr = (C.c_void_p * max(len(profs), 1))(*[p.inner if p is not None else None for p in profs])
        nq = len(profs) if nq is None else nq
        idbuf = np.zeros(max(nq, 1) * max(min(k, box.n), 1), dtype=np.int64)
        o = C.POINTER(ps.CBatch)()
        rc = L.psb_box_search(name, arr, nq, 10, 1, database.inner if database is not None else None, k,
                              idbuf.ctypes.data_as(C.c_void_p) if ids else None, C.byref(o) if out else None)
        assert rc != 0
        return rc

    assert search(b"sw_trace_striped_sat", [prof]) == PSB_EINVAL and "psb_box_search: not a profile function name" in err()
    assert search(b"not_a_function", [prof]) == PSB_EINVAL
    assert search(name, [prof], nq=0) == PSB_EINVAL and "psb_box_search: 0 queries" in err()
    assert search(name, [prof], k=0) == PSB_EINVAL
    assert search(name, [prof], ids=False) == PSB_EINVAL and err() == "psb_box_search: NULL argument"
    assert search(name, [prof], out=False) == PSB_EINVAL
    assert search(name, [prof], database=None) == PSB_EINVAL
    assert search(name, [prof, None, prof]) == PSB_EINVAL and err() == "psb_box_search: profiles[1] is NULL"
    assert search(name, [prof, prof, dna_prof]) == PSB_EINVAL and err() == (
        "psb_box_search: profiles[2]: profile and database were built with different alphabets")
    assert search(b"sw_table_striped_profile_sat", [prof]) == PSB_EUNSUPPORTED and "_table/_rowcol" in err()
    assert search(b"sw_rowcol_striped_profile_sat", [prof]) == PSB_EUNSUPPORTED
    big = np.zeros(1, dtype=np.int64)
    o = C.POINTER(ps.CBatch)()
    assert L.psb_box_search(name, (C.c_void_p * 1)(prof.inner), (2**31) // min(400, box.n) + 1, 10, 1, box.inner, 400,
                            big.ctypes.data_as(C.c_void_p), C.byref(o)) == PSB_EUNSUPPORTED and "2^31-1 rows" in err()

    scan_name = b"sw_striped_profile_sat"
    assert L.psb_box_scan(name, prof.inner, 10, 1, box.inner, C.byref(o)) == PSB_EUNSUPPORTED and err().startswith("psb_box_scan: trace/table/rowcol")
    assert L.psb_box_scan(b"sw_striped_sat", prof.inner, 10, 1, box.inner, C.byref(o)) == PSB_EINVAL and "psb_box_scan: not a profile" in err()
    assert L.psb_box_scan(scan_name, None, 10, 1, box.inner, C.byref(o)) == PSB_EINVAL and err() == "psb_box_scan: NULL profile"
    assert L.psb_box_scan(scan_name, prof.inner, 10, 1, None, C.byref(o)) == PSB_EINVAL and err() == "psb_box_scan: NULL argument"
    assert L.psb_box_scan(scan_name, prof.inner, 10, 1, box.inner, None) == PSB_EINVAL
    assert L.psb_box_scan(scan_name, dna_prof.inner, 10, 1, box.inner, C.byref(o)) == PSB_EINVAL and err() == (
        "psb_box_scan: profile and database were built with different alphabets")

    ids = np.array([0, box.n], dtype=np.int64)
    p_ids = ids.ctypes.data_as(C.c_void_p)
    assert L.psb_box_align(name, prof.inner, 10, 1, box.inner, p_ids, 2, C.byref(o)) == PSB_EINVAL and err() == (
        f"psb_box_align: ids[1] = {box.n} is not a subject of a database of {box.n}")
    assert L.psb_box_align(name, prof.inner, 10, 1, box.inner, None, 5, C.byref(o)) == PSB_EINVAL and err() == (
        f"psb_box_align: 5 ids for a database of {box.n} subjects")
    assert L.psb_box_align(name, prof.inner, 10, 1, box.inner, p_ids, 0, C.byref(o)) == PSB_EINVAL
    assert L.psb_box_align(b"sw_table_striped_profile_sat", prof.inner, 10, 1, box.inner, p_ids, 1, C.byref(o)) == PSB_EUNSUPPORTED
    assert L.psb_box_align(name, dna_prof.inner, 10, 1, box.inner, p_ids, 1, C.byref(o)) == PSB_EINVAL and "psb_box_align: profile and" in err()
    assert L.psb_box_align(name, prof.inner, 10, 1, None, p_ids, 1, C.byref(o)) == PSB_EINVAL

    assert L.psb_box_db_subject(box.inner, box.n, None, 0) == PSB_EINVAL and err() == (
        f"psb_box_db_subject: id {box.n} is not a subject of a database of {box.n}")
    assert L.psb_box_db_subject(box.inner, -1, None, 0) == PSB_EINVAL
    assert L.psb_box_db_subject(box.inner, 0, None, 5) == PSB_EINVAL and "NULL argument or negative capacity" in err()
    assert L.psb_box_db_subject(None, 0, None, 0) == PSB_EINVAL
    assert L.psb_box_db_shards(None, None, None) == PSB_EINVAL
    assert L.psb_box_db_count(None) == 0
    L.psb_box_db_free(None)

    with pytest.raises(ps.DeviceError, match="devices\\[1\\] = 99 is not a device"):
        ps.BoxDatabase((cat, off), b62, devices=[0, 99])
    with pytest.raises(ps.DeviceError, match="devices\\[0\\] = -1 is not a device"):
        ps.BoxDatabase((cat, off), b62, devices=[-1])
    with pytest.raises(ps.DeviceError, match="psb_box_db_create: 0 shards"):
        ps.BoxDatabase((cat, off), b62, devices=[])
    with pytest.raises(ps.DeviceError, match="psb_box_db_create: NULL argument or empty database"):
        ps.BoxDatabase([], b62, devices=[0])
    bad = off.copy()
    bad[-1] = bad[0]
    with pytest.raises(ps.DeviceError, match="psb_box_db_create: offsets are not increasing"):
        ps.BoxDatabase((cat, bad), b62, devices=[0])
    with pytest.raises(ps.Panic):
        ps.Aligner.new().local().matrix(b62).use_trace().build().search_many(box, [prof], 10)
    assert ps.launches() == launches   # none of the refused calls reached a device


@pytest.mark.gpu
def test_fewer_shards_than_asked(ps, b62):
    subs = [psb_data.random_seq(3700, i, 50 + i) for i in range(3)]
    box = ps.BoxDatabase(subs, b62, devices=[0] * 5)
    assert [(f, e) for f, e, d in box.shards] == [(0, 1), (1, 2), (2, 3)]
    db = ps.Database(subs, b62)
    prof = ps.Profile.new(subs[1], False, b62)
    a = aligner(ps, "local", prof, out="trace")
    assert_same_search(box, db, a, [prof], 10, "three subjects")


@pytest.mark.gpu
def test_several_devices(ps, b62, mixed):
    if ps._lib.lib().psb_device_count() < 2:
        pytest.skip("needs at least 2 visible GPUs")
    queries, cat, off, db = mixed
    ndev = ps._lib.lib().psb_device_count()
    for devices in (None, [1, 0]):
        box = ps.BoxDatabase((cat, off), b62, devices=devices)
        assert [d for f, e, d in box.shards] == (list(range(ndev)) if devices is None else [1, 0])
        for out in ("trace", ""):
            profs = [ps.Profile.new(q, False, b62) for q in queries]
            for mode in ("local", "global_"):
                a = aligner(ps, mode, profs[0], out=out)
                for k in (1, 50, db.n + 7):
                    assert_same_search(box, db, a, profs, k, f"devices {devices} {a.fn_name} k={k}")
        for stats in (False, True):
            a = aligner(ps, "local", ps.Profile.new(queries[6], stats, b62))
            assert_same_rows(a.scan(box), a.scan(db), f"devices {devices} scan stats={stats}", retried=True)
        for f, e, d in box.shards:
            assert box.subject(f) == db.subject(f) and box.subject(e - 1) == db.subject(e - 1)


def test_no_gpu_fails_loudly(ps):
    """without a CUDA device a box database is refused, not built on the CPU"""
    if ps._lib.lib().psb_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(ps.DeviceError) as e:
        ps.BoxDatabase([b"ACGT", b"ACGGT"], ps.Matrix.default())
    assert "no CPU fallback" in str(e.value)
    with pytest.raises(ps.DeviceError) as e:
        ps.BoxDatabase([b"ACGT", b"ACGGT"], ps.Matrix.default(), devices=[0, 0])
    assert "no CPU fallback" in str(e.value)
