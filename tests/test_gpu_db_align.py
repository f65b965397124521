"""Alignments of the hits of a database scan, read out of the resident, packed database (psb_db_align,
Aligner.search / align_subjects, Database.subject): against the CPU oracle on the same (query, subject) pairs,
against psb_scan where both compute the same thing, and under the error cases of the C ABI."""
import ctypes as C
import threading

import numpy as np
import pytest

import psb_data
from test_oracle_properties import cigar_rescore

pytestmark = pytest.mark.gpu

KEYS3 = ("score", "end_query", "end_ref")
KEYS6 = KEYS3 + ("matches", "similar", "length")
TRACE_KEYS = KEYS3 + ("beg_query", "beg_ref", "cigar_off", "cigar_ops")
MODES = {"local": 2, "global_": 0, "semi_global": 1}
PSB_EINVAL, PSB_EUNSUPPORTED = -1, -5


@pytest.fixture(scope="module")
def ps():
    import __graft_entry__ as g
    g.build()
    import parasail_rs_b200 as ps
    return ps


@pytest.fixture(scope="module")
def c2(ps):
    """reduced C2: 6 000 proteins with planted hits, a 400-aa query, resident under BLOSUM62"""
    query = psb_data.random_seq(2001, 0, 400)
    cat, off = psb_data.protein_db(2002, 2003, 6000, query=query, planted_frac=0.02)
    b62 = ps.Matrix.from_name("blosum62")
    return query, cat, off, b62, ps.Database((cat, off), b62)


def aligner(ps, mode, prof, o=10, e=1, trace=True, width=None, flags=None):
    b = getattr(ps.Aligner.new(), mode)().gap_open(o).gap_extend(e).profile(prof)
    if flags is not None:
        b = b.allow_query_gaps([g for g, f in (("prefix", flags[0]), ("suffix", flags[1])) if f])
        b = b.allow_ref_gaps([g for g, f in (("prefix", flags[2]), ("suffix", flags[3])) if f])
    if width is not None:
        b = b.solution_width(width)
    return (b.use_trace() if trace else b).build()


def subjects(cat, off, ids):
    return psb_data.concat([cat[off[i]:off[i + 1]] for i in ids])


def oracle_hits(oracle, omat, query, cat, off, ids, mode, o, e, flags=(1, 1, 1, 1), **kw):
    rc, ro = subjects(cat, off, ids)
    return oracle.align_batch(query, np.array([0, len(query)]), rc, ro, omat, mode=mode, open=o, gap=e, s1_beg=flags[0],
                              s1_end=flags[1], s2_beg=flags[2], s2_end=flags[3], shared_query=True, threads=0, **kw)


def assert_same(got, exp, keys, tag=""):
    for k in keys:
        g, x = getattr(got, k), exp[k] if isinstance(exp, dict) else getattr(exp, k)
        if not np.array_equal(g, x):
            bad = np.nonzero(g != x)[0] if len(g) == len(x) else [0]
            raise AssertionError(f"{tag} {k}: first difference at {bad[0]} (lengths {len(g)} / {len(x)})")


def assert_rescores(hits, query, cat, off, ids, omat, o, e, mode):
    """every CIGAR re-scores to its pair's score and lands on its end cell (free leading I/D runs of sg/sw aside)"""
    for i, sid in enumerate(ids):
        ops = hits.cigar_ops[hits.cigar_off[i]:hits.cigar_off[i + 1]]
        r = cat[off[sid]:off[sid + 1]]
        sc, ei, ej, *_ = cigar_rescore(ops, query, r, int(hits.beg_query[i]), int(hits.beg_ref[i]), omat, o, e)
        if mode == 2 and hits.score[i] == 0:
            continue
        assert (ei, ej) == (hits.end_query[i], hits.end_ref[i]), i
        if mode != 0 and len(ops) and (int(ops[0]) & 15) in (1, 2):
            n = int(ops[0]) >> 4
            sc += o + (n - 1) * e
        assert sc == hits.score[i], i


@pytest.mark.parametrize("mode", ["local", "global_", "semi_global"])
def test_search_c2_reduced_against_oracle(ps, oracle, blosum62, c2, mode):
    query, cat, off, b62, db = c2
    prof = ps.Profile.new(query, False, b62)
    ids, hits = aligner(ps, mode, prof).search(db, 200)
    assert len(ids) == 200 and hits.n == 200
    scan = aligner(ps, mode, prof, trace=False).scan(db)
    order = np.lexsort((np.arange(scan.n), -scan.score))[:200]
    assert np.array_equal(ids, order)
    exp = oracle_hits(oracle, blosum62, query, cat, off, ids, MODES[mode], 10, 1, cigar=True)
    assert_same(hits, exp, TRACE_KEYS, mode)
    assert np.array_equal(hits.score, scan.score[ids])
    if mode == "local":
        for k in KEYS3:
            assert np.array_equal(getattr(hits, k), getattr(scan, k)[ids]), k
        assert hits.score[0] > 200   # a planted segment


@pytest.mark.parametrize("mode,flags", [("local", None), ("semi_global", (1, 0, 0, 1))])
def test_stats_over_every_subject(ps, oracle, blosum62, mode, flags):
    query = psb_data.random_seq(2011, 0, 300)
    cat, off = psb_data.protein_db(2012, 2013, 2000, query=query, planted_frac=0.05)
    b62 = ps.Matrix.from_name("blosum62")
    db = ps.Database((cat, off), b62)
    a = aligner(ps, mode, ps.Profile.new(query, True, b62), trace=False, flags=flags)
    assert "_stats" in a.fn_name
    got = a.align_subjects(db)
    assert got.n == db.n
    assert_same(got, a.scan(db), KEYS6, f"{mode} vs psb_scan")
    exp = oracle_hits(oracle, blosum62, query, cat, off, np.arange(db.n), MODES[mode], 10, 1, flags or (1, 1, 1, 1), stats=True)
    assert_same(got, exp, KEYS6, f"{mode} vs oracle")


def test_off_the_packed_path(ps, oracle, blosum62):
    b62 = ps.Matrix.from_name("blosum62")
    # a 70 kb subject (beyond the 16-bit column range: 32-bit classes) among ordinary ones
    query = psb_data.random_seq(2021, 0, 400)
    subs = [psb_data.random_seq(2022, i, 50 + 37 * i) for i in range(12)]
    subs[4] = np.concatenate([psb_data.random_seq(2023, 0, 30000), psb_data.mutate(query, 2023, 1, 0.1, 0.02),
                              psb_data.random_seq(2023, 2, 39600)])
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), b62)
    ids = np.array([4, 0, 11, 4, 7])
    for mode in ("local", "global_"):
        hits = aligner(ps, mode, ps.Profile.new(query, False, b62)).align_subjects(db, ids)
        exp = oracle_hits(oracle, blosum62, query, cat, off, ids, MODES[mode], 10, 1, cigar=True)
        assert_same(hits, exp, TRACE_KEYS, f"70 kb {mode}")
        assert_rescores(hits, query, cat, off, ids, blosum62, 10, 1, MODES[mode])
    # a 2 500-residue query against 3 kb subjects: the traced wavefront launch and its walk
    query = psb_data.random_seq(2024, 0, 2500)
    subs = [np.concatenate([psb_data.random_seq(2025, i, 200), psb_data.mutate(query[300 * i: 300 * i + 2000], 2025, 10 + i, 0.12, 0.03),
                            psb_data.random_seq(2026, i, 800)])[:3000] for i in range(4)]
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), b62)
    ids = np.array([3, 1, 0, 2])
    for mode in ("local", "semi_global"):
        hits = aligner(ps, mode, ps.Profile.new(query, False, b62)).align_subjects(db, ids)
        exp = oracle_hits(oracle, blosum62, query, cat, off, ids, MODES[mode], 10, 1, cigar=True)
        assert_same(hits, exp, TRACE_KEYS, f"long query {mode}")
        assert_rescores(hits, query, cat, off, ids, blosum62, 10, 1, MODES[mode])


def test_dna_two_and_three_bit(ps, oracle):
    dna, odna = ps.Matrix.create(b"ACGT", 2, -3), oracle.Matrix.create(b"ACGT", 2, -3)
    query = psb_data.random_seq(2031, 0, 150, protein=False)
    subs = [psb_data.random_seq(2031, 1 + i, 40 + 13 * i, protein=False) for i in range(40)]
    subs[3] = np.concatenate([subs[3][:20], psb_data.mutate(query[20:120], 2031, 99, 0.05, 0.02, protein=False)])
    for with_n, bits in ((False, 2), (True, 3)):
        ss = [s.copy() for s in subs]
        if with_n:
            ss[7][5] = ord("N"); ss[3][30] = ord("n"); ss[9][0] = ord("a")
        cat, off = psb_data.concat(ss)
        db = ps.Database((cat, off), dna)
        assert db.bits == bits
        for mode in ("local", "semi_global", "global_"):
            ids, hits = aligner(ps, mode, ps.Profile.new(query, False, dna), 5, 2).search(db, 15)
            exp = oracle_hits(oracle, odna, query, cat, off, ids, MODES[mode], 5, 2, cigar=True)
            assert_same(hits, exp, TRACE_KEYS, f"{bits}-bit {mode}")


def expected_subject(ps_matrix, raw):
    alphabet = np.frombuffer(ps_matrix.inner.contents.alphabet, dtype=np.uint8)
    return alphabet[ps_matrix.mapper()[raw]].tobytes()


def test_loaded_databases_and_subject_read_back(ps, blosum62, c2, tmp_path):
    query, cat, off, b62, db = c2
    fa = tmp_path / "db.fa"
    with open(fa, "wb") as f:
        for i in range(len(off) - 1):
            f.write(b">s%d\n" % i + bytes(cat[off[i]:off[i + 1]]) + b"\n")
    db.save(tmp_path / "db.psbdb")
    a = aligner(ps, "local", ps.Profile.new(query, False, b62))
    ids, base = a.search(db, 100)
    for other, tag in ((ps.Database.load(tmp_path / "db.psbdb", b62), "load"), (ps.Database.from_fasta(fa, b62), "from_fasta")):
        ids2, got = a.search(other, 100)
        assert np.array_equal(ids2, ids), tag
        assert_same(got, base, TRACE_KEYS, tag)
    # every subject of a small database read back, original and loaded; lower case and unknown letters included
    small_cat, small_off = cat[: off[300]].copy(), off[:301]
    small_cat[5] = ord("a"); small_cat[17] = ord("J"); small_cat[small_off[7]] = ord("?")
    small = ps.Database((small_cat, small_off), b62)
    small.save(tmp_path / "small.psbdb")
    loaded = ps.Database.load(tmp_path / "small.psbdb", b62)
    for d, tag in ((small, "original"), (loaded, "loaded")):
        for i in range(300):
            assert d.subject(i) == expected_subject(b62, small_cat[small_off[i]:small_off[i + 1]]), (tag, i)
    assert small.subject(0)[5:6] == b"A"
    dna = ps.Matrix.create(b"ACGT", 2, -3)
    dcat, doff = psb_data.concat([np.frombuffer(b"ACGTNacgtn", dtype=np.uint8), np.frombuffer(b"T", dtype=np.uint8)])
    ddb = ps.Database((dcat, doff), dna)
    assert (ddb.subject(0), ddb.subject(1)) == (b"ACGT*ACGT*", b"T")


def test_passes_equal_single_call(ps, c2, monkeypatch):
    query, cat, off, b62, db = c2
    ids = np.concatenate([np.arange(db.n), np.arange(db.n)[::-1]])   # 12 000 ids, ~4 MB of subjects
    a = aligner(ps, "local", ps.Profile.new(query, False, b62))
    one = a.align_subjects(db, ids)
    monkeypatch.setenv("PSB_PAIRS_PASS_MB", "1")
    passes = a.align_subjects(db, ids)
    assert_same(passes, one, TRACE_KEYS, "1 MB passes")
    assert passes.cells == one.cells


def test_order_and_repeats(ps, c2):
    query, cat, off, b62, db = c2
    rng = np.random.default_rng(7)
    ids = rng.permutation(np.concatenate([rng.choice(db.n, 300, replace=False), np.full(5, db.n - 1), np.zeros(5, dtype=np.int64)]))
    a = aligner(ps, "semi_global", ps.Profile.new(query, False, b62))
    got = a.align_subjects(db, ids)
    uniq = np.unique(ids)
    ref = a.align_subjects(db, uniq)
    row = {int(s): i for i, s in enumerate(uniq)}
    for i, s in enumerate(ids):
        j = row[int(s)]
        for k in KEYS3 + ("beg_query", "beg_ref"):
            assert getattr(got, k)[i] == getattr(ref, k)[j], (i, k)
        assert got.cigar(i) == ref.cigar(j), i


def test_explicit_16_bit_width_flags_saturation_like_scan(ps):
    m = ps.Matrix.create(b"ACGT", 100, -90)
    q = psb_data.random_seq(2601, 0, 400, protein=False)
    subs = [psb_data.random_seq(2602, i, 100 + 7 * i, protein=False) for i in range(30)]
    subs[5] = q.copy()
    subs[11] = np.concatenate([subs[11][:50], q[20:390]])
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), m)
    prof = ps.Profile.new(q, False, m)
    scan = aligner(ps, "local", prof, 5, 2, trace=False, width=16).scan(db)
    hits = aligner(ps, "local", prof, 5, 2, width=16).align_subjects(db)
    assert hits.saturated[5] == 1 and hits.saturated.sum() >= 2
    assert np.array_equal(hits.saturated, scan.saturated)
    for k in KEYS3:
        assert np.array_equal(getattr(hits, k), getattr(scan, k)), k


def test_first_use_from_two_threads(ps):
    # the database is aligned from two other threads while its creating stream may still be packing: the first
    # call builds the inverse permutation behind the packing, the other waits for it
    b62 = ps.Matrix.from_name("blosum62")
    query = psb_data.random_seq(2041, 0, 300)
    cat, off = psb_data.protein_db(2042, 2043, 200000, query=query, planted_frac=0.01)
    ids = np.arange(0, 200000, 401)
    a = aligner(ps, "local", ps.Profile.new(query, False, b62))
    db = ps.Database((cat, off), b62)
    go = threading.Barrier(2)
    out, errors = [None, None], []

    def work(t):
        try:
            go.wait()
            out[t] = a.align_subjects(db, ids)
        except Exception as e:  # noqa: BLE001
            errors.append(repr(e))
    th = [threading.Thread(target=work, args=(t,)) for t in range(2)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert not errors, errors
    single = a.align_subjects(db, ids)
    for t in range(2):
        assert_same(out[t], single, TRACE_KEYS, f"thread {t}")


def test_errors(ps, c2):
    query, cat, off, b62, db = c2
    L = ps._lib.lib()
    prof = ps.Profile.new(query, False, b62)

    def call(name, ids, n, profile=prof):
        out = C.POINTER(ps.CBatch)()
        arr = None if ids is None else np.ascontiguousarray(ids, dtype=np.int64)
        rc = L.psb_db_align(name, profile.inner, 10, 1, db.inner, None if arr is None else arr.ctypes.data_as(C.c_void_p), n, C.byref(out))
        if rc == 0:
            L.psb_batch_free(out)
        return rc

    name = b"sw_trace_striped_profile_sat"
    assert call(name, [0, 1, db.n - 1], 3) == 0
    assert call(name, None, db.n) == 0
    assert call(name, [0, -1], 2) == PSB_EINVAL and "ids[1]" in ps._lib.last_error()
    assert call(name, [0, 1, 2, db.n], 4) == PSB_EINVAL and "ids[3]" in ps._lib.last_error()
    assert call(name, [0], 0) == PSB_EINVAL
    assert call(name, None, db.n - 1) == PSB_EINVAL
    assert call(b"sw_table_striped_profile_sat", [0], 1) == PSB_EUNSUPPORTED
    assert call(b"sw_rowcol_striped_profile_sat", [0], 1) == PSB_EUNSUPPORTED
    assert call(b"sw_trace_striped_sat", [0], 1) == PSB_EINVAL     # not a profile name
    dna_prof = ps.Profile.new(b"ACGTACGT", False, ps.Matrix.create(b"ACGT", 2, -3))
    assert call(name, [0], 1, dna_prof) == PSB_EINVAL                # another alphabet
    out = C.POINTER(ps.CBatch)()
    assert L.psb_scan(name, prof.inner, 10, 1, db.inner, C.byref(out)) == PSB_EUNSUPPORTED   # database scans stay score/stats only
    assert L.psb_db_subject(db.inner, db.n, None, 0) == PSB_EINVAL
    assert L.psb_db_subject(db.inner, 3, None, 0) == off[4] - off[3]
    with pytest.raises(ps.Panic):
        ps.Aligner.new().local().matrix(b62).use_trace().build().search(db, 10)
