"""Every launch route of the database scan (psb_scan) against the oracle: subjects routed to the wavefront kernel
(longer than 65 535), the head launch, the main launch, strip-wise long queries, and the 32-bit re-run of subjects
that leave the 16-bit range -- alone and together, at the exact boundaries between them.

Each case also asserts the route it was written for, from the `[psb] sw16:` line PSB_DEBUG_TIMING prints (nroute,
nhead), the launch count of the scan, or the piece line of a host-memory scan, so that a later change of a threshold
cannot move a case off its route unnoticed."""
import re

import numpy as np
import pytest

import psb_data

pytestmark = pytest.mark.gpu

KEYS3 = ("score", "end_query", "end_ref")
KEYS6 = KEYS3 + ("matches", "similar", "length")


@pytest.fixture(scope="module")
def ps():
    import __graft_entry__ as g
    g.build()
    import parasail_rs_b200 as ps
    return ps


# ---- how a case observes its route ----------------------------------------------------------------------------------
SW16_LINE = re.compile(r"\[psb\] sw16: n (\d+) residues (\d+) est \S+ ms long_len (\S+) nroute (\d+) nhead (\d+) top (\d+)")
PIECES_LINE = re.compile(r"\[psb\] scan_host\(dev \d+\): pieces \(MB\):([^;]*);")


def sw16_routes(err):
    """every `[psb] sw16: n ... nroute ... nhead ...` line of a scan's stderr, as dicts"""
    return [dict(n=int(m[1]), residues=int(m[2]), long_len=float(m[3]), nroute=int(m[4]), nhead=int(m[5]), top=int(m[6]))
            for m in SW16_LINE.finditer(err)]


def traced(fn, capfd, monkeypatch):
    """fn() with PSB_DEBUG_TIMING set; returns (its result, what it printed to stderr)"""
    monkeypatch.setenv("PSB_DEBUG_TIMING", "1")
    capfd.readouterr()
    try:
        out = fn()
    finally:
        monkeypatch.delenv("PSB_DEBUG_TIMING")
    return out, capfd.readouterr().err


def route_of(err):
    """the one packed-scan plan line of a resident scan; fails clearly if the scan did not take the packed path"""
    lines = sw16_routes(err)
    assert len(lines) == 1, f"expected one '[psb] sw16: n ... nroute ... nhead ...' line, got {len(lines)}:\n{err[-2000:]}"
    return lines[0]


def expected_nhead(lens, nroute, multi):
    """plan_scan's head for a database whose long-subject threshold is 1024 (asserted beside it): the subjects after
    the routed ones that are longer than 1024, rounded up to a multiple of 4, at most an eighth of the rest; none
    for a query of several strips"""
    if multi:
        return 0
    srt = sorted(lens, reverse=True)
    cnt = sum(1 for L in srt[nroute:] if L > 1024)
    return min((cnt + 3) // 4 * 4, (len(srt) - nroute) // 8 // 4 * 4)


def strip_count(lq):
    """strips of a packed scan: one per 400 query rows (sw16_prepare)"""
    return (lq + 399) // 400


def scan_traced(a, db, capfd, monkeypatch, nroute, nhead):
    """a.scan(db) with its route asserted: exactly nroute routed subjects and nhead head subjects"""
    got, err = traced(lambda: a.scan(db), capfd, monkeypatch)
    r = route_of(err)
    assert (r["nroute"], r["nhead"]) == (nroute, nhead), r
    return got, r


# ---- how a case checks its results ----------------------------------------------------------------------------------
def oracle_scan(oracle, query, cat, off, omat, mode=2, o=10, e=1, stats=False):
    return oracle.align_batch(query, np.array([0, len(query)]), cat, off, omat, mode=mode, open=o, gap=e, shared_query=True,
                              stats=stats, threads=0)


def oracle_some(oracle, query, cat, off, ids, omat, mode=2, o=10, e=1):
    """the oracle on the listed subjects only"""
    ids = np.asarray(sorted(set(int(i) for i in ids)), dtype=np.int64)
    sub = [cat[off[i]:off[i + 1]] for i in ids]
    c2, o2 = psb_data.concat(sub)
    return ids, oracle_scan(oracle, query, c2, o2, omat, mode, o, e)


def assert_same(got, exp, keys, tag="", ids=None):
    for k in keys:
        g = getattr(got, k) if ids is None else getattr(got, k)[ids]
        x = exp[k]
        if not np.array_equal(g, x):
            bad = np.nonzero(g != x)[0]
            at = bad[0] if ids is None else ids[bad[0]]
            raise AssertionError(f"{tag} {k}: {len(bad)} mismatches, first at subject {at}: got {g[bad[0]]} expected {x[bad[0]]}")


def assert_equal_results(a, b, keys=KEYS3, tag=""):
    for k in keys:
        x, y = getattr(a, k), getattr(b, k)
        if not np.array_equal(x, y):
            bad = np.nonzero(x != y)[0]
            raise AssertionError(f"{tag} {k}: {len(bad)} differences, first at subject {bad[0]}: {x[bad[0]]} against {y[bad[0]]}")


def host_paths_equal(ps, a, cat, off, ref, tag):
    """psb_scan_host from pageable and from page-locked memory, and psb_scan_box over all / one GPU, equal the
    resident scan; each piece is sorted, packed, routed and re-run on its own, so only the bounds of n_retried hold"""
    import torch
    pc = torch.empty(len(cat), dtype=torch.uint8, pin_memory=True); pc.numpy()[:] = cat
    po = torch.empty(len(off), dtype=torch.int64, pin_memory=True); po.numpy()[:] = off
    runs = [("pageable", lambda: a.scan_host((cat, off))), ("pinned", lambda: a.scan_host((pc.numpy(), po.numpy()))),
            ("box 0", lambda: a.scan_box((cat, off), 0)), ("box 1", lambda: a.scan_box((cat, off), 1))]
    nlong = int(np.sum(np.diff(off) > 65535))
    for name, run in runs:
        got = run()
        assert_equal_results(got, ref, KEYS3, f"{tag} {name}")
        assert nlong <= got.n_retried <= got.n, (tag, name, got.n_retried)


# ---- matrices -------------------------------------------------------------------------------------------------------
def protein(ps, oracle):
    return ps.Matrix.from_name("blosum62"), oracle.Matrix.from_table(psb_data.BLOSUM62_ALPHABET, psb_data.blosum62_table())


def dna(ps, oracle, match, mismatch):
    return ps.Matrix.create(b"ACGT", match, mismatch), oracle.Matrix.create(b"ACGT", match, mismatch)


def local_aligner(ps, prof, o, e, width="sat", mode="local"):
    return getattr(ps.Aligner.new(), mode)().gap_open(o).gap_extend(e).solution_width(width).profile(prof).build()


def rnd(seed, i, n, is_protein):
    return psb_data.random_seq(seed, i, n, protein=is_protein)


# ---- 1. routed subjects -----------------------------------------------------------------------------------------------
def routed_db(seed, q, nroute, is_protein, with_n=False, nshort=40):
    """subjects of 65 535 residues (packed; the query planted at its end, so the best cell is in the last column), and
    nroute routed ones of 65 536, 70 000, 66 000 residues (query planted inside), plus nshort short subjects"""
    lq = len(q)
    subs = [np.concatenate([rnd(seed, 1, 65535 - lq, is_protein), q])]
    for i, L in enumerate((65536, 70000, 66000)[:nroute]):
        seg = psb_data.mutate(q, seed, 10 + i, 0.1, 0.02, is_protein)
        a = 1000 + 20000 * i
        subs.append(np.concatenate([rnd(seed, 20 + i, a, is_protein), seg, rnd(seed, 30 + i, L - a - len(seg), is_protein)]))
    for i in range(nshort):
        L = 30 + 17 * i
        if i % 5 == 0:
            seg = q[: min(lq, L)]
            subs.append(np.concatenate([seg, rnd(seed, 40 + i, L - len(seg), is_protein)]))
        else:
            subs.append(rnd(seed, 40 + i, L, is_protein))
    if with_n:
        for s in subs[:3]:
            s[7] = ord("N")
    order = np.random.default_rng(seed).permutation(len(subs))
    subs = [subs[i] for i in order]
    return psb_data.concat(subs)


ROUTED_CASES = [  # (query length, routed subjects, alphabet)
    (17, 1, "protein"), (64, 2, "protein"), (65, 3, "protein"), (400, 1, "protein"), (401, 2, "protein"), (1601, 3, "protein"),
    (64, 3, "dna2"), (401, 1, "dna2"), (17, 2, "dna3"), (401, 3, "dna3"),
]


@pytest.mark.parametrize("lq,nroute,alpha", ROUTED_CASES)
def test_routed_subjects(ps, oracle, lq, nroute, alpha, capfd, monkeypatch):
    # queries of <= 64 residues run the route with K = 1, longer ones with K = 2; 401 and 1601 residues add the
    # strip-wise launches, whose boundary lines start at an offset of nroute subjects
    is_protein = alpha == "protein"
    m, om = protein(ps, oracle) if is_protein else dna(ps, oracle, 2, -3)
    o, e = (10, 1) if is_protein else (5, 2)
    q = rnd(700 + lq, 0, lq, is_protein)
    cat, off = routed_db(710 + lq, q, nroute, is_protein, with_n=alpha == "dna3")
    lens = np.diff(off)
    db = ps.Database((cat, off), m)
    assert db.bits == {"protein": 5, "dna2": 2, "dna3": 3}[alpha]
    a = local_aligner(ps, ps.Profile.new(q, False, m), o, e)
    multi = strip_count(lq) > 1
    got, r = scan_traced(a, db, capfd, monkeypatch, nroute, expected_nhead(lens, nroute, multi))
    assert r["long_len"] == 1024 and r["top"] == lens.max()
    if multi:
        assert ps.launches() == 3 + strip_count(lq) + 1   # route (unpack, sweep, reduce), one per strip, re-run
    exp = oracle_scan(oracle, q, cat, off, om, o=o, e=e)
    assert_same(got, exp, KEYS3, f"lq {lq} nroute {nroute} {alpha}")
    assert got.n_retried == nroute
    i65535 = int(np.nonzero(lens == 65535)[0][0])
    assert got.end_ref[i65535] == 65534 and got.end_query[i65535] == lq - 1
    if (lq, nroute) in ((64, 2), (401, 2)):
        host_paths_equal(ps, a, cat, off, got, f"routed lq {lq}")


@pytest.mark.parametrize("lq", [64, 401])
def test_every_subject_routed(ps, oracle, lq, capfd, monkeypatch):
    # no subject left for the packed kernel (nshort == 0): the route alone fills the results
    m, om = protein(ps, oracle)
    q = rnd(720, lq, lq, True)
    subs = [np.concatenate([rnd(721, i, 2000 + 3000 * i, True), psb_data.mutate(q, 722, i, 0.1, 0.02), rnd(723, i, L, True)])
            for i, L in enumerate((64000, 66000, 68000))]
    cat, off = psb_data.concat(subs)
    a = local_aligner(ps, ps.Profile.new(q, False, m), 10, 1)
    got, _ = scan_traced(a, ps.Database((cat, off), m), capfd, monkeypatch, 3, 0)
    assert_same(got, oracle_scan(oracle, q, cat, off, om), KEYS3, f"all routed lq {lq}")
    assert got.n_retried == 3


# ---- 2. head, main and routed launches together, with 16-bit re-runs in each ----------------------------------------
def mixed_db(seed, q):
    """one routed subject (70 000), 8 head subjects (3 000 .. 2 300) and 80 main subjects (1 000 .. 131), all of distinct
    lengths, so that the sorted order -- and with it the pairing into items -- is fixed.  Copies of the query sit in
    the routed subject, at sorted position 3 (head) and at sorted position 20 (main).  Returns cat, off, and the caller
    id of every sorted position."""
    lq = len(q)
    lens = [70000] + [3000 - 100 * i for i in range(8)] + [1000 - 11 * i for i in range(80)]
    subs = [rnd(seed, i, L, False) for i, L in enumerate(lens)]
    for pos in (0, 3, 20):
        a = (len(subs[pos]) - lq) // 3
        subs[pos] = np.concatenate([subs[pos][:a], q, subs[pos][a + lq:]])
        assert len(subs[pos]) == lens[pos]
    caller = np.random.default_rng(seed).permutation(len(subs))   # caller id of sorted position s: where(caller == s)
    cat, off = psb_data.concat([subs[i] for i in caller])
    pos_to_id = np.argsort(caller)
    return cat, off, pos_to_id


def items_with(pos, first, count):
    """the item (pair of adjacent sorted positions, counted from the launch's first subject) that holds `pos`"""
    a = first + (pos - first) // 2 * 2
    return [s for s in (a, a + 1) if s < first + count]


@pytest.mark.parametrize("lq", [400, 800])
def test_head_main_and_routed_with_reruns(ps, oracle, lq, capfd, monkeypatch):
    # single strip: head launch over sorted positions 1..8, main launch over 9..88, each with an overflowing item;
    # 800 residues: two strip launches over positions 1..88.  Every re-run pushes its launch's first position plus
    # the index inside the launch (sid_base), so every result must come back exact.
    # Penalties: gaps as dear as the packed profile allows keep random subjects far below the 16-bit limit.
    match, o, e = (100, 27, 27) if lq == 400 else (60, 60, 60)
    m, om = dna(ps, oracle, match, -90 if lq == 400 else -60)
    q = rnd(730, lq, lq, False)
    cat, off, pos_to_id = mixed_db(731 + lq, q)
    n = len(off) - 1
    db = ps.Database((cat, off), m)
    a = local_aligner(ps, ps.Profile.new(q, False, m), o, e)
    multi = lq > 400
    got, r = scan_traced(a, db, capfd, monkeypatch, 1, 0 if multi else 8)
    assert r["long_len"] == 1024
    exp = oracle_scan(oracle, q, cat, off, om, o=o, e=e)
    assert_same(got, exp, KEYS3, f"mixed lq {lq}")
    limit = 32767 - o - match
    over = [s for s in range(n) if exp["score"][pos_to_id[s]] >= limit]
    assert over == [0, 3, 20], over
    launches = [(1, n - 1)] if multi else [(1, 8), (9, n - 9)]
    items = set()
    for s in over[1:]:
        first, count = next(fc for fc in launches if fc[0] <= s < fc[0] + fc[1])
        items.add(tuple(items_with(s, first, count)))
    assert items == {(3, 4), (19, 20)}
    assert got.n_retried == 1 + sum(len(t) for t in items)
    if multi:
        assert ps.launches() == 3 + 2 + 1
    host_paths_equal(ps, a, cat, off, got, f"mixed lq {lq}")


# ---- 3. the re-run threshold exactly ----------------------------------------------------------------------------------
@pytest.mark.parametrize("lq", [359, 600])
def test_rerun_threshold_exactly(ps, oracle, lq, capfd, monkeypatch):
    # DNA +91/-91, gap 1: a 359-residue core scores 32 669.  The limit is 32 767 - open - 91: open 6 leaves the score
    # one below it (exact in 16 bit, no re-run), open 7 puts it on the limit and open 8 above (both re-run)
    m, om = dna(ps, oracle, 91, -91)
    core = rnd(740, 0, 359, False)
    pre = (lq - 359) // 3
    q = np.concatenate([rnd(740, 1, pre, False), core, rnd(740, 2, lq - 359 - pre, False)])
    subs = [core.copy()] + [rnd(741, i, 300 - 7 * i, False) for i in range(30)]
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), m)
    prof = ps.Profile.new(q, False, m)
    for o, rerun in ((6, False), (7, True), (8, True)):
        got, _ = scan_traced(local_aligner(ps, prof, o, 1), db, capfd, monkeypatch, 0, 0)
        exp = oracle_scan(oracle, q, cat, off, om, o=o, e=1)
        assert exp["score"][0] == 32669 and 32767 - o - 91 == 32670 - (o - 6)
        assert_same(got, exp, KEYS3, f"threshold lq {lq} open {o}")
        assert got.n_retried == (2 if rerun else 0), (o, got.n_retried)
        if lq > 400:
            assert ps.launches() == strip_count(lq) + 1


# ---- 4. strip-wise queries ---------------------------------------------------------------------------------------------
def strip_rows(lq):
    """rows of every strip but the last (sw16_prepare): the smallest class of 16 * K rows whose strips cover the query"""
    s = strip_count(lq)
    if s == 1:
        return lq
    return next(16 * k for k in (12, 16, 20, 25) if 16 * k * s >= lq)


STRIP_LENGTHS = [400, 401, 768, 769, 800, 801, 1200, 1201, 6400]


@pytest.mark.parametrize("lq", STRIP_LENGTHS)
def test_strip_wise_query_lengths(ps, oracle, lq, capfd, monkeypatch):
    # segments planted across every strip boundary, mutated, in a small protein database
    m, om = protein(ps, oracle)
    q = rnd(750, lq, lq, True)
    rows = strip_rows(lq)
    subs = [rnd(751, i, 40 + 9 * i, True) for i in range(60)]
    for k, b in enumerate(range(rows, lq, rows)):
        seg = psb_data.mutate(q[max(0, b - 60): b + 60], 752, k, 0.1, 0.03)
        subs.append(np.concatenate([rnd(753, k, 25, True), seg, rnd(754, k, 15, True)]))
    subs.append(q[-150:].copy())
    cat, off = psb_data.concat(subs)
    a = local_aligner(ps, ps.Profile.new(q, False, m), 10, 1)
    got, _ = scan_traced(a, ps.Database((cat, off), m), capfd, monkeypatch, 0, 0)
    assert ps.launches() == (strip_count(lq) if lq > 400 else 1) + 1
    assert_same(got, oracle_scan(oracle, q, cat, off, om), KEYS3, f"strip-wise lq {lq}")
    assert got.n_retried == 0
    if lq in (801, 1201):
        host_paths_equal(ps, a, cat, off, got, f"strip-wise lq {lq}")


def test_query_beyond_sixteen_strips_takes_the_32_bit_scan(ps, oracle, capfd, monkeypatch):
    # 6 401 residues need 17 strips: no packed profile, the whole scan runs on the 32-bit kernel (no sw16 line)
    m, om = protein(ps, oracle)
    q = rnd(755, 0, 6401, True)
    subs = [rnd(756, i, 50 + 7 * i, True) for i in range(40)] + [q[6000:6300].copy(), q[100:300].copy()]
    cat, off = psb_data.concat(subs)
    a = local_aligner(ps, ps.Profile.new(q, False, m), 10, 1)
    got, err = traced(lambda: a.scan(ps.Database((cat, off), m)), capfd, monkeypatch)
    assert sw16_routes(err) == [], err[-2000:]
    assert ps.launches() == 1
    assert_same(got, oracle_scan(oracle, q, cat, off, om), KEYS3, "6401")


def test_strip_wise_rerun_counts_each_subject_once(ps, oracle, capfd, monkeypatch):
    # a 1 200-residue query in three strips; its copy (DNA +60/-60) leaves the 16-bit range in strips 2 and 3.  The
    # item is re-run once: n_retried counts the distinct re-run subjects (2), never more than the database holds
    m, om = dna(ps, oracle, 60, -60)
    q = rnd(760, 0, 1200, False)
    subs = [rnd(761, i, 900 - 13 * i, False) for i in range(40)]
    subs[6] = np.concatenate([rnd(762, 0, 100, False), q])
    cat, off = psb_data.concat(subs)
    a = local_aligner(ps, ps.Profile.new(q, False, m), 60, 60)
    got, _ = scan_traced(a, ps.Database((cat, off), m), capfd, monkeypatch, 0, 0)
    assert ps.launches() == 3 + 1
    exp = oracle_scan(oracle, q, cat, off, om, o=60, e=60)
    assert_same(got, exp, KEYS3, "strip-wise re-run")
    assert exp["score"][6] == 72000 and np.sum(exp["score"] >= 32767 - 60 - 60) == 1
    assert got.n_retried == 2 <= got.n


# ---- 5. ties through psb_scan ---------------------------------------------------------------------------------------------
def test_ties_through_the_scan(ps, oracle, capfd, monkeypatch):
    m, om = dna(ps, oracle, 2, -3)
    unit = np.frombuffer(b"ACGTTGCAAGCT", dtype=np.uint8)
    q = np.concatenate([rnd(770, 0, 40, False), unit, rnd(770, 1, 60, False)])
    subs = [
        # the query segment several times in one subject: the smallest end_ref wins
        np.concatenate([rnd(771, 0, 30, False), unit, rnd(771, 1, 20, False), unit, rnd(771, 2, 9, False), unit]),
        # equal maxima in both subjects of one word: adjacent in sorted order (lengths 300 and 150, nothing in
        # between), the same first 150 columns with the segment in them; the shorter subject's pad columns lie past
        # its end, where the longer one goes on
        np.concatenate([rnd(772, 0, 60, False), unit, rnd(772, 1, 300 - 60 - len(unit), False)]),
    ] + [rnd(774, i, 20 + i, False) for i in range(20)]
    subs.insert(2, subs[1][:150].copy())
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), m)
    prof = ps.Profile.new(q, False, m)
    got, _ = scan_traced(local_aligner(ps, prof, 5, 2), db, capfd, monkeypatch, 0, 0)
    exp = oracle_scan(oracle, q, cat, off, om, o=5, e=2)
    assert_same(got, exp, KEYS3, "ties")
    assert exp["score"][1] == exp["score"][2] and exp["end_ref"][1] == exp["end_ref"][2] < 150
    # a homopolymer: every cell of a diagonal band ties; at 0/0 and at open == gap
    hq = np.full(50, ord("A"), dtype=np.uint8)
    hs = [np.full(L, ord("A"), dtype=np.uint8) for L in (80, 50, 49, 17)] + [rnd(775, i, 30, False) for i in range(6)]
    hcat, hoff = psb_data.concat(hs)
    hdb = ps.Database((hcat, hoff), m)
    hprof = ps.Profile.new(hq, False, m)
    for o, e in ((0, 0), (3, 3)):
        got, _ = scan_traced(local_aligner(ps, hprof, o, e), hdb, capfd, monkeypatch, 0, 0)
        assert_same(got, oracle_scan(oracle, hq, hcat, hoff, om, o=o, e=e), KEYS3, f"homopolymer {o}/{e}")
    # equal maxima in two strips: the unit at query rows 100 and 700 (strips 1 and 3 of 320 rows)
    lq = 900
    sq = rnd(776, 0, lq, False)
    sq[100:100 + len(unit)] = unit; sq[700:700 + len(unit)] = unit
    ss = [np.concatenate([rnd(777, 0, 25, False), unit, rnd(777, 1, 13, False)]), unit.copy(),
          np.concatenate([unit, rnd(777, 2, 5, False), unit])] + [rnd(778, i, 40 + i, False) for i in range(10)]
    scat, soff = psb_data.concat(ss)
    got, _ = scan_traced(local_aligner(ps, ps.Profile.new(sq, False, m), 5, 2), ps.Database((scat, soff), m), capfd,
                         monkeypatch, 0, 0)
    assert ps.launches() == strip_count(lq) + 1
    assert_same(got, oracle_scan(oracle, sq, scat, soff, om, o=5, e=2), KEYS3, "ties across strips")


# ---- 6. penalty edges of the packed path, and its per-open profile cache ------------------------------------------
def test_penalty_edges_and_profile_cache(ps, oracle, capfd, monkeypatch):
    # the packed profile holds S + open in a byte: open + max(S) = 127 stays packed, 128 takes the 32-bit scan;
    # open < gap is not packed either; open == gap and 0/0 are
    m, om = protein(ps, oracle)
    q = rnd(780, 0, 300, True)
    cat, off = psb_data.protein_db(781, 782, 300, query=q, planted_frac=0.1)
    db = ps.Database((cat, off), m)
    prof = ps.Profile.new(q, False, m)
    for o, e, packed in ((116, 1, True), (117, 1, False), (3, 5, False), (4, 4, True), (0, 0, True)):
        got, err = traced(lambda: local_aligner(ps, prof, o, e).scan(db), capfd, monkeypatch)
        assert len(sw16_routes(err)) == (1 if packed else 0), (o, e, err[-2000:])
        assert_same(got, oracle_scan(oracle, q, cat, off, om, o=o, e=e), KEYS3, f"open {o} gap {e}")
    # one Profile, packed once per gap-open value: 10/1, 11/1, then 10/1 again from the cache
    for o in (10, 11, 10):
        got, _ = scan_traced(local_aligner(ps, prof, o, 1), db, capfd, monkeypatch, 0, expected_nhead(np.diff(off), 0, False))
        assert_same(got, oracle_scan(oracle, q, cat, off, om, o=o, e=1), KEYS3, f"cached profile open {o}")


# ---- 7. explicit solution widths on a scan ---------------------------------------------------------------------------
def test_explicit_widths_on_a_scan(ps, oracle, capfd, monkeypatch):
    # _8 / _16 run the packed path, then flag what does not fit: a local score s saturates a width of b bits when
    # s + max(S) > 2^(b-1) - 1; such a subject is flagged and its score and ends are zeroed.  _32 / _64 run the
    # 32-bit scan and equal _sat.
    m, om = dna(ps, oracle, 100, -90)
    q = rnd(790, 0, 400, False)
    subs = [rnd(791, i, 30 + 9 * i, False) for i in range(40)]
    subs[4] = q.copy()                                   # 40 000: saturates 16 bit too
    subs[9] = q[:2].copy()                               # 200: saturates 8 bit only, as every random subject does
    subs[13] = np.full(25, ord("N"), dtype=np.uint8)     # no residue of the query: 0 fits 8 bit
    subs[17] = np.full(60, ord("N"), dtype=np.uint8)
    cat, off = psb_data.concat(subs)
    db = ps.Database((cat, off), m)
    prof = ps.Profile.new(q, False, m)
    sat, _ = scan_traced(local_aligner(ps, prof, 27, 27), db, capfd, monkeypatch, 0, 0)
    assert_same(sat, oracle_scan(oracle, q, cat, off, om, o=27, e=27), KEYS3, "sat")
    for width, hi in ((8, 127), (16, 32767)):
        got, _ = scan_traced(local_aligner(ps, prof, 27, 27, width), db, capfd, monkeypatch, 0, 0)
        flagged = sat.score.astype(np.int64) + 100 > hi
        assert flagged.any() and not flagged.all()
        assert np.array_equal(got.saturated.astype(bool), flagged), width
        for k in KEYS3:
            assert np.all(getattr(got, k)[flagged] == 0) and np.array_equal(getattr(got, k)[~flagged], getattr(sat, k)[~flagged]), (width, k)
    for width in (32, 64):
        got, err = traced(lambda: local_aligner(ps, prof, 27, 27, width).scan(db), capfd, monkeypatch)
        assert sw16_routes(err) == []
        assert_equal_results(got, sat, KEYS3, f"width {width}")


# ---- 8. the 32-bit scan -------------------------------------------------------------------------------------------------
SCAN_MODES = [("global_", 0), ("semi_global", 1), ("local", 2)]


@pytest.mark.parametrize("mode,om_", SCAN_MODES)
def test_32_bit_scan_with_statistics(ps, oracle, mode, om_, capfd, monkeypatch):
    # statistics take the 32-bit scan.  Narrow statistics word: a 300-residue query against subjects of at most
    # 1 000; wide: a 1 100-residue query (min(lq, maxlen) >= 1024) against subjects of 5 000 and 70 000 residues,
    # a query longer than 32 * K rows of the largest class, so strips hand their bottom rows over through scratch
    m, om = protein(ps, oracle)
    for lq, lens in ((300, [1000, 700] + [40 + 9 * i for i in range(30)]), (1100, [70000, 5000] + [40 + 9 * i for i in range(30)])):
        q = rnd(800, lq, lq, True)
        subs = [rnd(801, i, L, True) for i, L in enumerate(lens)]
        for i in (0, 1, 5):
            seg = psb_data.mutate(q[lq // 4: lq // 4 + min(250, len(subs[i]) - 20)], 802, i, 0.1, 0.03)
            subs[i] = np.concatenate([subs[i][:10], seg, subs[i][10 + len(seg):]])[:lens[i]]
        cat, off = psb_data.concat(subs)
        db = ps.Database((cat, off), m)
        for stats in (False, True):
            a = getattr(ps.Aligner.new(), mode)().gap_open(10).gap_extend(1).profile(ps.Profile.new(q, stats, m)).build()
            if not stats and mode == "local":
                continue
            got, err = traced(lambda: a.scan(db), capfd, monkeypatch)
            assert sw16_routes(err) == [] and ps.launches() == 1
            exp = oracle_scan(oracle, q, cat, off, om, mode=om_, stats=stats)
            assert_same(got, exp, KEYS6 if stats else KEYS3, f"{mode} lq {lq} stats {stats}")


def test_32_bit_scan_with_a_pssm(ps, oracle, capfd, monkeypatch):
    # a PSSM profile is never packed: the scan reads it through the coarse kernel family
    m, om = protein(ps, oracle)
    q = rnd(810, 0, 700, True)
    pssm = m.to_pssm(q)
    cat, off = psb_data.protein_db(811, 812, 200, query=q[:300], planted_frac=0.1)
    db = ps.Database((cat, off), m)
    for mode, om_ in SCAN_MODES:
        a = getattr(ps.Aligner.new(), mode)().gap_open(10).gap_extend(1).profile(ps.Profile.new(q, False, pssm)).build()
        got, err = traced(lambda: a.scan(db), capfd, monkeypatch)
        assert sw16_routes(err) == []
        assert_same(got, oracle_scan(oracle, q, cat, off, om, mode=om_), KEYS3, f"pssm {mode}")


# ---- 9. a host-memory scan of several pieces, with a routed and an overflowing subject in a later piece -------------
def test_host_scan_pieces_with_routed_and_rerun_subjects(ps, oracle, capfd, monkeypatch):
    m, om = dna(ps, oracle, 100, -90)
    o, e = 27, 27
    q = rnd(820, 0, 400, False)
    n_bulk = 160000                                        # ~59 MB of DNA subjects, 280 .. 460 residues
    lens = 280 + (np.arange(n_bulk) * 7919) % 181
    bulk = rnd(821, 0, int(lens.sum()), False)
    tail = [np.concatenate([rnd(822, 0, 30000, False), q, rnd(822, 1, 40000, False)]),   # routed, 70 400
            np.concatenate([rnd(823, 0, 50, False), q]), rnd(824, 0, 449, False)]        # overflows; its partner
    tcat, toff = psb_data.concat(tail)
    cat = np.concatenate([bulk, tcat])
    off = np.concatenate([np.concatenate([[0], np.cumsum(lens)]), toff[1:] + lens.sum()]).astype(np.int64)
    n = len(off) - 1
    assert cat.nbytes >= 40 * 2 ** 20
    a = local_aligner(ps, ps.Profile.new(q, False, m), o, e)
    ref, r = scan_traced(a, ps.Database((cat, off), m), capfd, monkeypatch, 1, 0)
    w32 = local_aligner(ps, ps.Profile.new(q, False, m), o, e, 32).scan(ps.Database((cat, off), m))
    assert_equal_results(ref, w32, KEYS3, "packed against 32-bit")
    sample = list(np.random.default_rng(825).choice(n_bulk, 300, replace=False)) + [n - 3, n - 2, n - 1]
    ids, exp = oracle_some(oracle, q, cat, off, sample, om, o=o, e=e)
    assert_same(ref, exp, KEYS3, "host db sample", ids)
    assert ref.score[n - 3] == 40000 and ref.score[n - 2] == 40000
    assert ref.n_retried == 3
    for name, run in (("pageable", lambda: a.scan_host((cat, off))), ("box", lambda: a.scan_box((cat, off), 1))):
        got, err = traced(run, capfd, monkeypatch)
        pieces = PIECES_LINE.findall(err)
        if name == "pageable":
            assert pieces and len(pieces[0].split()) >= 2, err[-2000:]
            assert sum(x["nroute"] for x in sw16_routes(err)) == 1
        assert_equal_results(got, ref, KEYS3, f"host {name}")
        assert 1 <= got.n_retried <= n
