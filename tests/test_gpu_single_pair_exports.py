"""The single-pair exports an unmodified parasail-rs reads after Aligner::align -- full tables (`_table`,
`_stats_table`), last row and column (`_rowcol`, `_stats_rowcol`), the trace table, the CIGAR and the traceback
strings -- against the CPU oracle, cell for cell.

Query lengths are chosen to cross every row-per-lane class and strip boundary of both kernel families: the coarse
family (K = 4 / 8 / 16 rows per lane, strips of 128 / 256 / 512 rows) that every table and row/column request takes,
and the fine family (K = 1 ... 16, strips of 32 K rows) that traces byte-sized scoring schemes.  Scoring schemes reach
each family: byte-sized DNA and BLOSUM62 schemes (fine trace), a matrix with values beyond a byte and a PSSM (coarse
trace, 32-bit values in the tables).  Failure messages name the pair's lengths, mode, end-gap flags, scheme and the
first differing cell (i, j)."""
import re

import numpy as np
import pytest

import psb_data
from test_oracle_properties import SG_FLAGS, cigar_rescore

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ps():
    import __graft_entry__ as g
    g.build()
    import parasail_rs_b200 as ps
    return ps


MODE_NAME = {0: "nw", 1: "sg", 2: "sw"}
ALL_FREE = (1, 1, 1, 1)
# scheme: (protein residues, gap open, gap extend)
SCHEMES = {
    "b62": (True, 10, 1),
    "dna5/2": (False, 5, 2),
    "dna4/4": (False, 4, 4),     # open == extend
    "dna1/4": (False, 1, 4),     # open < extend
    "dna0/0": (False, 0, 0),     # every gap decision a tie
    "big30/4": (False, 30, 4),   # match 200, mismatch -150: beyond a signed byte, coarse family
    "pssm": (True, 10, 1),       # BLOSUM62 converted to a PSSM of the query; the oracle uses the square matrix
}
FINE_SCHEMES = ("b62", "dna5/2", "dna4/4", "dna1/4", "dna0/0")
COARSE_SCHEMES = ("big30/4", "pssm")
PLANES = ("score", "matches", "similar", "length")


def matrices(ps, oracle, blosum62, scheme, q):
    """(product matrix, oracle matrix) of a scheme; a PSSM is built from the pair's own query"""
    if scheme == "b62":
        return ps.Matrix.from_name("blosum62"), blosum62
    if scheme == "pssm":
        return ps.Matrix.from_name("blosum62").to_pssm(q), blosum62
    if scheme == "big30/4":
        return ps.Matrix.create(b"ACGT", 200, -150), oracle.Matrix.create(b"ACGT", 200, -150)
    return ps.Matrix.create(b"ACGT", 2, -3), oracle.Matrix.create(b"ACGT", 2, -3)


def make_pair(seed, lq, lr, protein):
    """a query and a reference that holds a mutated copy of the query's tail after an unrelated prefix, cut or
    padded to lr: long diagonals, gaps, and overhangs at both ends so that every end-gap flag matters"""
    q = psb_data.random_seq(seed, 0, lq, protein)
    core = psb_data.mutate(q[lq // 5:], seed, 1, 0.12, 0.03, protein)
    r = np.concatenate([psb_data.random_seq(seed, 2, lr // 6, protein), core, psb_data.random_seq(seed, 3, lr, protein)])[:lr]
    return q, r


def aligner(ps, mode, flags, m, o, e, stats=False, out="", width=None, profile=None):
    b = getattr(ps.Aligner.new(), {0: "global_", 1: "semi_global", 2: "local"}[mode])()
    if mode == 1:
        b = b.allow_query_gaps([g for g, f in (("prefix", flags[0]), ("suffix", flags[1])) if f])
        b = b.allow_ref_gaps([g for g, f in (("prefix", flags[2]), ("suffix", flags[3])) if f])
    b = b.matrix(m).gap_open(o).gap_extend(e)
    if stats:
        b = b.use_stats()
    b = {"table": b.use_table, "rowcol": b.use_last_rowcol, "trace": b.use_trace}.get(out, lambda: b)()
    if width is not None:
        b = b.solution_width(width)
    if profile is not None:
        b = b.profile(profile)
    return b.build()


def oracle_align(oracle, q, r, om, mode, flags, o, e, **kw):
    return oracle.align(q, r, om, mode=mode, open=o, gap=e, s1_beg=flags[0], s1_end=flags[1], s2_beg=flags[2],
                        s2_end=flags[3], **kw)


def tag_of(lq, lr, mode, flags, scheme, what=""):
    return f"(lq, lr) = ({lq}, {lr}) {MODE_NAME[mode]} flags {flags} {scheme}{' ' + what if what else ''}"


def same(got, exp, what, tag, cell=None):
    """bit-exact; a 1-D export names its cell through `cell` (k -> (i, j))"""
    got, exp = np.asarray(got), np.asarray(exp)
    assert got.shape == exp.shape, f"{tag} {what}: shape {got.shape}, expected {exp.shape}"
    bad = np.argwhere(got != exp)
    if len(bad):
        at = tuple(int(x) for x in bad[0])
        ij = cell(at[0]) if cell else at
        raise AssertionError(f"{tag} {what}: {len(bad)} cells differ, first at (i, j) = {ij}: got {got[at]} expected {exp[at]}")


def check_getters(a, tag, table=False, rowcol=False, stats=False, trace=False):
    got = (a.is_table(), a.is_rowcol(), a.is_stats_table(), a.is_stats_rowcol(), a.is_trace(), a.is_stats())
    exp = (table, rowcol, stats and table, stats and rowcol, trace, stats)
    assert got == exp, f"{tag}: (is_table, is_rowcol, is_stats_table, is_stats_rowcol, is_trace, is_stats) = {got}, expected {exp}"
    assert not a.is_saturated(), tag


def check_result(a, exp, tag, stats=False):
    got = (a.get_score(), a.get_end_query(), a.get_end_ref())
    assert got == (exp["score"], exp["end_query"], exp["end_ref"]), f"{tag}: (score, end_query, end_ref) = {got}, oracle {exp['score'], exp['end_query'], exp['end_ref']}"
    if stats:
        got = (a.get_matches(), a.get_similar(), a.get_length())
        assert got == (exp["matches"], exp["similar"], exp["length"]), f"{tag}: (matches, similar, length) = {got}, oracle {exp['matches'], exp['similar'], exp['length']}"


# ---- tables and last row / column ------------------------------------------------------------------------------------
def check_tables(ps, oracle, blosum62, q, r, mode, flags, scheme, m=None, om=None):
    """_stats_table, _table, _stats_rowcol and _rowcol of one pair against the oracle and against each other.
    Returns the four results (for route comparisons)."""
    _, o, e = SCHEMES[scheme]
    if m is None:
        m, om = matrices(ps, oracle, blosum62, scheme, q)
    lq, lr = len(q), len(r)
    tag = tag_of(lq, lr, mode, flags, scheme)
    exp = oracle_align(oracle, q, r, om, mode, flags, o, e, tables=True, rowcol=True)
    row, col = (lambda j: (lq - 1, j)), (lambda i: (i, lr - 1))
    res = {}
    for stats in (True, False):
        planes = PLANES if stats else PLANES[:1]
        kind = "_stats_table" if stats else "_table"
        a = aligner(ps, mode, flags, m, o, e, stats=stats, out="table").align(q, r)
        check_getters(a, tag + " " + kind, table=True, stats=stats)
        check_result(a, exp, tag + " " + kind, stats)
        for p in planes:
            same(getattr(a, f"get_{p}_table")(), exp[f"{p}_table"], f"{kind} {p}_table", tag)
        if not stats:
            with pytest.raises(ps.NoStatsTable):
                a.get_matches_table()
        res[kind] = a
        kind = "_stats_rowcol" if stats else "_rowcol"
        b = aligner(ps, mode, flags, m, o, e, stats=stats, out="rowcol").align(q, r)
        check_getters(b, tag + " " + kind, rowcol=True, stats=stats)
        check_result(b, exp, tag + " " + kind, stats)
        for p in planes:
            same(getattr(b, f"get_{p}_row")(), exp[f"{p}_row"], f"{kind} {p}_row", tag, row)
            same(getattr(b, f"get_{p}_col")(), exp[f"{p}_col"], f"{kind} {p}_col", tag, col)
            # oracle-free: the row / column runs hand out the table run's last row / column
            t = getattr(a, f"get_{p}_table")()
            same(getattr(b, f"get_{p}_row")(), t[-1, :], f"{kind} {p}_row vs last row of the table", tag, row)
            same(getattr(b, f"get_{p}_col")(), t[:, -1], f"{kind} {p}_col vs last column of the table", tag, col)
        res[kind] = b
    if mode == 0:
        assert res["_table"].get_score_table()[-1, -1] == res["_table"].get_score(), f"{tag}: nw corner of the table is not the score"
    return res


TABLE_LQ = (1, 33, 128, 129, 256, 257, 511, 512, 513, 1024, 1025, 1537)
TABLE_SCHEMES = ("dna5/2", "b62", "big30/4", "pssm", "dna4/4", "dna1/4", "dna0/0")
# each query length meets a short and a long reference; the schemes rotate over the shapes
TABLE_SHAPES = [(lq, lr) for k, lq in enumerate(TABLE_LQ) for lr in ((1, 2, 31, 32, 33)[k % 5], (95, 300, 777)[k % 3])]
TABLE_CASES = [(mode, lq, lr, TABLE_SCHEMES[k % len(TABLE_SCHEMES)]) for k, (lq, lr) in enumerate(TABLE_SHAPES) for mode in (0, 2)]


@pytest.mark.parametrize("mode,lq,lr,scheme", TABLE_CASES, ids=[f"{MODE_NAME[c[0]]}-{c[1]}x{c[2]}-{c[3]}" for c in TABLE_CASES])
def test_tables_and_rowcol(ps, oracle, blosum62, mode, lq, lr, scheme):
    q, r = make_pair(7000 + lq * 3 + lr, lq, lr, SCHEMES[scheme][0])
    check_tables(ps, oracle, blosum62, q, r, mode, ALL_FREE, scheme)


# ---- trace table, CIGAR, traceback strings ---------------------------------------------------------------------------
_OPS = "MIDNSHP=X"


def cigar_words(text):
    return [int(n) << 4 | _OPS.index(op) for n, op in re.findall(r"(\d+)([MIDNSHP=X])", text)]


def check_rescore(ops, q, r, beg, a, om, mode, flags, o, e, tag):
    """oracle-free: the CIGAR re-scores to the pair's score and ends on its end cell.  A run of n gaps costs
    o + (n - 1) min(o, e): with open < extend every gap opens anew.  A walk that runs off the top (left) edge emits the
    rest of the reference (query) as one leading D (I) run, which costs what the boundary row (column) holds:
    nothing where that edge is free, o + (n - 1) e elsewhere."""
    if not ops or (mode == 2 and a.get_score() == 0):
        return
    sc, ei, ej, *_ = cigar_rescore(ops, q, r, beg[0], beg[1], om, o, min(o, e))
    top_free = mode == 2 or (mode == 1 and flags[0])
    left_free = mode == 2 or (mode == 1 and flags[2])
    first, n = ops[0] & 15, ops[0] >> 4
    if first in (1, 2):
        sc += o + (n - 1) * min(o, e)
        if not ((first == 2 and top_free) or (first == 1 and left_free)):
            sc -= o + (n - 1) * e
    assert (sc, ei, ej) == (a.get_score(), a.get_end_query(), a.get_end_ref()), \
        f"{tag}: the CIGAR re-scores to (score, end_query, end_ref) = {(sc, ei, ej)}, the result says {(a.get_score(), a.get_end_query(), a.get_end_ref())}"


def check_trace(ps, oracle, blosum62, q, r, mode, flags, scheme, m=None, om=None, table_twice=False):
    _, o, e = SCHEMES[scheme]
    if m is None:
        m, om = matrices(ps, oracle, blosum62, scheme, q)
    tag = tag_of(len(q), len(r), mode, flags, scheme, "_trace")
    exp = oracle_align(oracle, q, r, om, mode, flags, o, e, trace=True)
    a = aligner(ps, mode, flags, m, o, e, out="trace").align(q, r)
    check_getters(a, tag, trace=True)
    check_result(a, exp, tag)
    cig = a.get_cigar(q, r)
    if cig != exp["cigar"]:
        k = next((k for k, (x, y) in enumerate(zip(cig, exp["cigar"])) if x != y), min(len(cig), len(exp["cigar"])))
        raise AssertionError(f"{tag}: CIGAR differs from character {k}: got ...{cig[max(0, k - 20):k + 20]} expected ...{exp['cigar'][max(0, k - 20):k + 20]}")
    assert a.cigar_beg == (exp["beg_query"], exp["beg_ref"]), f"{tag}: CIGAR begins at {a.cigar_beg}, oracle {(exp['beg_query'], exp['beg_ref'])}"
    tb = a.get_traceback_strings(q, r)
    assert (tb.query, tb.comparison, tb.reference) == exp["traceback"], f"{tag}: traceback strings differ"
    for _ in range(2 if table_twice else 1):
        same(a.get_trace_table(), exp["trace"], "trace table", tag)
    check_rescore(cigar_words(cig), q, r, a.cigar_beg, a, om, mode, flags, o, e, tag)
    return a


FINE_K = (1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 12, 14, 16)
TRACE_LQ = [n for K in FINE_K for n in (32 * K, 32 * K + 1)] + [1000, 1600, 2047]
TRACE_LR = (1, 2, 31, 32, 33, 95, 300, 777)
TRACE_CASES = [(mode, lq, TRACE_LR[k % len(TRACE_LR)], FINE_SCHEMES[k % len(FINE_SCHEMES)])
               for k, lq in enumerate(TRACE_LQ) for mode in (0, 2)]
COARSE_TRACE_SHAPES = ((1, 95), (128, 33), (129, 300), (257, 31), (513, 777), (1025, 95), (1537, 300))
TRACE_CASES += [(mode, lq, lr, COARSE_SCHEMES[(k + mode // 2) % 2]) for k, (lq, lr) in enumerate(COARSE_TRACE_SHAPES) for mode in (0, 2)]


@pytest.mark.parametrize("mode,lq,lr,scheme", TRACE_CASES, ids=[f"{MODE_NAME[c[0]]}-{c[1]}x{c[2]}-{c[3]}" for c in TRACE_CASES])
def test_trace_exports(ps, oracle, blosum62, mode, lq, lr, scheme):
    q, r = make_pair(8000 + lq * 3 + lr, lq, lr, SCHEMES[scheme][0])
    check_trace(ps, oracle, blosum62, q, r, mode, ALL_FREE, scheme)


# ---- semi-global end-gap variants ------------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", SG_FLAGS, ids=["".join(map(str, f)) for f in SG_FLAGS])
def test_sg_flags_exports(ps, oracle, blosum62, flags):
    # every semi-global variant parasail defines, on a two-strip table pair (coarse K = 16), a two-strip fine trace
    # pair, a two-strip coarse trace pair and a small pair (tables and trace)
    q, r = make_pair(9001, 600, 300, False)
    check_tables(ps, oracle, blosum62, q, r, 1, flags, "dna5/2")
    q, r = make_pair(9002, 700, 250, True)
    check_trace(ps, oracle, blosum62, q, r, 1, flags, "b62")
    q, r = make_pair(9003, 530, 200, False)
    check_trace(ps, oracle, blosum62, q, r, 1, flags, "big30/4")
    q, r = make_pair(9004, 45, 60, False)
    check_tables(ps, oracle, blosum62, q, r, 1, flags, "dna4/4")
    check_trace(ps, oracle, blosum62, q, r, 1, flags, "dna0/0")


# ---- long pairs: traced wavefront walk, trace table from the lazy flag-byte re-run -------------------------------------
LONG_CASES = [(lq, lr, mode, flags) for lq, lr in ((2048, 2100), (2300, 700))
              for mode, flags in ((0, ALL_FREE), (2, ALL_FREE), (1, ALL_FREE), (1, (1, 0, 0, 1)), (1, (0, 1, 1, 0)))]


@pytest.mark.parametrize("lq,lr,mode,flags", LONG_CASES, ids=[f"{MODE_NAME[c[2]]}{''.join(map(str, c[3])) if c[2] == 1 else ''}-{c[0]}x{c[1]}" for c in LONG_CASES])
def test_long_pair_trace_exports(ps, oracle, blosum62, lq, lr, mode, flags):
    # queries of 2048 rows and more: CIGAR and begin coordinates come from the walk over the traced wavefront launch,
    # the table from the pair once more on the one-warp kernel when it is first asked for; it is asked for twice
    q, r = make_pair(9100 + lq + lr, lq, lr, False)
    check_trace(ps, oracle, blosum62, q, r, mode, flags, "dna5/2", table_twice=True)


# ---- residues outside the alphabet, other routes to the same exports --------------------------------------------------
def test_lower_case_and_unknown_letters(ps, oracle, blosum62):
    # lower-case letters score as their upper-case forms; letters outside the alphabet (J, O, U, ?, #) as the wildcard
    q, r = make_pair(9201, 300, 280, True)
    q, r = q.copy(), r.copy()
    q[::7] = np.frombuffer(bytes(q[::7]).lower(), dtype=np.uint8)
    r[3::5] = np.frombuffer(bytes(r[3::5]).lower(), dtype=np.uint8)
    q[::13] = np.frombuffer((b"JOU?#" * 10)[: len(q[::13])], dtype=np.uint8)
    r[5::17] = np.frombuffer((b"#?UOJ" * 10)[: len(r[5::17])], dtype=np.uint8)
    for mode in (0, 1, 2):
        check_tables(ps, oracle, blosum62, q, r, mode, ALL_FREE, "b62")
        check_trace(ps, oracle, blosum62, q, r, mode, ALL_FREE, "b62")


def exports(a, kind, q, r):
    """everything a result of this kind hands out"""
    out = {"ends": (a.get_score(), a.get_end_query(), a.get_end_ref())}
    if kind == "trace":
        out.update(cigar=a.get_cigar(q, r), beg=a.cigar_beg, trace=a.get_trace_table())
        tb = a.get_traceback_strings(q, r)
        out["tb"] = (tb.query, tb.comparison, tb.reference)
    else:
        out["stats"] = (a.get_matches(), a.get_similar(), a.get_length())
        for p in PLANES:
            if kind == "table":
                out[p] = getattr(a, f"get_{p}_table")()
            else:
                out[p] = (getattr(a, f"get_{p}_row")(), getattr(a, f"get_{p}_col")())
    return out


def same_exports(x, y, tag):
    assert x.keys() == y.keys(), tag
    for k in x:
        if isinstance(x[k], tuple) and x[k] and isinstance(x[k][0], np.ndarray):
            for g, h in zip(x[k], y[k]):
                same(g, h, k, tag)
        elif isinstance(x[k], np.ndarray):
            same(x[k], y[k], k, tag)
        else:
            assert x[k] == y[k], f"{tag} {k}: {x[k]} vs {y[k]}"


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_profile_route_equals_direct_route(ps, oracle, blosum62, mode):
    # Aligner.profile(Profile.new(q, stats, m)).align(None, r) -- the pfunction route -- hands out what the direct
    # route does: multi-strip coarse tables and row/column, a multi-strip fine trace
    b62 = ps.Matrix.from_name("blosum62")
    q, r = make_pair(9301, 700, 300, True)
    direct = check_tables(ps, oracle, blosum62, q, r, mode, ALL_FREE, "b62", b62, blosum62)
    for kind in ("table", "rowcol"):
        via = aligner(ps, mode, ALL_FREE, b62, 10, 1, out=kind, profile=ps.Profile.new(q, True, b62)).align(None, r)
        check_getters(via, f"profile route _stats_{kind}", table=kind == "table", rowcol=kind == "rowcol", stats=True)
        same_exports(exports(via, kind, q, r), exports(direct[f"_stats_{kind}"], kind, q, r), f"{MODE_NAME[mode]} profile route _stats_{kind}")
    a = check_trace(ps, oracle, blosum62, q, r, mode, ALL_FREE, "b62", b62, blosum62)
    via = aligner(ps, mode, ALL_FREE, b62, 10, 1, out="trace", profile=ps.Profile.new(q, False, b62)).align(None, r)
    same_exports(exports(via, "trace", q, r), exports(a, "trace", q, r), f"{MODE_NAME[mode]} profile route _trace")


@pytest.mark.parametrize("width", [32, 64])
def test_explicit_width_equals_sat(ps, oracle, blosum62, width):
    # an explicit 32- or 64-bit solution width computes exactly what `_sat` does
    b62 = ps.Matrix.from_name("blosum62")
    q, r = make_pair(9401, 600, 257, True)
    for mode in (0, 1, 2):
        for kind, stats in (("table", True), ("rowcol", True), ("trace", False)):
            sat = aligner(ps, mode, ALL_FREE, b62, 10, 1, stats=stats, out=kind).align(q, r)
            wide = aligner(ps, mode, ALL_FREE, b62, 10, 1, stats=stats, out=kind, width=width).align(q, r)
            assert not wide.is_saturated()
            same_exports(exports(wide, kind, q, r), exports(sat, kind, q, r), f"{MODE_NAME[mode]} _{kind} width {width}")
