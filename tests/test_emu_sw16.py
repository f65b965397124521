"""The packed 16-bit scan kernel source (csrc/kern_sw16.cuh) on the CPU SIMT emulation vs the
oracle: score, end_query, end_ref bit-exact; overflowing subjects must land on the retry list."""
import numpy as np
import pytest

import emu_harness
import psb_data


def check(oracle, mat, query, subjects, o, e, bits=5):
    outs, retry = emu_harness.sw16(query, subjects, mat, o, e, bits)
    for i, s in enumerate(subjects):
        if i in retry:
            continue
        exp = oracle.align(query, s, mat, mode=2, open=o, gap=e)
        got = (outs["score"][i], outs["end_query"][i], outs["end_ref"][i])
        assert got == (exp["score"], exp["end_query"], exp["end_ref"]), (i, len(query), len(s))
    return outs, retry


@pytest.mark.parametrize("lq", [40, 100, 400])
def test_protein_scan(oracle, blosum62, lq):
    q = psb_data.random_seq(7, 0, lq)
    subs = []
    for i in range(7):
        L = [35, 90, 91, 150, 17, 64, 33][i]
        if i % 2 == 0:
            seg = psb_data.mutate(q[: min(lq, L)], 7, 100 + i, 0.2, 0.05)[:L]
            s = np.concatenate([seg, psb_data.random_seq(8, i, max(0, L - len(seg)))])[:L]
        else:
            s = psb_data.random_seq(8, i, L)
        subs.append(s)
    _, retry = check(oracle, blosum62, q, subs, 10, 1)
    assert retry == []


def test_ties_and_zero(oracle):
    mat = oracle.Matrix.create(b"ACGT", 2, -3)
    q = np.frombuffer(b"ACTACGGG", dtype=np.uint8)
    subs = [np.frombuffer(s, dtype=np.uint8) for s in (b"ACTTAC", b"AC", b"TTTT", b"ACGGGACGGG", b"GG")]
    check(oracle, mat, q, subs, 5, 2)
    check(oracle, mat, q, subs, 0, 0)
    check(oracle, mat, q, subs, 5, 2, bits=5)


def test_overflow_goes_to_retry(oracle):
    # 400 matches at +100 exceed the 16-bit range: both subjects of that item are re-run at 32 bit,
    # everything else stays exact
    mat = oracle.Matrix.create(b"ACGT", 100, -90)
    q = psb_data.random_seq(9, 0, 400, protein=False)
    subs = [q.copy(), psb_data.random_seq(9, 1, 380, protein=False), psb_data.random_seq(9, 2, 60, protein=False),
            psb_data.random_seq(9, 3, 50, protein=False)]
    _, retry = check(oracle, mat, q, subs, 5, 2)
    assert retry == [0, 1]


def test_high_scores_stay_in_16_bit(oracle, blosum62):
    # an identical 400-aa protein scores ~2100: no re-run needed any more
    q = psb_data.random_seq(9, 0, 400)
    subs = [q.copy(), psb_data.random_seq(9, 1, 380), np.concatenate([psb_data.random_seq(9, 2, 60), q[50:300]])]
    outs, retry = check(oracle, blosum62, q, subs, 10, 1)
    assert retry == [] and outs["score"][0] > 2000


@pytest.mark.parametrize("lq,rows", [(100, 64), (130, 64), (300, 128), (400, 192)])
def test_strip_wise_scan_of_long_queries(oracle, blosum62, lq, rows):
    # queries longer than one strip: one sweep per strip, bottom rows handed over, per-strip bests merged with
    # (score, smaller end_ref, smaller end_query).  Every strip but the last is exactly 16*K rows high (the
    # bottom row of lane 15 must be a real query row)
    q = psb_data.random_seq(17, 0, lq)
    subs = []
    for i, L in enumerate([35, 90, 91, 150, 17, 64, 33, 200]):
        if i % 2 == 0:
            a = (i * 13) % max(1, lq - 30)
            seg = psb_data.mutate(q[a: a + L], 17, 100 + i, 0.2, 0.05)[:L]
            s = np.concatenate([seg, psb_data.random_seq(18, i, max(0, L - len(seg)))])[:L]
        else:
            s = psb_data.random_seq(18, i, L)
        subs.append(s)
    subs.append(np.concatenate([q[rows - 5: rows + 25], q[rows - 5: rows + 25]]))   # a match that straddles the strip boundary, twice
    outs, retry = emu_harness.sw16_strips(q, subs, blosum62, 10, 1, rows)
    assert retry == []
    for i, s in enumerate(subs):
        exp = oracle.align(q, s, blosum62, mode=2, open=10, gap=1)
        assert (outs["score"][i], outs["end_query"][i], outs["end_ref"][i]) == (exp["score"], exp["end_query"], exp["end_ref"]), (i, lq, len(s))


def test_strip_wise_scan_ties_across_strips(oracle):
    # the same maximum in two strips: the smaller end_ref must win whichever strip finds it
    mat = oracle.Matrix.create(b"ACGT", 2, -3)
    unit = np.frombuffer(b"ACGTTGCA", dtype=np.uint8)
    q = np.concatenate([unit, psb_data.random_seq(19, 0, 60, protein=False), unit, psb_data.random_seq(19, 1, 40, protein=False)])
    subs = [np.concatenate([psb_data.random_seq(19, 2, 11, protein=False), unit, psb_data.random_seq(19, 3, 9, protein=False)]),
            unit.copy(), np.concatenate([unit, unit]), psb_data.random_seq(19, 4, 50, protein=False)]
    outs, _ = emu_harness.sw16_strips(q, subs, mat, 5, 2, 64, bits=3)
    for i, s in enumerate(subs):
        exp = oracle.align(q, s, mat, mode=2, open=5, gap=2)
        assert (outs["score"][i], outs["end_query"][i], outs["end_ref"][i]) == (exp["score"], exp["end_query"], exp["end_ref"]), i


# ---- the re-run list: global sorted positions, the exact threshold, one entry per subject -------------------------
def sw16_limit(mat, o):
    """the packed kernel re-runs an item once a half's score reaches 32767 - open - max(S)"""
    return 32767 - o - int(np.max(mat.table))


def test_head_and_main_sub_ranges_push_global_positions(oracle):
    # the engine's launches over sorted positions: subject 0 routed elsewhere (not launched), a head launch over
    # positions 1..4 and a main launch over the rest; each launch's pointers start at its first position and its
    # re-run pushes add sid_base = first.  Overflowing subjects sit in both launches.  Gaps as dear as the matrix
    # allows (open + max(S) = 127) keep random subjects far below the limit: only the planted copies overflow.
    mat = oracle.Matrix.create(b"ACGT", 100, -90)
    o, e = 27, 27
    q = psb_data.random_seq(41, 0, 400, protein=False)
    lens = [900, 800, 700, 600, 520, 480, 450, 430, 410, 405, 300, 200, 150]   # distinct: the sort order is fixed
    subs = [psb_data.random_seq(42, i, L, protein=False) for i, L in enumerate(lens)]
    subs[2] = np.concatenate([psb_data.random_seq(43, 0, 300, protein=False), q])           # position 2: head
    subs[7] = np.concatenate([q, psb_data.random_seq(43, 1, 30, protein=False)])            # position 7: main
    caller = np.random.default_rng(44).permutation(len(subs))                                # caller order != sorted order
    shuffled = [subs[i] for i in caller]
    ranges = [(1, 4), (5, len(subs) - 5)]
    outs, pushed = emu_harness.sw16(q, shuffled, mat, o, e, ranges=ranges, raw=True)
    exp = [oracle.align(q, s, mat, mode=2, open=o, gap=e) for s in subs]
    over = [x["score"] >= sw16_limit(mat, o) for x in exp]
    assert over[2] and over[7] and sum(over) == 2
    want = set()
    for first, count in ranges:
        for a in range(first, first + count, 2):
            item = [s for s in (a, a + 1) if s < first + count]
            if any(over[s] for s in item):
                want.update(item)
    assert sorted(pushed) == sorted(want) == [1, 2, 7, 8]
    # sorted position s holds subs[s]; the caller passed it at index where(caller == s)
    where = {int(c): i for i, c in enumerate(caller)}
    for s in range(1, len(subs)):
        if s in want:
            continue
        i = where[s]
        assert (outs["score"][i], outs["end_query"][i], outs["end_ref"][i]) == (exp[s]["score"], exp[s]["end_query"], exp[s]["end_ref"]), s
    assert outs["score"][where[0]] == -777   # the routed subject is no launch's


def threshold_case(psb_data_seed, lq):
    """DNA +91/-91: a 359-residue core scores 359 * 91 = 32669.  The query is the core, or the core with random
    flanks (lq > 359); the first subject is the core itself, the others are shorter random subjects."""
    core = psb_data.random_seq(psb_data_seed, 0, 359, protein=False)
    pre = (lq - 359) // 3
    q = np.concatenate([psb_data.random_seq(psb_data_seed, 1, pre, protein=False), core,
                        psb_data.random_seq(psb_data_seed, 2, lq - 359 - pre, protein=False)])
    subs = [core.copy()] + [psb_data.random_seq(psb_data_seed, 3 + i, L, protein=False) for i, L in enumerate((300, 200, 100))]
    return q, subs


@pytest.mark.parametrize("lq,rows", [(359, None), (600, 256)])
def test_rerun_threshold_exactly(oracle, lq, rows):
    # limit = 32767 - open - 91: open 6 puts the score one below it (exact in 16 bit), open 7 on it, open 8 above
    mat = oracle.Matrix.create(b"ACGT", 91, -91)
    q, subs = threshold_case(31, lq)
    for o, rerun in ((6, False), (7, True), (8, True)):
        exp = [oracle.align(q, s, mat, mode=2, open=o, gap=1) for s in subs]
        assert exp[0]["score"] == 32669 and sw16_limit(mat, o) == 32669 + 1 - (o - 6)
        if rows is None:
            outs, retry = emu_harness.sw16(q, subs, mat, o, 1)
        else:
            outs, retry = emu_harness.sw16_strips(q, subs, mat, o, 1, rows)
        assert retry == ([0, 1] if rerun else []), o
        for i, s in enumerate(subs):
            if i not in retry:
                assert (outs["score"][i], outs["end_query"][i], outs["end_ref"][i]) == (exp[i]["score"], exp[i]["end_query"], exp[i]["end_ref"]), (o, i)


def test_strip_wise_rerun_lists_a_subject_once(oracle):
    # a 768-residue query in three strips of 256 rows; its copy overflows in strips 2 and 3.  Each subject of the
    # item goes on the re-run list once, not once per strip in which it is still over the limit.
    mat = oracle.Matrix.create(b"ACGT", 100, -90)
    q = psb_data.random_seq(9, 0, 768, protein=False)
    subs = [q.copy(), psb_data.random_seq(9, 1, 500, protein=False), psb_data.random_seq(9, 2, 60, protein=False),
            psb_data.random_seq(9, 3, 50, protein=False)]
    outs, retry = emu_harness.sw16_strips(q, subs, mat, 5, 2, 256)
    assert retry == [0, 1]
    for i in (2, 3):
        exp = oracle.align(q, subs[i], mat, mode=2, open=5, gap=2)
        assert (outs["score"][i], outs["end_query"][i], outs["end_ref"][i]) == (exp["score"], exp["end_query"], exp["end_ref"]), i
