"""The general 32-bit kernel source (csrc/kern_gotoh32.cuh), stepped on CPU threads through the
SIMT emulation, must agree with the oracle bit for bit: score, ends, stats, trace bytes."""
import numpy as np
import pytest

import emu_harness
import psb_data
from test_oracle_properties import SG_FLAGS, rand_pair


def compare(oracle, mat, qs, rs, K, mode, o, e, flags=(1, 1, 1, 1), stats=False, trace=False, wide=False, profile=False):
    got = emu_harness.gotoh32(qs, rs, mat, K, mode, o, e, flags, stats, trace, wide, profile=profile)
    for i, (q, r) in enumerate(zip(qs, rs)):
        exp = oracle.align(q, r, mat, mode=mode, open=o, gap=e, s1_beg=flags[0], s1_end=flags[1],
                           s2_beg=flags[2], s2_end=flags[3], trace=trace)
        tag = (i, K, mode, flags, len(q), len(r))
        assert (got["score"][i], got["end_query"][i], got["end_ref"][i]) == (exp["score"], exp["end_query"], exp["end_ref"]), tag
        if stats:
            assert (got["matches"][i], got["similar"][i], got["length"][i]) == (exp["matches"], exp["similar"], exp["length"]), tag
        if trace:
            assert np.array_equal(got["trace"][i], exp["trace"]), tag


def pairs(seed, n, lq_rng, lr_rng, protein):
    rng = np.random.default_rng(seed)
    qs, rs = [], []
    for i in range(n):
        q, r = rand_pair(seed, i, int(rng.integers(*lq_rng)), int(rng.integers(*lr_rng)), protein)
        qs.append(q); rs.append(r)
    return qs, rs


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("K", [1, 2, 4])
def test_score_ends_protein(oracle, blosum62, mode, K):
    qs, rs = pairs(11 + K, 4, (1, 150), (1, 90), True)   # several strips for small K
    compare(oracle, blosum62, qs, rs, K, mode, 10, 1)


@pytest.mark.parametrize("flags", SG_FLAGS)
def test_sg_flags(oracle, flags):
    mat = oracle.Matrix.create(b"ACGT", 2, -3)
    qs, rs = pairs(21, 3, (1, 70), (1, 70), False)
    compare(oracle, mat, qs, rs, 2, 1, 5, 2, flags)


@pytest.mark.parametrize("gaps", [(0, 0), (3, 3), (1, 4)])
def test_odd_gap_penalties(oracle, dna_default, gaps):
    qs, rs = pairs(31, 3, (1, 60), (1, 60), False)
    for mode in (0, 1, 2):
        compare(oracle, dna_default, qs, rs, 2, mode, gaps[0], gaps[1], stats=True)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("wide", [False, True])
def test_stats(oracle, blosum62, mode, wide):
    qs, rs = pairs(41, 3, (1, 140), (1, 80), True)
    compare(oracle, blosum62, qs, rs, 3, mode, 10, 1, stats=True, wide=wide)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("K", [2, 8])
def test_trace(oracle, blosum62, mode, K):
    qs, rs = pairs(51, 3, (1, 100), (1, 60), True)
    compare(oracle, blosum62, qs, rs, K, mode, 10, 1, trace=True)


def test_planted_ties(oracle):
    mat = oracle.Matrix.create(b"ACGT", 2, -3)
    qs = [np.frombuffer(b"AC", dtype=np.uint8), np.frombuffer(b"ACTAC", dtype=np.uint8),
          np.frombuffer(b"TTAC", dtype=np.uint8), np.frombuffer(b"ACGTACGTACGTACGTACGTACGTACGTACGTACGTACGT" * 3, dtype=np.uint8)]
    rs = [np.frombuffer(b"ACTTAC", dtype=np.uint8), np.frombuffer(b"AC", dtype=np.uint8),
          np.frombuffer(b"ACGG", dtype=np.uint8), np.frombuffer(b"ACGTACGT" * 9, dtype=np.uint8)]
    for mode in (0, 1, 2):
        compare(oracle, mat, qs, rs, 1, mode, 5, 2, stats=True)
        compare(oracle, mat, qs, rs, 2, mode, 0, 0)


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("variant", ["score", "stats", "trace"])
def test_per_warp_profile_variant(oracle, blosum62, mode, variant):
    # the PROF=true instantiation (int8 per-warp query profile instead of matrix reads)
    qs, rs = pairs(61, 3, (1, 150), (1, 80), True)
    compare(oracle, blosum62, qs, rs, 3, mode, 10, 1, stats=variant == "stats", trace=variant == "trace", profile=True)
    mat = oracle.Matrix.create(b"ACGT", 2, -3)
    qs, rs = pairs(62, 3, (1, 90), (1, 90), False)
    compare(oracle, mat, qs, rs, 2, mode, 0, 0, stats=variant == "stats", trace=variant == "trace", profile=True)


@pytest.mark.parametrize("protein", [False, True])
@pytest.mark.parametrize("K", [1, 2])
def test_table_planes(oracle, blosum62, K, protein):
    # the TABLE instantiation (single-pair _table / _rowcol exports): every cell of the score, matches, similar and
    # length planes, with strips of 32 or 64 rows so that the pairs cross several strip boundaries (and end mid-strip)
    mat = blosum62 if protein else oracle.Matrix.create(b"ACGT", 2, -3)
    o, e = (10, 1) if protein else (5, 2)
    qs, rs = pairs(81 + K, 3, (70, 150), (1, 90), protein)
    qs[1] = qs[1][:32 * K + 1]   # one row into the second strip
    cases = [(mode, (1, 1, 1, 1)) for mode in (0, 1, 2)] + [(1, f) for f in ((1, 0, 0, 0), (0, 1, 1, 0), (0, 0, 0, 1), (0, 1, 0, 1))]
    for mode, flags in cases:
        got = emu_harness.gotoh32(qs, rs, mat, K, mode, o, e, flags, table=True)
        for i, (q, r) in enumerate(zip(qs, rs)):
            exp = oracle.align(q, r, mat, mode=mode, open=o, gap=e, s1_beg=flags[0], s1_end=flags[1],
                               s2_beg=flags[2], s2_end=flags[3], tables=True)
            tag = (i, K, mode, flags, len(q), len(r))
            assert (got["score"][i], got["end_query"][i], got["end_ref"][i]) == (exp["score"], exp["end_query"], exp["end_ref"]), tag
            assert (got["matches"][i], got["similar"][i], got["length"][i]) == (exp["matches"], exp["similar"], exp["length"]), tag
            for name in emu_harness.TABLE_PLANES:
                bad = np.argwhere(got[name][i] != exp[name])
                assert len(bad) == 0, f"{tag} {name}: {len(bad)} cells differ, first at (i, j) = {tuple(bad[0])}: " \
                                      f"got {got[name][i][tuple(bad[0])]} expected {exp[name][tuple(bad[0])]}"


@pytest.mark.parametrize("bits,protein", [(5, True), (2, False)])
def test_packed_subjects_and_device_count(oracle, blosum62, bits, protein):
    # database-scan form: one query, subjects read from the 5-bit / 2-bit packed store, results
    # scattered through out_map, number of work items read from device memory
    mat = blosum62 if protein else oracle.Matrix.create(b"ACG", 2, -3)   # 4 columns incl. wildcard -> 2 bits
    q = psb_data.random_seq(71, 0, 70, protein) if protein else np.frombuffer(b"ACGACGGACCAGCAGGCA", dtype=np.uint8)
    subs = [psb_data.random_seq(72, i, 20 + 13 * i, protein) for i in range(5)]
    if not protein:
        subs = [np.frombuffer(bytes(s).replace(b"T", b"A"), dtype=np.uint8) for s in subs]
    for mode in (0, 2):
        got = emu_harness.gotoh32([q], subs, mat, 2, mode, 5, 2, shared_query=True, profile=True, packed_bits=bits, stats=True)
        for i, s_ in enumerate(subs):
            exp = oracle.align(q, s_, mat, mode=mode, open=5, gap=2)
            assert (got["score"][i], got["end_query"][i], got["end_ref"][i], got["matches"][i], got["length"][i]) == \
                (exp["score"], exp["end_query"], exp["end_ref"], exp["matches"], exp["length"]), (mode, i)
