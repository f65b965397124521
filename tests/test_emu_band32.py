"""The band kernel (csrc/kern_band32.cuh) and its walk (walk_band_kernel), stepped on CPU threads through the SIMT
emulation, must agree with the oracle's banded nw bit for bit: score, end cell, statistics, every in-band trace
byte, the CIGAR and its begin coordinates."""
import numpy as np
import pytest

import band_oracle
import emu_band32
import psb_data


def band_trace(oracle_trace, lq, lr, k):
    """the oracle's row-major trace table in band layout (row i, offset t = j - i - lo); cells outside the table 0"""
    lo, _, W = emu_band32.band_geom(lq, lr, k)
    out = np.zeros((lq, W), dtype=np.uint8)
    for i in range(lq):
        for t in range(W):
            j = i + lo + t
            if 0 <= j < lr:
                out[i, t] = np.uint8(oracle_trace[i, j])
    return out


def regs_for(W):
    """offsets per lane of the register variant the device takes for a band of W offsets (0: shared memory)"""
    for R in (2, 4, 8, 16):
        if W <= 32 * R:
            return R
    return 0


def compare(oracle, mat, qs, rs, k, o, e, R=None, rr=0):
    """every output of the emulated kernel against oracle.align(..., band=k)"""
    for stats, trace in ((False, False), (True, False), (False, True), (True, True)):
        if R is None:
            Rk = max(regs_for(emu_band32.band_geom(len(q), len(r), k)[2]) for q, r in zip(qs, rs))
        else:
            Rk = R
        got = emu_band32.band32(qs, rs, mat, k, o, e, Rk, stats=stats, trace=trace, rr=rr)
        for i, (q, r) in enumerate(zip(qs, rs)):
            exp = oracle.align(q, r, mat, mode=oracle.NW, open=o, gap=e, trace=trace, band=k)
            lq = mat.length if mat.is_pssm else len(q)
            tag = dict(pair=i, lq=lq, lr=len(r), k=k, R=Rk, rr=rr, stats=stats, trace=trace)
            assert (got["score"][i], got["end_query"][i], got["end_ref"][i]) == (exp["score"], exp["end_query"], exp["end_ref"]), tag
            if stats:
                assert (got["matches"][i], got["similar"][i], got["length"][i]) == (exp["matches"], exp["similar"], exp["length"]), tag
            if trace:
                want = band_trace(exp["trace"], lq, len(r), k)
                diff = np.argwhere(got["trace"][i] != want)
                assert diff.size == 0, (tag, "first differing (row, offset)", diff[:1].tolist())
                assert np.array_equal(got["cigar_ops"][i], exp["cigar_ops"]), tag
                assert (got["beg_query"][i], got["beg_ref"][i]) == (exp["beg_query"], exp["beg_ref"]), tag


def related(seed, n, lq, lr, protein=True):
    """pairs of the given lengths whose second sequence is a mutated copy of the first (so that the band matters)"""
    qs, rs = [], []
    for i in range(n):
        q = psb_data.random_seq(seed, 2 * i, lq, protein)
        r = psb_data.mutate(q, seed, 2 * i + 1, 0.15, 0.05, protein)
        r = np.concatenate([r, psb_data.random_seq(seed, 2 * i + 1, lr, protein)])[:lr]
        qs.append(q); rs.append(r)
    return qs, rs


@pytest.fixture(scope="module")
def dna(oracle):
    return oracle.Matrix.create(b"ACGT", 2, -3)


# W = 2k + |lr - lq| + 1: each register variant at its capacity 32R - 1 and 32R, and 32R + 1 on the next variant
@pytest.mark.parametrize("R", [2, 4, 8, 16])
@pytest.mark.parametrize("dW", [-1, 0, 1])
def test_register_variants_at_capacity(oracle, blosum62, R, dW):
    W = 32 * R + dW
    d = (W - 1) % 2            # W odd: equal lengths; W even: lengths differ by one
    k = (W - 1 - d) // 2
    qs, rs = related(100 + R, 2, 120, 120 + d)
    compare(oracle, blosum62, qs, rs, k, 10, 1, R=R if dW <= 0 else (2 * R if R < 16 else 0),
            rr=0 if dW <= 0 or R < 16 else 18)


def test_shared_memory_variant_just_above_registers(oracle, dna):
    # W = 513: one offset more than the widest register variant, 18 offsets per lane
    qs, rs = related(7, 2, 300, 300, protein=False)
    compare(oracle, dna, qs, rs, 256, 5, 2, R=0, rr=18)


def test_shared_memory_variant_small_band(oracle, blosum62):
    # the shared-memory code path on a narrow band (the same results as the register variants)
    qs, rs = related(8, 3, 90, 100)
    compare(oracle, blosum62, qs, rs, 5, 10, 1, R=0, rr=2)


@pytest.mark.parametrize("lq,lr,k", [(40, 120, 5), (120, 40, 5), (200, 60, 31), (60, 200, 33), (1, 1, 1), (1, 3, 1),
                                     (3, 1, 2), (2, 3, 1), (3, 3, 1), (1, 40, 2), (40, 1, 2)])
def test_shapes(oracle, blosum62, dna, lq, lr, k):
    qs, rs = related(lq * 7 + lr, 2, lq, lr)
    compare(oracle, blosum62, qs, rs, k, 10, 1)
    qs, rs = related(lq * 7 + lr + 1, 2, lq, lr, protein=False)
    compare(oracle, dna, qs, rs, k, 5, 2)


@pytest.mark.parametrize("k", [1, 2, 5, 17])
def test_scoring_schemes(oracle, blosum62, dna, k):
    qs, rs = related(20 + k, 2, 100, 110, protein=False)
    compare(oracle, dna, qs, rs, k, 5, 2)       # DNA 2/-3 with 5/2
    compare(oracle, dna, qs, rs, k, 1, 4)       # open < gap
    compare(oracle, dna, qs, rs, k, 0, 0)       # every gap free: ties everywhere
    big = oracle.Matrix.create(b"ACGT", 200, -150)
    compare(oracle, big, qs, rs, k, 30, 4)      # values far beyond a byte
    qs, rs = related(30 + k, 2, 100, 90)
    compare(oracle, blosum62, qs, rs, k, 10, 1)


@pytest.mark.parametrize("k", [3, 40])
def test_pssm(oracle, blosum62, k):
    q = psb_data.random_seq(5, 0, 80, True)
    mq = blosum62.mapper[q]
    pssm = oracle.Matrix(blosum62.table[mq], blosum62.mapper, is_pssm=True)
    r = psb_data.mutate(q, 5, 1, 0.2, 0.05, True)
    compare(oracle, pssm, [q, q], [r, r[: 60]], k, 10, 1)


def test_band_oracle_batch_equals_single_pairs(oracle, blosum62):
    # the batch form of the banded oracle (band_oracle.align_batch) is the single-pair oracle, pair by pair
    qs, rs = related(41, 12, 70, 90)
    qs += [np.frombuffer(s, dtype=np.uint8) for s in (b"A", b"ACD", b"W" * 50)]
    rs += [np.frombuffer(s, dtype=np.uint8) for s in (b"ACDEF", b"A", b"W" * 3)]
    qcat, qoff = psb_data.concat(qs)
    rcat, roff = psb_data.concat(rs)
    for k in (1, 4, 30):
        got = band_oracle.align_batch(qcat, qoff, rcat, roff, blosum62, 10, 1, k, stats=True, cigar=True)
        for i, (q, r) in enumerate(zip(qs, rs)):
            exp = oracle.align(q, r, blosum62, mode=oracle.NW, open=10, gap=1, trace=True, band=k)
            st = oracle.align(q, r, blosum62, mode=oracle.NW, open=10, gap=1, band=k)
            for f in ("score", "end_query", "end_ref", "beg_query", "beg_ref"):
                assert got[f][i] == exp[f], (k, i, f)
            for f in ("matches", "similar", "length"):
                assert got[f][i] == st[f], (k, i, f)
            assert np.array_equal(got["cigar_ops"][got["cigar_off"][i]: got["cigar_off"][i + 1]], exp["cigar_ops"]), (k, i)
