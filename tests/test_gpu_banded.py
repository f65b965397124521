"""Banded global alignment on the band kernel (psb_align_pairs_banded, Aligner.banded_nw_batch, parasail_nw_banded):
against the CPU oracle's banded nw bit for bit, against the unbanded path where the band covers the table, and under
the error cases of the C ABI."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import band_oracle
import psb_data
from test_oracle_properties import cigar_rescore

pytestmark = pytest.mark.gpu

PSB_EINVAL, PSB_EUNSUPPORTED = -1, -5
FLAG_NW, FLAG_BANDED, FLAG_NOVEC, FLAG_STRIPED, FLAG_STATS, FLAG_TRACE = 1, 1 << 7, 1 << 8, 1 << 11, 1 << 16, 1 << 19
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ps():
    import __graft_entry__ as g
    g.build()
    import parasail_rs_b200 as ps
    return ps


def related(seed, n, lq, lr, protein=True, p_indel=0.02):
    qs, rs = [], []
    for i in range(n):
        q = psb_data.random_seq(seed, 2 * i, lq, protein)
        r = psb_data.mutate(q, seed, 2 * i + 1, 0.1, p_indel, protein)
        r = np.concatenate([r, psb_data.random_seq(seed, 2 * i + 1, lr, protein)])[:lr]
        qs.append(q); rs.append(r)
    return qs, rs


def schemes(ps, oracle):
    dna = (ps.Matrix.create(b"ACGT", 2, -3), oracle.Matrix.create(b"ACGT", 2, -3), False)
    big = (ps.Matrix.create(b"ACGT", 200, -150), oracle.Matrix.create(b"ACGT", 200, -150), False)
    b62 = (ps.Matrix.from_name("blosum62"), oracle.Matrix.from_table(psb_data.BLOSUM62_ALPHABET, psb_data.blosum62_table()), True)
    return {"dna_5_2": dna + (5, 2), "dna_1_4": dna + (1, 4), "dna_0_0": dna + (0, 0), "big_30_4": big + (30, 4),
            "b62_10_1": b62 + (10, 1)}


def run(ps, mat, o, e, k, qs, rs, out=""):
    b = ps.Aligner.new().global_().matrix(mat).gap_open(o).gap_extend(e).bandwidth(k)
    if out == "trace":
        b = b.use_trace()
    elif out == "stats":
        b = b.use_stats()
    return b.build().banded_nw_batch(qs, rs)


def check(got, exp, out, tag):
    keys = ["score", "end_query", "end_ref"] + (["matches", "similar", "length"] if out == "stats" else []) + \
           (["beg_query", "beg_ref", "cigar_off", "cigar_ops"] if out == "trace" else [])
    for key in keys:
        g, x = getattr(got, key), exp[key]
        if not np.array_equal(g, x):
            bad = np.flatnonzero(g != x)[:1] if len(g) == len(x) else "length"
            raise AssertionError(f"{tag}: {key} differs, first at {bad}")


def oracle_of(omat, o, e, k, qs, rs, out):
    qc, qo = psb_data.concat(qs)
    rc, ro = psb_data.concat(rs)
    return band_oracle.align_batch(qc, qo, rc, ro, omat, o, e, k, stats=out == "stats", cigar=out == "trace")


@pytest.mark.parametrize("k", [1, 2, 5, 31, 32, 33, 100, 255, 256, 257, 511, 512, 513, 2000])
@pytest.mark.parametrize("out", ["", "stats", "trace"])
def test_against_oracle_band_widths(ps, oracle, k, out):
    mat, omat, prot, o, e = schemes(ps, oracle)["b62_10_1"]
    qs, rs = related(k, 6, 700, 720)
    qs += [qs[0][:3], qs[1][:500], qs[2]]
    rs += [rs[0][:400], rs[1][:60], rs[2][:1]]
    check(run(ps, mat, o, e, k, qs, rs, out), oracle_of(omat, o, e, k, qs, rs, out), out, f"k={k} out={out}")


@pytest.mark.parametrize("scheme", ["dna_5_2", "dna_1_4", "dna_0_0", "big_30_4", "b62_10_1"])
@pytest.mark.parametrize("out", ["", "stats", "trace"])
def test_against_oracle_schemes_and_mixed_batches(ps, oracle, scheme, out):
    mat, omat, prot, o, e = schemes(ps, oracle)[scheme]
    rng = np.random.default_rng(len(scheme))
    qs, rs = [], []
    for i in range(60):   # mixed lengths: band pairs and pairs whose band covers their table
        lq, lr = int(rng.integers(1, 900)), int(rng.integers(1, 900))
        a, b = related(1000 + i, 1, lq, lr, prot)
        qs += a; rs += b
    for k in (3, 40, 300):
        check(run(ps, mat, o, e, k, qs, rs, out), oracle_of(omat, o, e, k, qs, rs, out), out, f"{scheme} k={k} out={out}")


def test_pssm(ps, oracle):
    b62 = ps.Matrix.from_name("blosum62")
    q = psb_data.random_seq(77, 0, 300)
    pssm = b62.to_pssm(bytes(q))
    ob62 = oracle.Matrix.from_table(psb_data.BLOSUM62_ALPHABET, psb_data.blosum62_table())
    opssm = oracle.Matrix(ob62.table[ob62.mapper[q]], ob62.mapper, is_pssm=True)
    rs = [psb_data.mutate(q, 77, i, 0.15, 0.03) for i in range(1, 9)] + [q[:40], q[:5]]
    qs = [q] * len(rs)
    for out in ("", "stats", "trace"):
        for k in (4, 50):
            check(run(ps, pssm, 10, 1, k, qs, rs, out), oracle_of(opssm, 10, 1, k, qs, rs, out), out, f"pssm k={k} {out}")


@pytest.mark.parametrize("out", ["", "stats", "trace"])
def test_whole_table_bands_equal_unbanded(ps, oracle, out):
    b62 = ps.Matrix.from_name("blosum62")
    qs, rs = related(5, 40, 60, 70)
    b = ps.Aligner.new().global_().matrix(b62).gap_open(10).gap_extend(1)
    b = b.use_trace() if out == "trace" else (b.use_stats() if out == "stats" else b)
    full = b.build().align_batch(qs, rs)
    got = run(ps, b62, 10, 1, 100, qs, rs, out)   # lo <= -lq and hi >= lr for every pair
    for key in ("score", "end_query", "end_ref", "matches", "similar", "length", "beg_query", "beg_ref", "cigar_off", "cigar_ops"):
        a, x = getattr(got, key), getattr(full, key)
        assert (a is None and x is None) or np.array_equal(a, x), key
    assert got.flag == full.flag | FLAG_BANDED


def single(ps, mat, o, e, k, q, r, env_off=False):
    a = ps.Aligner.new().global_().matrix(mat).gap_open(o).gap_extend(e).bandwidth(k).build()
    res = a.banded_nw(bytes(q), bytes(r))
    return res.get_score(), res.get_end_query(), res.get_end_ref(), res.inner.contents.flag


def test_single_pair_against_oracle(ps, oracle):
    mat, omat, prot, o, e = schemes(ps, oracle)["b62_10_1"]
    for lq, lr, k in ((300, 310, 3), (500, 200, 64), (2000, 2100, 600), (30000, 30000, 64)):
        q, r = (x[0] for x in related(lq + k, 1, lq, lr, p_indel=0.01))
        exp = oracle.align(q, r, omat, mode=oracle.NW, open=o, gap=e, band=k)
        sc, eq, er, flag = single(ps, mat, o, e, k, q, r)
        assert (sc, eq, er) == (exp["score"], exp["end_query"], exp["end_ref"]), (lq, lr, k)
        assert flag & FLAG_BANDED and flag & FLAG_NW and flag & FLAG_NOVEC and not flag & FLAG_STRIPED


SINGLE_SCRIPT = r"""
import sys, json
sys.path[:0] = [sys.argv[1], sys.argv[1] + '/tests']
import numpy as np, psb_data, parasail_rs_b200 as ps
out = []
b62 = ps.Matrix.from_name('blosum62')
for lq, lr, k in ((300, 310, 3), (500, 200, 64), (3000, 3100, 5000), (2500, 2600, 30)):
    q = psb_data.random_seq(lq, 0, lq); r = psb_data.mutate(q, lq, 1, 0.1, 0.02)[:lr]
    res = ps.Aligner.new().global_().matrix(b62).gap_open(10).gap_extend(1).bandwidth(k).build().banded_nw(bytes(q), bytes(r))
    out.append([res.get_score(), res.get_end_query(), res.get_end_ref(), res.inner.contents.flag])
print(json.dumps(out))
"""


def test_single_pair_equals_masked_path(ps):
    # parasail_nw_banded on the band kernel and on the masked general kernel (PSB_NO_BAND_KERNEL): score, ends, flags
    runs = []
    for env in ({}, {"PSB_NO_BAND_KERNEL": "1"}):
        r = subprocess.run([sys.executable, "-c", SINGLE_SCRIPT, ROOT], capture_output=True, text=True, env={**os.environ, **env})
        assert r.returncode == 0, r.stderr
        runs.append(r.stdout.strip().splitlines()[-1])
    assert runs[0] == runs[1]


def test_long_pair_100kb(ps, oracle):
    b62 = ps.Matrix.from_name("blosum62")
    q = psb_data.random_seq(9, 0, 100_000)
    r = psb_data.mutate(q, 9, 1, 0.05, 0.0004)   # indels balance: the drift stays well inside k = 128
    k = 128
    tr = run(ps, b62, 10, 1, k, [q], [r], "trace")
    st = run(ps, b62, 10, 1, k, [q], [r], "stats")
    full = ps.Aligner.new().global_().matrix(b62).gap_open(10).gap_extend(1).build().align_batch([q], [r])
    assert tr.score[0] == st.score[0] == full.score[0]
    assert (tr.beg_query[0], tr.beg_ref[0]) == (0, 0)
    omat = oracle.Matrix.from_table(psb_data.BLOSUM62_ALPHABET, psb_data.blosum62_table())
    ops = tr.cigar_ops[tr.cigar_off[0]: tr.cigar_off[1]]
    rescored = cigar_rescore(ops, q, r, 0, 0, omat, 10, 1)   # (score, end cell, matches, similar, length)
    assert rescored[:3] == (tr.score[0], len(q) - 1, len(r) - 1), rescored[:3]
    assert (st.matches[0], st.similar[0], st.length[0]) == rescored[3:]


@pytest.mark.parametrize("lanes", ["1", "2"])
def test_passes(ps, lanes):
    script = r"""
import sys, hashlib
sys.path[:0] = [sys.argv[1], sys.argv[1] + '/tests']
import numpy as np, psb_data, parasail_rs_b200 as ps
qs, rs = psb_data.dna_read_pairs(31, 6000, read_len=150, win_len=180)
dna = ps.Matrix.create(b'ACGT', 2, -3)
b = ps.Aligner.new().global_().matrix(dna).gap_open(5).gap_extend(2).bandwidth(8).use_trace().build().banded_nw_batch(qs, rs)
h = hashlib.sha256()
for a in (b.score, b.end_query, b.end_ref, b.beg_query, b.beg_ref, b.cigar_off, b.cigar_ops):
    h.update(np.ascontiguousarray(a).tobytes())
print(h.hexdigest())
"""
    outs = []
    for env in ({}, {"PSB_PAIRS_PASS_MB": "1", "PSB_PAIRS_LANES": lanes}):
        r = subprocess.run([sys.executable, "-c", script, ROOT], capture_output=True, text=True, env={**os.environ, **env})
        assert r.returncode == 0, r.stderr
        outs.append(r.stdout.strip().splitlines()[-1])
    assert outs[0] == outs[1]


def call(ps, name, k, qs, rs, mat=None, null=None):
    from parasail_rs_b200 import _lib
    L = _lib.lib()
    mat = mat or ps.Matrix.from_name("blosum62")
    qc, qo = psb_data.concat(qs)
    rc, ro = psb_data.concat(rs)
    out = C.POINTER(_lib.CBatch)()
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    args = [name, mat.inner, 10, 1, k, p(qc), p(qo), p(rc), p(ro), len(ro) - 1, C.byref(out)]
    if null is not None:
        args[null] = None
    rc_ = L.psb_align_pairs_banded(*args)
    if rc_ == 0:
        b = out.contents
        res = dict(flag=b.flag, score=[b.score[i] for i in range(b.n)], sat=[b.saturated[i] for i in range(b.n)])
        L.psb_batch_free(out)
        return rc_, res
    return rc_, None


def test_errors_and_flags(ps):
    q = [psb_data.random_seq(3, 0, 200)]
    r = [psb_data.random_seq(3, 1, 210)]
    assert call(ps, b"sw_striped_32", 5, q, r)[0] == PSB_EINVAL
    assert call(ps, b"sg_striped_32", 5, q, r)[0] == PSB_EINVAL
    assert call(ps, b"nw_striped_32", 0, q, r)[0] == PSB_EINVAL
    assert call(ps, b"nw_striped_32", -3, q, r)[0] == PSB_EINVAL
    assert call(ps, b"nw_bogus", 5, q, r)[0] == PSB_EINVAL
    assert call(ps, b"nw_striped_32", 5, q, r, null=1)[0] == PSB_EINVAL
    assert call(ps, b"nw_striped_32", 5, q, r, null=7)[0] == PSB_EINVAL
    assert call(ps, b"nw_striped_32", 5, q, [np.zeros(0, dtype=np.uint8)])[0] == PSB_EINVAL
    assert call(ps, b"nw_table_striped_32", 5, q, r)[0] == PSB_EUNSUPPORTED
    assert call(ps, b"nw_stats_rowcol_striped_32", 5, q, r)[0] == PSB_EUNSUPPORTED
    wide_q, wide_r = [psb_data.random_seq(4, 0, 9000)], [psb_data.random_seq(4, 1, 9000)]
    rc, _ = call(ps, b"nw_striped_32", 2048, wide_q, wide_r)   # W = 4097
    err = ps.last_error()
    assert rc == PSB_EUNSUPPORTED and "4097" in err and "4096" in err
    assert call(ps, b"nw_striped_32", 2047, wide_q, wide_r)[0] == 0   # W = 4095
    assert call(ps, b"nw_striped_32", 9000, wide_q, wide_r)[0] == 0   # covers the table
    for name, extra in ((b"nw_striped_32", 0), (b"nw_trace_striped_sat", FLAG_TRACE), (b"nw_stats_scan_16", FLAG_STATS)):
        rc, res = call(ps, name, 5, q, r)
        assert rc == 0 and res["flag"] & FLAG_BANDED and res["flag"] & FLAG_NW and (res["flag"] & extra) == extra, name
    # saturation at explicit narrow widths: a long pair of mismatches overflows 8 bit, not 16 bit
    bad_q, bad_r = [np.frombuffer(b"W" * 300, dtype=np.uint8)], [np.frombuffer(b"P" * 300, dtype=np.uint8)]
    rc8, res8 = call(ps, b"nw_striped_8", 5, bad_q, bad_r)
    rc16, res16 = call(ps, b"nw_striped_16", 5, bad_q, bad_r)
    assert rc8 == rc16 == 0 and res8["sat"] == [1] and res8["score"] == [0] and res16["sat"] == [0] and res16["score"][0] < -128


def test_python_errors(ps):
    b62 = ps.Matrix.from_name("blosum62")
    with pytest.raises(ps.NoBandwidth):
        ps.Aligner.new().global_().matrix(b62).build().banded_nw_batch([b"ACD"], [b"ACD"])
    with pytest.raises(ps.Panic):
        ps.Aligner.new().local().matrix(b62).bandwidth(3).build().banded_nw_batch([b"ACD"], [b"ACD"])
    prof = ps.Profile.new(b"ACDEF", False, b62)
    with pytest.raises(ps.Panic):
        ps.Aligner.new().global_().matrix(b62).profile(prof).bandwidth(3).build().banded_nw_batch([b"ACD"], [b"ACD"])
