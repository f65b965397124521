"""CPU-only: the C-ABI library loads and exports every symbol include/parasail_b200.h declares;
host-side logic (matrices, name grammar, error behaviour) works without a GPU; and the product
fails loudly -- never falls back -- when no CUDA device exists."""
import ctypes as C
import json
import os
import re

import numpy as np
import pytest

import psb_data

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ps():
    import __graft_entry__ as g
    g.build()
    import parasail_rs_b200 as ps
    return ps


def header_symbols():
    text = open(os.path.join(ROOT, "include", "parasail_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    names = set(re.findall(r"\b((?:parasail|psb)_[a-z0-9_]+)\s*\(", text))
    # macro-stamped profile creators
    for st in ("", "_stats"):
        for isa in ("", "_sse_128", "_avx_256", "_neon_128", "_altivec_128"):
            for w in ("8", "16", "32", "64", "sat"):
                names.add(f"parasail_profile_create{st}{isa}_{w}")
    names = {n for n in names if not n.endswith("_t") and "##" not in n}
    names.discard("parasail_profile_create")
    names.discard("parasail_profile_create_stats")
    return names


def test_every_declared_symbol_is_exported(ps):
    from parasail_rs_b200 import _lib
    L = _lib.lib()
    declared = header_symbols()
    assert len(declared) >= 105 + 15
    missing = [n for n in sorted(declared) if not hasattr(L, n)]
    assert not missing, missing
    assert set(_lib.ALL_SYMBOLS) <= declared


def test_reference_binds_105_functions(ps):
    # the four `use libparasail_sys::{..}` blocks of parasail-rs, stored in tests/golden/reference_bindings.json:
    # aligner 4 + profile 52 + matrix 8 + alignment 41
    from parasail_rs_b200 import _lib
    L = _lib.lib()
    mods = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_bindings.json")))["modules"]
    assert {m: len(set(v)) for m, v in mods.items()} == {"aligner": 4, "profile": 52, "matrix": 8, "alignment": 41}
    fns = set().union(*mods.values())
    assert len(fns) == 105
    assert fns <= header_symbols()
    assert not [n for n in sorted(fns) if not hasattr(L, n)]


def test_matrix_construction(ps, tmp_path):
    # [REF tests/test_parasail.rs:4-34]
    ps.Matrix.default()
    m = ps.Matrix.create(b"ACGT", 3, -2)
    assert m.size == 5 and m.length == 5 and m.type_ == 0
    v = m.values()
    assert v[0, 0] == 3 and v[0, 1] == -2 and v[4, 0] == 0 and v[0, 4] == 0
    m.set_value(2, 2, 100)
    assert m.values()[2, 2] == 100
    with pytest.raises(ps.InvalidIndex):
        m.set_value(4, 0, 1)  # bound is size-2
    b62 = ps.Matrix.from_name("blosum62")
    assert np.array_equal(b62.values(), psb_data.blosum62_table())
    with pytest.raises(ps.NotBuiltIn):
        b62.set_value(0, 0, 1)
    with pytest.raises(ps.FailedLookup):
        ps.Matrix.from_name("nosuchmatrix")
    pssm = b62.to_pssm(b"ACGT")
    assert pssm.type_ == 1 and pssm.length == 4 and pssm.size == 24
    assert np.array_equal(pssm.values()[1], psb_data.blosum62_table()[4])  # 'C' row
    sq = ps.Matrix.from_file(os.path.join(ROOT, "tests", "golden", "square.txt"))
    assert sq.type_ == 0 and sq.size == 17 and sq.values()[0, 0] == 5 and sq.values()[16, 16] == -5
    assert sq.mapper()[ord("u")] == 15 and sq.mapper()[ord("?")] == 16
    ps_ = ps.Matrix.from_file(os.path.join(ROOT, "tests", "golden", "pssm.txt"))
    assert ps_.type_ == 1 and ps_.length == 10 and ps_.size == 21 and ps_.values()[0, 2] == 3
    with pytest.raises(ps.FileNotFound):
        ps.Matrix.from_file(str(tmp_path / "missing.txt"))
    p2 = ps.Matrix.create_pssm("abcdef", list(range(12)), 2)
    assert p2.type_ == 1 and p2.length == 2 and p2.size == 7
    c = m.clone()
    assert np.array_equal(c.values(), m.values())
    assert str(ps.Matrix.create(b"AC", 1, -1)).splitlines()[0].strip() == "1 -1 0"


def test_default_matrix_maps_like_upstream(ps):
    # Matrix::default() uses "ACGTA": the duplicate A maps 'A' to index 4 [REF src/matrix/mod.rs:246-250]
    m = ps.Matrix.default()
    mp = m.mapper()
    assert m.size == 6 and mp[ord("A")] == 4 and mp[ord("a")] == 4 and mp[ord("C")] == 1 and mp[ord("N")] == 5


def test_name_grammar(ps):
    # [REF src/aligner/mod.rs:289-331]
    b = ps.Aligner.new()
    assert b.get_parasail_fn_name() == "nw_striped_sat"
    assert ps.Aligner.new().local().use_stats().scan().solution_width(16).get_parasail_fn_name() == "sw_stats_scan_16"
    b = ps.Aligner.new().semi_global().allow_query_gaps(["prefix"]).allow_ref_gaps(["suffix"]).use_stats().use_last_rowcol()
    assert b.get_parasail_fn_name() == "sg_qb_de_stats_rowcol_striped_sat"
    b = ps.Aligner.new().semi_global().allow_query_gaps(["prefix", "suffix"]).allow_ref_gaps(["prefix", "suffix"])
    assert b.get_parasail_fn_name() == "sg_striped_sat"
    assert ps.Aligner.new().use_stats().use_trace().get_parasail_fn_name() == "nw_trace_striped_sat"
    assert ps.Aligner.new().use_trace().use_table().get_parasail_fn_name() == "nw_table_striped_sat"
    from parasail_rs_b200 import _lib
    L = _lib.lib()
    good = ["nw_striped_sat", "parasail_sw_trace_scan_16", "sg_qb_de_stats_rowcol_diag_8", "sg_dx_table_striped_64",
            "sg_qe_db_striped_32"]
    bad = ["nw", "sw_striped", "sg_qx_db_striped_sat", "nw_trace_stats_striped_sat", "xx_striped_sat",
           "nw_striped_sat_", "nw_striped_profile_sat"]
    for n in good:
        assert L.parasail_lookup_function(n.encode()), n
    for n in bad:
        assert not L.parasail_lookup_function(n.encode()), n
    assert L.parasail_lookup_pfunction(b"sw_striped_profile_sat")
    assert L.parasail_lookup_pfunction(b"sg_stats_scan_profile_16")
    assert not L.parasail_lookup_pfunction(b"sw_diag_profile_sat")
    assert not L.parasail_lookup_pfunction(b"sw_striped_sat")
    # distinct names resolve to distinct entry points (the pointer carries the configuration)
    ptrs = {L.parasail_lookup_function(n.encode()) for n in good}
    assert len(ptrs) == len(good)
    with pytest.raises(ps.Panic):
        ps.Aligner.new().semi_global().allow_query_gaps(["prefix", "suffix"]).allow_ref_gaps(["prefix"]).build()


def test_profile_and_aligner_construction(ps):
    # [REF tests/test_parasail.rs:36-62]
    q = b"ATGGCACTATAA"
    ps.Profile.new(q, False, ps.Matrix.default())
    ps.Profile.new(q, True, ps.Matrix.default())
    with pytest.raises(ps.QueryIsEmpty):
        ps.Profile.new(b"", False, ps.Matrix.default())
    ps.Profile.builder(q, ps.Matrix.default()).use_stats().solution_width("Bit16").instruction_set("AVX2").build()
    ps.Aligner.new().build()
    ps.Aligner.new().matrix(ps.Matrix.default()).gap_open(10).gap_extend(1).profile(ps.Profile.default()) \
        .allow_query_gaps(["prefix", "suffix"]).striped().use_stats().build()
    with pytest.raises(ps.InteriorNulByte):
        ps.Aligner.new().build().align(b"AC\0GT", b"ACGT")
    with pytest.raises(ps.Panic):
        ps.Aligner.new().build().align(None, b"ACGT")
    with pytest.raises(ps.NoBandwidth):
        ps.Aligner.new().build().banded_nw(b"ACGT", b"ACGT")


def test_shard_plan_balances_residues(ps):
    lens = psb_data.lognormal_lengths(2002, 20000)
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    off[1:] = np.cumsum(lens)
    for k in (2, 4, 8):
        shard = ps.shard_plan(off, k)
        loads = np.bincount(shard, weights=lens, minlength=k)
        assert loads.max() - loads.min() <= lens.max()
        assert set(shard) == set(range(k))


def test_no_gpu_fails_loudly(ps):
    """On a box without a CUDA device the product must fail, not fall back."""
    from parasail_rs_b200 import _lib
    if _lib.lib().psb_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(ps.DeviceError) as e:
        ps.Aligner.new().build().align_batch([b"ACGT"], [b"ACGT"])
    assert "no CPU fallback" in str(e.value)
    a = ps.Aligner.new().build().align(b"ACGT", b"ACGT")
    assert a.is_saturated() and a.get_score() == 0  # flagged, not a silently wrong answer
    with pytest.raises(ps.DeviceError):
        ps.Database([b"ACGT"], ps.Matrix.default())
