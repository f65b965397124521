#!/usr/bin/env python
"""What searching many queries in one call (psb_db_search, Aligner.search_many) saves against the per-query composition.

usage: python tools/search_probe.py [--db 1000000] [--small 10000] [--nq 64] [--reps 5] [--out FILE.json]

The resident database of bench.py's synthetic proteins (C2 size by default) and a small one of --small subjects from the
same generator; BLOSUM62 open 10 / extend 1, local alignment with traceback (sw_trace_striped_profile_sat).
  many L       nq queries of L residues (100 / 250 / 400), k = 100: psb_db_search against the old composition, per
               query psb_scan (score-only) -> psb_batch_topk -> psb_db_align, called directly from here
  single k     Aligner.search(db, k) (now the one-query psb_db_search) against the same composition for one query,
               bench.py's 400-aa query, k = 100 / 1 000 / 10 000
The two sides of a case alternate within the run, after a warm-up of each; the figures are medians of --reps calls:
wall ms of the call ending in a device synchronise, and for psb_db_search its psb_last_kernel_ms / psb_last_launches
(the whole call); for the composition the sums over its calls.  Checked inside the run: both sides return the same ids
and the same rows, field for field, CIGARs included.  The card's name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)
import bench  # noqa: E402
from db_align_probe import card  # noqa: E402

NAME = b"sw_trace_striped_profile_sat"
SCORE_ONLY = b"sw_striped_profile_sat"
FIELDS = ("score", "end_query", "end_ref", "beg_query", "beg_ref", "saturated", "cigar_off", "cigar_ops")


def composition(ps, profs, db, k):
    """per query: psb_scan, psb_batch_topk on the host, psb_db_align of the k hits"""
    L = ps._lib.lib()
    ids, batches, ms, launches = [], [], 0.0, 0
    for p in profs:
        out = C.POINTER(ps.CBatch)()
        assert L.psb_scan(SCORE_ONLY, p.inner, bench.OPEN, bench.GAP, db.inner, C.byref(out)) == 0, ps._lib.last_error()
        ms += ps.kernel_ms(); launches += ps.launches()
        idx, _ = ps.BatchResult(out).topk(k)
        hits = C.POINTER(ps.CBatch)()
        assert L.psb_db_align(NAME, p.inner, bench.OPEN, bench.GAP, db.inner, idx.ctypes.data_as(C.c_void_p), len(idx), C.byref(hits)) == 0
        ms += ps.kernel_ms(); launches += ps.launches()
        ids.append(idx); batches.append(ps.BatchResult(hits))
    return (np.stack(ids), batches), ms, launches


def searched(ps, aligner, profs, db, k):
    out = aligner.search_many(db, profs, k)
    return out, ps.kernel_ms(), ps.launches()


def same(new, old):
    (ids, got), (oids, obs) = new, old
    assert np.array_equal(ids, oids)
    kk = ids.shape[1]
    for q, ob in enumerate(obs):
        for f in FIELDS[:6]:
            assert np.array_equal(getattr(got, f)[q * kk:(q + 1) * kk], getattr(ob, f)), (q, f)
        for r in range(kk):
            assert got.cigar(q * kk + r) == ob.cigar(r), (q, r)


def alternate(ps, sides, reps):
    """{name: fn} -> {name: medians}; each fn returns (result, kernel_ms, launches); one warm-up call each"""
    rows = {n: [] for n in sides}
    results = {n: fn()[0] for n, fn in sides.items()}
    for _ in range(reps):
        for n, fn in sides.items():
            t0 = time.perf_counter()
            res, ms, la = fn()
            ps._lib.lib().psb_synchronize()
            rows[n].append(((time.perf_counter() - t0) * 1e3, ms, la))
            results[n] = res
    med = lambda r, i: statistics.median(x[i] for x in r)
    return results, {n: {"wall_ms": round(med(r, 0), 3), "wall_ms_min": round(min(x[0] for x in r), 3), "wall_ms_max": round(max(x[0] for x in r), 3),
                         "kernel_ms": round(med(r, 1), 3), "launches": int(med(r, 2))} for n, r in rows.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--db", type=int, default=1000000)
    ap.add_argument("--small", type=int, default=10000)
    ap.add_argument("--nq", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from __graft_entry__ import build
    build()
    import parasail_rs_b200 as ps
    import psb_data

    b62 = ps.Matrix.from_name("blosum62")
    query, cat, off = bench.make_inputs(args.db)
    scat, soff = cat[: off[args.small]].copy(), off[: args.small + 1].copy()
    dbs = {"C2": (ps.Database((cat, off), b62), int(off[-1])), "small": (ps.Database((scat, soff), b62), int(soff[-1]))}
    res = {"workload": f"bench.py's synthetic proteins ({args.db} subjects, {int(off[-1])} residues; small: the first {args.small}, "
                       f"{int(soff[-1])} residues), BLOSUM62 open {bench.OPEN} ext {bench.GAP}, {NAME.decode()}",
           "reps": args.reps, "nq": args.nq, **card(), "cases": {}}

    for dname, (db, residues) in dbs.items():
        for lq in (100, 250, 400):
            profs = [ps.Profile.new(psb_data.random_seq(4100 + lq, i, lq), False, b62) for i in range(args.nq)]
            a = ps.Aligner.new().local().gap_open(bench.OPEN).gap_extend(bench.GAP).profile(profs[0]).use_trace().build()
            results, t = alternate(ps, {"psb_db_search": lambda: searched(ps, a, profs, db, 100),
                                        "composition": lambda: composition(ps, profs, db, 100)}, args.reps)
            same(results["psb_db_search"], results["composition"])
            case = {"scan_cells": float(lq) * residues * args.nq, **t, "checked": "same ids and rows, CIGARs included"}
            case["saved_ms_per_query"] = round((t["composition"]["wall_ms"] - t["psb_db_search"]["wall_ms"]) / args.nq, 3)
            res["cases"][f"{dname} many {lq}"] = case
            print(f"{dname} many {lq}: {json.dumps(case)}", flush=True)

    db = dbs["C2"][0]
    prof = ps.Profile.new(query, False, b62)
    a = ps.Aligner.new().local().gap_open(bench.OPEN).gap_extend(bench.GAP).profile(prof).use_trace().build()
    for k in (100, 1000, 10000):
        def one():
            ids, hits = a.search(db, k)
            return (ids[None, :], hits), ps.kernel_ms(), ps.launches()
        results, t = alternate(ps, {"Aligner.search": one, "composition": lambda: composition(ps, [prof], db, k)}, args.reps)
        same(results["Aligner.search"], results["composition"])
        res["cases"][f"single {k}"] = {**t, "checked": "same ids and rows, CIGARs included"}
        print(f"single {k}: {json.dumps(res['cases'][f'single {k}'])}", flush=True)

    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
