#!/usr/bin/env python
"""A resident database sharded over the GPUs of the box (BoxDatabase: psb_box_scan, psb_box_search) against the same
database on one device (Database: psb_scan, psb_db_search).

usage: python tools/box_search_probe.py [--db 1000000] [--nq 64] [--reps 5] [--out FILE.json]

bench.py's C2 database (its synthetic proteins and 400-aa query), BLOSUM62 open 10 / extend 1, built as a box of N
shards on devices 0 .. N-1 for N = 1, 2, 4, 8 (as many as are visible).  Per N:
  build        wall seconds of BoxDatabase(...) (the single-device Database once, beside it)
  scan         Aligner.scan with a fresh profile per call (profile creation + upload + scan), score-only
               sw_striped_profile_sat; GCUPS = query length x residues / wall time
  search       Aligner.search(db, 100) with sw_trace_striped_profile_sat for the 400-aa query
  many L       Aligner.search_many with --nq queries of L = 100 and 400 residues, k = 100, with traceback
The two sides of a case (box, then one device) alternate within the run after a warm-up of each; figures are medians of
--reps calls: wall ms of the call ending in a device synchronise, and psb_last_kernel_ms (the box: its slowest device)
and psb_last_launches.  Checked inside the run: both sides return the same ids and the same rows, field for field,
CIGARs included.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)
import bench  # noqa: E402
from db_align_probe import card  # noqa: E402
from search_probe import alternate  # noqa: E402

FIELDS = ("score", "end_query", "end_ref", "saturated", "beg_query", "beg_ref", "cigar_off", "cigar_ops")


def same_rows(a, b):
    assert a.n == b.n and a.cells == b.cells
    for f in FIELDS:
        x, y = getattr(a, f), getattr(b, f)
        assert (x is None) == (y is None) and (x is None or np.array_equal(x, y)), f


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--db", type=int, default=1000000)
    ap.add_argument("--nq", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from __graft_entry__ import build
    build()
    import parasail_rs_b200 as ps
    import psb_data

    ndev = ps._lib.lib().psb_device_count()
    if ndev <= 0:
        raise SystemExit("no CUDA device: nothing to measure")
    b62 = ps.Matrix.from_name("blosum62")
    query, cat, off = bench.make_inputs(args.db)
    residues = int(off[-1])
    t0 = time.perf_counter()
    db = ps.Database((cat, off), b62)
    ps._lib.lib().psb_synchronize()
    res = {"workload": f"bench.py's C2 database ({args.db} subjects, {residues} residues), BLOSUM62 open {bench.OPEN} ext {bench.GAP}",
           "reps": args.reps, "nq": args.nq, "visible_gpus": ndev, **card(),
           "single_device_build_s": round(time.perf_counter() - t0, 3), "boxes": {}}
    print(json.dumps({k: v for k, v in res.items() if k != "boxes"}), flush=True)
    many = {lq: [ps.Profile.new(psb_data.random_seq(4100 + lq, i, lq), False, b62) for i in range(args.nq)] for lq in (100, 400)}
    prof = ps.Profile.new(query, False, b62)

    def trace_aligner(p):
        return ps.Aligner.new().local().gap_open(bench.OPEN).gap_extend(bench.GAP).profile(p).use_trace().build()

    def scan(d):
        p = ps.Profile.new(query, False, b62)   # fresh each call: creation and upload are part of the figure
        out = ps.Aligner.new().local().gap_open(bench.OPEN).gap_extend(bench.GAP).profile(p).build().scan(d)
        return out, ps.kernel_ms(), ps.launches()

    def search(d, a, profs, k):
        out = a.search_many(d, profs, k)
        return out, ps.kernel_ms(), ps.launches()

    for n in [x for x in (1, 2, 4, 8) if x <= ndev]:
        t0 = time.perf_counter()
        box = ps.BoxDatabase((cat, off), b62, devices=list(range(n)))
        build_s = time.perf_counter() - t0
        row = {"build_s": round(build_s, 3), "shards": box.shards, "cases": {}}
        results, t = alternate(ps, {"box": lambda: scan(box), "one device": lambda: scan(db)}, args.reps)
        same_rows(results["box"], results["one device"])
        for side in t.values():
            side["gcups"] = round(len(query) * residues / (side["wall_ms"] * 1e-3) / 1e9, 1)
        row["cases"]["scan"] = t
        a = trace_aligner(prof)
        results, t = alternate(ps, {"box": lambda: search(box, a, [prof], 100), "one device": lambda: search(db, a, [prof], 100)}, args.reps)
        assert np.array_equal(results["box"][0], results["one device"][0])
        same_rows(results["box"][1], results["one device"][1])
        row["cases"]["search 400 k=100"] = t
        for lq, profs in many.items():
            a = trace_aligner(profs[0])
            results, t = alternate(ps, {"box": lambda: search(box, a, profs, 100), "one device": lambda: search(db, a, profs, 100)}, args.reps)
            assert np.array_equal(results["box"][0], results["one device"][0])
            same_rows(results["box"][1], results["one device"][1])
            row["cases"][f"many {args.nq} x {lq} k=100"] = t
        row["checked"] = "every case: same ids and rows as the single-device database, CIGARs included"
        res["boxes"][str(n)] = row
        print(f"N={n}: {json.dumps(row)}", flush=True)
        del box

    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
