"""Kernel time of banded global alignment (psb_align_pairs_banded, parasail_nw_banded) on the band kernel, and of
the masked full-table path it replaces (PSB_NO_BAND_KERNEL=1).  Writes one JSON file (default
profiles/r6a_band_probe.json): per case the kernel ms (psb_last_kernel_ms), band cells per second and launches.

    python tools/band_probe.py [--out PATH] [--quick]
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402

import psb_data  # noqa: E402


def band_cells(lq, lr, k):
    d = lr - lq
    lo, hi = -k + min(d, 0), k + max(d, 0)

    def tri(m, n):
        return 0 if m <= 0 else (m * (m + 1) // 2 if m <= n else n * m - n * (n - 1) // 2)
    return lq * lr - tri(lr - hi - 1, lq) - tri(lq + lo - 1, lr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6a_band_probe.json"))
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    import __graft_entry__ as g
    g.build()
    import parasail_rs_b200 as ps
    from parasail_rs_b200 import _lib
    L = _lib.lib()
    b62 = ps.Matrix.from_name("blosum62")
    import subprocess
    import torch
    dev = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    if q.returncode == 0:
        dev += ", power limit " + q.stdout.strip()
    cases = []

    def record(name, lq, lr, k, n, ms, launches, **kw):
        cells = band_cells(lq, lr, k) * n
        cases.append(dict(case=name, lq=lq, lr=lr, k=k, pairs=n, kernel_ms=round(ms, 4), launches=launches,
                          band_cells=cells, band_cells_per_s=cells / (ms / 1e3) if ms > 0 else None, **kw))
        print(json.dumps(cases[-1]), flush=True)

    def best(fn):
        out = None
        for _ in range(args.reps):
            fn()
            ms, la = float(L.psb_last_kernel_ms()), int(L.psb_last_launches())
            out = (ms, la) if out is None or ms < out[0] else out
        return out

    def pair(n_res, seed):
        q = psb_data.random_seq(seed, 0, n_res)
        r = psb_data.mutate(q, seed, 1, 0.05, 0.002)
        return q, r

    for n_res in (20_000, 100_000):
        q, r = pair(n_res, n_res)
        for k in (16, 64, 256, 1024, 4096):
            a = ps.Aligner.new().global_().matrix(b62).gap_open(10).gap_extend(1).bandwidth(k).build()
            try:
                ms, la = best(lambda: a.banded_nw_batch([q], [r]))
                record("single pair, psb_align_pairs_banded", len(q), len(r), k, 1, ms, la)
            except ps.DeviceError as ex:
                cases.append(dict(case="single pair, psb_align_pairs_banded", lq=len(q), lr=len(r), k=k, error=str(ex)))
                print(json.dumps(cases[-1]), flush=True)
    q, r = pair(20_000, 20_000)
    a = ps.Aligner.new().global_().matrix(b62).gap_open(10).gap_extend(1).bandwidth(64).build()
    ms_band, la = best(lambda: a.banded_nw(bytes(q), bytes(r)))
    record("parasail_nw_banded, band kernel", len(q), len(r), 64, 1, ms_band, la)
    os.environ["PSB_NO_BAND_KERNEL"] = "1"
    ms_mask, la = best(lambda: a.banded_nw(bytes(q), bytes(r)))
    del os.environ["PSB_NO_BAND_KERNEL"]
    record("parasail_nw_banded, PSB_NO_BAND_KERNEL=1 (masked full table)", len(q), len(r), 64, 1, ms_mask, la,
           speedup_of_band_kernel=round(ms_mask / ms_band, 1))
    qs, rs = [], []
    for i in range(10_000):
        x = psb_data.random_seq(7, 2 * i, 10_000)
        qs.append(x); rs.append(psb_data.mutate(x, 7, 2 * i + 1, 0.05, 0.002))
    qc, qo = psb_data.concat(qs)
    rc, ro = psb_data.concat(rs)
    lq_sum = None
    for out in ("", "stats", "trace"):
        b = ps.Aligner.new().global_().matrix(b62).gap_open(10).gap_extend(1).bandwidth(64)
        b = b.use_stats() if out == "stats" else (b.use_trace() if out == "trace" else b)
        al = b.build()
        ms, la = best(lambda: al.banded_nw_batch((qc, qo), (rc, ro)))
        cells = sum(band_cells(int(qo[i + 1] - qo[i]), int(ro[i + 1] - ro[i]), 64) for i in range(len(qs)))
        cases.append(dict(case=f"batch of 10^4 pairs of 10 kb, nw{'_' + out if out else ''}", k=64, pairs=len(qs), kernel_ms=round(ms, 3),
                          launches=la, band_cells=cells, band_cells_per_s=cells / (ms / 1e3)))
        print(json.dumps(cases[-1]), flush=True)
    res = dict(device=dev, note="kernel ms = psb_last_kernel_ms, best of %d; BLOSUM62 10/1; pairs are mutated copies "
               "(5%% substitutions, 0.2%% indels)" % args.reps, cases=cases)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
