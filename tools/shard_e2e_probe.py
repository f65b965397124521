#!/usr/bin/env python
"""probe: psb_scan_host on a 1/N shard of the C2 database (what each device of psb_scan_box sees at N GPUs), with the
library's own piece plan.  usage: python tools/shard_e2e_probe.py [nshards]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch, bench
import parasail_rs_b200 as ps

nsh = int(sys.argv[1]) if len(sys.argv) > 1 else 8
query, cat, off = bench.make_inputs(1000000)
total = int(off[-1])
cut = int(np.searchsorted(off, total // nsh))
sc, so = cat[: off[cut]], off[: cut + 1]
pc = torch.empty(len(sc), dtype=torch.uint8, pin_memory=True); pc.numpy()[:] = sc
po = torch.empty(len(so), dtype=torch.int64, pin_memory=True); po.numpy()[:] = so
b62 = ps.Matrix.from_name("blosum62")
a = ps.Aligner.new().local().gap_open(10).gap_extend(1).profile(ps.Profile.new(query, False, b62)).build()
cells = 400.0 * float(so[-1])
fresh = os.environ.get("PROBE_FRESH") == "1"   # a new Profile + Aligner for every call, as bench.py's e2e leg does
def call():
    al = ps.Aligner.new().local().gap_open(10).gap_extend(1).profile(ps.Profile.new(query, False, b62)).build() if fresh else a
    return al.scan_host((pc.numpy(), po.numpy()))
for _ in range(6): call()
ts = []
for _ in range(10):
    t0 = time.perf_counter(); call(); ts.append(time.perf_counter() - t0)
print(f"shard 1/{nsh} ({so[-1] / 1e6:.1f} MB): median {np.median(ts) * 1e3:.3f} ms, min {min(ts) * 1e3:.3f} ms, kernels {ps.kernel_ms():.3f} ms, "
      f"{cells / np.median(ts) / 1e9:.0f} GCUPS", flush=True)
# one call with the host and device timelines on stderr
os.environ["PSB_DEBUG_TIMING"] = "1"
call()
