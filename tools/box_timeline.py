#!/usr/bin/env python
"""probe: one psb_scan_box call with PSB_DEBUG_TIMING (host and device timelines per device) after warm-up.
usage: python tools/box_timeline.py [n_gpus]"""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch, bench
import parasail_rs_b200 as ps

ng = min(int(sys.argv[1]) if len(sys.argv) > 1 else 8, torch.cuda.device_count())
query, cat, off = bench.make_inputs(1000000)
pc = torch.empty(len(cat), dtype=torch.uint8, pin_memory=True); pc.numpy()[:] = cat
po = torch.empty(len(off), dtype=torch.int64, pin_memory=True); po.numpy()[:] = off
a = ps.Aligner.new().local().gap_open(10).gap_extend(1).profile(ps.Profile.new(query, False, ps.Matrix.from_name("blosum62"))).build()
args = (pc.numpy(), po.numpy())
cells = 400.0 * float(off[-1])
for _ in range(6): a.scan_box(args, ng)
ts = []
for _ in range(10):
    t0 = time.perf_counter(); a.scan_box(args, ng); ts.append(time.perf_counter() - t0)
print(f"scan_box n_gpus {ng}: median {np.median(ts) * 1e3:.3f} ms (min {min(ts) * 1e3:.3f}), {cells / np.median(ts) / 1e9:.0f} GCUPS, "
      f"slowest device's kernels {ps.kernel_ms():.3f} ms", flush=True)
os.environ["PSB_DEBUG_TIMING"] = "1"
a.scan_box(args, ng)
sys.stderr.flush()
