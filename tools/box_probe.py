#!/usr/bin/env python
"""probe (multi-GPU box): where does a psb_scan_box call spend its time?
 1. plain concurrent host->device copies from ONE pinned buffer to 1, 2, 4, ... devices: the PCIe / host-memory ceiling
 2. psb_scan_box timeline (PSB_DEBUG_TIMING) at the largest device count
 3. psb_scan_box wall time at 1, 2, 4, ... devices, with the library's own piece plan
usage: python tools/box_probe.py [n_gpus]"""
import os, sys, time, threading
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np, torch, bench
import parasail_rs_b200 as ps

ng_max = min(int(sys.argv[1]) if len(sys.argv) > 1 else 8, torch.cuda.device_count())
query, cat, off = bench.make_inputs(1000000)
pc = torch.empty(len(cat), dtype=torch.uint8, pin_memory=True); pc.numpy()[:] = cat
po = torch.empty(len(off), dtype=torch.int64, pin_memory=True); po.numpy()[:] = off
total = len(cat)

# 1. raw copies
for ng in [g for g in (1, 2, 4, 8) if g <= ng_max]:
    share = total // ng
    dst = [torch.empty(share, dtype=torch.uint8, device=f"cuda:{d}") for d in range(ng)]
    streams = [torch.cuda.Stream(device=d) for d in range(ng)]
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(ng)]
    for rep in range(3):
        for d in range(ng): torch.cuda.synchronize(d)
        t0 = time.perf_counter()
        for d in range(ng):
            with torch.cuda.device(d), torch.cuda.stream(streams[d]):
                ev[d][0].record(); dst[d].copy_(pc[d * share:(d + 1) * share], non_blocking=True); ev[d][1].record()
        for d in range(ng): torch.cuda.synchronize(d)
        wall = time.perf_counter() - t0
    per = [ev[d][0].elapsed_time(ev[d][1]) for d in range(ng)]
    print(f"raw H2D, {ng} devices x {share / 1e6:.1f} MB: wall {wall * 1e3:.3f} ms, per device ms {['%.3f' % x for x in per]}, "
          f"aggregate {total // ng * ng / wall / 1e9:.1f} GB/s, per device {share / max(per) / 1e6:.1f} GB/s", flush=True)
    del dst

b62 = ps.Matrix.from_name("blosum62")
a = ps.Aligner.new().local().gap_open(10).gap_extend(1).profile(ps.Profile.new(query, False, b62)).build()
cells = 400.0 * float(off[-1])
args = (pc.numpy(), po.numpy())

def timed(ng, reps=8):
    for _ in range(4): a.scan_box(args, ng)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter(); a.scan_box(args, ng); ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), min(ts)

# 3. wall time per device count
for ng in [g for g in (1, 2, 4, 8) if g <= ng_max]:
    med, mn = timed(ng)
    print(f"scan_box n_gpus {ng}: median {med * 1e3:.3f} ms (min {mn * 1e3:.3f}), {cells / med / 1e9:.0f} GCUPS, slowest device's kernels {ps.kernel_ms():.3f} ms", flush=True)

# 2. one timeline
sys.stdout.flush()
os.environ["PSB_DEBUG_TIMING"] = "1"
t0 = time.perf_counter(); a.scan_box(args, ng_max); dt = time.perf_counter() - t0
sys.stderr.flush()
print(f"timeline call: {dt * 1e3:.3f} ms", flush=True)
