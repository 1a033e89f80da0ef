#!/usr/bin/env python
"""Host-to-host latency of one align through the host API: packed points (ndt2d_align) and one LaserScan (ndt2d_align_batch_ranges).
  python tools/single_latency_probe.py   (GPU box)"""
import os, sys, time, json, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gtsam_ndt_b200 as g
from gtsam_ndt_b200 import synth
sc = synth.SCAN_1080
ranges, poses = synth.scans(4, traj_len=10000, first=0, step=1, **sc)
pts = synth.polar_to_points(ranges, sc["angle_min"], sc["angle_inc"])
init = poses + synth.uniform3(4) * np.array([0.03, 0.03, np.radians(0.3)])
map_xy = synth.make_map(2048, traj_len=2048, **sc)
m = g.NdtMatcher2D([0.25], device=0)
m.set_grid(-100.0, -100.0, 200.0, 200.0); m.set_target(map_xy)
one = np.ascontiguousarray(pts[0]); r1 = ranges[:1].copy()
out = {}
for name, fn in (("align_xy", lambda: m.align(one, init[0])), ("align_ranges", lambda: m.align_batch_ranges(r1, sc["angle_min"], sc["angle_inc"], init[:1], range_scale=1.0))):
    for _ in range(10): fn()
    lat = []
    for _ in range(200):
        t0 = time.perf_counter(); r = fn(); lat.append((time.perf_counter() - t0) * 1e6)
    out[name] = {"median_us": round(float(np.median(lat)), 1), "min_us": round(min(lat), 1), "iters": int(np.atleast_1d(r)["iterations"][0])}
print(json.dumps(out))
