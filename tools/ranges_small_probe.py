#!/usr/bin/env python
"""Small LaserScan batches (ndt2d_align_batch_ranges[_device]): block-per-scan kernel against the warp-per-scan kernel with helper
warps, kernel ms per batch, identical records, and the host-API latency of a single scan.  python tools/ranges_small_probe.py  (GPU box)"""
import os, sys, time, json, numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import gtsam_ndt_b200 as g
from gtsam_ndt_b200 import synth
sc = synth.SCAN_1080
ranges, poses = synth.scans(1250, traj_len=10000, first=0, step=1, **sc)
init = poses + synth.uniform3(1250) * np.array([0.03, 0.03, np.radians(0.3)])
map_xy = synth.make_map(2048, traj_len=2048, **sc)
dev = torch.device('cuda', 0)
for B in (1, 148, 600, 1184, 1250):
    row = {"scans": B}
    for mode in ("block", "help"):
        os.environ["NDT2D_BLOCK_ALIGN_MAX"] = str(1 << 30) if mode == "block" else "0"
        os.environ["NDT2D_ALIGN_HELP"] = "1"
        m = g.NdtMatcher2D([0.25], device=0, stream=torch.cuda.current_stream().cuda_stream)
        m.set_grid(-100.0, -100.0, 200.0, 200.0); m.set_target(map_xy)
        d_r = torch.from_numpy(ranges[:B]).to(dev); d_i = torch.from_numpy(np.ascontiguousarray(init[:B])).to(dev)
        d_res = torch.zeros(B * 144, dtype=torch.uint8, device=dev)
        f = lambda: m._ck(m._L.ndt2d_align_batch_ranges_device(m._h, g.matcher._ptr(d_r), 0, B, 1080, sc["angle_min"], sc["angle_inc"], 1.0, 0.0, 3e38, g.matcher._ptr(d_i), g.matcher._ptr(d_res)))
        for _ in range(5): f()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); [f() for _ in range(20)]; e1.record(); torch.cuda.synchronize()
        row[mode + "_ms"] = round(e0.elapsed_time(e1) / 20, 4)
        row[mode + "_sha"] = hash(d_res.cpu().numpy().tobytes()) & 0xffffff
        if B == 1:
            h = ranges[:1].copy()
            for _ in range(5): m.align_batch_ranges(h, sc["angle_min"], sc["angle_inc"], init[:1], range_scale=1.0)
            t0 = time.perf_counter()
            for _ in range(50): m.align_batch_ranges(h, sc["angle_min"], sc["angle_inc"], init[:1], range_scale=1.0)
            row[mode + "_host_api_us"] = round((time.perf_counter() - t0) / 50 * 1e6, 1)
        m.close()
    row["identical"] = row["block_sha"] == row["help_sha"]
    print(json.dumps(row), flush=True)
