#!/usr/bin/env python
"""Loop-closure search against submaps: ndt2d_relocalize_submaps (one call for all candidates) against the host loop of
ndt2d_set_target_scans(members) + ndt2d_relocalize per candidate on the same handle, and ndt2d_align_submaps against the loop
of ndt2d_set_target_scans + ndt2d_align.

M candidate submaps of S keyframes of 1080 beams each (keyframes 0.19 m apart, a submap = S consecutive keyframes relative to
its middle one), one query scan, centres about 0.5 m / 5 deg off, a 21 x 21 x 13 = 5733-hypothesis window, k = 4, a
2.0 / 1.0 / 0.5 m pyramid, the sweep on the 1 m level. Prints the GPU's name and power limit, then one JSON line per (S, M):
median ms per call of each form over --reps timed calls after a warm-up, kernel launches per call, and whether every index,
score and record is byte-equal between the two forms. Needs a CUDA GPU; fails without one.
  python tools/submap_search_probe.py [--members 5 20] [--candidates 1 16 64 256] [--reps 5]"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

WINDOW = (10, 10, 6, 0.1, 0.1, math.radians(1.0))
K, LEVEL, RES = 4, 1, [2.0, 1.0, 0.5]


def parse_args():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--members", type=int, nargs="+", default=[5, 20], help="keyframes per submap")
    ap.add_argument("--candidates", type=int, nargs="+", default=[1, 16, 64, 256], help="candidate submaps per call")
    ap.add_argument("--reps", type=int, default=5)
    return ap.parse_args()


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def between(a, b):
    c, s = math.cos(a[2]), math.sin(a[2])
    dx, dy = b[0] - a[0], b[1] - a[1]
    return np.array([c * dx + s * dy, -s * dx + c * dy, b[2] - a[2]])


def timed(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out)), r


def main():
    a = parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("submap_search_probe: no CUDA GPU visible; this tool measures the GPU and has no CPU fallback")
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    print(json.dumps({"gpu": gpu_info()}), flush=True)
    m = g.NdtMatcher2D(RES)
    sc = synth.SCAN_1080
    for S in a.members:
        for M in a.candidates:
            nkf = M + S
            ranges, poses = synth.scans(nkf + 1, traj_len=8000, first=1000, step=2, sigma=0.01, **sc)
            scans = synth.polar_to_points(ranges, sc["angle_min"], sc["angle_inc"])
            q = nkf                                                      # the query: the last scan
            submaps, anchors = [], []
            for c in range(M):
                anchor = c + S // 2
                submaps.append((list(range(c, c + S)), [between(poses[anchor], poses[j]) for j in range(c, c + S)]))
                anchors.append(anchor)
            rng = np.random.default_rng(3)
            drift = rng.uniform(-1, 1, size=(M, 3)) * [0.5, 0.5, math.radians(5)]
            centres = np.array([between(poses[an], poses[q]) for an in anchors]) + drift
            pairs = [(c, q) for c in range(M)]
            xy, off = synth.pack(scans)
            so, ms, mp = g.pack_submaps(submaps)
            members = [synth.pack([scans[j] for j in idx]) + (np.asarray(pp),) for idx, pp in submaps]
            hyps = [g.window_hypotheses(c, WINDOW) for c in centres]

            def reloc_batched():
                return m.relocalize_submaps(xy, off, so, ms, mp, pairs, centres, WINDOW, k=K, level=LEVEL)

            def reloc_loop():
                bi = np.full((M, K), -1, np.int64)
                rr = np.zeros((M, K), g.RESULT_DTYPE)
                for c in range(M):
                    m.set_target_scans(*members[c])
                    bi[c], rr[c] = m.relocalize(scans[q], hyps[c], k=K, level=LEVEL)
                return bi, rr

            def align_batched():
                return m.align_submaps(xy, off, so, ms, mp, pairs, centres)

            def align_loop():
                rr = np.zeros(M, g.RESULT_DTYPE)
                for c in range(M):
                    m.set_target_scans(*members[c])
                    rr[c] = m.align(scans[q], centres[c])
                return rr

            row = {"members": S, "candidates": M, "points_per_submap": int(off[S] - off[0]), "hyp_per_pair": len(hyps[0]), "k": K}
            for name, fb, fl in (("relocalize", reloc_batched, reloc_loop), ("align", align_batched, align_loop)):
                fb(), fl()                                               # warm-up: modules, buffers
                n0 = m.kernel_launches
                fb()
                lb = m.kernel_launches - n0
                n0 = m.kernel_launches
                fl()
                ll = m.kernel_launches - n0
                tb, rb = timed(fb, a.reps)
                tl, rl = timed(fl, a.reps)
                if name == "relocalize":
                    bi, bs, rr = rb
                    li, lr = rl
                    ls = np.zeros((M, K))
                    for c in range(M):                                   # the loop's sweep scores (untimed)
                        m.set_target_scans(*members[c])
                        ls[c] = m.sweep(scans[q], hyps[c], k=K, level=LEVEL, want_scores=False)[2]
                    equal = bool(np.array_equal(bi, li) and rr.tobytes() == lr.tobytes() and bs.tobytes() == np.where(li >= 0, ls, 0.0).tobytes())
                    conv = int((rr["status"][:, 0] == g.CONVERGED).sum())
                else:
                    equal = rb.tobytes() == rl.tobytes()
                    conv = int((rb["status"] == g.CONVERGED).sum())
                row[name] = {"batched_ms": round(tb, 3), "loop_ms": round(tl, 3), "loop_ms_per_candidate": round(tl / M, 4),
                             "speedup": round(tl / tb, 2), "launches_batched": lb, "launches_loop": ll, "byte_equal": equal,
                             "converged_best": conv}
            print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
