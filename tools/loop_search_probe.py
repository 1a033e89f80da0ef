#!/usr/bin/env python
"""Loop-closure search: ndt2d_relocalize_pairs (one call for all candidates) against the host loop of ndt2d_set_target +
ndt2d_relocalize per candidate on the same handle. 720- and 1080-beam keyframes near a drifted pose, centres about 0.5 m / 5 deg
off, a 21 x 21 x 13 = 5733-hypothesis window, k = 4, a 2.0 / 1.0 / 0.5 m pyramid, the sweep on the 1 m level.
Prints one JSON line per (beams, npairs): ms per call of each form, hypotheses/s of the whole call, kernel launches per call,
and whether every index, score and record is byte-equal between the two forms.
--against map: relocalisation in a saved map instead, ndt2d_relocalize_batch (one call for nscans scans) against the loop of
ndt2d_relocalize(scan, window_hypotheses(centre), k, level) per scan on the same handle, with a synth.make_map target;
nscans 1 / 16 / 256 / 4096 scans of 1080 beams, centres up to 0.5 m / 5 deg off their map poses, the same window, k and pyramid.
  python tools/loop_search_probe.py [--against pairs|map] [--reps 5]   (GPU box)"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gtsam_ndt_b200 as g  # noqa: E402
from gtsam_ndt_b200 import synth  # noqa: E402

WINDOW = (10, 10, 6, 0.1, 0.1, math.radians(1.0))
K, LEVEL, RES = 4, 1, [2.0, 1.0, 0.5]
MAP_TRAJ = 8000


def between(a, b):
    c, s = math.cos(a[2]), math.sin(a[2])
    dx, dy = b[0] - a[0], b[1] - a[1]
    return np.array([c * dx + s * dy, -s * dx + c * dy, b[2] - a[2]])


def candidates(nbeams, npairs, seed=3):
    """One query scan (the last) against npairs keyframes within a few metres of it."""
    sc = dict(nbeams=nbeams, angle_min=-0.75 * math.pi, angle_inc=1.5 * math.pi / nbeams)
    nkf = npairs + 1
    ranges, poses = synth.scans(nkf, traj_len=8000, first=1000, step=2, sigma=0.01, **sc)
    scans = synth.polar_to_points(ranges, sc["angle_min"], sc["angle_inc"])
    q = nkf - 1
    rng = np.random.default_rng(seed)
    pairs = [(i, q) for i in range(npairs)]
    drift = rng.uniform(-1, 1, size=(npairs, 3)) * [0.5, 0.5, math.radians(5)]
    centres = np.array([between(poses[t], poses[s]) for t, s in pairs]) + drift
    return scans, pairs, centres


def timed(fn, reps):
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        out.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(out)), r


def measure(m, batched, loop, loop_scores, n, reps):
    """Times both forms (median of reps after a warm-up) and compares their outputs byte for byte."""
    batched(), loop()                                   # warm-up: modules, buffers
    n0 = m.kernel_launches
    batched()
    launches_b = m.kernel_launches - n0
    n0 = m.kernel_launches
    loop()
    launches_l = m.kernel_launches - n0
    tb, (bi, bs, rr) = timed(batched, reps)
    tl, (li, _, lr) = timed(loop, reps)
    ls = loop_scores()                                  # the loop's sweep scores, for the score comparison (untimed)
    equal = bool(np.array_equal(bi, li) and rr.tobytes() == lr.tobytes() and bs.tobytes() == np.where(li >= 0, ls, 0.0).tobytes())
    conv = rr["status"] == g.CONVERGED
    H = (2 * WINDOW[0] + 1) * (2 * WINDOW[1] + 1) * (2 * WINDOW[2] + 1)
    return {"hyp_per_pair": H, "k": K, "batched_ms": round(tb, 3), "loop_ms": round(tl, 3), "speedup": round(tl / tb, 2),
            "batched_hyp_per_s": round(n * H / (tb * 1e-3)), "loop_hyp_per_s": round(n * H / (tl * 1e-3)),
            "launches_batched": launches_b, "launches_loop": launches_l, "byte_equal": equal, "converged_best": int(conv[:, 0].sum())}


def against_pairs(m, npairs_list, reps):
    for nbeams in (720, 1080):
        for npairs in npairs_list:
            scans, pairs, centres = candidates(nbeams, npairs)
            xy, off = synth.pack(scans)
            hyps = [g.window_hypotheses(c, WINDOW) for c in centres]

            def batched():
                return m.relocalize_pairs(xy, off, pairs, centres, WINDOW, k=K, level=LEVEL)

            def loop():
                bi = np.full((npairs, K), -1, np.int64)
                bs = np.zeros((npairs, K))
                rr = np.zeros((npairs, K), g.RESULT_DTYPE)
                for p, (t, s) in enumerate(pairs):
                    m.set_target(scans[t])
                    bi[p], rr[p] = m.relocalize(scans[s], hyps[p], k=K, level=LEVEL)
                return bi, bs, rr

            def loop_scores():
                ls = np.zeros((npairs, K))
                for p, (t, s) in enumerate(pairs):
                    m.set_target(scans[t])
                    _, _, ls[p] = m.sweep(scans[s], hyps[p], k=K, level=LEVEL, want_scores=False)
                return ls

            print(json.dumps({"beams": nbeams, "npairs": npairs, **measure(m, batched, loop, loop_scores, npairs, reps)}), flush=True)


def against_map(m, nscans_list, reps):
    m.set_target(synth.make_map(200, traj_len=MAP_TRAJ))
    for nscans in nscans_list:
        ranges, poses = synth.scans(nscans, traj_len=MAP_TRAJ, first=3, step=max(1, MAP_TRAJ // nscans), sigma=0.01, **synth.SCAN_1080)
        scans = synth.polar_to_points(ranges, synth.SCAN_1080["angle_min"], synth.SCAN_1080["angle_inc"])
        centres = poses + np.random.default_rng(3).uniform(-1, 1, size=(nscans, 3)) * [0.5, 0.5, math.radians(5)]
        xy, off = synth.pack(scans)
        hyps = [g.window_hypotheses(c, WINDOW) for c in centres]

        def batched():
            return m.relocalize_batch(xy, off, centres, WINDOW, k=K, level=LEVEL)

        def loop():
            bi = np.full((nscans, K), -1, np.int64)
            rr = np.zeros((nscans, K), g.RESULT_DTYPE)
            for b in range(nscans):
                bi[b], rr[b] = m.relocalize(scans[b], hyps[b], k=K, level=LEVEL)
            return bi, None, rr

        def loop_scores():
            return np.array([m.sweep(scans[b], hyps[b], k=K, level=LEVEL, want_scores=False)[2] for b in range(nscans)])

        print(json.dumps({"beams": 1080, "nscans": nscans, **measure(m, batched, loop, loop_scores, nscans, reps)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--against", choices=["pairs", "map"], default="pairs")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--npairs", type=int, nargs="+", default=None, help="npairs (pairs) or nscans (map) per call")
    a = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print(json.dumps({"gpu": q.stdout.strip().splitlines()[0] if q.stdout.strip() else "unknown"}), flush=True)
    m = g.NdtMatcher2D(RES)
    if a.against == "pairs":
        against_pairs(m, a.npairs or [1, 16, 64, 256], a.reps)
    else:
        against_map(m, a.npairs or [1, 16, 256, 4096], a.reps)


if __name__ == "__main__":
    main()
