"""Map rebuild from keyframes at new poses (SPEC.md section 7.2): time of the routes a SLAM front end has after a loop
closure, on the same seeded keyframes (synth.scans), at 0.25 m single level and on the 2 / 1 / 0.5 m pyramid.

  (a) host route: synth.transform of every keyframe on the CPU, then set_target of the map-frame points
  (b) set_target_scans from host buffers
  (c) set_target_scans_device and set_target_ranges_device (u16 ranges) with the keyframes resident on the GPU
  and add_target / add_target_ranges of one scan into the rebuilt map.

Prints one JSON line per measurement: host-to-host milliseconds (median of --reps after a warm-up), device milliseconds
(CUDA events on the handle's stream) and kernel launches per call, with the GPU's name and power limit. --check compares
the cells and sums of (c) with the CPU spec oracle (with SPEC 7.2, tests/posed_oracle.py) byte for byte. Needs a CUDA GPU; fails without one.

    python tools/map_rebuild_probe.py [--keyframes 2000] [--reps 10] [--check] [--out results.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def parse_args():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--keyframes", type=int, default=2000)
    ap.add_argument("--beams", type=int, default=1080)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--check", action="store_true", help="compare (c) with the CPU spec oracle")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    return ap.parse_args()


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    a = parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("map_rebuild_probe: no CUDA GPU visible; this tool measures the GPU and has no CPU fallback")
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    card = gpu_info()
    amin = -0.75 * np.pi
    ainc = 1.5 * np.pi / a.beams
    ranges, poses = synth.scans(a.keyframes, nbeams=a.beams, angle_min=amin, angle_inc=ainc)
    pts = synth.polar_to_points(ranges, amin, ainc)
    xy, off = synth.pack(pts)
    scale = 0.001
    u16 = np.clip(np.round(ranges / scale), 0, 65535).astype(np.uint16)
    dev = torch.device("cuda", 0)
    d_xy, d_off, d_p, d_u16 = (torch.from_numpy(np.ascontiguousarray(v)).to(dev) for v in (xy, off, poses, u16))
    rmin = 1e-3       # the synthetic scans mark a missing return with 0
    lines = []

    def emit(**kw):
        kw.update(gpu=card, keyframes=a.keyframes, points=int(off[-1]))
        line = json.dumps(kw)
        print(line, flush=True)
        lines.append(line)

    def timed(m, fn):
        ext = torch.cuda.ExternalStream(m.stream)
        fn()
        m.synchronize()
        host, devt, launches = [], [], []
        for _ in range(a.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n0 = m.kernel_launches
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record(ext)
            fn()
            e1.record(ext)
            m.synchronize()
            host.append((time.perf_counter() - t0) * 1e3)
            e1.synchronize()
            devt.append(e0.elapsed_time(e1))
            launches.append(m.kernel_launches - n0)
        return dict(host_ms=float(np.median(host)), device_ms=float(np.median(devt)), launches=int(np.median(launches)))

    for res in ([0.25], [2.0, 1.0, 0.5]):
        m = g.NdtMatcher2D(res)
        kw = dict(res=res)
        emit(route="a_host_transform_set_target", **kw,
             **timed(m, lambda: m.set_target(np.concatenate([synth.transform(p, q) for p, q in zip(pts, poses)]))))
        emit(route="b_set_target_scans_host", **kw, **timed(m, lambda: m.set_target_scans(xy, off, poses)))
        emit(route="c_set_target_scans_device", **kw,
             **timed(m, lambda: m.set_target_scans_device(d_xy, d_off, a.keyframes, int(off[-1]), d_p)))
        cells_c = [m.cells(l) for l in range(len(res))]
        sums_c = [m.sums(l) for l in range(len(res))]
        emit(route="c_set_target_ranges_device_u16", **kw,
             **timed(m, lambda: m.set_target_ranges_device(d_u16, True, a.keyframes, a.beams, amin, ainc, d_p, range_scale=scale,
                                                           range_min=rmin)))
        cells_u = [m.cells(l) for l in range(len(res))]
        sums_u = [m.sums(l) for l in range(len(res))]
        emit(route="add_target_one_scan_host_transform", **kw, **timed(m, lambda: m.add_target(synth.transform(pts[0], poses[0]))))
        emit(route="add_target_ranges_one_scan", **kw,
             **timed(m, lambda: m.add_target_ranges(ranges[:1], amin, ainc, poses[:1], range_min=rmin)))
        if a.check:
            import oracle
            from tests.posed_oracle import PosedOracle
            o = PosedOracle(res)
            o.set_target_scans(xy, off, poses)
            ok = all(cells_c[l].tobytes() == o.cells(l).tobytes() and all(np.array_equal(u, v) for u, v in zip(sums_c[l], o.sums(l)))
                     for l in range(len(res)))
            ou = PosedOracle(res)
            upts = [oracle.polar_to_points(r, amin, ainc, range_scale=scale, range_min=rmin) for r in u16]
            ou.set_target_scans(*synth.pack(upts), poses)
            ok_u = all(cells_u[l].tobytes() == ou.cells(l).tobytes() and all(np.array_equal(u, v) for u, v in zip(sums_u[l], ou.sums(l)))
                       for l in range(len(res)))
            emit(route="check_c_against_oracle", res=res, scans_bytes_equal=bool(ok), ranges_u16_bytes_equal=bool(ok_u))
            if not (ok and ok_u):
                sys.exit("map_rebuild_probe: (c) differs from the CPU spec oracle")
        m.close()
    if a.out:
        with open(a.out, "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
