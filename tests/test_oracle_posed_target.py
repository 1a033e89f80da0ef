"""Targets from posed scans in the CPU spec oracle (SPEC.md section 7.2, tests/posed_oracle.py): identity and translation-only poses against
set_target of the points transformed in numpy, partitions over add calls, LaserScan input, non-finite points and empty
scans, and the precision of the cell means at |t| = 100 m against an f64 numpy model."""
import math

import numpy as np
import pytest

from tests.posed_oracle import PosedOracle


def _scans(n=12, first=3, step=97):
    from gtsam_ndt_b200 import synth
    ranges, poses = synth.scans(n, traj_len=2000, first=first, step=step, **synth.SCAN_1080)
    return ranges, poses, synth.polar_to_points(ranges, synth.SCAN_1080["angle_min"], synth.SCAN_1080["angle_inc"])


def _same(o1, o2, nlevels):
    for l in range(nlevels):
        assert o1.geometry(l) == o2.geometry(l)
        n1, s1 = o1.sums(l)
        n2, s2 = o2.sums(l)
        assert np.array_equal(n1, n2) and np.array_equal(s1, s2)
        assert o1.cells(l).tobytes() == o2.cells(l).tobytes()


@pytest.mark.parametrize("overlap", [0, 1])
def test_identity_and_translation_poses_equal_set_target(overlap):
    import oracle
    from gtsam_ndt_b200 import synth
    _, _, pts = _scans()
    # points on a 2^-10 m raster, so that x + t (t a multiple of 2^-4, |x + t| < 2^13) is exact in f32 and in f64
    pts = [np.round(p * 1024.0).astype(np.float32) / np.float32(1024.0) for p in pts]
    pts[0][:5] = [[-0.0, 1.0], [2.0, -0.0], [-0.0, -0.0], [0.0, 0.0], [0.5, 0.25]]   # -0 becomes +0; SPEC 2-3 cannot tell
    xy, off = synth.pack(pts)
    res = [2.0, 1.0, 0.5]
    for trans in (np.zeros((len(pts), 2)), np.random.default_rng(5).integers(-800, 800, (len(pts), 2)) / 16.0):
        poses = np.concatenate([trans, np.zeros((len(pts), 1))], axis=1)
        moved = np.concatenate([(p.astype(np.float64) + t).astype(np.float32) for p, t in zip(pts, trans)])
        assert np.array_equal(moved.astype(np.float64), np.concatenate([p.astype(np.float64) + t for p, t in zip(pts, trans)]))
        a, b = PosedOracle(res, overlap=overlap), oracle.Oracle(res, overlap=overlap)
        a.set_target_scans(xy, off, poses)
        b.set_target(moved)
        _same(a, b, len(res))


def test_zero_angle_is_exact_identity():
    import oracle
    assert oracle.sincos(0.0) == (0.0, 1.0) and math.copysign(1.0, oracle.sincos(0.0)[0]) == 1.0


@pytest.mark.parametrize("grid", [None, (-100.0, -100.0, 200.0, 200.0)])
def test_partitions_over_add_calls_equal_one_set(grid):
    from gtsam_ndt_b200 import synth
    _, poses, pts = _scans()
    xy, off = synth.pack(pts)
    res = [1.0, 0.5]

    def make():
        o = PosedOracle(res, overlap=1)
        if grid:
            o.set_grid(*grid)
        return o

    whole = make()
    whole.set_target_scans(xy, off, poses)
    parts = [[0, 3], [3, 4], [4, 4], [4, 12]] if grid else [[0, 12]]
    for first_call in ("set", "add"):
        o = make()
        for j, (s0, s1) in enumerate(parts):
            pxy, poff = synth.pack(pts[s0:s1])
            (o.add_target_scans if j or first_call == "add" else o.set_target_scans)(pxy, poff, poses[s0:s1])
        _same(whole, o, len(res))


def test_ranges_through_polar_to_points():
    import oracle
    from gtsam_ndt_b200 import synth
    ranges, poses, pts = _scans(6)
    ranges = ranges.copy()
    ranges[1, 10:20] = np.nan
    ranges[2, 30:35] = np.inf
    amin, ainc = synth.SCAN_1080["angle_min"], synth.SCAN_1080["angle_inc"]
    per = [oracle.polar_to_points(r, amin, ainc, range_scale=1.0, range_min=0.05, range_max=40.0) for r in ranges]
    ref = synth.polar_to_points(ranges, amin, ainc, range_min=0.05, range_max=40.0)
    for a, b in zip(per, ref):
        assert a.tobytes() == b.tobytes()
    o1, o2 = PosedOracle([0.5]), PosedOracle([0.5])
    o1.set_target_scans(*synth.pack(per), poses)
    o2.set_target_scans(*synth.pack(ref), poses)
    _same(o1, o2, 1)


@pytest.mark.parametrize("grid", [None, (-100.0, -100.0, 200.0, 200.0)])
def test_non_finite_points_and_empty_scans_are_ignored(grid):
    from gtsam_ndt_b200 import synth
    _, poses, pts = _scans(5)
    bad = np.array([[np.nan, 1.0], [1.0, np.nan], [np.inf, 0.0], [0.0, -np.inf], [np.inf, -np.inf], [np.nan, np.nan]], np.float32)
    dirty = [np.concatenate([p[:100], bad, p[100:]]) for p in pts]
    empty = np.zeros((0, 2), np.float32)
    dirty_list = [empty, dirty[0], empty, empty] + dirty[1:] + [empty]
    dirty_poses = np.concatenate([[[1e3, -1e3, 2.0]], poses[:1], [[0.0, 0.0, 0.0], [5.0, 5.0, 5.0]], poses[1:], [[0.0, 0.0, 1.0]]])
    res = [1.0, 0.25]
    o1, o2 = PosedOracle(res), PosedOracle(res)
    if grid:
        o1.set_grid(*grid)
        o2.set_grid(*grid)
    o1.set_target_scans(*synth.pack(pts), poses)
    o2.set_target_scans(*synth.pack(dirty_list), dirty_poses)
    _same(o1, o2, len(res))


def _spec_transform(p, pose):
    import oracle
    sn, cs = oracle.sincos(pose[2])
    x, y = p[:, 0].astype(np.float64), p[:, 1].astype(np.float64)
    return cs * x - sn * y + pose[0], sn * x + cs * y + pose[1]


def test_cell_means_at_100m_are_within_the_fixed_point_unit():
    """Each cell mean of the posed build is within U/2 of the f64 mean of its points; the f32 map-frame route is not."""
    import oracle
    from gtsam_ndt_b200 import synth
    _, poses, pts = _scans(16)
    poses = poses + [100.0, -100.0, 0.0]        # the same scene with its origin 100 m away
    xy, off = synth.pack(pts)
    res = 0.25
    o = PosedOracle([res], min_points=3)
    o.set_target_scans(xy, off, poses)
    f32 = oracle.Oracle([res], min_points=3)
    f32.set_grid(*[float(v) for v in (o.geometry()["ox"], o.geometry()["oy"])],
                 o.geometry()["nhx"] * res, o.geometry()["nhy"] * res)
    f32.set_target(np.concatenate([synth.transform(p, q) for p, q in zip(pts, poses)]))
    g = o.geometry()
    assert f32.geometry() == g
    ox, oy, st = float(g["ox"]), float(g["oy"]), float(g["st"])
    inv = 1.0 / st
    U = res * 2.0 ** -22
    X, Y, Xs, Ys = [], [], [], []
    for p, q in zip(pts, poses):
        c, s = math.cos(q[2]), math.sin(q[2])
        x, y = p[:, 0].astype(np.float64), p[:, 1].astype(np.float64)
        X.append(c * x - s * y + q[0]); Y.append(s * x + c * y + q[1])
        a, b = _spec_transform(p, q)
        Xs.append(a); Ys.append(b)
    X, Y, Xs, Ys = map(np.concatenate, (X, Y, Xs, Ys))
    hx, hy = np.floor((X - ox) * inv).astype(np.int64), np.floor((Y - oy) * inv).astype(np.int64)
    hxs, hys = np.floor((Xs - ox) * inv).astype(np.int64), np.floor((Ys - oy) * inv).astype(np.int64)
    key = hy * g["njx"] + hx
    flipped = set(key[(hx != hxs) | (hy != hys)]) | set((hys * g["njx"] + hxs)[(hx != hxs) | (hy != hys)])
    n, sums = o.sums()
    n, sums = n.ravel(), sums.reshape(-1, 5)
    n32, s32 = f32.sums()
    n32, s32 = n32.ravel(), s32.reshape(-1, 5)
    order = np.argsort(key, kind="stable")
    ks, starts = np.unique(key[order], return_index=True)
    ends = np.append(starts[1:], len(order))
    err, err32, checked = 0.0, 0.0, 0
    for k, a, b in zip(ks, starts, ends):
        if k in flipped or b - a < 3:
            continue
        idx = order[a:b]
        jx, jy = k % g["njx"], k // g["njx"]
        cx = ox + float(jx) * st + 0.5 * res
        cy = oy + float(jy) * st + 0.5 * res
        assert n[k] == b - a
        mx, my = X[idx].mean(), Y[idx].mean()
        gx, gy = cx + sums[k, 0] / n[k] * U, cy + sums[k, 1] / n[k] * U
        err = max(err, abs(gx - mx), abs(gy - my))
        if n32[k] == n[k]:
            err32 = max(err32, abs(cx + s32[k, 0] / n32[k] * U - mx), abs(cy + s32[k, 1] / n32[k] * U - my))
        checked += 1
    print(f"cells checked {checked} (skipped {len(flipped)} with flipped membership): posed build max |mean error| {err:.3g} m, "
          f"U/2 = {U / 2:.3g} m; f32 map-frame route {err32:.3g} m")
    assert checked > 1000
    assert err <= U / 2 + 1e-9
    assert err32 > 10 * err
