"""Windowed search over scan pairs (ndt2d_relocalize_pairs, SPEC.md section 6.1): every pair must give the bytes of
ndt2d_set_target(target scan) + ndt2d_relocalize(source scan, the window's hypotheses, k, level) on the GPU and of the same
two steps of the CPU spec oracle; plus edge inputs, the device form, side effects, launch count, search quality and errors.
The first tests need no GPU."""
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _window_loop(c, w):
    nx, ny, nth, sx, sy, st = w
    out = []
    for ix in range(-nx, nx + 1):
        for iy in range(-ny, ny + 1):
            for it in range(-nth, nth + 1):
                out.append([np.float32(float(c[0]) + float(ix) * sx), np.float32(float(c[1]) + float(iy) * sy),
                            np.float32(float(c[2]) + float(it) * st)])
    return np.array(out, np.float32)


def test_window_hypotheses_match_the_formula():
    from gtsam_ndt_b200.matcher import window_hypotheses
    for c, w in [((0.1, -2.3, 0.7), (3, 2, 4, 0.1, 0.25, math.radians(1.5))), ((1e4 + 1 / 3, -7.77, 3.1), (0, 5, 1, 0.0, 0.013, 0.3)),
                 ((0.0, 0.0, 0.0), (0, 0, 0, 1.0, 1.0, 1.0))]:
        h = window_hypotheses(c, w)
        ref = _window_loop(c, w)
        assert h.dtype == np.float32 and h.tobytes() == ref.tobytes()
    # index order: ix outermost, it innermost
    h = window_hypotheses((0, 0, 0), (1, 1, 1, 1.0, 10.0, 100.0))
    assert h[1].tolist() == [-1.0, -10.0, 0.0] and h[3].tolist() == [-1.0, 0.0, -100.0] and h[9].tolist() == [0.0, -10.0, -100.0]


CPP = r'''
#include <cstdio>
#include "ndt2d.hpp"
int main()
{
    try {
        ndt2d::Matcher m;
        m.setResolutions({1.0f, 0.5f});
        std::vector<ndt2d::Point2f> pts;
        for (int i = 0; i < 400; ++i) pts.push_back({0.05f * (float)i - 10.0f, (i % 2) ? 3.0f : -3.0f + 0.01f * (float)i});
        for (int i = 0; i < 400; ++i) pts.push_back({pts[(size_t)i].x + 0.1f, pts[(size_t)i].y - 0.05f});
        std::vector<std::int64_t> off = {0, 400, 800};
        std::vector<std::pair<std::int32_t, std::int32_t>> pairs = {{0, 1}, {1, 0}};
        std::vector<ndt2d::Pose2d> centres(2);
        ndt2d_window w{2, 2, 1, 0, 0.1, 0.1, 0.01};
        std::vector<std::int64_t> idx;
        std::vector<double> sc;
        std::vector<ndt2d::Result> r = m.relocalizePairs(pts, off, pairs, centres, w, 3, 0, &idx, &sc);
        for (int p = 0; p < 2; ++p) {
            m.setTarget(std::vector<ndt2d::Point2f>(pts.begin() + off[(size_t)pairs[(size_t)p].first], pts.begin() + off[(size_t)pairs[(size_t)p].first + 1]));
            std::vector<float> hyp;
            for (int ix = -2; ix <= 2; ++ix)
                for (int iy = -2; iy <= 2; ++iy)
                    for (int it = -1; it <= 1; ++it) {
                        hyp.push_back((float)(0.0 + (double)ix * w.step_x));
                        hyp.push_back((float)(0.0 + (double)iy * w.step_y));
                        hyp.push_back((float)(0.0 + (double)it * w.step_th));
                    }
            std::vector<ndt2d::Point2f> src(pts.begin() + off[(size_t)pairs[(size_t)p].second], pts.begin() + off[(size_t)pairs[(size_t)p].second + 1]);
            std::vector<ndt2d::Result> one = m.relocalize(src, hyp, 3, 0);
            for (int j = 0; j < 3; ++j)
                if (std::memcmp(&one[(size_t)j], &r[(size_t)(3 * p + j)], sizeof(ndt2d::Result)) != 0) { std::printf("mismatch %d %d\n", p, j); return 1; }
        }
        std::printf("relocalizePairs ok %lld %.6f\n", (long long)idx[0], sc[0]);
        return 0;
    } catch (const std::exception &e) {
        std::fprintf(stderr, "%s\n", e.what());
        return 2;
    }
}
'''


def _compile_cpp(tmp_path):
    from gtsam_ndt_b200 import build
    assert os.path.exists(build.LIB_CUDA)
    libdir = os.path.dirname(build.LIB_CUDA)
    src = tmp_path / "reloc_pairs.cpp"
    src.write_text("#include <cstring>\n" + CPP)
    exe = str(tmp_path / "reloc_pairs")
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-L", libdir,
           "-lndt2d", f"-Wl,-rpath,{libdir}", "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_cpp_relocalize_pairs_compiles(tmp_path):
    _compile_cpp(tmp_path)


@pytest.mark.gpu
def test_cpp_relocalize_pairs_runs(tmp_path):
    r = subprocess.run([_compile_cpp(tmp_path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "relocalizePairs ok" in r.stdout, r.stdout + r.stderr


# ---- GPU ---------------------------------------------------------------------------------------------------------


def _between(a, b):
    c, s_ = math.cos(a[2]), math.sin(a[2])
    dx, dy = b[0] - a[0], b[1] - a[1]
    return np.array([c * dx + s_ * dy, -s_ * dx + c * dy, b[2] - a[2]])


@pytest.fixture(scope="module")
def world():
    from gtsam_ndt_b200 import synth
    sc = synth.SCAN_1080
    ranges, poses = synth.scans(14, traj_len=4000, first=50, step=9, sigma=0.01, **sc)      # neighbours 0.85 m apart
    scans = synth.polar_to_points(ranges, sc["angle_min"], sc["angle_inc"])
    scans = [s[:: (1 + i % 3)] for i, s in enumerate(scans)]                                # ragged: 1080 / 540 / 360 points
    scans += [np.zeros((0, 2), np.float32), scans[0][:4], np.full((30, 2), np.nan, np.float32)]
    E, T, N = 14, 15, 16                                                                    # empty, tiny, all-NaN
    pairs = [(i, i + 1) for i in range(0, 13, 2)] + [(i + 1, i) for i in range(0, 13, 4)] + [(5, 5), (0, 4), (3, 9), (0, 2),
             (E, 0), (0, E), (T, 1), (1, T), (N, 2), (2, N)]
    pp = np.vstack([poses, np.zeros((3, 3))])
    rng = np.random.default_rng(7)
    centres = np.array([_between(pp[t], pp[s]) + rng.normal(size=3) * [0.05, 0.05, 0.01] for t, s in pairs])
    return dict(scans=scans, pairs=pairs, centres=centres, poses=poses)


def _sequential(m, o, scans, t, s, hyp, k, level):
    """set_target + relocalize on the GPU handle and the oracle's set_target + sweep + top-k + align."""
    m.set_target(scans[t])
    bi, res = m.relocalize(scans[s], hyp, k=k, level=level)
    _, _, bs = m.sweep(scans[s], hyp, k=k, level=level, want_scores=False)
    bs = np.where(bi >= 0, bs, 0.0)
    o.set_target(scans[t])
    so, _, _ = o.sweep(scans[s], hyp, level=level)
    order = sorted((i for i in range(len(hyp)) if so[i] == so[i]), key=lambda i: (-so[i], i))[:k]
    oi = np.array(order + [-1] * (k - len(order)), np.int64)
    ores = np.zeros(k, res.dtype)
    for j, i in enumerate(order):
        ores[j] = o.align(scans[s], hyp[i].astype(np.float64))
    ores["status"][len(order):] = 3
    return bi, bs, res, oi, so, ores


CFGS = [dict(res=[0.5]), dict(res=[2.0, 1.0, 0.5]), dict(res=[1.0, 0.5], overlap=1), dict(res=[0.5], grid=(-120.0, -120.0, 240.0, 240.0)),
        dict(res=[1.0, 0.5], fused=0), dict(res=[1.0], chunk_bytes=3_000_000, fused=0), dict(res=[0.3, 0.1]),
        dict(res=[1.0, 0.5], min_points=5, eig_ratio=0.05)]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CFGS)
def test_relocalize_pairs_equals_set_target_plus_relocalize(world, cfg, monkeypatch):
    import gtsam_ndt_b200 as g
    import oracle
    from gtsam_ndt_b200 import synth
    cfg = dict(cfg)
    grid, chunk, res = cfg.pop("grid", None), cfg.pop("chunk_bytes", None), cfg.pop("res")
    if chunk:
        monkeypatch.setenv("NDT2D_PAIRS_BYTES", str(chunk))
    if cfg.pop("fused", 1) == 0:
        monkeypatch.setenv("NDT2D_PAIRS_FUSED", "0")
    m, o = g.NdtMatcher2D(res, **cfg), oracle.Oracle(res, **cfg)
    if grid:
        m.set_grid(*grid)
        o.set_grid(*grid)
    scans, pairs, centres = world["scans"], world["pairs"], world["centres"]
    xy, off = synth.pack(scans)
    win = (2, 1, 2, 0.05, 0.04, math.radians(0.7))                                          # 75 hypotheses
    for kk, k in enumerate((1, 4, 32)):
        level = kk % len(res)
        bi, bs, rr = m.relocalize_pairs(xy, off, pairs, centres, win, k=k, level=level)
        assert bi.shape == bs.shape == rr.shape == (len(pairs), k)
        for p, (t, s_) in enumerate(pairs):
            hyp = g.window_hypotheses(centres[p], win)
            si, ss, sr, oi, so, orr = _sequential(m, o, scans, t, s_, hyp, k, level)
            assert np.array_equal(bi[p], si) and bs[p].tobytes() == ss.tobytes() and rr[p].tobytes() == sr.tobytes(), (p, k, level)
            assert np.array_equal(bi[p], oi) and rr[p].tobytes() == orr.tobytes(), (p, k, level)
            assert bs[p].tobytes() == np.array([so[i] if i >= 0 else 0.0 for i in oi]).tobytes()


@pytest.mark.gpu
def test_edge_windows(world):
    """A zero-size window with k = 3: one candidate and two empty slots; step_x = 0: exact ties go to the smaller index."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    m = g.NdtMatcher2D([1.0, 0.5])
    scans, pairs, centres = world["scans"], world["pairs"][:6], world["centres"][:6]
    xy, off = synth.pack(scans)
    bi, bs, rr = m.relocalize_pairs(xy, off, pairs, centres, (0, 0, 0, 0.1, 0.1, 0.1), k=3)
    assert (bi[:, 0] == 0).all() and (bi[:, 1:] == -1).all() and (bs[:, 1:] == 0).all()
    empty = np.zeros(1, g.RESULT_DTYPE)
    empty["status"] = g.NO_OVERLAP
    assert all(rr[p, j].tobytes() == empty[0].tobytes() for p in range(len(pairs)) for j in (1, 2))
    for p, (t, s_) in enumerate(pairs):
        m.set_target(scans[t])
        assert rr[p, 0].tobytes() == m.align(scans[s_], g.window_hypotheses(centres[p], (0, 0, 0, 0.1, 0.1, 0.1))[0].astype(np.float64)).tobytes()
    win = (3, 1, 1, 0.0, 0.05, 0.01)                                                        # 7 identical copies of every (y, theta)
    bi, bs, rr = m.relocalize_pairs(xy, off, pairs, centres, win, k=4)
    for p in range(len(pairs)):
        ref = g.window_hypotheses(centres[p], win)
        assert (np.diff(bi[p][bs[p] == bs[p][0]]) > 0).all()
        assert bi[p][0] < 9                                                                  # the best (y, theta) first occurs at ix = -3
        assert np.array_equal(bi[p], bi[p][0] + 9 * np.arange(4)) and (ref[bi[p]] == ref[bi[p][0]]).all()


@pytest.mark.gpu
def test_long_targets_take_the_general_path(monkeypatch):
    """Targets too long for the shared-memory tables (40 000 points): the general path, still set_target + relocalize byte for byte."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    rng = np.random.default_rng(21)
    wall = np.stack([np.linspace(-40, 40, 40000), 5.0 + 0.02 * rng.normal(size=40000)], 1).astype(np.float32)
    box = np.concatenate([wall[::50], np.stack([wall[::50, 1] - 10, wall[::50, 0] / 4], 1)]).astype(np.float32)
    scans = [wall, box, (box + np.float32([0.1, 0.05])).astype(np.float32)]
    pairs = [(0, 1), (1, 2), (2, 1)]
    centres = np.zeros((3, 3))
    xy, off = synth.pack(scans)
    m = g.NdtMatcher2D([1.0])
    win = (2, 2, 1, 0.1, 0.1, 0.01)
    bi, bs, rr = m.relocalize_pairs(xy, off, pairs, centres, win, k=2)
    for p, (t, s_) in enumerate(pairs):
        m.set_target(scans[t])
        si, sres = m.relocalize(scans[s_], g.window_hypotheses(centres[p], win), k=2)
        assert np.array_equal(bi[p], si) and rr[p].tobytes() == sres.tobytes(), p


@pytest.mark.gpu
def test_device_form_side_effects_and_launches(world, small_world):
    import torch
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    scans, pairs, centres = world["scans"], world["pairs"], world["centres"]
    xy, off = synth.pack(scans)
    win = (3, 3, 2, 0.05, 0.05, 0.01)
    m = g.NdtMatcher2D([1.0, 0.5])
    m.set_target(small_world["map_xy"])
    before = m.align(small_world["scans"][2], small_world["init"][2])
    bi, bs, rr = m.relocalize_pairs(xy, off, pairs, centres, win, k=4)
    assert m.align(small_world["scans"][2], small_world["init"][2]).tobytes() == before.tobytes()     # the handle's map is untouched
    dev = torch.device("cuda", 0)
    d_xy, d_off = torch.from_numpy(xy).to(dev), torch.from_numpy(off).to(dev)
    d_c = torch.from_numpy(np.ascontiguousarray(centres)).to(dev)
    d_bi = torch.empty((len(pairs), 4), dtype=torch.int64, device=dev)
    d_bs = torch.empty((len(pairs), 4), dtype=torch.float64, device=dev)
    d_res = torch.empty((len(pairs), 4 * g.RESULT_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    m.relocalize_pairs_device(d_xy, d_off, off, pairs, d_c, win, 4, d_bi, d_bs, d_res)
    m.synchronize()
    assert np.array_equal(d_bi.cpu().numpy(), bi) and d_bs.cpu().numpy().tobytes() == bs.tobytes()
    assert d_res.cpu().numpy().tobytes() == rr.tobytes()
    # launches per call on the shared-memory path do not grow with the number of pairs
    many = [pairs[i % 13] for i in range(200)]
    cm = np.array([centres[i % 13] for i in range(200)])
    grow = []
    for pp, cc in ((pairs[:1], centres[:1]), (many, cm)):
        n0 = m.kernel_launches
        m.relocalize_pairs(xy, off, pp, cc, win, k=4)
        grow.append(m.kernel_launches - n0)
    assert grow[0] == grow[1] <= 4, grow


@pytest.mark.gpu
def test_search_finds_the_relative_pose():
    """Loop-closure style: drifted centres (0.5 m, 5 deg off), a 21 x 21 x 13 window; the best refined result is the true pose."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    sc = synth.SCAN_1080
    ranges, poses = synth.scans(24, traj_len=4000, first=200, step=3, sigma=0.01, **sc)
    scans = synth.polar_to_points(ranges, sc["angle_min"], sc["angle_inc"])
    rng = np.random.default_rng(5)
    pairs = [(i, i + 2) for i in range(0, 22)] + [(i + 2, i) for i in range(0, 20, 2)]
    truth = np.array([_between(poses[t], poses[s]) for t, s in pairs])
    drift = rng.uniform(-1, 1, size=(len(pairs), 3)) * [0.5, 0.5, math.radians(5)]
    xy, off = synth.pack(scans)
    m = g.NdtMatcher2D([2.0, 1.0, 0.5])
    bi, bs, rr = m.relocalize_pairs(xy, off, pairs, truth + drift, (10, 10, 6, 0.1, 0.1, math.radians(1.0)), k=4, level=1)
    good = 0
    for p in range(len(pairs)):
        ok = rr[p][rr[p]["status"] == g.CONVERGED]
        if len(ok) == 0:
            continue
        best = ok[np.argmax(ok["score"])]["pose"]
        d = best - truth[p]
        good += abs(d[0]) <= 0.03 and abs(d[1]) <= 0.03 and abs((d[2] + math.pi) % (2 * math.pi) - math.pi) <= 3e-3
    assert good >= 0.9 * len(pairs), (good, len(pairs))


@pytest.mark.gpu
def test_errors(world):
    """Each bad argument is refused with a message (a handle always has resolutions, so that case cannot arise)."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    scans, pairs, centres = world["scans"], world["pairs"][:3], world["centres"][:3]
    xy, off = synth.pack(scans)
    m = g.NdtMatcher2D([1.0, 0.5])
    win = (1, 1, 1, 0.1, 0.1, 0.01)
    bad = [dict(k=0), dict(k=33), dict(window=(-1, 1, 1, 0.1, 0.1, 0.01)), dict(window=(1, 1, 1, float("nan"), 0.1, 0.01)),
           dict(window=(1, 1, 1, 0.1, float("inf"), 0.01)), dict(window=(40000, 40000, 0, 0.1, 0.1, 0.01)), dict(level=2),
           dict(level=-1), dict(pairs=[(0, len(scans))]), dict(pairs=[(-1, 0)])]
    for b in bad:
        kw = dict(k=2, window=win, level=0, pairs=pairs)
        kw.update(b)
        pp = kw.pop("pairs")
        with pytest.raises(g.NdtError, match="relocalize_pairs|out of range"):
            m.relocalize_pairs(xy, off, pp, centres[:len(pp)], kw.pop("window"), **kw)
    bi, _, _ = m.relocalize_pairs(xy, off, pairs, centres, win, k=2)                         # the handle still works
    assert (bi >= 0).all()
