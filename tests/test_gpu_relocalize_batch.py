"""Windowed search of a batch of scans against the handle's target (ndt2d_relocalize_batch, SPEC.md section 6.2): every scan
must give the bytes of ndt2d_relocalize(scan, the window's hypotheses, k, level) on the same GPU handle and of the CPU spec
oracle's set_target + sweep + top-k + align; plus awkward scans, edge windows, the device form, side effects, launch count,
search quality and errors. The C++ compile test needs no GPU."""
import math
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CPP = r'''
#include <cstdio>
#include <cstring>
#include "ndt2d.hpp"
int main()
{
    try {
        ndt2d::Matcher m;
        m.setResolutions({1.0f, 0.5f});
        std::vector<ndt2d::Point2f> pts;
        for (int i = 0; i < 400; ++i) pts.push_back({0.05f * (float)i - 10.0f, (i % 2) ? 3.0f : -3.0f + 0.01f * (float)i});
        for (int i = 0; i < 400; ++i) pts.push_back({pts[(size_t)i].x + 0.1f, pts[(size_t)i].y - 0.05f});
        m.setTarget(pts);
        std::vector<std::int64_t> off = {0, 400, 800};
        std::vector<ndt2d::Pose2d> centres = {{0.0, 0.0, 0.0}, {-0.1, 0.05, 0.002}};
        ndt2d_window w{2, 2, 1, 0, 0.1, 0.1, 0.01};
        std::vector<std::int64_t> idx;
        std::vector<double> sc;
        std::vector<ndt2d::Result> r = m.relocalizeBatch(pts, off, centres, w, 3, 0, &idx, &sc);
        for (int b = 0; b < 2; ++b) {
            const double *c = reinterpret_cast<const double *>(&centres[(size_t)b]);
            std::vector<float> hyp;
            for (int ix = -2; ix <= 2; ++ix)
                for (int iy = -2; iy <= 2; ++iy)
                    for (int it = -1; it <= 1; ++it) {
                        hyp.push_back((float)(c[0] + (double)ix * w.step_x));
                        hyp.push_back((float)(c[1] + (double)iy * w.step_y));
                        hyp.push_back((float)(c[2] + (double)it * w.step_th));
                    }
            std::vector<ndt2d::Point2f> scan(pts.begin() + off[(size_t)b], pts.begin() + off[(size_t)b + 1]);
            std::vector<ndt2d::Result> one = m.relocalize(scan, hyp, 3, 0);
            for (int j = 0; j < 3; ++j)
                if (std::memcmp(&one[(size_t)j], &r[(size_t)(3 * b + j)], sizeof(ndt2d::Result)) != 0) { std::printf("mismatch %d %d\n", b, j); return 1; }
        }
        std::printf("relocalizeBatch ok %lld %.6f\n", (long long)idx[0], sc[0]);
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
    src = tmp_path / "reloc_batch.cpp"
    src.write_text(CPP)
    exe = str(tmp_path / "reloc_batch")
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-L", libdir,
           "-lndt2d", f"-Wl,-rpath,{libdir}", "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_cpp_relocalize_batch_compiles(tmp_path):
    _compile_cpp(tmp_path)


@pytest.mark.gpu
def test_cpp_relocalize_batch_runs(tmp_path):
    r = subprocess.run([_compile_cpp(tmp_path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "relocalizeBatch ok" in r.stdout, r.stdout + r.stderr


# ---- GPU ---------------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def batch(small_world):
    """Scans of the small_world map with centres near their true poses; ragged (1080 / 540 / 360 points)."""
    scans = [s[:: (1 + i % 3)] for i, s in enumerate(small_world["scans"][:8])]
    rng = np.random.default_rng(11)
    centres = small_world["poses"][:8] + rng.normal(size=(8, 3)) * [0.05, 0.05, 0.01]
    return dict(map_xy=small_world["map_xy"], scans=scans, centres=centres)


def _per_scan(m, scan, hyp, k, level):
    """relocalize + sweep top-k scores of one scan on the GPU handle (empty slots: index -1, score 0)."""
    bi, res = m.relocalize(scan, hyp, k=k, level=level)
    _, _, bs = m.sweep(scan, hyp, k=k, level=level, want_scores=False)
    return bi, np.where(bi >= 0, bs, 0.0), res


def _oracle(o, scan, hyp, k, level, dtype):
    """The oracle's sweep + top-k by (-score, index) with NaN skipped + align from each of the k."""
    so, _, _ = o.sweep(scan, hyp, level=level)
    order = sorted((i for i in range(len(hyp)) if so[i] == so[i]), key=lambda i: (-so[i], i))[:k]
    oi = np.array(order + [-1] * (k - len(order)), np.int64)
    ores = np.zeros(k, dtype)
    for j, i in enumerate(order):
        ores[j] = o.align(scan, hyp[i].astype(np.float64))
    ores["status"][len(order):] = 3
    return oi, np.array([so[i] if i >= 0 else 0.0 for i in oi]), ores


CFGS = [dict(res=[0.5]), dict(res=[2.0, 1.0, 0.5]), dict(res=[1.0, 0.5], overlap=1), dict(res=[0.5], grid=(-100.0, -100.0, 200.0, 200.0)),
        dict(res=[1.0, 0.5], min_points=5, eig_ratio=0.05), dict(res=[0.3, 0.1])]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CFGS)
def test_relocalize_batch_equals_relocalize(batch, cfg):
    import gtsam_ndt_b200 as g
    import oracle
    from gtsam_ndt_b200 import synth
    cfg = dict(cfg)
    grid, res = cfg.pop("grid", None), cfg.pop("res")
    m, o = g.NdtMatcher2D(res, **cfg), oracle.Oracle(res, **cfg)
    if grid:
        m.set_grid(*grid)
        o.set_grid(*grid)
    m.set_target(batch["map_xy"])
    o.set_target(batch["map_xy"])
    scans, centres = batch["scans"], batch["centres"]
    xy, off = synth.pack(scans)
    win = (2, 1, 2, 0.05, 0.04, math.radians(0.7))                                          # 75 hypotheses
    for kk, k in enumerate((1, 4, 32)):
        level = kk % len(res)
        bi, bs, rr = m.relocalize_batch(xy, off, centres, win, k=k, level=level)
        assert bi.shape == bs.shape == rr.shape == (len(scans), k)
        for b, scan in enumerate(scans):
            hyp = g.window_hypotheses(centres[b], win)
            si, ss, sr = _per_scan(m, scan, hyp, k, level)
            assert np.array_equal(bi[b], si) and bs[b].tobytes() == ss.tobytes() and rr[b].tobytes() == sr.tobytes(), (b, k, level)
            oi, os_, orr = _oracle(o, scan, hyp, k, level, rr.dtype)
            assert np.array_equal(bi[b], oi) and bs[b].tobytes() == os_.tobytes() and rr[b].tobytes() == orr.tobytes(), (b, k, level)


@pytest.mark.gpu
def test_awkward_scans(batch):
    """Ragged, empty, 4-point, all-NaN and a 20 000-point scan (too long for the staged sweep) in one batch."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    scans = list(batch["scans"][:4])
    rng = np.random.default_rng(3)
    long = np.concatenate([batch["scans"][0] + rng.normal(size=batch["scans"][0].shape) * 0.01 for _ in range(19)])[:20000]
    scans += [np.zeros((0, 2), np.float32), scans[0][:4], np.full((30, 2), np.nan, np.float32), long.astype(np.float32)]
    centres = np.vstack([batch["centres"][:4], batch["centres"][[0, 0, 1, 0]]])
    xy, off = synth.pack(scans)
    m = g.NdtMatcher2D([2.0, 1.0, 0.5])
    m.set_target(batch["map_xy"])
    win = (2, 2, 1, 0.1, 0.1, 0.01)
    for k, level in ((4, 1), (32, 0)):
        bi, bs, rr = m.relocalize_batch(xy, off, centres, win, k=k, level=level)
        for b, scan in enumerate(scans):
            si, ss, sr = _per_scan(m, scan, g.window_hypotheses(centres[b], win), k, level)
            assert np.array_equal(bi[b], si) and bs[b].tobytes() == ss.tobytes() and rr[b].tobytes() == sr.tobytes(), (b, k, level)


@pytest.mark.gpu
def test_edge_windows(batch):
    """A zero-size window with k = 3: one candidate and two empty slots; step_x = 0: exact ties go to the smaller index."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    m = g.NdtMatcher2D([1.0, 0.5])
    m.set_target(batch["map_xy"])
    scans, centres = batch["scans"][:6], batch["centres"][:6]
    xy, off = synth.pack(scans)
    bi, bs, rr = m.relocalize_batch(xy, off, centres, (0, 0, 0, 0.1, 0.1, 0.1), k=3)
    assert (bi[:, 0] == 0).all() and (bi[:, 1:] == -1).all() and (bs[:, 1:] == 0).all()
    empty = np.zeros(1, g.RESULT_DTYPE)
    empty["status"] = g.NO_OVERLAP
    assert all(rr[b, j].tobytes() == empty[0].tobytes() for b in range(len(scans)) for j in (1, 2))
    for b, scan in enumerate(scans):
        h0 = g.window_hypotheses(centres[b], (0, 0, 0, 0.1, 0.1, 0.1))[0].astype(np.float64)
        assert rr[b, 0].tobytes() == m.align(scan, h0).tobytes()
    win = (3, 1, 1, 0.0, 0.05, 0.01)                                                        # 7 identical copies of every (y, theta)
    bi, bs, rr = m.relocalize_batch(xy, off, centres, win, k=4)
    for b in range(len(scans)):
        ref = g.window_hypotheses(centres[b], win)
        assert bi[b][0] < 9                                                                  # the best (y, theta) first occurs at ix = -3
        assert np.array_equal(bi[b], bi[b][0] + 9 * np.arange(4)) and (ref[bi[b]] == ref[bi[b][0]]).all()


@pytest.mark.gpu
def test_device_form_side_effects_and_launches(batch, small_world):
    import torch
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    scans, centres = batch["scans"], batch["centres"]
    xy, off = synth.pack(scans)
    win = (3, 3, 2, 0.05, 0.05, 0.01)
    m = g.NdtMatcher2D([1.0, 0.5])
    m.set_target(small_world["map_xy"])
    before = m.align(small_world["scans"][2], small_world["init"][2])
    bi, bs, rr = m.relocalize_batch(xy, off, centres, win, k=4)
    assert m.align(small_world["scans"][2], small_world["init"][2]).tobytes() == before.tobytes()     # the map is untouched
    dev = torch.device("cuda", 0)
    d_xy, d_off = torch.from_numpy(xy).to(dev), torch.from_numpy(off).to(dev)
    d_c = torch.from_numpy(np.ascontiguousarray(centres)).to(dev)
    n = len(scans)
    d_bi = torch.empty((n, 4), dtype=torch.int64, device=dev)
    d_bs = torch.empty((n, 4), dtype=torch.float64, device=dev)
    d_res = torch.empty((n, 4 * g.RESULT_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    m.relocalize_batch_device(d_xy, d_off, n, int(np.diff(off).max()), d_c, win, 4, d_bi, d_bs, d_res)
    m.synchronize()
    assert np.array_equal(d_bi.cpu().numpy(), bi) and d_bs.cpu().numpy().tobytes() == bs.tobytes()
    assert d_res.cpu().numpy().tobytes() == rr.tobytes()
    assert m.align(small_world["scans"][2], small_world["init"][2]).tobytes() == before.tobytes()
    # launches per call do not grow with the number of scans
    many = [scans[i % len(scans)] for i in range(200)]
    mxy, moff = synth.pack(many)
    mc = np.array([centres[i % len(scans)] for i in range(200)])
    grow = []
    for (pxy, poff, cc) in ((*synth.pack(scans[:1]), centres[:1]), (mxy, moff, mc)):
        n0 = m.kernel_launches
        m.relocalize_batch(pxy, poff, cc, win, k=4)
        grow.append(m.kernel_launches - n0)
    assert grow[0] == grow[1] <= 4, grow


@pytest.mark.gpu
def test_search_finds_the_map_pose(small_world):
    """Relocalisation in the map: centres drifted by up to 0.5 m / 5 deg, a 21 x 21 x 13 window; the best refined result is the
    true pose."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    scans, truth = small_world["scans"], small_world["poses"]
    rng = np.random.default_rng(5)
    drift = rng.uniform(-1, 1, size=(len(scans), 3)) * [0.5, 0.5, math.radians(5)]
    xy, off = synth.pack(scans)
    m = g.NdtMatcher2D([2.0, 1.0, 0.5])
    m.set_target(small_world["map_xy"])
    bi, bs, rr = m.relocalize_batch(xy, off, truth + drift, (10, 10, 6, 0.1, 0.1, math.radians(1.0)), k=4, level=1)
    good = 0
    for b in range(len(scans)):
        ok = rr[b][rr[b]["status"] == g.CONVERGED]
        if len(ok) == 0:
            continue
        best = ok[np.argmax(ok["score"])]["pose"]
        d = best - truth[b]
        good += abs(d[0]) <= 0.03 and abs(d[1]) <= 0.03 and abs((d[2] + math.pi) % (2 * math.pi) - math.pi) <= 3e-3
    assert good >= 0.9 * len(scans), (good, len(scans))


@pytest.mark.gpu
def test_errors(batch):
    """Each bad argument is refused with a message, and the handle works afterwards."""
    import torch
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    scans, centres = batch["scans"][:3], batch["centres"][:3]
    xy, off = synth.pack(scans)
    m = g.NdtMatcher2D([1.0, 0.5])
    win = (1, 1, 1, 0.1, 0.1, 0.01)
    with pytest.raises(g.NdtError, match="no target"):
        m.relocalize_batch(xy, off, centres, win, k=2)
    m.set_target(batch["map_xy"])
    bad = [dict(k=0), dict(k=33), dict(window=(-1, 1, 1, 0.1, 0.1, 0.01)), dict(window=(1, 1, 1, float("nan"), 0.1, 0.01)),
           dict(window=(1, 1, 1, 0.1, float("inf"), 0.01)), dict(window=(40000, 40000, 0, 0.1, 0.1, 0.01)), dict(level=2),
           dict(level=-1)]
    for b in bad:
        kw = dict(k=2, window=win, level=0)
        kw.update(b)
        with pytest.raises(g.NdtError, match="relocalize_batch|out of range"):
            m.relocalize_batch(xy, off, centres, kw.pop("window"), **kw)
    dev = torch.device("cuda", 0)
    d_xy, d_off = torch.from_numpy(xy).to(dev), torch.from_numpy(off).to(dev)
    d_c = torch.from_numpy(np.ascontiguousarray(centres)).to(dev)
    d_bi = torch.empty((3, 32), dtype=torch.int64, device=dev)
    d_res = torch.empty((3, 32 * g.RESULT_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    with pytest.raises(g.NdtError, match=r"relocalize_batch: nscans \* k"):                 # checked before anything is read
        m.relocalize_batch_device(d_xy, d_off, 1 << 26, 1080, d_c, win, 32, d_bi, None, d_res)
    with pytest.raises(g.NdtError, match="relocalize_batch"):
        m.relocalize_batch_device(d_xy, d_off, 3, -1, d_c, win, 2, d_bi, None, d_res)
    bi, _, _ = m.relocalize_batch(xy, off, centres, win, k=2)                                # the handle still works
    assert (bi >= 0).all()
