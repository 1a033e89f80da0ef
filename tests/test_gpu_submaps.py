"""Pairs against submaps of posed scans (ndt2d_align_submaps / ndt2d_relocalize_submaps, SPEC.md section 7.3): every pair
must give the bytes of ndt2d_set_target_scans(the submap's members) + ndt2d_align / ndt2d_relocalize on the GPU, and of the
same steps of the CPU spec oracle with SPEC 7.2 (tests/posed_oracle.py) for a subset; single-member identity submaps
against align_pairs / relocalize_pairs; device forms, side effects and launch counts; errors; search quality; the C++
mirror. pack_submaps and the C++ compile need no GPU."""
import math
import os
import subprocess

import numpy as np
import pytest

from tests.posed_oracle import PosedOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_pack_submaps_shapes_and_dtypes():
    from gtsam_ndt_b200 import pack_submaps
    so, ms, mp = pack_submaps([([3, 1], [[0, 0, 0], [1.0, 2.0, 0.5]]), ([], np.zeros((0, 3))), ([7], [(5.0, 6.0, -1.0)])])
    assert so.dtype == np.int64 and ms.dtype == np.int32 and mp.dtype == np.float64
    assert so.tolist() == [0, 2, 2, 3] and ms.tolist() == [3, 1, 7] and mp.shape == (3, 3) and mp.flags.c_contiguous
    assert mp[1].tolist() == [1.0, 2.0, 0.5] and mp[2].tolist() == [5.0, 6.0, -1.0]
    so, ms, mp = pack_submaps([])
    assert so.tolist() == [0] and ms.shape == (0,) and mp.shape == (0, 3)
    with pytest.raises(ValueError):
        pack_submaps([([1, 2], [[0, 0, 0]])])


CPP = r'''
#include <cmath>
#include <cstdio>
#include <cstring>
#include "ndt2d.hpp"
int main()
{
    try {
        ndt2d::Matcher m;
        m.setResolutions({1.0f, 0.5f});
        std::vector<ndt2d::Point2f> pts;
        std::vector<std::int64_t> off = {0};
        for (int s = 0; s < 4; ++s) {
            for (int i = 0; i < 500; ++i) {
                const double phi = 0.0125 * i;
                const float r = (float)(5.0 + std::sin(3.0 * phi) + 0.05 * s);
                pts.push_back({r * (float)std::cos(phi), r * (float)std::sin(phi)});
            }
            off.push_back((std::int64_t)pts.size());
        }
        std::vector<ndt2d::Submap> sub(2);
        sub[0].scans = {0, 1, 2};
        sub[0].poses = {{0.0, 0.0, 0.0}, {0.2, -0.1, 0.05}, {-0.3, 0.1, -0.02}};
        sub[1].scans = {3};
        sub[1].poses = {{100.0, -50.0, 3.1}};
        std::vector<std::pair<std::int32_t, std::int32_t>> pairs = {{0, 3}, {1, 0}};
        std::vector<ndt2d::Pose2d> centres = {{0.1, 0.0, 0.01}, {100.0, -50.0, 3.1}};
        ndt2d_window w{2, 2, 1, 0, 0.1, 0.1, 0.01};
        std::vector<std::int64_t> idx;
        std::vector<double> sc;
        std::vector<ndt2d::Result> r = m.relocalizeSubmaps(pts, off, sub, pairs, centres, w, 3, 0, &idx, &sc);
        std::vector<ndt2d::Result> a = m.alignSubmaps(pts, off, sub, pairs, centres);
        for (int p = 0; p < 2; ++p) {
            const ndt2d::Submap &s = sub[(size_t)pairs[(size_t)p].first];
            std::vector<ndt2d::Point2f> tp;
            std::vector<std::int64_t> to = {0};
            for (std::int32_t b : s.scans) {
                tp.insert(tp.end(), pts.begin() + off[(size_t)b], pts.begin() + off[(size_t)b + 1]);
                to.push_back((std::int64_t)tp.size());
            }
            m.setTargetScans(tp, to, s.poses);
            std::vector<float> hyp;
            for (int ix = -2; ix <= 2; ++ix)
                for (int iy = -2; iy <= 2; ++iy)
                    for (int it = -1; it <= 1; ++it) {
                        hyp.push_back((float)(centres[(size_t)p].x + (double)ix * w.step_x));
                        hyp.push_back((float)(centres[(size_t)p].y + (double)iy * w.step_y));
                        hyp.push_back((float)(centres[(size_t)p].theta + (double)it * w.step_th));
                    }
            std::vector<ndt2d::Point2f> src(pts.begin() + off[(size_t)pairs[(size_t)p].second], pts.begin() + off[(size_t)pairs[(size_t)p].second + 1]);
            std::vector<ndt2d::Result> one = m.relocalize(src, hyp, 3, 0);
            for (int j = 0; j < 3; ++j)
                if (std::memcmp(&one[(size_t)j], &r[(size_t)(3 * p + j)], sizeof(ndt2d::Result)) != 0) { std::printf("mismatch %d %d\n", p, j); return 1; }
            ndt2d::Result al = m.align(src, centres[(size_t)p]);
            if (std::memcmp(&al, &a[(size_t)p], sizeof(ndt2d::Result)) != 0) { std::printf("align mismatch %d\n", p); return 1; }
        }
        std::printf("submaps ok %lld %.6f\n", (long long)idx[0], sc[0]);
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
    src = tmp_path / "submaps.cpp"
    src.write_text(CPP)
    exe = str(tmp_path / "submaps")
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-L", libdir,
           "-lndt2d", f"-Wl,-rpath,{libdir}", "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_cpp_submaps_compiles(tmp_path):
    _compile_cpp(tmp_path)


def test_submap_search_probe_command_line():
    import sys
    tool = os.path.join(ROOT, "tools", "submap_search_probe.py")
    r = subprocess.run([sys.executable, tool, "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "--candidates" in r.stdout, r.stderr
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, tool, "--candidates", "1"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode != 0 and "GPU" in r.stderr, r.stdout + r.stderr


@pytest.mark.gpu
def test_cpp_submaps_runs(tmp_path):
    r = subprocess.run([_compile_cpp(tmp_path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "submaps ok" in r.stdout, r.stdout + r.stderr


# ---- GPU ---------------------------------------------------------------------------------------------------------


def _between(a, b):
    c, s_ = math.cos(a[2]), math.sin(a[2])
    dx, dy = b[0] - a[0], b[1] - a[1]
    return np.array([c * dx + s_ * dy, -s_ * dx + c * dy, b[2] - a[2]])


@pytest.fixture(scope="module")
def world():
    """26 keyframes 0.85 m apart (ragged), an empty, a tiny and an all-NaN scan; anchor-relative submaps of 0, 1, 5, 12 and 20
    members, with repeated members, the source among the members, members near |t| = 100 m and theta near +-pi."""
    from gtsam_ndt_b200 import synth
    sc = synth.SCAN_1080
    ranges, poses = synth.scans(26, traj_len=4000, first=50, step=9, sigma=0.01, **sc)
    scans = synth.polar_to_points(ranges, sc["angle_min"], sc["angle_inc"])
    scans = [s[:: (1 + i % 3)] for i, s in enumerate(scans)]                                # 1080 / 540 / 360 points
    scans += [np.zeros((0, 2), np.float32), scans[0][:4], np.full((30, 2), np.nan, np.float32)]
    E, T, N = 26, 27, 28
    rel = lambda a, js: [_between(poses[a], poses[j]) for j in js]                          # noqa: E731
    far = [[100.0 + 1 / 3, -100.0, math.pi - 0.01], [-99.5, 100.25, -math.pi + 0.02], [100.0, 100.0, 3.14159]]
    submaps = [
        ([], np.zeros((0, 3))),                                                             # 0: empty
        ([4], [[0.0, 0.0, 0.0]]),                                                           # 1: one member at the identity
        ([2, 3, 4, 5, 6], rel(4, [2, 3, 4, 5, 6])),                                         # 2: five, anchor 4
        (list(range(0, 20)), rel(10, range(0, 20))),                                        # 3: twenty, anchor 10
        ([7, 7, 8, 7], rel(8, [7, 7, 8]) + [_between(poses[8], poses[7]) + [0.3, -0.2, 0.01]]),   # 4: repeated members
        ([9, 10, 11], [far[0], far[1], far[2]]),                                            # 5: far members
        ([E, 12, T, N, 13], rel(12, [12, 12, 12, 12, 13])),                                 # 6: empty / tiny / NaN members
        (list(range(14, 26)), rel(20, range(14, 26))),                                      # 7: twelve, anchor 20
    ]
    pairs = [(2, 4), (2, 7), (2, 1), (3, 10), (3, 21), (4, 8), (4, 9), (5, 9), (6, 12), (6, 14), (7, 20), (7, 13), (1, 5), (0, 3),
             (2, E), (3, T), (7, N), (5, 10)]
    anchor = {0: 0, 1: 4, 2: 4, 3: 10, 4: 8, 5: 9, 6: 12, 7: 20}
    rng = np.random.default_rng(11)
    pp = np.vstack([poses, np.zeros((3, 3))])
    centres = []
    for g, s in pairs:
        c = _between(pp[anchor[g]], pp[s]) if s < 26 else np.zeros(3)
        if g == 5:
            c = np.array(far[0]) + [0.1, -0.1, 0.0]
        centres.append(c + rng.normal(size=3) * [0.05, 0.05, 0.01])
    return dict(scans=scans, poses=poses, submaps=submaps, pairs=pairs, centres=np.array(centres))


def _members(world, g):
    from gtsam_ndt_b200 import synth
    idx, pp = world["submaps"][g]
    xy, off = synth.pack([world["scans"][j] for j in idx])
    return xy, off, np.asarray(pp, np.float64).reshape(-1, 3)


def _make(cfg, monkeypatch, oracle=False):
    import gtsam_ndt_b200 as g
    cfg = dict(cfg)
    grid, chunk, res = cfg.pop("grid", None), cfg.pop("chunk_bytes", None), cfg.pop("res")
    if chunk:
        monkeypatch.setenv("NDT2D_PAIRS_BYTES", str(chunk))
    m = g.NdtMatcher2D(res, **cfg)
    o = PosedOracle(res, **cfg) if oracle else None
    if grid:
        m.set_grid(*grid)
        if o:
            o.set_grid(*grid)
    return m, o


CFGS = [dict(res=[0.5]), dict(res=[2.0, 1.0, 0.5]), dict(res=[1.0, 0.5], overlap=1), dict(res=[0.5], grid=(-120.0, -120.0, 240.0, 240.0)),
        dict(res=[1.0], chunk_bytes=3_000_000), dict(res=[1.0, 0.5], min_points=5, eig_ratio=0.05)]
ORACLE_PAIRS = (0, 5, 7, 8)       # five members, repeated members, far members, degenerate members


def _cases(world, cfg):
    """The pairs a configuration runs: with overlapping grids, submaps are limited to 10 922 points, so the twenty-member
    submap is left out."""
    keep = [p for p, (g, _) in enumerate(world["pairs"]) if not (cfg.get("overlap") and g == 3)]
    return [world["pairs"][p] for p in keep], world["centres"][keep]


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CFGS)
def test_align_submaps_equals_set_target_scans_plus_align(world, cfg, monkeypatch):
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    m, o = _make(cfg, monkeypatch, oracle=True)
    pairs, centres = _cases(world, cfg)
    xy, off = synth.pack(world["scans"])
    so, ms, mp = g.pack_submaps(world["submaps"])
    rr = m.align_submaps(xy, off, so, ms, mp, pairs, centres)
    assert rr.shape == (len(pairs),)
    for p, (sm, s_) in enumerate(pairs):
        txy, toff, tp = _members(world, sm)
        m.set_target_scans(txy, toff, tp)
        ref = m.align(world["scans"][s_], centres[p])
        assert rr[p].tobytes() == ref.tobytes(), (p, sm, s_)
        if p in ORACLE_PAIRS:
            o.set_target_scans(txy, toff, tp)
            assert rr[p].tobytes() == o.align(world["scans"][s_], centres[p]).tobytes(), (p, sm, s_)


def _sequential(m, scans, txy, toff, tp, s, hyp, k, level):
    m.set_target_scans(txy, toff, tp)
    bi, res = m.relocalize(scans[s], hyp, k=k, level=level)
    _, _, bs = m.sweep(scans[s], hyp, k=k, level=level, want_scores=False)
    return bi, np.where(bi >= 0, bs, 0.0), res


def _oracle_search(o, scans, txy, toff, tp, s, hyp, k, level):
    o.set_target_scans(txy, toff, tp)
    so, _, _ = o.sweep(scans[s], hyp, level=level)
    order = sorted((i for i in range(len(hyp)) if so[i] == so[i]), key=lambda i: (-so[i], i))[:k]
    import gtsam_ndt_b200 as g
    ores = np.zeros(k, g.RESULT_DTYPE)
    for j, i in enumerate(order):
        ores[j] = o.align(scans[s], hyp[i].astype(np.float64))
    ores["status"][len(order):] = g.NO_OVERLAP
    return np.array(order + [-1] * (k - len(order)), np.int64), ores


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", CFGS)
def test_relocalize_submaps_equals_set_target_scans_plus_relocalize(world, cfg, monkeypatch):
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    m, o = _make(cfg, monkeypatch, oracle=True)
    pairs, centres = _cases(world, cfg)
    xy, off = synth.pack(world["scans"])
    so, ms, mp = g.pack_submaps(world["submaps"])
    res = cfg["res"]
    win = (2, 1, 2, 0.05, 0.04, math.radians(0.7))                                          # 75 hypotheses
    for kk, k in enumerate((1, 4, 32)):
        level = kk % len(res)
        bi, bs, rr = m.relocalize_submaps(xy, off, so, ms, mp, pairs, centres, win, k=k, level=level)
        assert bi.shape == bs.shape == rr.shape == (len(pairs), k)
        for p, (sm, s_) in enumerate(pairs):
            hyp = g.window_hypotheses(centres[p], win)
            txy, toff, tp = _members(world, sm)
            si, ss, sr = _sequential(m, world["scans"], txy, toff, tp, s_, hyp, k, level)
            assert np.array_equal(bi[p], si) and bs[p].tobytes() == ss.tobytes() and rr[p].tobytes() == sr.tobytes(), (p, k, level)
            if k == 4 and p in ORACLE_PAIRS:
                oi, orr = _oracle_search(o, world["scans"], txy, toff, tp, s_, hyp, k, level)
                assert np.array_equal(bi[p], oi) and rr[p].tobytes() == orr.tobytes(), (p, k, level)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [None, "0"])
def test_identity_submaps_equal_pairs(world, fused, monkeypatch):
    """Single-member submaps at the identity pose: align_pairs / relocalize_pairs byte for byte (SPEC 7.2 identity rule),
    whichever path the pairs calls take."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    if fused is not None:
        monkeypatch.setenv("NDT2D_PAIRS_FUSED", fused)
    scans = world["scans"]
    xy, off = synth.pack(scans)
    pairs = [(i, i + 1) for i in range(0, 24, 2)] + [(5, 5), (0, 26), (26, 0), (27, 1), (1, 27), (28, 2), (2, 28)]
    so, ms, mp = g.pack_submaps([([t], np.zeros((1, 3))) for t in range(len(scans))])
    rng = np.random.default_rng(3)
    centres = rng.normal(size=(len(pairs), 3)) * [0.3, 0.3, 0.02]
    for res in ([1.0], [2.0, 1.0, 0.5]):
        m = g.NdtMatcher2D(res)
        a = m.align_pairs(xy, off, pairs, centres)
        b = m.align_submaps(xy, off, so, ms, mp, pairs, centres)
        assert a.tobytes() == b.tobytes()
        win = (3, 2, 2, 0.05, 0.05, 0.01)
        for k in (1, 4):
            ai, as_, ar = m.relocalize_pairs(xy, off, pairs, centres, win, k=k, level=len(res) - 1)
            bi, bs, br = m.relocalize_submaps(xy, off, so, ms, mp, pairs, centres, win, k=k, level=len(res) - 1)
            assert np.array_equal(ai, bi) and as_.tobytes() == bs.tobytes() and ar.tobytes() == br.tobytes()


@pytest.mark.gpu
def test_device_forms_side_effects_and_launches(world, small_world, monkeypatch):
    import torch
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    scans, pairs, centres = world["scans"], world["pairs"], world["centres"]
    xy, off = synth.pack(scans)
    so, ms, mp = g.pack_submaps(world["submaps"])
    win = (3, 3, 2, 0.05, 0.05, 0.01)
    m = g.NdtMatcher2D([1.0, 0.5])
    m.set_target(small_world["map_xy"])
    cells = [m.cells(l).tobytes() for l in range(2)]
    before = m.align(small_world["scans"][2], small_world["init"][2])
    n0 = m.kernel_launches
    ra = m.align_submaps(xy, off, so, ms, mp, pairs, centres)
    n1 = m.kernel_launches
    bi, bs, rr = m.relocalize_submaps(xy, off, so, ms, mp, pairs, centres, win, k=4)
    n2 = m.kernel_launches
    # one pose-table launch per call; per chunk (one here) the build and the align, or build, sweep, top-k, align and clear
    assert (n1 - n0, n2 - n1) == (3, 6), (n1 - n0, n2 - n1)
    assert [m.cells(l).tobytes() for l in range(2)] == cells                               # the handle's target is untouched
    assert m.align(small_world["scans"][2], small_world["init"][2]).tobytes() == before.tobytes()
    dev = torch.device("cuda", 0)
    d_xy, d_off = torch.from_numpy(xy).to(dev), torch.from_numpy(off).to(dev)
    d_mp = torch.from_numpy(mp).to(dev)
    d_c = torch.from_numpy(np.ascontiguousarray(centres)).to(dev)
    d_res1 = torch.empty((len(pairs), g.RESULT_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    n0 = m.kernel_launches
    m.align_submaps_device(d_xy, d_off, off, so, ms, d_mp, pairs, d_c, d_res1)
    m.synchronize()
    assert m.kernel_launches - n0 == 3
    assert d_res1.cpu().numpy().tobytes() == ra.tobytes()
    d_bi = torch.empty((len(pairs), 4), dtype=torch.int64, device=dev)
    d_bs = torch.empty((len(pairs), 4), dtype=torch.float64, device=dev)
    d_res = torch.empty((len(pairs), 4 * g.RESULT_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    n0 = m.kernel_launches
    m.relocalize_submaps_device(d_xy, d_off, off, so, ms, d_mp, pairs, d_c, win, 4, d_bi, d_bs, d_res)
    m.synchronize()
    assert m.kernel_launches - n0 == 6
    assert np.array_equal(d_bi.cpu().numpy(), bi) and d_bs.cpu().numpy().tobytes() == bs.tobytes()
    assert d_res.cpu().numpy().tobytes() == rr.tobytes()
    # several chunks: one pose table, then five launches per chunk
    monkeypatch.setenv("NDT2D_PAIRS_BYTES", "3000000")
    m1 = g.NdtMatcher2D([1.0])
    n0 = m1.kernel_launches
    m1.relocalize_submaps(xy, off, so, ms, mp, pairs, centres, win, k=4)
    launches = m1.kernel_launches - n0
    assert launches > 6 and (launches - 1) % 5 == 0, launches
    assert cells == [m.cells(l).tobytes() for l in range(2)]


@pytest.mark.gpu
def test_errors(world):
    """Every refused argument, on the host and the device forms; the handle works afterwards."""
    import torch
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    scans = world["scans"]
    xy, off = synth.pack(scans)
    so, ms, mp = g.pack_submaps(world["submaps"])
    pairs, centres = world["pairs"][:3], world["centres"][:3]
    m = g.NdtMatcher2D([1.0, 0.5])
    win = (1, 1, 1, 0.1, 0.1, 0.01)
    big = g.pack_submaps([(list(range(0, 26, 3)) * 7, np.zeros((63, 3)))])                 # 63 members, ~45 000 points
    nan_mp, inf_mp = mp.copy(), mp.copy()
    nan_mp[3, 1] = np.nan
    inf_mp[5, 2] = np.inf
    bad_ms_hi, bad_ms_lo = ms.copy(), ms.copy()
    bad_ms_hi[2] = len(scans)
    bad_ms_lo[4] = -1
    bad_so0 = so.copy()
    bad_so0[0] = 1
    bad_mono = so.copy()
    bad_mono[2], bad_mono[3] = bad_mono[3], bad_mono[2]
    cases = [dict(so=bad_so0, match="submap_offsets"), dict(so=bad_mono, match="not monotone"), dict(ms=bad_ms_hi, match="out of range"),
             dict(ms=bad_ms_lo, match="out of range"), dict(pairs=[(len(so) - 1, 0)], match="submap index"),
             dict(pairs=[(-1, 0)], match="submap index"), dict(pairs=[(0, len(scans))], match="scan index"),
             dict(so=big[0], ms=big[1], mp=big[2], pairs=[(0, 1)], match="65536 table slots"),
             dict(mp=nan_mp, match="not finite", host_only=True), dict(mp=inf_mp, match="not finite", host_only=True)]
    dev = torch.device("cuda", 0)
    d_xy, d_off = torch.from_numpy(xy).to(dev), torch.from_numpy(off).to(dev)
    out = torch.zeros((4 * 32 * 144,), dtype=torch.uint8, device=dev)
    d_bi = torch.zeros((4 * 32,), dtype=torch.int64, device=dev)
    for c in cases:
        kso, kms, kmp, kpairs = c.get("so", so), c.get("ms", ms), c.get("mp", mp), c.get("pairs", pairs)
        kc = centres[:len(kpairs)] if len(kpairs) <= len(centres) else np.zeros((len(kpairs), 3))
        with pytest.raises(g.NdtError, match=c["match"]):
            m.align_submaps(xy, off, kso, kms, kmp, kpairs, kc)
        with pytest.raises(g.NdtError, match=c["match"]):
            m.relocalize_submaps(xy, off, kso, kms, kmp, kpairs, kc, win, k=2)
        if c.get("host_only"):
            continue
        d_mp = torch.from_numpy(np.ascontiguousarray(kmp)).to(dev)
        d_c = torch.from_numpy(np.ascontiguousarray(kc)).to(dev)
        with pytest.raises(g.NdtError, match=c["match"]):
            m.align_submaps_device(d_xy, d_off, off, kso, kms, d_mp, kpairs, d_c, out)
        with pytest.raises(g.NdtError, match=c["match"]):
            m.relocalize_submaps_device(d_xy, d_off, off, kso, kms, d_mp, kpairs, d_c, win, 2, d_bi, None, out)
    for b in (dict(k=0), dict(k=33), dict(level=2), dict(window=(-1, 1, 1, 0.1, 0.1, 0.01))):
        kw = dict(k=2, window=win, level=0)
        kw.update(b)
        with pytest.raises(g.NdtError, match="relocalize_submaps"):
            m.relocalize_submaps(xy, off, so, ms, mp, pairs, centres, kw.pop("window"), **kw)
    # one submap whose auto-fitted lattice exceeds 2^31 cells: reported, its pairs NO_OVERLAP, every other pair as without it
    sub = list(world["submaps"][:3]) + [([3, 4], [[0.0, 0.0, 0.0], [3e5, 3e5, 0.0]])]
    so2, ms2, mp2 = g.pack_submaps(sub)
    pairs2 = [(2, 4), (3, 5), (1, 7), (3, 3), (2, 1)]
    c2 = np.zeros((5, 3))
    with pytest.raises(g.NdtError, match="submap exceeds 2"):
        m.align_submaps(xy, off, so2, ms2, mp2, pairs2, c2)
    with pytest.raises(g.NdtError, match="submap exceeds 2"):
        m.relocalize_submaps(xy, off, so2, ms2, mp2, pairs2, c2, win, k=2)
    keep = [0, 2, 4]
    ra = m.align_submaps(xy, off, so2, ms2, mp2, [pairs2[i] for i in keep], c2[keep])
    bi, bs, rr = m.relocalize_submaps(xy, off, so2, ms2, mp2, [pairs2[i] for i in keep], c2[keep], win, k=2)
    d_mp2 = torch.from_numpy(mp2).to(dev)
    d_c2 = torch.from_numpy(c2).to(dev)
    d_res = torch.zeros((5, 144), dtype=torch.uint8, device=dev)
    m.align_submaps_device(d_xy, d_off, off, so2, ms2, d_mp2, pairs2, d_c2, d_res)        # the device form reports nothing
    m.synchronize()
    got = np.frombuffer(d_res.cpu().numpy().tobytes(), g.RESULT_DTYPE)
    assert got[keep].tobytes() == ra.tobytes()
    assert (got["status"][[1, 3]] == g.NO_OVERLAP).all()
    d_res2 = torch.zeros((5 * 2, 144), dtype=torch.uint8, device=dev)
    d_bi2 = torch.zeros((5, 2), dtype=torch.int64, device=dev)
    d_bs2 = torch.zeros((5, 2), dtype=torch.float64, device=dev)
    m.relocalize_submaps_device(d_xy, d_off, off, so2, ms2, d_mp2, pairs2, d_c2, win, 2, d_bi2, d_bs2, d_res2)
    m.synchronize()
    got = np.frombuffer(d_res2.cpu().numpy().tobytes(), g.RESULT_DTYPE).reshape(5, 2)
    gi, gs = d_bi2.cpu().numpy(), d_bs2.cpu().numpy()
    assert got[keep].tobytes() == rr.tobytes() and np.array_equal(gi[keep], bi) and gs[keep].tobytes() == bs.tobytes()
    assert (got["status"][[1, 3]] == g.NO_OVERLAP).all()
    # the handle still works
    ra2 = m.align_submaps(xy, off, so, ms, mp, pairs, centres)
    assert (ra2["status"] != g.NO_OVERLAP).all()


@pytest.mark.gpu
def test_submap_search_finds_the_relative_pose():
    """Loop-closure style: sources taken 1.1 m from the nearest keyframe, centres drifted by up to 0.5 m / 5 deg, a
    21 x 21 x 13 window. Against a five-keyframe submap relative to the nearest keyframe, the best converged result is the
    true relative pose for every candidate. The count the single-keyframe search gets on the same candidates is printed."""
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    sc = synth.SCAN_1080
    nk = 14
    kr, kp = synth.scans(nk, traj_len=4000, first=300, step=24, sigma=0.01, **sc)           # keyframes 2.3 m apart
    sr, sp = synth.scans(nk - 4, traj_len=4000, first=300 + 2 * 24 + 12, step=24, sigma=0.01, **sc)   # half-way between keyframes
    keys = synth.polar_to_points(kr, sc["angle_min"], sc["angle_inc"])
    srcs = synth.polar_to_points(sr, sc["angle_min"], sc["angle_inc"])
    xy, off = synth.pack(keys + srcs)
    submaps, pairs, single, truth = [], [], [], []
    for i in range(len(srcs)):
        a = i + 2                                                                           # nearest keyframe (one of two)
        dist = math.hypot(*(sp[i][:2] - kp[a][:2]))
        assert dist >= 1.0, dist
        submaps.append((list(range(a - 2, a + 3)), [_between(kp[a], kp[j]) for j in range(a - 2, a + 3)]))
        pairs.append((i, nk + i))
        single.append((a, nk + i))
        truth.append(_between(kp[a], sp[i]))
    truth = np.array(truth)
    rng = np.random.default_rng(5)
    drift = rng.uniform(-1, 1, size=truth.shape) * [0.5, 0.5, math.radians(5)]
    so, ms, mp = g.pack_submaps(submaps)
    m = g.NdtMatcher2D([2.0, 1.0, 0.5])
    win = (10, 10, 6, 0.1, 0.1, math.radians(1.0))

    def good(rr):
        ok = 0
        for p in range(len(pairs)):
            c = rr[p][rr[p]["status"] == g.CONVERGED]
            if len(c) == 0:
                continue
            d = c[np.argmax(c["score"])]["pose"] - truth[p]
            ok += abs(d[0]) <= 0.05 and abs(d[1]) <= 0.05 and abs((d[2] + math.pi) % (2 * math.pi) - math.pi) <= math.radians(0.5)
        return ok

    _, _, rs = m.relocalize_submaps(xy, off, so, ms, mp, pairs, truth + drift, win, k=4, level=1)
    _, _, r1 = m.relocalize_pairs(xy, off, single, truth + drift, win, k=4, level=1)
    n_sub, n_single = good(rs), good(r1)
    print(f"\nwithin 5 cm / 0.5 deg: five-keyframe submaps {n_sub}/{len(pairs)}, single keyframe {n_single}/{len(pairs)}")
    assert n_sub == len(pairs), (n_sub, n_single, len(pairs))
