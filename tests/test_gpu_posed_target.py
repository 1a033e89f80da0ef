"""Targets from posed scans on the GPU (ndt2d_set/add_target_scans, ndt2d_set/add_target_ranges and their device forms,
SPEC.md section 7.2): cells and sums byte-identical to the CPU spec oracle with SPEC 7.2 added (tests/posed_oracle.py) for every input form, overlap mode, pyramid,
lattice choice and set / sparse add / dense add; device forms against host forms; identity poses against set_target;
align_batch and relocalize_batch on a posed map against the oracle; argument errors; launch count; the C++ mirror; the
measurement tool's command line. The C++ compile test and the tool test need no GPU."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.posed_oracle import PosedOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CPP = r'''
#include <cmath>
#include <cstdio>
#include <cstring>
#include "ndt2d.hpp"
int main()
{
    try {
        const int nb = 360, ns = 4;
        const double amin = -3.14159265358979, ainc = 2.0 * 3.14159265358979 / nb;
        std::vector<float> ranges;
        std::vector<ndt2d::Point2f> pts;
        std::vector<std::int64_t> off = {0};
        std::vector<ndt2d::Pose2d> poses;
        for (int s = 0; s < ns; ++s) {
            poses.push_back({0.3 * s + 50.0, -0.2 * s - 40.0, 0.1 * s});
            for (int i = 0; i < nb; ++i) {
                const double phi = amin + (double)i * ainc;
                const float r = (float)(4.0 + std::sin(3.0 * phi) + 0.1 * s);
                ranges.push_back(r);
                pts.push_back({r * (float)std::cos(phi), r * (float)std::sin(phi)});
            }
            off.push_back((std::int64_t)pts.size());
        }
        ndt2d::Matcher a, b;
        a.setResolutions({1.0f, 0.5f});
        b.setResolutions({1.0f, 0.5f});
        a.setGrid(40.0f, -50.0f, 20.0f, 20.0f);
        b.setGrid(40.0f, -50.0f, 20.0f, 20.0f);
        a.setTargetScans(pts, off, poses);
        std::vector<float> r0(ranges.begin(), ranges.begin() + nb), r1(ranges.begin() + nb, ranges.end());
        b.setTargetRanges(r0, nb, amin, ainc, 0.0f, 100.0f, {poses[0]});
        b.addRangesToTarget(r1, nb, amin, ainc, 0.0f, 100.0f, std::vector<ndt2d::Pose2d>(poses.begin() + 1, poses.end()));
        std::vector<ndt2d::Point2f> p1(pts.begin(), pts.begin() + nb);
        ndt2d::Matcher c;
        c.setResolutions({1.0f, 0.5f});
        c.setGrid(40.0f, -50.0f, 20.0f, 20.0f);
        c.setTargetScans(p1, {0, nb}, {poses[0]});
        std::vector<ndt2d::Point2f> rest(pts.begin() + nb, pts.end());
        c.addScansToTarget(rest, {0, nb, 2 * nb, 3 * nb}, std::vector<ndt2d::Pose2d>(poses.begin() + 1, poses.end()));
        for (int l = 0; l < 2; ++l) {
            float g[5];
            int32_t d[4];
            if (ndt2d_level_geometry(a.handle(), l, g, d) != NDT2D_OK) return 3;
            std::vector<float> ca((size_t)d[2] * d[3] * 8), cb(ca.size()), cc(ca.size());
            if (ndt2d_get_cells(a.handle(), l, ca.data()) || ndt2d_get_cells(b.handle(), l, cb.data()) || ndt2d_get_cells(c.handle(), l, cc.data())) return 3;
            if (std::memcmp(ca.data(), cb.data(), ca.size() * 4) || std::memcmp(ca.data(), cc.data(), ca.size() * 4)) { std::printf("mismatch level %d\n", l); return 1; }
        }
        ndt2d::Result r = a.align(p1, {50.1, -40.1, 0.01});
        std::printf("posed target ok %.4f %.4f %d\n", r.pose[0], r.pose[1], r.status);
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
    src = tmp_path / "posed_target.cpp"
    src.write_text(CPP)
    exe = str(tmp_path / "posed_target")
    cmd = ["/usr/bin/g++", "-std=c++17", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-L", libdir,
           "-lndt2d", f"-Wl,-rpath,{libdir}", "-o", exe]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return exe


def test_cpp_posed_target_compiles(tmp_path):
    _compile_cpp(tmp_path)


@pytest.mark.gpu
def test_cpp_posed_target_runs(tmp_path):
    r = subprocess.run([_compile_cpp(tmp_path)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "posed target ok" in r.stdout, r.stdout + r.stderr


def test_map_rebuild_probe_command_line():
    tool = os.path.join(ROOT, "tools", "map_rebuild_probe.py")
    r = subprocess.run([sys.executable, tool, "--help"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and "--keyframes" in r.stdout, r.stderr
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, tool, "--keyframes", "4"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode != 0 and "GPU" in r.stderr, r.stdout + r.stderr


# ---- GPU ---------------------------------------------------------------------------------------------------------

SCALE = 0.001


@pytest.fixture(scope="module")
def data(small_world):
    """Ten 1080-beam scans of the small world at their poses (moved 60 m away), as f32 ranges, u16 ranges and packed points."""
    from gtsam_ndt_b200 import synth
    import oracle
    amin, ainc = synth.SCAN_1080["angle_min"], synth.SCAN_1080["angle_inc"]
    r32 = small_world["ranges"][:10].astype(np.float32).copy()
    r32[3, 100:110] = np.nan
    r32[4, 200:204] = np.inf
    u16 = np.where(np.isfinite(r32), np.clip(np.round(np.nan_to_num(r32) / SCALE), 0, 65535), 0).astype(np.uint16)
    poses = small_world["poses"][:10] + [60.0, -60.0, 0.0]
    rmin, rmax = 0.05, 1e30

    def pts_of(r, is_u16, decim=1):
        return [oracle.polar_to_points(row, amin, ainc * decim, range_scale=SCALE if is_u16 else 1.0, range_min=rmin, range_max=rmax)
                for row in r]
    return dict(r32=r32, u16=u16, poses=poses, amin=amin, ainc=ainc, rmin=rmin, rmax=rmax, pts_of=pts_of)


def _cmp(m, o, nlevels, what):
    for l in range(nlevels):
        g = o.geometry(l)
        gm = m.geometry(l)
        assert all(gm[k] == g[k] for k in g), (what, l, gm, g)
        n1, s1 = m.sums(l)
        n2, s2 = o.sums(l)
        assert np.array_equal(n1, n2) and np.array_equal(s1, s2), (what, l)
        assert m.cells(l).tobytes() == o.cells(l).tobytes(), (what, l)


def _call(m, op, form, d, scans, decim=1):
    """op: set / add; form: xy / f32 / u16; scans: slice of the data's scans (decim: every decim-th beam)."""
    from gtsam_ndt_b200 import synth
    poses = d["poses"][scans]
    if form == "xy":
        xy, off = synth.pack(d["pts_of"](d["r32"][scans, ::decim], False, decim))
        (m.set_target_scans if op == "set" else m.add_target_scans)(xy, off, poses)
    else:
        r = (d["r32"] if form == "f32" else d["u16"])[scans, ::decim]
        (m.set_target_ranges if op == "set" else m.add_target_ranges)(r, d["amin"], d["ainc"] * decim, poses, range_scale=SCALE,
                                                                       range_min=d["rmin"], range_max=d["rmax"])


def _ocall(o, op, form, d, scans, decim=1):
    from gtsam_ndt_b200 import synth
    xy, off = synth.pack(d["pts_of"]((d["r32"] if form != "u16" else d["u16"])[scans, ::decim], form == "u16", decim))
    (o.set_target_scans if op == "set" else o.add_target_scans)(xy, off, d["poses"][scans])


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["xy", "f32", "u16"])
@pytest.mark.parametrize("overlap", [0, 1])
@pytest.mark.parametrize("res", [[0.5], [2.0, 1.0, 0.5]])
@pytest.mark.parametrize("grid", [None, (0.0, -120.0, 150.0, 90.0)])
def test_set_and_add_equal_the_oracle(data, form, overlap, res, grid):
    """set (4 scans), sparse add (every 10th beam of one scan), dense add (5 scans); the explicit grid cuts the scene."""
    import gtsam_ndt_b200 as g
    m, o = g.NdtMatcher2D(res, overlap=overlap), PosedOracle(res, overlap=overlap)
    if grid:
        m.set_grid(*grid)
        o.set_grid(*grid)
    K = 4 if overlap else 1
    steps = [("set", slice(0, 4), 1), ("add", slice(4, 5), 10), ("add", slice(5, 10), 1)]
    for op, scans, decim in steps:
        _call(m, op, form, data, scans, decim)
        _ocall(o, op, form, data, scans, decim)
        _cmp(m, o, len(res), (op, scans, decim))
    # the second step takes the sparse path (touched cells only); the third is dense on every pyramid
    cells = [o.geometry(l)["njx"] * o.geometry(l)["njy"] for l in range(len(res))]
    assert all((1080 // 10) * K * 8 < c for c in cells)
    assert len(res) == 1 or not all(5 * 1080 * K * 8 < c for c in cells)


@pytest.mark.gpu
@pytest.mark.parametrize("res", [[0.5], [2.0, 1.0, 0.5]])
def test_device_forms_equal_host_forms(data, res):
    import torch
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    dev = torch.device("cuda", 0)
    xy, off = synth.pack(data["pts_of"](data["r32"], False))
    poses = np.ascontiguousarray(data["poses"])
    d_xy, d_off, d_p = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (xy, off, poses))
    kw = dict(range_scale=SCALE, range_min=data["rmin"], range_max=data["rmax"])
    for grid in (None, (0.0, -120.0, 150.0, 90.0)):
        for form in ("xy", "f32", "u16"):
            h, dv = g.NdtMatcher2D(res), g.NdtMatcher2D(res)
            if grid:
                h.set_grid(*grid)
                dv.set_grid(*grid)
            if form == "xy":
                h.set_target_scans(xy[:off[6]], off[:7], poses[:6])
                h.add_target_scans(xy[off[6]:], off[6:] - off[6], poses[6:])
                dv.set_target_scans_device(d_xy, d_off, 6, int(off[6]), d_p)
                d_off2 = (d_off[6:] - d_off[6]).contiguous()
                dv.add_target_scans_device(d_xy[int(off[6]):], d_off2, 4, int(off[-1] - off[6]), d_p[6:])
            else:
                r = np.ascontiguousarray(data["r32"] if form == "f32" else data["u16"])
                d_r = torch.from_numpy(r).to(dev)
                h.set_target_ranges(r[:6], data["amin"], data["ainc"], poses[:6], **kw)
                h.add_target_ranges(r[6:], data["amin"], data["ainc"], poses[6:], **kw)
                dv.set_target_ranges_device(d_r, form == "u16", 6, r.shape[1], data["amin"], data["ainc"], d_p, **kw)
                dv.add_target_ranges_device(d_r[6:], form == "u16", 4, r.shape[1], data["amin"], data["ainc"], d_p[6:], **kw)
            dv.synchronize()
            for l in range(len(res)):
                assert h.cells(l).tobytes() == dv.cells(l).tobytes() and h.geometry(l) == dv.geometry(l), (grid, form, l)
                assert all(np.array_equal(a, b) for a, b in zip(h.sums(l), dv.sums(l)))


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [0, 1])
def test_identity_poses_equal_set_target(data, overlap):
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    pts = data["pts_of"](data["r32"], False)
    pts[0] = np.concatenate([[[-0.0, 1.0], [np.nan, 2.0], [1.0, np.inf]], pts[0]]).astype(np.float32)
    xy, off = synth.pack(pts + [np.zeros((0, 2), np.float32)])
    res = [2.0, 1.0, 0.5]
    a, b = g.NdtMatcher2D(res, overlap=overlap), g.NdtMatcher2D(res, overlap=overlap)
    a.set_target_scans(xy, off, np.zeros((len(off) - 1, 3)))
    b.set_target(xy)
    for l in range(len(res)):
        assert a.geometry(l) == b.geometry(l) and a.cells(l).tobytes() == b.cells(l).tobytes()
        assert all(np.array_equal(u, v) for u, v in zip(a.sums(l), b.sums(l)))


@pytest.mark.gpu
def test_align_and_relocalize_on_a_posed_map(data, small_world):
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    res = [1.0, 0.5]
    m, o = g.NdtMatcher2D(res), PosedOracle(res)
    m.set_target_ranges(data["r32"], data["amin"], data["ainc"], data["poses"], range_scale=SCALE, range_min=data["rmin"],
                        range_max=data["rmax"])
    _ocall(o, "set", "f32", data, slice(0, 10))
    scans = [s[::2] for s in small_world["scans"][10:14]]
    init = small_world["poses"][10:14] + [60.0, -60.0, 0.0] + synth.uniform3(4) * [0.1, 0.1, 0.02]
    xy, off = synth.pack(scans)
    assert m.align_batch(xy, off, init).tobytes() == o.align_batch(xy, off, init).tobytes()
    win = (2, 2, 1, 0.1, 0.1, 0.01)
    bi, bs, rr = m.relocalize_batch(xy, off, init, win, k=3, level=1)
    for b, s in enumerate(scans):
        hyp = g.window_hypotheses(init[b], win)
        so, _, _ = o.sweep(s, hyp, level=1)
        order = sorted((i for i in range(len(hyp)) if so[i] == so[i]), key=lambda i: (-so[i], i))[:3]
        assert list(bi[b]) == order
        assert np.array_equal(bs[b], so[order])
        for j, i in enumerate(order):
            assert rr[b, j].tobytes() == o.align(s, hyp[i].astype(np.float64)).tobytes()


@pytest.mark.gpu
def test_bad_arguments_leave_the_target(data):
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    m = g.NdtMatcher2D([1.0, 0.5])
    xy, off = synth.pack(data["pts_of"](data["r32"][:3], False))
    poses = np.ascontiguousarray(data["poses"][:3])
    m.set_target_scans(xy, off, poses)
    before = [m.cells(l).tobytes() for l in range(2)]
    L, h = m._L, m._h
    P = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    bad_pose = poses.copy()
    bad_pose[1, 2] = np.nan
    inf_pose = poses.copy()
    inf_pose[2, 0] = np.inf
    off1 = off.copy()
    off1[0] = 1
    off2 = off.copy()
    off2[2] = off2[1] - 1
    r = np.ascontiguousarray(data["r32"][:3])
    for fn in (L.ndt2d_set_target_scans, L.ndt2d_add_target_scans):
        assert fn(h, P(xy), P(off), 3, P(bad_pose)) == 1
        assert fn(h, P(xy), P(off), 3, P(inf_pose)) == 1
        assert fn(h, P(xy), P(off), -1, P(poses)) == 1
        assert fn(h, P(xy), P(off1), 3, P(poses)) == 1
        assert fn(h, P(xy), P(off2), 3, P(poses)) == 1
    for fn in (L.ndt2d_set_target_ranges, L.ndt2d_add_target_ranges):
        assert fn(h, P(r), 0, 3, r.shape[1], data["amin"], data["ainc"], 1.0, 0.0, 1e30, P(bad_pose)) == 1
        assert fn(h, P(r), 0, 3, 0, data["amin"], data["ainc"], 1.0, 0.0, 1e30, P(poses)) == 1
        assert fn(h, P(r), 0, -2, r.shape[1], data["amin"], data["ainc"], 1.0, 0.0, 1e30, P(poses)) == 1
    for fn in (L.ndt2d_set_target_ranges_device, L.ndt2d_add_target_ranges_device):
        assert fn(h, None, 0, 3, 0, data["amin"], data["ainc"], 1.0, 0.0, 1e30, None) == 1
    for fn in (L.ndt2d_set_target_scans_device, L.ndt2d_add_target_scans_device):
        assert fn(h, None, None, -1, 0, None) == 1
        assert fn(h, None, None, 0, 5, None) == 1      # points without a scan
    assert [m.cells(l).tobytes() for l in range(2)] == before
    # add onto a target loaded without sums is refused
    cells = m.cells(1)
    m.set_cells(cells, level=1)
    with pytest.raises(g.NdtError):
        m.add_target_scans(xy, off, poses)


@pytest.mark.gpu
def test_launches_per_call(data):
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200 import synth
    xy, off = synth.pack(data["pts_of"](data["r32"], False))
    m = g.NdtMatcher2D([2.0, 1.0, 0.5])
    for call in (lambda: m.set_target_scans(xy, off, data["poses"]),
                 lambda: m.set_target_ranges(data["r32"], data["amin"], data["ainc"], data["poses"], range_min=data["rmin"])):
        n0 = m.kernel_launches
        call()
        assert m.kernel_launches - n0 <= 4      # pose table + bounding box + accumulate + finalise
    m.set_grid(-200.0, -200.0, 400.0, 400.0)
    n0 = m.kernel_launches
    m.set_target_scans(xy, off, data["poses"])
    assert m.kernel_launches - n0 == 3          # explicit grid: no bounding box
    # a scan added to a large map finalises only the cells it touches: one accumulate and one finalise launch for all levels
    scan = data["pts_of"](data["r32"][:1], False)[0]
    for res in ([2.0, 1.0, 0.5], [0.5]):
        m = g.NdtMatcher2D(res)
        m.set_grid(-200.0, -200.0, 400.0, 400.0)
        m.set_target(xy)
        assert all(len(scan) * 8 < m.geometry(l)["njx"] * m.geometry(l)["njy"] for l in range(len(res)))   # the sparse path
        n0 = m.kernel_launches
        m.add_target(scan)
        assert m.kernel_launches - n0 == 2, res
