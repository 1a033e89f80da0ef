"""Entry-point behaviour of the calls over packed scans (ndt2d_align_pairs, ndt2d_relocalize_pairs, ndt2d_relocalize_batch)
that the per-call parity tests do not reach: the device form of align_pairs, a target whose auto-fitted lattice is too
large, and rejected offsets and pair indices. Return codes are read from the C ABI, since the Python wrappers check
some of these inputs themselves."""
import ctypes as C
import math

import numpy as np
import pytest

NDT2D_EINVAL = 1
WINDOW = (2, 2, 1, 0.05, 0.05, 0.01)


def _between(a, b):
    c, s_ = math.cos(a[2]), math.sin(a[2])
    dx, dy = b[0] - a[0], b[1] - a[1]
    return np.array([c * dx + s_ * dy, -s_ * dx + c * dy, b[2] - a[2]])


@pytest.fixture(scope="module")
def scans():
    """Eight 1080-beam scans 0.85 m apart (ragged: 1080 / 540 / 360 points), consecutive and repeated pairs, initial poses
    near the truth, and a ninth scan: scan 0 plus one point 1e8 m away, whose auto-fitted lattice at 0.5 m has more than
    2^31 cells."""
    from gtsam_ndt_b200 import synth
    sc = synth.SCAN_1080
    ranges, poses = synth.scans(8, traj_len=4000, first=50, step=9, sigma=0.01, **sc)
    pts = synth.polar_to_points(ranges, sc["angle_min"], sc["angle_inc"])
    pts = [s[:: (1 + i % 3)] for i, s in enumerate(pts)]
    far = np.vstack([pts[0], np.float32([[1e8, 0.0]])]).astype(np.float32)
    pairs = [(i, i + 1) for i in range(7)] + [(3, 1), (5, 5), (0, 2)]
    rng = np.random.default_rng(17)
    init = np.array([_between(poses[t], poses[s]) + rng.normal(size=3) * [0.03, 0.03, 0.003] for t, s in pairs])
    xy, off = synth.pack(pts + [far])
    return dict(xy=np.ascontiguousarray(xy, np.float32), off=np.ascontiguousarray(off, np.int64), pairs=np.int32(pairs),
                init=init, far=len(pts))


def _with_bad_pair(d, at=3):
    """The pairs and poses with (far target, scan 1) inserted at index `at`."""
    pairs = np.insert(d["pairs"], at, [d["far"], 1], axis=0).astype(np.int32)
    poses = np.insert(d["init"], at, [0.0, 0.0, 0.0], axis=0)
    return np.ascontiguousarray(pairs), np.ascontiguousarray(poses)


def _align_pairs_c(m, xy, off, pairs, init):
    from gtsam_ndt_b200 import RESULT_DTYPE
    from gtsam_ndt_b200.matcher import _ptr
    res = np.zeros(len(pairs), RESULT_DTYPE)
    rc = m._L.ndt2d_align_pairs(m._h, _ptr(xy), _ptr(off), len(off) - 1, _ptr(pairs), len(pairs), _ptr(init), _ptr(res))
    return rc, res


def _relocalize_pairs_c(m, xy, off, pairs, centres, k=3):
    from gtsam_ndt_b200 import RESULT_DTYPE
    from gtsam_ndt_b200.matcher import _ptr, _window
    bi = np.full((len(pairs), k), -1, np.int64)
    bs = np.zeros((len(pairs), k), np.float64)
    res = np.zeros((len(pairs), k), RESULT_DTYPE)
    rc = m._L.ndt2d_relocalize_pairs(m._h, 0, _ptr(xy), _ptr(off), len(off) - 1, _ptr(pairs), len(pairs), _ptr(centres),
                                     C.byref(_window(WINDOW)), k, _ptr(bi), _ptr(bs), _ptr(res))
    return rc, bi, bs, res


def _last_error(m):
    return m._L.ndt2d_last_error(m._h).decode()


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [1, 0])
def test_align_pairs_device_equals_host(scans, fused, monkeypatch):
    """align_pairs_device writes the records of align_pairs, byte for byte, on the shared-memory path and the general path."""
    import torch
    import gtsam_ndt_b200 as g
    if not fused:
        monkeypatch.setenv("NDT2D_PAIRS_FUSED", "0")
    m = g.NdtMatcher2D([1.0, 0.5])
    ref = m.align_pairs(scans["xy"], scans["off"], scans["pairs"], scans["init"])
    assert (ref["status"] == g.CONVERGED).sum() >= 6
    dev = torch.device("cuda", 0)
    d_xy, d_off = torch.from_numpy(scans["xy"]).to(dev), torch.from_numpy(scans["off"]).to(dev)
    d_init = torch.from_numpy(np.ascontiguousarray(scans["init"])).to(dev)
    d_res = torch.zeros((len(scans["pairs"]), g.RESULT_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    m.align_pairs_device(d_xy, d_off, scans["off"], scans["pairs"], d_init, d_res)
    m.synchronize()
    assert d_res.cpu().numpy().tobytes() == ref.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [1, 0])
def test_lattice_overflow_is_reported(scans, fused, monkeypatch):
    """A target whose lattice exceeds 2^31 cells: the host calls fail with the message, that pair's record is NO_OVERLAP,
    and every other pair's outputs are those of a call without it."""
    import gtsam_ndt_b200 as g
    if not fused:
        monkeypatch.setenv("NDT2D_PAIRS_FUSED", "0")
    xy, off = scans["xy"], scans["off"]
    pairs, init = _with_bad_pair(scans)
    m = g.NdtMatcher2D([0.5])

    with pytest.raises(g.NdtError, match=r"align_pairs: .*exceeds 2\^31 cells"):
        m.align_pairs(xy, off, pairs, init)
    rc, res = _align_pairs_c(m, xy, off, pairs, init)
    assert rc == NDT2D_EINVAL and "exceeds 2^31 cells" in _last_error(m)
    assert res[3]["status"] == g.NO_OVERLAP
    ref = m.align_pairs(xy, off, scans["pairs"], scans["init"])
    assert np.delete(res, 3).tobytes() == ref.tobytes()

    with pytest.raises(g.NdtError, match=r"relocalize_pairs: .*exceeds 2\^31 cells"):
        m.relocalize_pairs(xy, off, pairs, init, WINDOW, k=3)
    rc, bi, bs, rr = _relocalize_pairs_c(m, xy, off, pairs, init)
    assert rc == NDT2D_EINVAL and "exceeds 2^31 cells" in _last_error(m)
    rbi, rbs, rrr = m.relocalize_pairs(xy, off, scans["pairs"], scans["init"], WINDOW, k=3)
    assert (rbi >= 0).all()
    assert np.delete(bi, 3, axis=0).tobytes() == rbi.tobytes()
    assert np.delete(bs, 3, axis=0).tobytes() == rbs.tobytes()
    assert np.delete(rr, 3, axis=0).tobytes() == rrr.tobytes()


@pytest.mark.gpu
def test_bad_offsets_and_pairs_are_rejected(scans):
    """Non-monotone offsets, a negative first offset and an out-of-range pair index return NDT2D_EINVAL from the host forms of
    align_pairs, relocalize_pairs and relocalize_batch and from the device forms that read host offsets; the handle works
    afterwards."""
    import torch
    import gtsam_ndt_b200 as g
    from gtsam_ndt_b200.matcher import _ptr, _window
    xy, off, pairs, init = scans["xy"], scans["off"], scans["pairs"], scans["init"]
    nb = len(off) - 1
    swapped = off.copy()
    swapped[2], swapped[3] = off[3], off[2]                     # scan 1 ends after scan 2 starts: not monotone
    negative = off - 5
    out_of_range = pairs.copy()
    out_of_range[4] = [2, nb]

    m = g.NdtMatcher2D([1.0, 0.5])
    m.set_target(xy[off[1]:off[2]])
    dev = torch.device("cuda", 0)
    d_xy, d_off = torch.from_numpy(xy).to(dev), torch.from_numpy(off).to(dev)
    d_init = torch.from_numpy(np.ascontiguousarray(init)).to(dev)
    k, n = 3, len(pairs)
    d_bi = torch.empty((n, k), dtype=torch.int64, device=dev)
    d_bs = torch.empty((n, k), dtype=torch.float64, device=dev)
    d_res = torch.empty((n, k * g.RESULT_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    w = _window(WINDOW)
    for o, pp in [(swapped, pairs), (negative, pairs), (off, out_of_range)]:
        assert _align_pairs_c(m, xy, o, pp, init)[0] == NDT2D_EINVAL
        assert m._L.ndt2d_align_pairs_device(m._h, _ptr(d_xy), _ptr(d_off), _ptr(o), nb, _ptr(pp), n, _ptr(d_init),
                                             _ptr(d_res)) == NDT2D_EINVAL
        assert _relocalize_pairs_c(m, xy, o, pp, init, k)[0] == NDT2D_EINVAL
        assert m._L.ndt2d_relocalize_pairs_device(m._h, 0, _ptr(d_xy), _ptr(d_off), _ptr(o), nb, _ptr(pp), n, _ptr(d_init), C.byref(w),
                                                  k, _ptr(d_bi), _ptr(d_bs), _ptr(d_res)) == NDT2D_EINVAL
    centres = np.zeros((nb, 3))
    bi = np.full((nb, k), -1, np.int64)
    bs = np.zeros((nb, k), np.float64)
    res = np.zeros((nb, k), g.RESULT_DTYPE)
    for o in (swapped, negative):                                # relocalize_batch has no pairs
        assert m._L.ndt2d_relocalize_batch(m._h, 0, _ptr(xy), _ptr(o), nb, _ptr(centres), C.byref(w), k, _ptr(bi), _ptr(bs),
                                           _ptr(res)) == NDT2D_EINVAL
    m.synchronize()
    ref = m.align_pairs(xy, off, pairs, init)
    assert (ref["status"] == g.CONVERGED).sum() >= 6
    bi, _, _ = m.relocalize_batch(xy, off, np.zeros((nb, 3)), WINDOW, k=2)
    assert (bi >= 0).all()
