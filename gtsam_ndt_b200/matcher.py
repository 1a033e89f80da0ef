"""Host-side mirror of the matcher interface named by BASELINE.json's north_star: set target map or scan,
set cell resolution, align(scan, initial pose) -> pose, score, Hessian; plus the batched and sweep paths.

Python front end over the C ABI (include/ndt2d.h); the C++ mirror is include/ndt2d.hpp. Reference
class/signature: none citable (the mount is /root/reference/README.md:1 only, SURVEY.md 8b).
All compute runs in libndt2d.so on the GPU; nothing here (or below) falls back to the CPU.
"""
import ctypes as C

import numpy as np

from . import _lib

RESULT_DTYPE = np.dtype([("pose", "f8", 3), ("score", "f8"), ("grad", "f8", 3), ("hessian", "f8", (3, 3)),
                         ("iterations", "i4"), ("status", "i4"), ("count", "i4"), ("reserved", "i4")])
assert RESULT_DTYPE.itemsize == 144

CONVERGED, MAX_ITERATIONS, STALLED, NO_OVERLAP = 0, 1, 2, 3


class NdtError(RuntimeError):
    pass


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(C.c_void_p)
    if hasattr(a, "data_ptr"):            # torch tensor (device or pinned host): plumbing only
        return C.c_void_p(a.data_ptr())
    return C.c_void_p(int(a))


def pinned_array(shape, dtype, write_combined=False):
    """A numpy array in page-locked host memory from the library's allocator (ndt2d_host_alloc_flags): full-speed copies for
    the host-buffer calls. write_combined: for input buffers the CPU only writes. The memory is freed with the array."""
    L = _lib.load()
    dt = np.dtype(dtype)
    n = int(np.prod(shape)) * dt.itemsize
    p = C.c_void_p()
    if L.ndt2d_host_alloc_flags(C.byref(p), n, 1 if write_combined else 0) != 0:
        raise NdtError(f"ndt2d_host_alloc_flags({n}) failed: {L.ndt2d_last_error(None).decode()}")

    class _Owner:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            L.ndt2d_host_free(self.ptr)

    buf = (C.c_ubyte * max(n, 1)).from_address(p.value)
    buf._owner = _Owner(p)          # keeps the allocation alive as long as any view of `buf` exists
    return np.frombuffer(buf, dtype=dt, count=int(np.prod(shape))).reshape(shape)


def _window(window):
    """A search window as ndt2d_window: a _lib.Window, or (nx, ny, nth, step_x, step_y, step_th)."""
    if isinstance(window, _lib.Window):
        return window
    nx, ny, nth, sx, sy, st = window
    return _lib.Window(int(nx), int(ny), int(nth), 0, float(sx), float(sy), float(st))


def window_hypotheses(centre, window):
    """The hypotheses of a search window around centre, as ndt2d_relocalize_pairs sweeps them (SPEC.md section 6.1):
    f32 (H, 3), index j = ((ix + nx)(2ny + 1) + (iy + ny))(2nth + 1) + (it + nth), value (float)(c + (double)i * step)."""
    w = _window(window)
    if min(w.nx, w.ny, w.nth) < 0:
        raise ValueError("window half-widths must be >= 0")
    c = np.asarray(centre, np.float64).reshape(3)
    ix, iy, it = np.meshgrid(np.arange(-w.nx, w.nx + 1, dtype=np.float64), np.arange(-w.ny, w.ny + 1, dtype=np.float64),
                             np.arange(-w.nth, w.nth + 1, dtype=np.float64), indexing="ij")
    # numpy evaluates each f64 product and sum on its own (no fused multiply-add), then rounds once to f32
    return np.stack([c[0] + ix * w.step_x, c[1] + iy * w.step_y, c[2] + it * w.step_th], -1).reshape(-1, 3).astype(np.float32)


def pack_submaps(submaps):
    """Submaps for align_submaps / relocalize_submaps (SPEC.md section 7.3) from a list of (scan_indices, poses[n, 3]):
    returns (submap_offsets int64 [nsubmaps + 1], member_scans int32 [nmembers], member_poses float64 [nmembers, 3])."""
    offsets, scans, poses = [0], [], []
    for idx, pp in submaps:
        idx = np.asarray(idx, np.int64).reshape(-1)
        pp = np.asarray(pp, np.float64).reshape(-1, 3)
        if len(idx) != len(pp):
            raise ValueError("every member scan needs one pose")
        scans.append(idx)
        poses.append(pp)
        offsets.append(offsets[-1] + len(idx))
    member_scans = np.concatenate(scans).astype(np.int32) if scans else np.zeros(0, np.int32)
    member_poses = np.ascontiguousarray(np.concatenate(poses) if poses else np.zeros((0, 3)), np.float64)
    return np.array(offsets, np.int64), member_scans, member_poses


def _submap_args(submap_offsets, member_scans, member_poses=None):
    so = np.ascontiguousarray(submap_offsets, np.int64).reshape(-1)
    ms = np.ascontiguousarray(member_scans, np.int32).reshape(-1)
    if len(so) < 1 or so[-1] != len(ms):
        raise ValueError("submap_offsets must have nsubmaps + 1 entries and end at the number of member scans")
    if member_poses is None:
        return so, ms
    mp = np.ascontiguousarray(member_poses, np.float64).reshape(-1, 3)
    if len(mp) != len(ms):
        raise ValueError("member_scans / member_poses sizes disagree")
    return so, ms, mp


class NdtMatcher2D:
    """One handle = one CUDA device + one stream (not thread-safe)."""

    def __init__(self, resolutions=(1.0,), device=0, stream=None, **params):
        self._L = _lib.load()
        h = C.c_void_p()
        rc = (self._L.ndt2d_create(device, C.byref(h)) if stream is None
              else self._L.ndt2d_create_on_stream(device, C.c_void_p(stream), C.byref(h)))
        if rc != 0:
            raise NdtError(f"ndt2d_create failed ({rc}): {self._L.ndt2d_last_error(None).decode()}")
        self._h = h
        self.device = device
        self.params = _lib.Params()
        self._L.ndt2d_default_params(C.byref(self.params))
        if params:
            self.set_params(**params)
        self.set_resolutions(resolutions)

    # -- lifecycle -------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._L.ndt2d_destroy(self._h)
            self._h = None

    __del__ = close

    def _ck(self, rc):
        if rc != 0:
            raise NdtError(f"libndt2d error {rc}: {self._L.ndt2d_last_error(self._h).decode()}")

    def synchronize(self):
        self._ck(self._L.ndt2d_synchronize(self._h))

    def set_upload_relay(self, relay_device, fraction=0.5):
        """About `fraction` of the input chunks of the host-buffer batch calls go host -> relay_device -> this GPU (that GPU's
        PCIe link, then NVLink) instead of over this GPU's own link; relay_device < 0 switches it off (ndt2d_set_upload_relay)."""
        self._ck(self._L.ndt2d_set_upload_relay(self._h, int(relay_device), float(fraction)))

    @property
    def stream(self):
        return self._L.ndt2d_stream(self._h) or 0

    @property
    def kernel_launches(self):
        return self._L.ndt2d_kernel_launches(self._h)

    # -- configuration ---------------------------------------------------------------------------
    def set_params(self, **kw):
        for k, v in kw.items():
            if not hasattr(self.params, k):
                raise AttributeError(k)
            setattr(self.params, k, v)
        self._ck(self._L.ndt2d_set_params(self._h, C.byref(self.params)))

    def set_resolution(self, res):
        self.set_resolutions([res])

    def set_resolutions(self, res):
        r = np.ascontiguousarray(np.atleast_1d(res), np.float32)
        self.nlevels = len(r)
        self._ck(self._L.ndt2d_set_resolutions(self._h, r.ctypes.data_as(_lib.c_f32p), len(r)))

    def set_grid(self, ox, oy, extent_x, extent_y):
        self._ck(self._L.ndt2d_set_grid(self._h, ox, oy, extent_x, extent_y))

    # -- target ----------------------------------------------------------------------------------
    def set_target(self, xy):
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        self._ck(self._L.ndt2d_set_target(self._h, _ptr(xy), len(xy)))

    def add_target(self, xy):
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        self._ck(self._L.ndt2d_add_target(self._h, _ptr(xy), len(xy)))

    def set_target_device(self, d_xy, n):
        self._ck(self._L.ndt2d_set_target_device(self._h, _ptr(d_xy), n))

    def add_target_device(self, d_xy, n):
        self._ck(self._L.ndt2d_add_target_device(self._h, _ptr(d_xy), n))

    def set_target_scans(self, xy, offsets, poses):
        """Target from packed scans (SPEC.md section 7.2): scan b = xy[offsets[b]:offsets[b+1]] at f64 poses[b] = (tx, ty, theta),
        transformed into the map frame in f64 inside the build (never rounded to f32)."""
        self._target_scans(self._L.ndt2d_set_target_scans, xy, offsets, poses)

    def add_target_scans(self, xy, offsets, poses):
        """add_target of posed scans: equals one set_target_scans of every scan added so far, bit for bit (SPEC 7)."""
        self._target_scans(self._L.ndt2d_add_target_scans, xy, offsets, poses)

    def _target_scans(self, fn, xy, offsets, poses):
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        offsets = np.ascontiguousarray(offsets, np.int64)
        poses = np.ascontiguousarray(poses, np.float64).reshape(-1, 3)
        nb = len(offsets) - 1
        if nb < 0 or len(poses) != nb or (nb and offsets[-1] > len(xy)):
            raise ValueError("offsets / poses / xy sizes disagree")
        self._ck(fn(self._h, _ptr(xy), _ptr(offsets), nb, _ptr(poses)))

    def set_target_scans_device(self, d_xy, d_offsets, nscans, npoints, d_poses):
        self._ck(self._L.ndt2d_set_target_scans_device(self._h, _ptr(d_xy), _ptr(d_offsets), nscans, npoints, _ptr(d_poses)))

    def add_target_scans_device(self, d_xy, d_offsets, nscans, npoints, d_poses):
        self._ck(self._L.ndt2d_add_target_scans_device(self._h, _ptr(d_xy), _ptr(d_offsets), nscans, npoints, _ptr(d_poses)))

    def set_target_ranges(self, ranges, angle_min, angle_inc, poses, range_scale=0.001, range_min=0.0, range_max=3.0e38):
        """Target from LaserScan ranges[nscans, nbeams] (float32 metres or uint16 * range_scale, SPEC.md section 8) at f64
        poses[nscans, 3] (SPEC 7.2)."""
        self._target_ranges(self._L.ndt2d_set_target_ranges, ranges, angle_min, angle_inc, poses, range_scale, range_min, range_max)

    def add_target_ranges(self, ranges, angle_min, angle_inc, poses, range_scale=0.001, range_min=0.0, range_max=3.0e38):
        self._target_ranges(self._L.ndt2d_add_target_ranges, ranges, angle_min, angle_inc, poses, range_scale, range_min, range_max)

    def _target_ranges(self, fn, ranges, angle_min, angle_inc, poses, range_scale, range_min, range_max):
        r = np.ascontiguousarray(ranges)
        if r.dtype not in (np.float32, np.uint16):
            r = r.astype(np.float32)
        r = np.atleast_2d(r)
        poses = np.ascontiguousarray(poses, np.float64).reshape(-1, 3)
        if r.ndim != 2 or len(poses) != r.shape[0]:
            raise ValueError("ranges must be (nscans, nbeams) with one pose per scan")
        self._ck(fn(self._h, _ptr(r), int(r.dtype == np.uint16), r.shape[0], r.shape[1], angle_min, angle_inc, range_scale,
                    range_min, range_max, _ptr(poses)))

    def set_target_ranges_device(self, d_ranges, is_u16, nscans, nbeams, angle_min, angle_inc, d_poses, range_scale=0.001,
                                 range_min=0.0, range_max=3.0e38):
        self._ck(self._L.ndt2d_set_target_ranges_device(self._h, _ptr(d_ranges), int(is_u16), nscans, nbeams, angle_min, angle_inc,
                                                        range_scale, range_min, range_max, _ptr(d_poses)))

    def add_target_ranges_device(self, d_ranges, is_u16, nscans, nbeams, angle_min, angle_inc, d_poses, range_scale=0.001,
                                 range_min=0.0, range_max=3.0e38):
        self._ck(self._L.ndt2d_add_target_ranges_device(self._h, _ptr(d_ranges), int(is_u16), nscans, nbeams, angle_min, angle_inc,
                                                        range_scale, range_min, range_max, _ptr(d_poses)))

    def geometry(self, level=0):
        g = np.zeros(5, np.float32)
        d = np.zeros(4, np.int32)
        self._ck(self._L.ndt2d_level_geometry(self._h, level, g.ctypes.data_as(_lib.c_f32p), d.ctypes.data_as(_lib.c_i32p)))
        return dict(res=g[0], st=g[1], inv_st=g[2], ox=g[3], oy=g[4], nhx=int(d[0]), nhy=int(d[1]), njx=int(d[2]), njy=int(d[3]))

    def cells(self, level=0):
        g = self.geometry(level)
        out = np.zeros((g["njy"], g["njx"], 8), np.float32)
        self._ck(self._L.ndt2d_get_cells(self._h, level, _ptr(out)))
        return out

    def set_cells(self, cells, level=0):
        """Load a cell table (njy, njx, 8) for `level`; the lattice must exist (set_grid or a target)."""
        cells = np.ascontiguousarray(cells, np.float32)
        if cells.ndim != 3 or cells.shape[2] != 8:
            raise ValueError("cells must have shape (njy, njx, 8)")
        self._ck(self._L.ndt2d_set_cells(self._h, level, _ptr(cells), cells.shape[0] * cells.shape[1]))
        g = self.geometry(level)
        if cells.shape[:2] != (g["njy"], g["njx"]):     # same record count, other shape: rows would be sheared
            raise ValueError(f"cells has shape {cells.shape[:2]}, level {level} is ({g['njy']}, {g['njx']})")

    def sums(self, level=0):
        g = self.geometry(level)
        n = np.zeros((g["njy"], g["njx"]), np.uint32)
        s = np.zeros((g["njy"], g["njx"], 5), np.int64)
        self._ck(self._L.ndt2d_get_sums(self._h, level, _ptr(n), _ptr(s)))
        return n, s

    def cells_device(self, level=0):
        return self._L.ndt2d_cells_device(self._h, level)

    def save_map(self, path, with_sums=True):
        """Persist the target through the C ABI (ndt2d_save_map): every level's lattice exactly as built, the parameters that
        shaped the cells, the records and (with_sums) the integer sums, so add_target continues the loaded map bit for bit."""
        self._ck(self._L.ndt2d_save_map(self._h, str(path).encode(), 1 if with_sums else 0))

    def load_map(self, path):
        """Inverse of save_map (ndt2d_load_map): replaces resolutions, grid, overlap/min_points/eig_ratio and the target."""
        self._ck(self._L.ndt2d_load_map(self._h, str(path).encode()))
        self._ck(self._L.ndt2d_get_params(self._h, C.byref(self.params)))
        n = 0
        g = np.zeros(5, np.float32)
        d = np.zeros(4, np.int32)
        while n < 8 and self._L.ndt2d_level_geometry(self._h, n, g.ctypes.data_as(_lib.c_f32p), d.ctypes.data_as(_lib.c_i32p)) == 0:
            n += 1
        self.nlevels = n

    # -- evaluation ------------------------------------------------------------------------------
    def cell_index(self, xy, pose=None, level=0):
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        idx = np.zeros(len(xy), np.int32)
        pose = None if pose is None else np.ascontiguousarray(pose, np.float64)
        self._ck(self._L.ndt2d_cell_index(self._h, level, _ptr(xy), len(xy), _ptr(pose), _ptr(idx)))
        return idx

    def evaluate(self, xy, poses, level=0):
        """poses (3,) or (m,3) -> (out[10] or out[m,10], count)."""
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        p = np.ascontiguousarray(poses, np.float64)
        single = p.ndim == 1
        p = p.reshape(-1, 3)
        out = np.zeros((len(p), 10), np.float64)
        cnt = np.zeros(len(p), np.int32)
        self._ck(self._L.ndt2d_evaluate(self._h, level, _ptr(xy), len(xy), _ptr(p), len(p), _ptr(out), _ptr(cnt)))
        return (out[0], int(cnt[0])) if single else (out, cnt)

    def evaluate_device(self, d_xy, n, d_poses, npose, d_out, d_count=None, level=0):
        self._ck(self._L.ndt2d_evaluate_device(self._h, level, _ptr(d_xy), n, _ptr(d_poses), npose, _ptr(d_out), _ptr(d_count)))

    def point_terms(self, xy, pose, level=0):
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        pose = np.ascontiguousarray(pose, np.float64)
        K = 4 if self.params.overlap else 1
        out = np.zeros((len(xy), K, 10), np.float32)
        self._ck(self._L.ndt2d_point_terms(self._h, level, _ptr(xy), len(xy), _ptr(pose), _ptr(out)))
        return out

    # -- align -----------------------------------------------------------------------------------
    @staticmethod
    def _check_out(out, n):
        """A caller-supplied result buffer is written by the C side as n x 144 bytes: refuse anything else."""
        if not (isinstance(out, np.ndarray) and out.dtype == RESULT_DTYPE and out.flags.c_contiguous and out.size >= n):
            raise ValueError(f"out must be a C-contiguous array of RESULT_DTYPE with at least {n} entries")
        return out

    def align(self, xy, init):
        """align(scan, initial pose) -> record with pose, score, hessian (+ grad, iterations, status, count)."""
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        init = np.ascontiguousarray(init, np.float64)
        r = np.zeros(1, RESULT_DTYPE)
        self._ck(self._L.ndt2d_align(self._h, _ptr(xy), len(xy), _ptr(init), _ptr(r)))
        return r[0]

    def align_batch(self, xy, offsets, init, out=None):
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        offsets = np.ascontiguousarray(offsets, np.int64)
        init = np.ascontiguousarray(init, np.float64).reshape(-1, 3)
        nb = len(offsets) - 1
        if nb < 0 or len(init) != nb or (nb and (offsets[0] < 0 or offsets[-1] > len(xy))):
            raise ValueError("offsets / init / xy sizes disagree")
        r = np.zeros(nb, RESULT_DTYPE) if out is None else self._check_out(out, nb)
        self._ck(self._L.ndt2d_align_batch(self._h, _ptr(xy), _ptr(offsets), nb, _ptr(init), _ptr(r)))
        return r

    def align_batch_device(self, d_xy, d_offsets, nscans, max_points, d_init, d_res):
        self._ck(self._L.ndt2d_align_batch_device(self._h, _ptr(d_xy), _ptr(d_offsets), nscans, max_points, _ptr(d_init), _ptr(d_res)))

    def align_batch_ranges(self, ranges, angle_min, angle_inc, init, range_scale=0.001, range_min=0.0,
                           range_max=3.0e38, out=None):
        """LaserScan input: ranges[nscans, nbeams] float32 metres or uint16 * range_scale (SPEC.md section 8)."""
        r = np.ascontiguousarray(ranges)
        if r.dtype not in (np.float32, np.uint16):
            r = r.astype(np.float32)
        r = np.atleast_2d(r)
        init = np.ascontiguousarray(init, np.float64).reshape(-1, 3)
        if r.ndim != 2 or len(init) != r.shape[0]:
            raise ValueError("ranges must be (nscans, nbeams) with one initial pose per scan")
        res = np.zeros(len(r), RESULT_DTYPE) if out is None else self._check_out(out, len(r))
        self._ck(self._L.ndt2d_align_batch_ranges(self._h, _ptr(r), int(r.dtype == np.uint16), r.shape[0], r.shape[1],
                                                  angle_min, angle_inc, range_scale, range_min, range_max, _ptr(init), _ptr(res)))
        return res

    def align_batch_ranges_device(self, d_ranges, is_u16, nscans, nbeams, angle_min, angle_inc, d_init, d_res,
                                  range_scale=0.001, range_min=0.0, range_max=3.0e38):
        self._ck(self._L.ndt2d_align_batch_ranges_device(self._h, _ptr(d_ranges), int(is_u16), nscans, nbeams, angle_min,
                                                         angle_inc, range_scale, range_min, range_max, _ptr(d_init), _ptr(d_res)))

    # -- sweep -----------------------------------------------------------------------------------
    def sweep(self, xy, hyp, k=1, level=0, want_scores=True):
        """hyp[m,3] f32 -> (scores[m] or None, best_idx[k], best_score[k])."""
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        hyp = np.ascontiguousarray(hyp, np.float32).reshape(-1, 3)
        scores = np.zeros(len(hyp), np.float64) if want_scores else None
        bi = np.full(max(k, 1), -1, np.int64)
        bs = np.zeros(max(k, 1), np.float64)
        self._ck(self._L.ndt2d_sweep(self._h, level, _ptr(xy), len(xy), _ptr(hyp), len(hyp), _ptr(scores), k, _ptr(bi), _ptr(bs)))
        return scores, bi[:k], bs[:k]

    def sweep_device(self, d_xy, n, d_hyp, nhyp, d_scores, k, d_best_idx, d_best_score, level=0):
        self._ck(self._L.ndt2d_sweep_device(self._h, level, _ptr(d_xy), n, _ptr(d_hyp), nhyp, _ptr(d_scores), k,
                                            _ptr(d_best_idx), _ptr(d_best_score)))

    def align_pairs(self, xy, offsets, pairs, init):
        """Batched scan-to-scan: pairs[p] = (target scan, source scan) of the packed batch; equals set_target(target) +
        align(source, init[p]) for every pair, in one call (per-target grids in hash tables)."""
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        offsets = np.ascontiguousarray(offsets, np.int64)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        init = np.ascontiguousarray(init, np.float64).reshape(-1, 3)
        nb = len(offsets) - 1
        if nb < 0 or len(init) != len(pairs) or (nb and (offsets[0] < 0 or offsets[-1] > len(xy))):
            raise ValueError("offsets / pairs / init / xy sizes disagree")
        res = np.zeros(len(pairs), RESULT_DTYPE)
        self._ck(self._L.ndt2d_align_pairs(self._h, _ptr(xy), _ptr(offsets), len(offsets) - 1, _ptr(pairs), len(pairs), _ptr(init), _ptr(res)))
        return res

    def align_pairs_device(self, d_xy, d_offsets, offsets, pairs, d_init, d_res):
        """Device-resident scans / initial poses / results; offsets (host copy) and pairs on the host. Asynchronous."""
        offsets = np.ascontiguousarray(offsets, np.int64)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        self._ck(self._L.ndt2d_align_pairs_device(self._h, _ptr(d_xy), _ptr(d_offsets), _ptr(offsets), len(offsets) - 1, _ptr(pairs),
                                                  len(pairs), _ptr(d_init), _ptr(d_res)))

    def relocalize_pairs(self, xy, offsets, pairs, centres, window, k=4, level=0):
        """Windowed search over scan pairs (loop-closure candidates): for pairs[p] = (target scan, source scan), sweep the window
        hypotheses around centres[p] on `level`, keep the k best by (-score, index) and align the source from each of them.
        Equals set_target(target) + relocalize(source, window_hypotheses(centres[p], window), k, level) for every pair.
        Returns (best_idx[npairs, k], best_score[npairs, k], res[npairs, k]); an empty slot has index -1."""
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        offsets = np.ascontiguousarray(offsets, np.int64)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        centres = np.ascontiguousarray(centres, np.float64).reshape(-1, 3)
        nb = len(offsets) - 1
        if nb < 0 or len(centres) != len(pairs) or (nb and (offsets[0] < 0 or offsets[-1] > len(xy))):
            raise ValueError("offsets / pairs / centres / xy sizes disagree")
        kk = max(int(k), 0)
        bi = np.full((len(pairs), kk), -1, np.int64)
        bs = np.zeros((len(pairs), kk), np.float64)
        res = np.zeros((len(pairs), kk), RESULT_DTYPE)
        w = _window(window)
        self._ck(self._L.ndt2d_relocalize_pairs(self._h, level, _ptr(xy), _ptr(offsets), nb, _ptr(pairs), len(pairs), _ptr(centres),
                                                C.byref(w), int(k), _ptr(bi), _ptr(bs), _ptr(res)))
        return bi, bs, res

    def relocalize_pairs_device(self, d_xy, d_offsets, offsets, pairs, d_centres, window, k, d_best_idx, d_best_score, d_res,
                                level=0):
        """Device-resident scans / centres / outputs ([npairs * k] each; d_best_score may be None); offsets (host copy) and
        pairs on the host. Asynchronous on the handle's stream."""
        offsets = np.ascontiguousarray(offsets, np.int64)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        w = _window(window)
        self._ck(self._L.ndt2d_relocalize_pairs_device(self._h, level, _ptr(d_xy), _ptr(d_offsets), _ptr(offsets), len(offsets) - 1,
                                                       _ptr(pairs), len(pairs), _ptr(d_centres), C.byref(w), int(k), _ptr(d_best_idx),
                                                       _ptr(d_best_score), _ptr(d_res)))

    def align_submaps(self, xy, offsets, submap_offsets, member_scans, member_poses, pairs, init):
        """Batched align against submaps of posed scans (SPEC.md section 7.3; pack_submaps builds the three submap arrays):
        pairs[p] = (submap, source scan); equals set_target_scans(the submap's member scans, their poses) + align(source,
        init[p]) for every pair, in one call. The handle's own target is not touched."""
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        offsets = np.ascontiguousarray(offsets, np.int64)
        so, ms, mp = _submap_args(submap_offsets, member_scans, member_poses)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        init = np.ascontiguousarray(init, np.float64).reshape(-1, 3)
        nb = len(offsets) - 1
        if nb < 0 or len(init) != len(pairs) or (nb and (offsets[0] < 0 or offsets[-1] > len(xy))):
            raise ValueError("offsets / pairs / init / xy sizes disagree")
        res = np.zeros(len(pairs), RESULT_DTYPE)
        self._ck(self._L.ndt2d_align_submaps(self._h, _ptr(xy), _ptr(offsets), nb, _ptr(so), len(so) - 1, _ptr(ms), _ptr(mp),
                                             _ptr(pairs), len(pairs), _ptr(init), _ptr(res)))
        return res

    def align_submaps_device(self, d_xy, d_offsets, offsets, submap_offsets, member_scans, d_member_poses, pairs, d_init, d_res):
        """Device-resident scans / member poses / initial poses / results; offsets (host copy), submap offsets, member scans
        and pairs on the host. Asynchronous."""
        offsets = np.ascontiguousarray(offsets, np.int64)
        so, ms = _submap_args(submap_offsets, member_scans)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        self._ck(self._L.ndt2d_align_submaps_device(self._h, _ptr(d_xy), _ptr(d_offsets), _ptr(offsets), len(offsets) - 1, _ptr(so),
                                                    len(so) - 1, _ptr(ms), _ptr(d_member_poses), _ptr(pairs), len(pairs), _ptr(d_init),
                                                    _ptr(d_res)))

    def relocalize_submaps(self, xy, offsets, submap_offsets, member_scans, member_poses, pairs, centres, window, k=4, level=0):
        """Windowed search against submaps of posed scans (SPEC.md section 7.3): for pairs[p] = (submap, source scan), equals
        set_target_scans(the submap's members) + relocalize(source, window_hypotheses(centres[p], window), k, level).
        Returns (best_idx[npairs, k], best_score[npairs, k], res[npairs, k]); an empty slot has index -1."""
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        offsets = np.ascontiguousarray(offsets, np.int64)
        so, ms, mp = _submap_args(submap_offsets, member_scans, member_poses)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        centres = np.ascontiguousarray(centres, np.float64).reshape(-1, 3)
        nb = len(offsets) - 1
        if nb < 0 or len(centres) != len(pairs) or (nb and (offsets[0] < 0 or offsets[-1] > len(xy))):
            raise ValueError("offsets / pairs / centres / xy sizes disagree")
        kk = max(int(k), 0)
        bi = np.full((len(pairs), kk), -1, np.int64)
        bs = np.zeros((len(pairs), kk), np.float64)
        res = np.zeros((len(pairs), kk), RESULT_DTYPE)
        w = _window(window)
        self._ck(self._L.ndt2d_relocalize_submaps(self._h, level, _ptr(xy), _ptr(offsets), nb, _ptr(so), len(so) - 1, _ptr(ms), _ptr(mp),
                                                  _ptr(pairs), len(pairs), _ptr(centres), C.byref(w), int(k), _ptr(bi), _ptr(bs), _ptr(res)))
        return bi, bs, res

    def relocalize_submaps_device(self, d_xy, d_offsets, offsets, submap_offsets, member_scans, d_member_poses, pairs, d_centres,
                                  window, k, d_best_idx, d_best_score, d_res, level=0):
        """Device-resident scans / member poses / centres / outputs ([npairs * k] each; d_best_score may be None); offsets
        (host copy), submap offsets, member scans, pairs and the window on the host. Asynchronous on the handle's stream."""
        offsets = np.ascontiguousarray(offsets, np.int64)
        so, ms = _submap_args(submap_offsets, member_scans)
        pairs = np.ascontiguousarray(pairs, np.int32).reshape(-1, 2)
        w = _window(window)
        self._ck(self._L.ndt2d_relocalize_submaps_device(self._h, level, _ptr(d_xy), _ptr(d_offsets), _ptr(offsets), len(offsets) - 1,
                                                         _ptr(so), len(so) - 1, _ptr(ms), _ptr(d_member_poses), _ptr(pairs), len(pairs),
                                                         _ptr(d_centres), C.byref(w), int(k), _ptr(d_best_idx), _ptr(d_best_score),
                                                         _ptr(d_res)))

    def relocalize_batch(self, xy, offsets, centres, window, k=4, level=0):
        """Windowed relocalisation of a batch of scans in the handle's map (SPEC.md section 6.2): for scan b, sweep the window
        hypotheses around centres[b] on `level`, keep the k best by (-score, index) and align the scan from each of them.
        Equals relocalize(scan b, window_hypotheses(centres[b], window), k, level) for every scan.
        Returns (best_idx[nscans, k], best_score[nscans, k], res[nscans, k]); an empty slot has index -1."""
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        offsets = np.ascontiguousarray(offsets, np.int64)
        centres = np.ascontiguousarray(centres, np.float64).reshape(-1, 3)
        nb = len(offsets) - 1
        if nb < 0 or len(centres) != nb or (nb and (offsets[0] < 0 or offsets[-1] > len(xy))):
            raise ValueError("offsets / centres / xy sizes disagree")
        kk = max(int(k), 0)
        bi = np.full((nb, kk), -1, np.int64)
        bs = np.zeros((nb, kk), np.float64)
        res = np.zeros((nb, kk), RESULT_DTYPE)
        w = _window(window)
        self._ck(self._L.ndt2d_relocalize_batch(self._h, level, _ptr(xy), _ptr(offsets), nb, _ptr(centres), C.byref(w), int(k),
                                                _ptr(bi), _ptr(bs), _ptr(res)))
        return bi, bs, res

    def relocalize_batch_device(self, d_xy, d_offsets, nscans, max_points, d_centres, window, k, d_best_idx, d_best_score, d_res,
                                level=0):
        """Device-resident scans / offsets / centres / outputs ([nscans * k] each; d_best_score may be None); max_points >= the
        longest scan. Asynchronous on the handle's stream."""
        w = _window(window)
        self._ck(self._L.ndt2d_relocalize_batch_device(self._h, level, _ptr(d_xy), _ptr(d_offsets), int(nscans), int(max_points),
                                                       _ptr(d_centres), C.byref(w), int(k), _ptr(d_best_idx), _ptr(d_best_score),
                                                       _ptr(d_res)))

    # ---- multi-GPU sweep: best-hypothesis exchange over peer memory (one process per GPU) ----
    def exchange_create(self, world, rank, nslots=64):
        """Allocate this rank's exchange table; returns its 64-byte CUDA IPC handle (bytes) for the other ranks."""
        h = (C.c_ubyte * 64)()
        self._ck(self._L.ndt2d_exchange_create(self._h, world, rank, nslots, C.cast(h, C.c_void_p)))
        return bytes(h)

    def exchange_open(self, handles):
        """handles: world x 64 bytes (entry r from rank r)."""
        buf = np.frombuffer(b"".join(handles) if isinstance(handles, (list, tuple)) else bytes(handles), np.uint8).copy()
        self._ck(self._L.ndt2d_exchange_open(self._h, _ptr(buf)))

    def sweep_publish(self, d_xy, n, d_hyp, nhyp, d_scores, index_offset, query, level=0):
        """Sweep this rank's shard on the device and store its best (global index, score) into every rank's table."""
        self._ck(self._L.ndt2d_sweep_publish(self._h, level, _ptr(d_xy), n, _ptr(d_hyp), nhyp, _ptr(d_scores), index_offset, query))

    def exchange_wait(self, query, timeout_ms=10000):
        """Global best (index, score) of `query` once every rank has published it (host-side poll of the own table)."""
        bi, bs = C.c_int64(-1), C.c_double(0.0)
        self._ck(self._L.ndt2d_exchange_wait(self._h, query, timeout_ms, C.byref(bi), C.byref(bs)))
        return bi.value, bs.value

    def exchange_close(self):
        self._ck(self._L.ndt2d_exchange_close(self._h))

    # ---- multi-GPU relocalisation over peer memory (one process per GPU; distributed.PeerRelocalizer wraps these) ----
    def reloc_create(self, world, rank, nslots=16, kmax=8):
        h = (C.c_ubyte * 64)()
        self._ck(self._L.ndt2d_reloc_create(self._h, world, rank, nslots, kmax, C.cast(h, C.c_void_p)))
        return bytes(h)

    def reloc_open(self, handles):
        buf = np.frombuffer(b"".join(handles) if isinstance(handles, (list, tuple)) else bytes(handles), np.uint8).copy()
        self._ck(self._L.ndt2d_reloc_open(self._h, _ptr(buf)))

    def relocalize_publish(self, d_xy, n, d_hyp, nhyp, index_offset, k, query, level=0):
        """Sweep this rank's shard, refine its k best and store the k candidates into every rank's table (asynchronous)."""
        self._ck(self._L.ndt2d_relocalize_publish(self._h, level, _ptr(d_xy), n, _ptr(d_hyp), nhyp, index_offset, k, query))

    def relocalize_wait(self, query, k, timeout_ms=10000):
        """Global (idx[k], res[k]) of `query` once every rank has published: what relocalize() returns on one GPU."""
        bi = np.full(k, -1, np.int64)
        res = np.zeros(k, RESULT_DTYPE)
        self._ck(self._L.ndt2d_relocalize_wait(self._h, query, timeout_ms, k, _ptr(bi), _ptr(res)))
        return bi, res

    def reloc_close(self):
        self._ck(self._L.ndt2d_reloc_close(self._h))

    def relocalize_device(self, d_xy, n, d_hyp, nhyp, k, d_best_idx, d_res, level=0):
        """Sweep + top-k + k refinements, everything on the device, asynchronous (ndt2d_relocalize_device)."""
        self._ck(self._L.ndt2d_relocalize_device(self._h, level, _ptr(d_xy), n, _ptr(d_hyp), nhyp, k, _ptr(d_best_idx), _ptr(d_res)))

    def relocalize(self, xy, hyp, k=4, level=0):
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        hyp = np.ascontiguousarray(hyp, np.float32).reshape(-1, 3)
        bi = np.full(k, -1, np.int64)
        res = np.zeros(k, RESULT_DTYPE)
        self._ck(self._L.ndt2d_relocalize(self._h, level, _ptr(xy), len(xy), _ptr(hyp), len(hyp), k, _ptr(bi), _ptr(res)))
        return bi, res
