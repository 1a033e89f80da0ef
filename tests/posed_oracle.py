"""The CPU spec oracle with SPEC.md section 7.2 (targets from posed scans) added: test infrastructure only.

tests/oracle_posed_target.c compiles the oracle's source unchanged and adds oracle_set_target_scans /
oracle_add_target_scans. The library is built with the oracle's compiler flags into a temporary directory (the source
tree may be read-only) and cached there by the hash of its sources; PosedOracle is oracle.Oracle on that library.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE_DIR = os.path.join(os.path.dirname(_HERE), "oracle")
_SRC = os.path.join(_HERE, "oracle_posed_target.c")
# oracle/Makefile's CFLAGS: fma() is one rounding and nothing else is contracted
_CFLAGS = ["-O2", "-std=c11", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-mavx2"]

_lib = None


def build():
    h = hashlib.sha256(" ".join(_CFLAGS).encode())
    for f in (_SRC, os.path.join(_ORACLE_DIR, "ndt2d_oracle.c"), os.path.join(_ORACLE_DIR, "ndt2d_oracle.h")):
        with open(f, "rb") as fh:
            h.update(fh.read())
    out_dir = os.path.join(tempfile.gettempdir(), "ndt2d_posed_oracle_%d" % os.getuid())
    os.makedirs(out_dir, exist_ok=True)
    so = os.path.join(out_dir, "libndt2d_oracle_posed_%s.so" % h.hexdigest()[:16])
    if not os.path.exists(so):
        tmp = "%s.%d.tmp" % (so, os.getpid())
        subprocess.check_call(["gcc"] + _CFLAGS + ["-shared", "-I", _ORACLE_DIR, "-o", tmp, _SRC, "-lm"])
        os.replace(tmp, so)
    return so


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        L.oracle_create.restype = C.c_void_p
        L.oracle_expneg.restype = C.c_float
        L.oracle_expneg.argtypes = [C.c_float]
        for name in ("oracle_destroy", "oracle_default_params"):
            getattr(L, name).restype = None
        _lib = L
    return _lib


class PosedOracle(oracle.Oracle):
    """oracle.Oracle plus set_target_scans / add_target_scans (SPEC 7.2)."""

    def __init__(self, resolutions=(1.0,), **params):
        self.L = lib()
        self.h = C.c_void_p(self.L.oracle_create())
        self.params = oracle.Params()
        self.L.oracle_default_params(C.byref(self.params))
        self.set_params(**params)
        self.set_resolutions(resolutions)

    def _target_scans(self, fn, xy, offsets, poses):
        xy = np.ascontiguousarray(xy, np.float32).reshape(-1, 2)
        offsets = np.ascontiguousarray(offsets, np.int64)
        poses = np.ascontiguousarray(poses, np.float64).reshape(-1, 3)
        nb = len(offsets) - 1
        assert len(poses) == nb and (nb == 0 or offsets[-1] <= len(xy))
        P = lambda a, t: a.ctypes.data_as(C.POINTER(t))   # noqa: E731
        self._ck(fn(self.h, P(xy, C.c_float), P(offsets, C.c_int64), nb, P(poses, C.c_double)), fn.__name__)

    def set_target_scans(self, xy, offsets, poses):
        """SPEC 7.2: target from packed scans (offsets[0..B]) at f64 poses[B, 3]."""
        self._target_scans(self.L.oracle_set_target_scans, xy, offsets, poses)

    def add_target_scans(self, xy, offsets, poses):
        self._target_scans(self.L.oracle_add_target_scans, xy, offsets, poses)
