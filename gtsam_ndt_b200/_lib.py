"""ctypes binding of libndt2d.so (the C ABI in include/ndt2d.h). Fails loudly: no CPU fallback exists."""
import ctypes as C
import os

from . import build as _build

c_i64p = C.POINTER(C.c_int64)
c_f32p = C.POINTER(C.c_float)
c_f64p = C.POINTER(C.c_double)
c_i32p = C.POINTER(C.c_int32)


class Params(C.Structure):
    """ndt2d_params (include/ndt2d.h, SPEC.md section 1)."""
    _fields_ = [(n, C.c_double) for n in ("eig_ratio", "eps_trans", "eps_rot", "max_step_trans", "max_step_rot",
                                          "lambda_init", "lambda_min", "lambda_max", "lambda_up", "lambda_down",
                                          "lambda_fail_up")] + \
               [(n, C.c_int32) for n in ("min_points", "max_iterations", "overlap", "reserved")]


class Window(C.Structure):
    """ndt2d_window (include/ndt2d.h, SPEC.md section 6.1): half-widths and steps of a search window."""
    _fields_ = [(n, C.c_int32) for n in ("nx", "ny", "nth", "reserved")] + [(n, C.c_double) for n in ("step_x", "step_y", "step_th")]


# every symbol include/ndt2d.h declares: name -> (restype, argtypes)
_V = C.c_void_p
SIGNATURES = {
    "ndt2d_version": (C.c_int, []),
    "ndt2d_create": (C.c_int, [C.c_int, C.POINTER(_V)]),
    "ndt2d_create_on_stream": (C.c_int, [C.c_int, _V, C.POINTER(_V)]),
    "ndt2d_destroy": (None, [_V]),
    "ndt2d_last_error": (C.c_char_p, [_V]),
    "ndt2d_stream": (_V, [_V]),
    "ndt2d_synchronize": (C.c_int, [_V]),
    "ndt2d_kernel_launches": (C.c_int64, [_V]),
    "ndt2d_default_params": (None, [C.POINTER(Params)]),
    "ndt2d_set_params": (C.c_int, [_V, C.POINTER(Params)]),
    "ndt2d_get_params": (C.c_int, [_V, C.POINTER(Params)]),
    "ndt2d_set_resolution": (C.c_int, [_V, C.c_float]),
    "ndt2d_set_resolutions": (C.c_int, [_V, c_f32p, C.c_int]),
    "ndt2d_set_grid": (C.c_int, [_V, C.c_float, C.c_float, C.c_float, C.c_float]),
    "ndt2d_set_target": (C.c_int, [_V, _V, C.c_int64]),
    "ndt2d_set_target_device": (C.c_int, [_V, _V, C.c_int64]),
    "ndt2d_add_target": (C.c_int, [_V, _V, C.c_int64]),
    "ndt2d_add_target_device": (C.c_int, [_V, _V, C.c_int64]),
    "ndt2d_set_target_scans": (C.c_int, [_V, _V, _V, C.c_int, _V]),
    "ndt2d_add_target_scans": (C.c_int, [_V, _V, _V, C.c_int, _V]),
    "ndt2d_set_target_scans_device": (C.c_int, [_V, _V, _V, C.c_int, C.c_int64, _V]),
    "ndt2d_add_target_scans_device": (C.c_int, [_V, _V, _V, C.c_int, C.c_int64, _V]),
    "ndt2d_set_target_ranges": (C.c_int, [_V, _V, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_float, C.c_float,
                                          C.c_float, _V]),
    "ndt2d_add_target_ranges": (C.c_int, [_V, _V, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_float, C.c_float,
                                          C.c_float, _V]),
    "ndt2d_set_target_ranges_device": (C.c_int, [_V, _V, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_float,
                                                 C.c_float, C.c_float, _V]),
    "ndt2d_add_target_ranges_device": (C.c_int, [_V, _V, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_float,
                                                 C.c_float, C.c_float, _V]),
    "ndt2d_level_geometry": (C.c_int, [_V, C.c_int, c_f32p, c_i32p]),
    "ndt2d_get_cells": (C.c_int, [_V, C.c_int, _V]),
    "ndt2d_get_sums": (C.c_int, [_V, C.c_int, _V, _V]),
    "ndt2d_cells_device": (_V, [_V, C.c_int]),
    "ndt2d_set_cells": (C.c_int, [_V, C.c_int, _V, C.c_int64]),
    "ndt2d_save_map": (C.c_int, [_V, C.c_char_p, C.c_int]),
    "ndt2d_load_map": (C.c_int, [_V, C.c_char_p]),
    "ndt2d_cell_index": (C.c_int, [_V, C.c_int, _V, C.c_int, _V, _V]),
    "ndt2d_evaluate": (C.c_int, [_V, C.c_int, _V, C.c_int, _V, C.c_int, _V, _V]),
    "ndt2d_evaluate_device": (C.c_int, [_V, C.c_int, _V, C.c_int, _V, C.c_int, _V, _V]),
    "ndt2d_point_terms": (C.c_int, [_V, C.c_int, _V, C.c_int, _V, _V]),
    "ndt2d_align": (C.c_int, [_V, _V, C.c_int, _V, _V]),
    "ndt2d_align_batch": (C.c_int, [_V, _V, _V, C.c_int, _V, _V]),
    "ndt2d_align_batch_device": (C.c_int, [_V, _V, _V, C.c_int, C.c_int, _V, _V]),
    "ndt2d_align_batch_ranges": (C.c_int, [_V, _V, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_float,
                                           C.c_float, C.c_float, _V, _V]),
    "ndt2d_align_batch_ranges_device": (C.c_int, [_V, _V, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_float,
                                                  C.c_float, C.c_float, _V, _V]),
    "ndt2d_align_pairs": (C.c_int, [_V, _V, _V, C.c_int, _V, C.c_int, _V, _V]),
    "ndt2d_align_pairs_device": (C.c_int, [_V, _V, _V, _V, C.c_int, _V, C.c_int, _V, _V]),
    "ndt2d_relocalize_pairs": (C.c_int, [_V, C.c_int, _V, _V, C.c_int, _V, C.c_int, _V, C.POINTER(Window), C.c_int, _V, _V, _V]),
    "ndt2d_relocalize_pairs_device": (C.c_int, [_V, C.c_int, _V, _V, _V, C.c_int, _V, C.c_int, _V, C.POINTER(Window), C.c_int,
                                                _V, _V, _V]),
    "ndt2d_align_submaps": (C.c_int, [_V, _V, _V, C.c_int, _V, C.c_int, _V, _V, _V, C.c_int, _V, _V]),
    "ndt2d_align_submaps_device": (C.c_int, [_V, _V, _V, _V, C.c_int, _V, C.c_int, _V, _V, _V, C.c_int, _V, _V]),
    "ndt2d_relocalize_submaps": (C.c_int, [_V, C.c_int, _V, _V, C.c_int, _V, C.c_int, _V, _V, _V, C.c_int, _V, C.POINTER(Window),
                                           C.c_int, _V, _V, _V]),
    "ndt2d_relocalize_submaps_device": (C.c_int, [_V, C.c_int, _V, _V, _V, C.c_int, _V, C.c_int, _V, _V, _V, C.c_int, _V,
                                                  C.POINTER(Window), C.c_int, _V, _V, _V]),
    "ndt2d_relocalize_batch": (C.c_int, [_V, C.c_int, _V, _V, C.c_int, _V, C.POINTER(Window), C.c_int, _V, _V, _V]),
    "ndt2d_relocalize_batch_device": (C.c_int, [_V, C.c_int, _V, _V, C.c_int, C.c_int, _V, C.POINTER(Window), C.c_int, _V, _V, _V]),
    "ndt2d_sweep":(C.c_int, [_V, C.c_int, _V, C.c_int, _V, C.c_int64, _V, C.c_int, _V, _V]),
    "ndt2d_sweep_device": (C.c_int, [_V, C.c_int, _V, C.c_int, _V, C.c_int64, _V, C.c_int, _V, _V]),
    "ndt2d_relocalize": (C.c_int, [_V, C.c_int, _V, C.c_int, _V, C.c_int64, C.c_int, _V, _V]),
    "ndt2d_relocalize_device": (C.c_int, [_V, C.c_int, _V, C.c_int, _V, C.c_int64, C.c_int, _V, _V]),
    "ndt2d_exchange_create": (C.c_int, [_V, C.c_int, C.c_int, C.c_int, _V]),
    "ndt2d_exchange_open": (C.c_int, [_V, _V]),
    "ndt2d_sweep_publish": (C.c_int, [_V, C.c_int, _V, C.c_int, _V, C.c_int64, _V, C.c_int64, C.c_uint64]),
    "ndt2d_exchange_wait": (C.c_int, [_V, C.c_uint64, C.c_int, c_i64p, c_f64p]),
    "ndt2d_exchange_close": (C.c_int, [_V]),
    "ndt2d_reloc_create": (C.c_int, [_V, C.c_int, C.c_int, C.c_int, C.c_int, _V]),
    "ndt2d_reloc_open": (C.c_int, [_V, _V]),
    "ndt2d_relocalize_publish": (C.c_int, [_V, C.c_int, _V, C.c_int, _V, C.c_int64, C.c_int64, C.c_int, C.c_uint64]),
    "ndt2d_relocalize_wait": (C.c_int, [_V, C.c_uint64, C.c_int, C.c_int, _V, _V]),
    "ndt2d_reloc_close": (C.c_int, [_V]),
    "ndt2d_host_alloc": (C.c_int, [C.POINTER(_V), C.c_size_t]),
    "ndt2d_host_alloc_flags": (C.c_int, [C.POINTER(_V), C.c_size_t, C.c_int]),
    "ndt2d_host_free": (C.c_int, [_V]),
    "ndt2d_set_upload_relay": (C.c_int, [_V, C.c_int, C.c_double]),
}

_lib = None


def load():
    """Load libndt2d.so (built in-tree by gtsam_ndt_b200.build). Raises if it is missing: no fallback."""
    global _lib
    if _lib is None:
        so = os.environ.get("NDT2D_LIB") or _build.LIB_CUDA  # NDT2D_LIB: a tuning-experiment build of the same sources
        if not os.path.exists(so):
            raise ImportError(f"{so} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(needs nvcc). There is no CPU fallback for the NDT path.")
        lib = C.CDLL(so)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib
