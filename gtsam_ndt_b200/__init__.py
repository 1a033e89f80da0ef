"""gtsam_ndt_b200: B200-native 2D NDT scan matching behind the matcher API of a GTSAM/iSAM pipeline.

Only the hot path lives here: csrc/ (hand-written sm_100a kernels + the C ABI of include/ndt2d.h) and a thin
host mirror of the matcher interface. The CUDA library is mandatory; there is no CPU fallback.
"""
from .matcher import NdtMatcher2D, NdtError, RESULT_DTYPE, CONVERGED, MAX_ITERATIONS, STALLED, NO_OVERLAP, pinned_array, window_hypotheses, pack_submaps  # noqa: F401

__all__ = ["NdtMatcher2D", "NdtError", "RESULT_DTYPE", "CONVERGED", "MAX_ITERATIONS", "STALLED", "NO_OVERLAP", "pinned_array", "window_hypotheses", "pack_submaps"]
