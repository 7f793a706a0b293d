"""ctypes binding of the C-ABI in include/pilot_b200.h (pilot_b200/csrc/libpilot_b200.so).

There is deliberately no fallback: if the shared library is missing or a call
fails, an exception is raised.  Nothing in this package computes on the CPU.
"""
from __future__ import annotations

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# PILOT_B200_LIB: another build of the same library (A/B measurements of kernel variants only)
LIB_PATH = os.environ.get("PILOT_B200_LIB") or os.path.join(_HERE, "csrc", "libpilot_b200.so")

ABI_VERSION = 4

# constants mirrored from include/pilot_b200.h
F32, F64 = 0, 1
METRICS = {"cosine": 0, "cos": 0, "euclidean": 1, "euclid": 1, "eu": 1, "e": 1, "l2": 1,
           "sqeuclidean": 2, "sqe": 2, "sqeuclid": 2,
           "cityblock": 3, "cblock": 3, "cb": 3, "c": 3, "manhattan": 3, "taxicab": 3, "l1": 3,
           "chebyshev": 4, "chebychev": 4, "chebyshev": 4, "cheby": 4, "cheb": 4, "ch": 4, "linf": 4,
           "correlation": 5, "co": 5,
           "braycurtis": 6, "canberra": 7, "minkowski": 8, "mi": 8, "m": 8, "pnorm": 8,
           "seuclidean": 9, "se": 9, "s": 9, "hamming": 10, "hamm": 10, "ha": 10, "h": 10, "matching": 10}
PAIRS_FULL, PAIRS_UPPER, PAIRS_RECT = 0, 1, 2
PRECISIONS = {"f64": F64, "fp64": F64, "float64": F64, "double": F64,
              "f32": F32, "fp32": F32, "float32": F32, "single": F32}


def precision_code(precision) -> int:
    """'f64' (1e-9 parity tier, the default everywhere) or 'f32' (1e-4 tier) -> PILOT_F64 / PILOT_F32."""
    if precision in (F32, F64) and not isinstance(precision, str):
        return int(precision)
    try:
        return PRECISIONS[str(precision).lower()]
    except KeyError:
        raise ValueError(f"precision must be 'f64' or 'f32', got {precision!r}") from None
ST_CONVERGED, ST_MAXITER, ST_NUMERIC, ST_UNBOUNDED = 0, 1, 2, 3
WS_MEDIAN, WS_SINKHORN, WS_EMD = 0, 1, 2
SIL_PRECOMPUTED = 100

EXPORTS = (
    "pilot_abi_version", "pilot_last_error", "pilot_range_count", "pilot_workspace_bytes", "pilot_launch_count",
    "pilot_hist", "pilot_props_finalize", "pilot_centroid_median", "pilot_cdist",
    "pilot_sinkhorn_pairs", "pilot_emd_pairs", "pilot_sinkhorn_plans", "pilot_emd_plans", "pilot_unpack_pairs",
    "pilot_knn_rows", "pilot_silhouette_rows", "pilot_pipe_peak",
)


class PairRange(ctypes.Structure):
    """pilot_pair_range (include/pilot_b200.h).  ``rows``: the row count S_a in PAIRS_RECT, 0 otherwise;
    ``reserved`` is its former name and still accepted."""
    _fields_ = [("total", ctypes.c_int64), ("block", ctypes.c_int64), ("nranks", ctypes.c_int32),
                ("rank", ctypes.c_int32), ("mode", ctypes.c_int32), ("rows", ctypes.c_int32),
                ("first", ctypes.c_int64)]
    reserved = property(lambda self: self.rows, lambda self, v: setattr(self, "rows", v))


class PilotLibraryError(RuntimeError):
    pass


_lib = None


def lib():
    """Load the shared library (once) and declare every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PilotLibraryError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C pilot_b200/csrc`).  pilot_b200 has no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, dbl, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double, ctypes.c_size_t
    prp = ctypes.POINTER(PairRange)
    L.pilot_abi_version.restype = i32
    L.pilot_abi_version.argtypes = []
    L.pilot_last_error.restype = ctypes.c_char_p
    L.pilot_last_error.argtypes = []
    L.pilot_range_count.restype = i64
    L.pilot_range_count.argtypes = [prp]
    L.pilot_workspace_bytes.restype = sz
    L.pilot_workspace_bytes.argtypes = [i32, i64, i32, i32, i32]
    L.pilot_launch_count.restype = ctypes.c_uint64
    L.pilot_launch_count.argtypes = []
    L.pilot_hist.restype = i32
    L.pilot_hist.argtypes = [vp, vp, i64, i32, i32, vp, vp, vp, vp]
    L.pilot_props_finalize.restype = i32
    L.pilot_props_finalize.argtypes = [vp, i32, i32, vp, vp, i32, i32, i64, dbl, i32, vp, vp, vp, vp]
    L.pilot_centroid_median.restype = i32
    L.pilot_centroid_median.argtypes = [vp, i32, i64, i32, i64, vp, i32, vp, vp, vp, sz, vp]
    L.pilot_cdist.restype = i32
    L.pilot_cdist.argtypes = [vp, i32, i32, i32, vp, vp, vp, vp]
    L.pilot_sinkhorn_pairs.restype = i32
    L.pilot_sinkhorn_pairs.argtypes = [vp, i32, i32, vp, dbl, i32, dbl, dbl, i32, prp, i32, i32, vp, vp, vp, vp,
                                       vp, sz, vp]
    L.pilot_emd_pairs.restype = i32
    L.pilot_emd_pairs.argtypes = [vp, i32, i32, vp, i64, prp, i32, vp, vp, vp, vp, sz, vp]
    L.pilot_sinkhorn_plans.restype = i32
    L.pilot_sinkhorn_plans.argtypes = [vp, i32, i32, vp, dbl, i32, dbl, dbl, i32, vp, vp, i64, vp, vp, vp, vp, vp, vp,
                                       sz, vp]
    L.pilot_emd_plans.restype = i32
    L.pilot_emd_plans.argtypes = [vp, i32, i32, vp, i64, vp, vp, i64, vp, vp, vp, vp, sz, vp]
    L.pilot_unpack_pairs.restype = i32
    L.pilot_unpack_pairs.argtypes = [vp, i64, i32, prp, dbl, vp, vp]
    L.pilot_knn_rows.restype = i32
    L.pilot_knn_rows.argtypes = [vp, i32, i32, vp, vp, vp, sz, vp]
    L.pilot_silhouette_rows.restype = i32
    L.pilot_silhouette_rows.argtypes = [vp, i32, i32, vp, vp, vp, i32, vp, vp, sz, vp]
    L.pilot_pipe_peak.restype = i32
    L.pilot_pipe_peak.argtypes = [i32, ctypes.POINTER(ctypes.c_double), vp]
    if L.pilot_abi_version() != ABI_VERSION:
        raise PilotLibraryError(f"ABI mismatch: library {L.pilot_abi_version()} != binding {ABI_VERSION}")
    _lib = L
    return L


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().pilot_last_error().decode("utf-8", "replace")
        raise PilotLibraryError(f"{what or 'pilot_b200'} failed (rc={rc}): {msg}")


def launch_count() -> int:
    """Kernels launched by the library in this process so far."""
    return int(lib().pilot_launch_count())


def range_count(r: PairRange) -> int:
    return int(lib().pilot_range_count(ctypes.byref(r)))
