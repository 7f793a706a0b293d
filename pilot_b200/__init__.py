"""pilot_b200 -- B200-native drop-in for PILOT's patient-distance hot path.

``pilot_b200.tl.wasserstein_distance`` mirrors ``pilotpy.tl.wasserstein_distance``
(/root/reference/pilotpy/tools/Trajectory.py:36-116) and writes the same seven
``adata.uns`` entries; the four computations under it (proportion histogram,
median centroids + cdist, all-pairs stabilised Sinkhorn, all-pairs exact EMD)
run in hand-written sm_100a CUDA kernels reached through the C ABI declared in
``include/pilot_b200.h``.  ``install()`` patches an importable ``pilotpy`` in
place so existing notebooks pick the GPU path up unchanged.
"""
from __future__ import annotations

import sys

from . import _lib, h5ad, ops, pairs, pl, tl  # noqa: F401
from .tl import (Cluster_Representations, Precomputed_distance, Sil_computing, cost_matrix,  # noqa: F401
                 extract_data_anno_pathomics_from_h5ad, extract_data_anno_scRNA_from_h5ad, load_h5ad,
                 return_real_labels,
                 set_path_for_results, transport_plan, wasserstein_d, wasserstein_d_cross, wasserstein_d_extend,
                 wasserstein_distance, wasserstein_plans)

__version__ = "0.1.0"

_PATCHED = ("wasserstein_distance", "Cluster_Representations", "cost_matrix", "wasserstein_d",
            "return_real_labels", "extract_data_anno_scRNA_from_h5ad",
            "extract_data_anno_pathomics_from_h5ad", "set_path_for_results", "Precomputed_distance",
            "Sil_computing")


def install() -> list:
    """Replace the hot-path functions of an importable ``pilotpy`` with the GPU versions.

    Patches every namespace that re-exports them by star-import
    (pilotpy/tools/Trajectory.py, pilotpy/tools/patients_sub_clustering.py:10,
    pilotpy/tools/__init__.py:1-5, pilotpy/tl.py:1).  Returns the patched module names.
    """
    import importlib

    importlib.import_module("pilotpy")  # raises ImportError if pilotpy is not installed
    patched = []
    for name in ("pilotpy.tools.Trajectory", "pilotpy.tools.patients_sub_clustering", "pilotpy.tools",
                 "pilotpy.tl"):
        mod = sys.modules.get(name)
        if mod is None:
            try:
                mod = importlib.import_module(name)
            except ImportError:
                continue
        for fn in _PATCHED:
            if hasattr(mod, fn):
                setattr(mod, fn, getattr(tl, fn))
        patched.append(name)
    return patched
