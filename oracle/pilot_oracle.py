"""oracle/pilot_oracle.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

CPU restatement of the reference's patient-distance hot path
(/root/reference/pilotpy/tools/Trajectory.py:36-116, 377-523, 617-642) in
NumPy/pandas, plus thin ctypes wrappers around the C restatements of the two
POT calls (oracle/emd_oracle.c, oracle/sinkhorn_oracle.c).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s cpu_baseline /
``--impl reference`` legs may import this module.  The product package
``pilot_b200`` never does.

Pinning status
--------------
* Stages 1-2 (proportions, cost matrix): pinned against the reference itself.
  ``oracle/ref_exec.py`` ast-extracts the reference functions from
  /root/reference (when mounted) and ``tests/golden/make_golden.py`` commits
  their outputs; ``tests/test_oracle_golden.py`` checks this restatement
  against those fixtures bit-for-bit.
* Stage 3 (ot.emd2 / ot.sinkhorn2): the arithmetic is in POT (pot>=0.9.1,<0.10,
  setup.py:19), absent from /root/reference and not installable here ->
  **parity unpinned** against POT; anchored on SciPy-HiGHS (EMD optimum),
  closed-form known answers, and Sinkhorn marginal invariants.
  The pin closes by itself wherever POT exists: ``pot()`` returns the real
  module when ``import ot`` works (site-packages or baseline/_ref), and then
  tests/test_oracle_vs_pot.py checks this restatement against it and
  bench.py's reference arm times POT itself (``kind: "pot <version>"``).
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from typing import Dict, Tuple

import numpy as np
import pandas as pd
import scipy.spatial.distance as ssd

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libpilot_oracle.so")
_lib = None
_pot = False  # not probed yet


def pot():
    """The real POT module (``ot``) if it can be imported -- from site-packages or from an offline
    install under baseline/_ref -- else None.  Never required; when present it pins the restatement."""
    global _pot
    if _pot is False:
        import importlib
        import sys
        ref = os.path.join(os.path.dirname(_HERE), "baseline", "_ref")
        added = False
        if os.path.isdir(ref) and ref not in sys.path:
            sys.path.append(ref)
            added = True
        try:
            mod = importlib.import_module("ot")
            _pot = mod if hasattr(mod, "emd2") and hasattr(mod, "sinkhorn2") else None
        except Exception:
            _pot = None
        if _pot is None and added:
            sys.path.remove(ref)
    return _pot


def pot_version():
    m = pot()
    return None if m is None else str(getattr(m, "__version__", "unknown"))


class _EmdStats(ctypes.Structure):
    _fields_ = [("pivots", ctypes.c_longlong), ("arcs_priced", ctypes.c_longlong),
                ("pot_updates", ctypes.c_longlong), ("cycle_steps", ctypes.c_longlong)]


class _SkInfo(ctypes.Structure):
    _fields_ = [("iters", ctypes.c_int), ("absorptions", ctypes.c_int),
                ("status", ctypes.c_int), ("err", ctypes.c_double)]


def build(force: bool = False) -> str:
    """Compile the C restatements (gcc, -O2, no fast-math, no FMA contraction)."""
    srcs = [os.path.join(_HERE, "emd_oracle.c"), os.path.join(_HERE, "sinkhorn_oracle.c")]
    if not force and os.path.exists(_LIB_PATH) and all(
            os.path.getmtime(_LIB_PATH) >= os.path.getmtime(s) for s in srcs):
        return _LIB_PATH
    cmd = ["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-o", _LIB_PATH] + srcs + ["-lm"]
    subprocess.check_call(cmd)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_LIB_PATH)
        dp = ctypes.POINTER(ctypes.c_double)
        L.pilot_oracle_emd.restype = ctypes.c_int
        L.pilot_oracle_emd.argtypes = [ctypes.c_int, ctypes.c_int, dp, dp, dp, ctypes.c_longlong,
                                       dp, dp, dp, dp, ctypes.POINTER(_EmdStats)]
        L.pilot_oracle_emd_rows.restype = ctypes.c_int
        L.pilot_oracle_emd_rows.argtypes = [ctypes.c_int, ctypes.c_int, dp, dp, ctypes.c_int,
                                            ctypes.c_int, dp, ctypes.POINTER(_EmdStats)]
        L.pilot_oracle_sinkhorn2.restype = ctypes.c_double
        L.pilot_oracle_sinkhorn2.argtypes = [ctypes.c_int, ctypes.c_int, dp, dp, dp, ctypes.c_double,
                                             ctypes.c_int, ctypes.c_double, ctypes.c_double,
                                             ctypes.c_int, ctypes.POINTER(_SkInfo)]
        L.pilot_oracle_sinkhorn_rows.restype = None
        L.pilot_oracle_sinkhorn_rows.argtypes = [ctypes.c_int, ctypes.c_int, dp, dp, ctypes.c_double,
                                                 ctypes.c_int, ctypes.c_int, dp,
                                                 ctypes.POINTER(ctypes.c_int),
                                                 ctypes.POINTER(ctypes.c_int)]
        _lib = L
    return _lib


def _dp(x: np.ndarray):
    return x.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


# --------------------------------------------------------------------------
# Stage 1: proportions  (Trajectory.py:377-436)
# --------------------------------------------------------------------------
def cluster_representations(df: pd.DataFrame, cell_col=0, sample_col=1, regulizer=0.2,
                            normalization=True) -> Dict[object, np.ndarray]:
    """Per-sample cell-type proportions, restating Cluster_Representations.

    * cell types / samples in order of first appearance (``.unique()``, :402,:412)
    * prior_k = n_k / (N - 1) * regulizer                       (:405-409)
    * counts scattered into the first-appearance order          (:418-425)
    * (c + prior) / (sum(c) + sum(prior)) with *sequential* sums (:428-430)
    """
    cell_name = df.columns[cell_col]
    samp_name = df.columns[sample_col]
    ct_codes, ct_uniques = pd.factorize(df[cell_name], sort=False)
    sm_codes, sm_uniques = pd.factorize(df[samp_name], sort=False)
    K, S, N = len(ct_uniques), len(sm_uniques), len(df)
    counts = np.bincount(sm_codes.astype(np.int64) * K + ct_codes, minlength=S * K)
    counts = counts.reshape(S, K).astype(np.float64)
    n_k = counts.sum(axis=0)                      # exact integers
    prior = (n_k / (N - 1)) * regulizer
    out: Dict[object, np.ndarray] = {}
    if normalization:
        sp = 0                                    # python sum(): 0 + p0 + p1 + ...
        for p in prior:
            sp = sp + p
        for s in range(S):
            sc = 0
            for c in counts[s]:
                sc = sc + c
            out[sm_uniques[s]] = (counts[s] + prior) / (sc + sp)
    else:
        for s in range(S):
            out[sm_uniques[s]] = counts[s].copy()
    return out


# --------------------------------------------------------------------------
# Stage 2: cost matrix  (Trajectory.py:441-475)
# --------------------------------------------------------------------------
def centroid_medians(annot: pd.DataFrame, data) -> np.ndarray:
    """Per-type, per-dimension median in the input dtype (:465-466)."""
    ct_codes, ct_uniques = pd.factorize(annot[annot.columns[0]], sort=False)
    X = np.asarray(data)
    K = len(ct_uniques)
    cent = np.empty((K, X.shape[1]), dtype=X.dtype if X.dtype.kind == "f" else np.float64)
    for k in range(K):
        cent[k] = np.nanmedian(X[ct_codes == k], axis=0)
    return cent


def cost_matrix(annot: pd.DataFrame, data, metric="cosine") -> Tuple[np.ndarray, pd.DataFrame]:
    cent = centroid_medians(annot, data)
    dis = ssd.squareform(ssd.pdist(cent.astype(np.float64), metric=metric), force="no", checks=True)
    names = annot[annot.columns[0]].unique()
    cost = pd.DataFrame(dis.copy())
    cost.columns = names
    cost["cell_types"] = names
    cost = cost.set_index("cell_types")
    return dis, cost


# --------------------------------------------------------------------------
# Stage 3a: ot.emd2  (Trajectory.py:511; POT ot/lp/__init__.py::emd2, A.1)
# --------------------------------------------------------------------------
def emd2(a, b, M, numItermax=100000, return_stats=False):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    M = np.ascontiguousarray(np.asarray(M, dtype=np.float64))
    if len(a) == 0:
        a = np.ones((M.shape[0],), dtype=np.float64) / M.shape[0]
    if len(b) == 0:
        b = np.ones((M.shape[1],), dtype=np.float64) / M.shape[1]
    assert a.shape[0] == M.shape[0] and b.shape[0] == M.shape[1], \
        "Dimension mismatch, check dimensions of M with a and b"
    np.testing.assert_almost_equal(a.sum(0), b.sum(0, keepdims=True),
                                   err_msg="a and b vector must have the same sum", decimal=6)
    b = np.ascontiguousarray(b * a.sum(0) / b.sum(0, keepdims=True))
    a = np.ascontiguousarray(a)
    cost = ctypes.c_double(0.0)
    st = _EmdStats()
    code = lib().pilot_oracle_emd(M.shape[0], M.shape[1], _dp(a), _dp(b), _dp(M), int(numItermax),
                                  ctypes.byref(cost), None, None, None, ctypes.byref(st))
    if return_stats:
        return float(cost.value), code, dict(pivots=st.pivots, arcs_priced=st.arcs_priced,
                                             pot_updates=st.pot_updates, cycle_steps=st.cycle_steps)
    return float(cost.value)


def emd_plan(a, b, M):
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    M = np.ascontiguousarray(M, dtype=np.float64)
    b = np.ascontiguousarray(b * a.sum() / b.sum())
    G = np.zeros_like(M)
    cost = ctypes.c_double(0.0)
    code = lib().pilot_oracle_emd(M.shape[0], M.shape[1], _dp(a), _dp(b), _dp(M), 100000,
                                  ctypes.byref(cost), _dp(G), None, None, None)
    return G, float(cost.value), code


# --------------------------------------------------------------------------
# Stage 3b: ot.sinkhorn2(..., method="sinkhorn_stabilized")  (Trajectory.py:515, A.2)
# --------------------------------------------------------------------------
def sinkhorn_stabilized_np(a, b, M, reg, numItermax=1000, tau=1e3, stopThr=1e-9,
                           print_period=20, return_info=False):
    """NumPy restatement in the reference form (plan returned, like POT)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    M = np.asarray(M, dtype=np.float64)
    dim_a, dim_b = len(a), len(b)
    alpha, beta = np.zeros(dim_a), np.zeros(dim_b)
    u, v = np.ones(dim_a) / dim_a, np.ones(dim_b) / dim_b

    def get_K(al, be):
        return np.exp(-(M - al.reshape((dim_a, 1)) - be.reshape((1, dim_b))) / reg)

    def get_Gamma(al, be, u_, v_):
        return np.exp(-(M - al.reshape((dim_a, 1)) - be.reshape((1, dim_b))) / reg
                      + np.log(u_.reshape((dim_a, 1))) + np.log(v_.reshape((1, dim_b))))

    K = get_K(alpha, beta)
    err = 1.0
    n_abs = 0
    iters = 0
    status = 1
    with np.errstate(all="ignore"):
        for ii in range(numItermax):
            iters = ii + 1
            uprev, vprev = u, v
            v = b / np.dot(K.T, u)
            u = a / np.dot(K, v)
            if np.max(np.abs(u)) > tau or np.max(np.abs(v)) > tau:
                alpha, beta = alpha + reg * np.log(u), beta + reg * np.log(v)
                u, v = np.ones(dim_a) / dim_a, np.ones(dim_b) / dim_b
                K = get_K(alpha, beta)
                n_abs += 1
            if ii % print_period == 0:
                transp = get_Gamma(alpha, beta, u, v)
                err = np.linalg.norm(np.sum(transp, axis=0) - b)
            if err <= stopThr:
                status = 0
                break
            if np.any(np.isnan(u)) or np.any(np.isnan(v)):
                u, v = uprev, vprev
                status = 2
                break
        G = get_Gamma(alpha, beta, u, v)
    if return_info:
        return G, dict(iters=iters, absorptions=n_abs, status=status, err=float(err))
    return G


def sinkhorn2_np(a, b, M, reg, **kw):
    M = np.asarray(M, dtype=np.float64)
    return float(np.sum(M * sinkhorn_stabilized_np(a, b, M, reg, **kw)))


def sinkhorn2(a, b, M, reg, numItermax=1000, stopThr=1e-9, tau=1e3, return_info=False, check_every=20):
    """C restatement (same statements as sinkhorn_stabilized_np).  check_every is POT's print_period: the
    marginal error is evaluated when ii % check_every == 0."""
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    M = np.ascontiguousarray(M, dtype=np.float64)
    info = _SkInfo()
    c = lib().pilot_oracle_sinkhorn2(M.shape[0], M.shape[1], _dp(a), _dp(b), _dp(M), float(reg),
                                     int(numItermax), float(tau), float(stopThr), int(check_every),
                                     ctypes.byref(info))
    if return_info:
        return float(c), dict(iters=info.iters, absorptions=info.absorptions,
                              status=info.status, err=info.err)
    return float(c)


# --------------------------------------------------------------------------
# Stage 3: all ordered pairs  (Trajectory.py:479-523)
# --------------------------------------------------------------------------
def wasserstein_d(Clu_rep: dict, cost, regularized="unreg", reg=0.1, use_numpy_sinkhorn=False):
    ids = list(Clu_rep.keys())
    n = len(ids)
    EMD = np.zeros((n, n))
    cost = np.asarray(cost, dtype=np.float64)
    if regularized == "unreg":
        for i in range(n):
            for j in range(n):
                EMD[i, j] = emd2(Clu_rep[ids[i]], Clu_rep[ids[j]], cost)
    else:
        f = sinkhorn2_np if use_numpy_sinkhorn else sinkhorn2
        for i in range(n):
            for j in range(n):
                EMD[i, j] = f(Clu_rep[ids[i]], Clu_rep[ids[j]], cost, reg)
    emd = pd.DataFrame(EMD.T.copy())   # DataFrame.from_dict(ndarray).T == transpose (:518)
    emd.columns = ids
    emd["sampleID"] = ids
    emd = emd.set_index("sampleID")
    return EMD, emd


def emd_rows(P: np.ndarray, M: np.ndarray, row0: int, row1: int, return_stats=False):
    """C-level batch of ordered pairs rows [row0,row1) x all columns (baseline timing)."""
    P = np.ascontiguousarray(P, dtype=np.float64)
    M = np.ascontiguousarray(M, dtype=np.float64)
    S, K = P.shape
    out = np.empty((row1 - row0, S))
    st = _EmdStats()
    bad = lib().pilot_oracle_emd_rows(S, K, _dp(P), _dp(M), row0, row1, _dp(out), ctypes.byref(st))
    if return_stats:
        return out, bad, dict(pivots=st.pivots, arcs_priced=st.arcs_priced,
                              pot_updates=st.pot_updates, cycle_steps=st.cycle_steps)
    return out


def sinkhorn_rows(P: np.ndarray, M: np.ndarray, reg: float, row0: int, row1: int):
    P = np.ascontiguousarray(P, dtype=np.float64)
    M = np.ascontiguousarray(M, dtype=np.float64)
    S, K = P.shape
    out = np.empty((row1 - row0, S))
    iters = np.empty((row1 - row0, S), dtype=np.int32)
    absn = np.empty((row1 - row0, S), dtype=np.int32)
    ip = ctypes.POINTER(ctypes.c_int)
    lib().pilot_oracle_sinkhorn_rows(S, K, _dp(P), _dp(M), float(reg), row0, row1, _dp(out),
                                     iters.ctypes.data_as(ip), absn.ctypes.data_as(ip))
    return out, iters, absn


# --------------------------------------------------------------------------
# Labels  (Trajectory.py:617-642)
# --------------------------------------------------------------------------
def return_real_labels(df: pd.DataFrame, category="status", sample_col=1):
    scol = df.columns[sample_col]
    first = df.drop_duplicates(subset=scol, keep="first")
    return list(first[category])


# --------------------------------------------------------------------------
# `ot` shim so that the *verbatim* reference wasserstein_d (ast-extracted by
# oracle/ref_exec.py) can run without POT.
# --------------------------------------------------------------------------
class OtShim:
    """Minimal stand-in for the two POT entry points PILOT calls."""

    def __init__(self, numpy_sinkhorn=True):
        self._np = numpy_sinkhorn

    @staticmethod
    def emd2(a, b, M, **kw):
        return emd2(a, b, M)

    def sinkhorn2(self, a, b, M, reg, method="sinkhorn", **kw):
        if method.lower() != "sinkhorn_stabilized":
            raise NotImplementedError("the oracle restates only method='sinkhorn_stabilized' "
                                      "(the one PILOT uses, Trajectory.py:515)")
        return sinkhorn2_np(a, b, M, reg) if self._np else sinkhorn2(a, b, M, reg)
