"""Device-level operators: one Python function per C-ABI entry point.

PyTorch is plumbing only here (device buffers, the current CUDA stream); all
arithmetic is done by the hand-written sm_100a kernels behind the C ABI.
Every function takes/returns CUDA tensors and is asynchronous on the current
stream.  No CPU fallback exists: without a GPU or without the shared library
these functions raise.
"""
from __future__ import annotations

import ctypes
from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import PairRange, check, lib


def _require_cuda(*tensors: torch.Tensor) -> None:
    if not torch.cuda.is_available():
        raise _lib.PilotLibraryError("pilot_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise ValueError("expected a CUDA tensor")


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


_ws_cache = {}


def _workspace(nbytes: int, device) -> torch.Tensor:
    """Per-device, per-stream grow-only scratch buffer."""
    key = (str(device), _stream())
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    return buf


def make_range(total: int, mode: int, nranks: int = 1, rank: int = 0, block: Optional[int] = None,
               rows: int = 0, first: int = 0) -> PairRange:
    """rows: the row count S_a of the PAIRS_RECT space (0 for FULL / UPPER)."""
    if block is None:
        block = max(1, min(4096, -(-total // (nranks * 4)))) if nranks > 1 else max(1, total)
    return PairRange(total=int(total), block=int(block), nranks=int(nranks), rank=int(rank), mode=int(mode),
                     rows=int(rows), first=int(first))


def n_pairs(S: int, mode: int, rows: int = 0) -> int:
    """Problems in the pair space of S samples (PAIRS_RECT: S_a = rows against the other S - rows)."""
    if mode == _lib.PAIRS_RECT:
        return rows * (S - rows)
    return S * S if mode == _lib.PAIRS_FULL else S * (S - 1) // 2


# ---------------------------------------------------------------------------
def hist(ct_code: torch.Tensor, smp_code: torch.Tensor, K: int, S: int
         ) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """counts[S,K] (int64), first_ct[K], first_smp[S] -- see pilot_hist."""
    _require_cuda(ct_code, smp_code)
    assert ct_code.dtype == torch.int32 and smp_code.dtype == torch.int32
    assert ct_code.is_contiguous() and smp_code.is_contiguous() and ct_code.numel() == smp_code.numel()
    dev = ct_code.device
    counts = torch.empty((S, K), dtype=torch.int64, device=dev)
    first_ct = torch.empty((K,), dtype=torch.int64, device=dev)
    first_smp = torch.empty((S,), dtype=torch.int64, device=dev)
    check(lib().pilot_hist(_ptr(ct_code), _ptr(smp_code), ct_code.numel(), K, S, _ptr(counts), _ptr(first_ct),
                           _ptr(first_smp), _stream()), "pilot_hist")
    return counts, first_ct, first_smp


def props_finalize(counts_raw: torch.Tensor, perm_k: Optional[torch.Tensor], perm_s: Optional[torch.Tensor],
                   n_cells: int, regulizer: float, normalization: bool
                   ) -> Tuple[torch.Tensor, torch.Tensor]:
    """props[S,K] (float64) and the permuted counts[S,K] (int64)."""
    _require_cuda(counts_raw)
    S_raw, K_raw = counts_raw.shape
    K = K_raw if perm_k is None else perm_k.numel()
    S = S_raw if perm_s is None else perm_s.numel()
    for p in (perm_k, perm_s):
        assert p is None or (p.dtype == torch.int32 and p.is_cuda and p.is_contiguous())
    props = torch.empty((S, K), dtype=torch.float64, device=counts_raw.device)
    counts = torch.empty((S, K), dtype=torch.int64, device=counts_raw.device)
    prior = torch.empty((K + 1,), dtype=torch.float64, device=counts_raw.device)
    check(lib().pilot_props_finalize(_ptr(counts_raw), K_raw, S_raw, _ptr(perm_k), _ptr(perm_s), K, S, n_cells,
                                     float(regulizer), 1 if normalization else 0, _ptr(props), _ptr(counts),
                                     _ptr(prior), _stream()), "pilot_props_finalize")
    return props, counts


def centroid_median(X: torch.Tensor, ct_code: torch.Tensor, K: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per-code, per-dimension median of the rows of X (n x D, f32 or f64).  Returns
    (centroids in X.dtype [K,D], centroids as float64 [K,D])."""
    _require_cuda(X, ct_code)
    assert X.dim() == 2 and X.stride(1) == 1 and ct_code.dtype == torch.int32
    if X.dtype == torch.float32:
        dt = _lib.F32
    elif X.dtype == torch.float64:
        dt = _lib.F64
    else:
        raise TypeError(f"embedding dtype {X.dtype} not supported (float32/float64)")
    n, D = X.shape
    cent = torch.empty((K, D), dtype=X.dtype, device=X.device)
    cent64 = torch.empty((K, D), dtype=torch.float64, device=X.device)
    nbytes = lib().pilot_workspace_bytes(_lib.WS_MEDIAN, n, K, 0, D)
    ws = _workspace(nbytes, X.device)
    check(lib().pilot_centroid_median(_ptr(X), dt, n, D, X.stride(0), _ptr(ct_code), K, _ptr(cent), _ptr(cent64),
                                      _ptr(ws), ws.numel(), _stream()), "pilot_centroid_median")
    return cent, cent64


def median_fallbacks(K: int, D: int, device=None) -> int:
    """Diagnostic: how many (type, dim) pairs of the LAST centroid_median call on this stream took
    the exact full-column fallback of the streaming path (reads the workspace; synchronises)."""
    device = device or torch.device("cuda", torch.cuda.current_device())
    ws = _workspace(1, device)
    return int(ws[0:4].view(torch.int32).item())  # MsHeader.fail is the first word of the workspace


def cdist(cent64: torch.Tensor, metric: str = "cosine") -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """(cost[K,K], cost / cost.max(), cost.max()) for a scipy pdist metric name."""
    _require_cuda(cent64)
    assert cent64.dtype == torch.float64 and cent64.is_contiguous()
    key = metric.lower() if isinstance(metric, str) else metric
    if key not in _lib.METRICS:
        raise ValueError(f"Unknown Distance Metric: {metric} (pilot_b200 implements "
                         f"{sorted(set(_lib.METRICS))}; no CPU fallback)")
    K, D = cent64.shape
    cost = torch.empty((K, K), dtype=torch.float64, device=cent64.device)
    cost_norm = torch.empty_like(cost)
    cmax = torch.empty((1,), dtype=torch.float64, device=cent64.device)
    check(lib().pilot_cdist(_ptr(cent64), K, D, _lib.METRICS[key], _ptr(cost), _ptr(cost_norm), _ptr(cmax),
                            _stream()), "pilot_cdist")
    return cost, cost_norm, cmax


def sinkhorn_pairs(props: torch.Tensor, cost: torch.Tensor, reg: float, rng: PairRange, algo: int = 0,
                   num_iter_max: int = 1000, stop_thr: float = 1e-9, tau: float = 1e3, check_every: int = 20,
                   want_info: bool = False, out: Optional[torch.Tensor] = None, precision="f64"):
    """Packed Sinkhorn costs of the problems `rng` assigns to rng.rank."""
    _require_cuda(props, cost)
    assert props.dtype == torch.float64 and cost.dtype == torch.float64
    assert props.is_contiguous() and cost.is_contiguous()
    S, K = props.shape
    assert cost.shape == (K, K)
    n = _lib.range_count(rng)
    dev = props.device
    if out is None:
        out = torch.empty((max(n, 1),), dtype=torch.float64, device=dev)
    iters = absn = status = None
    if want_info:
        iters = torch.zeros((max(n, 1),), dtype=torch.int32, device=dev)
        absn = torch.zeros_like(iters)
        status = torch.zeros_like(iters)
    nbytes = lib().pilot_workspace_bytes(_lib.WS_SINKHORN, n, K, S, 0)
    ws = _workspace(nbytes, dev)
    check(lib().pilot_sinkhorn_pairs(_ptr(props), S, K, _ptr(cost), float(reg), int(num_iter_max), float(stop_thr),
                                     float(tau), int(check_every), ctypes.byref(rng), int(algo),
                                     _lib.precision_code(precision), _ptr(out),
                                     _ptr(iters), _ptr(absn), _ptr(status), _ptr(ws), ws.numel(), _stream()),
          "pilot_sinkhorn_pairs")
    if want_info:
        return out[:n], iters[:n], absn[:n], status[:n]
    return out[:n]


def emd_pairs(props: torch.Tensor, cost: torch.Tensor, rng: PairRange, max_pivots: int = 100000,
              want_info: bool = False, out: Optional[torch.Tensor] = None, precision="f64"):
    """Packed exact-EMD costs of the problems `rng` assigns to rng.rank."""
    _require_cuda(props, cost)
    assert props.dtype == torch.float64 and cost.dtype == torch.float64
    assert props.is_contiguous() and cost.is_contiguous()
    S, K = props.shape
    assert cost.shape == (K, K)
    n = _lib.range_count(rng)
    dev = props.device
    if out is None:
        out = torch.empty((max(n, 1),), dtype=torch.float64, device=dev)
    status = pivots = None
    if want_info:
        status = torch.zeros((max(n, 1),), dtype=torch.int32, device=dev)
        pivots = torch.zeros_like(status)
    ws = _workspace(lib().pilot_workspace_bytes(_lib.WS_EMD, n, K, S, 0), dev)
    check(lib().pilot_emd_pairs(_ptr(props), S, K, _ptr(cost), int(max_pivots), ctypes.byref(rng),
                                _lib.precision_code(precision), _ptr(out), _ptr(status), _ptr(pivots), _ptr(ws),
                                ws.numel(), _stream()), "pilot_emd_pairs")
    if want_info:
        return out[:n], status[:n], pivots[:n]
    return out[:n]


def _plan_inputs(props: torch.Tensor, cost: torch.Tensor, pair_a, pair_b):
    """Checked shapes and int32 device copies of the pair lists (a list, an ndarray or a tensor)."""
    _require_cuda(props, cost)
    assert props.dtype == torch.float64 and cost.dtype == torch.float64
    assert props.is_contiguous() and cost.is_contiguous()
    S, K = props.shape
    assert cost.shape == (K, K)
    dev = props.device
    pa, pb = (torch.as_tensor(p, dtype=torch.int32).to(dev).contiguous().reshape(-1) for p in (pair_a, pair_b))
    if pa.numel() != pb.numel():
        raise ValueError(f"pair_a has {pa.numel()} entries and pair_b {pb.numel()}")
    n = pa.numel()
    plans = torch.empty((n, K, K), dtype=torch.float64, device=dev)
    out = torch.empty((n,), dtype=torch.float64, device=dev)
    return S, K, n, pa, pb, plans, out


def emd_plans(props: torch.Tensor, cost: torch.Tensor, pair_a, pair_b, max_pivots: int = 100000,
              want_info: bool = False):
    """Exact-EMD transport plans of the problems (props[pair_a[l]], props[pair_b[l]]), FP64, no mirroring:
    (plans [n, K, K], out [n]) with plans[l, r, c] the mass moved from type r of a to type c of b (emd2's rescaled
    b) and out[l] the cost pilot_emd_pairs computes for that pair; with want_info also status [n].  A pair index
    outside [0, S) gives a NaN plan, a NaN cost and ST_NUMERIC."""
    S, K, n, pa, pb, plans, out = _plan_inputs(props, cost, pair_a, pair_b)
    status = torch.zeros((n,), dtype=torch.int32, device=props.device) if want_info else None
    ws = _workspace(lib().pilot_workspace_bytes(_lib.WS_EMD, n, K, S, 0), props.device)
    check(lib().pilot_emd_plans(_ptr(props), S, K, _ptr(cost), int(max_pivots), _ptr(pa), _ptr(pb), n, _ptr(plans),
                                _ptr(out), _ptr(status), _ptr(ws), ws.numel(), _stream()), "pilot_emd_plans")
    if want_info:
        return plans, out, status
    return plans, out


def sinkhorn_plans(props: torch.Tensor, cost: torch.Tensor, reg: float, pair_a, pair_b, num_iter_max: int = 1000,
                   stop_thr: float = 1e-9, tau: float = 1e3, check_every: int = 20, want_info: bool = False):
    """Stabilised-Sinkhorn transport plans of the problems (props[pair_a[l]], props[pair_b[l]]), FP64, in POT's
    reference form: (plans [n, K, K], out [n]), out bit-identical to sinkhorn_pairs(algo=1) for the same pair; with
    want_info also (iters, absorptions, status) [n] each.  A pair index outside [0, S) gives a NaN plan, a NaN
    cost and ST_NUMERIC."""
    S, K, n, pa, pb, plans, out = _plan_inputs(props, cost, pair_a, pair_b)
    iters = absn = status = None
    if want_info:
        iters = torch.zeros((n,), dtype=torch.int32, device=props.device)
        absn = torch.zeros_like(iters)
        status = torch.zeros_like(iters)
    ws = _workspace(lib().pilot_workspace_bytes(_lib.WS_SINKHORN, n, K, S, 0), props.device)
    check(lib().pilot_sinkhorn_plans(_ptr(props), S, K, _ptr(cost), float(reg), int(num_iter_max), float(stop_thr),
                                     float(tau), int(check_every), _ptr(pa), _ptr(pb), n, _ptr(plans), _ptr(out),
                                     _ptr(iters), _ptr(absn), _ptr(status), _ptr(ws), ws.numel(), _stream()),
          "pilot_sinkhorn_plans")
    if want_info:
        return plans, out, iters, absn, status
    return plans, out


def unpack_pairs(packed: torch.Tensor, chunk_stride: int, S: int, rng: PairRange, diag_value: float = 0.0,
                 dense: Optional[torch.Tensor] = None) -> torch.Tensor:
    """All-gathered packed chunks -> dense float64 matrix: S x S, or S_a x (S - S_a) for PAIRS_RECT."""
    _require_cuda(packed)
    assert packed.dtype == torch.float64 and packed.is_contiguous()
    if dense is None:
        shape = (rng.rows, S - rng.rows) if rng.mode == _lib.PAIRS_RECT else (S, S)
        dense = torch.empty(shape, dtype=torch.float64, device=packed.device)
    check(lib().pilot_unpack_pairs(_ptr(packed), int(chunk_stride), S, ctypes.byref(rng), float(diag_value),
                                   _ptr(dense), _stream()), "pilot_unpack_pairs")
    return dense


def knn_rows(X: torch.Tensor, k: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """k nearest rows of every row of X (S x S float64, rows = points), Euclidean, self included, sorted by
    (distance, index): (idx int32 [S,k], dist float64 [S,k]).  The Gram matrix is a library GEMM (cuBLAS DGEMM
    through torch.mm); selection and distances run in pilot_knn_rows."""
    _require_cuda(X)
    assert X.dim() == 2 and X.dtype == torch.float64
    S = X.shape[0]
    gram = torch.mm(X, X.t())
    idx = torch.empty((S, k), dtype=torch.int32, device=X.device)
    dist = torch.empty((S, k), dtype=torch.float64, device=X.device)
    ws = _workspace(max(S * 8, 256), X.device)
    check(lib().pilot_knn_rows(_ptr(gram), S, int(k), _ptr(idx), _ptr(dist), _ptr(ws), ws.numel(), _stream()),
          "pilot_knn_rows")
    return idx, dist


def silhouette_rows(X: torch.Tensor, labels, metric: str = "cosine") -> torch.Tensor:
    """Silhouette coefficient of every row of X (S x S float64, rows = points; metric 'cosine' or 'euclidean') or
    of every sample of the distance matrix X (metric 'precomputed') under the clustering ``labels``: float64 [S].
    The Gram matrix is a library GEMM (torch.mm); distances and the per-cluster reductions run in
    pilot_silhouette_rows.  Label bookkeeping (sklearn's LabelEncoder + a stable sort by label) is host NumPy."""
    _require_cuda(X)
    assert X.dim() == 2 and X.shape[0] == X.shape[1] and X.dtype == torch.float64
    S = X.shape[0]
    codes = np.unique(np.asarray(labels), return_inverse=True)[1].astype(np.int32).ravel()
    if codes.shape[0] != S:
        raise ValueError(f"Found input variables with inconsistent numbers of samples: [{S}, {codes.shape[0]}]")
    L = int(codes.max()) + 1
    if not 1 < L < S:
        raise ValueError("Number of labels is %d. Valid values are 2 to n_samples - 1 (inclusive)" % L)
    perm = np.argsort(codes, kind="stable").astype(np.int32)
    seg = np.concatenate([[0], np.cumsum(np.bincount(codes, minlength=L))]).astype(np.int32)
    if metric == "precomputed":
        mid, mat = _lib.SIL_PRECOMPUTED, X.contiguous()
    elif metric in ("cosine", "euclidean"):
        mid, mat = _lib.METRICS[metric], torch.mm(X, X.t())
    else:
        raise ValueError(f"silhouette metric {metric!r}: 'cosine', 'euclidean' or 'precomputed' (no CPU fallback)")
    dev = X.device
    perm_d, seg_d, lab_d = (torch.from_numpy(a).to(dev) for a in (perm, seg, codes))
    out = torch.empty(S, dtype=torch.float64, device=dev)
    ws = _workspace(max(S * 8, 256), dev)
    check(lib().pilot_silhouette_rows(_ptr(mat), S, int(mid), _ptr(perm_d), _ptr(seg_d), _ptr(lab_d), L, _ptr(out),
                                      _ptr(ws), ws.numel(), _stream()), "pilot_silhouette_rows")
    return out


def pipe_peak(kind: int) -> float:
    """Measured FP64-FMA (0), FP32-FMA (1) or FP64-mma.sync (2) throughput in TFLOP/s."""
    _require_cuda()
    v = ctypes.c_double(0.0)
    check(lib().pilot_pipe_peak(int(kind), ctypes.byref(v), _stream()), "pilot_pipe_peak")
    return float(v.value)
