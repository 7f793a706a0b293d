"""Host-side mirror of the reference's patient-distance interface.

Same names, argument meaning, return containers and error behaviour as
``/root/reference/pilotpy/tools/Trajectory.py`` (``wasserstein_distance`` :36-116,
``set_path_for_results`` :146-164, ``extract_data_anno_*`` :234-299,
``Cluster_Representations`` :377-436, ``cost_matrix`` :441-475,
``wasserstein_d`` :479-523, ``return_real_labels`` :617-642) so that a PILOT
user can switch ``pl.tl.wasserstein_distance`` for this one and everything
downstream (trajectory, clustering, statistics) runs unchanged.

The arithmetic of the four stages runs in hand-written sm_100a CUDA kernels
behind the C ABI (``include/pilot_b200.h``); this module only factorises
labels, moves buffers and assembles the pandas/NumPy containers of the
``adata.uns`` contract (SURVEY.md Appendix C).  There is no CPU fallback.
"""
from __future__ import annotations

import os
import warnings
from typing import Dict, List, Optional, Tuple

import numpy as np
import pandas as pd
import torch

from . import ops, pairs
from . import pairs as _pairs  # wasserstein_plans takes an argument named `pairs`
from .h5ad import load_h5ad  # noqa: F401  (pilotpy.tl.load_h5ad, Trajectory.py:121-137)

warnings.filterwarnings("ignore")  # the reference silences everything at import (Trajectory.py:32)

path_to_results = None  # module global read by pilotpy's cell_importance (Trajectory.py:708)


# ---------------------------------------------------------------------------
# extraction (host-only; Trajectory.py:146-164, 234-299)
# ---------------------------------------------------------------------------
def set_path_for_results():
    """Create ./Results_PILOT/plots like the reference and return the path."""
    if not os.path.exists("Results_PILOT/plots"):
        os.makedirs("Results_PILOT/plots")
    return "Results_PILOT/plots"


def extract_data_anno_scRNA_from_h5ad(adata, emb_matrix="PCA", clusters_col="cell_type", sample_col="sampleID",
                                      status="status"):
    """(data, annot) DataFrames from adata.obsm[emb_matrix] and three obs columns."""
    global path_to_results
    data = adata.obsm[emb_matrix]
    cols = ["PCA_" + str(i) for i in range(1, adata.obsm[emb_matrix].shape[1] + 1)]
    # copy=False: share the embedding's memory like pandas 2.0.x (the version the reference pins,
    # setup.py:21) does for ndarray input, instead of pandas >= 3's transposing 200 MB copy
    data = pd.DataFrame(data, columns=cols, copy=False)
    data = data.reset_index(drop=True)
    annot = adata.obs[[clusters_col, sample_col, status]]
    annot.columns = ["cell_type", "sampleID", "status"]
    annot = annot.reset_index(drop=True)
    path_to_results = set_path_for_results()
    return data, annot


def extract_data_anno_pathomics_from_h5ad(adata, var_names=[], clusters_col="Cell_type", sample_col="sampleID",
                                          status="status"):
    """(data, annot) DataFrames from adata[:, var_names].X and three obs columns."""
    global path_to_results
    data = adata[:, var_names].X
    data = pd.DataFrame(data, columns=var_names, copy=False)
    data = data.reset_index(drop=True)
    annot = adata.obs[[clusters_col, sample_col, status]]
    annot.columns = ["cell_type", "sampleID", "status"]
    annot = annot.reset_index(drop=True)
    path_to_results = set_path_for_results()
    return data, annot


# ---------------------------------------------------------------------------
# host factorisation helpers
# ---------------------------------------------------------------------------
def _raw_codes(col: pd.Series) -> Tuple[np.ndarray, object]:
    """Integer codes of a label column without hashing when it is Categorical.
    Returns (codes, labels-by-code); the codes keep the narrow dtype pandas stores them in (int8 for
    < 128 categories: 1 MB instead of 4 MB per million cells over PCIe) and are widened on the device.
    Missing labels are an error."""
    if isinstance(col.dtype, pd.CategoricalDtype):
        codes = col.cat.codes.to_numpy()
        labels = col.cat.categories
    else:
        cached = _factor_cache_get(col) if col.dtype == object else None
        if cached is not None:
            codes, labels = cached
        else:
            fast = _factorize_object_column(col) if col.dtype == object else None
            codes, labels = fast if fast is not None else pd.factorize(col, sort=False)
            codes = codes.astype(np.int32, copy=False)
            if col.dtype == object:
                _factor_cache_put(col, codes, labels)
    if len(codes) and codes.min() < 0:
        raise ValueError(f"column {col.name!r} contains missing labels")
    if codes.dtype not in (np.int8, np.int16, np.int32):
        codes = codes.astype(np.int32)
    return np.ascontiguousarray(codes), labels


# Factorising a column of Python str objects costs ~0.2 us per cell when every cell is its own object (1.1 s per
# 5 M-cell column, more than every GPU stage together); the same labels usually come back -- a second call with
# another metric or regularisation, the resolution sweeps of the consumers.  The result is therefore remembered,
# and a hit is validated EXACTLY: the cache entry holds its own references to the column's objects (so they stay
# alive, and str is immutable) and the new column must hold the same object pointer in every cell (one memcmp of
# 8 bytes per cell, ~5 ms per 5 M cells).  At most 4 columns are remembered.
_factor_cache: Dict[tuple, tuple] = {}
_FACTOR_CACHE_MAX = 4


def _object_pointers(vals: np.ndarray) -> np.ndarray:
    import ctypes
    return np.ctypeslib.as_array((ctypes.c_ssize_t * len(vals)).from_address(vals.ctypes.data))


def _factor_cache_key(vals: np.ndarray):
    if vals.dtype != object or vals.ndim != 1 or not vals.flags.c_contiguous or len(vals) < 50_000:
        return None, None
    ptrs = _object_pointers(vals)
    n = len(ptrs)
    return (n, int(ptrs[0]), int(ptrs[n // 2]), int(ptrs[-1])), ptrs


def _factor_cache_get(col: pd.Series):
    key, ptrs = _factor_cache_key(col.to_numpy())
    hit = _factor_cache.get(key) if key is not None else None
    if hit is None:
        return None
    held, codes, labels = hit
    if not np.array_equal(_object_pointers(held), ptrs):
        return None
    return codes, labels


def _factor_cache_put(col: pd.Series, codes, labels) -> None:
    vals = col.to_numpy()
    key, _ = _factor_cache_key(vals)
    if key is None:
        return
    if len(_factor_cache) >= _FACTOR_CACHE_MAX and key not in _factor_cache:
        _factor_cache.pop(next(iter(_factor_cache)))
    _factor_cache[key] = (vals.copy(), codes, labels)


_host_lib = {"lib": None, "tried": False}


def _host_helper():
    """libpilot_host.so (csrc/host_ingest.c), loaded with the GIL held; None when it has not been built."""
    if not _host_lib["tried"]:
        _host_lib["tried"] = True
        import ctypes
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "libpilot_host.so")
        if os.path.isfile(path):
            lib = ctypes.PyDLL(path)
            lib.pilot_factorize_str.restype = ctypes.c_int64
            lib.pilot_factorize_str.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p,
                                                ctypes.c_int64]
            _host_lib["lib"] = lib
    return _host_lib["lib"]


def _factorize_str_native(vals: np.ndarray):
    """(codes int32, labels object ndarray) of a contiguous object array of str, in order of first appearance, by
    the C helper; None when it does not apply (helper missing, non-str cells, > 2^20 labels)."""
    import ctypes
    lib = _host_helper()
    n = len(vals)
    if lib is None or n == 0:
        return None
    max_unique = min(n, 1 << 20)
    codes = np.empty(n, dtype=np.int32)
    uniq = np.zeros(max_unique, dtype=np.uintp)
    m = lib.pilot_factorize_str(vals.ctypes.data, n, codes.ctypes.data, uniq.ctypes.data, max_unique)
    if m < 0:
        return None
    labels = np.empty(m, dtype=object)
    for i in range(m):
        labels[i] = ctypes.cast(int(uniq[i]), ctypes.py_object).value   # borrowed from `vals`, which is alive
    return codes, labels


def _factorize_object_column(col: pd.Series):
    """pd.factorize(col, sort=False) for an object column that holds few distinct Python objects -- the usual
    case for label columns (a million references to a few dozen str objects).  Hashing Python objects costs
    ~35 ns per cell; factorising the object POINTERS as integers first and the few distinct objects afterwards
    costs ~8 ns per cell (default user input: str labels, Trajectory.py:261-263).  Returns None when it does
    not apply (then the caller uses pd.factorize directly)."""
    import ctypes
    vals = col.to_numpy()
    n = len(vals)
    if n < 50_000 or vals.dtype != object or not vals.flags.c_contiguous:
        return None
    native = _factorize_str_native(vals)
    if native is not None:
        return native
    ptrs = np.ctypeslib.as_array((ctypes.c_ssize_t * n).from_address(vals.ctypes.data))
    pcodes, puniq = pd.factorize(ptrs, sort=False)  # by identity, in order of first appearance
    if len(puniq) > max(4096, n // 16):
        return None  # (nearly) every cell its own object: no gain
    # the few distinct objects (borrowed from `vals`, which keeps them alive); equal values may sit in different
    # objects: merge them by value, still in order of first appearance; missing values keep pandas' code -1
    objs = np.empty(len(puniq), dtype=object)
    for i, p in enumerate(puniq):
        objs[i] = ctypes.cast(int(p), ctypes.py_object).value
    vcodes, labels = pd.factorize(objs, sort=False)
    return vcodes[pcodes], labels


def _unique_in_order(col: pd.Series, labels, perm: np.ndarray):
    """What ``col.unique()`` returns (same container type), built from the codes."""
    if isinstance(col.dtype, pd.CategoricalDtype):
        return pd.Categorical.from_codes(perm, dtype=col.dtype)
    if isinstance(labels, pd.Index):
        taken = labels.take(perm)
        # extension dtypes (pandas >= 3 `str`) come back from .unique() as their ExtensionArray
        return taken.array if isinstance(taken.dtype, pd.api.extensions.ExtensionDtype) else taken.to_numpy()
    return np.asarray(labels)[perm]


def _device() -> torch.device:
    if not torch.cuda.is_available():
        raise ops._lib.PilotLibraryError("pilot_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _to_device(arr: np.ndarray) -> torch.Tensor:
    return torch.from_numpy(arr).to(_device(), non_blocking=False)


# Host staging.  A pageable source makes cudaMemcpy stage through the driver's bounce buffer and block
# the host; label codes therefore go through a grow-only pinned buffer of our own and are copied
# asynchronously.  The buffer is reused by the next call, which is safe because every public function
# ends with a device-to-host read of its result (a full stream sync).
_pinned_stage = {"buf": None, "used": 0}
_copy_streams: Dict[int, "torch.cuda.Stream"] = {}


def _stage_reset() -> None:
    _pinned_stage["used"] = 0


_TORCH_DTYPE = {"int8": torch.int8, "int16": torch.int16, "int32": torch.int32, "int64": torch.int64,
                "uint8": torch.uint8, "float32": torch.float32, "float64": torch.float64}


def _to_device_staged(arr: np.ndarray) -> torch.Tensor:
    dev = _device()
    nbytes = (arr.nbytes + 255) // 256 * 256
    off = _pinned_stage["used"]
    buf = _pinned_stage["buf"]
    if buf is None or off + nbytes > buf.numel():
        if off != 0:  # would have to move live data: plain blocking copy instead
            return _to_device(arr)
        buf = torch.empty(max(nbytes * 2, 1 << 22), dtype=torch.uint8, pin_memory=True)
        _pinned_stage["buf"] = buf
    _pinned_stage["used"] = off + nbytes
    host = buf[off:off + arr.nbytes].view(_TORCH_DTYPE[arr.dtype.name]).view(arr.shape)
    host.numpy()[...] = arr
    return host.to(dev, non_blocking=True)


_ring = {"bufs": None, "events": None}
_RING_CHUNK_BYTES = 32 << 20


def _ring_copy(dst: torch.Tensor, src: torch.Tensor, dev: torch.device) -> "torch.cuda.Event":
    """Copy the pageable CPU tensor ``src`` into the device tensor ``dst`` (same shape, both contiguous) in chunks
    through two page-locked buffers on the copy stream; returns the event the compute stream has to wait for."""
    if _ring["bufs"] is None:
        _ring["bufs"] = [torch.empty(_RING_CHUNK_BYTES, dtype=torch.uint8, pin_memory=True) for _ in range(2)]
        _ring["events"] = [None, None]
    main = torch.cuda.current_stream(dev)
    side = _copy_stream(dev)
    side.wait_stream(main)  # dst was allocated in compute-stream order
    s8 = src.reshape(-1).view(torch.uint8)
    d8 = dst.reshape(-1).view(torch.uint8)
    total = s8.numel()
    for c, off in enumerate(range(0, total, _RING_CHUNK_BYTES)):
        m = min(_RING_CHUNK_BYTES, total - off)
        buf, ev = _ring["bufs"][c & 1], _ring["events"][c & 1]
        if ev is not None:
            ev.synchronize()                      # the DMA that last read this chunk has finished
        buf[:m].copy_(s8[off:off + m])            # host copy (intra-op threads)
        with torch.cuda.stream(side):
            d8[off:off + m].copy_(buf[:m], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(side)
        _ring["events"][c & 1] = ev
    dst.record_stream(side)
    done = torch.cuda.Event()
    done.record(side)
    return done


def _copy_stream(dev: torch.device) -> "torch.cuda.Stream":
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if idx not in _copy_streams:
        _copy_streams[idx] = torch.cuda.Stream(device=dev)
    return _copy_streams[idx]


class _Labels:
    """Device-resident factorised annotation shared by the stages of one call."""

    def __init__(self, annot: pd.DataFrame, cell_col_name, sample_col_name):
        _stage_reset()  # previous calls ended with a sync: their staged copies are done
        self.n = len(annot)
        self.cell_col = annot[cell_col_name]
        self.samp_col = annot[sample_col_name]
        ct, self.ct_labels = _raw_codes(self.cell_col)
        sm, self.sm_labels = _raw_codes(self.samp_col)
        self.K_raw, self.S_raw = len(self.ct_labels), len(self.sm_labels)
        self.ct_dev = _to_device_staged(ct).to(torch.int32)
        self.sm_dev = _to_device_staged(sm).to(torch.int32)
        self.counts_raw, first_ct, first_smp = ops.hist(self.ct_dev, self.sm_dev, self.K_raw, self.S_raw)
        first = torch.cat([first_ct, first_smp]).cpu().numpy()  # the only sync of stage 1
        fk, fs = first[: self.K_raw], first[self.K_raw:]
        pk = np.argsort(fk, kind="stable")
        ps = np.argsort(fs, kind="stable")
        self.perm_k = np.ascontiguousarray(pk[fk[pk] < self.n], dtype=np.int32)  # raw codes in .unique() order
        self.perm_s = np.ascontiguousarray(ps[fs[ps] < self.n], dtype=np.int32)
        self.first_smp = fs[self.perm_s]
        self.perm_k_dev = _to_device(self.perm_k)
        self.perm_s_dev = _to_device(self.perm_s)
        self.K, self.S = len(self.perm_k), len(self.perm_s)
        self.cells = _unique_in_order(self.cell_col, self.ct_labels, self.perm_k)
        self.samples = _unique_in_order(self.samp_col, self.sm_labels, self.perm_s)

    def proportions(self, regulizer, normalization) -> Tuple[torch.Tensor, torch.Tensor]:
        return ops.props_finalize(self.counts_raw, self.perm_k_dev, self.perm_s_dev, self.n, regulizer,
                                  bool(normalization == True))  # noqa: E712  (reference: `normalization == True`)


def _shard_min_bytes() -> int:
    return int(os.environ.get("PILOT_SHARD_H2D_MIN_BYTES", str(32 << 20)))


def _embedding_to_device(data, group=None) -> torch.Tensor:
    """Stage the embedding.  Page-locked input (e.g. a torch pinned tensor's numpy view) is copied on a
    side stream so that the label factorisation, the histogram and the proportion table -- host work
    plus small kernels -- run while the 200 MB cross PCIe; the compute stream waits for the copy before
    it is first read (stage 2).  Pageable input is a plain blocking copy.

    Several ranks (torch.distributed initialised; every rank holds the same host array, as in any SPMD
    launch of the same script): rank r uploads only rows [r n/N, (r+1) n/N) over ITS PCIe link and the
    slices are exchanged with one in-place NCCL all-gather over NVLink right before stage 2 -- the host
    memory system no longer serves N full copies at once (round 1: the 8-rank end-to-end step took 2x
    the 1-rank one for this reason)."""
    X = data.to_numpy() if isinstance(data, pd.DataFrame) else np.asarray(data)
    if X.dtype not in (np.float32, np.float64):
        X = X.astype(np.float64)  # pandas' nanmedian promotes non-float input to float64
    if X.ndim != 2:
        raise ValueError("embedding must be 2-dimensional")
    if not X.flags.c_contiguous:
        X = np.ascontiguousarray(X)
    host = torch.from_numpy(X)
    dev = _device()
    nranks, rank = pairs.world(group)
    n = X.shape[0]
    if nranks > 1 and X.nbytes >= _shard_min_bytes():
        per = -(-n // nranks)
        full = torch.empty((per * nranks, X.shape[1]), dtype=host.dtype, device=dev)
        r0, r1 = min(n, rank * per), min(n, (rank + 1) * per)
        src, dst = host[r0:r1], full[r0:r1]
        gather = (per, rank, group)
    else:
        full = None
        src, dst, gather = host, None, None
    if not host.is_pinned():
        # pageable input (a user's plain ndarray): through a ring of two page-locked chunks -- the host copy into
        # one chunk (multi-threaded) overlaps the DMA of the other, instead of the driver's single-threaded bounce
        # buffer; small arrays take the plain blocking copy
        if gather is None:
            if X.nbytes < (64 << 20):
                return _to_device(X)
            full = torch.empty(host.shape, dtype=host.dtype, device=dev)
            dst = full
        done = _ring_copy(dst, src, dev)
        X_dev = full[:n]
        X_dev._pilot_ready = done
        if gather is not None:
            X_dev._pilot_gather = (full,) + gather
        return X_dev
    main = torch.cuda.current_stream(dev)
    side = _copy_stream(dev)
    if gather is None:
        full = torch.empty(host.shape, dtype=host.dtype, device=dev)  # allocated in compute-stream order
        dst = full
    side.wait_stream(main)
    with torch.cuda.stream(side):
        dst.copy_(src, non_blocking=True)
    full.record_stream(side)  # the allocator must not hand the block out again while the copy is in flight
    done = torch.cuda.Event()
    done.record(side)
    X_dev = full[:n]
    X_dev._pilot_ready = done  # consumed by _cost_device
    if gather is not None:
        X_dev._pilot_gather = (full,) + gather
    return X_dev


def _props_dict(samples, props_host: np.ndarray) -> Dict[object, np.ndarray]:
    return {s: props_host[i].copy() for i, s in enumerate(samples)}


def _labelled_square(mat_T: np.ndarray, labels, name: str) -> pd.DataFrame:
    """What the reference's three statements build --
        f = pd.DataFrame.from_dict(mat).T; f.columns = labels; f[name] = labels; f = f.set_index(name)
    (Trajectory.py:470-473 and :518-521) -- constructed in one step: ~0.4 ms instead of ~1.3 ms of
    pandas bookkeeping.  The index types follow the same pandas code paths: the columns are the
    labels' Index after inserting and deleting `name` (which is what turns a CategoricalIndex or an
    integer Index into an object one), the row index is built from the column the assignment would
    have created.  tests/test_host_logic.py checks it against the literal statements."""
    cols = pd.Index(labels) if not isinstance(labels, pd.Index) else labels
    cols = cols.insert(len(cols), name)[:-1]
    idx = pd.Index(pd.Series(labels, name=name)._values, name=name)
    return pd.DataFrame(np.ascontiguousarray(mat_T), index=idx, columns=cols, copy=False)


def _labelled_square_reference(mat: np.ndarray, labels, name: str) -> pd.DataFrame:
    f = pd.DataFrame.from_dict(mat).T
    f.columns = labels
    f[name] = labels
    return f.set_index(name)


def _cost_frame(dis: np.ndarray, cells) -> pd.DataFrame:
    if len(cells) == 0 or np.asarray(cells).dtype.kind in "iu":  # RangeIndex special cases: literal path
        return _labelled_square_reference(dis, cells, "cell_types")
    return _labelled_square(dis.T, cells, "cell_types")


def _emd_frame(EMD: np.ndarray, samples_id: List, EMD_T: Optional[np.ndarray] = None) -> pd.DataFrame:
    # DataFrame.from_dict(EMD).T (Trajectory.py:518) is the transpose; EMD_T, when given, is an independent
    # C-contiguous copy of it that the frame takes over without another pass over S x S doubles
    if len(samples_id) == 0 or np.asarray(samples_id).dtype.kind in "iu":
        return _labelled_square_reference(EMD, samples_id, "sampleID")
    return _labelled_square(EMD.T if EMD_T is None else EMD_T, samples_id, "sampleID")


# ---------------------------------------------------------------------------
# Stage 1: proportions (Trajectory.py:377-436)
# ---------------------------------------------------------------------------
def Cluster_Representations(df, cell_col=0, sample_col=1, regulizer=0.2, normalization=True):
    """Per-sample, Dirichlet-smoothed cell-type proportions.

    Returns ``{sample: float64[K]}`` with samples and cell types in order of first
    appearance.  Like the reference, the frame must carry the columns
    ``'cell_type'`` and ``'sampleID'`` (hard-coded at Trajectory.py:405,407,429).
    """
    cell_name = df.columns[cell_col]
    samp_name = df.columns[sample_col]
    if "cell_type" not in df.columns:
        raise KeyError("cell_type")
    if normalization == True and "sampleID" not in df.columns:  # noqa: E712
        raise KeyError("sampleID")
    if cell_name != "cell_type" or (normalization == True and samp_name != "sampleID"):  # noqa: E712
        raise ValueError("Cluster_Representations: cell_col/sample_col must select the 'cell_type'/'sampleID' "
                         "columns (the reference hard-codes these names, Trajectory.py:405-429)")
    lab = _Labels(df, cell_name, samp_name)
    props, counts = lab.proportions(regulizer, normalization)
    counts_h = counts.cpu().numpy()
    if int(counts_h.sum()) != lab.n:
        raise ValueError("label codes out of range")
    return _props_dict(lab.samples, props.cpu().numpy())


# ---------------------------------------------------------------------------
# Stage 2: cost matrix (Trajectory.py:441-475)
# ---------------------------------------------------------------------------
def _embedding_ready(X_dev: torch.Tensor) -> torch.Tensor:
    """Make the compute stream wait for the staged embedding (side-stream copy, rank slices)."""
    ready = getattr(X_dev, "_pilot_ready", None)
    if ready is not None:
        torch.cuda.current_stream(X_dev.device).wait_event(ready)
        X_dev._pilot_ready = None
    gather = getattr(X_dev, "_pilot_gather", None)
    if gather is not None:
        # every rank uploaded its row slice: exchange them over NVLink (in place: rank r's slice is already
        # where the all-gather would put it)
        import torch.distributed as dist
        full, per, rank, group = gather
        dist.all_gather_into_tensor(full.view(-1), full[rank * per:(rank + 1) * per].reshape(-1), group=group)
        X_dev._pilot_gather = None
    return X_dev


def _cost_device(lab: _Labels, X_dev: torch.Tensor, metric) -> Tuple[torch.Tensor, torch.Tensor]:
    _embedding_ready(X_dev)
    if X_dev.shape[0] != lab.n:
        raise ValueError(f"Item wrong length {lab.n} instead of {X_dev.shape[0]}.")
    _, cent64_raw = ops.centroid_median(X_dev, lab.ct_dev, lab.K_raw)
    cent64 = cent64_raw.index_select(0, lab.perm_k_dev.long()).contiguous()
    cost, cost_norm, _ = ops.cdist(cent64, metric)
    return cost, cost_norm


def cost_matrix(annot, data, metric="cosine"):
    """Median centroid of every cell type, then their pairwise distances.

    Returns ``(dis, cost)``: the K x K ndarray and the labelled DataFrame
    (index name ``'cell_types'``), both un-normalised.
    """
    lab = _Labels(annot, annot.columns[0], annot.columns[1] if annot.shape[1] > 1 else annot.columns[0])
    cost, _ = _cost_device(lab, _embedding_to_device(data), metric)
    dis = cost.cpu().numpy()
    return dis, _cost_frame(dis, lab.cells)


# ---------------------------------------------------------------------------
# Stage 3: all-pairs OT (Trajectory.py:479-523)
# ---------------------------------------------------------------------------
def _check_emd_inputs(P: np.ndarray, cost: np.ndarray) -> None:
    # what ot.emd2 asserts per pair (POT ot/lp/__init__.py::emd2)
    assert P.shape[1] == cost.shape[0] and P.shape[1] == cost.shape[1], \
        "Dimension mismatch, check dimensions of M with a and b"
    sums = P.sum(axis=1)
    if sums.size and float(sums.max() - sums.min()) >= 1.5e-6:
        raise AssertionError("\nArrays are not almost equal to 6 decimals\n"
                             "a and b vector must have the same sum")


def _stack_props(Clu_rep) -> Tuple[list, np.ndarray]:
    """(sample ids, proportions [S, K] float64) of a {sample: proportions} dict."""
    ids = list(Clu_rep.keys())
    if not ids:
        return ids, np.zeros((0, 0))
    return ids, np.ascontiguousarray(np.stack([np.asarray(Clu_rep[s], dtype=np.float64) for s in ids]))


def wasserstein_d(Clu_rep, cost, regularized="unreg", reg=0.1, precision="f64"):
    """All ordered sample pairs: exact EMD (``regularized == "unreg"``) or stabilised
    Sinkhorn (anything else).  Returns ``(EMD ndarray [S,S], DataFrame indexed by sampleID)``.
    ``precision`` is an extension of the reference signature: "f64" (default, within 1e-9 of POT) or
    "f32" (single-precision solvers, within 1e-4)."""
    samples_id, P = _stack_props(Clu_rep)
    C = np.ascontiguousarray(np.asarray(cost, dtype=np.float64))
    if len(samples_id) == 0:
        EMD = np.zeros((0, 0))
        return EMD, _emd_frame(EMD, samples_id)
    sym = None
    if regularized == "unreg":
        _check_emd_inputs(P, C)
        sym = pairs.cost_is_symmetric_metric_like(C)  # K x K on the host: no device round trip
    EMD, EMD_T = pairs.all_pairs_host(_to_device(P), _to_device(C), regularized, reg, symmetric=sym,
                                      with_transpose=True, precision=precision)
    return EMD, _emd_frame(EMD, samples_id, EMD_T)




def _check_two_sets(P_a: np.ndarray, P_b: np.ndarray, C: np.ndarray, regularized) -> None:
    """Checks of wasserstein_d_cross / _extend made before any device work: the same number of cell types in
    both sets and the cost, and under "unreg" equal masses across both sets (_check_emd_inputs)."""
    if P_a.shape[1] != P_b.shape[1]:
        raise ValueError(f"the two sample sets have {P_a.shape[1]} and {P_b.shape[1]} cell types")
    if C.shape != (P_a.shape[1], P_a.shape[1]):
        raise ValueError(f"cost has shape {C.shape}, expected {P_a.shape[1]} x {P_a.shape[1]} (one row and "
                         "column per cell type)")
    if regularized == "unreg":
        _check_emd_inputs(np.concatenate([P_a, P_b]), C)


def wasserstein_d_cross(Clu_rep_a, Clu_rep_b, cost, regularized="unreg", reg=0.1, precision="f64"):
    """OT costs between two sample sets that share the cell types and the cost matrix, for example a
    discovery and a validation cohort: exact EMD (``regularized == "unreg"``) or stabilised Sinkhorn.

    Returns ``(D ndarray [S_a, S_b], DataFrame)`` with ``D[i, j]`` the cost of (a_i, b_j); the frame is
    indexed by the ids of ``Clu_rep_a`` (index name ``sampleID``) and its columns are the ids of
    ``Clu_rep_b`` (not transposed).  Only the S_a x S_b problems are solved, and ``D`` is bit-identical to
    the same entries of ``wasserstein_d({**Clu_rep_a, **Clu_rep_b}, cost, ...)`` when the ids are distinct."""
    ids_a, P_a = _stack_props(Clu_rep_a)
    ids_b, P_b = _stack_props(Clu_rep_b)
    if ids_a and ids_b:
        C = np.ascontiguousarray(np.asarray(cost, dtype=np.float64))
        _check_two_sets(P_a, P_b, C, regularized)
        D = pairs.cross_pairs_host(_to_device(P_a), _to_device(P_b), _to_device(C), regularized, reg,
                                   precision=precision)
    else:
        D = np.zeros((len(ids_a), len(ids_b)))
    frame = pd.DataFrame(D.copy(), index=pd.Index(ids_a, name="sampleID"), columns=pd.Index(ids_b))
    return D, frame


def wasserstein_d_extend(Clu_rep, EMD, Clu_rep_new, cost, regularized="unreg", reg=0.1, precision="f64"):
    """Extend the matrix ``EMD`` of the samples ``Clu_rep`` with the samples ``Clu_rep_new``.

    Returns ``(EMD, EMD_df)`` over old ∪ new (old samples first), bit-identical to
    ``wasserstein_d({**Clu_rep, **Clu_rep_new}, cost, regularized, reg, precision)``, frame included, while
    solving only the problems that involve a new sample: old x new and new x new, and new x old unless the
    exact solver mirrors (symmetric cost), as the square does.  Sinkhorn with K <= 16 solves the whole union
    instead when the old cohort is below 448 samples and the union is not (the solver changes there).  ``EMD`` must be this library's
    ``wasserstein_d(Clu_rep, cost, ...)`` output with the same arguments; that is not checked (only its shape
    is), and the old corner is copied as given.  An id present in both sets raises."""
    ids_old, P_old = _stack_props(Clu_rep)
    ids_new, P_new = _stack_props(Clu_rep_new)
    if not ids_old:
        return wasserstein_d(Clu_rep_new, cost, regularized, reg, precision)
    if not ids_new:
        EMD = np.array(EMD, dtype=np.float64)
        return EMD, _emd_frame(EMD, ids_old)
    shared = set(ids_old).intersection(ids_new)
    if shared:
        raise ValueError(f"wasserstein_d_extend: sample ids in both sets: {sorted(map(str, shared))[:5]}")
    EMD = np.asarray(EMD, dtype=np.float64)
    S_old, S_new = len(ids_old), len(ids_new)
    if EMD.shape != (S_old, S_old):
        raise ValueError(f"EMD is {EMD.shape}, expected ({S_old}, {S_old}) for the samples of Clu_rep")
    C = np.ascontiguousarray(np.asarray(cost, dtype=np.float64))
    _check_two_sets(P_old, P_new, C, regularized)
    if regularized != "unreg" and pairs.sinkhorn_form_changes(S_old, S_old + S_new, C.shape[0]):
        # the union crosses the cohort size at which Sinkhorn changes solver for K <= 16, so EMD's bits are not
        # those of the union's square: solve it all (S_old <= 447 here, at most 200 000 extra problems)
        return wasserstein_d({**Clu_rep, **Clu_rep_new}, cost, regularized, reg, precision)
    sym = pairs.cost_is_symmetric_metric_like(C) if regularized == "unreg" else None
    old_new, new_rows = pairs.extend_pairs(_to_device(P_old), _to_device(P_new), _to_device(C), regularized, reg,
                                           symmetric=sym, precision=precision)
    S = S_old + S_new
    out = np.empty((S, S), dtype=np.float64)
    out[:S_old, S_old:] = old_new.cpu().numpy()
    out[S_old:] = new_rows.cpu().numpy()
    out[:S_old, :S_old] = EMD
    # the square's frame takes its transpose; a mirrored matrix is its own transpose
    return out, _emd_frame(out, ids_old + ids_new, out.copy() if sym else None)


_PLAN_CHUNK_BYTES = 256 << 20  # device memory of the plans of one chunk (512 plans at K = 256)


def wasserstein_plans(Clu_rep, cost, pairs, regularized="unreg", reg=0.1, Clu_rep_b=None):
    """Transport plans of chosen sample pairs: what the distance between two samples is made of.

    ``pairs`` is a sequence of ``(id_a, id_b)``.  Without ``Clu_rep_b`` both ids are keys of ``Clu_rep`` and the
    plans follow ``wasserstein_d(Clu_rep, cost, regularized, reg)``; with it ``id_a`` is a key of ``Clu_rep`` and
    ``id_b`` of ``Clu_rep_b``, and they follow ``wasserstein_d_cross(Clu_rep, Clu_rep_b, ...)``.  Returns
    ``(plans ndarray [n, K, K], costs ndarray [n])``: ``plans[l, r, c]`` is the mass that cell type r of id_a
    sends to cell type c of id_b, and ``sum(cost * plans[l])`` is the distance.  Exact EMD
    (``regularized == "unreg"``): ``costs`` equal the matrix entries bit for bit (a mirrored matrix gives the
    transposed plan of (id_b, id_a), and ``diag(a)`` with cost 0 on its diagonal).  Sinkhorn: POT's reference form
    of the plan, costs within 1e-12 relative of the matrix entries.  Solved on the GPU in FP64, in chunks."""
    ids_a, P_a = _stack_props(Clu_rep)
    ids_b, P_b = _stack_props(Clu_rep_b) if Clu_rep_b is not None else (ids_a, P_a)
    pos_a = {s: i for i, s in enumerate(ids_a)}
    pos_b = {s: i for i, s in enumerate(ids_b)}
    rows = np.array([pos_a[a] for a, _ in pairs], dtype=np.int64)  # KeyError for an unknown id
    cols = np.array([pos_b[b] for _, b in pairs], dtype=np.int64)
    C = np.ascontiguousarray(np.asarray(cost, dtype=np.float64))
    if rows.size == 0:
        K = C.shape[0] if C.ndim == 2 else 0
        return np.zeros((0, K, K)), np.zeros((0,))
    _check_two_sets(P_a, P_b, C, regularized)
    if Clu_rep_b is not None:  # the block between two sets never mirrors
        P = np.concatenate([P_a, P_b])
        cols = cols + len(ids_a)
        sym = False
    else:
        P = P_a
        sym = _pairs.cost_is_symmetric_metric_like(C) if regularized == "unreg" else None
    K = C.shape[0]
    n = rows.size
    plans = np.empty((n, K, K), dtype=np.float64)
    costs = np.empty((n,), dtype=np.float64)
    P_d, C_d = _to_device(np.ascontiguousarray(P)), _to_device(C)
    chunk = max(1, _PLAN_CHUNK_BYTES // (8 * K * K))
    for s in range(0, n, chunk):
        g, c = _pairs.entry_plans(P_d, C_d, rows[s:s + chunk], cols[s:s + chunk], regularized, reg, symmetric=sym)
        plans[s:s + chunk] = g.cpu().numpy()
        costs[s:s + chunk] = c.cpu().numpy()
    return plans, costs


def transport_plan(adata, sample_a, sample_b, regularized="unreg", reg=0.1):
    """The transport plan between two samples after ``wasserstein_distance``: ``(DataFrame K x K, cost)``, index =
    the cell types of ``sample_a`` (the mass it sends), columns = those of ``sample_b``, both named as in
    ``adata.uns['cost']``.  The cost is normalised as ``wasserstein_distance`` does (``cost / cost.max()``, the same
    IEEE division), so with that call's ``regularized`` and ``reg`` an exact-EMD cost equals
    ``adata.uns['EMD'][i, j]`` bit for bit."""
    cost_df = adata.uns["cost"]
    C = np.asarray(cost_df.to_numpy(), dtype=np.float64)
    plans, costs = wasserstein_plans(adata.uns["proportions"], C / C.max(), [(sample_a, sample_b)], regularized, reg)
    frame = pd.DataFrame(plans[0], index=cost_df.index.copy(), columns=cost_df.columns.copy())
    return frame, float(costs[0])


# ---------------------------------------------------------------------------
# labels (Trajectory.py:617-642)
# ---------------------------------------------------------------------------
def return_real_labels(df, category="status", sample_col=1):
    """First ``category`` value of every sample, samples in order of first appearance."""
    scol = df.columns[sample_col]
    first = ~df[scol].duplicated(keep="first")
    return list(df[category][first])


# ---------------------------------------------------------------------------
# entry point (Trajectory.py:36-116)
# ---------------------------------------------------------------------------
def wasserstein_distance(adata, emb_matrix="X_PCA", clusters_col="cell_types", sample_col="sampleID",
                         status="status", metric="cosine", regulizer=0.2, normalization=True,
                         regularized="unreg", reg=0.1, res=0.01, steper=0.01, data_type="scRNA",
                         return_sil_ari=False, precision="f64"):
    """Drop-in for ``pilotpy.tl.wasserstein_distance``: writes ``data``, ``annot``,
    ``proportions``, ``cost``, ``EMD_df``, ``EMD`` and ``real_labels`` into ``adata.uns``."""
    if return_sil_ari:
        _require_clustering_tail()  # fail before any device work or side effect, not after (ADVICE r1)
    X_dev = None
    if data_type == "scRNA":
        # stage the embedding straight from the caller's array (no detour through the DataFrame) and
        # first of all: the copy overlaps everything up to the median kernel
        X_dev = _embedding_to_device(adata.obsm[emb_matrix])
        data, annot = extract_data_anno_scRNA_from_h5ad(adata, emb_matrix=emb_matrix, clusters_col=clusters_col,
                                                        sample_col=sample_col, status=status)
    else:
        data, annot = extract_data_anno_pathomics_from_h5ad(adata, var_names=list(adata.var_names),
                                                            clusters_col=clusters_col, sample_col=sample_col,
                                                            status=status)
        X_dev = _embedding_to_device(data)
    adata.uns["data"] = data
    adata.uns["annot"] = annot

    lab = _Labels(annot, "cell_type", "sampleID")
    props, counts = lab.proportions(regulizer, normalization)
    cost, cost_norm = _cost_device(lab, X_dev, metric)
    # enqueue the pair stage before the first device-to-host read, so that the host-side checks and the
    # construction of the result containers overlap it (its result is dropped if a check raises)
    if lab.S * lab.S * 8 >= (1 << 28):
        # big matrix: band pipeline, the rows cross PCIe while later bands are solved (pairs.all_pairs_host)
        props_h = props.cpu().numpy()
        if int(counts.sum().item()) != lab.n:
            raise ValueError("label codes out of range")
        if regularized == "unreg":
            _check_emd_inputs(props_h, np.empty((lab.K, lab.K)))
        EMD, EMD_T = pairs.all_pairs_host(props, cost_norm, regularized, reg, with_transpose=True, precision=precision)
    else:
        emd_dev = pairs.all_pairs(props, cost_norm, regularized, reg, precision=precision)
        props_h = props.cpu().numpy()
        if int(counts.sum().item()) != lab.n:
            raise ValueError("label codes out of range")
        if regularized == "unreg":
            _check_emd_inputs(props_h, np.empty((lab.K, lab.K)))
        EMD, EMD_T = emd_dev.cpu().numpy(), None

    adata.uns["proportions"] = _props_dict(lab.samples, props_h)
    dis = cost.cpu().numpy()
    adata.uns["cost"] = _cost_frame(dis, lab.cells)
    adata.uns["EMD_df"] = _emd_frame(EMD, list(adata.uns["proportions"].keys()), EMD_T)
    adata.uns["EMD"] = EMD

    if return_sil_ari:
        # the reference's Leiden / ARI / silhouette tail (Trajectory.py:107-113) is a consumer of the matrix
        # (scanpy + leidenalg + sklearn, SURVEY.md 8f #2): run the reference's own functions on it
        Clustering, Sil_computing = _require_clustering_tail()
        predicted_labels, ARI, real_labels = Clustering(EMD / EMD.max(), annot, metric=metric, res=res, steper=steper)
        adata.uns["real_labels"] = real_labels
        adata.uns["Sil"] = Sil_computing(EMD / EMD.max(), real_labels, metric=metric)
        adata.uns["ARI"] = ARI
    else:
        # first status per sample, via the first-appearance cell index the histogram kernel produced
        adata.uns["real_labels"] = list(annot["status"].iloc[lab.first_smp])


def Sil_computing(EMD, real_labels, metric="cosine"):
    """Silhouette score of the samples (``Trajectory.py:593-612``: ``sklearn.metrics.silhouette_score(EMD,
    real_labels, metric=metric)``, the ROWS of the matrix as points).  GPU: one library DGEMM for the Gram matrix,
    distances and per-cluster reductions in ``pilot_silhouette_rows`` (SURVEY.md 8f #2).  ``EMD``: ndarray or CUDA
    tensor; metrics 'cosine' (the reference's default), 'euclidean' and 'precomputed'."""
    if not torch.cuda.is_available():
        raise ops._lib.PilotLibraryError("pilot_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    E = EMD if isinstance(EMD, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(EMD, dtype=np.float64)).cuda()
    if metric == "precomputed" and bool((torch.diagonal(E).abs() > 1e-10).any()):
        raise ValueError("The precomputed distance matrix contains non-zero elements on the diagonal. "
                         "Use np.fill_diagonal(X, 0).")           # scikit-learn's own check and message
    sil = ops.silhouette_rows(E.contiguous(), real_labels, metric)
    return float(sil.cpu().numpy().mean())


def _require_clustering_tail():
    """``Clustering`` of the reference (Trajectory.py:527-588): scanpy neighbours + Leiden + Rand index.  Graph
    clustering is not re-implemented here (it needs scanpy and leidenalg and cannot be pinned without them); the
    silhouette half of the tail is ``Sil_computing`` above."""
    try:
        from pilotpy.tools.Trajectory import Clustering  # type: ignore
    except Exception as exc:
        raise NotImplementedError(
            "return_sil_ari=True runs the reference's Leiden/ARI tail (Trajectory.py:107-113), which needs pilotpy "
            "with scanpy + leidenalg importable; it is a consumer of the distance matrix, outside the "
            f"patient-distance hot path (SURVEY.md 8f #2, #4).  Import failed with: {exc!r}") from exc
    return Clustering, Sil_computing


def Precomputed_distance(adata, distances, cost_df, features_matrix, emb_matrix="X_PCA", clusters_col="cell_types",
                         sample_col="sampleID", status="status", data_type="scRNA"):
    """Store externally computed sample distances in ``adata.uns`` (Trajectory.py:1687-1727): the reference's
    bring-your-own-backend seam.  The reference body reads an undefined ``data_type`` (:1716, a NameError in
    2.0.6); here it is a keyword argument with the value the other entry points default to."""
    if data_type == "scRNA":
        data, annot = extract_data_anno_scRNA_from_h5ad(adata, emb_matrix=emb_matrix, clusters_col=clusters_col,
                                                        sample_col=sample_col, status=status)
    else:
        data, annot = extract_data_anno_pathomics_from_h5ad(adata, var_names=list(adata.var_names),
                                                            clusters_col=clusters_col, sample_col=sample_col,
                                                            status=status)
    adata.uns["data"] = data
    adata.uns["annot"] = annot
    adata.uns["proportions"] = features_matrix
    adata.uns["cost"] = cost_df
    adata.uns["EMD"] = distances
    adata.uns["real_labels"] = return_real_labels(annot)
