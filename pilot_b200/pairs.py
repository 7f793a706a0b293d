"""All-pairs OT on one or several GPUs.

The pair space is partitioned over the ranks of the current ``torch.distributed``
process group exactly as ``pilot_pair_range`` (include/pilot_b200.h) describes:
blocks of consecutive problems dealt round-robin.  Every rank solves its blocks
with the CUDA kernels, the packed results are assembled with ONE all-gather
(NCCL over NVLink on a B200 box) and unpacked (and mirrored for the symmetric
exact-EMD case) into the dense S x S matrix on every rank.

``all_pairs``      -> dense matrix on the device (one window over the whole pair space)
``all_pairs_host`` -> dense matrix in host memory: the pair space is cut into bands of whole
                      matrix rows; band b's rows cross PCIe on a copy stream while band b+1
                      is being solved, so the 3.2 GB of a 20 000-sample matrix cost no time
                      on top of the kernels.
``cross_pairs`` / ``cross_pairs_host`` -> the S_a x S_b block between two sample sets (the RECT
                      pair space over their concatenation), on the device / in host memory.
``extend_pairs``   -> the entries a matrix over S_old samples lacks once S_new samples join.
Every block is bit-identical to the same entries of the square over the concatenated samples.

Replaces the double loop of the reference's ``wasserstein_d``
(/root/reference/pilotpy/tools/Trajectory.py:505-515).
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, ops
from ._lib import PairRange


def world(group=None) -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(group), dist.get_rank(group)
    return 1, 0


# ---- host-side statement of the partition (mirrors common.cuh; used for sizing and tests) ----
def range_count(total: int, block: int, nranks: int, rank: int) -> int:
    if total <= 0:
        return 0
    nblocks = -(-total // block)
    mine = nblocks // nranks + (1 if (nblocks % nranks) > rank else 0)
    if mine == 0:
        return 0
    last_block = (mine - 1) * nranks + rank
    cnt = mine * block
    if last_block == nblocks - 1:
        cnt -= nblocks * block - total
    return cnt


def local_to_global(l: int, block: int, nranks: int, rank: int) -> int:
    lb, off = divmod(l, block)
    return (lb * nranks + rank) * block + off


def global_to_local(g: int, block: int, nranks: int) -> Tuple[int, int]:
    b, off = divmod(g, block)
    return b % nranks, (b // nranks) * block + off


def global_to_ij(g: int, S: int, mode: int, rows: int = 0) -> Tuple[int, int]:
    if mode == _lib.PAIRS_FULL:
        return divmod(g, S)
    if mode == _lib.PAIRS_RECT:  # rows 0..rows-1 against columns rows..S-1
        i, jp = divmod(g, S - rows)
        return i, rows + jp
    i = 0
    # rows before i hold i*(2S-i-1)/2 entries
    lo, hi = 0, S - 2
    while lo < hi:
        mid = (lo + hi + 1) // 2
        if mid * (2 * S - mid - 1) // 2 <= g:
            lo = mid
        else:
            hi = mid - 1
    i = lo
    return i, g - i * (2 * S - i - 1) // 2 + i + 1


def row_start(i: int, S: int, mode: int, rows: int = 0) -> int:
    """Linear index of the first problem of matrix row i (i == number of rows: one past the end)."""
    if mode == _lib.PAIRS_RECT:
        return i * (S - rows)
    return i * S if mode == _lib.PAIRS_FULL else i * (2 * S - i - 1) // 2


def band_rows(S: int, mode: int, n_bands: int, rows: int = 0) -> List[int]:
    """Row boundaries r_0 = 0 < r_1 < ... < r_B = R of bands holding about the same number of problems
    (upper-triangle rows get shorter, so later bands take more rows).  R = S, or `rows` in PAIRS_RECT."""
    total = ops.n_pairs(S, mode, rows)
    R = rows if mode == _lib.PAIRS_RECT else S
    n_bands = max(1, min(n_bands, R))
    edges = [0]
    for b in range(1, n_bands):
        target = total * b // n_bands
        lo, hi = edges[-1], R
        while lo < hi:  # first row whose start is >= target
            mid = (lo + hi) // 2
            if row_start(mid, S, mode, rows) >= target:
                hi = mid
            else:
                lo = mid + 1
        if lo > edges[-1] and lo < R:
            edges.append(lo)
    edges.append(R)
    return edges


def sinkhorn_form_changes(S_a: int, S_b: int, K: int) -> bool:
    """True when pilot_sinkhorn_pairs picks different solvers for cohorts of S_a and of S_b samples: for K <= 16
    the warp form runs when S*S < 200 000 and the DMMA panels otherwise (sinkhorn.cu).  The two agree within a few
    ulp but not bit for bit, so a matrix solved at one size is not a block of the square at the other."""
    return K <= 16 and (S_a * S_a < 200_000) != (S_b * S_b < 200_000)


def choose_block(total: int, nranks: int) -> int:
    """>= 4 blocks per rank when possible, at most 4096 problems per block."""
    if nranks <= 1:
        return max(1, total)
    return max(1, min(4096, -(-total // (nranks * 4))))


def gather_packed(local: torch.Tensor, chunk: int, group=None) -> torch.Tensor:
    """All-gather equally padded per-rank chunks -> [nranks * chunk]."""
    nranks, _ = world(group)
    if nranks == 1:
        return local
    assert local.numel() == chunk
    out = torch.empty((nranks * chunk,), dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, local, group=group)
    return out


def cost_is_symmetric_metric_like(cost) -> bool:
    """True when mirroring the exact-EMD matrix is parity-safe: cost symmetric, zero
    diagonal and non-negative, so EMD(a,b) == EMD(b,a) and EMD(a,a) == 0.  A host array is
    checked on the host; a device tensor costs ONE read-back."""
    if isinstance(cost, np.ndarray):
        return bool((cost == cost.T).all() and (np.diagonal(cost) == 0).all() and (cost >= 0).all())
    c = cost
    return bool(((c == c.t()).all() & (torch.diagonal(c) == 0).all() & (c >= 0).all()).item())


def _mode_for(regularized, cost_norm, symmetric: Optional[bool], rect: bool = False) -> Tuple[bool, int]:
    exact = isinstance(regularized, str) and regularized == "unreg"
    if rect:  # a block between two sample sets holds no mirrored pair, whatever the cost
        return exact, _lib.PAIRS_RECT
    if exact:
        if symmetric is None:
            symmetric = cost_is_symmetric_metric_like(cost_norm)
        return True, (_lib.PAIRS_UPPER if symmetric else _lib.PAIRS_FULL)
    return False, _lib.PAIRS_FULL  # Sinkhorn is neither symmetric nor zero on the diagonal (SURVEY fact 6)


def plan_rule(rows, cols, S: int, mirrored: bool) -> Tuple[np.ndarray, np.ndarray, np.ndarray, np.ndarray]:
    """Which problem produced each entry (rows[l], cols[l]) of a matrix: (pair_a, pair_b, transpose, diagonal).
    Without mirroring the entry is the problem (i, j).  A mirrored matrix (exact EMD, symmetric metric-like cost)
    holds (i, j) for i < j, the transpose of (j, i) for i > j, and an exact 0 on the diagonal: there the plan is
    diag(props[i]), which is optimal for a symmetric, non-negative, zero-diagonal cost, and nothing is solved.
    An index outside [0, S) is passed through, so that the solver reports it (NaN)."""
    i = np.asarray(rows, dtype=np.int64).reshape(-1)
    j = np.asarray(cols, dtype=np.int64).reshape(-1)
    if i.shape != j.shape:
        raise ValueError(f"{i.size} row indices and {j.size} column indices")
    if not mirrored:
        none = np.zeros(i.shape, dtype=bool)
        return i, j, none, none
    flip = i > j
    diag = (i == j) & (i >= 0) & (i < S)
    return np.where(flip, j, i), np.where(flip, i, j), flip, diag


def entry_plans(props: torch.Tensor, cost_norm: torch.Tensor, rows, cols, regularized="unreg", reg: float = 0.1,
                symmetric: Optional[bool] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Transport plans behind the entries (rows[l], cols[l]) of ``all_pairs(props, cost_norm, regularized, reg,
    symmetric=symmetric)``: (plans [n, K, K], costs [n]) on the device, plans[l, r, c] the mass that row sample's
    type r sends to column sample's type c.  Each plan is that of the problem that produced the entry (plan_rule),
    so an exact-EMD cost equals the matrix entry bit for bit; a Sinkhorn plan comes from the reference form
    (ops.sinkhorn_plans), within 1e-12 relative of the entry."""
    S, K = props.shape
    exact, mode = _mode_for(regularized, cost_norm, symmetric)
    pa, pb, flip, diag = plan_rule(rows, cols, S, exact and mode == _lib.PAIRS_UPPER)
    n = pa.size
    dev = props.device
    plans = torch.empty((n, K, K), dtype=torch.float64, device=dev)
    costs = torch.empty((n,), dtype=torch.float64, device=dev)
    solve = np.nonzero(~diag)[0]
    if solve.size:
        if exact:
            g, c = ops.emd_plans(props, cost_norm, pa[solve], pb[solve])
        else:
            g, c = ops.sinkhorn_plans(props, cost_norm, reg, pa[solve], pb[solve])
        f = torch.from_numpy(flip[solve]).to(dev).view(-1, 1, 1)
        sel = torch.from_numpy(solve).to(dev)
        plans[sel] = torch.where(f, g.transpose(1, 2), g)
        costs[sel] = c
    d = np.nonzero(diag)[0]
    if d.size:
        sel = torch.from_numpy(d).to(dev)
        plans[sel] = torch.diag_embed(props[torch.from_numpy(pa[d]).to(dev)])
        costs[sel] = 0.0
    return plans, costs


def _solve_window(props, cost_norm, exact: bool, reg: float, mode: int, first: int, total: int, nranks: int,
                  rank: int, group, algo: int, precision, dense: torch.Tensor, want_info: bool = False,
                  marks: Optional[list] = None, rows: int = 0):
    """Solve the window [first, first + total) of the pair space over the ranks, all-gather, unpack into
    `dense` (rows: S_a of PAIRS_RECT).  Everything is asynchronous on the current stream."""
    S = props.shape[0]
    block = choose_block(total, nranks)
    rng = PairRange(total=total, block=block, nranks=nranks, rank=rank, mode=mode, rows=rows, first=first)
    chunk = max(1, range_count(total, block, nranks, 0))  # rank 0 always holds the largest share
    packed = torch.zeros((chunk,), dtype=torch.float64, device=props.device) if nranks > 1 else None

    def mark(name):
        if marks is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            marks.append((name, ev))

    mark("start")
    if exact:
        res = ops.emd_pairs(props, cost_norm, rng, want_info=want_info, out=packed, precision=precision)
    else:
        res = ops.sinkhorn_pairs(props, cost_norm, reg, rng, algo=algo, want_info=want_info, out=packed,
                                 precision=precision)
    mark("solve")
    info = None
    if want_info:
        info = res[1:]
        res = res[0]
    if nranks > 1:
        gathered = gather_packed(packed, chunk, group)
    else:
        gathered = res
        chunk = max(1, total)
    mark("gather")
    ops.unpack_pairs(gathered.contiguous(), chunk, S, rng, 0.0, dense=dense)
    mark("unpack")
    return info


def all_pairs(props: torch.Tensor, cost_norm: torch.Tensor, regularized="unreg", reg: float = 0.1,
              group=None, algo: int = 0, symmetric: Optional[bool] = None, want_info: bool = False,
              precision="f64", single_rank: bool = False, marks: Optional[list] = None, rows: int = 0):
    """Dense S x S matrix EMD[i, j] = OT(props[i], props[j]) on every rank (device tensor).

    regularized == "unreg" -> exact EMD, anything else -> stabilised Sinkhorn
    (the string comparison is the reference's, Trajectory.py:507).
    single_rank=True solves everything on this rank, whatever the process group (parity checks).
    marks: optional list receiving (name, cuda event) pairs around solve / gather / unpack.
    rows > 0: only the rows x (S - rows) block of props[:rows] against props[rows:] (PAIRS_RECT).
    """
    S, K = props.shape
    nranks, rank = (1, 0) if single_rank else world(group)
    exact, mode = _mode_for(regularized, cost_norm, symmetric, rect=rows > 0)
    shape = (rows, S - rows) if rows > 0 else (S, S)
    total = ops.n_pairs(S, mode, rows)
    if total == 0:
        dense = torch.zeros(shape, dtype=torch.float64, device=props.device)
        return (dense, None) if want_info else dense
    dense = torch.empty(shape, dtype=torch.float64, device=props.device)
    info = _solve_window(props, cost_norm, exact, reg, mode, 0, total, nranks, rank, group, algo, precision, dense,
                         want_info, marks, rows)
    if want_info:
        return dense, info
    return dense


_copy_streams = {}


def _copy_stream(dev: torch.device) -> "torch.cuda.Stream":
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    if idx not in _copy_streams:
        _copy_streams[idx] = torch.cuda.Stream(device=dev)
    return _copy_streams[idx]


def all_pairs_host(props: torch.Tensor, cost_norm: torch.Tensor, regularized="unreg", reg: float = 0.1,
                   group=None, algo: int = 0, symmetric: Optional[bool] = None, precision="f64",
                   n_bands: Optional[int] = None, with_transpose: bool = False, rows: int = 0
                   ) -> Tuple[np.ndarray, Optional[np.ndarray]]:
    """The dense S x S matrix in HOST memory on every rank, and optionally an independent ndarray holding
    its transpose (the reference hands out the ndarray and a DataFrame of the transpose, Trajectory.py:518).

    The pair space is cut into bands of whole matrix rows holding equal numbers of problems.  All bands are
    enqueued at once (solve -> all-gather -> unpack, asynchronous); the host then walks the bands and copies
    band b's rows out on a copy stream as soon as its unpack has finished, i.e. while the kernels of the
    later bands run.  With the upper-triangle mode a band's rows are final once it is unpacked (their
    left part was mirrored in by the earlier bands) and the transpose is the matrix itself; otherwise the
    transpose is formed on the device after the last band and copied out then.
    rows > 0: only the rows x (S - rows) block of props[:rows] against props[rows:] (PAIRS_RECT); the bands
    are rows of the block, and with_transpose does not apply.
    """
    S, K = props.shape
    nranks, rank = world(group)
    if rows > 0 and with_transpose:
        raise ValueError("all_pairs_host: with_transpose is not available for a block (rows > 0)")
    exact, mode = _mode_for(regularized, cost_norm, symmetric, rect=rows > 0)
    shape = (rows, S - rows) if rows > 0 else (S, S)
    total = ops.n_pairs(S, mode, rows)
    out = np.empty(shape, dtype=np.float64)
    out_T = np.empty((S, S), dtype=np.float64) if with_transpose else None
    if S == 0 or total == 0:
        out[...] = 0.0
        if out_T is not None:
            out_T[...] = 0.0
        return out, out_T
    dev = props.device
    if n_bands is None:
        # small matrices: one band (the copy takes microseconds); big ones: ~256 MB of rows per band
        n_bands = max(1, min(64, (shape[0] * shape[1] * 8) >> 28))
    edges = band_rows(S, mode, n_bands, rows)
    dense = torch.empty(shape, dtype=torch.float64, device=dev)
    main = torch.cuda.current_stream(dev)
    side = _copy_stream(dev)
    done = []
    for b in range(len(edges) - 1):
        first = row_start(edges[b], S, mode, rows)
        cnt = row_start(edges[b + 1], S, mode, rows) - first
        if cnt > 0:
            _solve_window(props, cost_norm, exact, reg, mode, first, cnt, nranks, rank, group, algo, precision, dense,
                          rows=rows)
        else:  # the last row of the upper triangle holds no pair: only its diagonal entry
            dense[edges[b]:edges[b + 1]].diagonal(offset=edges[b]).zero_()
        ev = torch.cuda.Event()
        ev.record(main)
        done.append(ev)
    dense_T = None
    if with_transpose and mode == _lib.PAIRS_FULL:
        dense_T = dense.t().contiguous()
        ev = torch.cuda.Event()
        ev.record(main)
        done.append(ev)
    host, host_T = torch.from_numpy(out), (torch.from_numpy(out_T) if with_transpose else None)
    with torch.cuda.stream(side):
        for b in range(len(edges) - 1):
            side.wait_event(done[b])
            r0, r1 = edges[b], edges[b + 1]
            host[r0:r1].copy_(dense[r0:r1])  # pageable destination: returns when the rows have arrived
            if with_transpose and dense_T is None:
                host_T[r0:r1].copy_(dense[r0:r1])  # symmetric by construction (mirrored entries)
        if dense_T is not None:
            side.wait_event(done[-1])
            for r0 in range(0, S, 2048):
                host_T[r0:r0 + 2048].copy_(dense_T[r0:r0 + 2048])
            dense_T.record_stream(side)
    dense.record_stream(side)
    return out, out_T


def _concat(props_a: torch.Tensor, props_b: torch.Tensor) -> torch.Tensor:
    if props_a.shape[1] != props_b.shape[1]:
        raise ValueError(f"the two sample sets have {props_a.shape[1]} and {props_b.shape[1]} cell types")
    return torch.cat([props_a, props_b]).contiguous()


def cross_pairs(props_a: torch.Tensor, props_b: torch.Tensor, cost_norm: torch.Tensor, regularized="unreg",
                reg: float = 0.1, group=None, algo: int = 0, want_info: bool = False, precision="f64",
                single_rank: bool = False):
    """Dense S_a x S_b matrix D[i, j] = OT(props_a[i], props_b[j]) on every rank (device tensor): the RECT pair
    space over the concatenated sets, partitioned and all-gathered as in all_pairs.  Bit-identical to the same
    entries of all_pairs over torch.cat([props_a, props_b])."""
    S_a, S_b = props_a.shape[0], props_b.shape[0]
    if S_a == 0 or S_b == 0:
        dense = torch.zeros((S_a, S_b), dtype=torch.float64, device=props_a.device)
        return (dense, None) if want_info else dense
    return all_pairs(_concat(props_a, props_b), cost_norm, regularized, reg, group, algo, want_info=want_info,
                     precision=precision, single_rank=single_rank, rows=S_a)


def cross_pairs_host(props_a: torch.Tensor, props_b: torch.Tensor, cost_norm: torch.Tensor, regularized="unreg",
                     reg: float = 0.1, group=None, algo: int = 0, precision="f64",
                     n_bands: Optional[int] = None) -> np.ndarray:
    """cross_pairs with the result in HOST memory, through the band pipeline of all_pairs_host."""
    S_a, S_b = props_a.shape[0], props_b.shape[0]
    if S_a == 0 or S_b == 0:
        return np.zeros((S_a, S_b), dtype=np.float64)
    out, _ = all_pairs_host(_concat(props_a, props_b), cost_norm, regularized, reg, group, algo, precision=precision,
                            n_bands=n_bands, rows=S_a)
    return out


def extend_pairs(props_old: torch.Tensor, props_new: torch.Tensor, cost_norm: torch.Tensor, regularized="unreg",
                 reg: float = 0.1, group=None, algo: int = 0, symmetric: Optional[bool] = None, precision="f64",
                 single_rank: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """What the square over S = S_old + S_new samples holds beyond its S_old x S_old corner, solving only
    those problems: (old_new [S_old, S_new], new_rows [S_new, S]) on every rank (device tensors), the rows
    S_old.. and the columns S_old.. of rows 0..S_old-1 of all_pairs(torch.cat([props_old, props_new])),
    bit for bit.

    old x new is the RECT block.  The rows of the new samples are the window of the square's own pair space
    that holds them, over the concatenated samples, so every problem runs as the square runs it.  Where the
    square mirrors its upper triangle (exact EMD, symmetric cost) that window holds new x new only, and
    new x old is the transposed old x new block."""
    S_old, S_new = props_old.shape[0], props_new.shape[0]
    props = _concat(props_old, props_new)
    S = S_old + S_new
    nranks, rank = (1, 0) if single_rank else world(group)
    exact, mode = _mode_for(regularized, cost_norm, symmetric)
    old_new = cross_pairs(props_old, props_new, cost_norm, regularized, reg, group, algo, precision=precision,
                          single_rank=single_rank)
    # unpack addresses the window's entries in the S x S matrix; only rows S_old.. are read back
    dense = torch.empty((S, S), dtype=torch.float64, device=props.device)
    first = row_start(S_old, S, mode)
    total = ops.n_pairs(S, mode) - first
    if total > 0:
        _solve_window(props, cost_norm, exact, reg, mode, first, total, nranks, rank, group, algo, precision, dense)
    new_rows = dense[S_old:]
    if mode == _lib.PAIRS_UPPER:
        new_rows[:, :S_old] = old_new.t()
        new_rows[:, S_old:].diagonal().zero_()  # unpack writes it too, but not when one new sample leaves no pair
    return old_new, new_rows
