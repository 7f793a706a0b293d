"""Every Sinkhorn solver against the oracle away from POT's default schedule (numItermax 1000, stopThr 1e-9,
tau 1e3, print_period 20), where each solver restates POT's loop with its own bookkeeping: the warp form, the DMMA
panels and their warp-form tail, the cluster panels, the FP32 kernel, the reference form and its plan variant.
Each schedule point decides one branch of that loop (table below).  The oracle is first pinned at these points
against its NumPy twin (CPU test at the top); the GPU tests then demand equal iteration counts, absorption counts
and status, and costs within 1e-9 relative, of every FP64 path.  The exact-EMD pivot cap is checked at the end."""
import functools

import numpy as np
import pytest
import torch

from oracle import pilot_oracle as po
from pilot_b200 import _lib, ops, pairs, synth

SK_RTOL = 1e-9
gpu = pytest.mark.gpu

# name: (num_iter_max, stop_thr, tau, check_every)                   what it decides
POINTS = {
    "A": (1000, 1e-9, 1e3, 1),      # a marginal check on every iteration
    "B": (1000, 1e-9, 1e3, 7),      # a check interval that does not divide the cap
    "C": (21, 1e-9, 1e3, 20),       # a pending check on the cap iteration
    "D": (37, 1e-9, 1e3, 20),       # the cap between two checks
    "E": (1, 1e-9, 1e3, 20),        # a single iteration
    "F": (60, 1e-9, 2.0, 3),        # an absorption on every iteration
    "G": (1000, 0.0, 1e300, 20),    # never converges, never absorbs (run at reg 0.002)
    "H": (1000, 1e-3, 1e3, 20),     # early convergence
    "I": (21, 1e-3, 1e3, 20),       # the check on the cap iteration converges: converged wins over the cap
}
ALL = sorted(POINTS)


def grid(Ks, points=ALL):
    """(point, K) cases.  F is left out at K = 2: there tau = 2 equals the value max(u, v) tends to after an
    absorption (v -> K), so every absorption test is a rounding tie and POT's own trajectory changes with a 1e-15
    change of the input (37 or 22 iterations), often without converging in 60 iterations."""
    return [(p, K) for p in points for K in Ks if not (p == "F" and K == 2)]


def point_kw(point):
    n, thr, tau, ce = POINTS[point]
    return dict(num_iter_max=n, stop_thr=thr, tau=tau, check_every=ce)


def point_reg(point):
    return 0.002 if point == "G" else 0.1


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def problems(K, S, seed, asym=False):
    P, M = synth.make_pairs(S, K, seed=seed)
    if K == 1:
        M = np.zeros((1, 1))
    if asym:
        M = np.random.default_rng(seed).random((K, K))
        M /= M.max()
    return P, M


def oracle_pairs(P, M, reg, point, idx):
    """(cost, iters, absorptions, status) of the C oracle for the flat pair indices idx (i * S + j)."""
    n, thr, tau, ce = POINTS[point]
    S = P.shape[0]
    res = np.empty((4, len(idx)))
    for l, g in enumerate(idx):
        c, info = po.sinkhorn2(P[g // S], P[g % S], M, reg, numItermax=n, stopThr=thr, tau=tau, return_info=True,
                               check_every=ce)
        res[:, l] = (c, info["iters"], info["absorptions"], info["status"])
    return res[0], res[1].astype(np.int32), res[2].astype(np.int32), res[3].astype(np.int32)


@functools.lru_cache(maxsize=None)
def oracle_case(K, S, seed, asym, point, reg):
    P, M = problems(K, S, seed, asym)
    return oracle_pairs(P, M, reg, point, np.arange(S * S))


def solve(P, M, reg, point, algo=0, precision="f64", rng=None):
    S = P.shape[0]
    rng = rng or ops.make_range(S * S, _lib.PAIRS_FULL)
    out, iters, absn, status = ops.sinkhorn_pairs(dev(P), dev(M), reg, rng, algo=algo, want_info=True,
                                                  precision=precision, **point_kw(point))
    got = tuple(t.cpu().numpy() for t in (out, iters, absn, status))
    return got, ops.sinkhorn_counters()


def assert_same_schedule(got, want):
    out, iters, absn, status = got
    wout, witers, wabs, wst = want
    np.testing.assert_array_equal(iters, witers, err_msg="iteration counts")
    np.testing.assert_array_equal(absn, wabs, err_msg="absorption counts")
    np.testing.assert_array_equal(status, wst, err_msg="status")
    np.testing.assert_allclose(out, wout, rtol=SK_RTOL, atol=1e-300)


def check_fp64_path(K, S, seed, asym, point, algo):
    reg = point_reg(point)
    P, M = problems(K, S, seed, asym)
    want = oracle_case(K, S, seed, asym, point, reg)
    got, ctr = solve(P, M, reg, point, algo=algo)
    if point == "G" and K > 1:
        # stop_thr 0 converges only on an error of exactly 0.0, which a problem (a, a) may reach in one iteration
        # by the luck of its rounding: the point is about the others (at K = 1 every problem is exact at once)
        off = ~np.eye(S, dtype=bool).ravel()
        got, want = tuple(g[off] for g in got), tuple(w[off] for w in want)
        assert (want[3] == _lib.ST_MAXITER).all()
    assert_same_schedule(got, want)
    if point == "I" and K > 1:
        assert (want[3][want[1] == POINTS["I"][0]] == _lib.ST_CONVERGED).any(), "no check converges on the cap"
    return ctr


# ---------------------------------------------------------------- the oracle at these points (CPU)
@pytest.mark.parametrize("reg", [0.1, 0.01])
@pytest.mark.parametrize("point", ALL)
def test_oracle_c_matches_numpy_at_schedule_points(point, reg):
    """The C oracle and its NumPy twin (print_period = check_every) agree on iterations, absorptions and status
    exactly and on the cost within 1e-12, at every schedule point (and point G also at its own reg 0.002)."""
    n, thr, tau, ce = POINTS[point]
    regs = (reg, 0.002) if point == "G" and reg == 0.01 else (reg,)
    P, M = synth.make_pairs(4, 20, seed=20)
    for r in regs:
        for i, j in ((0, 1), (2, 3), (1, 1), (3, 0)):
            c, ci = po.sinkhorn2(P[i], P[j], M, r, numItermax=n, stopThr=thr, tau=tau, return_info=True,
                                 check_every=ce)
            G, ni = po.sinkhorn_stabilized_np(P[i], P[j], M, r, numItermax=n, tau=tau, stopThr=thr,
                                              print_period=ce, return_info=True)
            assert (ci["iters"], ci["absorptions"], ci["status"]) == (ni["iters"], ni["absorptions"], ni["status"])
            assert abs(c - np.sum(M * G)) <= 1e-12 * abs(c)
            assert ci["iters"] <= n and (ci["status"] != _lib.ST_MAXITER or ci["iters"] == n)


def test_oracle_check_every_default_is_pots():
    P, M = synth.make_pairs(2, 12, seed=3)
    assert po.sinkhorn2(P[0], P[1], M, 0.1, return_info=True) == \
        po.sinkhorn2(P[0], P[1], M, 0.1, return_info=True, check_every=20)
    c, info = po.sinkhorn2(P[0], P[1], M, 0.1, return_info=True, check_every=7)
    assert info["status"] == _lib.ST_CONVERGED and (info["iters"] - 1) % 7 == 0


# ---------------------------------------------------------------- FP64 paths
@gpu
@pytest.mark.parametrize("point,K", grid([2, 16, 17, 32]))
def test_warp_form(point, K):
    """algo 0 with a symmetric cost and S * S < 200 000: one warp per problem with K0 in registers."""
    ctr = check_fp64_path(K, 4, 100 + K, False, point, 0)
    assert ctr["n_redo"] == 0, "a problem left the warp form for the reference form"


@gpu
@pytest.mark.parametrize("point,K,algo", [(p, K, 3) for p, K in grid([1, 2, 3, 16, 40, 64])] +
                         [(p, 64, 0) for p in ALL])
def test_dmma_panels(point, K, algo):
    ctr = check_fp64_path(K, 4, 200 + K, False, point, algo)
    assert ctr["n_redo"] == 0, "a problem left the panels for the reference form"


@gpu
@pytest.mark.parametrize("asym", [False, True])
@pytest.mark.parametrize("K", [65, 128, 256])
@pytest.mark.parametrize("point", ALL)
def test_cluster_panels(point, K, asym):
    ctr = check_fp64_path(K, 4, 300 + K, asym, point, 0)
    assert ctr["n_redo"] == 0, "a problem left the cluster panels for the reference form"


@gpu
@pytest.mark.parametrize("K", [40, 200])
@pytest.mark.parametrize("point", ALL)
def test_reference_form(point, K):
    check_fp64_path(K, 4, 400 + K, False, point, 1)


@gpu
@pytest.mark.parametrize("K,point,reg", [(64, "A", 0.1), (64, "B", 0.1), (64, "H", 0.1), (64, "B", 0.02),
                                         (12, "B", 0.1), (40, "A", 0.1)])
def test_panel_tail_handover(K, point, reg):
    """A batch large enough that the panels hand stragglers to the warp-form tail kernel mid-schedule (the
    n_tail counter proves it): every problem against the reference form, two rows against the oracle.  At reg
    0.02 the handed-over problems carry absorptions (rea / reb and the hasabs flag)."""
    S = 100
    P, M = problems(K, S, 500 + K)
    got, ctr = solve(P, M, reg, point, algo=3)
    assert ctr["n_tail"] > 0, "no problem was handed to the tail kernel"
    assert ctr["n_redo"] == 0
    ref, _ = solve(P, M, reg, point, algo=1)
    assert_same_schedule(got, ref)
    if reg < 0.1:
        assert got[2].max() > 0
    rows = np.arange(2 * S)
    assert_same_schedule(tuple(g[rows] for g in got), oracle_pairs(P, M, reg, point, rows))


@gpu
@pytest.mark.parametrize("K", [40, 64])
@pytest.mark.parametrize("point", ["B", "F"])
def test_panels_bit_reproducible(point, K):
    """Repeated runs of the panel path, and a 3-rank partition of its pair space, give the same bits."""
    S, reg = 40, point_reg(point)
    P, M = problems(K, S, 600 + K)
    (ref, *_), _ = solve(P, M, reg, point, algo=3)
    (again, *_), _ = solve(P, M, reg, point, algo=3)
    assert np.array_equal(ref, again)
    got = np.empty_like(ref)
    nranks, block = 3, 17
    for rank in range(nranks):
        r = _lib.PairRange(total=S * S, block=block, nranks=nranks, rank=rank, mode=_lib.PAIRS_FULL, reserved=0)
        (out, *_), _ = solve(P, M, reg, point, algo=3, rng=r)
        got[[pairs.local_to_global(l, block, nranks, rank) for l in range(len(out))]] = out
    assert np.array_equal(got, ref)
    rows = np.arange(S)
    np.testing.assert_allclose(ref[rows], oracle_pairs(P, M, reg, point, rows)[0], rtol=SK_RTOL)


# ---------------------------------------------------------------- FP32
@gpu
@pytest.mark.parametrize("point,K", grid([2, 3, 17, 31, 33, 63, 64]))
def test_fp32_kernel(point, K):
    """Within 1e-4 of the FP64 oracle at the same schedule; the float stop floor (5e-7) is the only allowed
    source of a different iteration count, so every count is a check iteration or the cap."""
    n, thr, tau, ce = POINTS[point]
    reg, S = point_reg(point), 4
    P, M = problems(K, S, 700 + K)
    wout, witers, wabs, wst = oracle_case(K, S, 700 + K, False, point, reg)
    (out, iters, absn, status), ctr = solve(P, M, reg, point, precision="f32")
    np.testing.assert_allclose(out, wout, rtol=1e-4, atol=1e-7)
    assert (iters >= 1).all() and (iters <= n).all()
    assert (((iters - 1) % ce == 0) | (iters == n)).all()
    assert np.isin(status, [_lib.ST_CONVERGED, _lib.ST_MAXITER]).all()
    assert (status[iters < n] == _lib.ST_CONVERGED).all()
    if thr >= 5e-7:
        np.testing.assert_array_equal(iters, witers)
        np.testing.assert_array_equal(status, wst)
    else:
        # the float floor may stop a problem earlier than the FP64 schedule, never later (at G: stop_thr 0
        # never converges in FP64, while the float kernel stops at an error below 5e-7)
        assert (iters <= witers).all()
    if point not in ("F", "G"):
        assert ctr["n_redo"] == 0, "a problem left the FP32 kernel for the FP64 reference form"


# ---------------------------------------------------------------- plans
@gpu
@pytest.mark.parametrize("K", [12, 100])
@pytest.mark.parametrize("point", ["B", "C", "F", "I"])
def test_sinkhorn_plans_at_schedule_points(point, K):
    S, reg = 5, point_reg(point)
    P, M = problems(K, S, 800 + K)
    rng_ = np.random.default_rng(K)
    pa, pb = rng_.integers(0, S, 6), rng_.integers(0, S, 6)
    plans, out, iters, absn, status = ops.sinkhorn_plans(dev(P), dev(M), reg, pa, pb, want_info=True,
                                                         **point_kw(point))
    plans, out = plans.cpu().numpy(), out.cpu().numpy()
    iters, absn, status = iters.cpu().numpy(), absn.cpu().numpy(), status.cpu().numpy()
    n, thr, tau, ce = POINTS[point]
    for l, (i, j) in enumerate(zip(pa, pb)):
        G, info = po.sinkhorn_stabilized_np(P[i], P[j], M, reg, numItermax=n, tau=tau, stopThr=thr,
                                            print_period=ce, return_info=True)
        np.testing.assert_allclose(plans[l], G, rtol=0, atol=1e-9 * G.max())
        assert (iters[l], absn[l], status[l]) == (info["iters"], info["absorptions"], info["status"])
    (ref, *_), _ = solve(P, M, reg, point, algo=1)
    assert np.array_equal(out.view(np.int64), ref[pa * S + pb].view(np.int64))


# ---------------------------------------------------------------- exact EMD: the pivot cap
@gpu
@pytest.mark.parametrize("K,precision", [(10, "f64"), (40, "f64"), (64, "f64"), (10, "f32"), (40, "f32"),
                                         (64, "f32")])
def test_emd_pivot_cap_bitmask_kernel(K, precision):
    """max_pivots = m stops a problem that needs more than m pivots with PILOT_ST_MAXITER and m + 1 in the pivot
    count (the entering arc of pivot m + 1 was found, not pivoted); every other problem is untouched, bit for bit.
    The start basis is feasible, so a stopped problem reports the cost of a feasible basis: never below the
    optimum, and its plan still has the marginals a and b."""
    S = 8
    P, M = synth.make_pairs(S, K, seed=900 + K)
    Pd, Md = dev(P), dev(M)
    rng = ops.make_range(S * S, _lib.PAIRS_FULL)
    free, fst, fpiv = (t.cpu().numpy() for t in ops.emd_pairs(Pd, Md, rng, want_info=True, precision=precision))
    assert (fst == _lib.ST_CONVERGED).all()
    want = po.emd_rows(P, M, 0, S).ravel()
    slack = 1e-12 if precision == "f64" else 1e-5
    caps = sorted({1, 5, max(1, int(np.median(fpiv)))})
    for m in caps:
        out, st, piv = (t.cpu().numpy() for t in ops.emd_pairs(Pd, Md, rng, max_pivots=m, want_info=True,
                                                               precision=precision))
        capped = fpiv > m
        assert capped.any()
        assert (st[capped] == _lib.ST_MAXITER).all() and (st[~capped] == _lib.ST_CONVERGED).all()
        assert (piv[capped] == m + 1).all() and np.array_equal(piv[~capped], fpiv[~capped])
        assert np.array_equal(out[~capped].view(np.int64), free[~capped].view(np.int64))
        assert (out[capped] >= want[capped] * (1 - slack)).all()
        if precision == "f64":
            ia, ib = np.divmod(np.arange(S * S), S)
            plans, pout, pst = (t.cpu().numpy() for t in ops.emd_plans(Pd, Md, ia, ib, max_pivots=m,
                                                                        want_info=True))
            np.testing.assert_array_equal(pst, st)
            assert np.array_equal(pout.view(np.int64), out.view(np.int64))
            assert (plans >= 0).all()
            for l in range(S * S):
                a, b = P[ia[l]], P[ib[l]]
                np.testing.assert_allclose(plans[l].sum(axis=1), a, rtol=0, atol=1e-13)
                np.testing.assert_allclose(plans[l].sum(axis=0), b * a.sum() / b.sum(), rtol=0, atol=1e-13)
                np.testing.assert_allclose(np.sum(M * plans[l]), out[l], rtol=1e-13, atol=0)


@gpu
@pytest.mark.parametrize("K", [100, 200])
def test_emd_pivot_cap_general_kernel(K):
    """The general network simplex (65..256 types) stops at max_pivots like the bit-mask kernel: PILOT_ST_MAXITER
    and m + 1 pivots exactly where the uncapped run needed more than m, the uncapped result bit for bit
    elsewhere.  It starts from POT's artificial big-M star, so a stopped problem may still route mass over
    artificial arcs; its cost is the real arcs' part only (finite, >= 0, and no bound on the optimum holds)."""
    S = 5
    P, M = synth.make_pairs(S, K, seed=950 + K)
    Pd, Md = dev(P), dev(M)
    rng = ops.make_range(S * S, _lib.PAIRS_FULL)
    free, fst, fpiv = (t.cpu().numpy() for t in ops.emd_pairs(Pd, Md, rng, want_info=True))
    assert (fst == _lib.ST_CONVERGED).all()
    for m in sorted({1, 5, max(1, int(np.median(fpiv)))}):
        out, st, piv = (t.cpu().numpy() for t in ops.emd_pairs(Pd, Md, rng, max_pivots=m, want_info=True))
        capped = fpiv > m
        assert capped.any()
        assert (st[capped] == _lib.ST_MAXITER).all() and (st[~capped] == _lib.ST_CONVERGED).all()
        assert (piv[capped] == m + 1).all() and np.array_equal(piv[~capped], fpiv[~capped])
        assert np.array_equal(out[~capped].view(np.int64), free[~capped].view(np.int64))
        assert np.isfinite(out).all() and (out >= 0).all()
