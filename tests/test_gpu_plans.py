"""GPU checks of the transport plans (pilot_emd_plans, pilot_sinkhorn_plans and the layers above them).  The contract:
an exact-EMD plan matches the oracle's plan and is a feasible basis whose cost equals the distance-matrix entry bit for
bit; a Sinkhorn plan matches POT's reference statement, with identical iteration and absorption counts and a cost
bit-identical to the reference-form pair solver; plans do not depend on where a problem sits in the list."""
import numpy as np
import pytest
import torch

from oracle import pilot_oracle as po
from pilot_b200 import _lib, ops, pairs, synth, tl

pytestmark = pytest.mark.gpu


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def bits(x):
    return np.ascontiguousarray(x).view(np.int64)


def asym_cost(M, seed):
    A = M + 0.3 * np.triu(np.random.default_rng(seed).random(M.shape), 1)
    return A / A.max()


def some_pairs(S, n, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, S, size=n), rng.integers(0, S, size=n)


# ---------------- exact EMD ----------------
@pytest.mark.parametrize("K", [2, 10, 32, 33, 64, 65, 128, 256])
def test_emd_plans_match_the_oracle(K):
    S = 12
    P, M = synth.make_pairs(S, K, seed=1000 + K)
    pa, pb = some_pairs(S, 10, K)
    plans, out, status = ops.emd_plans(dev(P), dev(M), pa, pb, want_info=True)
    plans, out, status = plans.cpu().numpy(), out.cpu().numpy(), status.cpu().numpy()
    assert (status == _lib.ST_CONVERGED).all()
    for l, (i, j) in enumerate(zip(pa, pb)):
        a, b = P[i], P[j]
        G = plans[l]
        want, _, code = po.emd_plan(a, b, M)
        np.testing.assert_allclose(G, want, rtol=0, atol=1e-12)
        assert (G >= 0).all() and np.count_nonzero(G) <= 2 * K - 1
        np.testing.assert_allclose(G.sum(axis=1), a, rtol=0, atol=1e-13)
        np.testing.assert_allclose(G.sum(axis=0), b * a.sum() / b.sum(), rtol=0, atol=1e-13)
        np.testing.assert_allclose(np.sum(M * G), out[l], rtol=1e-14, atol=0)


@pytest.mark.parametrize("K", [24, 100])
def test_emd_plan_costs_equal_the_mirrored_matrix(K):
    """Symmetric cost: all_pairs solves the upper triangle and mirrors it.  i < j is solved, i > j is the
    transposed plan of (j, i), the diagonal is diag(a) with cost 0.0 -- and every cost is the entry's bits."""
    S = 16
    P, M = synth.make_pairs(S, K, seed=1100 + K)
    assert pairs.cost_is_symmetric_metric_like(M)
    D = pairs.all_pairs(dev(P), dev(M), "unreg", single_rank=True).cpu().numpy()
    rows, cols = np.meshgrid(np.arange(S), np.arange(S), indexing="ij")
    rows, cols = rows.ravel(), cols.ravel()
    plans, costs = pairs.entry_plans(dev(P), dev(M), rows, cols, "unreg")
    plans, costs = plans.cpu().numpy(), costs.cpu().numpy()
    assert np.array_equal(bits(costs), bits(D[rows, cols]))
    G = plans.reshape(S, S, K, K)
    for i in range(S):
        assert np.array_equal(G[i, i], np.diag(P[i])) and costs[i * S + i] == 0.0
        for j in range(i + 1, S):
            assert np.array_equal(G[j, i], G[i, j].T)
    # the solved problems are (i, j), i < j, as given
    up = rows < cols
    direct, _ = ops.emd_plans(dev(P), dev(M), rows[up], cols[up])
    assert np.array_equal(bits(plans[up]), bits(direct.cpu().numpy()))


@pytest.mark.parametrize("K", [24, 100])
def test_emd_plan_costs_equal_the_full_matrix_for_an_asymmetric_cost(K):
    S = 14
    P, M = synth.make_pairs(S, K, seed=1200 + K)
    M = asym_cost(M, K)
    D = pairs.all_pairs(dev(P), dev(M), "unreg", single_rank=True).cpu().numpy()
    rows, cols = some_pairs(S, 40, K)
    rows[:3] = cols[:3]  # diagonal entries are solved too: the matrix does not mirror
    plans, costs = pairs.entry_plans(dev(P), dev(M), rows, cols, "unreg")
    assert np.array_equal(bits(costs.cpu().numpy()), bits(D[rows, cols]))
    direct, _ = ops.emd_plans(dev(P), dev(M), rows, cols)
    assert np.array_equal(bits(plans.cpu().numpy()), bits(direct.cpu().numpy()))


def _reps(P, prefix, start=0):
    return {f"{prefix}{start + i}": P[i] for i in range(P.shape[0])}


@pytest.mark.parametrize("regularized", ["unreg", "reg"])
@pytest.mark.parametrize("K", [24, 100])
def test_wasserstein_plans_follow_wasserstein_d_and_cross(K, regularized):
    P, M = synth.make_pairs(20, K, seed=1300 + K)
    a, b = _reps(P[:12], "a"), _reps(P[12:], "b")
    # one set: the plans follow wasserstein_d (mirrored under "unreg")
    D, _ = tl.wasserstein_d(a, M, regularized, 0.1)
    ids = list(a)
    prs = [(ids[i], ids[j]) for i, j in ((0, 5), (5, 0), (3, 3), (11, 2), (2, 11))]
    plans, costs = tl.wasserstein_plans(a, M, prs, regularized, 0.1)
    want = np.array([D[ids.index(x), ids.index(y)] for x, y in prs])
    if regularized == "unreg":
        assert np.array_equal(bits(costs), bits(want))
    else:
        np.testing.assert_allclose(costs, want, rtol=1e-12, atol=0)
    np.testing.assert_allclose(np.einsum("nrc,rc->n", plans, M), costs, rtol=1e-13, atol=1e-300)
    # two sets: the plans follow wasserstein_d_cross (never mirrored)
    Dx, _ = tl.wasserstein_d_cross(a, b, M, regularized, 0.1)
    ib = list(b)
    prs = [(ids[i], ib[j]) for i, j in ((0, 0), (11, 7), (4, 2), (4, 3))]
    plans, costs = tl.wasserstein_plans(a, M, prs, regularized, 0.1, Clu_rep_b=b)
    want = np.array([Dx[ids.index(x), ib.index(y)] for x, y in prs])
    if regularized == "unreg":
        assert np.array_equal(bits(costs), bits(want))
    else:
        np.testing.assert_allclose(costs, want, rtol=1e-12, atol=0)


def test_transport_plan_equals_the_emd_entry():
    X, obs = synth.make_cells(20_000, 12, 9, 10, seed=77)
    adata = synth.FakeAnnData(obs, obsm={"X_PCA": X})
    tl.wasserstein_distance(adata, regularized="unreg")
    ids = list(adata.uns["proportions"])
    E = adata.uns["EMD"]
    cost_df = adata.uns["cost"]
    for i, j in ((0, 1), (1, 0), (4, 4), (9, 3)):
        frame, c = tl.transport_plan(adata, ids[i], ids[j])
        assert bits(np.array([c]))[0] == bits(np.array([E[i, j]]))[0]
        assert frame.index.equals(cost_df.index) and frame.columns.equals(cost_df.columns)
        G = frame.to_numpy()
        np.testing.assert_allclose(G.sum(axis=1), adata.uns["proportions"][ids[i]], rtol=0, atol=1e-13)
        np.testing.assert_allclose(G.sum(axis=0), adata.uns["proportions"][ids[j]], rtol=0, atol=1e-13)
        C = cost_df.to_numpy()
        np.testing.assert_allclose(np.sum(C / C.max() * G), c, rtol=1e-13, atol=1e-300)


# ---------------- Sinkhorn ----------------
@pytest.mark.parametrize("reg", [0.1, 0.01])
@pytest.mark.parametrize("K", [10, 40, 64, 100, 200, 256])
def test_sinkhorn_plans_match_the_oracle(K, reg):
    S = 6
    P, M = synth.make_pairs(S, K, seed=1400 + K)
    pa, pb = some_pairs(S, 4, K + 1)
    plans, out, iters, absn, status = ops.sinkhorn_plans(dev(P), dev(M), reg, pa, pb, want_info=True)
    plans, out = plans.cpu().numpy(), out.cpu().numpy()
    iters, absn, status = iters.cpu().numpy(), absn.cpu().numpy(), status.cpu().numpy()
    for l, (i, j) in enumerate(zip(pa, pb)):
        G, info = po.sinkhorn_stabilized_np(P[i], P[j], M, reg, return_info=True)
        np.testing.assert_allclose(plans[l], G, rtol=0, atol=1e-12 * G.max())
        assert (iters[l], absn[l], status[l]) == (info["iters"], info["absorptions"], info["status"])
    # the cost: bit-identical to the reference-form pair solver, within 1e-12 of the default solvers' matrix
    Pd, Md = dev(P), dev(M)
    ref = ops.sinkhorn_pairs(Pd, Md, reg, ops.make_range(S * S, _lib.PAIRS_FULL), algo=1).cpu().numpy()
    assert np.array_equal(bits(out), bits(ref[pa * S + pb]))
    D = pairs.all_pairs(Pd, Md, "reg", reg, single_rank=True).cpu().numpy()
    np.testing.assert_allclose(out, D[pa, pb], rtol=1e-12, atol=0)
    # the plan sums, in the kernel's order, to the cost
    np.testing.assert_allclose(np.einsum("nrc,rc->n", plans, M), out, rtol=1e-13, atol=0)


def test_sinkhorn_reaches_absorptions_and_the_iteration_cap():
    """reg 0.01 at these sizes absorbs and runs into the 1000-iteration cap on some problems (so the two tests above
    cover both); asserted here so that a change of the inputs cannot silently drop that coverage."""
    hit_cap = absorbed = False
    for K in (40, 64, 100):
        P, M = synth.make_pairs(6, K, seed=1400 + K)
        pa, pb = some_pairs(6, 4, K + 1)
        _, _, iters, absn, _ = ops.sinkhorn_plans(dev(P), dev(M), 0.01, pa, pb, want_info=True)
        hit_cap |= bool((iters.cpu().numpy() == 1000).any())
        absorbed |= bool((absn.cpu().numpy() > 0).any())
    assert absorbed and hit_cap


# ---------------- reproducibility, refilled slots, bad indices ----------------
@pytest.mark.parametrize("kind,K,n", [("emd", 32, 20_000), ("emd", 64, 20_000), ("emd", 128, 10_000),
                                      ("sinkhorn", 64, 4_000), ("sinkhorn", 256, 600)])
def test_plans_do_not_depend_on_the_list(kind, K, n):
    """A list of at least 4x the warps (EMD: 32 per SM; general kernel: 16) or CTAs (Sinkhorn: the occupancy of
    the reference form, one per SM at K = 256) resident at once, so that most problems run in refilled slots.
    The same problem gives the same plan bytes alone and inside the list, and two runs are byte-identical."""
    S = 300
    P, M = synth.make_pairs(S, K, seed=1500 + K)
    Pd, Md = dev(P), dev(M)
    pa, pb = some_pairs(S, n, K)

    def run(a, b):
        g, c = ops.emd_plans(Pd, Md, a, b) if kind == "emd" else ops.sinkhorn_plans(Pd, Md, 0.1, a, b)
        return g.cpu().numpy(), c.cpu().numpy()

    g1, c1 = run(pa, pb)
    g2, c2 = run(pa, pb)
    assert g1.tobytes() == g2.tobytes() and c1.tobytes() == c2.tobytes()
    for l in (0, n // 2, n - 1):
        ga, ca = run(pa[l:l + 1], pb[l:l + 1])
        assert ga[0].tobytes() == g1[l].tobytes() and ca[0].tobytes() == c1[l].tobytes()


@pytest.mark.parametrize("kind,K", [("emd", 10), ("emd", 100), ("sinkhorn", 10), ("sinkhorn", 200)])
def test_out_of_range_pair_indices_give_nan(kind, K):
    S = 5
    P, M = synth.make_pairs(S, K, seed=1600 + K)
    pa = np.array([0, -1, 2, S, 1, 2 ** 31 - 1])
    pb = np.array([1, 2, -7, 0, S + 3, 4])
    if kind == "emd":
        g, c, st = ops.emd_plans(dev(P), dev(M), pa, pb, want_info=True)
    else:
        g, c, _, _, st = ops.sinkhorn_plans(dev(P), dev(M), 0.1, pa, pb, want_info=True)
    g, c, st = g.cpu().numpy(), c.cpu().numpy(), st.cpu().numpy()
    bad = np.array([False, True, True, True, True, True])
    assert np.isnan(c[bad]).all() and np.isnan(g[bad]).all()
    assert (st[bad] == _lib.ST_NUMERIC).all()
    assert np.isfinite(c[~bad]).all() and np.isfinite(g[~bad]).all() and st[0] == _lib.ST_CONVERGED
