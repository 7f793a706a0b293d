"""CPU-side checks of the transport-plan feature: the argument checks of pilot_emd_plans / pilot_sinkhorn_plans, the
errors tl.wasserstein_plans raises before any device work, and the host statement of which problem produced a
matrix entry (pairs.plan_rule)."""
import numpy as np
import pytest

from pilot_b200 import _lib, pairs, tl

WS = 1 << 30  # large enough for any K: the checks below must fail on their own argument


def emd_plans(props=1, S=10, K=8, cost=1, pa=1, pb=1, n=4, plans=1, out=1, ws=1):
    return _lib.lib().pilot_emd_plans(props, S, K, cost, 0, pa, pb, n, plans, out, None, ws, WS, None)


def sinkhorn_plans(props=1, S=10, K=8, cost=1, pa=1, pb=1, n=4, plans=1, out=1, ws=1):
    return _lib.lib().pilot_sinkhorn_plans(props, S, K, cost, 0.1, 1000, 1e-9, 1e3, 20, pa, pb, n, plans, out, None,
                                           None, None, ws, WS, None)


def test_abi_version_is_4():
    assert _lib.ABI_VERSION == 4 and _lib.lib().pilot_abi_version() == 4


@pytest.mark.parametrize("entry", [emd_plans, sinkhorn_plans], ids=["emd", "sinkhorn"])
@pytest.mark.parametrize("kw,msg", [
    (dict(props=None), b"NULL pointer"), (dict(cost=None), b"NULL pointer"), (dict(pa=None), b"NULL pointer"),
    (dict(pb=None), b"NULL pointer"), (dict(plans=None), b"NULL pointer"), (dict(out=None), b"NULL pointer"),
    (dict(ws=None), b"NULL pointer"),
    (dict(S=0), b"S=0"), (dict(S=-3), b"S=-3"),
    (dict(K=0), b"K=0 outside"), (dict(K=257), b"K=257 outside"),
    (dict(n=-1), b"n=-1"),
])
def test_entry_points_reject_bad_arguments(entry, kw, msg):
    assert entry(**kw) < 0
    assert msg in _lib.lib().pilot_last_error()


@pytest.mark.parametrize("entry", [emd_plans, sinkhorn_plans], ids=["emd", "sinkhorn"])
def test_no_problems_is_a_no_op(entry):
    assert entry(n=0) == 0


def test_sinkhorn_plans_rejects_bad_parameters():
    L = _lib.lib()
    assert L.pilot_sinkhorn_plans(1, 10, 8, 1, 0.0, 1000, 1e-9, 1e3, 20, 1, 1, 4, 1, 1, None, None, None, 1, WS,
                                  None) < 0
    assert b"reg must be > 0" in L.pilot_last_error()
    assert L.pilot_sinkhorn_plans(1, 10, 8, 1, 0.1, 1000, 1e-9, 1e3, 0, 1, 1, 4, 1, 1, None, None, None, 1, WS,
                                  None) < 0
    assert b"iteration parameters" in L.pilot_last_error()


def test_workspace_too_small_is_rejected():
    L = _lib.lib()
    assert L.pilot_emd_plans(1, 10, 8, 1, 0, 1, 1, 4, 1, 1, None, 1, 16, None) < 0
    assert b"workspace" in L.pilot_last_error()
    assert L.pilot_sinkhorn_plans(1, 10, 8, 1, 0.1, 1000, 1e-9, 1e3, 20, 1, 1, 4, 1, 1, None, None, None, 1, 16,
                                  None) < 0
    assert b"workspace" in L.pilot_last_error()


# ---- tl.wasserstein_plans: errors before any device work ----
def _reps(n, K, seed, prefix):
    P = np.random.default_rng(seed).dirichlet(np.ones(K), size=n)
    return {f"{prefix}{i}": P[i] for i in range(n)}


def _cost(K):
    c = np.abs(np.subtract.outer(np.arange(K), np.arange(K))).astype(np.float64)
    return c / c.max()


@pytest.mark.parametrize("regularized", ["unreg", "reg"])
def test_unknown_ids_raise_key_error(regularized):
    a, b = _reps(3, 5, 0, "a"), _reps(3, 5, 1, "b")
    with pytest.raises(KeyError, match="zz"):
        tl.wasserstein_plans(a, _cost(5), [("a0", "a1"), ("a0", "zz")], regularized)
    with pytest.raises(KeyError, match="a1"):  # with Clu_rep_b, id_b is a key of Clu_rep_b
        tl.wasserstein_plans(a, _cost(5), [("a0", "a1")], regularized, Clu_rep_b=b)
    with pytest.raises(KeyError, match="b0"):
        tl.wasserstein_plans(a, _cost(5), [("b0", "b1")], regularized, Clu_rep_b=b)


def test_shape_errors_raise_value_error():
    a = _reps(3, 5, 0, "a")
    with pytest.raises(ValueError, match="cell types"):
        tl.wasserstein_plans(a, _cost(5), [("a0", "b0")], Clu_rep_b=_reps(3, 6, 1, "b"))
    with pytest.raises(ValueError, match="cost has shape"):
        tl.wasserstein_plans(a, _cost(4), [("a0", "a1")], regularized="reg")
    with pytest.raises(ValueError, match="cost has shape"):
        tl.wasserstein_plans(a, _cost(4), [("a0", "b0")], Clu_rep_b=_reps(3, 5, 1, "b"))


def test_unequal_masses_under_unreg_raise():
    a = _reps(3, 5, 0, "a")
    a["a2"] = 2.0 * a["a2"]
    with pytest.raises(AssertionError, match="same sum"):
        tl.wasserstein_plans(a, _cost(5), [("a0", "a1")])
    b = {k: 2.0 * v for k, v in _reps(3, 5, 1, "b").items()}
    with pytest.raises(AssertionError, match="same sum"):
        tl.wasserstein_plans(_reps(3, 5, 0, "a"), _cost(5), [("a0", "b0")], Clu_rep_b=b)


def test_empty_pair_list_returns_empty_arrays():
    plans, costs = tl.wasserstein_plans(_reps(3, 5, 0, "a"), _cost(5), [])
    assert plans.shape == (0, 5, 5) and costs.shape == (0,)
    plans, costs = tl.wasserstein_plans({}, _cost(5), [], Clu_rep_b={})
    assert plans.shape == (0, 5, 5) and costs.shape == (0,)


# ---- pairs.plan_rule: which problem produced an entry ----
def test_plan_rule_mirrored_matrix():
    rows = [0, 3, 2, 2, 4, 1, 7, -1]
    cols = [3, 0, 2, 4, 2, 1, 7, -1]
    pa, pb, flip, diag = pairs.plan_rule(rows, cols, S=5, mirrored=True)
    assert pa.tolist() == [0, 0, 2, 2, 2, 1, 7, -1]
    assert pb.tolist() == [3, 3, 2, 4, 4, 1, 7, -1]
    assert flip.tolist() == [False, True, False, False, True, False, False, False]
    # the diagonal of the mirrored matrix is not solved; out-of-range indices go to the solver, which reports them
    assert diag.tolist() == [False, False, True, False, False, True, False, False]


def test_plan_rule_without_mirror_solves_every_entry_as_given():
    rows, cols = [0, 3, 2, 4], [3, 0, 2, 2]
    pa, pb, flip, diag = pairs.plan_rule(rows, cols, S=5, mirrored=False)
    assert pa.tolist() == rows and pb.tolist() == cols
    assert not flip.any() and not diag.any()


def test_plan_rule_rejects_unequal_lengths():
    with pytest.raises(ValueError, match="2 row indices and 3 column"):
        pairs.plan_rule([0, 1], [0, 1, 2], S=3, mirrored=True)

