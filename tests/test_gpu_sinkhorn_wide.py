"""GPU tests of stabilised Sinkhorn for 65..256 cell types: the cluster-split DMMA panels (sinkhorn_wide.cu),
the reference form with its Gibbs matrix in the workspace, and the dispatch between them."""
import functools

import numpy as np
import pytest
import torch

from oracle import pilot_oracle as po
from pilot_b200 import _lib, ops, synth, tl

pytestmark = pytest.mark.gpu

SK_RTOL = 1e-9


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


@functools.lru_cache(maxsize=None)
def _case(K, reg, S, seed):
    P, M = synth.make_pairs(S, K, seed=seed)
    want, witers, wabs = po.sinkhorn_rows(P, M, reg, 0, S)
    return P, M, want, witers, wabs


def _full(S):
    return ops.make_range(S * S, _lib.PAIRS_FULL)


def _check_oracle(P, M, reg, algo, want, witers, wabs):
    S = P.shape[0]
    out, iters, absn, status = ops.sinkhorn_pairs(dev(P), dev(M), reg, _full(S), algo=algo, want_info=True)
    np.testing.assert_array_equal(iters.cpu().numpy().reshape(S, S), witers)
    np.testing.assert_array_equal(absn.cpu().numpy().reshape(S, S), wabs)
    np.testing.assert_allclose(out.cpu().numpy().reshape(S, S), want, rtol=SK_RTOL, atol=1e-300)
    assert np.isin(status.cpu().numpy(), [0, 1]).all()
    return iters.cpu().numpy(), status.cpu().numpy()


@pytest.mark.parametrize("algo", [0, 1, 3])
@pytest.mark.parametrize("K", [65, 72, 120, 128, 136, 150, 151, 192, 193, 200, 250, 256])
def test_wide_matches_oracle(K, algo):
    P, M, want, witers, wabs = _case(K, 0.1, 4, 1000 + K)
    _check_oracle(P, M, 0.1, algo, want, witers, wabs)


@pytest.mark.parametrize("algo", [0, 1])
@pytest.mark.parametrize("K,reg,seed", [(100, 0.01, 2100), (192, 0.01, 2192), (200, 0.02, 2200), (256, 0.02, 2257)])
def test_wide_many_absorptions(K, reg, seed, algo):
    """Small reg: many absorptions, and problems that run into the iteration cap."""
    P, M, want, witers, wabs = _case(K, reg, 3, seed)
    assert wabs.max() > 0 and (witers == 1000).any()
    iters, status = _check_oracle(P, M, reg, algo, want, witers, wabs)
    assert (status[iters == 1000] == 1).all()  # PILOT_ST_MAXITER


@pytest.mark.parametrize("K", [100, 200, 256])
def test_wide_asymmetric_cost(K):
    """A non-symmetric cost runs the general variant (K0 and K0^T stripes, clusters of up to 8 CTAs: 8 at K = 256)."""
    S = 4
    P, _ = synth.make_pairs(S, K, seed=77)
    M = np.random.default_rng(3).random((K, K))
    M /= M.max()
    want, witers, wabs = po.sinkhorn_rows(P, M, 0.1, 0, S)
    _check_oracle(P, M, 0.1, 0, want, witers, wabs)


@pytest.mark.parametrize("cap", ["0", None])
@pytest.mark.parametrize("K", [100, 200])
def test_wide_zero_masses_take_reference_form(K, cap, monkeypatch):
    if cap is not None:
        monkeypatch.setenv("PILOT_SK_REDO_CAP", cap)  # the marker scan finds every queued problem
    S = 6
    P, M = synth.make_pairs(S, K, seed=31)
    P[::2, 2] = 0.0
    P /= P.sum(axis=1, keepdims=True)
    out, iters, absn, status = ops.sinkhorn_pairs(dev(P), dev(M), 0.05, _full(S), want_info=True)
    ref = ops.sinkhorn_pairs(dev(P), dev(M), 0.05, _full(S), algo=1).cpu().numpy()
    got = out.cpu().numpy()
    assert (status.cpu().numpy() >= 0).all(), "a problem was left unsolved"
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    np.testing.assert_allclose(got, ref, rtol=1e-12, equal_nan=True)
    want, _, _ = po.sinkhorn_rows(P, M, 0.05, 0, S)
    np.testing.assert_allclose(got.reshape(S, S), want, rtol=SK_RTOL, equal_nan=True)


@pytest.mark.parametrize("mode", [_lib.PAIRS_FULL, _lib.PAIRS_UPPER])
def test_wide_partition_invariance_and_determinism(mode):
    S, K = 13, 200
    P, M = synth.make_pairs(S, K, seed=12)
    Pd, Md = dev(P), dev(M)
    total = ops.n_pairs(S, mode)
    ref = ops.sinkhorn_pairs(Pd, Md, 0.1, ops.make_range(total, mode)).cpu().numpy()
    again = ops.sinkhorn_pairs(Pd, Md, 0.1, ops.make_range(total, mode)).cpu().numpy()
    assert np.array_equal(ref, again), "two runs must be bit-identical"
    rng_all = ops.make_range(total, mode)
    want = ops.unpack_pairs(dev(ref), total, S, rng_all, 0.0).cpu().numpy()
    for nranks, block in ((2, 7), (4, 5), (8, 3)):
        chunk = max(1, _lib.range_count(_lib.PairRange(total=total, block=block, nranks=nranks, rank=0, mode=mode,
                                                       reserved=0)))
        packed = torch.zeros((nranks * chunk,), dtype=torch.float64, device="cuda")
        for r in range(nranks):
            rng = _lib.PairRange(total=total, block=block, nranks=nranks, rank=r, mode=mode, reserved=0)
            if _lib.range_count(rng):
                ops.sinkhorn_pairs(Pd, Md, 0.1, rng, out=packed[r * chunk:(r + 1) * chunk])
        rng0 = _lib.PairRange(total=total, block=block, nranks=nranks, rank=0, mode=mode, reserved=0)
        dense = ops.unpack_pairs(packed, chunk, S, rng0, 0.0).cpu().numpy()
        assert np.array_equal(dense, want), f"nranks={nranks}: partitioned result must be bit-identical"


@pytest.mark.parametrize("K", [100, 200])
def test_wide_batch_independence(K):
    """The same problem in another slot, team and CTA gives the same bits."""
    P40, M = synth.make_pairs(40, K, seed=55)
    P6 = P40[:6].copy()
    big = ops.sinkhorn_pairs(dev(P40), dev(M), 0.1, _full(40)).cpu().numpy().reshape(40, 40)
    small = ops.sinkhorn_pairs(dev(P6), dev(M), 0.1, _full(6)).cpu().numpy().reshape(6, 6)
    assert np.array_equal(big[:6, :6], small)


def _slot_bound(K, sym):
    """An upper bound on the problems the wide kernel holds at once: at most one CTA per SM, clusters of
    ceil(KC / stripe) CTAs, at most 8 teams of 8 slots per CTA (sinkhorn_wide.cu)."""
    KC = -(-K // 8) * 8
    CL = -(-KC // (64 if sym else 32))
    return torch.cuda.get_device_properties(0).multi_processor_count // CL * 8 * 8


@pytest.mark.parametrize("K,sym,reg", [(100, True, 0.02), (200, True, 0.02), (100, False, 0.1), (200, False, 0.1),
                                       (256, False, 0.1)])
def test_wide_refilled_slots(K, sym, reg):
    """A batch at least 4x the slots the kernel can hold: every problem from local index _slot_bound on is taken
    by a team after it finished an earlier one (member 0 draws it, every member reuses the slot's columns, its
    rea / reb and state).  All of them against the reference form, the last rows against the oracle, and a block
    of refilled problems bit for bit against the same problems solved first in a small batch.  At reg 0.02 almost
    every problem absorbs, so refilled slots follow problems that left rea / reb behind."""
    bound = _slot_bound(K, sym)
    S = int(np.ceil(np.sqrt(4 * bound)))
    P, M = synth.make_pairs(S, K, seed=4000 + K)
    if not sym:
        M = np.random.default_rng(K).random((K, K))
        M /= M.max()
    Pd, Md = dev(P), dev(M)
    out, iters, absn, status = ops.sinkhorn_pairs(Pd, Md, reg, _full(S), want_info=True)
    got, iters, absn = out.cpu().numpy(), iters.cpu().numpy(), absn.cpu().numpy()
    assert np.isin(status.cpu().numpy(), [0, 1]).all()
    ref, riters, rabs, _ = ops.sinkhorn_pairs(Pd, Md, reg, _full(S), algo=1, want_info=True)
    np.testing.assert_array_equal(iters, riters.cpu().numpy())
    np.testing.assert_array_equal(absn, rabs.cpu().numpy())
    np.testing.assert_allclose(got, ref.cpu().numpy(), rtol=SK_RTOL, atol=1e-300)
    r0 = S - 2
    assert r0 * S >= bound  # refilled rows
    want, witers, wabs = po.sinkhorn_rows(P, M, reg, r0, S)
    np.testing.assert_array_equal(iters.reshape(S, S)[r0:], witers)
    np.testing.assert_array_equal(absn.reshape(S, S)[r0:], wabs)
    np.testing.assert_allclose(got.reshape(S, S)[r0:], want, rtol=SK_RTOL, atol=1e-300)
    again = ops.sinkhorn_pairs(Pd, Md, reg, _full(S)).cpu().numpy()
    assert np.array_equal(got, again), "two runs must be bit-identical"
    b0 = S - 6
    assert b0 * S >= bound
    small = ops.sinkhorn_pairs(dev(P[b0:]), Md, reg, _full(6)).cpu().numpy().reshape(6, 6)
    assert np.array_equal(got.reshape(S, S)[b0:, b0:], small)


@pytest.mark.parametrize("algo", [0, 1])
def test_more_than_256_types_is_rejected(algo):
    P, M = synth.make_pairs(3, 257, seed=1)
    with pytest.raises(_lib.PilotLibraryError, match="K=257"):
        ops.sinkhorn_pairs(dev(P), dev(M), 0.1, _full(3), algo=algo)


@pytest.mark.parametrize("K", [100, 200])
def test_fp32_request_above_64_types_runs_fp64(K):
    P, M, want, _, _ = _case(K, 0.1, 4, 1000 + K)
    got = ops.sinkhorn_pairs(dev(P), dev(M), 0.1, _full(4), precision="f32").cpu().numpy().reshape(4, 4)
    np.testing.assert_allclose(got, want, rtol=1e-4)


def test_wasserstein_distance_with_200_types(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    X, obs = synth.make_cells(60_000, 16, 200, 5, seed=8)
    adata = synth.FakeAnnData(obs, obsm={"X_PCA": X})
    tl.wasserstein_distance(adata, regularized="reg", reg=0.1)
    annot, data = adata.uns["annot"], adata.uns["data"]
    props = po.cluster_representations(annot)
    assert len(next(iter(props.values()))) > 150
    dis, _ = po.cost_matrix(annot, data, "cosine")
    want, _ = po.wasserstein_d(props, dis / dis.max(), regularized="reg", reg=0.1)
    np.testing.assert_allclose(adata.uns["EMD"], want, rtol=1e-9, atol=1e-15)
