"""GPU checks of the RECT pair space and of tl.wasserstein_d_cross / tl.wasserstein_d_extend.  The contract: a block
between two sample sets is BIT-IDENTICAL to the same entries of the square matrix over the
concatenated samples, for both solvers, every kernel (EMD bit-mask and general, Sinkhorn warp form, panels and
tail, wide, FP32 and reference form), any window and any partition."""
import numpy as np
import pytest
import torch

from oracle import pilot_oracle as po
from pilot_b200 import _lib, ops, pairs, synth, tl

pytestmark = pytest.mark.gpu


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def square(P, M, regularized, reg=0.1, precision="f64"):
    return pairs.all_pairs(dev(P), dev(M), regularized, reg, precision=precision, single_rank=True).cpu().numpy()


def block(P, M, S_a, regularized, reg=0.1, precision="f64"):
    return pairs.cross_pairs(dev(P[:S_a]), dev(P[S_a:]), dev(M), regularized, reg, precision=precision,
                             single_rank=True).cpu().numpy()


def bits(x):
    """the entries' bit patterns: equal bits, NaN results included"""
    return np.ascontiguousarray(x).view(np.int64)


def check_block(P, M, S_a, regularized, reg=0.1, precision="f64"):
    sq = square(P, M, regularized, reg, precision)
    got = block(P, M, S_a, regularized, reg, precision)
    assert got.shape == (S_a, P.shape[0] - S_a)
    assert np.array_equal(bits(got), bits(sq[:S_a, S_a:])), \
        "block differs from the square over the concatenated samples"
    # the host band pipeline (bands = rows of the block) gives the same bytes
    host = pairs.cross_pairs_host(dev(P[:S_a]), dev(P[S_a:]), dev(M), regularized, reg, precision=precision,
                                  n_bands=3)
    assert np.array_equal(bits(host), bits(got))
    return got


def asym_cost(M, seed):
    A = M + 0.3 * np.triu(np.random.default_rng(seed).random(M.shape), 1)
    return A / A.max()


@pytest.mark.parametrize("regularized", ["unreg", "reg"])
@pytest.mark.parametrize("K", [10, 16, 24, 40, 64, 100, 200, 256])
def test_block_equals_square(K, regularized):
    S_a, S_b = (37, 29) if K <= 64 else (19, 13)
    P, M = synth.make_pairs(S_a + S_b, K, seed=900 + K)
    check_block(P, M, S_a, regularized)


@pytest.mark.parametrize("K", [10, 16])
def test_sinkhorn_selection_boundary(K):
    """K <= 16 picks the warp form or the panels from the size of the concatenated samples (S*S < 200 000);
    a block takes the choice of the square over them on both sides of the boundary."""
    for S_a, S_b in ((420, 40), (40, 420), (200, 40)):
        P, M = synth.make_pairs(S_a + S_b, K, seed=910 + K)
        check_block(P, M, S_a, "reg")


@pytest.mark.parametrize("K", [40, 64, 100])
def test_small_reg_absorptions_and_iteration_cap(K):
    P, M = synth.make_pairs(30, K, seed=920 + K)
    check_block(P, M, 17, "reg", reg=0.01)


@pytest.mark.parametrize("regularized", ["unreg", "reg"])
@pytest.mark.parametrize("K", [10, 40, 64, 100])
def test_asymmetric_cost(K, regularized):
    P, M = synth.make_pairs(31, K, seed=930 + K)
    check_block(P, asym_cost(M, K), 12, regularized)


@pytest.mark.parametrize("regularized", ["unreg", "reg"])
@pytest.mark.parametrize("K", [10, 24, 64])
def test_zero_masses_take_the_reference_form(K, regularized):
    P, M = synth.make_pairs(26, K, seed=940 + K)
    P[::3, 1] = 0.0
    P[1::4, K - 1] = 0.0
    P /= P.sum(axis=1, keepdims=True)
    check_block(P, M, 11, regularized, reg=0.01)


@pytest.mark.parametrize("regularized", ["unreg", "reg"])
@pytest.mark.parametrize("K", [10, 40, 64])
def test_fp32_block_equals_fp32_square(K, regularized):
    P, M = synth.make_pairs(33, K, seed=950 + K)
    check_block(P, M, 14, regularized, precision="f32")


@pytest.mark.parametrize("nranks,blk", [(1, None), (2, 7), (4, 5), (8, 64)])
def test_rect_windows_and_virtual_ranks(nranks, blk):
    """Every window of the RECT space, split over virtual ranks and unpacked from the packed layout an
    all-gather produces, writes exactly its own entries of the block."""
    S_a, S_b, K = 23, 17, 40
    P, M = synth.make_pairs(S_a + S_b, K, seed=960)
    Pd, Md = dev(P), dev(M)
    total = S_a * S_b
    for regularized in ("unreg", "reg"):
        want = square(P, M, regularized)[:S_a, S_a:]
        for first, cnt in ((0, total), (S_b * 5, S_b * 7), (13, 101), (total - 9, 9)):
            b = blk or cnt
            chunk = max(1, pairs.range_count(cnt, b, nranks, 0))
            packed = torch.zeros((nranks * chunk,), dtype=torch.float64, device="cuda")
            for r in range(nranks):
                rng = ops.make_range(cnt, _lib.PAIRS_RECT, nranks, r, b, rows=S_a, first=first)
                if _lib.range_count(rng):
                    out = packed[r * chunk:(r + 1) * chunk]
                    if regularized == "unreg":
                        ops.emd_pairs(Pd, Md, rng, out=out)
                    else:
                        ops.sinkhorn_pairs(Pd, Md, 0.1, rng, out=out)
            dense = torch.full((S_a, S_b), -1.0, dtype=torch.float64, device="cuda")
            ops.unpack_pairs(packed, chunk, S_a + S_b, ops.make_range(cnt, _lib.PAIRS_RECT, nranks, 0, b, rows=S_a,
                                                                     first=first), dense=dense)
            got = dense.cpu().numpy().ravel()
            sel = np.arange(first, first + cnt)
            assert np.array_equal(got[sel], want.ravel()[sel])
            assert (np.delete(got, sel) == -1.0).all(), "a window wrote outside its entries"


def _reps(P, prefix, start=0):
    return {f"{prefix}{start + i}": P[i] for i in range(P.shape[0])}


@pytest.mark.parametrize("S_new", [1, 9])
@pytest.mark.parametrize("cost_kind", ["symmetric", "asymmetric"])
@pytest.mark.parametrize("regularized", ["unreg", "reg"])
def test_extend_equals_wasserstein_d_on_the_union(regularized, cost_kind, S_new):
    S_old, K = 30, 24
    P, M = synth.make_pairs(S_old + S_new, K, seed=970 + S_new)
    if cost_kind == "asymmetric":
        M = asym_cost(M, 5)
    old, new = _reps(P[:S_old], "s"), _reps(P[S_old:], "s", S_old)
    EMD_old, _ = tl.wasserstein_d(old, M, regularized, 0.1)
    got, got_df = tl.wasserstein_d_extend(old, EMD_old, new, M, regularized, 0.1)
    want, want_df = tl.wasserstein_d({**old, **new}, M, regularized, 0.1)
    assert np.array_equal(got, want)
    assert np.array_equal(got_df.to_numpy(), want_df.to_numpy())
    assert got_df.index.equals(want_df.index) and got_df.columns.equals(want_df.columns)
    assert got_df.index.name == want_df.index.name == "sampleID"


@pytest.mark.parametrize("regularized", ["unreg", "reg"])
def test_extend_integer_ids_and_small_cohort_boundary(regularized):
    """Integer sample ids (the frame's literal pandas path), and a K <= 16 cohort whose union crosses the
    warp-form / panel boundary of the Sinkhorn selection while the old set alone does not (Sinkhorn then solves
    the whole union: the two forms differ in the last bits)."""
    S_old, S_new, K = 430, 30, 12
    P, M = synth.make_pairs(S_old + S_new, K, seed=980)
    old = {i: P[i] for i in range(S_old)}
    new = {S_old + i: P[S_old + i] for i in range(S_new)}
    EMD_old, _ = tl.wasserstein_d(old, M, regularized, 0.1)
    got, got_df = tl.wasserstein_d_extend(old, EMD_old, new, M, regularized, 0.1)
    want, want_df = tl.wasserstein_d({**old, **new}, M, regularized, 0.1)
    assert np.array_equal(got, want)
    assert np.array_equal(got_df.to_numpy(), want_df.to_numpy()) and got_df.index.equals(want_df.index)


@pytest.mark.parametrize("regularized", ["unreg", "reg"])
@pytest.mark.parametrize("K", [12, 64, 130])
def test_cross_matches_oracle(K, regularized):
    S_a, S_b = 14, 9
    P, M = synth.make_pairs(S_a + S_b, K, seed=990 + K)
    a, b = _reps(P[:S_a], "a"), _reps(P[S_a:], "b")
    D, frame = tl.wasserstein_d_cross(a, b, M, regularized, 0.1)
    if regularized == "unreg":
        want = po.emd_rows(P, M, 0, S_a)[:, S_a:]
    else:
        want = po.sinkhorn_rows(P, M, 0.1, 0, S_a)[0][:, S_a:]
    np.testing.assert_allclose(D, want, rtol=1e-9, atol=1e-15)
    assert list(frame.index) == list(a) and list(frame.columns) == list(b) and frame.index.name == "sampleID"
    assert np.array_equal(frame.to_numpy(), D)
    sq, _ = tl.wasserstein_d({**a, **b}, M, regularized, 0.1)
    assert np.array_equal(D, sq[:S_a, S_a:])
