"""CPU-side checks of the RECT pair space (two sample sets concatenated in props): the host statement of the
mapping and of the bands, the library's argument checks, and the argument errors of tl.wasserstein_d_cross /
tl.wasserstein_d_extend that are raised before any device work."""
import ctypes

import numpy as np
import pytest

from pilot_b200 import _lib, ops, pairs, tl


@pytest.mark.parametrize("S,rows", [(2, 1), (5, 1), (5, 4), (7, 3), (40, 17)])
def test_rect_mapping_matches_enumeration(S, rows):
    want = [(i, j) for i in range(rows) for j in range(rows, S)]
    assert ops.n_pairs(S, _lib.PAIRS_RECT, rows) == len(want)
    assert [pairs.global_to_ij(g, S, _lib.PAIRS_RECT, rows) for g in range(len(want))] == want
    for i in range(rows + 1):
        assert pairs.row_start(i, S, _lib.PAIRS_RECT, rows) == sum(1 for p in want if p[0] < i)


@pytest.mark.parametrize("S,rows,n_bands", [(10, 3, 1), (10, 3, 2), (10, 3, 8), (300, 299, 7), (300, 1, 5)])
def test_rect_bands_cover_the_block_rows(S, rows, n_bands):
    edges = pairs.band_rows(S, _lib.PAIRS_RECT, n_bands, rows)
    assert edges[0] == 0 and edges[-1] == rows
    assert all(a < b for a, b in zip(edges, edges[1:]))
    assert len(edges) - 1 == min(n_bands, rows)


@pytest.mark.parametrize("total,block,nranks", [(17 * 23, 5, 3), (1, 1, 2), (4000 * 200, 4096, 8)])
def test_rect_partition_covers_every_pair_once(total, block, nranks):
    counts = []
    for rank in range(nranks):
        r = ops.make_range(total, _lib.PAIRS_RECT, nranks, rank, block, rows=17)
        c = _lib.range_count(r)
        assert c == pairs.range_count(total, block, nranks, rank)
        counts.append(c)
    assert sum(counts) == total


def test_pair_range_rows_field_keeps_its_former_name():
    r = _lib.PairRange(total=1, block=1, nranks=1, rank=0, mode=0, reserved=0)
    assert r.rows == 0
    r = _lib.PairRange(total=1, block=1, nranks=1, rank=0, mode=_lib.PAIRS_RECT, rows=3)
    assert r.reserved == 3
    assert ctypes.sizeof(_lib.PairRange) == 40


@pytest.mark.parametrize("rows,total,first,msg", [(0, 1, 0, b"RECT row count 0"), (10, 1, 0, b"RECT row count 10"),
                                                  (-1, 1, 0, b"RECT row count -1"),
                                                  (4, 25, 0, b"window"), (4, 1, 24, b"window")])
def test_library_rejects_a_bad_rect_range(rows, total, first, msg):
    L = _lib.lib()
    S = 10  # rows = 4: a 4 x 6 block of 24 pairs
    r = ops.make_range(total, _lib.PAIRS_RECT, rows=rows, first=first)
    assert L.pilot_unpack_pairs(1, 1, S, ctypes.byref(r), 0.0, 1, None) < 0
    assert msg in L.pilot_last_error()
    assert L.pilot_emd_pairs(1, S, 3, 1, 0, ctypes.byref(r), 1, 1, None, None, 1, 1 << 20, None) < 0
    assert msg in L.pilot_last_error()
    assert L.pilot_sinkhorn_pairs(1, S, 3, 1, 0.1, 1000, 1e-9, 1e3, 20, ctypes.byref(r), 0, 1, 1, None, None, None,
                                  1, 1 << 30, None) < 0
    assert msg in L.pilot_last_error()


def _reps(n, K, seed, prefix):
    rng = np.random.default_rng(seed)
    P = rng.dirichlet(np.ones(K), size=n)
    return {f"{prefix}{i}": P[i] for i in range(n)}


def _cost(K):
    c = np.abs(np.subtract.outer(np.arange(K), np.arange(K))).astype(np.float64)
    return c / c.max()


def test_cross_rejects_different_cell_types():
    with pytest.raises(ValueError, match="cell types"):
        tl.wasserstein_d_cross(_reps(3, 5, 0, "a"), _reps(3, 6, 1, "b"), _cost(5))
    with pytest.raises(ValueError, match="cost has shape"):
        tl.wasserstein_d_cross(_reps(3, 5, 0, "a"), _reps(3, 5, 1, "b"), _cost(4), regularized="reg")


def test_cross_rejects_unequal_masses_across_the_sets():
    b = {k: 2.0 * v for k, v in _reps(3, 5, 1, "b").items()}
    with pytest.raises(AssertionError, match="same sum"):
        tl.wasserstein_d_cross(_reps(3, 5, 0, "a"), b, _cost(5))


def test_cross_with_an_empty_set_is_empty():
    D, frame = tl.wasserstein_d_cross({}, _reps(3, 5, 1, "b"), _cost(5))
    assert D.shape == (0, 3) and list(frame.columns) == ["b0", "b1", "b2"] and frame.index.name == "sampleID"


def test_extend_argument_errors():
    old, new = _reps(4, 5, 0, "s"), _reps(2, 5, 1, "t")
    EMD = np.zeros((4, 4))
    with pytest.raises(ValueError, match="in both sets"):
        tl.wasserstein_d_extend(old, EMD, {"s1": new["t0"]}, _cost(5))
    with pytest.raises(ValueError, match="expected"):
        tl.wasserstein_d_extend(old, np.zeros((3, 3)), new, _cost(5))
    with pytest.raises(ValueError, match="cell types"):
        tl.wasserstein_d_extend(old, EMD, _reps(2, 6, 1, "t"), _cost(5))
    with pytest.raises(AssertionError, match="same sum"):
        tl.wasserstein_d_extend(old, EMD, {k: 3.0 * v for k, v in new.items()}, _cost(5))


def test_extend_without_new_samples_returns_the_matrix():
    old = _reps(3, 5, 0, "s")
    EMD = np.arange(9.0).reshape(3, 3)
    out, frame = tl.wasserstein_d_extend(old, EMD, {}, _cost(5))
    assert np.array_equal(out, EMD) and out is not EMD
    assert np.array_equal(frame.to_numpy(), EMD.T) and list(frame.index) == list(old)


def test_sinkhorn_form_boundary():
    assert pairs.sinkhorn_form_changes(430, 460, 12) and pairs.sinkhorn_form_changes(460, 430, 16)
    assert not pairs.sinkhorn_form_changes(430, 440, 12)
    assert not pairs.sinkhorn_form_changes(448, 20000, 16)
    assert not pairs.sinkhorn_form_changes(430, 460, 17)
