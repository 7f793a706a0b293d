"""GPU parity of stages 1-2 (histogram/proportions, median centroids, cdist) against the oracle.
Everything goes through the C ABI (pilot_b200.ops).  Bit-exact for integer work and proportions."""
import numpy as np
import pandas as pd
import pytest
import scipy.spatial.distance as ssd
import torch

from oracle import pilot_oracle as po
from pilot_b200 import ops, synth, tl

pytestmark = pytest.mark.gpu


def dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


@pytest.mark.parametrize("n,K,S", [(0, 3, 2), (1, 1, 1), (3, 2, 2), (1001, 7, 5), (200_003, 10, 20),
                                   (300_000, 64, 2000), (50_000, 200, 300)])
def test_hist_counts_and_first_index(n, K, S):
    rng = np.random.default_rng(n + K)
    ct = rng.integers(0, K, size=n).astype(np.int32)
    sm = rng.integers(0, S, size=n).astype(np.int32)
    if n > 10:  # leave some codes unused
        ct[ct == K - 1] = 0
    counts, fct, fsm = ops.hist(dev(ct), dev(sm), K, S)
    want = np.bincount(sm.astype(np.int64) * K + ct, minlength=S * K).reshape(S, K)
    assert np.array_equal(counts.cpu().numpy(), want)
    wf = np.full(K, n, dtype=np.int64)
    np.minimum.at(wf, ct, np.arange(n))
    ws = np.full(S, n, dtype=np.int64)
    np.minimum.at(ws, sm, np.arange(n))
    assert np.array_equal(fct.cpu().numpy(), wf)
    assert np.array_equal(fsm.cpu().numpy(), ws)


@pytest.mark.parametrize("labels", ["str", "categorical", "int"])
@pytest.mark.parametrize("regulizer,normalization", [(0.2, True), (1.3, True), (0.2, False)])
def test_cluster_representations_bit_exact(labels, regulizer, normalization):
    X, obs = synth.make_cells(60_000, 4, 13, 37, 17, labels=labels)
    annot = obs.rename(columns={"cell_types": "cell_type"})
    got = tl.Cluster_Representations(annot, regulizer=regulizer, normalization=normalization)
    want = po.cluster_representations(annot, regulizer=regulizer, normalization=normalization)
    assert list(got.keys()) == list(want.keys())
    for k in want:
        assert got[k].dtype == np.float64
        assert np.array_equal(got[k], want[k]), k


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n,K,D", [(1, 1, 1), (2, 1, 3), (7, 2, 5), (5000, 6, 9), (120_001, 10, 30)])
def test_centroid_median_bit_exact(dtype, n, K, D):
    rng = np.random.default_rng(n * 7 + D)
    X = rng.normal(size=(n, D)).astype(dtype)
    if n >= 5000:
        X[rng.integers(0, n, 200), rng.integers(0, D, 200)] = np.nan      # NaNs are skipped
        X[: n // 3, 0] = np.round(X[: n // 3, 0], 1)                      # heavy duplicates
        X[:, 1] = np.abs(X[:, 1]) * (rng.random(n) < 0.5)                 # zero inflated
    code = rng.integers(0, K, size=n).astype(np.int32)
    code[:K] = np.arange(K)  # every type present
    cent, cent64 = ops.centroid_median(dev(X), dev(code), K)
    want = np.stack([np.nanmedian(X[code == k], axis=0) for k in range(K)])
    assert cent.cpu().numpy().dtype == dtype
    np.testing.assert_array_equal(cent.cpu().numpy(), want.astype(dtype))
    np.testing.assert_array_equal(cent64.cpu().numpy(), want.astype(np.float64))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("case", ["gauss", "duplicates", "nan", "skewed_types", "adversarial_sample"])
def test_centroid_median_streaming_path(dtype, case):
    """n >= 64K and D >= 32 take the sampled-pivot single-pass path; results must stay exact,
    including when the sample misleads the pivots (exact in-kernel fallback)."""
    rng = np.random.default_rng(hash(case) % 1000)
    n, K, D = 200_000, 10, 50
    X = rng.normal(size=(n, D)).astype(dtype)
    code = rng.integers(0, K, size=n).astype(np.int32)
    if case == "duplicates":
        X[:, :20] = np.round(X[:, :20], 1)          # ~60 distinct values per column
        X[:, 20:25] = (rng.random((n, 5)) < 0.7)    # 0/1 features (pathomics-like)
    elif case == "nan":
        X[rng.integers(0, n, 5000), rng.integers(0, D, 5000)] = np.nan
        X[code == 3, 7] = np.nan                    # an all-NaN (type, dim)
    elif case == "skewed_types":
        code = np.minimum((rng.exponential(1.2, size=n)).astype(np.int32), K - 1)  # one dominant, some rare
        code[:K] = np.arange(K)
    elif case == "adversarial_sample":
        # the rows the kernel samples (hash(row) % stride == 0, mn_hash / mn_plan_kernel in median.cu) carry
        # values far above the rest: every pivot bracket misses the true median and the pairs must take the
        # exact in-kernel fallback.  Columns 40.. are additionally sorted along the rows (harmless here; it
        # was the adversarial input of the round-1 design).
        i = np.arange(n, dtype=np.uint64)
        h = (i * np.uint64(0x9E3779B1)) & np.uint64(0xffffffff)
        h ^= h >> np.uint64(15)
        h = (h * np.uint64(0x85EBCA77)) & np.uint64(0xffffffff)
        h ^= h >> np.uint64(13)
        stride = np.array([max(1, -(-int((code == k).sum()) // 2048)) for k in range(K)], dtype=np.uint64)
        sampled = (h % stride[code]) == 0
        X[:, 40:] = np.sort(X[:, 40:], axis=0)
        X[sampled, :40] += 50.0
    cent, cent64 = ops.centroid_median(dev(X), dev(code), K)
    fallbacks = ops.median_fallbacks(K, D)
    if case == "adversarial_sample":
        assert fallbacks > 0, "the misleading sample must have triggered the exact fallback"
    elif case == "gauss":
        assert fallbacks == 0
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = np.stack([np.nanmedian(X[code == k], axis=0) for k in range(K)])
    np.testing.assert_array_equal(cent.cpu().numpy(), want.astype(dtype))
    np.testing.assert_array_equal(cent64.cpu().numpy(), want.astype(np.float64))


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
@pytest.mark.parametrize("n,K,D", [(70_001, 3, 50), (65_537, 64, 50), (100_003, 30, 33), (90_002, 5, 7), (66_001, 4, 1),
                                   (80_003, 40, 128), (70_003, 2, 512), (70_001, 2, 600), (200_003, 3000, 1)])
def test_centroid_median_run_form_shapes(dtype, n, K, D):
    """The run form of the stream pass: row counts that leave a short last chunk, column groups narrower than 32
    (several rows per step), D > 512, rows whose code is out of range (pandas' -1 for a missing label), which must be
    ignored, and a base pointer that is not 16-byte aligned.  3000 types are more than the run form's shared memory
    holds: that input takes the radix path."""
    rng = np.random.default_rng(n + D)
    X = rng.normal(size=(n, D)).astype(dtype)
    X[rng.integers(0, n, 300), rng.integers(0, D, 300)] = np.nan
    code = rng.integers(0, K, size=n).astype(np.int32)
    code[rng.integers(0, n, 500)] = -1
    code[rng.integers(0, n, 50)] = K + 3
    code[-1] = K - 1            # the very last row (in the short last chunk) counts
    X[-1] = 1e6
    cent, cent64 = ops.centroid_median(dev(X), dev(code), K)
    want = np.stack([np.nanmedian(X[code == k], axis=0) for k in range(K)])
    np.testing.assert_array_equal(cent.cpu().numpy(), want.astype(dtype))
    np.testing.assert_array_equal(cent64.cpu().numpy(), want.astype(np.float64))
    # a view that starts 4 bytes into an allocation, not 16-byte aligned: same result
    if D == 50:
        flat = torch.empty(n * D + 1, dtype=torch.from_numpy(X).dtype, device="cuda")
        Xo = flat[1:].view(n, D)
        Xo.copy_(torch.from_numpy(X))
        cent2, _ = ops.centroid_median(Xo, dev(code), K)
        np.testing.assert_array_equal(cent2.cpu().numpy(), want.astype(dtype))


def test_centroid_median_beyond_4gb():
    """12 M cells x 96 dims of float32 = 4.6 GB: byte offsets beyond 2^32 and tens of chunks per CTA in the stream
    pass.  The expectation is computed on the GPU (a full sort per type), exact like the kernel."""
    n, K, D = 12_000_000, 3, 96
    g = torch.Generator(device="cuda").manual_seed(7)
    X = torch.randn((n, D), device="cuda", dtype=torch.float32, generator=g)
    code = torch.randint(0, K, (n,), device="cuda", dtype=torch.int32, generator=g)
    X += code[:, None].to(torch.float32) * 0.25
    X[n - 1] = 1e6                                      # the very last row counts
    cent, cent64 = ops.centroid_median(X, code, K)
    assert ops.median_fallbacks(K, D) == 0
    for k in range(K):
        Xk = X[code == k]
        m = Xk.shape[0]
        srt = torch.sort(Xk, dim=0).values
        want = srt[(m - 1) // 2] if m % 2 else (srt[m // 2 - 1] + srt[m // 2]) / 2
        assert torch.equal(cent[k], want), k
        assert torch.equal(cent64[k], want.to(torch.float64)), k
        del Xk, srt


@pytest.mark.parametrize("order", ["by_type", "by_type_blocks", "one_type_dominates"])
def test_centroid_median_sorted_inputs_stay_on_the_fast_path(order):
    """AnnData objects are often sorted by cluster or by sample.  The run-form stream pass counting-sorts 4096-row
    chunks: a chunk then holds one type only (one long run cut into 128-row segments), and a type's candidates come
    from a few chunks -- the list replicas must still fill evenly (no overflow -> no exact fallback) and the result
    stays exact."""
    rng = np.random.default_rng(21)
    n, K, D = 400_000, 12, 50
    X = rng.normal(size=(n, D)).astype(np.float32)
    code = rng.integers(0, K, size=n).astype(np.int32)
    if order == "by_type":
        code = np.sort(code)
    elif order == "by_type_blocks":
        code = np.repeat(rng.permutation(np.arange(K * 8) % K), n // (K * 8) + 1)[:n].astype(np.int32)
    else:
        code = np.where(rng.random(n) < 0.9, 3, code).astype(np.int32)
    X += code[:, None].astype(np.float32)             # type-dependent location: a wrong row assignment would show
    cent, cent64 = ops.centroid_median(dev(X), dev(code), K)
    assert ops.median_fallbacks(K, D) == 0
    want = np.stack([np.nanmedian(X[code == k], axis=0) for k in range(K)])
    np.testing.assert_array_equal(cent.cpu().numpy(), want)
    np.testing.assert_array_equal(cent64.cpu().numpy(), want.astype(np.float64))


@pytest.mark.parametrize("metric", ["cosine", "euclidean", "sqeuclidean", "cityblock", "chebyshev", "correlation",
                                    "braycurtis", "canberra", "minkowski", "seuclidean", "hamming"])
def test_cdist_matches_scipy(metric):
    rng = np.random.default_rng(4)
    C = rng.normal(size=(37, 50))
    if metric == "hamming":
        C = np.round(C)                     # coordinates that actually coincide
    if metric == "canberra":
        C[:, 3] = 0.0                       # 0 / 0 terms contribute nothing
    cost, cost_norm, cmax = ops.cdist(dev(C), metric)
    want = ssd.squareform(ssd.pdist(C, metric))
    np.testing.assert_allclose(cost.cpu().numpy(), want, rtol=1e-12, atol=1e-14)
    got = cost.cpu().numpy()
    assert np.array_equal(cost_norm.cpu().numpy(), got / got.max())
    assert cmax.item() == got.max()
    assert np.array_equal(got, got.T) and (np.diag(got) == 0).all()


def test_cdist_unknown_metric_raises():
    with pytest.raises(ValueError):
        ops.cdist(dev(np.zeros((3, 3))), "jaccard")


@pytest.mark.parametrize("labels", ["str", "categorical"])
def test_cost_matrix_matches_oracle(labels):
    X, obs = synth.make_cells(80_000, 20, 9, 12, 5, labels=labels)
    annot = obs.rename(columns={"cell_types": "cell_type"})
    data = pd.DataFrame(X)
    dis, cost = tl.cost_matrix(annot, data, metric="cosine")
    wdis, wcost = po.cost_matrix(annot, data, metric="cosine")
    np.testing.assert_allclose(dis, wdis, rtol=1e-12, atol=1e-15)
    pd.testing.assert_index_equal(cost.index, wcost.index)
    assert list(cost.columns) == list(wcost.columns)
