"""(f)-3 host ingest: the built-in .h5ad (HDF5) reader and the real-data golden fixture.

The reader is checked on two real HDF5 files: the reference's tutorial data set (old-style groups, contiguous datasets,
variable-length strings in global heaps, categorical columns, attributes; only where a PILOT checkout is mounted) and
SciPy's MATLAB-7.3 test file (a copy in tests/golden; 512-byte user block, version-2 layout message; content known from
SciPy's own test).  Chunked, shuffled and deflated datasets come from a minimal writer of our own
(tests/h5_writer.py), so the tests need no HDF5 library.  Sparse X and version-2 object headers are implemented from the format specification only."""
import os

import numpy as np
import pandas as pd
import pytest

from oracle import pilot_oracle as po, ref_exec
from pilot_b200 import h5ad, tl

KIDNEY = os.path.join(ref_exec.REFERENCE_ROOT, "Tutorial", "Datasets", "Kidney_IgAN_G.h5ad")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "g6_kidney_igan_G.npz")
needs_file = pytest.mark.skipif(not os.path.isfile(KIDNEY), reason="reference tutorial data not mounted")


@needs_file
def test_reads_the_tutorial_file():
    ad = h5ad.load_h5ad(KIDNEY)
    assert ad.shape == (24227, 14) and ad.X.dtype == np.float32 and ad.X.flags.c_contiguous
    assert np.isfinite(ad.X).all()
    assert list(ad.obs.columns) == ["Cell_type", "sampleID", "status", "sex", "Age"]     # the stored column-order
    assert isinstance(ad.obs["sampleID"].dtype, pd.CategoricalDtype) and len(ad.obs["sampleID"].cat.categories) == 634
    assert sorted(ad.obs["status"].cat.categories) == sorted(set(ad.obs["status"].astype(str)))
    assert ad.obs["Cell_type"].dtype == np.int64 and ad.obs["Age"].dtype == np.float64
    assert len(ad.var_names) == 14 and all(isinstance(v, str) and v for v in ad.var_names)
    assert ad.obs.index.is_unique and isinstance(ad.obs.index[0], str)
    assert ad.to_df().shape == (24227, 14) and list(ad.to_df().columns) == list(ad.var_names)
    sub = ad[:, list(ad.var_names[:3])]
    assert np.array_equal(sub.X, ad.X[:, :3])
    # what the fixture stores is what the file holds
    g = np.load(GOLDEN, allow_pickle=True)
    assert np.array_equal(g["X"], ad.X)
    assert np.array_equal(g["sample_codes"], ad.obs["sampleID"].cat.codes.to_numpy())
    assert list(g["var_names"]) == list(ad.var_names)


@needs_file
def test_extract_matches_the_reference_on_the_real_file():
    """extract_data_anno_pathomics_from_h5ad (Trajectory.py:268-297) of the reference, exec'd verbatim, and the
    mirror in pilot_b200.tl give the same frames on the object the reader returns."""
    ad = h5ad.read_h5ad(KIDNEY)
    ref = ref_exec.load()
    names = list(ad.var_names)
    wd, wa = ref.extract_data_anno_pathomics_from_h5ad(ad, var_names=names, clusters_col="Cell_type",
                                                       sample_col="sampleID", status="status")
    gd, ga = tl.extract_data_anno_pathomics_from_h5ad(ad, var_names=names, clusters_col="Cell_type",
                                                      sample_col="sampleID", status="status")
    pd.testing.assert_frame_equal(gd, wd)
    pd.testing.assert_frame_equal(ga, wa)


def test_oracle_restatement_on_the_real_data_fixture():
    """Stages 1-2 of the oracle restatement against what the reference produced on the real file (bit-exact
    proportions, cost to 1e-12), and a few rows of the exact-EMD matrix."""
    g = np.load(GOLDEN, allow_pickle=True)
    annot = pd.DataFrame({
        "cell_type": g["cell_type"],
        "sampleID": pd.Categorical.from_codes(g["sample_codes"], categories=list(g["sample_categories"])),
        "status": pd.Categorical.from_codes(g["status_codes"], categories=list(g["status_categories"])),
    })
    data = pd.DataFrame(g["X"], columns=list(g["var_names"]))
    props = po.cluster_representations(annot)
    assert [str(k) for k in props.keys()] == list(g["samples"])
    assert np.array_equal(np.stack(list(props.values())), g["props"])
    dis, cost_df = po.cost_matrix(annot, data, "cosine")
    np.testing.assert_allclose(dis, g["cost"], rtol=1e-12, atol=1e-15)
    assert [str(x) for x in po.return_real_labels(annot)] == list(g["real_labels"])
    P, M = g["props"], g["cost"] / g["cost"].max()
    for r, row in zip(g["EMD_rows"][:3], g["EMD_sub"][:3]):
        got = np.array([po.emd2(P[r], P[j], M) for j in range(0, P.shape[0], 40)])
        np.testing.assert_allclose(got, row[::40], rtol=1e-12, atol=1e-15)


def test_matlab73_file_of_scipy():
    # a copy of SciPy's scipy/io/matlab/tests/data/testhdf5_7.4_GLNX86.mat (BSD-3-Clause)
    path = os.path.join(os.path.dirname(GOLDEN), "testhdf5_7.4_GLNX86.mat")
    f = h5ad.H5File(path)                       # HDF5 behind a 512-byte user block
    assert f.root.keys() == ["testdouble"]
    np.testing.assert_allclose(f["testdouble"].read().ravel(), np.linspace(0, 2 * np.pi, 9), rtol=1e-15)


def test_load_h5ad_missing_file_behaves_like_the_reference(capsys):
    assert h5ad.load_h5ad("/nonexistent/x.h5ad") is None          # Trajectory.py:133-137: a hint, no exception
    assert "There is no such data" in capsys.readouterr().out
    with pytest.raises(h5ad.H5Error):
        h5ad.H5File(__file__)


@pytest.mark.parametrize("dtype", [np.float32, np.float64, np.int32, np.int64])
def test_chunked_filtered_datasets(tmp_path, dtype):
    """Chunked layout with a version-1 chunk B-tree, shuffle + deflate, chunk shapes that do not divide the data
    (edge chunks), several chunks per dataset -- written by the minimal test writer (tests/h5_writer.py; no h5py in
    the image), read back with the product reader."""
    from h5_writer import Writer
    rng = np.random.default_rng(11)
    a2 = (rng.normal(size=(301, 14)) * 100).astype(dtype)
    a1 = (rng.normal(size=1000) * 1000).astype(dtype)
    w = Writer()
    w.dataset("plain", a2)
    w.dataset("chunked", a2, chunks=(64, 5))
    w.dataset("gz", a2, chunks=(128, 14), gzip=4)
    w.dataset("shuffled_gz", a2, chunks=(100, 8), shuffle=True, gzip=6)
    w.dataset("vec", a1, chunks=(333,), shuffle=True, gzip=1)
    path = tmp_path / "t.h5"
    path.write_bytes(w.finish())
    f = h5ad.H5File(str(path))
    assert sorted(f.root.keys()) == ["chunked", "gz", "plain", "shuffled_gz", "vec"]
    for name in ("plain", "chunked", "gz", "shuffled_gz"):
        got = f[name].read()
        assert got.dtype == np.dtype(dtype) and got.shape == a2.shape
        assert np.array_equal(got, a2), name
    assert np.array_equal(f["vec"].read(), a1)
