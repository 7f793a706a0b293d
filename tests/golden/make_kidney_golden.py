"""Golden fixture from the reference's OWN test case on REAL data.

    python tests/golden/make_kidney_golden.py          (build container only: /root/reference is mounted)

The reference's only test (test/test_pilot.py:7-15) runs
``pl.tl.wasserstein_distance(adata_G, clusters_col='Cell_type', sample_col='sampleID', status='status',
data_type='Pathomics')`` on ``Tutorial/Datasets/Kidney_IgAN_G.h5ad`` (24 227 glomeruli x 14 morphometric features,
634 biopsies).  Here that file is read with the built-in HDF5 reader (pilot_b200/h5ad.py; no anndata / h5py in the
image), the reference's functions -- ast-extracted verbatim by oracle/ref_exec.py -- are run on it with the oracle's
``ot`` shim, and the inputs the GPU path needs plus the reference's outputs are stored:
  * X (float32), the label columns as codes + category tables          -> inputs (the .h5ad cannot travel)
  * proportions, sample / cell-type order, cost matrix, real labels     -> reference code alone
  * 22 evenly spaced rows of the 634 x 634 EMD matrix, its column sums  -> reference loop + C oracle of ot.emd2
The file is kept under 1 MB; the embedding alone takes 0.78 MB of it.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import pilot_oracle, ref_exec  # noqa: E402
from pilot_b200 import h5ad  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(ref_exec.REFERENCE_ROOT, "Tutorial", "Datasets", "Kidney_IgAN_G.h5ad")


def main():
    adata = h5ad.read_h5ad(SRC)
    ref = ref_exec.load(pilot_oracle.OtShim(numpy_sinkhorn=False))
    cwd = os.getcwd()
    os.chdir("/tmp")  # the reference mkdirs ./Results_PILOT/plots
    try:
        ref.wasserstein_distance(adata, clusters_col="Cell_type", sample_col="sampleID", status="status",
                                 data_type="Pathomics")
    finally:
        os.chdir(cwd)
    u = adata.uns
    props = u["proportions"]
    E = u["EMD"]
    rows = np.linspace(0, E.shape[0] - 1, 64).astype(np.int64)[::3]
    obs = adata.obs
    np.savez_compressed(
        os.path.join(HERE, "g6_kidney_igan_G.npz"),
        X=np.asarray(adata.X),
        var_names=np.array([str(v) for v in adata.var_names], dtype=object),
        cell_type=obs["Cell_type"].to_numpy(),
        sample_codes=obs["sampleID"].cat.codes.to_numpy(),
        sample_categories=np.array([str(c) for c in obs["sampleID"].cat.categories], dtype=object),
        status_codes=obs["status"].cat.codes.to_numpy(),
        status_categories=np.array([str(c) for c in obs["status"].cat.categories], dtype=object),
        samples=np.array([str(x) for x in props.keys()], dtype=object),
        cells=np.array(list(u["cost"].columns)),
        props=np.stack([props[x] for x in props.keys()]),
        cost=u["cost"].to_numpy(),
        EMD_rows=rows,
        EMD_sub=E[rows],
        EMD_colsum=E.sum(axis=0),
        EMD_diag=np.diag(E).copy(),
        real_labels=np.array([str(x) for x in u["real_labels"]], dtype=object),
    )
    print("X", adata.X.shape, adata.X.dtype, "props", np.stack(list(props.values())).shape, "cost", u["cost"].shape,
          "EMD", E.shape, "max", E.max())


if __name__ == "__main__":
    main()
