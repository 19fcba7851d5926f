"""CPU checks of sparse multinomial input: the scipy -> 1-based CSC conversion, the host-side argument checks of
dpmm_create_sparse, the NIW refusals, load_data of a .npz and the NumPy predict on sparse data."""
import ctypes as C
import os
from types import SimpleNamespace

import numpy as np
import pytest
import scipy.sparse as sps

import dpmm_pkg


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    return dpmm_pkg.load()


def test_csc_conversion_sums_duplicates_and_sorts(pkg):
    from dpmmsubclusters_jl_b200.sweep import csc_1based
    # D = 5, N = 4; column 1 has its rows out of order and a duplicate (row 3 twice), column 2 is empty
    rows = np.array([4, 0, 3, 3, 2, 1, 0])
    cols = np.array([1, 1, 1, 1, 0, 3, 3])
    vals = np.array([1.0, 2.0, 3.0, 4.0, 5.0, 6.0, 7.0])
    x = sps.coo_matrix((vals, (rows, cols)), shape=(5, 4))
    for m in (x, x.tocsr(), sps.csc_matrix((vals, (rows, cols)), shape=(5, 4)), x.T.tocsr().T):
        colptr, rowval, nzval = csc_1based(m)
        assert colptr.dtype == np.int64 and rowval.dtype == np.int64 and nzval.dtype == np.float32
        np.testing.assert_array_equal(colptr, [1, 2, 5, 5, 7])
        np.testing.assert_array_equal(rowval, [3, 1, 4, 5, 1, 2])
        np.testing.assert_array_equal(nzval, [5, 2, 7, 1, 7, 6])
    assert x.nnz == 7   # the caller's matrix is not modified


def test_sparse_needs_the_multinomial_prior(pkg):
    x = sps.random(6, 40, density=0.3, format="csc", dtype=np.float32, random_state=1)
    with pytest.raises(ValueError):
        pkg.GpuSweep(x, pkg.NIW)
    with pytest.raises(ValueError):
        pkg.fit(x, 10.0, iters=2)
    with pytest.raises(ValueError):
        pkg.fit(x, pkg.niw_hyperparams(1.0, np.zeros(6), 9, np.eye(6)), 10.0, iters=2)


def _create(pkg, colptr, rowval, nzval, n, d):
    lib = pkg._lib.load()
    h = C.c_void_p()
    colptr = np.ascontiguousarray(colptr, np.int64)
    rowval = np.ascontiguousarray(rowval, np.int64)
    nzval = np.ascontiguousarray(nzval, np.float32)
    rc = lib.dpmm_create_sparse(C.byref(h), colptr.ctypes.data_as(C.POINTER(C.c_int64)),
                                rowval.ctypes.data_as(C.POINTER(C.c_int64)), nzval.ctypes.data_as(C.POINTER(C.c_float)),
                                n, d, 0, 1, 0)
    msg = lib.dpmm_last_error(None).decode()
    if rc == 0:
        lib.dpmm_destroy(h)
    return rc, msg


def test_create_sparse_host_checks(pkg):
    E = pkg._lib
    rc, msg = _create(pkg, [1, 2, 3], [1, 2], [1, 1], 2, 16385)
    assert rc == E.ELIMIT, msg
    rc, msg = _create(pkg, [0, 1, 2], [1, 2], [1, 1], 2, 10)
    assert rc == E.EINVAL and "colptr[0]" in msg, msg
    rc, msg = _create(pkg, [1, 2, 0], [1, 2], [1, 1], 2, 10)
    assert rc == E.EINVAL and "nnz" in msg, msg


def test_create_sparse_without_a_device(pkg):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    x = sps.random(30, 50, density=0.1, format="csc", dtype=np.float32, random_state=2)
    with pytest.raises(pkg._lib.DpmmError) as ei:
        pkg.GpuSweep(x, pkg.MULTINOMIAL)
    assert ei.value.code == pkg._lib.ECUDA
    assert "no CPU fallback" in str(ei.value)
    # empty columns and nnz = 0 pass the host checks too
    rc, msg = _create(pkg, [1, 1, 1], np.zeros(0), np.zeros(0), 2, 10)
    assert rc == pkg._lib.ECUDA, msg


def test_load_data_reads_npz(pkg, tmp_path):
    rng = np.random.default_rng(3)
    dense = (rng.random((40, 12)) < 0.2) * rng.integers(1, 5, (40, 12))     # N x D, as the reference's .npy
    sps.save_npz(str(tmp_path / "corpus.npz"), sps.csr_matrix(dense.astype(np.float32)))
    x = pkg.load_data(str(tmp_path) + os.sep, prefix="corpus")
    assert sps.issparse(x) and x.shape == (12, 40)
    np.testing.assert_array_equal(x.toarray(), dense.T)
    y = pkg.load_data(str(tmp_path) + os.sep, prefix="corpus", swapDimension=False)
    np.testing.assert_array_equal(y.toarray(), dense)


def test_numpy_predict_on_sparse_equals_dense(pkg):
    from dpmmsubclusters_jl_b200 import host as H, priors as P
    D, K, n = 200, 5, 300
    rng = np.random.default_rng(4)
    dense = ((rng.random((D, n)) < 0.05) * rng.integers(1, 4, (D, n))).astype(np.float32)
    cl = [SimpleNamespace(cluster_params=SimpleNamespace(cluster_params=SimpleNamespace(
        posterior_hyperparams=P.multinomial_hyper(rng.uniform(0.5, 60.0, D))))) for _ in range(K)]
    model = SimpleNamespace(group=SimpleNamespace(local_clusters=cl, weights=rng.dirichlet(np.ones(K)).astype(np.float32),
                                                  sweep=None))
    ld, pd = H.predict(model, dense, on_device=False)
    ls, ps = H.predict(model, sps.csc_matrix(dense), on_device=False)
    np.testing.assert_array_equal(ls, ld)
    np.testing.assert_allclose(ps, pd, atol=1e-6)
