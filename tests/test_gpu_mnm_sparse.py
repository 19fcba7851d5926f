"""Multinomial models on sparse counts (dpmm_create_sparse): a sparse context must compute what a dense context holding
the same matrix computes.  Where the dense kernels run the sequential ascending-d fmaf chain (the label kernels except
the tcgen05 one, the sub-label kernels at D > 128) that is byte identity of the log-likelihoods, labels, sub-labels,
counts and sums; at small D the sparse context is checked against the CPU oracle.  Then the device validation of the
caller's arrays, the -Inf convention, fit / predict end to end and one fit the dense path cannot hold."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sps

import dpmm_pkg
from oracle import dpmm_oracle as O
from tests.util import compare_sweeps, make_mnm_case

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    return dpmm_pkg.load()


def sparse_case(D, K, n, density, seed):
    """Counts at the given density with every 37th column empty and about 1 % of the stored entries explicit zeros;
    returns (dense [D, n] float32, the same matrix as CSC with the stored zeros kept, log_p, weights, lr_weights)."""
    rng = np.random.default_rng(seed)
    dense = np.zeros((D, n), np.float32)
    m = rng.random((D, n)) < density
    dense[m] = 1 + rng.poisson(1.0, int(m.sum()))
    dense[:, ::37] = 0
    x = sps.csc_matrix(dense)
    z = rng.random(x.nnz) < 0.01
    x.data[z] = 0
    dense = x.toarray().astype(np.float32)
    assert x.nnz > 0 and (x.data == 0).any()
    log_p = np.log(rng.dirichlet(np.ones(D) * 0.7, size=(K, 3))).astype(np.float32)
    w = rng.dirichlet(np.ones(K) * 5).astype(np.float32)
    lr = rng.dirichlet(np.ones(2) * 5, size=K).astype(np.float32)
    return dense, x, log_p, w, lr


@pytest.mark.parametrize("sampler,final", [(0, False), (1, False), (0, True)])
@pytest.mark.parametrize("D,K,n,density", [(300, 20, 4000, 0.2), (1000, 200, 3000, 0.05), (4096, 48, 3000, 0.01),
                                           (16384, 8, 2000, 0.001)])
def test_sparse_sweeps_are_byte_identical_to_dense(pkg, D, K, n, density, sampler, final):
    dense, x, log_p, w, lr = sparse_case(D, K, n, density, seed=D + K)
    a = pkg.GpuSweep(dense, pkg.MULTINOMIAL, seed=77)
    b = pkg.GpuSweep(x, pkg.MULTINOMIAL, seed=77)
    assert b.sparse and not a.sparse
    for s in (a, b):
        s.set_sampler(sampler)
        s.init_labels(K)
        s.set_params_multinomial(log_p, w, lr)
    assert a.debug_loglik(0).tobytes() == b.debug_loglik(0).tobytes()
    assert a.debug_loglik(1).tobytes() == b.debug_loglik(1).tobytes()
    for _ in range(5):
        for s in (a, b):
            s.sample_labels(final)
            s.sample_sublabels()
        np.testing.assert_array_equal(a.get_labels(), b.get_labels())
        np.testing.assert_array_equal(a.get_sublabels(), b.get_sublabels())
        ca, sa, _ = a.suff_stats()
        cb, sb, _ = b.suff_stats()
        np.testing.assert_array_equal(ca, cb)
        assert sa.tobytes() == sb.tobytes()
        assert a.debug_loglik(1).tobytes() == b.debug_loglik(1).tobytes()
    assert len(np.unique(a.get_labels())) > 1
    np.testing.assert_array_equal(sb[:, 0].sum(0), dense.sum(1).astype(np.float64))
    a.close(); b.close()


@pytest.mark.parametrize("D,K,n", [(20, 20, 6000), (100, 20, 6000), (20, 300, 6000), (100, 300, 6000)])
def test_small_d_oracle_parity(pkg, D, K, n):
    case = make_mnm_case(D, K, n, seed=500 + D + K)
    x = sps.csc_matrix(case["x"])
    g = pkg.GpuSweep(x, pkg.MULTINOMIAL, seed=9)
    o = O.OracleSweep(case["x"], O.MULTINOMIAL, seed=9)
    rep = compare_sweeps(g, o, case, np.random.default_rng(D + K))
    g.close()
    print(f"sparse mnm D={D} K={K} n={n}: {rep}")


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


def test_device_validation(pkg):
    E = pkg._lib
    ones = np.ones(6, np.float32)
    # columns: {1, 3} | {2} | {4, 5}  (d = 6) is valid, as are empty columns and nnz = 0
    assert _create(pkg, [1, 3, 4, 6], [1, 3, 2, 4, 5], ones[:5], 3, 6)[0] == 0
    assert _create(pkg, [1, 1, 3, 3], [2, 6], ones[:2], 3, 6)[0] == 0
    assert _create(pkg, [1, 1, 1], [], [], 2, 6)[0] == 0
    for colptr, rowval, col, what in (([1, 3, 4, 6], [1, 3, 2, 5, 4], 3, "unsorted"),
                                      ([1, 3, 4, 6], [1, 3, 2, 4, 4], 3, "duplicate"),
                                      ([1, 3, 4, 6], [1, 3, 7, 4, 5], 2, "out of range"),
                                      ([1, 3, 4, 6], [1, 3, 0, 4, 5], 2, "row 0"),
                                      ([1, 4, 3, 6], [1, 2, 3, 4, 5], 2, "decreasing colptr")):
        rc, msg = _create(pkg, colptr, rowval, ones[:5], 3, 6)
        assert rc == E.EINVAL, (what, rc, msg)
        assert f"column {col} " in msg, (what, msg)


def test_smart_project_refuses_a_sparse_context(pkg):
    x = sps.random(50, 400, density=0.1, format="csc", dtype=np.float32, random_state=3)
    x.data[:] = np.ceil(x.data * 4)
    g = pkg.GpuSweep(x, pkg.MULTINOMIAL, seed=1)
    g.init_labels(2)
    with pytest.raises(pkg._lib.DpmmError) as ei:
        g.smart_project(1, np.ones(50), np.zeros(50))
    assert ei.value.code == pkg._lib.ESTATE
    g.close()


def test_minus_inf_against_zero_counts(pkg):
    """A -Inf log-probability of a feature no point counts (absent in most columns, a stored zero in some): the sparse
    log-likelihoods are finite and equal those with any finite value in its place; the dense ones are NaN (0 * -Inf)."""
    D, K, n = 300, 6, 2000
    dense, x, log_p, w, lr = sparse_case(D, K, n, 0.05, seed=8)
    d0 = 17
    cols = np.nonzero(dense[d0] != 0)[0]
    xl = x.tolil()
    for j in cols:
        xl[d0, j] = 0          # a stored zero, not removed
    x = xl.tocsc()
    dense[d0] = 0
    assert (x.data == 0).any()
    lp_inf = log_p.copy()
    lp_inf[:, :, d0] = -np.inf
    s = pkg.GpuSweep(x, pkg.MULTINOMIAL, seed=1)
    s.init_labels(K)
    s.set_params_multinomial(lp_inf, w, lr)
    ll_inf, sl_inf = s.debug_loglik(0), s.debug_loglik(1)
    s.set_params_multinomial(log_p, w, lr)
    ll, sl = s.debug_loglik(0), s.debug_loglik(1)
    assert np.isfinite(ll_inf).all() and np.isfinite(sl_inf).all()
    assert ll_inf.tobytes() == ll.tobytes() and sl_inf.tobytes() == sl.tobytes()
    g = pkg.GpuSweep(dense, pkg.MULTINOMIAL, seed=1)
    g.init_labels(K)
    g.set_params_multinomial(lp_inf, w, lr)
    assert np.isnan(g.debug_loglik(0)).all()
    s.close(); g.close()


@pytest.mark.timeout(1200, method="thread")
def test_fit_sparse_equals_dense(pkg):
    """The D = 1 000, 40-cluster data of test_fit_past_the_table_limit: fit() on the CSC matrix returns what fit() on the
    dense array returns, on both parameter paths."""
    hyper = pkg.multinomial_hyper(np.ones(1000, np.float32))
    x, z, _ = pkg.generate_mnmm_data(20000, 1000, 40, 200, np.random.default_rng(0))
    xs = sps.csc_matrix(x)
    for dev in (True, False):
        for seed in (1, 2):
            rd = pkg.fit(x, hyper, 10.0, iters=150, seed=seed, burnout=10, device_params=dev)
            rs = pkg.fit(xs, hyper, 10.0, iters=150, seed=seed, burnout=10, device_params=dev)
            assert rs[8].group.sweep.sparse
            np.testing.assert_array_equal(rs[0], rd[0])
            np.testing.assert_array_equal(rs[7], rd[7])
            assert len(rs[1]) == len(rd[1])
            assert np.asarray(rs[2]).tobytes() == np.asarray(rd[2]).tobytes()
            print(f"sparse fit D=1000 device_params={dev} seed={seed}: K={len(rs[1])}")


def test_predict_on_device_sparse(pkg):
    from types import SimpleNamespace
    from dpmmsubclusters_jl_b200 import host as H, priors as P
    D, K, n = 5000, 12, 4000
    dense, x, *_ = sparse_case(D, K, n, 0.02, seed=21)
    rng = np.random.default_rng(22)
    cl = [SimpleNamespace(cluster_params=SimpleNamespace(cluster_params=SimpleNamespace(
        posterior_hyperparams=P.multinomial_hyper(rng.uniform(0.5, 60.0, D))))) for _ in range(K)]
    sw = pkg.GpuSweep(dense[:, :100], pkg.MULTINOMIAL)
    model = SimpleNamespace(group=SimpleNamespace(local_clusters=cl, weights=rng.dirichlet(np.ones(K)).astype(np.float32),
                                                  sweep=sw))
    ls, ps = H.predict(model, x, on_device=True)
    ld, pd = H.predict(model, dense, on_device=True)
    lh, ph = H.predict(model, x, on_device=False)
    np.testing.assert_array_equal(ls, ld)
    np.testing.assert_allclose(ps, pd, atol=1e-6)
    np.testing.assert_array_equal(ls, lh)
    np.testing.assert_allclose(ps, ph, atol=1e-6)
    sw.close()


def block_corpus(N, D, K, block, words, rng):
    """Seeded sparse bag-of-words corpus that is never dense: every document draws half of its words uniformly from
    its cluster's own `block`-word range and half uniformly from the whole vocabulary.  Returns (CSC [D, N], labels)."""
    z = rng.integers(0, K, N)
    h = words // 2
    own = rng.integers(0, block, (N, h)) + (block * z)[:, None]
    other = rng.integers(0, D, (N, words - h))
    rows = np.concatenate([own, other], axis=1).reshape(-1)
    cols = np.repeat(np.arange(N), words)
    x = sps.csc_matrix((np.ones(rows.size, np.float32), (rows, cols)), shape=(D, N))
    x.sum_duplicates()
    return x, z + 1


@pytest.mark.timeout(1800, method="thread")
def test_fit_at_d16384_without_densifying(pkg):
    from dpmmsubclusters_jl_b200.host import normalized_mutual_info
    D, N, K = 16384, 200_000, 20
    x, z = block_corpus(N, D, K, 400, 60, np.random.default_rng(11))
    hyper = pkg.multinomial_hyper(np.ones(D, np.float32))
    labels, clusters, *_ = pkg.fit(x, hyper, 10.0, iters=100, seed=3, burnout=10, device_params=True)
    nmi = normalized_mutual_info(z, labels)
    print(f"sparse fit D={D} N={N} nnz={x.nnz}: K={len(clusters)} NMI={nmi:.4f}")
    assert len(clusters) >= 10
    assert nmi >= 0.8


def test_two_gpu_sparse_statistics():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29617", os.path.join(ROOT, "tests", "mgpu_sparse_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "MGPU_SPARSE_OK" in out.stdout
