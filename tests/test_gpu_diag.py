"""The diagonal-covariance Gaussian prior on the B200: label / sub-label / statistics parity with the CPU oracle over
feature widths 1 .. 4 096 and K up to 300, the D = 1 identity with the NIW prior, the D = 16 384 / K = 1 024 limit,
fit() / predict / checkpoints, and two GPUs against one."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

import dpmm_pkg
from oracle import diag_oracle as DO
from tests.diag_util import axis_aligned_data, compare_diag_sweeps, make_diag_case, set_params_diag
from tests.util import check_draws, tie_tolerance

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    return dpmm_pkg.load()


@pytest.mark.timeout(900, method="thread")
@pytest.mark.parametrize("D,K,n,final", [(1, 5, 3001, False), (2, 40, 5003, False), (7, 300, 20011, False),
                                         (32, 5, 10007, True), (32, 1, 2000, False), (100, 40, 8009, False),
                                         (100, 300, 4000, True), (257, 300, 3001, False), (1000, 40, 3001, False),
                                         (4096, 5, 1501, False)])
def test_sweep_parity(pkg, D, K, n, final):
    case = make_diag_case(D, K, n, seed=D * 1000 + K)
    g = pkg.GpuSweep(case["x"], pkg.DIAG, seed=7)
    o = DO.DiagOracleSweep(case["x"], seed=7)
    rep = compare_diag_sweeps(g, o, case, np.random.default_rng(D + K), final=final)
    g.close()
    print(f"diag D={D} K={K} n={n} final={final}: {rep}")


@pytest.mark.timeout(600, method="thread")
@pytest.mark.parametrize("D,K", [(7, 6), (300, 40)])
def test_far_means_empty_and_zero_weight_clusters(pkg, D, K):
    """Means 10^3 sigma from the origin, one cluster without points and one of weight 0."""
    case = make_diag_case(D, K, 6007, seed=D + 5, offset=1e3, empty=True, zero_weight=True)
    g = pkg.GpuSweep(case["x"], pkg.DIAG, seed=3)
    o = DO.DiagOracleSweep(case["x"], seed=3)
    rep = compare_diag_sweeps(g, o, case, np.random.default_rng(D), final=False)
    set_params_diag(g, case)
    g.sample_labels(False)
    lab = g.get_labels()
    assert not (lab == 1).any() and not (lab == K).any()    # weight 0 / no points near
    g.close()
    print(f"far D={D} K={K}: {rep}")


@pytest.mark.timeout(300, method="thread")
def test_d1_is_the_niw_prior(pkg):
    case = make_diag_case(1, 12, 20000, seed=11)
    inv = (1.0 / case["var"].astype(np.float64)).astype(np.float32)[..., None]
    a = pkg.GpuSweep(case["x"], pkg.DIAG, seed=5)
    b = pkg.GpuSweep(case["x"], pkg.NIW, seed=5)
    rng = np.random.default_rng(0)
    u, us = rng.random(case["n"]), rng.random(case["n"])
    for s in (a, b):
        s.set_uniforms(u, us, None)
        s.init_labels(12)
    set_params_diag(a, case)
    b.set_params_niw(case["mu"], inv, case["logdet"], case["weights"], case["lr_weights"])
    for which in (0, 1):
        la, lb = a.debug_loglik(which).astype(np.float64), b.debug_loglik(which).astype(np.float64)
        assert (np.abs(la - lb) <= 1e-6 * np.maximum(np.abs(lb), 1.0)).all(), np.abs(la - lb).max()
    LL = b.debug_loglik(0)
    for final in (False, True):
        a.sample_labels(final); b.sample_labels(final)
        check_draws(LL, u, a.get_labels(), b.get_labels(), f"D = 1 labels (final={final})")
    b.set_labels(a.get_labels())
    SL = b.debug_loglik(1)
    a.sample_sublabels(); b.sample_sublabels()
    check_draws(SL, us, a.get_sublabels(), b.get_sublabels(), "D = 1 sub-labels")
    a.close(); b.close()


@pytest.mark.timeout(600, method="thread")
def test_limits(pkg):
    E = pkg._lib
    out = (ctypes.c_int32 * 3)()
    assert E.load().dpmm_limits(out) == 0
    assert out[1] == 16384 and out[2] == 1024
    with pytest.raises(E.DpmmError) as ei:
        pkg.GpuSweep(np.zeros((16385, 4), np.float32), pkg.DIAG)
    assert ei.value.code == E.ELIMIT
    D, K, n = 16384, 1024, 300
    rng = np.random.default_rng(3)
    x = (rng.standard_normal((D, n)) * 2 + 1).astype(np.float32)
    mu = rng.standard_normal((K, 3, D)).astype(np.float32)
    var = rng.uniform(0.5, 2.0, (K, 3, D)).astype(np.float32)
    ld = np.log(var.astype(np.float64)).sum(-1).astype(np.float32)
    g = pkg.GpuSweep(x, pkg.DIAG, seed=4)
    g.init_labels(K)
    g.set_params_diag(mu, var, ld, np.full(K, 1.0 / K, np.float32), np.full((K, 2), 0.5, np.float32))
    g.sample_labels(False)
    g.sample_sublabels()
    counts, sx, sxx = g.suff_stats()
    assert counts[:, 0].sum() == n and (counts[:, 0] == counts[:, 1] + counts[:, 2]).all()
    x64 = x.astype(np.float64)
    np.testing.assert_allclose(sx[:, 0].sum(0), x64.sum(1), rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(sxx[:, 0].sum(0), (x64 * x64).sum(1), rtol=1e-12)
    g.close()


def test_refusals(pkg):
    import scipy.sparse as sps
    E = pkg._lib
    x = np.random.default_rng(0).standard_normal((8, 500)).astype(np.float32)
    with pytest.raises(ValueError):
        pkg.GpuSweep(sps.csc_matrix(x), pkg.DIAG)
    g = pkg.GpuSweep(x, pkg.DIAG)
    for call in (lambda: g.set_hyper_multinomial(np.ones(8), 1.0), lambda: g.set_hyper_niw(1.0, np.zeros(8), 10.0, np.eye(8), 1.0),
                 lambda: g.sample_params(2), lambda: g.posterior_step(), lambda: g.get_params_niw(1),
                 lambda: g.get_params_multinomial(1), lambda: g.predict_multinomial(np.zeros((1, 8)), np.zeros(1)),
                 lambda: g.smart_project(1, np.ones(8), np.zeros(8)),
                 lambda: g.set_params_niw(np.zeros((1, 3, 8)), np.zeros((1, 3, 8, 8)), np.zeros((1, 3)), np.ones(1), np.ones((1, 2)))):
        with pytest.raises(E.DpmmError) as ei:
            call()
        assert ei.value.code == E.ESTATE
    g.close()


@pytest.mark.timeout(1500, method="thread")
@pytest.mark.parametrize("D", [128, 1024])
def test_fit_axis_aligned(pkg, D, tmp_path):
    from dpmmsubclusters_jl_b200 import checkpoint as CK, host as H, priors as P
    hyper = P.diag_niw_hyperparams(1.0, np.zeros(D), 10.0, np.ones(D))
    for seed in (1, 2, 3):
        x, z = axis_aligned_data(200_000, D, 20, seed, hyper)
        labels, clusters, *rest = pkg.fit(x, hyper, 10.0, iters=100, seed=seed, burnout=10)
        model = rest[-1]
        nmi = H.normalized_mutual_info(z, labels)
        print(f"diag fit D={D} seed={seed}: K={len(clusters)} NMI={nmi:.4f}")
        assert nmi >= 0.9 and abs(len(clusters) - 20) <= 3
        if seed == 1:
            lbl, probs = pkg.predict(model, x)
            assert (lbl == labels).mean() >= 0.99
            with pytest.raises(ValueError):
                pkg.predict(model, x, on_device=True)
    # checkpoint save and resume on the GPU
    x, z = axis_aligned_data(50_000, D, 8, 9, hyper)
    # (default burnout: a resume without a parameter file runs with the default settings)
    pkg.fit(x, hyper, 10.0, iters=20, seed=4, save_model=True, save_path=str(tmp_path) + "/", model_save_interval=10)
    fname = str(tmp_path / "checkpoint__20.npz")
    grp, mh, it, _, _ = CK.load_checkpoint(fname)
    assert it == 20 and isinstance(mh.distribution_hyper_params, P.diag_niw_hyperparams)
    resumed, iters, *_ = H.run_model_from_checkpoint(fname, verbose=False, data=x)
    assert len(iters) == 80
    assert H.normalized_mutual_info(z, resumed.group.sweep.get_labels()) >= 0.9


def test_two_gpu_statistics_at_d1000():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29617", os.path.join(ROOT, "tests", "mgpu_diag_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "MGPU_DIAG_OK" in out.stdout
