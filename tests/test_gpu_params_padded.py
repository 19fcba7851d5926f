"""Device-side parameter step of NIW models whose D has no kernels of its own (the context runs zero-padded to the next
instantiated width): posterior, log marginal likelihoods and merge table against the NumPy prior plugin, the moments of
the draws, the log-likelihoods the sweep computes from them, and fit() / predict / smart splits / checkpoint resume
with the parameter step on the device."""
import numpy as np
import pytest

import dpmm_pkg
from oracle import dpmm_oracle as O
from tests.util import check_loglik, make_niw_case

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900, method="thread")]


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    return dpmm_pkg.load()


def _setup(pkg, D, K, n, seed, alpha=10.0):
    from dpmmsubclusters_jl_b200 import priors as P
    case = make_niw_case(D, K, n, seed=seed, spread=4.0)
    rng = np.random.default_rng(seed)
    lab = rng.integers(1, K + 1, n)
    sub = rng.integers(1, 3, n)
    hyper = P.niw_hyperparams(1.5, rng.standard_normal(D) * 0.3, D + 3.5, np.eye(D) * 1.3 + 0.1)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=5)
    g.set_labels(lab); g.set_sublabels(sub)
    g.set_hyper_niw(hyper.κ, hyper.m, hyper.ν, hyper.ψ, alpha)
    return case, g, hyper, lab, sub, P


@pytest.mark.parametrize("D,K,n", [(9, 4, 3000), (20, 5, 4000), (33, 3, 3000), (50, 4, 5000), (63, 3, 4000)])
def test_padded_posterior_logml_and_merge_table_match_the_prior_plugin(pkg, D, K, n):
    case, g, hyper, lab, sub, P = _setup(pkg, D, K, n, seed=D + K)
    counts, logml, merge = g.posterior_step(None, splittable=np.ones(K, bool))
    sc, sx, sxx = g.suff_stats()
    assert sx.shape == (K, 3, D) and sxx.shape == (K, 3, D, D)
    np.testing.assert_array_equal(counts, sc)
    # (the absolute term covers one Float32 rounding of log_multivariate_gamma, accumulated in Float32 on both sides)
    for k in range(K):
        for s in range(3):
            ss = P.make_suff_stats(hyper, sc[k, s], sx[k, s], sxx[k, s])
            want = P.log_marginal_likelihood(hyper, P.calc_posterior(hyper, ss), ss) if sc[k, s] > 0 else 0.0
            assert abs(logml[k, s] - want) <= 1e-9 * max(1.0, abs(want)) + 2e-3, (k, s, logml[k, s], want)
    for i in range(K):
        for j in range(K):
            if i < j and sc[i, 0] > 0 and sc[j, 0] > 0:
                a = P.make_suff_stats(hyper, sc[i, 0], sx[i, 0], sxx[i, 0])
                b = P.make_suff_stats(hyper, sc[j, 0], sx[j, 0], sxx[j, 0])
                ab = P.aggregate_suff_stats(a, b)
                want = P.log_marginal_likelihood(hyper, P.calc_posterior(hyper, ab), ab)
                assert abs(merge[i, j] - want) <= 1e-9 * abs(want) + 2e-3, (i, j, merge[i, j], want)
            else:
                assert np.isnan(merge[i, j])
    # restricted call + table merge: cluster 1 <- {1 + 2, 1, 2}
    c2, l2, _ = g.posterior_step([2, 1])
    np.testing.assert_array_equal(c2, counts[[1, 0]])
    np.testing.assert_allclose(l2, logml[[1, 0]], rtol=5e-6, atol=1e-6)
    g.params_merge(1, 2)
    c3, l3, _ = g.posterior_step([1], from_table=True)
    np.testing.assert_array_equal(c3[0], [counts[0, 0] + counts[1, 0], counts[0, 0], counts[1, 0]])
    np.testing.assert_allclose(l3[0], [merge[0, 1], logml[0, 0], logml[1, 0]], rtol=5e-6, atol=1e-6)
    g.close()


@pytest.mark.parametrize("D", [10, 50])
def test_padded_device_draws_have_the_right_moments_and_feed_the_sweep(pkg, D):
    """Sigma ~ IW(nu', nu' psi')  =>  E[invSigma] = psi'^-1;  mu | Sigma ~ N(m', Sigma / kappa'); the arrays come back at
    the caller's D, and the sweep's log-likelihoods of them equal the oracle's on the caller's D features."""
    K, n, alpha = 3, 4000, 10.0
    case, g, hyper, lab, sub, P = _setup(pkg, D, K, n, seed=7, alpha=alpha)
    counts, logml, _ = g.posterior_step(None)
    sc, sx, sxx = g.suff_stats()
    R = 300
    inv_acc = np.zeros((K, 3, D, D)); w_acc = np.zeros(K)
    z_acc = np.zeros((K, 3, D)); z2_acc = np.zeros((K, 3, D))
    posts = [[P.calc_posterior(hyper, P.make_suff_stats(hyper, sc[k, s], sx[k, s], sxx[k, s])) for s in range(3)] for k in range(K)]
    for r in range(R):
        g.sample_params(K)
        mu, lf, ld, w, lr = g.get_params_niw(K)
        assert mu.shape == (K, 3, D) and lf.shape == (K, 3, D, D) and ld.shape == (K, 3)
        assert np.isfinite(mu).all() and np.isfinite(lf).all() and np.isfinite(ld).all()
        L = np.tril(lf)
        inv = L @ np.swapaxes(L, -1, -2)
        inv_acc += inv; w_acc += w
        np.testing.assert_allclose(ld, -np.linalg.slogdet(inv)[1], rtol=2e-5, atol=1e-4)
        for k in range(K):
            for s in range(3):
                zz = np.sqrt(posts[k][s].κ) * (L[k, s].T @ (mu[k, s] - posts[k][s].m))
                z_acc[k, s] += zz; z2_acc[k, s] += zz * zz
    for k in range(K):
        for s in range(3):
            want = np.linalg.inv(posts[k][s].ψ)
            got = inv_acc[k, s] / R
            scale = np.sqrt(np.outer(np.diag(want), np.diag(want)))
            assert np.abs(got - want).max() / scale.max() < 6 * np.sqrt(2.0 / (posts[k][s].ν * R)) + 1e-3
            assert np.abs(z_acc[k, s] / R).max() < 5 / np.sqrt(R)
            assert np.abs(z2_acc[k, s] / R - 1).max() < 6 * np.sqrt(2.0 / R)
    Ntot = sc[:, 0].sum() + alpha
    np.testing.assert_allclose(w_acc / R, sc[:, 0] / Ntot, atol=6 * np.sqrt(0.25 / Ntot / R) + 1e-4)
    # padding never leaks into a likelihood: label and sub-label log-likelihoods vs the oracle on the fetched values
    o = O.OracleSweep(case["x"], O.NIW, seed=5)
    o.set_labels(lab); o.set_sublabels(sub)
    o.set_params_niw(mu, inv.astype(np.float32), ld, w, lr)
    check_loglik(g.debug_loglik(0), o.debug_loglik(0), "device-sampled parameters, label log-likelihood")
    check_loglik(g.debug_loglik(1), o.debug_loglik(1), "device-sampled parameters, sub-label log-likelihood")
    # draws from the prior as well
    g.sample_params(K, from_prior=True)
    mu, lf, ld, _, _ = g.get_params_niw(K)
    assert mu.shape == (K, 3, D) and lf.shape == (K, 3, D, D) and np.isfinite(ld).all()
    g.close()


def test_padded_fit_device_and_host_parameter_paths_agree_over_seeds(pkg):
    """fit(x, 10.0) with the defaults at widths without their own kernels: final K and NMI with the parameter step
    on the device vs on the host (NumPy) over seeds."""
    from dpmmsubclusters_jl_b200 import host as H
    for D in (10, 20, 50):
        x, labels, _, _ = pkg.generate_gaussian_data(20000, D, 8, 100.0, np.random.default_rng(D))
        out = H.fit(x, 10.0, iters=40, seed=0, burnout=10)                   # the default path: device parameters
        assert out[1][0].μ.shape == (D,) and out[1][0].invΣ.shape == (D, D)
        res = {}
        for mode in (True, False):
            nmi, ks = [], []
            for seed in range(6):
                out = H.fit(x, 10.0, iters=60, seed=seed, burnout=10, device_params=mode)
                nmi.append(H.normalized_mutual_info(labels, out[0])); ks.append(len(out[1]))
            res[mode] = (np.array(nmi), np.array(ks))
        print(f"D={D}: device NMI {np.round(res[True][0], 3)} K {res[True][1]}; "
              f"host NMI {np.round(res[False][0], 3)} K {res[False][1]}")
        assert abs(res[True][0].mean() - res[False][0].mean()) < 0.05
        assert abs(res[True][1].mean() - res[False][1].mean()) <= 1.5


def test_padded_smart_splits_checkpoint_and_predict_on_the_device_path(pkg, tmp_path):
    from dpmmsubclusters_jl_b200 import host as H
    from dpmmsubclusters_jl_b200 import priors as P
    D, K = 20, 6
    x, labels, _, _ = pkg.generate_gaussian_data(12000, D, K, 100.0, np.random.default_rng(3))
    out = H.fit(x, 10.0, iters=60, seed=11, burnout=5, gt=labels, smart_splits=True, device_params=True)
    assert H.normalized_mutual_info(labels, out[0]) > 0.9
    # checkpoint at iteration 20, resumed on the device path
    H.dp_parallel(x, P.niw_hyperparams(1.0, np.zeros(D), D + 3, np.eye(D)), 10.0, iters=30, seed=4, verbose=False,
                  burnout=5, gt=labels, save_model=True, save_path=str(tmp_path) + "/", model_save_interval=20,
                  device_params=True)
    dp2, ic2, nmi2, _, _ = H.run_model_from_checkpoint(str(tmp_path / "checkpoint__20.npz"), verbose=False, gt=labels,
                                                       data=x, device_params=True)
    # the resumed run starts from the stored labels: its first NMI is already that of iteration ~20
    assert len(ic2) > 0 and nmi2[0] > 0.8 and nmi2[-1] > 0.9
    for c in dp2.group.local_clusters:
        assert c.cluster_params.cluster_params.distribution.μ.shape == (D,)
    # predict on the device against NumPy
    model = out[-1]
    xnew, _, _, _ = pkg.generate_gaussian_data(5000, D, K, 100.0, np.random.default_rng(4))
    xnew = np.concatenate([xnew, x[:, :3000]], axis=1)
    lg, pg = H.predict(model, xnew, on_device=True)
    lh, ph = H.predict(model, xnew, on_device=False)
    assert (lg == lh).mean() > 0.999
    np.testing.assert_allclose(pg, ph, atol=2e-3)


def test_padded_set_hyper_niw_validates_at_the_callers_dimension(pkg):
    from dpmmsubclusters_jl_b200 import _lib as E
    D = 10                                                   # the context runs at 12
    x = np.random.default_rng(0).standard_normal((D, 500)).astype(np.float32)
    g = pkg.GpuSweep(x, pkg.NIW, seed=1)
    g.set_hyper_niw(1.0, np.zeros(D), D - 0.5, np.eye(D), 1.0)      # nu > D - 1 at the caller's D
    for nu, psi in [(D - 1.0, np.eye(D)), (D + 3.0, np.diag(np.r_[np.ones(D - 1), -1.0]))]:
        with pytest.raises(E.DpmmError) as ei:
            g.set_hyper_niw(1.0, np.zeros(D), nu, psi, 1.0)
        assert ei.value.code == E.EINVAL
    g.close()
