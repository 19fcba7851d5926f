"""The diagonal-covariance Gaussian prior on the CPU: its plugin functions against the NIW prior at D = 1 feature by
feature, its sampler's moments, the host loop on the oracle, checkpoints and parameter files, and what it refuses."""
import os

import numpy as np
import pytest
import scipy.sparse as sps

import dpmm_pkg
from oracle import diag_oracle as DO
from tests.diag_util import axis_aligned_data

pkg = dpmm_pkg.load()
from dpmmsubclusters_jl_b200 import checkpoint as CK, host as H, priors as P  # noqa: E402


def _random_prior_and_stats(D, seed):
    rng = np.random.default_rng(seed)
    hyper = P.diag_niw_hyperparams(rng.uniform(0.5, 3), rng.standard_normal(D), D % 5 + 4.0, rng.uniform(0.3, 3, D))
    N = 37
    pts = rng.standard_normal((D, N)) * 2 + 1
    ss = P.diag_niw_sufficient_statistics(float(N), pts.sum(1), (pts * pts).sum(1))
    return hyper, ss, rng


def _niw_at(hyper, ss, d):
    h = P.niw_hyperparams(hyper.κ, hyper.m[d:d + 1], hyper.ν, hyper.ψ[d:d + 1, None])
    s = P.niw_sufficient_statistics(ss.N, ss.points_sum[d:d + 1], ss.S_diag[d:d + 1, None])
    return h, s


@pytest.mark.parametrize("D", [1, 7, 300])
def test_prior_is_the_niw_prior_per_feature(D):
    hyper, ss, rng = _random_prior_and_stats(D, D)
    post = P.calc_posterior(hyper, ss)
    logml = P.log_marginal_likelihood(hyper, post, ss)
    x = rng.standard_normal((D, 50)) * 3
    pred = P.posterior_predictive(x, post)
    want_ml, want_pred = 0.0, np.zeros(50)
    for d in range(D):
        h, s = _niw_at(hyper, ss, d)
        p = P.calc_posterior(h, s)
        assert (p.κ, p.ν) == (post.κ, post.ν)
        np.testing.assert_allclose(post.m[d], p.m[0], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(post.ψ[d], p.ψ[0, 0], rtol=1e-12, atol=1e-12)
        want_ml += P.log_marginal_likelihood(h, p, s)
        want_pred += P.posterior_predictive(x[d:d + 1], p)
    assert abs(logml - want_ml) <= 1e-12 * max(1.0, abs(want_ml))
    np.testing.assert_allclose(pred, want_pred, rtol=1e-12, atol=1e-12 * np.abs(want_pred).max())
    # empty statistics leave the prior; aggregation adds every field
    assert P.calc_posterior(hyper, P.empty_suff_stats(hyper)) is hyper
    agg = P.aggregate_suff_stats(ss, ss)
    np.testing.assert_array_equal(agg.S_diag, 2 * ss.S_diag)
    assert agg.N == 2 * ss.N


def test_sampled_distribution_moments():
    rng = np.random.default_rng(1)
    hyper = P.diag_niw_hyperparams(2.0, np.array([0.0, 5.0, -3.0]), 10.0, np.array([1.0, 0.5, 4.0]))
    R = 100_000
    draws = [P.sample_distribution(hyper, rng) for _ in range(R)]
    mu = np.array([d.μ for d in draws], np.float64)
    var = np.array([d.σ2 for d in draws], np.float64)
    ld = np.array([d.logdetΣ for d in draws])
    np.testing.assert_allclose(ld, np.log(var).sum(1), rtol=1e-5, atol=1e-5)
    ev = hyper.ν * hyper.ψ / (hyper.ν - 2)                      # mean of the inverse-gamma sigma^2
    sv = ev * np.sqrt(2 / (hyper.ν - 4))                       # its standard deviation
    assert (np.abs(var.mean(0) - ev) <= 6 * sv / np.sqrt(R)).all(), (var.mean(0), ev)
    assert (np.abs(mu.mean(0) - hyper.m) <= 6 * np.sqrt(ev / hyper.κ / R)).all()
    np.testing.assert_allclose(mu.var(0), ev / hyper.κ, rtol=0.03)


def _oracle_factory(x, kind, seed, goff):
    return DO.DiagOracleSweep(x, kind, seed, goff)


def test_fit_on_the_oracle():
    hyper = P.diag_niw_hyperparams(1.0, np.zeros(20), 10.0, np.ones(20))
    x, z = axis_aligned_data(3000, 20, 5, 0, hyper)
    labels, clusters, *_ = pkg.fit(x, hyper, 10.0, iters=60, seed=3, burnout=10, sweep_factory=_oracle_factory)
    nmi = H.normalized_mutual_info(z, labels)
    assert nmi >= 0.9, (nmi, len(clusters))
    assert all(isinstance(c, P.diag_gaussian) for c in clusters)


def test_parameter_file_and_checkpoint_round_trip(tmp_path):
    hyper = P.diag_niw_hyperparams(1.0, np.zeros(6), 10.0, np.ones(6))
    x, z = axis_aligned_data(1500, 6, 3, 2, hyper)
    np.save(tmp_path / "pts.npy", x.T)
    pf = tmp_path / "params.jl"
    pf.write_text(f"""
data_path = "{tmp_path}/"
data_prefix = "pts"
iterations = 30
random_seed = 5
burnout_period = 5
alpha = 10.0
hyper_params = diag_niw_hyperparams(1.0, zeros(Float32, 6), 10.0, ones(Float32, 6))
enable_saving = true
model_save_interval = 20
save_path = "{tmp_path}/"
""")
    gp = CK.read_params(str(pf))
    assert isinstance(gp["hyper_params"], P.diag_niw_hyperparams) and gp["hyper_params"].m.shape == (6,)
    model, *_ = pkg.dp_parallel(str(pf), verbose=False, sweep_factory=_oracle_factory)
    assert H.normalized_mutual_info(z, model.group.sweep.get_labels()) >= 0.9
    fname = str(tmp_path / "checkpoint__20.npz")
    grp, mh, it, _, _ = CK.load_checkpoint(fname)
    assert it == 20 and isinstance(mh.distribution_hyper_params, P.diag_niw_hyperparams)
    c0 = grp["local_clusters"][0].cluster_params.cluster_params
    assert isinstance(c0.distribution, P.diag_gaussian) and c0.distribution.σ2.shape == (6,)
    assert isinstance(c0.suff_statistics, P.diag_niw_sufficient_statistics)
    assert isinstance(c0.posterior_hyperparams, P.diag_niw_hyperparams)
    # resume at iteration 21; a checkpoint of the resumed model restores its objects exactly
    resumed, *_ = H.run_model_from_checkpoint(fname, verbose=False, sweep_factory=_oracle_factory)
    assert H.normalized_mutual_info(z, resumed.group.sweep.get_labels()) >= 0.9
    again = CK.save_model(resumed, str(tmp_path) + "/", "again", 30, 0.0, str(pf))
    grp2, *_ = CK.load_checkpoint(again)
    np.testing.assert_array_equal(grp2["labels"], resumed.group.sweep.get_labels())
    assert len(grp2["local_clusters"]) == len(resumed.group.local_clusters)
    for c1, c2 in zip(resumed.group.local_clusters, grp2["local_clusters"]):
        for t1, t2 in ((c1.cluster_params.cluster_params, c2.cluster_params.cluster_params),
                       (c1.cluster_params.cluster_params_r, c2.cluster_params.cluster_params_r)):
            np.testing.assert_array_equal(t1.distribution.σ2, t2.distribution.σ2)
            np.testing.assert_array_equal(t1.distribution.μ, t2.distribution.μ)
            assert t1.distribution.logdetΣ == t2.distribution.logdetΣ
            np.testing.assert_array_equal(t1.suff_statistics.S_diag, t2.suff_statistics.S_diag)
            np.testing.assert_array_equal(t1.posterior_hyperparams.ψ, t2.posterior_hyperparams.ψ)
    lbl, probs = H.predict(resumed, x)
    assert (lbl == resumed.group.sweep.get_labels()).mean() >= 0.99
    np.testing.assert_allclose(probs.sum(1), 1.0, rtol=1e-5)


def test_refusals():
    hyper = P.diag_niw_hyperparams(1.0, np.zeros(4), 6.0, np.ones(4))
    x = np.random.default_rng(0).standard_normal((4, 100)).astype(np.float32)
    with pytest.raises(ValueError, match="sparse"):
        pkg.fit(sps.csc_matrix(x), hyper, 1.0, sweep_factory=_oracle_factory)
    with pytest.raises(ValueError, match="scatter matrix"):
        pkg.fit(x, hyper, 1.0, smart_splits=True, sweep_factory=_oracle_factory)
    with pytest.raises(ValueError, match="NIW and multinomial only|NIW and multinomial priors only"):
        pkg.fit(x, hyper, 1.0, device_params=True, sweep_factory=_oracle_factory)
