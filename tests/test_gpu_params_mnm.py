"""Device-side parameter step and predict of the multinomial prior on the GPU, through the C ABI:
deterministic parts (posterior alpha', log marginal likelihoods, merge table) against the NumPy prior plugin and the
reference's own checkpoint; the Dirichlet draws against their known moments; the device pack against the sweep
kernels' view of uploaded parameters; and fit() / predict() against the host-side paths."""
import os
import time
from types import SimpleNamespace

import numpy as np
import pytest

import dpmm_pkg
from oracle import dpmm_oracle as O
from tests.util import check_loglik, make_mnm_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    return dpmm_pkg.load()


def _setup(pkg, D, K, n, seed, alpha=10.0, prior=None):
    from dpmmsubclusters_jl_b200 import priors as P
    case = make_mnm_case(D, K, n, seed=seed)
    rng = np.random.default_rng(seed)
    lab = rng.integers(1, K + 1, n)
    sub = rng.integers(1, 3, n)
    sub[lab == K] = 1                                  # one side of the last cluster is empty
    hyper = P.multinomial_hyper(rng.uniform(0.3, 2.0, D) if prior is None else prior)
    g = pkg.GpuSweep(case["x"], pkg.MULTINOMIAL, seed=5)
    g.set_labels(lab); g.set_sublabels(sub)
    g.set_hyper_multinomial(hyper.α, alpha)
    return case, g, hyper, lab, sub, P


def _want_logml(P, hyper, n, sx):
    ss = P.make_suff_stats(hyper, n, sx)
    return P.log_marginal_likelihood(hyper, P.calc_posterior(hyper, ss), ss) if n > 0 else 0.0


@pytest.mark.parametrize("D,K,n", [(100, 20, 20000), (12, 3, 3000), (700, 4, 2000), (5, 1, 500)])
def test_posterior_logml_and_merge_table_match_the_prior_plugin(pkg, D, K, n):
    case, g, hyper, lab, sub, P = _setup(pkg, D, K, n, seed=D + K)
    counts, logml, merge = g.posterior_step(None, splittable=np.ones(K, bool))
    sc, sx, _ = g.suff_stats()
    np.testing.assert_array_equal(counts, sc)
    e = 1 if counts[K - 1, 1] == 0 else 2                 # the empty side of the last cluster
    assert counts[K - 1, e] == 0 and logml[K - 1, e] == 0.0
    for k in range(K):
        for s in range(3):
            want = _want_logml(P, hyper, sc[k, s], sx[k, s])
            assert abs(logml[k, s] - want) <= 1e-10 * max(1.0, abs(want)), (k, s, logml[k, s], want)
    for i in range(K):
        for j in range(K):
            if i < j and sc[i, 0] > 0 and sc[j, 0] > 0:
                ab = P.aggregate_suff_stats(P.make_suff_stats(hyper, sc[i, 0], sx[i, 0]),
                                            P.make_suff_stats(hyper, sc[j, 0], sx[j, 0]))
                want = P.log_marginal_likelihood(hyper, P.calc_posterior(hyper, ab), ab)
                assert abs(merge[i, j] - want) <= 1e-10 * max(1.0, abs(want)), (i, j, merge[i, j], want)
            elif merge is not None:
                assert np.isnan(merge[i, j])
    if K >= 2:
        c2, l2, _ = g.posterior_step([2, 1])
        np.testing.assert_array_equal(c2, counts[[1, 0]])
        np.testing.assert_array_equal(l2, logml[[1, 0]])
        g.params_merge(1, 2)
        c3, l3, _ = g.posterior_step([1], from_table=True)
        np.testing.assert_array_equal(c3[0], [counts[0, 0] + counts[1, 0], counts[0, 0], counts[1, 0]])
        np.testing.assert_allclose(l3[0], [merge[0, 1], logml[0, 0], logml[1, 0]], rtol=1e-12)
    g.close()


def test_device_posterior_on_the_reference_checkpoint(pkg, golden_dir):
    """Labels / sub-labels of the reference's multinomial checkpoint_20.jld2 with prior alpha = 1: the log marginal
    likelihoods must equal multinomial_prior.jl:34-39 evaluated on the posterior alpha' bytes the reference stored."""
    from dpmmsubclusters_jl_b200 import priors as P
    gm = np.load(os.path.join(golden_dir, "mnm_1k_checkpoint20.npz"))
    hyper = P.multinomial_hyper(np.ones(100, np.float32))
    g = pkg.GpuSweep(gm["x"], pkg.MULTINOMIAL)
    g.set_labels(gm["labels"]); g.set_sublabels(gm["sublabels"])
    g.set_hyper_multinomial(hyper.α, 10.0)
    counts, logml, _ = g.posterior_step(None)
    np.testing.assert_array_equal(counts, gm["counts"])
    for k in range(2):
        for s in range(3):
            stored = P.multinomial_hyper(gm["post_alpha"][k, s])
            want = P.log_marginal_likelihood(hyper, stored, None)
            assert abs(logml[k, s] - want) <= 1e-10 * max(1.0, abs(want)), (k, s, logml[k, s], want)
    g.close()


@pytest.mark.parametrize("D", [8, 100])
def test_device_draws_have_the_right_moments(pkg, D):
    """log p ~ log Dirichlet(alpha'):  E[p] = alpha' / sum alpha';  weights ~ Dir(N_1..N_K, alpha);
    lr ~ Dir(N_l + a/2, N_r + a/2).  Every log p is finite, also under a prior of alpha_d = 1e-3."""
    K, n, alpha, R = 3, 4000, 10.0, 300
    case, g, hyper, lab, sub, P = _setup(pkg, D, K, n, seed=7, alpha=alpha)
    g.posterior_step(None)
    sc, sx, _ = g.suff_stats()
    posts = np.array([[P.calc_posterior(hyper, P.make_suff_stats(hyper, sc[k, s], sx[k, s])).α for s in range(3)]
                      for k in range(K)], np.float64)
    p_acc = np.zeros((K, 3, D)); w_acc = np.zeros(K); lr_acc = np.zeros((K, 2))
    for _ in range(R):
        g.sample_params(K)
        lp, w, lr = g.get_params_multinomial(K)
        assert np.isfinite(lp).all()
        np.testing.assert_allclose(np.exp(lp.astype(np.float64)).sum(-1), 1.0, atol=1e-5)
        p_acc += np.exp(lp.astype(np.float64)); w_acc += w; lr_acc += lr
    A = posts.sum(-1, keepdims=True)
    m = posts / A
    sd = np.sqrt(m * (1 - m) / (A + 1) / R)
    assert (np.abs(p_acc / R - m) <= 6 * sd + 1e-6).all(), np.abs(p_acc / R - m).max()
    Ntot = sc[:, 0].sum() + alpha
    np.testing.assert_allclose(w_acc / R, sc[:, 0] / Ntot, atol=6 * np.sqrt(0.25 / Ntot / R) + 1e-4)
    want_lr = (sc[:, 1] + alpha / 2) / (sc[:, 1] + sc[:, 2] + alpha)
    np.testing.assert_allclose(lr_acc[:, 0] / R, want_lr, atol=0.01)
    # a sparse prior: most of the mass sits on few components, the rest far below Float32's smallest normal
    g.set_hyper_multinomial(np.full(D, 1e-3, np.float32), alpha)
    for _ in range(20):
        g.sample_params(K, from_prior=True)
        lp, _, _ = g.get_params_multinomial(K)
        assert np.isfinite(lp).all() and (lp <= 0).all()
        np.testing.assert_allclose(np.exp(lp.astype(np.float64)).sum(-1), 1.0, atol=1e-5)
    g.close()


@pytest.mark.parametrize("D,K", [(100, 20), (100, 40), (200, 5)])
def test_device_pack_feeds_the_sweep_like_uploaded_parameters(pkg, D, K):
    """The images the sweep kernels read after sample_params must be those dpmm_set_params_multinomial builds from the
    fetched parameters: label / sub-label log-likelihoods and draws bit for bit.  (100, 20) runs the tensor-core label
    kernel; K = 40 and D = 200 are past its limits."""
    n = 6000
    case, g, hyper, lab, sub, P = _setup(pkg, D, K, n, seed=D * K)
    rng = np.random.default_rng(1)
    u_label, u_sub = rng.random(n), rng.random(n)
    g.posterior_step(None)
    g.sample_params(K)

    def run():
        g.set_uniforms(u_label, u_sub, np.zeros(n, np.uint8))
        g.set_labels(lab); g.set_sublabels(sub)
        ll0, ll1 = g.debug_loglik(0), g.debug_loglik(1)
        g.sample_labels(False)
        g.sample_sublabels()
        return ll0, ll1, g.get_labels(), g.get_sublabels()

    a = run()
    lp, w, lr = g.get_params_multinomial(K)
    g.set_params_multinomial(lp, w, lr)
    b = run()
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()
    o = O.OracleSweep(case["x"], O.MULTINOMIAL, seed=5)
    o.set_params_multinomial(lp, w, lr)
    check_loglik(a[0], o.debug_loglik(0), "device-sampled parameters, label log-likelihood")
    g.close()


def _fit_nmi_k(H, x, labels, hyper, seeds, iters, burn, device_params):
    nmi, ks = [], []
    for seed in seeds:
        out = H.fit(x, hyper, 10.0, iters=iters, seed=seed, burnout=burn, device_params=device_params)
        nmi.append(H.normalized_mutual_info(labels, out[0])); ks.append(len(out[1]))
    return np.array(nmi), np.array(ks)


def test_fit_device_and_host_parameter_paths_agree_over_seeds(pkg):
    """N = 1e4, D = 100, K = 10 (10 seeds) and a 1e5-point slice of the C3 shape (D = 100, K = 20; 4 seeds): mean NMI
    and mean final K of fit() with the parameter step on the device and on the host (NumPy)."""
    from dpmmsubclusters_jl_b200 import host as H
    hyper = pkg.multinomial_hyper(np.ones(100, np.float32))
    for N, K, seeds in [(10 ** 4, 10, range(10)), (10 ** 5, 20, range(4))]:
        x, labels, _ = pkg.generate_mnmm_data(N, 100, K, 50, np.random.default_rng(5))
        dev = _fit_nmi_k(H, x, labels, hyper, seeds, 60, 10, True)
        host = _fit_nmi_k(H, x, labels, hyper, seeds, 60, 10, False)
        print(f"N={N}: device NMI {np.round(dev[0], 3)} K {dev[1]}; host NMI {np.round(host[0], 3)} K {host[1]}")
        assert abs(dev[0].mean() - host[0].mean()) < 0.05
        assert abs(dev[1].mean() - host[1].mean()) <= 1.5
    # test/module_tests.jl:49-60 on the device path
    x, labels, _ = pkg.generate_mnmm_data(10 ** 3, 100, 20, 50, np.random.default_rng(0))
    out = pkg.fit(x, hyper, 1e5, iters=39, seed=3, gt=labels, device_params=True)
    assert len(out[1]) > 1


@pytest.mark.timeout(300, method="thread")
def test_full_size_c3_fit_from_one_cluster(pkg):
    """fit() on the full C3 shape (N = 1e6, D = 100, K_true = 20) from K = 1 with the parameter step on the device."""
    from dpmmsubclusters_jl_b200.host import normalized_mutual_info
    x, z, _ = pkg.generate_mnmm_data(10 ** 6, 100, 20, 50, np.random.default_rng(0))
    hyper = pkg.multinomial_hyper(np.ones(100, np.float32))
    t0 = time.perf_counter()
    labels, clusters, weights, iter_count, *_ = pkg.fit(x, hyper, 10.0, iters=100, seed=1, burnout=20,
                                                        device_params=True)
    wall = time.perf_counter() - t0
    K = len(clusters)
    assert K == len(weights) == len(np.unique(labels)) and labels.min() == 1 and labels.max() == K
    assert float(np.sum(weights, dtype=np.float64)) <= 1.0 + 1e-6
    assert K > 1
    print(f"C3 device params: K={K} NMI={normalized_mutual_info(z, labels):.4f} "
          f"{len(iter_count) / sum(iter_count):.1f} it/s in the loop, {len(iter_count) / wall:.1f} it/s whole call")


def _numpy_scores(model, x):
    """parr of host.predict's NumPy branch (Float32)."""
    from dpmmsubclusters_jl_b200 import priors as P
    cl = model.group.local_clusters
    parr = np.zeros((x.shape[1], len(cl)), np.float32)
    for k, c in enumerate(cl):
        parr[:, k] = P.posterior_predictive(x, c.cluster_params.cluster_params.posterior_hyperparams)
    with np.errstate(divide="ignore"):
        parr += np.log(np.asarray(model.group.weights, np.float32))[None, :]
    return parr


def _check_predict(H, model, x):
    lg, pg = H.predict(model, x, on_device=True)
    lh, ph = H.predict(model, x, on_device=False)
    bad = np.nonzero(lg != lh)[0]
    if bad.size:
        s = np.sort(_numpy_scores(model, x[:, bad]), axis=1)
        assert (s[:, -1] - s[:, -2] <= np.spacing(np.abs(s[:, -1]))).all(), bad
    np.testing.assert_allclose(pg, ph, atol=1e-6)
    np.testing.assert_allclose(pg.sum(1), 1.0, atol=1e-5)
    return lg, int(bad.size)


def test_predict_on_device_matches_the_numpy_posterior_predictive(pkg):
    from dpmmsubclusters_jl_b200 import host as H, priors as P
    hyper = pkg.multinomial_hyper(np.ones(100, np.float32))
    x, z, _ = pkg.generate_mnmm_data(20000, 100, 20, 50, np.random.default_rng(3))
    out = H.fit(x, hyper, 10.0, iters=40, seed=2, burnout=10, device_params=True)
    model = out[-1]
    xnew, _, _ = pkg.generate_mnmm_data(5000, 100, 20, 50, np.random.default_rng(4))
    _, nb = _check_predict(H, model, xnew)
    lt, nt = _check_predict(H, model, x)
    print(f"D=100 K={len(out[1])}: near-tie mismatches {nb} (new points), {nt} (training points); "
          f"predict == fit labels on {(lt == out[0]).mean():.4f}")
    # K x D far past one shared-memory table (40 x 1000 Float64 = 320 KB): the score kernel tiles over clusters
    D, K = 1000, 40
    case = make_mnm_case(D, K, 3000, seed=11)
    rng = np.random.default_rng(12)
    cl = [SimpleNamespace(cluster_params=SimpleNamespace(cluster_params=SimpleNamespace(
        posterior_hyperparams=P.multinomial_hyper(rng.uniform(0.5, 60.0, D))))) for _ in range(K)]
    sw = pkg.GpuSweep(case["x"][:, :200], pkg.MULTINOMIAL)
    big = SimpleNamespace(group=SimpleNamespace(local_clusters=cl, weights=rng.dirichlet(np.ones(K)).astype(np.float32),
                                                sweep=sw))
    _check_predict(H, big, case["x"])
    sw.close()


PARAMS_JL = """
data_path = "{path}"
data_prefix = "pts"
iterations = 30
hard_clustering = false
initial_clusters = 1
argmax_sample_stop = 5
split_stop = 5
random_seed = 4
max_split_iter = 20
burnout_period = 5
max_clusters = Inf
α = 10.0
hyper_params = multinomial_hyper(ones(Float32,30))
outlier_mod = 0.0
enable_saving = true
model_save_interval = 10
save_path = "{path}"
overwrite_prec = false
save_file_prefix = "checkpoint_"
smart_splits = false
"""


def test_checkpoint_save_and_resume_on_the_device_path(pkg, tmp_path):
    """A multinomial fit with the parameter step on the device saves checkpoints (run_model :395-399) and resumes from
    one (run_model_from_checkpoint :428-449); the clusters it rebuilds carry multinomial_dist distributions."""
    from dpmmsubclusters_jl_b200 import host as H, priors as P
    from dpmmsubclusters_jl_b200 import checkpoint as CK
    x, labels, _ = pkg.generate_mnmm_data(5000, 30, 5, 50, np.random.default_rng(8))
    np.save(tmp_path / "pts.npy", x.T)
    f = tmp_path / "global_params.jl"
    f.write_text(PARAMS_JL.format(path=str(tmp_path) + "/"))
    dp, ic, nmi, _, kh = H.dp_parallel(str(f), verbose=False, gt=labels, device_params=True)
    assert len(ic) == 30
    for c in dp.group.local_clusters:
        assert isinstance(c.cluster_params.cluster_params.distribution, P.multinomial_dist)
    grp, mh, it, _, _ = CK.load_checkpoint(str(tmp_path / "checkpoint__20.npz"))
    assert it == 20 and isinstance(mh.distribution_hyper_params, P.multinomial_hyper)
    assert len(grp["local_clusters"]) == kh[19]
    for k, c in enumerate(grp["local_clusters"]):
        assert int((grp["labels"] == k + 1).sum()) == c.points_count
        assert isinstance(c.cluster_params.cluster_params.distribution, P.multinomial_dist)
    dp2, ic2, nmi2, _, kh2 = H.run_model_from_checkpoint(str(tmp_path / "checkpoint__20.npz"), verbose=False, gt=labels,
                                                        device_params=True)
    assert len(ic2) == 10 and kh2[-1] == len(dp2.group.local_clusters)
    for c in dp2.group.local_clusters:
        assert isinstance(c.cluster_params.cluster_params.distribution, P.multinomial_dist)
    print(f"fit: final K {kh[-1]}, NMI {nmi[-1]:.3f}; resumed at 20: final K {kh2[-1]}, NMI {nmi2[-1]:.3f}")


def test_error_paths(pkg):
    from dpmmsubclusters_jl_b200 import _lib as L
    case = make_mnm_case(8, 2, 500, seed=1)
    g = pkg.GpuSweep(case["x"], pkg.MULTINOMIAL)
    with pytest.raises(L.DpmmError) as e:
        g.posterior_step(None)
    assert e.value.code == L.ESTATE and "dpmm_set_hyper_multinomial" in str(e.value)
    for bad in (np.zeros(8), np.full(8, np.nan), np.full(8, np.inf), -np.ones(8)):
        with pytest.raises(L.DpmmError) as e:
            g.set_hyper_multinomial(bad, 1.0)
        assert e.value.code == L.EINVAL
    with pytest.raises(L.DpmmError) as e:
        g.set_hyper_multinomial(np.ones(8), 0.0)
    assert e.value.code == L.EINVAL
    g.set_hyper_multinomial(np.ones(8), 1.0)
    g.set_labels(np.ones(500, np.int64)); g.set_sublabels(np.ones(500, np.int64))
    g.posterior_step(None)
    g.sample_params(1)
    with pytest.raises(L.DpmmError) as e:
        g.get_params_niw(1)
    assert e.value.code == L.ESTATE
    with pytest.raises(L.DpmmError) as e:
        g.predict_niw(np.zeros((1, 8, 8)), np.zeros((1, 8)), np.zeros(1), np.ones(1))
    assert e.value.code == L.ESTATE
    g.close()
    x = np.random.default_rng(0).standard_normal((3, 300)).astype(np.float32)
    h = pkg.GpuSweep(x, pkg.NIW)
    for call in (lambda: h.set_hyper_multinomial(np.ones(3), 1.0), lambda: h.get_params_multinomial(1),
                 lambda: h.predict_multinomial(np.zeros((1, 3)), np.zeros(1))):
        with pytest.raises(L.DpmmError) as e:
            call()
        assert e.value.code == L.ESTATE
    h.close()
