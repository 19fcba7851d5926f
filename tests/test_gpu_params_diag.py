"""Device-side parameter step of the diagonal Gaussian prior on the GPU, through the C ABI: posteriors, log marginal
likelihoods and the merge table against the NumPy prior plugin; the draws against their known moments; the device pack
against the images dpmm_set_params_diag builds from the fetched parameters; the D = 16 384 / K = 1 024 limit; fit(),
checkpoints and two GPUs with device_params=True."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import dpmm_pkg
from tests.diag_util import axis_aligned_data, make_diag_case

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    return dpmm_pkg.load()


def _setup(pkg, D, K, n, seed, alpha=10.0, offset=0.0, nu=None):
    """A diagonal context with random labels / sub-labels (the left side of the last cluster empty) and a random
    diag_niw_hyperparams set on the device."""
    from dpmmsubclusters_jl_b200 import priors as P
    case = make_diag_case(D, K, n, seed=seed, offset=offset)
    rng = np.random.default_rng(seed)
    lab = rng.integers(1, K + 1, n)
    sub = rng.integers(1, 3, n)
    sub[lab == K] = 2
    hyper = P.diag_niw_hyperparams(rng.uniform(0.05, 2.0), rng.standard_normal(D) + offset,
                                   rng.uniform(2.5, 20.0) if nu is None else nu, rng.uniform(0.3, 3.0, D))
    g = pkg.GpuSweep(case["x"], pkg.DIAG, seed=5)
    g.set_labels(lab); g.set_sublabels(sub)
    g.set_hyper_diag(hyper.κ, hyper.m, hyper.ν, hyper.ψ, alpha)
    return case, g, hyper, P


def _ss(P, hyper, c, sx, sxx):
    return P.make_suff_stats(hyper, c, sx, sxx)


def _want_logml(P, hyper, ss):
    return P.log_marginal_likelihood(hyper, P.calc_posterior(hyper, ss), ss) if ss.N > 0 else 0.0


def _close(got, want, what):
    assert abs(got - want) <= 1e-9 * max(1.0, abs(want)), (what, got, want)


@pytest.mark.parametrize("D,K,n,offset", [(1, 3, 3000, 1e3), (128, 20, 20000, 1e3), (128, 20, 20000, 0.0),
                                          (4096, 8, 3000, 0.0)])
def test_posterior_logml_and_merge_table_match_the_prior_plugin(pkg, D, K, n, offset):
    """offset = 1e3: every mean 10^3 sigma from the origin, where psi' keeps a millionth of the size of its terms."""
    case, g, hyper, P = _setup(pkg, D, K, n, seed=D + K, offset=offset)
    counts, logml, merge = g.posterior_step(None, splittable=np.ones(K, bool))
    sc, sx, sxx = g.suff_stats()
    np.testing.assert_array_equal(counts, sc)
    assert counts[K - 1, 1] == 0 and logml[K - 1, 1] == 0.0          # the empty side
    ss = [[_ss(P, hyper, sc[k, s], sx[k, s], sxx[k, s]) for s in range(3)] for k in range(K)]
    for k in range(K):
        for s in range(3):
            _close(logml[k, s], _want_logml(P, hyper, ss[k][s]), ("logml", k, s))
    for i in range(K):
        for j in range(K):
            if i < j and sc[i, 0] > 0 and sc[j, 0] > 0:
                _close(merge[i, j], _want_logml(P, hyper, P.aggregate_suff_stats(ss[i][0], ss[j][0])), ("merge", i, j))
            else:
                assert np.isnan(merge[i, j])
    if K >= 3:
        # restricted update, then merge 1 <- {1 + 3, 1, 3} on the table and re-evaluate from it
        c2, l2, _ = g.posterior_step([1, 3])
        np.testing.assert_array_equal(c2, sc[[0, 2]])
        for a_ in range(2):
            for s in range(3):
                _close(l2[a_, s], logml[2 * a_, s], ("restricted", a_, s))
        g.params_merge(1, 3)
        c3, l3, _ = g.posterior_step([1], from_table=True)
        assert tuple(c3[0]) == (sc[0, 0] + sc[2, 0], sc[0, 0], sc[2, 0])
        _close(l3[0, 0], merge[0, 2], "merged c")
        assert l3[0, 1] == l2[0, 0] and l3[0, 2] == l2[1, 0]          # the same table rows, now as l and r
    g.close()


def test_draws_have_the_moments_of_the_host_sampler(pkg):
    """sigma^2 = nu' psi' / chi^2_nu', mu ~ N(m', sigma^2 / kappa'):  E[1/sigma^2] = 1/psi', E[mu] = m',
    Var mu = E[sigma^2] / kappa' (checked as (mu - m') sqrt(kappa' / sigma^2) ~ N(0, 1)); weights and sub-cluster
    weights as the Dirichlet draws of the other priors.  Every draw is finite with sigma^2 > 0, also under nu = 0.5."""
    D, K, n, alpha, R = 96, 3, 600, 10.0, 200
    case, g, hyper, P = _setup(pkg, D, K, n, seed=7, alpha=alpha)
    g.posterior_step(None)
    sc, sx, sxx = g.suff_stats()
    posts = [[P.calc_posterior(hyper, _ss(P, hyper, sc[k, s], sx[k, s], sxx[k, s])) for s in range(3)] for k in range(K)]
    psi = np.array([[p.ψ for p in r] for r in posts])
    m = np.array([[p.m for p in r] for r in posts])
    kap = np.array([[p.κ for p in r] for r in posts])
    nu = np.array([[p.ν for p in r] for r in posts])
    prec, z, w_acc, lr_acc = [], [], np.zeros(K), np.zeros((K, 2))
    for _ in range(R):
        g.sample_params(K)
        mu, var, ld, w, lr = g.get_params_diag(K)
        assert np.isfinite(mu).all() and np.isfinite(var).all() and (var > 0).all()
        np.testing.assert_allclose(ld, np.log(var.astype(np.float64)).sum(-1), rtol=1e-6, atol=1e-5)
        v64 = var.astype(np.float64)
        prec.append(psi / v64)
        z.append((mu.astype(np.float64) - m) * np.sqrt(kap[..., None] / v64))
        w_acc += w; lr_acc += lr
    prec, z = np.array(prec), np.array(z)                 # [R, K, 3, D]
    # per distribution, pooled over R draws x D features: 1/sigma^2 * psi' has mean 1 and variance 2 / nu'
    se = np.sqrt(2.0 / nu / (R * D))
    assert (np.abs(prec.mean(axis=(0, 3)) - 1.0) <= 6 * se).all(), prec.mean(axis=(0, 3))
    assert (np.abs(z.mean(axis=(0, 3))) <= 6 / np.sqrt(R * D)).all(), z.mean(axis=(0, 3))
    assert (np.abs(z.var(axis=(0, 3)) - 1.0) <= 6 * np.sqrt(2.0 / (R * D))).all(), z.var(axis=(0, 3))
    Ntot = sc[:, 0].sum() + alpha
    np.testing.assert_allclose(w_acc / R, sc[:, 0] / Ntot, atol=6 * np.sqrt(0.25 / Ntot / R) + 1e-4)
    want_lr = (sc[:, 1] + alpha / 2) / (sc[:, 1] + sc[:, 2] + alpha)
    np.testing.assert_allclose(lr_acc[:, 0] / R, want_lr, atol=0.02)
    # a prior of nu = 0.5: chi^2 draws of shape 1/4 (the boosted Gamma), heavy-tailed sigma^2
    g.set_hyper_diag(hyper.κ, hyper.m, 0.5, hyper.ψ, alpha)
    prec = []
    for _ in range(50):
        g.sample_params(K, from_prior=True)
        mu, var, ld, _, _ = g.get_params_diag(K)
        assert np.isfinite(mu).all() and np.isfinite(var).all() and (var > 0).all() and np.isfinite(ld).all()
        prec.append(hyper.ψ / var.astype(np.float64))
    prec = np.array(prec)
    assert abs(prec.mean() - 1.0) <= 6 * np.sqrt(2.0 / 0.5 / prec.size), prec.mean()
    g.close()


@pytest.mark.parametrize("D,K", [(128, 20), (1024, 300)])
def test_device_images_equal_those_of_uploaded_parameters(pkg, D, K):
    """sample_params -> get_params_diag -> set_params_diag on a second context: bit-identical label and sub-label
    log-likelihoods and identical draws.  (128, 20) runs the thread-per-point label kernel, (1024, 300) the streaming
    one."""
    n = 20000
    case, a, hyper, P = _setup(pkg, D, K, n, seed=D + K)
    a.posterior_step(None)
    a.sample_params(K)
    mu, var, ld, w, lr = a.get_params_diag(K)
    b = pkg.GpuSweep(case["x"], pkg.DIAG, seed=5)
    b.set_params_diag(mu, var, ld, w, lr)
    rng = np.random.default_rng(1)
    u_label, u_sub = rng.random(n), rng.random(n)
    lab = a.get_labels()
    out = []
    for g in (a, b):
        g.set_uniforms(u_label, u_sub, None)
        g.set_labels(lab)
        ll0, ll1 = g.debug_loglik(0), g.debug_loglik(1)
        g.sample_labels(False)
        g.sample_sublabels()
        out.append((ll0, ll1, g.get_labels(), g.get_sublabels()))
    for x, y in zip(*out):
        assert x.tobytes() == y.tobytes()
    assert np.isfinite(out[0][0]).all()
    a.close(); b.close()


def test_limits_d16384_k1024(pkg):
    """set_hyper_diag + posterior_step with the full merge table + sample_params at D = 16 384, K = 1 024."""
    D, K, n = 16384, 1024, 4096
    rng = np.random.default_rng(3)
    from dpmmsubclusters_jl_b200 import priors as P
    x = (rng.standard_normal((D, n)) * 2 + 1).astype(np.float32)
    lab = np.arange(n) % K + 1
    sub = rng.integers(1, 3, n)
    hyper = P.diag_niw_hyperparams(1.0, np.zeros(D), 10.0, np.ones(D))
    g = pkg.GpuSweep(x, pkg.DIAG, seed=4)
    g.set_labels(lab); g.set_sublabels(sub)
    g.set_hyper_diag(hyper.κ, hyper.m, hyper.ν, hyper.ψ, 10.0)
    g.posterior_step(None, splittable=np.ones(K, bool))           # warm-up (allocations, module load)
    g.sample_params(K); g.sync()
    t0 = time.perf_counter()
    counts, logml, merge = g.posterior_step(None, splittable=np.ones(K, bool))
    t1 = time.perf_counter()
    g.sample_params(K); g.sync()
    t2 = time.perf_counter()
    mu, var, ld, w, lr = g.get_params_diag(K)
    assert counts[:, 0].sum() == n and np.isfinite(logml).all()
    iu = np.triu_indices(K, 1)
    assert np.isfinite(merge[iu]).all()
    assert np.isfinite(mu).all() and (var > 0).all() and np.isfinite(var).all() and np.isfinite(ld).all()
    sc, sx, sxx = g.suff_stats([1, K])
    for a, k in enumerate((0, K - 1)):
        ss = [_ss(P, hyper, sc[a, s], sx[a, s], sxx[a, s]) for s in range(3)]
        for s in range(3):
            _close(logml[k, s], _want_logml(P, hyper, ss[s]), ("limit logml", k, s))
    _close(merge[0, K - 1], _want_logml(P, hyper, P.aggregate_suff_stats(
        _ss(P, hyper, sc[0, 0], sx[0, 0], sxx[0, 0]), _ss(P, hyper, sc[1, 0], sx[1, 0], sxx[1, 0]))), "limit merge")
    tables = 2 * 3 * K * (1 + 2 * D) * 8 + 2 * 3 * K * 4 * 8 + 3 * K * (2 * D + 1) * 4
    print(f"diag D={D} K={K}: posterior step + merge table {1e3 * (t1 - t0):.1f} ms, sample_params "
          f"{1e3 * (t2 - t1):.1f} ms; parameter-step tables {tables / 2 ** 30:.2f} GiB")
    g.close()


def _fit(pkg, x, hyper, seed, device_params, **kw):
    return pkg.fit(x, hyper, 10.0, iters=100, seed=seed, burnout=10, device_params=device_params, **kw)


@pytest.mark.timeout(1800, method="thread")
@pytest.mark.parametrize("D", [128, 1024])
def test_fit_device_and_host_parameter_paths_over_seeds(pkg, D):
    """test_fit_axis_aligned's floors (NMI >= 0.9, |K - 20| <= 3) on both paths; the device path returns finite
    diag_gaussian clusters and calculate_posterior runs on its model."""
    from dpmmsubclusters_jl_b200 import host as H, priors as P
    hyper = P.diag_niw_hyperparams(1.0, np.zeros(D), 10.0, np.ones(D))
    for seed in (1, 2):
        x, z = axis_aligned_data(200_000, D, 20, seed, hyper)
        res = {}
        for dev in (True, False):
            t0 = time.perf_counter()
            labels, clusters, weights, iters, *rest = _fit(pkg, x, hyper, seed, dev)
            wall = time.perf_counter() - t0
            nmi = H.normalized_mutual_info(z, labels)
            res[dev] = (nmi, len(clusters), len(iters) / sum(iters), len(iters) / wall)
            assert nmi >= 0.9 and abs(len(clusters) - 20) <= 3, (dev, nmi, len(clusters))
            if dev:
                model = rest[-1]
                assert len(weights) == len(clusters) == len(np.unique(labels))
                for c in clusters:
                    assert isinstance(c, P.diag_gaussian)
                    assert np.isfinite(c.μ).all() and np.isfinite(c.σ2).all() and (c.σ2 > 0).all()
                    assert np.isfinite(c.logdetΣ)
                assert np.isfinite(H.calculate_posterior(model))
        print(f"diag fit D={D} seed={seed}: device NMI {res[True][0]:.4f} K {res[True][1]} "
              f"({res[True][2]:.1f} it/s loop, {res[True][3]:.1f} it/s call); host NMI {res[False][0]:.4f} "
              f"K {res[False][1]} ({res[False][2]:.1f} it/s loop, {res[False][3]:.1f} it/s call)")


def test_checkpoint_save_and_resume_on_the_device_path(pkg, tmp_path):
    from dpmmsubclusters_jl_b200 import checkpoint as CK, host as H, priors as P
    D = 64
    hyper = P.diag_niw_hyperparams(1.0, np.zeros(D), 10.0, np.ones(D))
    x, z = axis_aligned_data(50_000, D, 8, 9, hyper)
    pkg.fit(x, hyper, 10.0, iters=20, seed=4, save_model=True, save_path=str(tmp_path) + "/", model_save_interval=10,
            device_params=True)
    fname = str(tmp_path / "checkpoint__20.npz")
    grp, mh, it, _, _ = CK.load_checkpoint(fname)
    assert it == 20 and isinstance(mh.distribution_hyper_params, P.diag_niw_hyperparams)
    for k, c in enumerate(grp["local_clusters"]):
        assert int((grp["labels"] == k + 1).sum()) == c.points_count
        assert isinstance(c.cluster_params.cluster_params.distribution, P.diag_gaussian)
    resumed, iters, *_ = H.run_model_from_checkpoint(fname, verbose=False, data=x, device_params=True)
    assert len(iters) == 80
    assert H.normalized_mutual_info(z, resumed.group.sweep.get_labels()) >= 0.9
    for c in resumed.group.local_clusters:
        assert isinstance(c.cluster_params.cluster_params.distribution, P.diag_gaussian)


def test_error_paths(pkg):
    import ctypes as C
    from dpmmsubclusters_jl_b200 import _lib as L
    D = 8
    x = np.random.default_rng(0).standard_normal((D, 500)).astype(np.float32)
    g = pkg.GpuSweep(x, pkg.DIAG)
    ok = dict(kappa=1.0, m=np.zeros(D), nu=3.0, psi=np.ones(D), alpha=1.0)
    bad = [dict(kappa=0.0), dict(kappa=-1.0), dict(nu=0.0), dict(nu=-2.0), dict(alpha=0.0), dict(kappa=np.nan),
           dict(m=np.r_[np.zeros(D - 1), np.nan]), dict(m=np.r_[np.inf, np.zeros(D - 1)]),
           dict(psi=np.r_[np.ones(D - 1), 0.0]), dict(psi=np.r_[-np.ones(1), np.ones(D - 1)]),
           dict(psi=np.r_[np.ones(D - 1), np.inf]), dict(psi=np.r_[np.nan, np.ones(D - 1)])]
    for b in bad:
        a = {**ok, **b}
        with pytest.raises(L.DpmmError) as e:
            g.set_hyper_diag(a["kappa"], a["m"], a["nu"], a["psi"], a["alpha"])
        assert e.value.code == L.EINVAL, b
    lib = L.load()
    m, psi = np.zeros(D), np.ones(D)
    for mp, pp in ((None, psi.ctypes.data_as(C.POINTER(C.c_double))), (m.ctypes.data_as(C.POINTER(C.c_double)), None)):
        assert lib.dpmm_set_hyper_diag(g.h, 1.0, mp, 3.0, pp, 1.0) == L.EINVAL
    for call in (lambda: g.posterior_step(None), lambda: g.sample_params(1), lambda: g.get_params_diag(1)):
        with pytest.raises(L.DpmmError) as e:
            call()
        assert e.value.code == L.ESTATE
    g.set_hyper_diag(**ok)
    g.set_labels(np.ones(500, np.int64)); g.set_sublabels(np.r_[np.ones(250, np.int64), np.full(250, 2)])
    with pytest.raises(L.DpmmError) as e:
        g.get_params_diag(1)                                  # nothing sampled yet
    assert e.value.code == L.ESTATE
    g.posterior_step(None)
    g.sample_params(1)
    mu, var, ld, w, lr = g.get_params_diag(1)
    assert np.isfinite(mu).all() and (var > 0).all()
    with pytest.raises(L.DpmmError) as e:
        g.get_params_diag(2)                                  # another K
    assert e.value.code == L.ESTATE
    for call in (lambda: g.set_hyper_multinomial(np.ones(D), 1.0), lambda: g.set_hyper_niw(1.0, np.zeros(D), 10.0, np.eye(D), 1.0),
                 lambda: g.get_params_niw(1), lambda: g.get_params_multinomial(1),
                 lambda: g.predict_multinomial(np.zeros((1, D)), np.zeros(1)),
                 lambda: g.predict_niw(np.zeros((1, D, D)), np.zeros((1, D)), np.zeros(1), np.ones(1)),
                 lambda: g.smart_project(1, np.ones(D), np.zeros(D))):
        with pytest.raises(L.DpmmError) as e:
            call()
        assert e.value.code == L.ESTATE
    g.close()
    for kind in (pkg.NIW, pkg.MULTINOMIAL):
        h = pkg.GpuSweep(np.round(np.abs(x)), kind)
        with pytest.raises(L.DpmmError) as e:
            h.set_hyper_diag(**ok)
        assert e.value.code == L.ESTATE
        with pytest.raises(L.DpmmError) as e:
            h.get_params_diag(1)
        assert e.value.code == L.ESTATE
        h.close()


def test_two_gpu_fit_draws_identical_parameters_on_every_rank():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29623", os.path.join(ROOT, "tests", "mgpu_params_diag_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "MGPU_PARAMS_DIAG_OK" in out.stdout
