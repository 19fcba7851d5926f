"""The outlier component (DESIGN.md 6.1) on the GPU: the device parameter step of cluster 1 under its own prior for the
three priors (posterior / log marginal likelihood, weights, draws), the C ABI refusals, and fit() of the Gaussian priors
with a uniform background on both parameter paths."""
import os
import subprocess
import sys

import numpy as np
import pytest

import dpmm_pkg
from tests.diag_util import axis_aligned_data
from tests.util import make_niw_case

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OMEGA = 0.05


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    return dpmm_pkg.load()


def _priors(P, kind, D, rng):
    """(model prior, outlier prior) of one kind at dimension D."""
    if kind == "niw":
        return (P.niw_hyperparams(1.5, rng.standard_normal(D) * 0.3, D + 3.5, np.eye(D) * 1.3 + 0.1),
                P.niw_hyperparams(0.05, rng.standard_normal(D), D + 2.0, np.eye(D) * 40.0))
    if kind == "diag":
        return (P.diag_niw_hyperparams(1.5, rng.standard_normal(D) * 0.3, 6.0, rng.uniform(0.5, 2.0, D)),
                P.diag_niw_hyperparams(0.05, rng.standard_normal(D), 3.0, np.full(D, 40.0)))
    return P.multinomial_hyper(np.ones(D, np.float32)), P.multinomial_hyper(np.full(D, 30.0, np.float32))


def _context(pkg, kind, D, K, n, seed, outlier):
    """A context with random labels / sub-labels, the model prior set and, with `outlier`, the component on."""
    from dpmmsubclusters_jl_b200 import priors as P
    rng = np.random.default_rng(seed)
    if kind == "mnm":
        x = rng.poisson(3.0, (D, n)).astype(np.float32)
        g = pkg.GpuSweep(x, pkg.MULTINOMIAL, seed=5)
    else:
        x = make_niw_case(D, K, n, seed=seed, spread=4.0)["x"] if kind == "niw" else rng.standard_normal((D, n)) * 3
        g = pkg.GpuSweep(x, pkg.NIW if kind == "niw" else pkg.DIAG, seed=5)
    g.set_labels(rng.integers(1, K + 1, n))
    g.set_sublabels(rng.integers(1, 3, n))
    hyper, out = _priors(P, kind, D, rng)
    _set(g, kind, hyper, None, 10.0)
    if outlier:
        _set(g, kind, None, out, OMEGA)
    return g, hyper, out, P


def _set(g, kind, hyper, out, w):
    if hyper is not None:
        {"niw": lambda: g.set_hyper_niw(hyper.κ, hyper.m, hyper.ν, hyper.ψ, w),
         "diag": lambda: g.set_hyper_diag(hyper.κ, hyper.m, hyper.ν, hyper.ψ, w),
         "mnm": lambda: g.set_hyper_multinomial(hyper.α, w)}[kind]()
    else:
        {"niw": lambda: g.set_outlier_niw(w, out.κ, out.m, out.ν, out.ψ),
         "diag": lambda: g.set_outlier_diag(w, out.κ, out.m, out.ν, out.ψ),
         "mnm": lambda: g.set_outlier_multinomial(w, out.α)}[kind]()


def _get(g, K):
    return {0: g.get_params_niw, 1: g.get_params_multinomial, 2: g.get_params_diag}[g.prior_kind](K)


@pytest.mark.parametrize("kind,D", [("niw", 2), ("niw", 32), ("niw", 50), ("diag", 128), ("mnm", 100)])
def test_posterior_step_uses_the_outlier_prior_for_cluster_1_only(pkg, kind, D):
    """The same statistics table evaluated with the component on and off (the statistics accumulate with atomics, so
    two contexts would differ in the last bits of their sums): only cluster 1 changes."""
    K, n = 5, 6000
    g, hyper, out, P = _context(pkg, kind, D, K, n, seed=D, outlier=True)
    c1, l1, m1 = g.posterior_step(None, splittable=np.ones(K, bool))
    _set(g, kind, None, out, 0.0)
    c0, l0, m0 = g.posterior_step(np.arange(1, K + 1), splittable=np.ones(K, bool), from_table=True)
    np.testing.assert_array_equal(c1, c0)
    assert l1[1:].tobytes() == l0[1:].tobytes()
    assert m1[1:, 1:].tobytes() == m0[1:, 1:].tobytes()
    sc, sx, sxx = g.suff_stats([1])
    for s in range(3):
        ss = P.make_suff_stats(out, sc[0, s], sx[0, s], None if sxx is None else sxx[0, s])
        want = P.log_marginal_likelihood(out, P.calc_posterior(out, ss), ss)
        # log_multivariate_gamma accumulates in Float32, as the reference does: a few of its ulps on top of 1e-9
        assert abs(l1[0, s] - want) <= 1e-9 * abs(want) + 8 * np.spacing(np.float32(abs(want))), (s, l1[0, s], want)
        assert l1[0, s] != l0[0, s]
    g.close()


@pytest.mark.parametrize("kind,D", [("niw", 2), ("diag", 16), ("mnm", 20)])
def test_weights_and_prior_draws(pkg, kind, D):
    K, n, calls = 5, 4000, 2000
    g, hyper, out, P = _context(pkg, kind, D, K, n, seed=7, outlier=True)
    counts, _, _ = g.posterior_step(None)
    alpha = np.float32(10.0)
    ws = []
    for _ in range(calls):
        g.sample_params(K)
        w = _get(g, K)[-2]
        assert w[0] == np.float32(OMEGA)
        ws.append(w)
    ws = np.asarray(ws, np.float64)
    a = np.concatenate([counts[1:, 0].astype(np.float64), [alpha]])
    a0 = a.sum()
    mean = (1 - OMEGA) * a[:-1] / a0
    sd = (1 - OMEGA) * np.sqrt(a[:-1] * (a0 - a[:-1]) / (a0 ** 2 * (a0 + 1)))
    assert (np.abs(ws[:, 1:].mean(0) - mean) <= 4 * sd / np.sqrt(calls)).all(), (ws[:, 1:].mean(0), mean)
    g.sample_params(K, unit_weights=True)
    w = _get(g, K)[-2]
    assert w[0] == np.float32(OMEGA) and np.allclose(w[1:], (1 - OMEGA) / (K - 1))
    # from_prior: cluster 1's three distributions come from the outlier prior, the others from the model's
    draws0, draws1 = [], []
    for _ in range(400):
        g.sample_params(K, from_prior=True)
        p = _get(g, K)
        draws0.append(p[0][0]); draws1.append(p[0][2])
    d0, d1 = np.asarray(draws0, np.float64), np.asarray(draws1, np.float64)
    if kind == "mnm":        # log p ~ log Dirichlet(alpha): the mean of p is alpha / sum alpha either way; the spread differs
        v0, v1 = np.exp(d0).var(0).mean(), np.exp(d1).var(0).mean()
        a_o, a_m = float(out.α[0]), float(hyper.α[0])
        want0 = (1 / D) * (1 - 1 / D) / (a_o * D + 1)
        want1 = (1 / D) * (1 - 1 / D) / (a_m * D + 1)
        assert abs(v0 / want0 - 1) < 0.3 and abs(v1 / want1 - 1) < 0.3
    else:                    # mu = m + N(0, Sigma / kappa): centre and spread of the outlier prior, not the model's
        m_o, m_m = out.m, hyper.m
        assert np.abs(d0.mean(0)[:, :] - m_o).max() < 0.5 * np.sqrt(d0.var(0)).max()
        assert np.abs(d1.mean(0)[:, :] - m_m).max() < 0.5 * np.sqrt(d1.var(0)).max()
        assert d0.var(0).mean() > 20 * d1.var(0).mean()
    g.close()


@pytest.mark.parametrize("kind,D", [("niw", 2), ("niw", 50), ("diag", 16), ("mnm", 20)])
def test_weight_zero_gives_the_bits_of_a_context_without_the_component(pkg, kind, D):
    """Byte for byte where the inputs are: draws from the prior, and the weights (integer counts).  Posterior draws
    read statistics sums whose last bits depend on the order of atomic additions in each context."""
    K, n = 4, 3000
    ref, *_ = _context(pkg, kind, D, K, n, seed=3, outlier=False)
    g, hyper, out, P = _context(pkg, kind, D, K, n, seed=3, outlier=True)
    _set(g, kind, None, out, 0.0)
    for sw in (ref, g):
        sw.posterior_step(None)
    for first in (True, False, False):
        ref.sample_params(K, from_prior=first, unit_weights=first)
        g.sample_params(K, from_prior=first, unit_weights=first)
        pr, pg = _get(ref, K), _get(g, K)
        for a, b in zip(pr if first else pr[-2:], pg if first else pg[-2:]):
            assert a.tobytes() == b.tobytes()
        if not first:
            for a, b in zip(pr[:-2], pg[:-2]):
                np.testing.assert_allclose(a, b, rtol=1e-4, atol=1e-5)
    ref.close(); g.close()


def test_abi_refusals(pkg):
    from dpmmsubclusters_jl_b200 import _lib as L
    from dpmmsubclusters_jl_b200 import priors as P
    D = 3
    x = np.abs(np.random.default_rng(0).standard_normal((D, 500))).astype(np.float32)
    niw = P.niw_hyperparams(1.0, np.zeros(D), D + 2.0, np.eye(D))

    def code(f):
        with pytest.raises(L.DpmmError) as e:
            f()
        return e.value.code
    g = pkg.GpuSweep(x, pkg.NIW)
    assert code(lambda: g.set_outlier_niw(0.05, 1.0, np.zeros(D), D + 2.0, np.eye(D))) == L.ESTATE   # before set_hyper
    g.set_hyper_niw(niw.κ, niw.m, niw.ν, niw.ψ, 10.0)
    assert code(lambda: g.set_outlier_multinomial(0.05, np.ones(D))) == L.ESTATE                     # wrong prior
    assert code(lambda: g.set_outlier_diag(0.05, 1.0, np.zeros(D), 3.0, np.ones(D))) == L.ESTATE
    for w in (1.0, -0.01, float("nan"), 1.5):
        assert code(lambda: g.set_outlier_niw(w, 1.0, np.zeros(D), D + 2.0, np.eye(D))) == L.EINVAL
    assert code(lambda: g.set_outlier_niw(0.05, 0.0, np.zeros(D), D + 2.0, np.eye(D))) == L.EINVAL    # kappa
    assert code(lambda: g.set_outlier_niw(0.05, 1.0, np.zeros(D), D - 1.5, np.eye(D))) == L.EINVAL    # nu
    assert code(lambda: g.set_outlier_niw(0.05, 1.0, np.zeros(D), D + 2.0, -np.eye(D))) == L.EINVAL   # psi
    g.init_labels(2, True)
    g.set_outlier_niw(0.05, 1.0, np.zeros(D), D + 2.0, np.eye(D))
    g.posterior_step(None)
    assert code(lambda: g.params_merge(1, 2)) == L.EINVAL
    assert code(lambda: g.params_merge(3, 1)) == L.EINVAL
    g.params_merge(2, 3)
    g.set_outlier_niw(0.0, 1.0, np.zeros(D), D + 2.0, np.eye(D))                                        # off again
    g.params_merge(1, 2)
    g.close()
    m = pkg.GpuSweep(np.round(x * 3), pkg.MULTINOMIAL)
    m.set_hyper_multinomial(np.ones(D), 10.0)
    assert code(lambda: m.set_outlier_multinomial(0.05, np.array([1.0, 0.0, 1.0]))) == L.EINVAL
    assert code(lambda: m.set_outlier_niw(0.05, 1.0, np.zeros(D), D + 2.0, np.eye(D))) == L.ESTATE
    m.close()
    d = pkg.GpuSweep(x, pkg.DIAG)
    assert code(lambda: d.set_outlier_diag(0.05, 1.0, np.zeros(D), 3.0, np.ones(D))) == L.ESTATE
    d.set_hyper_diag(1.0, np.zeros(D), 3.0, np.ones(D), 10.0)
    assert code(lambda: d.set_outlier_diag(0.05, 1.0, np.zeros(D), 3.0, np.array([1.0, -1.0, 1.0]))) == L.EINVAL
    assert code(lambda: d.set_outlier_diag(1.0, 1.0, np.zeros(D), 3.0, np.ones(D))) == L.EINVAL
    d.close()


# ---------------------------------------------------------------------------------------------- fit() --------
def _with_background(x, frac, rng):
    """x plus frac/(1-frac) of its size in points uniform over a box three times as wide as x's bounding box, and the
    outlier prior's centre and per-feature variance (those of the box).  Returns (points, background mask, m, var)."""
    D, n = x.shape
    nb = int(round(n * frac / (1 - frac)))
    c, h = (x.min(1) + x.max(1)) / 2.0, 1.5 * (x.max(1) - x.min(1))
    b = rng.uniform((c - h)[:, None], (c + h)[:, None], (D, nb))
    return (np.concatenate([x, b.astype(np.float32)], 1), np.concatenate([np.zeros(n, bool), np.ones(nb, bool)]),
            c, (2 * h) ** 2 / 12.0)


def _case(pkg, name):
    from dpmmsubclusters_jl_b200 import priors as P
    rng = np.random.default_rng(11)
    if name == "niw2":
        from tests.test_outlier_host import background_data, OUTLIER, PRIOR
        x, gt = background_data(1)
        return x, gt, gt == 0, PRIOR, OUTLIER, 300
    if name == "niw32":
        D = 32
        x, gt, _, _ = pkg.generate_gaussian_data(95_000, D, 10, 100.0, rng)
        x, bg, m, var = _with_background(x, 0.05, rng)
        out = P.niw_hyperparams(1.0, m, D + 3.0, np.diag(var))
        return x, np.concatenate([gt.astype(np.int64), np.zeros(bg.sum(), np.int64)]), bg, \
            P.niw_hyperparams(1.0, np.zeros(D), D + 3.0, np.eye(D)), out, 100
    D = 128
    hyper = P.diag_niw_hyperparams(1.0, np.zeros(D), 10.0, np.ones(D))
    x, gt = axis_aligned_data(30_000, D, 8, 5, hyper)
    x, bg, m, var = _with_background(x, 0.05, rng)
    out = P.diag_niw_hyperparams(1.0, m, 10.0, var)
    return x, np.concatenate([gt, np.zeros(bg.sum(), np.int64)]), bg, hyper, out, 100


@pytest.mark.timeout(900, method="thread")
@pytest.mark.parametrize("device_params", [True, False])
@pytest.mark.parametrize("name", ["niw2", "niw32", "diag128"])
def test_fit_puts_the_background_in_cluster_1(pkg, name, device_params):
    """niw2: the data and priors of tests/test_outlier_host.py; niw32 / diag128: background in a box three times as wide
    as the data, the outlier prior centred on it with its variance."""
    from dpmmsubclusters_jl_b200 import host as H
    x, gt, bg, hyper, out, iters = _case(pkg, name)
    for seed in (1, 2, 3):
        labels, _, weights, *_ = pkg.fit(x, hyper, 10.0, iters=iters, seed=seed, outlier_weight=OMEGA, outlier_params=out,
                                         device_params=device_params)
        assert weights[0] == np.float32(OMEGA) and weights[1:].sum() <= 0.95 + 1e-6
        cap, leak = (labels[bg] == 1).mean(), (labels[~bg] == 1).mean()
        nmi = H.normalized_mutual_info(gt[~bg], labels[~bg])
        print(f"{name} device_params={device_params} seed={seed}: K={len(weights)} background in 1: {cap:.3f}, "
              f"inliers in 1: {leak:.4f}, inlier NMI {nmi:.4f}")
        assert cap >= 0.80 and leak <= 0.01 and nmi >= 0.95


def test_two_gpu_parameters_identical_with_the_component():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29631", os.path.join(ROOT, "tests", "mgpu_outlier_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "MGPU_OUTLIER_OK" in out.stdout
