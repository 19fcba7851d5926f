"""Helpers of the diagonal Gaussian tests: synthetic cases and the GPU-vs-oracle comparison of one sweep, with the
tolerances and near-tie accounting of tests/util.py."""
import numpy as np

from oracle import diag_oracle as DO
from tests.util import STATS_RTOL, check_draws, check_loglik, tie_tolerance


def make_diag_case(D, K, n, seed, spread=2.5, offset=0.0, empty=False, zero_weight=False):
    """Overlapping axis-aligned clusters and 3K diagonal distributions near them (Float32 mu / sigma^2 / logdet).
    offset: every mean moves by offset x sigma from the origin.  empty: cluster K-1 lies far from all points.
    zero_weight: cluster 0 has weight exactly 0."""
    rng = np.random.default_rng(seed)
    centers = rng.standard_normal((K, D)) * spread + offset
    var = rng.uniform(0.5, 2.0, (K, D))
    z = rng.integers(0, K - 1 if (empty and K > 1) else K, n)
    x = (centers[z].T + np.sqrt(var[z].T) * rng.standard_normal((D, n))).astype(np.float32)
    if empty and K > 1:
        centers[K - 1] += 1e3
    mu = np.zeros((K, 3, D), np.float32)
    vv = np.zeros((K, 3, D), np.float32)
    for s in range(3):
        mu[:, s] = centers + (0 if s == 0 else (0.7 if s == 1 else -0.7)) * rng.standard_normal((K, D))
        vv[:, s] = var * rng.uniform(0.7, 1.3, (K, D))
    logdet = np.log(vv.astype(np.float64)).sum(-1).astype(np.float32)
    w = rng.dirichlet(np.ones(K) * 5).astype(np.float32)
    if zero_weight and K > 1:
        w[0] = 0
    lr = rng.dirichlet(np.ones(2) * 5, size=K).astype(np.float32)
    return dict(kind=DO.DIAG, x=x, mu=mu, var=vv, logdet=logdet, weights=w, lr_weights=lr, K=K, D=D, n=n)


def set_params_diag(sw, case):
    sw.set_params_diag(case["mu"], case["var"], case["logdet"], case["weights"], case["lr_weights"])


def check_diag_stats(gpu, ora, what):
    """Counts exact; sum x and sum x^2 within STATS_RTOL of the scales check_stats uses for NIW sum x and diag(S):
    sqrt(N S_dd) and S_dd."""
    gc, gsx, gsxx = gpu
    oc, osx, osxx = ora
    np.testing.assert_array_equal(gc, oc, err_msg=f"{what}: counts")
    assert gsxx.shape == osxx.shape == gsx.shape, f"{what}: shapes"
    sdd = np.maximum(osxx, 1e-300)
    e_xx = np.abs(gsxx - osxx) / sdd
    e_x = np.abs(gsx - osx) / np.maximum(np.sqrt(np.maximum(oc, 1)[..., None] * sdd), 1e-30)
    nz = oc > 0
    worst = max(e_xx[nz].max(initial=0.0), e_x[nz].max(initial=0.0))
    assert worst <= STATS_RTOL, f"{what}: max scaled err {worst:.3e}"
    assert not gsxx[~nz].any() and not gsx[~nz].any(), f"{what}: empty sets must give zeros"
    return float(worst)


def compare_diag_sweeps(g, o, case, rng, final=False):
    """tests/util.compare_sweeps for a diagonal context: the GPU state is copied into the oracle after every stage."""
    n, K = case["n"], case["K"]
    u_label, u_sub = rng.random(n), rng.random(n)
    bits = rng.integers(0, 2, n).astype(np.uint8)
    for s in (g, o):
        s.set_uniforms(u_label, u_sub, bits)
        set_params_diag(s, case)
    rep = {}
    LLo = o.debug_loglik(0)
    rep["ll_err"] = check_loglik(g.debug_loglik(0), LLo, "label log-likelihood")
    g.sample_labels(final); o.sample_labels(final)
    gl, ol = g.get_labels(), o.get_labels()
    if final:
        bad = np.nonzero(gl != ol)[0]
        if bad.size:
            srt = np.sort(LLo[bad], axis=1)
            assert ((srt[:, -1] - srt[:, -2]) <= tie_tolerance(LLo[bad])).all(), "argmax mismatch that is not a tie"
        rep["label_ties"] = int(bad.size)
    else:
        rep["label_ties"] = check_draws(LLo, u_label, gl, ol, "labels")
    o.set_labels(gl)
    SLo = o.debug_loglik(1)
    rep["sub_ll_err"] = check_loglik(g.debug_loglik(1), SLo, "sub-label log-likelihood")
    g.sample_sublabels(); o.sample_sublabels()
    gs = g.get_sublabels()
    rep["sub_ties"] = check_draws(SLo, u_sub, gs, o.get_sublabels(), "sub-labels")
    o.set_sublabels(gs)
    rep["stats_err"] = check_diag_stats(g.suff_stats(), o.suff_stats(), "suff stats (all)")
    sub_idx = [K, 1] if K > 1 else [1]
    check_diag_stats(g.suff_stats(sub_idx), o.suff_stats(sub_idx), "suff stats (restricted)")
    counts = np.bincount(gl, minlength=K + 1)[1:]
    big = int(np.argmax(counts)) + 1
    for s in (g, o):
        s.apply_split([big], [K + 1])
        s.K = K + 1
    np.testing.assert_array_equal(g.get_labels(), o.get_labels(), err_msg="split: labels")
    np.testing.assert_array_equal(g.get_sublabels(), o.get_sublabels(), err_msg="split: sub-labels")
    check_diag_stats(g.suff_stats([big, K + 1]), o.suff_stats([big, K + 1]), "suff stats after split")
    if K >= 2:
        i, j = (1 if big != 1 else 2), K + 1
        for s in (g, o):
            s.apply_merge([i], [j])
        np.testing.assert_array_equal(g.get_labels(), o.get_labels(), err_msg="merge: labels")
        check_diag_stats(g.suff_stats([i]), o.suff_stats([i]), "suff stats after merge")
    cnt = np.bincount(g.get_labels(), minlength=K + 2)[1:K + 2]
    for s in (g, o):
        s.remove_empty(cnt)
    np.testing.assert_array_equal(g.get_labels(), o.get_labels(), err_msg="remove_empty: labels")
    kk = int(g.get_labels().max())
    for s in (g, o):
        s.K = kk
    check_diag_stats(g.suff_stats(list(range(1, kk + 1))), o.suff_stats(list(range(1, kk + 1))), "suff stats after remove_empty")
    for s in (g, o):
        s.set_uniforms(None, None, None)
    return rep


def axis_aligned_data(N, D, K, seed, hyper):
    """Means ~ N(0, 100 I), per-feature variances drawn from the prior (nu psi / chi^2_nu), K clusters of random
    weights.  Returns (x [D, N] f32, labels [N] 1-based)."""
    rng = np.random.default_rng(seed)
    means = rng.standard_normal((K, D)) * 10.0
    var = hyper.ν * hyper.ψ[None, :] / rng.chisquare(hyper.ν, (K, D))
    w = rng.dirichlet(np.ones(K) * 5)
    z = rng.choice(K, N, p=w)
    x = (means[z].T + np.sqrt(var[z].T) * rng.standard_normal((D, N))).astype(np.float32)
    return x, z + 1
