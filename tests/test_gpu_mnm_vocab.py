"""Multinomial models past the shared-memory table: vocabularies up to D = 16 384 and any K up to 1 024.

The streaming label kernel (mnm_label_stream_kernel), the staged sub-label kernel (D > 1024) and the sliced
statistics kernel (D > 1024) do the same Float32 arithmetic as the kernels that serve the smaller shapes, so they are
checked byte for byte against those kernels (K split into 16-cluster contexts; zero-count padding features), and
against the CPU oracle, the prior plugin and the host paths."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

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


def test_k_split_loglik_is_byte_exact(pkg):
    """D = 1000, K = 200 runs the streaming kernel; every 16-cluster slice of the same parameters fits the table
    kernel.  The log-likelihood columns must agree bit for bit."""
    D, K, n = 1000, 200, 3000
    case = make_mnm_case(D, K, n, seed=31)
    g = pkg.GpuSweep(case["x"], pkg.MULTINOMIAL, seed=1)
    g.set_params_multinomial(case["log_p"], case["weights"], case["lr_weights"])
    full = g.debug_loglik(0)
    g.close()
    parts = []
    for k0 in range(0, K, 16):
        s = pkg.GpuSweep(case["x"], pkg.MULTINOMIAL, seed=1)
        s.set_params_multinomial(case["log_p"][k0:k0 + 16], case["weights"][k0:k0 + 16], case["lr_weights"][k0:k0 + 16])
        parts.append(s.debug_loglik(0))
        s.close()
    assert full.tobytes() == np.ascontiguousarray(np.concatenate(parts, axis=1)).tobytes()


@pytest.mark.parametrize("sampler,final", [(0, False), (1, False), (0, True)])
def test_zero_padded_vocabulary_gives_identical_sweeps(pkg, sampler, final):
    """D = 300 (table label kernel, thread-per-point sub-label kernel, one statistics slice) against the same model
    padded to D = 1200 with zero-count features of finite log-probability (streaming label kernel, staged sub-label
    kernel, two statistics slices): five Philox sweeps with fixed parameters agree exactly."""
    D, P, K, n = 300, 900, 20, 5000
    case = make_mnm_case(D, K, n, seed=5)
    xp = np.concatenate([case["x"], np.zeros((P, n), np.float32)])
    rng = np.random.default_rng(6)
    lp = np.log(np.concatenate([0.5 * np.exp(case["log_p"].astype(np.float64)),
                                0.5 * rng.dirichlet(np.ones(P), size=(K, 3))], axis=-1)).astype(np.float32)
    lp_small = np.ascontiguousarray(lp[..., :D])
    a = pkg.GpuSweep(case["x"], pkg.MULTINOMIAL, seed=77)
    b = pkg.GpuSweep(xp, pkg.MULTINOMIAL, seed=77)
    for s, l in ((a, lp_small), (b, lp)):
        s.set_sampler(sampler)
        s.init_labels(K)
        s.set_params_multinomial(l, case["weights"], case["lr_weights"])
    for _ in range(5):
        for s in (a, b):
            s.sample_labels(final)
            s.sample_sublabels()
        np.testing.assert_array_equal(a.get_labels(), b.get_labels())
        np.testing.assert_array_equal(a.get_sublabels(), b.get_sublabels())
        ca, sa, _ = a.suff_stats()
        cb, sb, _ = b.suff_stats()
        np.testing.assert_array_equal(ca, cb)
        assert sa.tobytes() == np.ascontiguousarray(sb[..., :D]).tobytes()
        assert not sb[..., D:].any()
    assert len(np.unique(a.get_labels())) > 1
    a.close(); b.close()


@pytest.mark.parametrize("D,K,n", [(1000, 200, 6000), (4096, 48, 3000), (16384, 8, 1500), (100, 500, 20000)])
def test_large_vocabulary_sweep_parity(pkg, D, K, n):
    case = make_mnm_case(D, K, n, seed=300 + D)
    g = pkg.GpuSweep(case["x"], pkg.MULTINOMIAL, seed=9)
    o = O.OracleSweep(case["x"], O.MULTINOMIAL, seed=9)
    rep = compare_sweeps(g, o, case, np.random.default_rng(D))
    g.close()
    print(f"mnm D={D} K={K} n={n}: {rep}")


def test_device_parameter_step_at_d12000(pkg):
    from dpmmsubclusters_jl_b200 import priors as P
    D, K, n = 12000, 4, 2000
    case = make_mnm_case(D, K, n, seed=12)
    rng = np.random.default_rng(12)
    lab = rng.integers(1, K + 1, n)
    sub = rng.integers(1, 3, n)
    hyper = P.multinomial_hyper(rng.uniform(0.3, 2.0, D))
    g = pkg.GpuSweep(case["x"], pkg.MULTINOMIAL, seed=5)
    g.set_labels(lab); g.set_sublabels(sub)
    g.set_hyper_multinomial(hyper.α, 10.0)
    counts, logml, merge = g.posterior_step(None, splittable=np.ones(K, bool))
    sc, sx, _ = g.suff_stats()
    np.testing.assert_array_equal(counts, sc)
    for k in range(K):
        for s in range(3):
            ss = P.make_suff_stats(hyper, sc[k, s], sx[k, s])
            want = P.log_marginal_likelihood(hyper, P.calc_posterior(hyper, ss), ss)
            assert abs(logml[k, s] - want) <= 1e-10 * max(1.0, abs(want)), (k, s, logml[k, s], want)
    for i in range(K):
        for j in range(i + 1, K):
            ab = P.aggregate_suff_stats(P.make_suff_stats(hyper, sc[i, 0], sx[i, 0]),
                                        P.make_suff_stats(hyper, sc[j, 0], sx[j, 0]))
            want = P.log_marginal_likelihood(hyper, P.calc_posterior(hyper, ab), ab)
            assert abs(merge[i, j] - want) <= 1e-10 * max(1.0, abs(want)), (i, j, merge[i, j], want)
    posts = np.array([[P.calc_posterior(hyper, P.make_suff_stats(hyper, sc[k, s], sx[k, s])).α for s in range(3)]
                      for k in range(K)], np.float64)
    R = 100
    p_acc = np.zeros((K, 3, D))
    for _ in range(R):
        g.sample_params(K)
        lp, w, lr = g.get_params_multinomial(K)
        assert np.isfinite(lp).all() and np.isfinite(w).all() and np.isfinite(lr).all()
        np.testing.assert_allclose(np.exp(lp.astype(np.float64)).sum(-1), 1.0, atol=1e-4)
        p_acc += np.exp(lp.astype(np.float64))
    A = posts.sum(-1, keepdims=True)
    m = posts / A
    sd = np.sqrt(m * (1 - m) / (A + 1) / R)
    assert (np.abs(p_acc / R - m) <= 6 * sd + 1e-6).all(), np.abs(p_acc / R - m).max()
    # the sampled parameters feed a sweep at this D
    g.sample_labels(False)
    g.sample_sublabels()
    assert g.suff_stats()[0][:, 0].sum() == n
    g.close()


def test_predict_on_device_at_d16384(pkg):
    from types import SimpleNamespace
    from dpmmsubclusters_jl_b200 import host as H, priors as P
    D, K, n = 16384, 6, 2000
    case = make_mnm_case(D, K, n, seed=16)
    rng = np.random.default_rng(17)
    cl = [SimpleNamespace(cluster_params=SimpleNamespace(cluster_params=SimpleNamespace(
        posterior_hyperparams=P.multinomial_hyper(rng.uniform(0.5, 60.0, D))))) for _ in range(K)]
    sw = pkg.GpuSweep(case["x"][:, :100], pkg.MULTINOMIAL)
    model = SimpleNamespace(group=SimpleNamespace(local_clusters=cl, weights=rng.dirichlet(np.ones(K)).astype(np.float32),
                                                  sweep=sw))
    lg, pg = H.predict(model, case["x"], on_device=True)
    lh, ph = H.predict(model, case["x"], on_device=False)
    np.testing.assert_array_equal(lg, lh)
    np.testing.assert_allclose(pg, ph, atol=1e-6)
    sw.close()


@pytest.mark.timeout(600, method="thread")
def test_fit_past_the_table_limit(pkg):
    """fit() on a 1 000-word vocabulary with 40 true clusters grows past K = 16 (the largest K the table kernel holds
    at this D) on both parameter paths; one shorter fit at D = 4 000."""
    from dpmmsubclusters_jl_b200.host import normalized_mutual_info
    hyper = pkg.multinomial_hyper(np.ones(1000, np.float32))
    x, z, _ = pkg.generate_mnmm_data(20000, 1000, 40, 200, np.random.default_rng(0))
    for dev in (True, False):
        for seed in (1, 2):
            labels, clusters, *_ = pkg.fit(x, hyper, 10.0, iters=150, seed=seed, burnout=10, device_params=dev)
            nmi = normalized_mutual_info(z, labels)
            print(f"D=1000 device_params={dev} seed={seed}: K={len(clusters)} NMI={nmi:.4f}")
            assert len(clusters) >= 17
            assert nmi >= 0.8
    hyper = pkg.multinomial_hyper(np.ones(4000, np.float32))
    x, z, _ = pkg.generate_mnmm_data(5000, 4000, 20, 400, np.random.default_rng(1))
    labels, clusters, *_ = pkg.fit(x, hyper, 10.0, iters=30, seed=2, burnout=5, device_params=True)
    print(f"D=4000: K={len(clusters)} NMI={normalized_mutual_info(z, labels):.4f}")
    assert len(clusters) > 1


def test_limits(pkg):
    E = pkg._lib
    out = (ctypes.c_int32 * 3)()
    assert E.load().dpmm_limits(out) == 0
    assert out[1] == 16384 and out[2] == 1024
    with pytest.raises(E.DpmmError) as ei:
        pkg.GpuSweep(np.zeros((16385, 4), np.float32), pkg.MULTINOMIAL)
    assert ei.value.code == E.ELIMIT
    D, K, n = 16384, 1024, 300
    rng = np.random.default_rng(3)
    x = rng.poisson(0.05, (D, n)).astype(np.float32)
    lp = np.log(rng.dirichlet(np.ones(D), size=(K, 3))).astype(np.float32)
    g = pkg.GpuSweep(x, pkg.MULTINOMIAL, seed=4)
    g.init_labels(K)
    g.set_params_multinomial(lp, np.full(K, 1.0 / K, np.float32), np.full((K, 2), 0.5, np.float32))
    g.sample_labels(False)
    g.sample_sublabels()
    counts, sx, _ = g.suff_stats()
    assert counts[:, 0].sum() == n and (counts[:, 0] == counts[:, 1] + counts[:, 2]).all()
    np.testing.assert_array_equal(sx[:, 0].sum(0), x.sum(1).astype(np.float64))
    g.close()


def test_two_gpu_statistics_at_d3000():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29613", os.path.join(ROOT, "tests", "mgpu_mnm_worker.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "MGPU_MNM_OK" in out.stdout
