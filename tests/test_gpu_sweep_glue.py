"""The work between the two tensor-core kernels of a D = 32 sweep: the label kernel counts the points whose label
changed, the sort after it skips its scatter when none did, the label histograms are double-buffered, the adaptive
path choice reads its counters from mapped host memory, and the risk slot of the statistics finalise is cleared by
the scatter.  Every check here is against the labels themselves or against statistics recomputed on the host."""
import numpy as np
import pytest

from tests.util import make_niw_case

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    ge.build()
    import dpmm_pkg
    return dpmm_pkg.load()


def set_params(g, case):
    g.set_params_niw(case["mu"], case["inv_sigma"], case["logdet"], case["weights"], case["lr_weights"])


def host_stats(x, labels, sub, K):
    """counts [K,3], sum x [K,3,D], sum x x' [K,3,D,D] (cluster, left, right) in Float64 from 1-based labels."""
    x = x.astype(np.float64)
    D = x.shape[0]
    c = np.zeros((K, 3), np.int64)
    sx = np.zeros((K, 3, D))
    sxx = np.zeros((K, 3, D, D))
    for k in range(K):
        for s, m in enumerate((labels == k + 1, (labels == k + 1) & (sub == 1), (labels == k + 1) & (sub == 2))):
            p = x[:, m]
            c[k, s] = p.shape[1]
            sx[k, s] = p.sum(1)
            sxx[k, s] = p @ p.T
    return c, sx, sxx


def assert_stats(got, x, labels, sub, K):
    c, sx, sxx = host_stats(x, labels, sub, K)
    assert np.array_equal(got[0], c)
    scale = max(np.abs(sxx).max(), 1.0)
    assert np.abs(got[1] - sx).max() <= 1e-5 * max(np.abs(sx).max(), 1.0)
    assert np.abs(got[2] - sxx).max() <= 1e-5 * scale


def assert_sorted(perm, labels):
    assert np.array_equal(np.sort(perm), np.arange(len(labels)))
    assert np.all(np.diff(labels[perm]) >= 0), "perm is not a sort of the labels"


def sweep(g):
    g.sample_labels(False)
    g.sample_sublabels()
    return g.suff_stats()


@pytest.fixture
def converged(pkg):
    """Well-separated clusters (C2-like converged state): after two sweeps no point changes label any more."""
    case = make_niw_case(32, 8, 30000, seed=11, spread=40.0)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=3)
    set_params(g, case)
    sweep(g)
    sweep(g)
    yield g, case
    g.close()


def test_no_movers_keeps_the_sort(converged):
    g, case = converged
    perm0, _ = g.sort_state()
    got = sweep(g)
    perm1, moved = g.sort_state()
    assert moved == 0
    assert np.array_equal(perm0, perm1), "the scatter ran although no label changed"
    lab, sub = g.get_labels(), g.get_sublabels()
    assert_sorted(perm1, lab - 1)
    assert_stats(got, case["x"], lab, sub, case["K"])


def test_movers_run_the_scatter(converged):
    g, case = converged
    before = g.get_labels()
    K = case["K"]
    rot = np.roll(np.arange(K), 1)          # cluster k gets the parameters of cluster k - 1: every point moves
    moved_case = dict(case, mu=case["mu"][rot], inv_sigma=case["inv_sigma"][rot], logdet=case["logdet"][rot],
                      weights=case["weights"][rot], lr_weights=case["lr_weights"][rot])
    set_params(g, moved_case)
    got = sweep(g)
    perm, moved = g.sort_state()
    lab, sub = g.get_labels(), g.get_sublabels()
    assert moved == case["n"]
    assert np.array_equal(lab, before % K + 1)
    assert_sorted(perm, lab - 1)
    assert_stats(got, case["x"], lab, sub, K)
    # and back: the next sweep finds nobody moving again
    got = sweep(g)
    assert g.sort_state()[1] == 0
    assert_stats(got, case["x"], g.get_labels(), g.get_sublabels(), K)


def test_relabel_forces_a_full_sort(converged):
    g, case = converged
    before = g.get_labels()
    g.apply_merge([1], [2])                 # cluster 2's points join cluster 1
    merged = g.get_labels()
    assert np.array_equal(merged, np.where(before == 2, 1, before))
    perm, _ = g.sort_state()
    assert_sorted(perm, merged - 1)
    got = sweep(g)                          # the parameters of cluster 2 take its points back
    perm, moved = g.sort_state()
    lab, sub = g.get_labels(), g.get_sublabels()
    assert moved == int((before == 2).sum())
    assert np.array_equal(lab, before)
    assert_sorted(perm, lab - 1)
    assert_stats(got, case["x"], lab, sub, case["K"])


def test_adaptive_switch_reads_mapped_counters(pkg, monkeypatch):
    monkeypatch.setenv("DPMM_LABEL_ADAPT", "1")
    case = make_niw_case(32, 12, 20000, seed=4, spread=0.3)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
    set_params(g, case)
    g.sample_labels(False)
    g.sync()                                # the counters of this call have arrived in host memory
    g.timing_enable(True)
    g.sample_labels(False)
    tim = g.timing_read()
    assert tim["label"][1] == 1 and tim["label_ovf"][1] == 0, tim      # the FMA kernel ran
    for _ in range(7):                      # the rest of the cool-down (8 calls)
        g.sample_labels(False)
    g.timing_read()
    g.sample_labels(False)                  # back on the tensor-core path, which the overflow kernel follows
    tim = g.timing_read()
    assert tim["label_ovf"][1] == 1, tim
    g.close()


def test_suff_stats_twice(converged):
    g, case = converged
    g.sample_labels(False)
    g.sample_sublabels()
    f0 = g.fused_stats()
    a = g.suff_stats()
    b = g.suff_stats()
    f1 = g.fused_stats()
    for u, v in zip(a, b):
        assert np.array_equal(u, v)
    assert f1[1] - f0[1] == 2 and f1[2] == f0[2], (f0, f1)   # both served from the fused accumulators, risk slot 0
    assert_stats(a, case["x"], g.get_labels(), g.get_sublabels(), case["K"])


def test_ragged_n_single_cluster(pkg):
    case = make_niw_case(32, 1, 128 * 40 + 37, seed=5)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=9)
    set_params(g, case)
    for _ in range(3):
        got = sweep(g)
        perm, moved = g.sort_state()
        assert moved == 0
        lab, sub = g.get_labels(), g.get_sublabels()
        assert np.all(lab == 1)
        assert_sorted(perm, lab - 1)
        assert_stats(got, case["x"], lab, sub, 1)
    g.close()
