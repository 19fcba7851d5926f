"""GPU parity tests (run with -m gpu on a B200): the CUDA path, called through the C ABI, against
the CPU oracle on the same seeded inputs and the same injected uniforms.

Bars (north_star / SURVEY.md 8c): labels, sub-labels and counts bit-exact except documented near-ties;
log-likelihoods within 1e-4 relative; sum x / sum xx' within 1e-4 (relative to sqrt(S_ii S_jj));
multinomial count vectors exact; relabelling exact."""
import os

import numpy as np
import pytest

import dpmm_pkg
from oracle import dpmm_oracle as O
from tests.util import (check_draws, check_loglik, check_stats, compare_sweeps, make_mnm_case, make_niw_case,
                        set_params, tie_tolerance)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as g
    g.build()
    return dpmm_pkg.load()


NIW_CASES = [  # (D, K, n)
    (2, 6, 10000),     # config C1
    (1, 3, 1000), (3, 10, 5000), (4, 2, 777), (5, 7, 4099), (6, 3, 1500), (7, 3, 1500), (8, 9, 3000),
    (12, 4, 2048), (16, 5, 4000), (24, 3, 2000),
    (32, 20, 20000),   # config C2 shape
    (48, 3, 1500),
    (64, 12, 3000),    # config C5 shape
    (32, 1, 5000), (5, 50, 8000),   # K = 1; config C4 shape
    (32, 100, 3000),   # K large enough that the staged clusters are chunked
    (9, 4, 3000), (10, 6, 2500), (20, 5, 3000), (30, 8, 6000), (50, 3, 2000),   # no instantiated width: zero-padded
    (3, 700, 4000),    # K beyond the 4-points-per-thread tile: one point per thread
]


@pytest.mark.parametrize("D,K,n", NIW_CASES)
def test_niw_full_sweep_parity(pkg, D, K, n):
    case = make_niw_case(D, K, n, seed=100 + D + K)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
    o = O.OracleSweep(case["x"], O.NIW, seed=7)
    rep = compare_sweeps(g, o, case, np.random.default_rng(D * 1000 + K))
    g.close()
    print(f"D={D} K={K} n={n}: {rep}")


@pytest.mark.parametrize("spread,K,n", [(0.3, 12, 20000), (0.0, 5, 8000), (1.0, 23, 12000)])
def test_niw_tensor_core_refine_path_with_overlapping_clusters(pkg, spread, K, n):
    """D=32 runs on gauss_label_tc2_kernel from a cold start.  Heavily overlapping (or identical-centre)
    clusters make most points multi-candidate, so the exact FP32 evaluations (in the kernel or in its
    full-K overflow kernel) decide the labels; parity with the oracle must hold there too (incl. the final
    argmax mode)."""
    case = make_niw_case(32, K, n, seed=int(10 * spread) + K, spread=spread)
    for final in (False, True):
        g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
        o = O.OracleSweep(case["x"], O.NIW, seed=7)
        rep = compare_sweeps(g, o, case, np.random.default_rng(K), final=final)
        g.close()
    import os
    os.environ["DPMM_TC_STATS"] = "1"
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
    set_params(g, case)
    g.sample_labels(False)
    npts, ncand = g.tc_stats()
    g.close()
    os.environ.pop("DPMM_TC_STATS")
    assert npts == n, "the tensor-core path did not run"
    print(f"spread={spread} K={K}: refined evaluations per point = {ncand / npts:.2f}")
    if spread <= 0.3:
        assert ncand > npts          # the refine path really was exercised


TC2_CASES = [  # (D, K, n, spread)
    (32, 20, 20000, 10.0),    # C2 shape, well separated: almost every point is decided by its pivot
    (32, 20, 20000, 2.5),     # moderately separated: several candidates per point
    (32, 40, 30000, 10.0),    # K > 23 (the limit of the first-generation kernel)
    (32, 100, 20000, 10.0),   # screen over the last 8 features (KS = 8), 7 chunks
    (32, 200, 30000, 10.0),
    (32, 3, 300, 2.5),        # ragged tiles, more tiles than points per cluster
    (32, 12, 20000, 0.3),     # everything overlaps: the overflow kernel decides
    (64, 12, 6000, 10.0),
    (64, 100, 20000, 10.0),   # config C5 shape
    (64, 30, 10000, 1.0),
]


@pytest.mark.parametrize("D,K,n,spread", TC2_CASES)
def test_niw_tc2_label_kernel_from_warm_labels(pkg, D, K, n, spread):
    """D = 32 / 64: gauss_label_tc2_kernel walks the points in the order of their CURRENT labels and uses the
    tile's old cluster as the pivot.  compare_sweeps(warm=True) starts from the labels of an argmax pass,
    as an iteration deep inside a run would, so the pivot / partial-screen / exact-candidate path decides
    the draws (cold starts, covered by test_niw_full_sweep_parity, mostly take the overflow kernel)."""
    case = make_niw_case(D, K, n, seed=1000 + D + K, spread=spread)
    for final in (False, True):
        g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
        o = O.OracleSweep(case["x"], O.NIW, seed=7)
        rep = compare_sweeps(g, o, case, np.random.default_rng(K + D), final=final, warm=True)
        g.close()
    os.environ["DPMM_TC_STATS"] = "1"
    try:
        g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
        set_params(g, case)
        g.sample_labels(True)
        g.sample_labels(False)
        npts, ncand, novf = g.tc_stats(overflow=True)
        g.close()
    finally:
        os.environ.pop("DPMM_TC_STATS")
    assert npts == n, "the tensor-core path did not run"
    print(f"D={D} K={K} n={n} spread={spread}: {rep}; exact evaluations per point {ncand / npts:.3f}, "
          f"overflow points {novf} ({novf / npts:.4f})")
    if spread >= 10.0:
        assert novf <= 0.02 * npts, "well separated clusters must be decided by the pivot path"


@pytest.mark.parametrize("spread,K,n", [(2.5, 20, 30000), (10.0, 20, 100000), (10.0, 3, 40000)])
def test_niw_fused_sublabel_statistics_kernel(pkg, spread, K, n):
    """D=32: dpmm_sample_sublabels runs niw_substats_tc_kernel (sub-label draw + left/right statistics in one
    pass on tcgen05) and dpmm_suff_stats is served from its accumulators.  Full parity against the oracle at
    cluster means far from the origin (|x| ~ 50: the centre shift has to be exact), the fused path must
    really have run, and it must agree with the separate FP32 sub-label / statistics kernels."""
    case = make_niw_case(32, K, n, seed=int(spread) + K, spread=spread)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
    o = O.OracleSweep(case["x"], O.NIW, seed=7)
    rep = compare_sweeps(g, o, case, np.random.default_rng(K))
    fused, served, redone = g.fused_stats()
    g.close()
    assert fused >= 1 and served >= 1, "the fused sub-label + statistics kernel did not run"
    print(f"spread={spread} K={K} n={n}: {rep}; fused launches {fused}, served {served}, recomputed {redone}")
    rng = np.random.default_rng(3)
    u_label, u_sub = rng.random(n), rng.random(n)
    res = []
    for mode in ("1", "0"):
        os.environ["DPMM_SUBSTATS_TC"] = mode
        try:
            g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
            g.set_uniforms(u_label, u_sub, np.zeros(n, np.uint8))
            set_params(g, case)
            g.sample_labels(False)
            ll = g.debug_loglik(1)
            g.sample_sublabels()
            res.append((ll, g.get_sublabels(), g.suff_stats(), g.fused_stats()))
            g.close()
        finally:
            os.environ.pop("DPMM_SUBSTATS_TC")
    (ll1, s1, st1, f1), (ll0, s0, st0, f0) = res
    assert f1[0] >= 1 and f0[0] == 0
    check_loglik(ll1, ll0, "fused vs FP32 sub-label log-likelihood")
    check_draws(ll0.astype(np.float32), u_sub, s1, s0, "fused vs FP32 sub-labels")
    if np.array_equal(s1, s0):
        check_stats(st1, st0, O.NIW, "fused vs separate statistics")


@pytest.mark.parametrize("spread,K,n,empty", [(2.5, 12, 30000, None), (30.0, 100, 60000, None), (10.0, 3, 129, None),
                                              (10.0, 4, 5000, 2), (40.0, 2, 1025, 0), (2.5, 40, 900, None)])
def test_niw_d64_tensor_core_sublabel_kernel(pkg, spread, K, n, empty):
    """D = 64: dpmm_sample_sublabels runs niw_sublabel_tc64_kernel (3-term TF32 product on tcgen05, M = N = 128).  Full
    parity against the oracle at cluster means far from the origin, ragged tiles and empty clusters, the kernel must
    really have run, and it must agree with the FP32 sub-label kernel on log-likelihoods and draws."""
    case = make_niw_case(64, K, n, seed=int(spread) + K + n, spread=spread)
    if empty is not None:
        w = case["weights"].astype(np.float64)
        w[empty] = 1e-30
        case["weights"] = (w / w.sum()).astype(np.float32)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
    o = O.OracleSweep(case["x"], O.NIW, seed=7)
    rep = compare_sweeps(g, o, case, np.random.default_rng(K))
    g.close()
    rng = np.random.default_rng(3)
    u_label, u_sub = rng.random(n), rng.random(n)
    res = []
    for mode in ("1", "0"):
        os.environ["DPMM_SUBLABEL_TC64"] = mode
        try:
            g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
            g.set_uniforms(u_label, u_sub, np.zeros(n, np.uint8))
            set_params(g, case)
            g.sample_labels(False)
            ll = g.debug_loglik(1)
            g.timing_enable(True)
            g.sample_sublabels()
            tim = g.timing_read()
            res.append((ll, g.get_sublabels(), tim["sublabel"][0]))
            g.close()
        finally:
            os.environ.pop("DPMM_SUBLABEL_TC64")
    (ll1, s1, t1), (ll0, s0, t0) = res
    check_loglik(ll1, ll0, "tcgen05 vs FP32 sub-label log-likelihood (D = 64)")
    check_draws(ll0.astype(np.float32), u_sub, s1, s0, "tcgen05 vs FP32 sub-labels (D = 64)")
    print(f"spread={spread} K={K} n={n}: {rep}; sub-label {t1 * 1e3:.1f} us (FP32 kernel {t0 * 1e3:.1f} us)")


@pytest.mark.parametrize("K,n,empty", [(3, 1, None), (5, 129, None), (4, 4000, 2), (2, 257, 0), (40, 900, None)])
def test_niw_fused_kernel_edge_shapes(pkg, K, n, empty):
    """Ragged and degenerate tile sequences of the fused D=32 kernel: a single point, one row past a tile,
    an empty cluster in the middle / at the front of the label-sorted order, more clusters than tiles."""
    case = make_niw_case(32, K, n, seed=K * 7 + n)
    if empty is not None:
        w = case["weights"].astype(np.float64)
        w[empty] = 1e-30                      # nobody draws this label: its segment is empty
        case["weights"] = (w / w.sum()).astype(np.float32)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=11)
    o = O.OracleSweep(case["x"], O.NIW, seed=11)
    rep = compare_sweeps(g, o, case, np.random.default_rng(n))
    fused, served, redone = g.fused_stats()
    g.close()
    assert fused >= 1 or n < 128          # contexts with fewer points than one tile stay on the FP32 kernels
    print(f"K={K} n={n} empty={empty}: {rep}; fused {fused}, served {served}, recomputed {redone}")


@pytest.mark.parametrize("K,n,spread,empty", [(12, 30000, 10.0, None), (100, 60000, 30.0, None), (3, 1, 10.0, None),
                                              (5, 129, 0.5, None), (4, 5000, 10.0, 2), (2, 1025, 40.0, 0), (40, 900, 2.5, None)])
def test_niw_d64_tensor_core_statistics_kernel(pkg, K, n, spread, empty):
    """niw_stats_tc64_kernel (D = 64, all clusters; M = 128 x N = 64 MN-major tcgen05 rank-8 updates) against the oracle
    and against the FP32 -> FP64 kernel it replaces: ragged tiles, empty clusters, runs far from the origin."""
    case = make_niw_case(64, K, n, seed=K * 3 + n, spread=spread)
    if empty is not None:
        w = case["weights"].astype(np.float64)
        w[empty] = 1e-30
        case["weights"] = (w / w.sum()).astype(np.float32)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=4)
    set_params(g, case)
    g.sample_labels(False); g.sample_sublabels()
    lab, sub = g.get_labels(), g.get_sublabels()
    g.timing_enable(True)
    got = g.suff_stats()
    tim = g.timing_read()
    o = O.OracleSweep(case["x"], O.NIW, seed=4)
    o.K = K
    o.set_labels(lab); o.set_sublabels(sub)
    err = check_stats(got, o.suff_stats(), O.NIW, "D=64 tensor-core statistics")
    os.environ["DPMM_STATS_TC"] = "0"
    try:
        ref = g.suff_stats()
    finally:
        os.environ.pop("DPMM_STATS_TC")
    check_stats(got, ref, O.NIW, "D=64 tensor-core vs FP32 statistics kernel")
    g.close()
    print(f"K={K} n={n}: stats_err {err:.2e}; stats {tim['stats'][0] * 1e3:.1f} us")


def test_small_dimension_statistics_kernel_on_a_large_input(pkg):
    """D <= 8 and n >= 2^18 points: the statistics run on niw_stats_small_kernel (one warp per run chunk)."""
    n, D, K = 300_000, 5, 12
    case = make_niw_case(D, K, n, seed=31)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=4)
    set_params(g, case)
    g.sample_labels(False); g.sample_sublabels()
    lab, sub = g.get_labels(), g.get_sublabels()
    counts, sx, sxx = g.suff_stats()
    o = O.OracleSweep(case["x"], O.NIW, seed=4)
    o.K = K
    o.set_labels(lab); o.set_sublabels(sub)
    check_stats((counts, sx, sxx), o.suff_stats(), O.NIW, "small-D statistics kernel")
    os.environ["DPMM_STATS_SMALL"] = "0"
    try:
        c2, sx2, sxx2 = g.suff_stats([2, 1])
    finally:
        os.environ.pop("DPMM_STATS_SMALL")
    check_stats((c2, sx2, sxx2), (counts[[1, 0]], sx[[1, 0]], sxx[[1, 0]]), O.NIW, "small-D vs cooperative kernel")
    g.close()


def test_suff_stats_out_argument_reuses_the_result_arrays(pkg):
    case = make_niw_case(32, 4, 3000, seed=2)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=3)
    set_params(g, case)
    g.sample_labels(False); g.sample_sublabels()
    a = g.suff_stats()
    b = g.suff_stats(out=tuple(np.full_like(v, -1) for v in a))
    for u, v in zip(a, b):
        np.testing.assert_array_equal(u, v)
    c = g.suff_stats(out=b)
    assert all(u is v for u, v in zip(b, c))
    with pytest.raises(ValueError):
        g.suff_stats([1], out=b)
    g.close()


def test_niw_fused_statistics_fall_back_when_a_run_is_far_from_its_centre(pkg):
    """The fused kernel accumulates sums about the cluster's centre c.  When the points of a run are much
    closer to the origin than to c in some component (here: x_0 ~ 0.01 while every mean says 30), the
    centred sums cannot resolve the un-centred sum x_0^2; the finalise kernel counts such entries and
    dpmm_suff_stats recomputes with the FP32/FP64 statistics kernel.  Parity must hold either way."""
    K, n = 4, 6000
    case = make_niw_case(32, K, n, seed=5)
    case["x"][0, :] = (0.01 * np.random.default_rng(1).standard_normal(n)).astype(np.float32)
    case["mu"][:, :, 0] = 30.0
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
    o = O.OracleSweep(case["x"], O.NIW, seed=7)
    compare_sweeps(g, o, case, np.random.default_rng(2))
    fused, served, redone = g.fused_stats()
    g.close()
    assert fused >= 1 and redone >= 1, (fused, served, redone)


@pytest.mark.parametrize("D,K,n", [(2, 6, 5000), (32, 20, 10000), (64, 4, 2000)])
def test_niw_final_argmax_parity(pkg, D, K, n):
    case = make_niw_case(D, K, n, seed=5)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
    o = O.OracleSweep(case["x"], O.NIW, seed=7)
    compare_sweeps(g, o, case, np.random.default_rng(1), final=True)
    g.close()


MNM_CASES = [(100, 20, 20000), (100, 2, 1000), (10, 5, 3000), (33, 17, 2500), (257, 3, 600), (7, 40, 4000)]


@pytest.mark.parametrize("D,K,n", MNM_CASES)
def test_multinomial_full_sweep_parity(pkg, D, K, n):
    case = make_mnm_case(D, K, n, seed=200 + D)
    g = pkg.GpuSweep(case["x"], pkg.MULTINOMIAL, seed=9)
    o = O.OracleSweep(case["x"], O.MULTINOMIAL, seed=9)
    rep = compare_sweeps(g, o, case, np.random.default_rng(D))
    g.close()
    print(f"mnm D={D} K={K} n={n}: {rep}")


def test_multinomial_final_argmax(pkg):
    case = make_mnm_case(100, 20, 5000, seed=4)
    g = pkg.GpuSweep(case["x"], pkg.MULTINOMIAL, seed=9)
    o = O.OracleSweep(case["x"], O.MULTINOMIAL, seed=9)
    compare_sweeps(g, o, case, np.random.default_rng(2), final=True)
    g.close()


def test_philox_streams_match_oracle(pkg):
    """Without injected uniforms both sides draw from Philox keyed by the global point index, so a
    whole sweep agrees (up to near-ties) and sharding does not change the stream."""
    case = make_niw_case(8, 5, 6000, seed=11)
    off = 2 ** 32 - 1000                      # crosses into the second counter word
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=0xDEADBEEFCAFE, global_offset=off)
    o = O.OracleSweep(case["x"], O.NIW, seed=0xDEADBEEFCAFE, global_offset=off)
    for s in (g, o):
        s.init_labels(3)
    np.testing.assert_array_equal(g.get_labels(), o.get_labels())
    np.testing.assert_array_equal(g.get_sublabels(), o.get_sublabels())
    assert set(np.unique(g.get_labels())) == {1, 2, 3}
    for s in (g, o):
        set_params(s, case)
        s.sample_labels(False)
    u = O.philox_uniform(0xDEADBEEFCAFE, O.STREAM_LABEL, o.call, o.gidx)
    check_draws(o.debug_loglik(0), u, g.get_labels(), o.get_labels(), "philox labels")
    o.set_labels(g.get_labels())
    for s in (g, o):
        s.sample_sublabels()
    u = O.philox_uniform(0xDEADBEEFCAFE, O.STREAM_SUBLABEL, o.call, o.gidx)
    check_draws(o.debug_loglik(1), u, g.get_sublabels(), o.get_sublabels(), "philox sub-labels")
    for s in (g, o):
        s.randomize_sublabels([2, 4])
    o.set_sublabels(np.where(np.isin(o.get_labels(), [2, 4]), o.get_sublabels(), g.get_sublabels()))
    np.testing.assert_array_equal(g.get_sublabels(), o.get_sublabels())
    g.close()


def test_golden_niw_checkpoint_through_cabi(pkg, golden_dir):
    """Stage 3 against the statistics stored in the reference's own checkpoint__50.jld2."""
    gd = np.load(os.path.join(golden_dir, "niw_2d1k_checkpoint50.npz"))
    g = pkg.GpuSweep(gd["x"].astype(np.float32), pkg.NIW)
    g.set_labels(gd["labels"]); g.set_sublabels(gd["sublabels"])
    g.K = 5
    got = g.suff_stats()
    check_stats(got, (gd["counts"], gd["sum_x"], gd["sum_xx"]), O.NIW, "golden NIW checkpoint")
    g.close()


def test_golden_multinomial_checkpoint_bytes_through_cabi(pkg, golden_dir):
    gd = np.load(os.path.join(golden_dir, "mnm_1k_checkpoint20.npz"))
    g = pkg.GpuSweep(gd["x"], pkg.MULTINOMIAL)
    g.set_labels(gd["labels"]); g.set_sublabels(gd["sublabels"])
    g.K = 2
    counts, sum_x, _ = g.suff_stats()
    np.testing.assert_array_equal(counts, gd["counts"])
    assert sum_x.astype(np.float32).tobytes() == gd["sum_x"].tobytes()   # byte-exact with the reference's Float32
    g.close()


def test_edge_cases(pkg):
    rng = np.random.default_rng(0)
    # a single point
    case = make_niw_case(3, 2, 1, seed=1)
    g = pkg.GpuSweep(case["x"], pkg.NIW); o = O.OracleSweep(case["x"], O.NIW)
    compare_sweeps(g, o, case, rng); g.close()
    # empty clusters (K larger than the labels in use) and empty sides give zero statistics
    case = make_niw_case(4, 6, 500, seed=2)
    g = pkg.GpuSweep(case["x"], pkg.NIW); o = O.OracleSweep(case["x"], O.NIW)
    lab = rng.integers(1, 3, 500); sub = np.ones(500, np.int64)
    for s in (g, o):
        set_params(s, case); s.set_labels(lab); s.set_sublabels(sub)
    gs, os_ = g.suff_stats(), o.suff_stats()
    check_stats(gs, os_, O.NIW, "empty clusters")
    assert (gs[0][2:] == 0).all() and (gs[0][:, 2] == 0).all()
    g.close()
    # NaN / -Inf log-likelihoods: a non-PD invSigma gives NaN for that cluster -> treated as -Inf when
    # sampling (utils.jl:21); all clusters NaN -> label 1
    case = make_niw_case(2, 3, 400, seed=3)
    case["inv_sigma"][1, 0] = np.array([[1, 2], [2, 1]], np.float32)   # indefinite
    g = pkg.GpuSweep(case["x"], pkg.NIW)
    set_params(g, case)
    ll = g.debug_loglik(0)
    assert np.isnan(ll[:, 1]).all() and np.isfinite(ll[:, [0, 2]]).all()
    g.set_uniforms(rng.random(400), None, None)
    g.sample_labels(False)
    assert not (g.get_labels() == 2).any()
    for k in range(3):
        case["inv_sigma"][k, 0] = np.array([[1, 2], [2, 1]], np.float32)
    set_params(g, case)
    g.sample_labels(False)
    assert (g.get_labels() == 1).all()
    g.sample_labels(True)          # argmax branch: NaN is maximal, first index wins
    assert (g.get_labels() == 1).all()
    g.close()


def test_ill_conditioned_inverse_covariance_stays_finite_and_matches_the_oracle(pkg):
    """ADVICE r1: a Float32-rounded invSigma of a nearly collinear cluster (condition number ~1e8) is not exactly
    positive definite any more; the reference's direct z' invSigma z (which the oracle follows) stays finite, and
    so must the factored form (tiny diagonal jitter in niw_pack_kernel), within the 1e-4 tolerance."""
    rng = np.random.default_rng(8)
    D, K, n = 8, 3, 4000
    case = make_niw_case(D, K, n, seed=9)
    v = rng.standard_normal(D); v /= np.linalg.norm(v)
    for k in range(K):
        Sig = np.linalg.inv(case["inv_sigma"][k, 0].astype(np.float64))
        Sig = Sig + 3e7 * np.outer(v, v)                 # one very long axis: cond(Sigma) ~ 1e8
        case["inv_sigma"][k, 0] = np.linalg.inv(Sig)     # Float64 inverse rounded to Float32
        case["logdet"][k, 0] = np.linalg.slogdet(Sig)[1]
    g = pkg.GpuSweep(case["x"], pkg.NIW); o = O.OracleSweep(case["x"], O.NIW)
    for s_ in (g, o):
        set_params(s_, case)
    got, want = g.debug_loglik(0), o.debug_loglik(0)
    assert np.isfinite(got).all() and np.isfinite(want).all()
    # the quadratic form itself is ill conditioned in Float32 on both sides: compare on the scale of the row
    err = np.abs(got.astype(np.float64) - want) / np.maximum(np.abs(want), 1.0)
    assert err.max() <= 2e-3, err.max()
    g.close()


def test_error_behaviour(pkg):
    E = pkg._lib
    x = np.zeros((2, 16), np.float32)
    g = pkg.GpuSweep(x, pkg.NIW)
    with pytest.raises(E.DpmmError) as ei:
        g.sample_labels()
    assert ei.value.code == E.ESTATE
    with pytest.raises(E.DpmmError) as ei:
        g.set_labels(np.zeros(16, np.int64))          # labels are 1-based
    assert ei.value.code == E.EINVAL
    with pytest.raises(E.DpmmError) as ei:
        g.set_params_multinomial(np.zeros((1, 3, 2), np.float32), np.ones(1, np.float32), np.ones(2, np.float32))
    assert ei.value.code == E.ESTATE
    g.close()
    with pytest.raises(E.DpmmError) as ei:
        pkg.GpuSweep(np.zeros((65, 4), np.float32), pkg.NIW)    # NIW: D <= 64
    assert ei.value.code == E.ELIMIT


def test_gumbel_sampler_is_statistically_equivalent(pkg):
    case = make_niw_case(2, 4, 200000, seed=21, spread=0.8)
    case["x"][:] = case["x"][:, :1]                    # every point identical -> one categorical law
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=3)
    set_params(g, case)
    ll = g.debug_loglik(0)[0].astype(np.float64)
    p = np.exp(ll - ll.max()); p /= p.sum()
    freqs = []
    for sampler in (pkg._lib.SAMPLER_INVERSE_CDF, pkg._lib.SAMPLER_GUMBEL):
        g.set_sampler(sampler)
        g.sample_labels(False)
        freqs.append(np.bincount(g.get_labels(), minlength=5)[1:] / case["n"])
    g.close()
    for f in freqs:
        np.testing.assert_allclose(f, p, atol=5e-3)


def test_full_size_properties_c2(pkg):
    """BASELINE config C2 shape (N=1e6, D=32, K=20): size-independent properties + oracle parity on a
    random sub-sample of points (the draw of a point depends only on that point and the parameters)."""
    n, D, K = 1_000_000, 32, 20
    case = make_niw_case(D, K, n, seed=77)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=123)
    set_params(g, case)
    g.sample_labels(False); g.sample_sublabels()
    lab, sub = g.get_labels(), g.get_sublabels()
    counts, sx, sxx = g.suff_stats()
    assert lab.min() >= 1 and lab.max() <= K and set(np.unique(sub)) <= {1, 2}
    np.testing.assert_array_equal(counts[:, 0], np.bincount(lab, minlength=K + 1)[1:])
    np.testing.assert_array_equal(counts[:, 1], np.bincount(lab[sub == 1], minlength=K + 1)[1:])
    np.testing.assert_array_equal(counts[:, 0], counts[:, 1] + counts[:, 2])
    np.testing.assert_allclose(sx[:, 0], sx[:, 1] + sx[:, 2], rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(sxx[:, 0], sxx[:, 1] + sxx[:, 2], rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(sx[:, 0].sum(0), case["x"].astype(np.float64).sum(1), rtol=1e-6)
    tot = case["x"].astype(np.float64) @ case["x"].astype(np.float64).T
    np.testing.assert_allclose(sxx[:, 0].sum(0), tot, rtol=1e-5, atol=1e-5 * np.abs(tot).max())
    # oracle on a sub-sample with the same Philox draws
    sel = np.sort(np.random.default_rng(0).choice(n, 20000, replace=False))
    o = O.OracleSweep(case["x"][:, sel], O.NIW, seed=123)
    o.gidx = sel.astype(np.uint64)
    set_params(o, case)
    o.sample_labels(False)
    u = O.philox_uniform(123, O.STREAM_LABEL, 1, o.gidx)
    check_draws(o.debug_loglik(0), u, lab[sel], o.get_labels(), "C2 labels (sub-sample)")
    o.set_labels(lab[sel])
    o.sample_sublabels()
    u = O.philox_uniform(123, O.STREAM_SUBLABEL, 2, o.gidx)
    check_draws(o.debug_loglik(1), u, sub[sel], o.get_sublabels(), "C2 sub-labels (sub-sample)")
    # idempotence of the statistics and a relabel round trip at full size
    c2, sx2, sxx2 = g.suff_stats()
    np.testing.assert_array_equal(counts, c2)
    np.testing.assert_allclose(sxx, sxx2, rtol=1e-6, atol=1e-6 * np.abs(sxx).max())
    g.apply_split([1], [K + 1])
    lab2 = g.get_labels()
    np.testing.assert_array_equal(lab2 == K + 1, (lab == 1) & (sub == 2))
    g.apply_merge([1], [K + 1])
    np.testing.assert_array_equal(g.get_labels(), lab)
    s2 = g.get_sublabels()
    np.testing.assert_array_equal(s2[lab == 1], sub[lab == 1])      # former-1 points -> 1, former-(K+1) -> 2
    g.close()


def test_full_size_properties_c3_multinomial(pkg):
    """BASELINE config C3 shape (multinomial, N=1e6, D=100, K=20): size-independent properties (count vectors are
    exact integers, so sums over clusters equal the column sums of X bit for bit) + oracle parity on a sub-sample."""
    n, D, K = 1_000_000, 100, 20
    case = make_mnm_case(D, K, n, seed=78)
    g = pkg.GpuSweep(case["x"], pkg.MULTINOMIAL, seed=321)
    set_params(g, case)
    g.sample_labels(False); g.sample_sublabels()
    lab, sub = g.get_labels(), g.get_sublabels()
    counts, sx, _ = g.suff_stats()
    assert lab.min() >= 1 and lab.max() <= K and set(np.unique(sub)) <= {1, 2}
    np.testing.assert_array_equal(counts[:, 0], np.bincount(lab, minlength=K + 1)[1:])
    np.testing.assert_array_equal(counts[:, 1], np.bincount(lab[sub == 1], minlength=K + 1)[1:])
    np.testing.assert_array_equal(sx[:, 0], sx[:, 1] + sx[:, 2])
    np.testing.assert_array_equal(sx[:, 0].sum(0), case["x"].astype(np.float64).sum(1))
    k0 = int(np.argmax(counts[:, 0]))
    np.testing.assert_array_equal(sx[k0, 1], case["x"][:, (lab == k0 + 1) & (sub == 1)].astype(np.float64).sum(1))
    sel = np.sort(np.random.default_rng(0).choice(n, 20000, replace=False))
    o = O.OracleSweep(case["x"][:, sel], O.MULTINOMIAL, seed=321)
    o.gidx = sel.astype(np.uint64)
    set_params(o, case)
    o.sample_labels(False)
    u = O.philox_uniform(321, O.STREAM_LABEL, 1, o.gidx)
    check_draws(o.debug_loglik(0), u, lab[sel], o.get_labels(), "C3 labels (sub-sample)")
    o.set_labels(lab[sel])
    o.sample_sublabels()
    u = O.philox_uniform(321, O.STREAM_SUBLABEL, 2, o.gidx)
    check_draws(o.debug_loglik(1), u, sub[sel], o.get_sublabels(), "C3 sub-labels (sub-sample)")
    g.apply_split([k0 + 1], [K + 1])
    np.testing.assert_array_equal(g.get_labels() == K + 1, (lab == k0 + 1) & (sub == 2))
    g.apply_merge([k0 + 1], [K + 1])
    np.testing.assert_array_equal(g.get_labels(), lab)
    g.close()


def test_full_size_properties_c4_image_segmentation_shape(pkg):
    """BASELINE config C4 shape (NIW, N=1e7, D=5, K=50): properties at full size + oracle parity on a sub-sample."""
    n, D, K = 10_000_000, 5, 50
    case = make_niw_case(D, K, n, seed=79, spread=3.0)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=55)
    set_params(g, case)
    g.sample_labels(False); g.sample_sublabels()
    lab, sub = g.get_labels(), g.get_sublabels()
    counts, sx, sxx = g.suff_stats()
    assert lab.min() >= 1 and lab.max() <= K and set(np.unique(sub)) <= {1, 2}
    np.testing.assert_array_equal(counts[:, 0], np.bincount(lab, minlength=K + 1)[1:])
    np.testing.assert_array_equal(counts[:, 1], np.bincount(lab[sub == 1], minlength=K + 1)[1:])
    np.testing.assert_array_equal(counts[:, 0], counts[:, 1] + counts[:, 2])
    np.testing.assert_allclose(sx[:, 0], sx[:, 1] + sx[:, 2], rtol=1e-12, atol=1e-9)
    np.testing.assert_allclose(sx[:, 0].sum(0), case["x"].astype(np.float64).sum(1), rtol=1e-6)
    tot = case["x"].astype(np.float64) @ case["x"].astype(np.float64).T
    np.testing.assert_allclose(sxx[:, 0].sum(0), tot, rtol=1e-5, atol=1e-5 * np.abs(tot).max())
    sel = np.sort(np.random.default_rng(0).choice(n, 20000, replace=False))
    o = O.OracleSweep(case["x"][:, sel], O.NIW, seed=55)
    o.gidx = sel.astype(np.uint64)
    set_params(o, case)
    o.sample_labels(False)
    u = O.philox_uniform(55, O.STREAM_LABEL, 1, o.gidx)
    check_draws(o.debug_loglik(0), u, lab[sel], o.get_labels(), "C4 labels (sub-sample)")
    o.set_labels(lab[sel])
    o.sample_sublabels()
    u = O.philox_uniform(55, O.STREAM_SUBLABEL, 2, o.gidx)
    check_draws(o.debug_loglik(1), u, sub[sel], o.get_sublabels(), "C4 sub-labels (sub-sample)")
    g.close()


def test_suff_stats_all_after_a_split_sizes_its_result_by_the_label_bound(pkg):
    """ADVICE r1: dpmm_suff_stats(indices = NULL) writes one row per label value in use; after apply_split that is
    K + 1.  The Python mirror sizes its arrays from dpmm_num_clusters, and a wrong n_indices is refused."""
    import ctypes as C
    case = make_niw_case(4, 3, 2000, seed=3)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=1)
    set_params(g, case)
    g.sample_labels(False); g.sample_sublabels()
    c0 = g.suff_stats()[0]
    assert c0.shape == (3, 3)
    g.apply_split([1], [4])
    c1 = g.suff_stats()[0]                       # no manual K patching
    assert c1.shape == (4, 3) and c1[:, 0].sum() == 2000 and c1[3, 0] == c0[0, 2]
    small = np.zeros((3, 3), np.int64)
    rc = g.lib.dpmm_suff_stats(g.h, None, 3, small.ctypes.data_as(C.POINTER(C.c_int64)), None, None)
    assert rc == pkg._lib.EINVAL
    g.close()


def test_label_path_adapts_to_overlapping_clusters(pkg, monkeypatch):
    """With heavily overlapping clusters nearly every cluster is a candidate of every point: the tensor-core kernel's
    counters say so, and the following calls run on a fallback label kernel instead for a while.  Either path gives
    the oracle's labels."""
    monkeypatch.setenv("DPMM_LABEL_ADAPT", "1")
    monkeypatch.setenv("DPMM_TC_STATS", "1")
    case = make_niw_case(32, 12, 20000, seed=4, spread=0.3)
    g = pkg.GpuSweep(case["x"], pkg.NIW, seed=7)
    o = O.OracleSweep(case["x"], O.NIW, seed=7)
    rng = np.random.default_rng(1)
    ran_tc = []
    for it in range(4):
        u = rng.random(case["n"])
        for s_ in (g, o):
            s_.set_uniforms(u, None, None)
            set_params(s_, case)
            s_.sample_labels(False)
        gl = g.get_labels()                      # (synchronises: the counters of this call have arrived)
        ran_tc.append(g.tc_stats()[0] == case["n"] if it == 0 else None)
        check_draws(o.debug_loglik(0), u, gl, o.get_labels(), f"labels, call {it}")
        o.set_labels(gl)
    assert ran_tc[0], "the first call must take the tensor-core kernel"
    g.timing_enable(True)
    g.sample_labels(False)
    tim = g.timing_read()
    g.close()
    # still cooling down: one launch of the fallback kernel, and no overflow kernel, which follows every tc2 launch
    assert tim["label"][1] == 1 and tim["label_ovf"][1] == 0, tim
