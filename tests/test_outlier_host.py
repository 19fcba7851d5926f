"""The outlier component (fit / dp_parallel `outlier_weight`, `outlier_params`; DESIGN.md 6.1) on the host parameter path,
with the oracle standing in for the workers: cluster 1 under its own prior at a fixed weight, never split, merged or
removed, the compaction that keeps it, the refusals, and the advanced mode / checkpoints."""
import numpy as np
import pytest

import dpmm_pkg
from oracle import dpmm_oracle as O

pkg = dpmm_pkg.load()
from dpmmsubclusters_jl_b200 import host as H  # noqa: E402
from dpmmsubclusters_jl_b200 import checkpoint as CK  # noqa: E402
from dpmmsubclusters_jl_b200 import priors as P  # noqa: E402

OMEGA = 0.05
OUTLIER = P.niw_hyperparams(0.01, np.zeros(2), 5, 2500.0 * np.eye(2))
PRIOR = P.niw_hyperparams(1.0, np.zeros(2), 5, np.eye(2))


def oracle_factory(x, kind, seed, goff):
    return O.OracleSweep(x, kind, seed=seed, global_offset=goff)


def background_data(seed, n_in=1900, n_bg=100):
    """Three sigma = 1 Gaussians 20 apart plus n_bg points uniform on [-100, 100]^2; labels 1..3, background 0."""
    rng = np.random.default_rng(seed)
    centres = np.array([[-20.0, 0.0], [0.0, 0.0], [20.0, 0.0]])
    gt = rng.integers(1, 4, n_in)
    x_in = centres[gt - 1].T + rng.standard_normal((2, n_in))
    x_bg = rng.uniform(-100, 100, (2, n_bg))
    return np.concatenate([x_in, x_bg], 1).astype(np.float32), np.concatenate([gt, np.zeros(n_bg, np.int64)])


def _checked_steps(monkeypatch, check):
    """Run `check(group, cfg)` after every group_step."""
    step = H.group_step

    def wrapped(group, no_more_splits, final, first, cfg, rng):
        step(group, no_more_splits, final, first, cfg, rng)
        check(group, cfg)
    monkeypatch.setattr(H, "group_step", wrapped)


def _check_outlier_invariants(group, cfg):
    c1 = group.local_clusters[0].cluster_params
    assert c1.cluster_params.hyperparams is OUTLIER
    labels = group.sweep.get_labels()
    assert labels.max() <= len(group.local_clusters)
    counts = np.bincount(labels, minlength=len(group.local_clusters) + 1)[1:]
    assert list(counts) == [c.points_count for c in group.local_clusters]


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_background_points_go_to_the_outlier_component(monkeypatch, seed):
    x, gt = background_data(seed)
    weights_seen = []

    def check(group, cfg):
        _check_outlier_invariants(group, cfg)
        weights_seen.append(np.asarray(group.weights).copy())
    _checked_steps(monkeypatch, check)
    labels, _, weights, _, _, _, kh, _, dp = H.fit(x, PRIOR, 10.0, iters=150, seed=seed, outlier_weight=OMEGA,
                                                   outlier_params=OUTLIER, sweep_factory=oracle_factory)
    assert len(weights_seen) == 150
    for w in weights_seen + [weights]:
        assert w[0] == np.float32(OMEGA) and w[1:].sum() <= 0.95 + 1e-6
    bg, inl = gt == 0, gt > 0
    assert (labels[bg] == 1).mean() >= 0.80
    assert (labels[inl] == 1).mean() <= 0.01
    assert H.normalized_mutual_info(gt[inl], labels[inl]) >= 0.95
    c1 = dp.group.local_clusters[0].cluster_params.cluster_params
    assert c1.hyperparams is OUTLIER
    # the posterior of cluster 1 is that of its own prior, and calculate_posterior / predict see it
    assert c1.posterior_hyperparams.κ == pytest.approx(OUTLIER.κ + c1.suff_statistics.N)
    assert np.isfinite(H.calculate_posterior(dp))
    pl, _ = H.predict(dp, x, on_device=False)
    assert (pl[bg] == 1).mean() >= 0.8


def test_weight_zero_is_the_model_without_the_component():
    x, _ = background_data(4, n_in=600, n_bg=30)
    a = H.fit(x, PRIOR, 10.0, iters=30, seed=5, sweep_factory=oracle_factory)
    b = H.fit(x, PRIOR, 10.0, iters=30, seed=5, sweep_factory=oracle_factory, outlier_weight=0, outlier_params=OUTLIER)
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[2], b[2])


@pytest.mark.parametrize("weight, params, what", [
    (1.0, OUTLIER, "outlier_weight"), (-0.1, OUTLIER, "outlier_weight"), (float("nan"), OUTLIER, "outlier_weight"),
    (0.05, None, "needs outlier_params"),
    (0.05, P.multinomial_hyper(np.ones(2)), "niw_hyperparams"),
    (0.05, P.diag_niw_hyperparams(1.0, np.zeros(2), 5, np.ones(2)), "niw_hyperparams"),
    (0.05, P.niw_hyperparams(1.0, np.zeros(3), 6, np.eye(3)), "dimension"),
])
def test_refusals(weight, params, what):
    x, _ = background_data(5, n_in=60, n_bg=6)
    with pytest.raises(ValueError, match=what):
        H.fit(x, PRIOR, 10.0, iters=2, seed=1, sweep_factory=oracle_factory, outlier_weight=weight, outlier_params=params)


def test_compaction_keeps_the_empty_outlier_cluster(monkeypatch):
    """No background: cluster 1 stays empty.  The counts sent to remove_empty must keep it on the sweep as well, or
    every label moves down by one while the host still holds cluster 1."""
    rng = np.random.default_rng(6)
    gt = rng.integers(0, 3, 900)
    x = (np.array([[-20.0, 0.0, 20.0], [0.0, 0.0, 0.0]])[:, gt] + rng.standard_normal((2, 900))).astype(np.float32)
    empty_seen = []

    def check(group, cfg):
        _check_outlier_invariants(group, cfg)
        empty_seen.append(group.local_clusters[0].points_count == 0)
    _checked_steps(monkeypatch, check)
    H.fit(x, PRIOR, 10.0, iters=40, seed=2, outlier_weight=OMEGA, outlier_params=OUTLIER, sweep_factory=oracle_factory)
    assert len(empty_seen) == 40 and all(empty_seen)


PARAMS_JL = """
data_path = "{data_path}"
data_prefix = "pts"
iterations = 30
initial_clusters = 1
random_seed = 7
burnout_period = 5
α = 10.0
hyper_params = niw_hyperparams(1.0, zeros(Float32,2), 5, Matrix{{Float32}}(I, 2, 2)*1.0)
outlier_mod = 0.05
outlier_hyper_params = niw_hyperparams(0.01, zeros(Float32,2), 5, Matrix{{Float32}}(I, 2, 2)*2500.0)
enable_saving = true
model_save_interval = 10
save_path = "{save_path}"
save_file_prefix = "checkpoint_"
"""


def test_advanced_mode_and_checkpoints_carry_the_component(tmp_path):
    x, gt = background_data(7, n_in=950, n_bg=50)
    np.save(tmp_path / "pts.npy", x.T)
    f = tmp_path / "global_params.jl"
    f.write_text(PARAMS_JL.format(data_path=str(tmp_path) + "/", save_path=str(tmp_path) + "/"))
    dp, ic, _, _, kh = H.dp_parallel(str(f), verbose=False, sweep_factory=oracle_factory, device_params=False)
    assert len(ic) == 30
    assert dp.group.weights[0] == np.float32(0.05)
    c1 = dp.group.local_clusters[0].cluster_params.cluster_params
    assert isinstance(c1.hyperparams, P.niw_hyperparams) and c1.hyperparams.κ == pytest.approx(0.01)
    grp, mh, it, _, _ = CK.load_checkpoint(str(tmp_path / "checkpoint__10.npz"))
    assert it == 10 and grp["outlier_weight"] == 0.05
    oh = grp["outlier_params"]
    np.testing.assert_allclose(oh.ψ, 2500.0 * np.eye(2))
    assert grp["local_clusters"][0].cluster_params.cluster_params.hyperparams is oh
    assert grp["local_clusters"][1].cluster_params.cluster_params.hyperparams is mh.distribution_hyper_params
    assert grp["weights"][0] == np.float32(0.05)
    dp2, ic2, _, _, _ = H.run_model_from_checkpoint(str(tmp_path / "checkpoint__10.npz"), verbose=False,
                                                   sweep_factory=oracle_factory, device_params=False)
    assert len(ic2) == 20 and dp2.outlier_weight == 0.05
    assert dp2.group.weights[0] == np.float32(0.05)
    r1 = dp2.group.local_clusters[0].cluster_params.cluster_params
    np.testing.assert_allclose(r1.hyperparams.ψ, 2500.0 * np.eye(2))
    assert int((dp2.group.sweep.get_labels() == 1).sum()) == dp2.group.local_clusters[0].points_count


def test_parameter_file_without_outlier_hyper_params_leaves_the_component_off(tmp_path):
    f = tmp_path / "p.jl"
    f.write_text(PARAMS_JL.replace("outlier_hyper_params = niw_hyperparams(0.01, zeros(Float32,2), 5, "
                                   "Matrix{{Float32}}(I, 2, 2)*2500.0)", "")
                 .format(data_path="x", save_path="y"))
    cfg = H._settings_from_params(CK.read_params(str(f)), False, None)
    assert cfg.outlier_mod == 0.0 and cfg.outlier_hyper_params is None
