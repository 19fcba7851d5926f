"""Checkpoint / data I/O of the advanced mode (SURVEY 8f-4): load_data (utils.jl:5-14), parameter files
(global_params.jl), save_model / run_model_from_checkpoint (dp-parallel-sampling.jl:428-456)."""
import os

import numpy as np
import pytest

import dpmm_pkg
from oracle import dpmm_oracle as O

pkg = dpmm_pkg.load()
from dpmmsubclusters_jl_b200 import host as H  # noqa: E402
from dpmmsubclusters_jl_b200 import checkpoint as CK  # noqa: E402
from dpmmsubclusters_jl_b200 import priors as P  # noqa: E402


def oracle_factory(x, kind, seed, goff):
    return O.OracleSweep(x, kind, seed=seed, global_offset=goff)


PARAMS_JL = """
#Data Loading specifics
data_path = "{data_path}"
data_prefix = "pts"  #If the data file name is bob.npy, this should be 'bob'

#Model Parameters
iterations = {iters}
hard_clustering = false  #Soft or hard assignments
initial_clusters = 1
argmax_sample_stop = 5 #Change to hard assignment from soft at iterations - argmax_sample_stop
split_stop  = 5#Stop split/merge moves at  iterations - split_stop

random_seed = 7 #When nothing, a random seed will be used.

max_split_iter = 20
burnout_period = 5
max_clusters = Inf

#Model hyperparams
α = 10.0 #Concetration Parameter
hyper_params = niw_hyperparams(1.0,
    zeros(Float32,2),
    5,
    Matrix{{Float32}}(I, 2, 2)*1.0)

outlier_mod = 0.05 #Concetration Parameter

#Saving specifics:
enable_saving = true
model_save_interval = {interval}
save_path = "{save_path}"
overwrite_prec = false
save_file_prefix = "checkpoint_"

smart_splits = false
"""


def test_load_data_matches_the_reference_loader(tmp_path):
    a = np.arange(12, dtype=np.float32).reshape(4, 3)
    a[1, 2] = np.nan
    np.save(tmp_path / "bob.npy", a)
    x = CK.load_data(str(tmp_path) + "/", prefix="bob")
    assert x.shape == (3, 4) and x[2, 1] == 0.0 and not np.isnan(x).any()
    np.testing.assert_array_equal(CK.load_data(str(tmp_path) + "/", prefix="bob", swapDimension=False)[0], a[0])


def test_load_data_reads_the_reference_fixtures(tmp_path, golden_dir):
    """The reference's data files examples/save_load_model/2d1ksample.npy (1000 x 2 Float64) and
    test/save_load_test/mnm_data.npy (1000 x 100 Float32), N x D on disk, restored from the golden fixtures that
    tests/golden/make_golden.py stored them in (D x N, same values)."""
    gn = np.load(os.path.join(golden_dir, "niw_2d1k_checkpoint50.npz"))
    gm = np.load(os.path.join(golden_dir, "mnm_1k_checkpoint20.npz"))
    np.save(tmp_path / "2d1ksample.npy", gn["x"].T)
    np.save(tmp_path / "mnm_data.npy", gm["x"].T)
    x = CK.load_data(str(tmp_path) + "/", prefix="2d1ksample")
    assert x.shape == (2, 1000)
    np.testing.assert_array_equal(x, gn["x"])
    m = CK.load_data(str(tmp_path) + "/", prefix="mnm_data")
    assert m.shape[0] == 100 and (m.sum(0) == 50).all()          # generate_mnmm_data: 50 trials per point
    np.testing.assert_array_equal(m, gm["x"])


def test_parameter_file_in_the_reference_style(tmp_path):
    f = tmp_path / "global_params.jl"
    f.write_text(PARAMS_JL.format(data_path=str(tmp_path) + "/", iters=30, interval=10, save_path=str(tmp_path) + "/"))
    gp = CK.read_params(str(f))
    assert gp["iterations"] == 30 and gp["hard_clustering"] is False and gp["random_seed"] == 7
    assert gp["max_clusters"] == np.inf and gp["α"] == 10.0 and gp["model_save_interval"] == 10
    hp = gp["hyper_params"]
    assert isinstance(hp, P.niw_hyperparams) and hp.ν == 5 and hp.m.shape == (2,)
    np.testing.assert_array_equal(hp.ψ, np.eye(2))


def _advanced_run(tmp_path, device_params, factory, iters=30, interval=10):
    x, labels, _, _ = pkg.generate_gaussian_data(1200, 2, 3, 100.0, np.random.default_rng(1))
    np.save(tmp_path / "pts.npy", x.T)                      # N x D on disk, as the reference expects (swapDimension)
    f = tmp_path / "global_params.jl"
    f.write_text(PARAMS_JL.format(data_path=str(tmp_path) + "/", iters=iters, interval=interval, save_path=str(tmp_path) + "/"))
    out = H.dp_parallel(str(f), verbose=False, gt=labels, sweep_factory=factory, device_params=device_params)
    return x, labels, f, out


def test_advanced_mode_saves_and_resumes_on_the_oracle(tmp_path):
    x, labels, f, out = _advanced_run(tmp_path, False, oracle_factory)
    dp_model, iter_count, nmi, _, kh = out
    assert len(iter_count) == 30 and nmi[-1] > 0.9
    for it in (10, 20, 30):
        assert os.path.exists(tmp_path / f"checkpoint__{it}.npz")     # path * prefix * "_" * iter (save_model :452)
    grp, mh, it, total_time, gparams = CK.load_checkpoint(str(tmp_path / "checkpoint__20.npz"))
    assert it == 20 and gparams["model_params"] == str(f) and grp["labels"].shape == (1200,)
    assert len(grp["local_clusters"]) == kh[19]
    # the stored posteriors are those of the stored statistics (what the golden test checks on the reference's file)
    for k, c in enumerate(grp["local_clusters"]):
        cp = c.cluster_params.cluster_params
        post = P.calc_posterior(mh.distribution_hyper_params, cp.suff_statistics)
        np.testing.assert_allclose(post.ψ, cp.posterior_hyperparams.ψ, rtol=1e-12)
        cnt = int((grp["labels"] == k + 1).sum())
        assert cnt == c.points_count == int(cp.suff_statistics.N)
    # resume: iterations 21..30 run, the model ends in the same place
    dp2, ic2, nmi2, _, kh2 = H.run_model_from_checkpoint(str(tmp_path / "checkpoint__20.npz"), verbose=False, gt=labels,
                                                        sweep_factory=oracle_factory, device_params=False)
    assert len(ic2) == 10 and nmi2[-1] > 0.9 and abs(kh2[-1] - kh[-1]) <= 1


def test_save_model_round_trip_multinomial(tmp_path):
    x, labels, _ = pkg.generate_mnmm_data(400, 12, 3, 30, np.random.default_rng(2))[:3]
    hyper = P.multinomial_hyper(np.ones(12))
    out = H.dp_parallel(x, hyper, 10.0, iters=12, seed=3, verbose=False, burnout=3, sweep_factory=oracle_factory,
                        save_model=True, save_path=str(tmp_path) + "/", model_save_interval=6)
    grp, mh, it, _, _ = CK.load_checkpoint(str(tmp_path / "checkpoint__12.npz"))
    assert it == 12 and isinstance(mh.distribution_hyper_params, P.multinomial_hyper)
    np.testing.assert_array_equal(grp["labels"], out[0].group.sweep.get_labels())
    for a, b in zip(grp["local_clusters"], out[0].group.local_clusters):
        np.testing.assert_array_equal(a.cluster_params.cluster_params.suff_statistics.points_sum,
                                      b.cluster_params.cluster_params.suff_statistics.points_sum)
        np.testing.assert_array_equal(a.cluster_params.cluster_params_l.distribution.α, b.cluster_params.cluster_params_l.distribution.α)


# ---------------------------------------------------------------------------------------------- GPU --------
@pytest.mark.gpu
@pytest.mark.parametrize("device_params", [True, False])
def test_advanced_mode_saves_and_resumes_on_the_gpu(tmp_path, device_params):
    import __graft_entry__ as g
    g.build()
    x, labels, f, out = _advanced_run(tmp_path, device_params, None, iters=40, interval=20)
    dp_model, iter_count, nmi, _, kh = out
    assert len(iter_count) == 40 and nmi[-1] > 0.9
    grp, mh, it, _, _ = CK.load_checkpoint(str(tmp_path / "checkpoint__20.npz"))
    assert it == 20 and len(grp["local_clusters"]) == kh[19]
    for k, c in enumerate(grp["local_clusters"]):
        assert int((grp["labels"] == k + 1).sum()) == c.points_count
    dp2, ic2, nmi2, _, kh2 = H.run_model_from_checkpoint(str(tmp_path / "checkpoint__20.npz"), verbose=False, gt=labels,
                                                        device_params=device_params)
    assert len(ic2) == 20 and nmi2[-1] > 0.9 and abs(kh2[-1] - kh[-1]) <= 1
    # the resumed run really started from the stored labels: its first NMI is already that of iteration ~20
    assert nmi2[0] > 0.8
