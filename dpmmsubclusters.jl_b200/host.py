"""Host side of the sampler: a Python mirror of the reference's MASTER functions, driving the sweep
through the C ABI (GpuSweep) exactly where the reference crosses to its workers.

Julia is not installed in this environment, so this module stands where the (unchanged) Julia host
would stand: same function names, same control flow, same defaults, citing the reference lines:
  fit / dp_parallel / run_model / calculate_posterior     src/dp-parallel-sampling.jl
  group_step and the master "!"-functions                  src/local_clusters_actions.jl
  sample_cluster_params / should_merge! / splits           src/shared_actions.jl
Only the worker calls differ: every `@spawnat ... _worker!` becomes one GpuSweep call.
"""
from __future__ import annotations

import copy
import os
import time
from dataclasses import dataclass, field

import numpy as np
import scipy.sparse as sps
from scipy.special import gammaln

from . import priors as P
from .sweep import GpuSweep, NIW, MULTINOMIAL, DIAG

F32 = np.float32


def _points(x):
    """The points as the sweep takes them: scipy.sparse matrices pass through (multinomial prior only; the sweep converts
    them to 1-based CSC once), everything else becomes a Float32 array."""
    return x if sps.issparse(x) else np.asarray(x, F32)


# ---------------------------------------------------------------- data structures (src/ds.jl) ----
@dataclass
class model_hyper_params:            # ds.jl:7-11
    distribution_hyper_params: object
    α: float
    total_dim: int


@dataclass
class cluster_parameters:            # ds.jl:13-18
    hyperparams: object
    distribution: object
    suff_statistics: object
    posterior_hyperparams: object


@dataclass
class splittable_cluster_params:     # ds.jl:20-27
    cluster_params: cluster_parameters
    cluster_params_l: cluster_parameters
    cluster_params_r: cluster_parameters
    lr_weights: np.ndarray
    splittable: bool
    logsublikelihood_hist: np.ndarray


@dataclass
class local_cluster:                 # ds.jl:43-49
    cluster_params: splittable_cluster_params
    total_dim: int
    points_count: int
    l_count: int
    r_count: int


@dataclass
class local_group:                   # ds.jl:51-58; points/labels/labels_subcluster live in the sweep
    model_hyperparams: model_hyper_params
    sweep: object
    local_clusters: list = field(default_factory=list)
    weights: np.ndarray = field(default_factory=lambda: np.zeros(0, F32))


@dataclass
class dp_parallel_sampling:          # ds.jl:76-79
    model_hyperparams: model_hyper_params
    group: local_group
    outlier_weight: float = 0.0          # the outlier component (DESIGN.md 6.1), recorded by save_model
    outlier_params: object = None


@dataclass
class Settings:
    """The module-level globals of the reference (src/global_params.jl, dp-parallel-sampling.jl:135-146)."""
    iterations: int = 100
    hard_clustering: bool = False
    initial_clusters: int = 1
    argmax_sample_stop: int = 5
    split_stop: int = 5
    burnout_period: int = 20
    max_num_of_clusters: float = np.inf
    outlier_mod: float = 0.0             # weight of the outlier component (cluster 1); 0 = no component
    outlier_hyper_params: object = None  # its prior, of the model prior's type and dimension
    use_verbose: bool = False
    ground_truth: object = None
    use_smart_splits: bool = False
    max_split_iter: int = 20             # global_params.jl:15
    # checkpoints (global_params.jl:34-40; dp-parallel-sampling.jl:395-399)
    should_save_model: bool = False
    model_save_interval: int = 1000
    save_path: str = ""
    save_file_prefix: str = "checkpoint_"
    data_path: str = ""
    data_prefix: str = ""
    global_params: object = "none"       # what save_model records as `global_params` (the parameter file's content)


# ---------------------------------------------------------------- shared_actions.jl --------------
def _neg_inf_hist(cfg):
    return np.full(cfg.burnout_period + 5, -np.inf)


def create_splittable_from_params(params, α, cfg, rng):
    """shared_actions.jl:2-9."""
    params_l = copy.deepcopy(params)
    params_l.distribution = P.sample_distribution(params.posterior_hyperparams, rng)
    params_r = copy.deepcopy(params)
    params_r.distribution = P.sample_distribution(params.posterior_hyperparams, rng)
    lr_weights = rng.dirichlet([α / 2, α / 2])
    return splittable_cluster_params(params, params_l, params_r, lr_weights, False, _neg_inf_hist(cfg))


def merge_clusters_to_splittable(cpl, cpr, α, cfg, rng):
    """shared_actions.jl:12-18."""
    suff_stats = P.aggregate_suff_stats(cpl.suff_statistics, cpr.suff_statistics)
    posterior = P.calc_posterior(cpl.hyperparams, suff_stats)
    lr_weights = rng.dirichlet([cpl.suff_statistics.N + α / 2, cpr.suff_statistics.N + α / 2])
    cp = cluster_parameters(cpl.hyperparams, cpl.distribution, suff_stats, posterior)
    return splittable_cluster_params(cp, cpl, cpr, lr_weights, False, _neg_inf_hist(cfg))


def should_merge(cpl, cpr, α, final, rng):
    """shared_actions.jl:21-38."""
    new_suff = P.aggregate_suff_stats(cpl.suff_statistics, cpr.suff_statistics)
    post = P.calc_posterior(cpl.hyperparams, new_suff)
    ll_l = P.log_marginal_likelihood(cpl.hyperparams, cpl.posterior_hyperparams, cpl.suff_statistics)
    ll_r = P.log_marginal_likelihood(cpr.hyperparams, cpr.posterior_hyperparams, cpr.suff_statistics)
    ll = P.log_marginal_likelihood(cpl.hyperparams, post, new_suff)
    Nl, Nr, N = cpl.suff_statistics.N, cpr.suff_statistics.N, new_suff.N
    log_HR = (-np.log(α) + gammaln(α) - 2 * gammaln(0.5 * α) + gammaln(N) - gammaln(N + α)
              + gammaln(Nl + 0.5 * α) - gammaln(Nl) - gammaln(Nr) + gammaln(Nr + 0.5 * α) + ll - ll_l - ll_r)
    return (log_HR > np.log(rng.random())) or (final and log_HR > np.log(0.1))


def sample_cluster_params(params, α, first, cfg, rng):
    """shared_actions.jl:41-66."""
    for cp in (params.cluster_params, params.cluster_params_l, params.cluster_params_r):
        cp.distribution = P.sample_distribution(cp.hyperparams if first else cp.posterior_hyperparams, rng)
    pc = np.array([params.cluster_params_l.suff_statistics.N, params.cluster_params_r.suff_statistics.N], np.float64) + α / 2
    params.lr_weights = rng.dirichlet(pc)
    ll_l = P.log_marginal_likelihood(params.cluster_params_l.hyperparams, params.cluster_params_l.posterior_hyperparams,
                                     params.cluster_params_l.suff_statistics)
    ll_r = P.log_marginal_likelihood(params.cluster_params_r.hyperparams, params.cluster_params_r.posterior_hyperparams,
                                     params.cluster_params_r.suff_statistics)
    b = cfg.burnout_period
    h = params.logsublikelihood_hist
    h[0:b - 1] = h[1:b].copy()
    h[b - 1] = ll_l + ll_r
    with np.errstate(invalid="ignore"):
        now = float(np.sum(h[:b] * (1 / (b - 0.1))))
    if now != -np.inf and not np.isnan(now) and now - h[b - 1] < 1e-2:
        params.splittable = True
    return params


# ---------------------------------------------------------------- local_clusters_actions.jl -------
def create_first_local_cluster(group, cfg, rng):
    """:1-20.  The worker call (split_first_cluster_worker!, :16-18) -> randomize_sublabels(all)."""
    hyper = group.model_hyperparams.distribution_hyper_params
    suff = P.empty_suff_stats(hyper)
    dist = P.sample_distribution(hyper, rng)
    cp = cluster_parameters(hyper, dist, suff, hyper)
    cpl, cpr = copy.deepcopy(cp), copy.deepcopy(cp)
    splittable = splittable_cluster_params(cp, cpl, cpr, np.array([0.5, 0.5]), False, _neg_inf_hist(cfg))
    cp.suff_statistics.N = group.sweep.n
    cluster = local_cluster(splittable, group.model_hyperparams.total_dim, group.sweep.n, 0, 0)
    group.sweep.randomize_sublabels(None)
    return cluster


def create_outlier_local_cluster(group, outlier_params, cfg, rng):
    """:42-61.  Cluster 1 of a model with the outlier component: its own prior, distributions drawn from it, lr
    weights (0.5, 0.5), no points (the initial labels start at 2)."""
    suff = P.empty_suff_stats(outlier_params)
    dist = P.sample_distribution(outlier_params, rng)
    cp = cluster_parameters(outlier_params, dist, suff, outlier_params)
    cpl, cpr = copy.deepcopy(cp), copy.deepcopy(cp)
    splittable = splittable_cluster_params(cp, cpl, cpr, np.array([0.5, 0.5]), False, _neg_inf_hist(cfg))
    return local_cluster(splittable, group.model_hyperparams.total_dim, 0, 0, 0)


def update_suff_stats_posterior(group, indices=None):
    """update_suff_stats_posterior! :206-254.  The fetch of the workers' dictionaries and their
    aggregate_suff_stats reduction (:229-248) is one dpmm_suff_stats call (all-reduce inside)."""
    if indices is None:
        indices = list(range(1, len(group.local_clusters) + 1))
    indices = [int(i) for i in indices]
    if not indices:
        return
    hyper = group.model_hyperparams.distribution_hyper_params
    counts, sum_x, sum_xx = group.sweep.suff_stats(indices)
    for a, v in enumerate(indices):
        cluster = group.local_clusters[v - 1]
        sp = cluster.cluster_params
        for s, cp in enumerate((sp.cluster_params, sp.cluster_params_l, sp.cluster_params_r)):
            cp.suff_statistics = P.make_suff_stats(hyper, counts[a, s], sum_x[a, s], None if sum_xx is None else sum_xx[a, s])
        cluster.points_count = int(counts[a, 0])                                   # :249
        for cp in (sp.cluster_params, sp.cluster_params_l, sp.cluster_params_r):   # update_splittable_cluster_params! :137-147
            cp.posterior_hyperparams = P.calc_posterior(cp.hyperparams, cp.suff_statistics)


def sample_clusters(group, first, cfg, rng):
    """sample_clusters! :417-437."""
    α = group.model_hyperparams.α
    points_count = []
    for cluster in group.local_clusters:
        cluster.cluster_params = sample_cluster_params(cluster.cluster_params, α, first, cfg, rng)
        cluster.points_count = int(cluster.cluster_params.cluster_params.suff_statistics.N)
        points_count.append(cluster.points_count)
    points_count.append(α)
    om = cfg.outlier_mod
    if om > 0:                                                      # cluster 1 keeps its fixed weight
        points_count = points_count[1:]
    pc = np.maximum(np.asarray(points_count, np.float64), 1e-300)   # Dirichlet needs positive parameters
    w = rng.dirichlet(pc)[:-1] * (1 - om)
    group.weights = (np.concatenate([[om], w]) if om > 0 else w).astype(F32)


def broadcast_cluster_params(group):
    """broadcast_cluster_params :518-549 with create_thin_cluster_params :439-444: pack the thin
    parameters (3 distributions + lr_weights per cluster) and the weights into one upload."""
    cl = group.local_clusters
    K = len(cl)
    lr = np.array([c.cluster_params.lr_weights for c in cl], F32).reshape(K, 2)
    trip = [(c.cluster_params.cluster_params.distribution, c.cluster_params.cluster_params_l.distribution,
             c.cluster_params.cluster_params_r.distribution) for c in cl]
    w = np.asarray(group.weights, F32)
    if isinstance(group.model_hyperparams.distribution_hyper_params, P.niw_hyperparams):
        mu = np.array([[d.μ for d in t] for t in trip], F32)
        inv = np.array([[d.invΣ for d in t] for t in trip], F32)
        ld = np.array([[d.logdetΣ for d in t] for t in trip], F32)
        group.sweep.set_params_niw(mu, inv, ld, w, lr)
    elif isinstance(group.model_hyperparams.distribution_hyper_params, P.diag_niw_hyperparams):
        mu = np.array([[d.μ for d in t] for t in trip], F32)
        var = np.array([[d.σ2 for d in t] for t in trip], F32)
        ld = np.array([[d.logdetΣ for d in t] for t in trip], F32)
        group.sweep.set_params_diag(mu, var, ld, w, lr)
    else:
        lp = np.array([[d.α for d in t] for t in trip], F32)
        group.sweep.set_params_multinomial(lp, w, lr)


def reset_bad_clusters(group, cfg):
    """reset_bad_clusters! :501-516."""
    bad = []
    for i, c in enumerate(group.local_clusters, start=1):
        if c.cluster_params.cluster_params_l.suff_statistics.N == 0 or c.cluster_params.cluster_params_r.suff_statistics.N == 0:
            bad.append(i)
            c.cluster_params.logsublikelihood_hist = _neg_inf_hist(cfg)
            c.cluster_params.splittable = False
    if bad:
        group.sweep.randomize_sublabels(bad)           # reset_bad_clusters_worker! :481-488
        update_suff_stats_posterior(group, bad)
    return bad


def should_split_local(cluster_params, α, final, rng):
    """should_split_local! :318-343."""
    cpl, cpr, cp = cluster_params.cluster_params_l, cluster_params.cluster_params_r, cluster_params.cluster_params
    if final or cpl.suff_statistics.N == 0 or cpr.suff_statistics.N == 0:
        return False
    post = P.calc_posterior(cp.hyperparams, cp.suff_statistics)
    lpost = P.calc_posterior(cp.hyperparams, cpl.suff_statistics)
    rpost = P.calc_posterior(cp.hyperparams, cpr.suff_statistics)
    ll_l = P.log_marginal_likelihood(cpl.hyperparams, lpost, cpl.suff_statistics)
    ll_r = P.log_marginal_likelihood(cpr.hyperparams, rpost, cpr.suff_statistics)
    ll = P.log_marginal_likelihood(cp.hyperparams, post, cp.suff_statistics)
    log_HR = (np.log(α) + gammaln(cpl.suff_statistics.N) + ll_l + gammaln(cpr.suff_statistics.N) + ll_r
              - (gammaln(cp.suff_statistics.N) + ll))
    return log_HR > np.log(rng.random())


def check_and_split(group, final, cfg, rng):
    """check_and_split! :345-382 (+ split_cluster_local! :280-291)."""
    α = group.model_hyperparams.α
    K = len(group.local_clusters)
    split = []
    for index, cluster in enumerate(group.local_clusters, start=1):
        if cfg.outlier_mod > 0 and index == 1:
            continue
        sp = cluster.cluster_params
        if sp.splittable and sp.cluster_params.suff_statistics.N > 1 and should_split_local(sp, α, final, rng):
            split.append(index)
    indices, new_indices = [], []
    new_index = K + 1
    for i in split:
        cluster = group.local_clusters[i - 1]
        l_split = copy.deepcopy(cluster)
        l_split.cluster_params = create_splittable_from_params(cluster.cluster_params.cluster_params_r, α, cfg, rng)
        cluster.cluster_params = create_splittable_from_params(cluster.cluster_params.cluster_params_l, α, cfg, rng)
        l_split.points_count = int(l_split.cluster_params.cluster_params.suff_statistics.N)
        cluster.points_count = int(cluster.cluster_params.cluster_params.suff_statistics.N)
        group.local_clusters.append(l_split)
        indices.append(i)
        new_indices.append(new_index)
        new_index += 1
    if indices:
        group.sweep.apply_split(indices, new_indices)      # split_cluster_local_worker! :265-278
        if cfg.use_smart_splits:                           # :374-378
            for i in indices + new_indices:
                smart_cluster_init(group, i, cfg)
    return indices + new_indices


def check_and_merge(group, final, cfg, rng):
    """check_and_merge! :385-413 (+ merge_clusters! :308-315)."""
    α = group.model_hyperparams.α
    cl = group.local_clusters
    indices, new_indices = [], []
    for i in range(len(cl)):
        if cfg.outlier_mod > 0 and i == 0:
            continue
        for j in range(i + 1, len(cl)):
            ci, cj = cl[i].cluster_params, cl[j].cluster_params
            if (ci.splittable and cj.splittable and ci.cluster_params.suff_statistics.N > 0
                    and cj.cluster_params.suff_statistics.N > 0
                    and should_merge(ci.cluster_params, cj.cluster_params, α, final, rng)):
                cl[i].cluster_params = merge_clusters_to_splittable(ci.cluster_params, cj.cluster_params, α, cfg, rng)
                cl[i].points_count += cl[j].points_count
                cl[j].points_count = 0
                cl[j].cluster_params.cluster_params.suff_statistics.N = 0
                cl[j].cluster_params.splittable = False
                indices.append(i + 1)
                new_indices.append(j + 1)
    if indices:
        group.sweep.apply_merge(indices, new_indices)      # merge_clusters_worker! :293-304
    return indices


def remove_empty_clusters(group, cfg):
    """remove_empty_clusters! :457-471.  The sweep drops exactly the clusters the host drops: a kept empty cluster (the
    outlier component, or cluster 2 while K = 2) is passed with a count of 1."""
    new_vec, pts_count = [], []
    n = len(group.local_clusters)
    for index, cluster in enumerate(group.local_clusters, start=1):
        keep = (cluster.points_count > 0 or (cfg.outlier_mod > 0 and index == 1)
                or (cfg.outlier_mod > 0 and index == 2 and n == 2))
        pts_count.append(max(int(cluster.points_count), 1) if keep else 0)
        if keep:
            new_vec.append(cluster)
    group.sweep.remove_empty(pts_count)                    # remove_empty_clusters_worker! :446-455
    group.local_clusters = new_vec


def smart_split_direction(N, sum_x, S):
    """The master-side linear algebra of smart_cluster_init! (:557-569): M = S/N - mu mu', eigen(M), and -- as the
    reference writes it -- ROW `mxindx` of the eigenvector matrix (`vecs[mxindx,:]`), not the eigenvector itself."""
    mu = np.asarray(sum_x, np.float64) / N
    M = np.asarray(S, np.float64) / N - np.outer(mu, mu)
    vals, vecs = np.linalg.eigh(M)
    return vecs[int(np.argmax(vals)), :].copy(), mu


def smart_kmeans(sweep, cluster_num, v1, mu, max_split_iter):
    """The worker-driving part of smart_cluster_init! (:570-623): projection + percentiles, the distributed 1-D
    2-means loop, and the sub-label write-back.  Shared by the host and the device parameter paths."""
    min_mean, max_mean, count = sweep.smart_project(cluster_num, v1, mu)
    if count == 0 or np.isnan(min_mean):                       # `if length(min_pts) == 0 return`
        return
    it, converged = 0, False
    while it < max_split_iter and not converged:
        s1, c1, s2, c2 = sweep.smart_kmeans_iter(min_mean, max_mean)
        with np.errstate(divide="ignore", invalid="ignore"):
            new_min, new_max = np.float64(s1) / np.float64(c1), np.float64(s2) / np.float64(c2)
        if new_min == min_mean and new_max == max_mean:
            converged = True
        else:
            min_mean, max_mean = float(new_min), float(new_max)
        it += 1
    sweep.smart_set_sublabels(cluster_num)


def smart_cluster_init(group, cluster_num, cfg):
    """smart_cluster_init! :555-623."""
    ss = group.local_clusters[cluster_num - 1].cluster_params.cluster_params.suff_statistics
    if ss.N == 0:
        return
    v1, mu = smart_split_direction(ss.N, ss.points_sum, ss.S)
    smart_kmeans(group.sweep, cluster_num, v1, mu, cfg.max_split_iter)


def group_step(group, no_more_splits, final, first, cfg, rng):
    """group_step :658-673."""
    sample_clusters(group, False, cfg, rng)
    broadcast_cluster_params(group)
    group.sweep.sample_labels(True if cfg.hard_clustering else final)   # sample_labels! :98-109
    group.sweep.sample_sublabels()                                       # sample_sub_clusters! :64-68
    update_suff_stats_posterior(group)
    reset_bad_clusters(group, cfg)
    if not no_more_splits:
        indices = check_and_split(group, final, cfg, rng)
        update_suff_stats_posterior(group, indices)
        check_and_merge(group, final, cfg, rng)
    remove_empty_clusters(group, cfg)


# ---------------------------------------------------------------- dp-parallel-sampling.jl ---------
def normalized_mutual_info(a, b):
    """Clustering.mutualinfo(a, b; normed=true): 2 I(a;b) / (H(a) + H(b))."""
    a = np.asarray(a).astype(np.int64)
    b = np.asarray(b).astype(np.int64)
    _, ai = np.unique(a, return_inverse=True)
    _, bi = np.unique(b, return_inverse=True)
    n = a.size
    C = np.zeros((ai.max() + 1, bi.max() + 1))
    np.add.at(C, (ai, bi), 1)
    pa, pb, pab = C.sum(1) / n, C.sum(0) / n, C / n
    nz = pab > 0
    I = (pab[nz] * np.log(pab[nz] / (pa[:, None] * pb[None, :])[nz])).sum()
    H = -(pa[pa > 0] * np.log(pa[pa > 0])).sum() - (pb[pb > 0] * np.log(pb[pb > 0])).sum()
    return float(2 * I / H) if H > 0 else 1.0


def calculate_posterior(model):
    """calculate_posterior :458-470."""
    α = model.model_hyperparams.α
    lp = gammaln(α) - gammaln(model.group.sweep.n_total + α)
    for c in model.group.local_clusters:
        cp = c.cluster_params.cluster_params
        if cp.suff_statistics.N == 0:
            continue
        lp += P.log_marginal_likelihood(cp.hyperparams, cp.posterior_hyperparams, cp.suff_statistics)
        lp += np.log(α) + gammaln(cp.suff_statistics.N)
    return float(lp)


def init_model_from_data(all_data, hyper_params, α, cfg, seed, sweep_factory, shard):
    """init_model_from_data :36-53: `distribute(all_data)` + random labels become dpmm_create +
    dpmm_init_labels.  `shard` = (global_offset, n_total) when the points are one shard of many."""
    all_data = _points(all_data)
    kind = (NIW if isinstance(hyper_params, P.niw_hyperparams)
            else DIAG if isinstance(hyper_params, P.diag_niw_hyperparams) else MULTINOMIAL)
    goff, n_total = shard if shard is not None else (0, all_data.shape[1])
    sweep_seed = int(seed) if seed is not None else int(np.random.default_rng().integers(2 ** 62))
    sweep = sweep_factory(all_data, kind, sweep_seed, goff)
    sweep.n_total = n_total
    mh = model_hyper_params(hyper_params, float(F32(α)), all_data.shape[1])
    sweep.init_labels(cfg.initial_clusters, cfg.outlier_mod > 0)
    return dp_parallel_sampling(mh, local_group(mh, sweep), cfg.outlier_mod, cfg.outlier_hyper_params)


def init_first_clusters(dp_model, cfg, rng):
    """init_first_clusters! :62-78."""
    g = dp_model.group
    om = cfg.outlier_mod
    if om > 0:                                             # :66-68: the outlier component is cluster 1
        g.local_clusters.append(create_outlier_local_cluster(g, cfg.outlier_hyper_params, cfg, rng))
    for _ in range(cfg.initial_clusters):
        g.local_clusters.append(create_first_local_cluster(g, cfg, rng))
    update_suff_stats_posterior(g)
    if cfg.use_smart_splits:                               # :70-75 (never the outlier component)
        for i in range(2 if om > 0 else 1, len(g.local_clusters) + 1):
            smart_cluster_init(g, i, cfg)
        update_suff_stats_posterior(g)
    sample_clusters(g, False, cfg, rng)
    K = len(g.local_clusters)
    if om > 0:
        g.weights = np.array([om] + [(1 - om) / (K - 1)] * (K - 1), F32)
    else:
        g.weights = np.full(K, 1.0 / K, F32) if K > 1 else np.ones(1, F32)
    broadcast_cluster_params(g)


def run_model(dp_model, first_iter, cfg, rng):
    """run_model :336-404."""
    iter_count, nmi_hist, ll_hist, k_hist = [], [], [], []
    g = dp_model.group
    start_time = time.time()
    for i in range(first_iter, cfg.iterations + 1):
        final = i >= cfg.iterations - cfg.argmax_sample_stop
        no_more_splits = (i >= cfg.iterations - cfg.split_stop) or (len(g.local_clusters) >= cfg.max_num_of_clusters)
        t0 = time.perf_counter()
        group_step(g, no_more_splits, final, i == 1, cfg, rng)
        iter_count.append(time.perf_counter() - t0)
        k_hist.append(len(g.local_clusters))
        if cfg.ground_truth is not None:
            nmi_hist.append(normalized_mutual_info(cfg.ground_truth, g.sweep.get_labels()))
        else:
            nmi_hist.append("no gt")
        if cfg.use_verbose:
            ll_hist.append(calculate_posterior(dp_model))
            print(f"Iteration: {i} || Clusters count: {k_hist[-1]} || Log posterior: {ll_hist[-1]} || "
                  f"NMI score: {nmi_hist[-1]} || Iter Time:{iter_count[-1]} || Total time:{sum(iter_count)}")
        else:
            ll_hist.append(1)
        if i % cfg.model_save_interval == 0 and cfg.should_save_model:      # :395-399
            from .checkpoint import save_model
            save_model(dp_model, cfg.save_path, cfg.save_file_prefix, i, time.time() - start_time, cfg.global_params)
    return dp_model, iter_count, nmi_hist, ll_hist, k_hist


def _gpu_factory(device=0):
    def make(x, kind, seed, goff):
        return GpuSweep(x, kind, seed=seed, global_offset=goff, device=device)
    return make


def _clusters_from_device(group, st, cfg):
    """Rebuild the reference's host objects (local_cluster list, weights) from the final device state, so that
    the tuple fit() returns, predict() and calculate_posterior() see what the host path would have left."""
    hyper = group.model_hyperparams.distribution_hyper_params
    om = cfg.outlier_mod
    sw = group.sweep
    K = st.K
    counts, sum_x, sum_xx = sw.suff_stats(list(range(1, K + 1)))
    params = getattr(st, "params", None)
    if params is not None and params[0].shape[0] != K:
        params = None                                     # K changed after the parameters were fetched (mid-run checkpoint)
    niw = isinstance(hyper, P.niw_hyperparams)
    diag = isinstance(hyper, P.diag_niw_hyperparams)
    if params is not None:
        if niw:
            mu, lfac, logdet, w, lr = params
        elif diag:
            mu, var, logdet, w, lr = params
        else:
            log_p, w, lr = params
    else:
        # no sampled parameters at hand: the posterior's centre stands in.  group_step re-draws every
        # distribution and weight before anything reads them (sample_clusters!, :659), so these never reach a sweep.
        tot = max(float(counts[:, 0].sum()), 1.0)
        w = counts[:, 0] / tot
        if om > 0:
            w = np.concatenate([[om], (1 - om) * counts[1:, 0] / max(float(counts[1:, 0].sum()), 1.0)])
        lr = (counts[:, 1:3] + 0.5) / (counts[:, 1:3] + 0.5).sum(axis=1, keepdims=True)
    group.local_clusters = []
    for k in range(K):
        h = cfg.outlier_hyper_params if (om > 0 and k == 0) else hyper     # cluster 1: the outlier component's prior
        cps = []
        for s_ in range(3):
            ss = P.make_suff_stats(hyper, counts[k, s_], sum_x[k, s_], None if sum_xx is None else sum_xx[k, s_])
            post = P.calc_posterior(h, ss)
            if diag:
                if params is not None:
                    dist = P.diag_gaussian(mu[k, s_].copy(), var[k, s_].copy(), float(logdet[k, s_]))
                else:
                    dist = P.diag_gaussian(post.m.astype(F32), post.ψ.astype(F32), float(F32(np.log(post.ψ).sum())))
            elif not niw:
                if params is not None:
                    dist = P.multinomial_dist(log_p[k, s_].copy())
                else:
                    a = post.α.astype(np.float64)
                    dist = P.multinomial_dist(np.log(a / a.sum()).astype(F32))
            elif params is not None:
                L = np.tril(lfac[k, s_])
                inv = L @ L.T
                with np.errstate(all="ignore"):
                    Sig = np.linalg.inv(inv) if np.isfinite(inv).all() else np.full_like(inv, np.nan)
                dist = P.mv_gaussian(mu[k, s_].astype(F32), Sig.astype(F32), inv.astype(F32), float(logdet[k, s_]), L.T.copy())
            else:
                inv = np.linalg.inv(post.ψ)
                dist = P.mv_gaussian(post.m.astype(F32), post.ψ.astype(F32), inv.astype(F32),
                                     float(np.linalg.slogdet(post.ψ)[1]), np.linalg.cholesky(inv).T)
            cps.append(cluster_parameters(h, dist, ss, post))
        sp = splittable_cluster_params(cps[0], cps[1], cps[2], lr[k].astype(np.float64), bool(st.splittable[k]),
                                       st.hist[k].copy())
        group.local_clusters.append(local_cluster(sp, group.model_hyperparams.total_dim, int(counts[k, 0]),
                                                  int(counts[k, 1]), int(counts[k, 2])))
    group.weights = np.asarray(w, F32)


def dp_parallel(all_data, local_hyper_params=None, α_param=None, iters=100, init_clusters=1, seed=None, verbose=True,
                save_model=False, burnout=15, gt=None, max_clusters=np.inf, outlier_weight=0, outlier_params=None,
                smart_splits=False, *, sweep_factory=None, shard=None, comm=None, device=0, device_params=None,
                save_path=None, save_file_prefix="checkpoint_", model_save_interval=1000):
    """dp_parallel :121-157.  `sweep_factory`, `shard`, `comm`, `device`, `device_params` have no reference
    counterpart: they select the device / inject a test double / attach the multi-GPU communicator / choose
    where the parameter step runs (default: on the device for the NIW prior, SURVEY 8f-1, and on the host for the
    multinomial and diagonal Gaussian priors, which take the device with device_params=True; False = the Python mirror
    of the reference's master functions below)."""
    if isinstance(all_data, (str, os.PathLike)):
        return dp_parallel_params_file(str(all_data), verbose=verbose, gt=gt, sweep_factory=sweep_factory, shard=shard,
                                       comm=comm, device=device, device_params=device_params)
    outlier_weight, outlier_params = _outlier_settings(local_hyper_params, outlier_weight, outlier_params)
    if save_model and save_path is None:
        raise ValueError("save_model=True needs save_path (global_params.jl:37 in the reference)")
    if sps.issparse(all_data) and isinstance(local_hyper_params, (P.niw_hyperparams, P.diag_niw_hyperparams)):
        raise ValueError("sparse points are supported for the multinomial prior only")
    if smart_splits and isinstance(local_hyper_params, P.diag_niw_hyperparams):
        raise ValueError("smart splits need the full scatter matrix: not available with the diagonal prior")
    if smart_splits and not isinstance(local_hyper_params, P.niw_hyperparams):
        raise ValueError("smart splits are Gaussian only (dp-parallel-sampling.jl:111)")
    if (comm is not None or shard is not None) and seed is None:
        # every rank must draw the same parameters and take the same split / merge decisions
        raise ValueError("multi-GPU runs (comm / shard) need an explicit seed shared by all ranks")
    cfg = Settings(iterations=int(iters), initial_clusters=int(init_clusters), burnout_period=int(burnout),
                   max_num_of_clusters=max_clusters, use_verbose=bool(verbose), ground_truth=gt,
                   use_smart_splits=bool(smart_splits), should_save_model=bool(save_model), save_path=save_path or "",
                   save_file_prefix=save_file_prefix, model_save_interval=int(model_save_interval),
                   outlier_mod=outlier_weight, outlier_hyper_params=outlier_params)
    return _run_from_settings(all_data, local_hyper_params, α_param, cfg, seed, sweep_factory, shard, comm, device,
                              device_params)


def _outlier_settings(hyper, weight, params):
    """(weight, prior) of the outlier component, validated; (0.0, None) when it is off (weight 0)."""
    weight = float(weight)
    if not 0.0 <= weight < 1.0:
        raise ValueError(f"outlier_weight must lie in [0, 1), got {weight}")
    if weight == 0.0:
        return 0.0, None
    if params is None:
        raise ValueError("outlier_weight > 0 needs outlier_params")
    if type(params) is not type(hyper):
        raise ValueError(f"outlier_params must be a {type(hyper).__name__}, as the model's prior, "
                         f"not a {type(params).__name__}")
    shape = lambda h: np.shape(h.α) if isinstance(h, P.multinomial_hyper) else (np.shape(h.m), np.shape(h.ψ))
    if shape(params) != shape(hyper):
        raise ValueError("outlier_params must have the dimension of the model's prior")
    return weight, params


def _run_from_settings(all_data, local_hyper_params, α_param, cfg, seed, sweep_factory, shard, comm, device, device_params,
                       restored=None):
    """init_model + init_first_clusters! + run_model for fresh runs; create_model_from_saved_data + run_model(iter + 1)
    when `restored` = (pts_less_group dict, iter) of a checkpoint."""
    if isinstance(local_hyper_params, P.diag_niw_hyperparams):
        if cfg.use_smart_splits:
            raise ValueError("smart splits need the full scatter matrix: not available with the diagonal prior")
    if restored is not None and seed is not None:
        seed = int(seed) + 1000003 * int(restored[1])     # a resumed run must not replay the random streams of iteration 1
    rng = np.random.default_rng(seed)
    dp_model = init_model_from_data(all_data, local_hyper_params, α_param, cfg, seed,
                                    sweep_factory or _gpu_factory(device), shard)
    sw = dp_model.group.sweep
    if comm is not None:
        sw.comm_init(*comm)
    niw = isinstance(local_hyper_params, P.niw_hyperparams)
    if device_params and isinstance(local_hyper_params, P.diag_niw_hyperparams) and not hasattr(sw, "sample_params"):
        raise ValueError("device_params: this sweep has no device parameter step; off the GPU, device_params is "
                         "accepted for the NIW and multinomial priors only, which fall back to the host loop")
    if device_params is None:                              # (multinomial, diagonal: the host loop unless asked for)
        device_params = niw and os.environ.get("DPMM_DEVICE_PARAMS", "1") != "0"
    first_iter = 1
    if restored is not None:                               # create_model_from_saved_data, ds.jl:89-92; :437-439
        grp, it = restored
        sw.set_labels(grp["labels"])
        sw.set_sublabels(grp["labels_subcluster"])
        dp_model.group.local_clusters = grp["local_clusters"]
        dp_model.group.weights = grp["weights"]
        first_iter = it + 1
    if device_params and hasattr(sw, "sample_params"):
        from . import host_device as HD
        st, iter_count, nmi, ll, kh = HD.run_model_device(dp_model, cfg, rng, normalized_mutual_info, first_iter=first_iter,
                                                          resume=restored is not None)
        _clusters_from_device(dp_model.group, st, cfg)
        return dp_model, iter_count, nmi, ll, kh
    if restored is None:
        init_first_clusters(dp_model, cfg, rng)
    return run_model(dp_model, first_iter, cfg, rng)


def _settings_from_params(gp, verbose, gt):
    """The component is on when the file sets outlier_mod > 0 and outlier_hyper_params (global_params.jl defaults to
    outlier_mod = 0.05 without hyper-parameters: off)."""
    om, ohp = 0.0, None
    if gp["outlier_hyper_params"] is not None and gp["outlier_mod"] > 0 and gp["hyper_params"] is not None:
        om, ohp = _outlier_settings(gp["hyper_params"], gp["outlier_mod"], gp["outlier_hyper_params"])
    return Settings(iterations=int(gp["iterations"]), hard_clustering=bool(gp["hard_clustering"]),
                    initial_clusters=int(gp["initial_clusters"]), argmax_sample_stop=int(gp["argmax_sample_stop"]),
                    split_stop=int(gp["split_stop"]), burnout_period=int(gp["burnout_period"]),
                    max_num_of_clusters=gp["max_clusters"], use_verbose=bool(verbose), ground_truth=gt,
                    use_smart_splits=bool(gp["smart_splits"]), max_split_iter=int(gp["max_split_iter"]),
                    should_save_model=bool(gp["enable_saving"]), model_save_interval=int(gp["model_save_interval"]),
                    save_path=gp["save_path"], save_file_prefix=gp["save_file_prefix"], data_path=gp["data_path"],
                    data_prefix=gp["data_prefix"], outlier_mod=om, outlier_hyper_params=ohp)


def dp_parallel_params_file(model_params, verbose=True, gt=None, **kw):
    """dp_parallel(model_params::String; verbose, gt) :317-334 -- the advanced mode: every setting, the prior and the
    data location come from a parameter file in the style of src/global_params.jl."""
    from .checkpoint import read_params, load_data
    gp = read_params(model_params)
    cfg = _settings_from_params(gp, verbose, gt)
    cfg.global_params = model_params
    if gp["hyper_params"] is None:
        raise ValueError("the parameter file must define hyper_params")
    data = _points(load_data(cfg.data_path, prefix=cfg.data_prefix))              # init_model :24-25
    return _run_from_settings(data, gp["hyper_params"], gp["α"], cfg, gp["random_seed"], kw.get("sweep_factory"),
                              kw.get("shard"), kw.get("comm"), kw.get("device", 0), kw.get("device_params"))


def run_model_from_checkpoint(filename, verbose=True, gt=None, data=None, **kw):
    """run_model_from_checkpoint :428-449: reload the group, re-read the parameter file recorded in the checkpoint and
    the data it points to (`data=` overrides), restore labels / sub-labels on the device, and continue at iter + 1."""
    from .checkpoint import load_checkpoint, read_params, load_data
    grp, mh, it, total_time, gparams = load_checkpoint(filename)
    params_file = gparams.get("model_params") if isinstance(gparams, dict) else None
    if params_file and os.path.exists(params_file):
        gp = read_params(params_file)                       # `include(global_params)`, :433
        cfg = _settings_from_params(gp, verbose, gt)
        cfg.global_params = params_file
        seed = gp["random_seed"]
    else:
        cfg = Settings(use_verbose=bool(verbose), ground_truth=gt)
        for k, v in (gparams or {}).items():
            if hasattr(cfg, k) and v is not None:
                setattr(cfg, k, v)
        cfg.global_params = gparams
        seed = (gparams or {}).get("random_seed")
    # the component is part of the saved model: cluster 1 of the restored list is it, or there is none
    cfg.outlier_mod, cfg.outlier_hyper_params = grp["outlier_weight"], grp["outlier_params"]
    if data is None:
        data = load_data(cfg.data_path, prefix=cfg.data_prefix)                   # :435
    data = _points(data)
    return _run_from_settings(data, mh.distribution_hyper_params, mh.α, cfg, seed, kw.get("sweep_factory"), kw.get("shard"),
                              kw.get("comm"), kw.get("device", 0), kw.get("device_params"), restored=(grp, it))


def fit(all_data, *args, iters=100, init_clusters=1, seed=None, verbose=False, save_model=False, burnout=20,
        gt=None, max_clusters=np.inf, outlier_weight=0, outlier_params=None, smart_splits=False, **kw):
    """fit(all_data, [local_hyper_params,] α_param; ...) :215-293.  Returns the reference's tuple:
    (labels, clusters, weights, iter_count, nmi_score_history, likelihood_history, cluster_count_history,
     sub_labels, dp_model)."""
    all_data = _points(all_data)
    if len(args) == 1:
        if sps.issparse(all_data):
            raise ValueError("sparse points need the multinomial prior: pass multinomial_hyper(...) and α")
        D = all_data.shape[0]
        hyper = P.niw_hyperparams(1.0, np.zeros(D), D + 3, np.eye(D))        # :272-274
        α = args[0]
    else:
        hyper, α = args
    dp_model, iter_count, nmi, ll, kh = dp_parallel(all_data, hyper, α, iters, init_clusters, seed, verbose,
                                                    save_model, burnout, gt, max_clusters, outlier_weight,
                                                    outlier_params, smart_splits, **kw)
    g = dp_model.group
    return (g.sweep.get_labels(), [c.cluster_params.cluster_params.distribution for c in g.local_clusters],
            g.weights, iter_count, nmi, ll, kh, g.sweep.get_sublabels(), dp_model)


def predict(dp_model, data, device=0, on_device=None):
    """predict / predict_points :23-40, :532-537: posterior-predictive hard labels + probabilities.
    NIW models run on the GPU by default (dpmm_predict_niw: Student-t densities, argmax and softmax per point; the
    host prepares the K factors); multinomial models do with on_device=True (dpmm_predict_multinomial: the host
    prepares log(alpha'/sum alpha') in Float64).  on_device=False, or a multinomial model by default, takes the NumPy
    formulas below.  Sparse data (scipy.sparse, D x N) runs on a sparse context on the device and as x' logp in NumPy.
    Diagonal Gaussian models always take the NumPy formula (a product of per-feature Student-t densities)."""
    data = _points(data)
    cl = dp_model.group.local_clusters
    posts = [c.cluster_params.cluster_params.posterior_hyperparams for c in cl]
    if posts and isinstance(posts[0], P.diag_niw_hyperparams):
        if on_device:
            raise ValueError("predict on the device runs the NIW and multinomial priors only")
        on_device = False
    w = np.asarray(dp_model.group.weights, F32)
    mnm = bool(posts) and isinstance(posts[0], P.multinomial_hyper)
    if on_device is None:
        on_device = not mnm and os.environ.get("DPMM_DEVICE_PREDICT", "1") != "0"
    if on_device and mnm and isinstance(dp_model.group.sweep, GpuSweep):
        logp = np.stack([np.log(a / a.sum()) for a in (p.α.astype(np.float64) for p in posts)])   # posterior_predictive
        with np.errstate(divide="ignore"):
            lw = np.log(w)
        g = GpuSweep(data, MULTINOMIAL, device=device)
        try:
            return g.predict_multinomial(logp, lw)
        finally:
            g.close()
    if on_device and posts and isinstance(posts[0], P.niw_hyperparams) and isinstance(dp_model.group.sweep, GpuSweep):
        D, K = data.shape[0], len(posts)
        u = np.zeros((K, D, D)); mu = np.zeros((K, D)); tc = np.zeros(K); dfs = np.zeros(K)
        with np.errstate(divide="ignore"):
            lw = np.log(w.astype(np.float64))
        for k, p in enumerate(posts):                    # niw.jl:68-76
            df = p.ν - D + 1
            Sig = ((p.κ + 1) / (p.κ * df)) * p.ν * p.ψ
            u[k] = np.linalg.cholesky(np.linalg.inv(Sig)).T          # Sig^-1 = U'U
            mu[k] = p.m
            dfs[k] = df
            tc[k] = (gammaln((df + D) / 2) - gammaln(df / 2) - 0.5 * D * np.log(df * np.pi)
                     - 0.5 * np.linalg.slogdet(Sig)[1] + lw[k])
        g = GpuSweep(data, NIW, device=device)
        try:
            return g.predict_niw(u, mu, tc, dfs)
        finally:
            g.close()
    parr = np.zeros((data.shape[1], len(cl)), F32)
    for k, c in enumerate(cl):
        parr[:, k] = P.posterior_predictive(data, c.cluster_params.cluster_params.posterior_hyperparams)
    with np.errstate(divide="ignore"):
        parr += np.log(w)[None, :]
    lbls = np.argmax(parr, axis=1) + 1
    parr = np.where(np.isnan(parr), -np.inf, parr)
    parr = np.exp(parr - parr.max(axis=1, keepdims=True))
    return lbls, parr / parr.sum(axis=1, keepdims=True)


def get_labels_histogram(labels):
    """utils.jl:39-48."""
    v, c = np.unique(np.asarray(labels), return_counts=True)
    return list(zip(v.tolist(), c.tolist()))
