"""Host loop for the device-side parameter step (NIW, multinomial and diagonal Gaussian priors; SURVEY.md 8f-1).

What stays here is what north_star leaves to the host once the K x D^2 (NIW) or K x D (multinomial, diagonal) work
has moved: cluster
bookkeeping and the Hastings accept / reject decisions on scalars.  Per iteration the host reads one
small block back from the device -- 3K counts, 3K log marginal likelihoods and the K x K table of merged
log marginal likelihoods (GpuSweep.posterior_step) -- and issues the relabel operations.  Written from the
formulas of SURVEY.md appendix B on arrays over clusters; the reference lines each step answers to:
  group_step                 src/local_clusters_actions.jl:658-673
  sample_cluster_params      src/shared_actions.jl:41-66   (history window / splittable rule, :51-63)
  reset_bad_clusters!        src/local_clusters_actions.jl:501-516
  should_split_local!        :318-343 ; check_and_split! :345-382
  should_merge! / check_and_merge!   src/shared_actions.jl:21-38 ; :385-413
  remove_empty_clusters!     :457-471
  run_model                  src/dp-parallel-sampling.jl:336-404
"""
from __future__ import annotations

import time

import numpy as np
from scipy.special import gammaln

from . import priors as P
from .sweep import DIAG, NIW


class DeviceState:
    """Per-cluster scalars the Hastings moves need (arrays over clusters, grown / compacted with K)."""

    def __init__(self, K, window):
        self.K = K
        self.window = window
        self.splittable = np.zeros(K, bool)
        self.hist = np.full((K, window), -np.inf)
        self.N = np.zeros((K, 3), np.int64)
        self.logml = np.zeros((K, 3), np.float64)

    def grow(self, extra):
        self.K += extra
        self.splittable = np.concatenate([self.splittable, np.zeros(extra, bool)])
        self.hist = np.concatenate([self.hist, np.full((extra, self.window), -np.inf)])
        self.N = np.concatenate([self.N, np.zeros((extra, 3), np.int64)])
        self.logml = np.concatenate([self.logml, np.zeros((extra, 3))])

    def keep(self, mask):
        self.K = int(mask.sum())
        self.splittable, self.hist, self.N, self.logml = (self.splittable[mask], self.hist[mask], self.N[mask],
                                                          self.logml[mask])


def _update(st, idx, counts, logml):
    st.N[idx] = counts
    st.logml[idx] = logml


def history_step(st, cfg):
    """The window update of sample_cluster_params (shared_actions.jl:51-63) for every cluster at once."""
    b = cfg.burnout_period
    h = st.hist
    h[:, 0:b - 1] = h[:, 1:b].copy()
    h[:, b - 1] = st.logml[:, 1] + st.logml[:, 2]
    with np.errstate(invalid="ignore"):
        now = (h[:, :b] * (1 / (b - 0.1))).sum(axis=1)
        ok = (now != -np.inf) & ~np.isnan(now) & (now - h[:, b - 1] < 1e-2)
    st.splittable |= ok


def group_step_device(sw, st, α, no_more_splits, final, cfg, rng, keep_params=False):
    """One Gibbs iteration; returns nothing, mutates `st` and the device state."""
    # sample_clusters! + broadcast (device)
    history_step(st, cfg)
    sw.sample_params(st.K)
    if keep_params:                                        # the distributions fit() returns (last iteration only)
        get = {NIW: sw.get_params_niw, DIAG: sw.get_params_diag}.get(sw.prior_kind, sw.get_params_multinomial)
        st.params = get(st.K)
    sw.sample_labels(True if cfg.hard_clustering else final)
    sw.sample_sublabels()
    # update_suff_stats_posterior! for every cluster; the merge table rides along when merges are possible
    want_merge = (not no_more_splits) and st.K > 1 and st.splittable.sum() > 1
    counts, logml, merge = sw.posterior_step(None, splittable=st.splittable if want_merge else None)
    st.N[:], st.logml[:] = counts[:st.K], logml[:st.K]
    # reset_bad_clusters!
    bad = np.nonzero((st.N[:, 1] == 0) | (st.N[:, 2] == 0))[0]
    if bad.size:
        st.hist[bad] = -np.inf
        st.splittable[bad] = False
        sw.randomize_sublabels(bad + 1)
        c, l, _ = sw.posterior_step(bad + 1)
        _update(st, bad, c, l)
    if not no_more_splits:
        # check_and_split!: log H = log a + lG(N_l) + L_l + lG(N_r) + L_r - lG(N) - L
        N = st.N.astype(np.float64)
        cand = st.splittable & (st.N[:, 0] > 1) & (st.N[:, 1] > 0) & (st.N[:, 2] > 0) & (not final)
        ci = np.nonzero(cand)[0]
        split = []
        if ci.size:
            log_hr = (np.log(α) + gammaln(N[ci, 1]) + st.logml[ci, 1] + gammaln(N[ci, 2]) + st.logml[ci, 2]
                      - gammaln(N[ci, 0]) - st.logml[ci, 0])
            split = ci[log_hr > np.log(rng.random(ci.size))]
        if len(split):
            if np.isfinite(cfg.max_num_of_clusters):
                split = split[:max(0, int(cfg.max_num_of_clusters) - st.K)]
        if len(split):
            new = st.K + np.arange(len(split))
            st.grow(len(split))
            both = np.concatenate([split, new])
            st.hist[both] = -np.inf                       # create_splittable_from_params: fresh window, not splittable
            st.splittable[both] = False
            sw.apply_split(split + 1, new + 1)
            if cfg.use_smart_splits:                      # check_and_split! :374-378
                smart_init_device(sw, both + 1, cfg)
            c, l, _ = sw.posterior_step(both + 1)
            _update(st, both, c, l)
        # check_and_merge!: pairs i < j in order, both splittable and non-empty
        if merge is not None:
            N = st.N.astype(np.float64)
            sp = st.splittable.copy()
            merged_i, merged_j = [], []
            const = -np.log(α) + gammaln(α) - 2 * gammaln(0.5 * α)
            idx = np.nonzero(sp & (st.N[:, 0] > 0))[0]
            idx = idx[idx < merge.shape[0]]
            for a_, i in enumerate(idx):
                if not sp[i]:
                    continue
                js = idx[a_ + 1:]
                js = js[sp[js]]
                if not js.size:
                    continue
                Ni, Nj = N[i, 0], N[js, 0]
                log_hr = (const + gammaln(Ni + Nj) - gammaln(Ni + Nj + α) + gammaln(Ni + 0.5 * α) - gammaln(Ni)
                          - gammaln(Nj) + gammaln(Nj + 0.5 * α) + merge[i, js] - st.logml[i, 0] - st.logml[js, 0])
                u = np.log(rng.random(js.size))
                acc = (log_hr > u) | (final & (log_hr > np.log(0.1)))
                hit = np.nonzero(acc)[0]
                if hit.size:                             # the first accepted partner; i is not splittable afterwards
                    j = int(js[hit[0]])
                    merged_i.append(int(i)); merged_j.append(j)
                    st.N[i] = (st.N[i, 0] + st.N[j, 0], st.N[i, 0], st.N[j, 0])
                    st.logml[i] = (merge[i, j], st.logml[i, 0], st.logml[j, 0])
                    st.N[j] = 0
                    sp[i] = sp[j] = False
                    st.hist[i] = -np.inf
            st.splittable = sp & st.splittable
            if merged_i:
                mi, mj = np.asarray(merged_i), np.asarray(merged_j)
                st.splittable[mi] = False
                st.splittable[mj] = False
                sw.apply_merge(mi + 1, mj + 1)
                for i, j in zip(merged_i, merged_j):
                    sw.params_merge(i + 1, j + 1)
                sw.posterior_step(mi + 1, from_table=True, fetch=False)
    # remove_empty_clusters!
    if (st.N[:, 0] == 0).any():
        sw.remove_empty(st.N[:, 0])
        mask = st.N[:, 0] > 0
        if keep_params and getattr(st, "params", None) is not None:
            kp = mask[:st.params[0].shape[0]]
            st.params = tuple(a[kp] for a in st.params)
        st.keep(mask)


def smart_init_device(sw, clusters, cfg):
    """smart_cluster_init! (:555-623) for the listed clusters (1-based): the cluster statistics come back through
    dpmm_suff_stats, the D x D eigen-decomposition stays on the host, the rest is the three worker calls."""
    from .host import smart_split_direction, smart_kmeans
    clusters = [int(c) for c in clusters]
    counts, sum_x, sum_xx = sw.suff_stats(clusters)
    for a, c in enumerate(clusters):
        if counts[a, 0] == 0:
            continue
        v1, mu = smart_split_direction(float(counts[a, 0]), sum_x[a, 0], sum_xx[a, 0])
        smart_kmeans(sw, c, v1, mu, cfg.max_split_iter)


def run_model_device(dp_model, cfg, rng, normalized_mutual_info, first_iter=1, resume=False):
    """init_first_clusters! (:62-78) + run_model (:336-404) with the parameter step on the device.  resume=True: the
    group was restored from a checkpoint (labels / sub-labels already on the device, local_clusters holding the
    history windows); the statistics and posterior tables are rebuilt from the labels."""
    g = dp_model.group
    sw = g.sweep
    hyper = g.model_hyperparams.distribution_hyper_params
    α = g.model_hyperparams.α
    if isinstance(hyper, P.niw_hyperparams):
        sw.set_hyper_niw(hyper.κ, hyper.m, hyper.ν, hyper.ψ, α)
    elif isinstance(hyper, P.diag_niw_hyperparams):
        sw.set_hyper_diag(hyper.κ, hyper.m, hyper.ν, hyper.ψ, α)
    else:
        sw.set_hyper_multinomial(hyper.α, α)
    if resume:
        K = len(g.local_clusters)
        st = DeviceState(K, cfg.burnout_period + 5)
        for k, c in enumerate(g.local_clusters):
            h = np.asarray(c.cluster_params.logsublikelihood_hist, np.float64)
            st.hist[k, :min(h.size, st.window)] = h[:st.window]
            st.splittable[k] = bool(c.cluster_params.splittable)
        counts, logml, _ = sw.posterior_step(np.arange(1, K + 1))
        st.N[:], st.logml[:] = counts[:K], logml[:K]
    else:
        st = DeviceState(cfg.initial_clusters, cfg.burnout_period + 5)
        for _ in range(cfg.initial_clusters):
            sw.randomize_sublabels(None)                       # split_first_cluster_worker! per first cluster
        counts, logml, _ = sw.posterior_step(None)
        if cfg.use_smart_splits:                               # init_first_clusters! :70-75
            smart_init_device(sw, np.arange(1, st.K + 1), cfg)
            counts, logml, _ = sw.posterior_step(None)
        st.N[:], st.logml[:] = counts[:st.K], logml[:st.K]
        history_step(st, cfg)                                  # sample_clusters!(group, false) of init_first_clusters!
        sw.sample_params(st.K, unit_weights=True)
    iter_count, nmi_hist, ll_hist, k_hist = [], [], [], []
    first = True
    start_time = time.time()
    for i in range(first_iter, cfg.iterations + 1):
        final = i >= cfg.iterations - cfg.argmax_sample_stop
        no_more_splits = (i >= cfg.iterations - cfg.split_stop) or (st.K >= cfg.max_num_of_clusters)
        t0 = time.perf_counter()
        if first:
            # the parameters of the first iteration were drawn above; group_step draws again, as the reference does
            first = False
        group_step_device(sw, st, α, no_more_splits, final, cfg, rng, keep_params=(i == cfg.iterations))
        iter_count.append(time.perf_counter() - t0)
        k_hist.append(st.K)
        if cfg.ground_truth is not None:
            nmi_hist.append(normalized_mutual_info(cfg.ground_truth, sw.get_labels()))
        else:
            nmi_hist.append("no gt")
        if cfg.use_verbose:
            nz = st.N[:, 0] > 0
            lp = (gammaln(α) - gammaln(sw.n_total + α)
                  + (st.logml[nz, 0] + np.log(α) + gammaln(st.N[nz, 0].astype(np.float64))).sum())
            ll_hist.append(float(lp))
            print(f"Iteration: {i} || Clusters count: {st.K} || Log posterior: {ll_hist[-1]} || "
                  f"NMI score: {nmi_hist[-1]} || Iter Time:{iter_count[-1]} || Total time:{sum(iter_count)}")
        else:
            ll_hist.append(1)
        if i % cfg.model_save_interval == 0 and cfg.should_save_model:      # run_model :395-399
            from .checkpoint import save_model
            from .host import _clusters_from_device
            _clusters_from_device(g, st, cfg)
            save_model(dp_model, cfg.save_path, cfg.save_file_prefix, i, time.time() - start_time, cfg.global_params)
    return st, iter_count, nmi_hist, ll_hist, k_hist
