"""Data and checkpoint I/O of the advanced mode (SURVEY 8f-4).

  load_data                  src/utils.jl:5-14            <path><prefix>.npy, NaN -> 0, transposed to D x N
  save_model                 src/dp-parallel-sampling.jl:451-456  + create_pts_less_group src/ds.jl:85-87
  run_model_from_checkpoint  src/dp-parallel-sampling.jl:428-449  + create_model_from_saved_data ds.jl:89-92
  dp_parallel(params_file)   src/dp-parallel-sampling.jl:317-334  with the globals of src/global_params.jl

The reference stores its checkpoints as JLD2 (serialised Julia structs).  Here a checkpoint is one `.npz` of plain
arrays holding the same five items -- `group` (the pts_less_group: hyper-parameters, labels, sub-labels, every
local_cluster, weights), `hyperparams`, `iter`, `total_time`, `global_params` -- which NPZ.jl (a dependency the
reference already has) reads on the Julia side.  A model with the outlier component also stores its weight and prior
as `outlier_weight` and `outlier_*` next to `prior_*`; files without them hold a model without the component.  Labels and sub-labels are restored through
dpmm_set_labels / dpmm_set_sublabels (`group.labels = distribute(group.labels)`, :437-439); X is reloaded from
`data_path`/`data_prefix` exactly as the reference does.
"""
from __future__ import annotations

import json
import os
import re

import numpy as np

from . import priors as P

F32 = np.float32
FORMAT = 1


# ------------------------------------------------------------------------------------------- data ----------
def load_data(path, prefix="", swapDimension=True):
    """utils.jl:5-14.  Also reads `path + prefix + ".npz"` written by scipy.sparse.save_npz when there is no ".npy":
    an N x D sparse matrix like the reference's array, returned as CSC (D x N when swapDimension)."""
    if not os.path.exists(path + prefix + ".npy") and os.path.exists(path + prefix + ".npz"):
        import scipy.sparse as sps
        m = sps.load_npz(path + prefix + ".npz")
        return sps.csc_matrix(m.T if swapDimension else m)
    arr = np.load(path + prefix + ".npy")
    if np.issubdtype(arr.dtype, np.floating):
        arr = np.where(np.isnan(arr), 0.0, arr)
    return arr.T if swapDimension else arr


# ------------------------------------------------------------------------------------ parameter files -------
_DEFAULTS = dict(                                   # src/global_params.jl
    data_path="/path/to/data/", data_prefix="data_prefix", iterations=100, hard_clustering=False, initial_clusters=1,
    argmax_sample_stop=5, split_stop=5, random_seed=None, max_split_iter=20, burnout_period=20, max_clusters=np.inf,
    α=10.0, hyper_params=None, outlier_mod=0.05, outlier_hyper_params=None, enable_saving=True,
    model_save_interval=1000, save_path="/path/to/save/dir/", overwrite_prec=False, save_file_prefix="checkpoint_",
    smart_splits=False)


def _jl_to_py(src):
    """The subset of Julia the reference's parameter files use (assignments of literals, `nothing`, `Inf`, `true`,
    `zeros(Float32,d)`, `ones(Float32,d)`, `Matrix{Float32}(I, d, d)`, niw_hyperparams(...), multinomial_hyper(...),
    diag_niw_hyperparams(...))."""
    out = []
    for line in src.splitlines():
        line = re.sub(r"#.*$", "", line).rstrip()
        line = re.sub(r"^\s*(global|const)\s+", "", line)
        line = re.sub(r"\bnothing\b", "None", line)
        line = re.sub(r"\btrue\b", "True", line)
        line = re.sub(r"\bfalse\b", "False", line)
        line = re.sub(r"\bInf\b", "np.inf", line)
        line = re.sub(r"Matrix\{Float(?:32|64)\}\(I\s*,\s*([^,]+),\s*([^)]+)\)", r"np.eye(int(\1), int(\2))", line)
        line = re.sub(r"\b(zeros|ones)\(Float(?:32|64)\s*,\s*([^)]+)\)", r"np.\1(int(\2))", line)
        line = re.sub(r"Float32\(([^)]+)\)", r"float(\1)", line)
        out.append(line)
    return "\n".join(out)


def read_params(params_file):
    """`include(model_params)` (dp-parallel-sampling.jl:318): a global_params.jl-style file (Julia subset above) or
    a Python file with the same variable names.  Returns the globals as a dict over the reference's defaults."""
    src = open(params_file, encoding="utf-8").read()
    if not params_file.endswith(".py"):
        src = _jl_to_py(src)
    ns = {"np": np, "niw_hyperparams": P.niw_hyperparams, "multinomial_hyper": P.multinomial_hyper,
          "diag_niw_hyperparams": P.diag_niw_hyperparams}
    exec(compile(src, params_file, "exec"), ns)        # a parameter file is code, in the reference as here
    g = dict(_DEFAULTS)
    g.update({k: v for k, v in ns.items() if k in _DEFAULTS or k == "alpha"})
    if "alpha" in ns:
        g["α"] = ns["alpha"]
    return g


# ------------------------------------------------------------------------------------- checkpoints ---------
def _hyper_arrays(h, tag, out):
    if isinstance(h, (P.niw_hyperparams, P.diag_niw_hyperparams)):
        out[tag + "kappa"], out[tag + "m"], out[tag + "nu"], out[tag + "psi"] = np.float64(h.κ), h.m, np.float64(h.ν), h.ψ
    else:
        out[tag + "alpha"] = np.asarray(h.α, F32)


def _hyper_from(z, tag, kind, idx=None):
    def get(name):
        a = z[tag + name]
        return a if idx is None else a[idx]
    if kind in ("niw", "diag"):
        T = P.niw_hyperparams if kind == "niw" else P.diag_niw_hyperparams
        return T(float(get("kappa")), np.array(get("m")), float(get("nu")), np.array(get("psi")))
    return P.multinomial_hyper(np.array(get("alpha")))


def save_model(model, path, filename, iter, total_time, global_params):
    """save_model :451-456.  `model` is the dp_parallel_sampling (its group still holds the sweep: labels and
    sub-labels are gathered as create_pts_less_group does with Array(group.labels)).  Returns the file name."""
    g = model.group
    hyper = model.model_hyperparams.distribution_hyper_params
    kind = ("niw" if isinstance(hyper, P.niw_hyperparams) else "diag" if isinstance(hyper, P.diag_niw_hyperparams)
            else "multinomial")
    K = len(g.local_clusters)
    out = {"labels": np.asarray(g.sweep.get_labels(), np.int64),
           "labels_subcluster": np.asarray(g.sweep.get_sublabels(), np.int64),
           "weights": np.asarray(g.weights, F32)}
    _hyper_arrays(hyper, "prior_", out)
    if getattr(model, "outlier_weight", 0) > 0:
        out["outlier_weight"] = np.float64(model.outlier_weight)
        _hyper_arrays(model.outlier_params, "outlier_", out)
    trip = lambda c: (c.cluster_params.cluster_params, c.cluster_params.cluster_params_l, c.cluster_params.cluster_params_r)
    stack = lambda f, dt=np.float64: np.array([[f(cp) for cp in trip(c)] for c in g.local_clusters], dt).reshape(
        (K, 3) + np.shape(f(trip(g.local_clusters[0])[0]))) if K else np.zeros((0, 3), dt)
    out["stats_N"] = stack(lambda cp: cp.suff_statistics.N)
    if kind == "niw":
        out["stats_sum"] = stack(lambda cp: cp.suff_statistics.points_sum)
        out["stats_S"] = stack(lambda cp: cp.suff_statistics.S)
        for name, f in (("kappa", lambda h: h.κ), ("m", lambda h: h.m), ("nu", lambda h: h.ν), ("psi", lambda h: h.ψ)):
            out["post_" + name] = stack(lambda cp, f=f: f(cp.posterior_hyperparams))
        out["dist_mu"] = stack(lambda cp: cp.distribution.μ, F32)
        out["dist_Sigma"] = stack(lambda cp: cp.distribution.Σ, F32)
        out["dist_invSigma"] = stack(lambda cp: cp.distribution.invΣ, F32)
        out["dist_logdet"] = stack(lambda cp: cp.distribution.logdetΣ, F32)
        D = hyper.m.shape[0]
        out["dist_invChol"] = stack(lambda cp: np.zeros((D, D)) if cp.distribution.invChol is None else cp.distribution.invChol)
    elif kind == "diag":                                # the NIW items, with vectors where NIW has matrices
        out["stats_sum"] = stack(lambda cp: cp.suff_statistics.points_sum)
        out["stats_S"] = stack(lambda cp: cp.suff_statistics.S_diag)
        for name, f in (("kappa", lambda h: h.κ), ("m", lambda h: h.m), ("nu", lambda h: h.ν), ("psi", lambda h: h.ψ)):
            out["post_" + name] = stack(lambda cp, f=f: f(cp.posterior_hyperparams))
        out["dist_mu"] = stack(lambda cp: cp.distribution.μ, F32)
        out["dist_var"] = stack(lambda cp: cp.distribution.σ2, F32)
        out["dist_logdet"] = stack(lambda cp: cp.distribution.logdetΣ, F32)
    else:
        out["stats_sum"] = stack(lambda cp: cp.suff_statistics.points_sum, F32)
        out["post_alpha"] = stack(lambda cp: cp.posterior_hyperparams.α, F32)
        out["dist_alpha"] = stack(lambda cp: cp.distribution.α, F32)
    out["lr_weights"] = np.array([c.cluster_params.lr_weights for c in g.local_clusters], np.float64).reshape(K, 2)
    out["splittable"] = np.array([c.cluster_params.splittable for c in g.local_clusters], bool)
    out["logsublikelihood_hist"] = np.array([c.cluster_params.logsublikelihood_hist for c in g.local_clusters], np.float64)
    out["points_count"] = np.array([[c.points_count, c.l_count, c.r_count] for c in g.local_clusters], np.int64).reshape(K, 3)
    gp = dict(global_params) if isinstance(global_params, dict) else {"model_params": global_params}
    meta = {"format": FORMAT, "kind": kind, "alpha": model.model_hyperparams.α, "total_dim": model.model_hyperparams.total_dim,
            "iter": int(iter), "total_time": float(total_time),
            "global_params": {k: (None if v is None else (float(v) if isinstance(v, (float, np.floating)) else v))
                              for k, v in gp.items() if isinstance(v, (int, float, str, bool, type(None), np.floating))}}
    out["meta"] = np.frombuffer(json.dumps(meta).encode(), np.uint8)
    fname = path + filename + "_" + str(iter) + ".npz"
    np.savez(fname, **out)
    return fname


def load_checkpoint(filename):
    """`@load filename group hyperparams iter total_time global_params` (:430): returns
    (pts_less_group as a dict {model_hyperparams, labels, labels_subcluster, local_clusters, weights},
     hyperparams, iter, total_time, global_params)."""
    from . import host as H
    z = np.load(filename)
    meta = json.loads(bytes(z["meta"]).decode())
    if meta["format"] != FORMAT:
        raise ValueError(f"checkpoint format {meta['format']} (this build reads {FORMAT})")
    kind = meta["kind"]
    prior = _hyper_from(z, "prior_", kind)
    mh = H.model_hyper_params(prior, meta["alpha"], meta["total_dim"])
    ow, op = 0.0, None
    if "outlier_weight" in z.files:
        ow, op = float(z["outlier_weight"]), _hyper_from(z, "outlier_", kind)
    K = z["stats_N"].shape[0]
    clusters = []
    for k in range(K):
        cps = []
        for s in range(3):
            if kind == "niw":
                ss = P.niw_sufficient_statistics(float(z["stats_N"][k, s]), np.array(z["stats_sum"][k, s]), np.array(z["stats_S"][k, s]))
                post = _hyper_from(z, "post_", kind, (k, s))
                dist = P.mv_gaussian(np.array(z["dist_mu"][k, s]), np.array(z["dist_Sigma"][k, s]), np.array(z["dist_invSigma"][k, s]),
                                     float(z["dist_logdet"][k, s]), np.array(z["dist_invChol"][k, s]))
            elif kind == "diag":
                ss = P.diag_niw_sufficient_statistics(float(z["stats_N"][k, s]), np.array(z["stats_sum"][k, s]),
                                                      np.array(z["stats_S"][k, s]))
                post = _hyper_from(z, "post_", kind, (k, s))
                dist = P.diag_gaussian(np.array(z["dist_mu"][k, s]), np.array(z["dist_var"][k, s]), float(z["dist_logdet"][k, s]))
            else:
                ss = P.multinomial_sufficient_statistics(float(z["stats_N"][k, s]), np.array(z["stats_sum"][k, s]))
                post = _hyper_from(z, "post_", kind, (k, s))
                dist = P.multinomial_dist(np.array(z["dist_alpha"][k, s]))
            cps.append(H.cluster_parameters(op if (ow > 0 and k == 0) else prior, dist, ss, post))
        sp = H.splittable_cluster_params(cps[0], cps[1], cps[2], np.array(z["lr_weights"][k]), bool(z["splittable"][k]),
                                         np.array(z["logsublikelihood_hist"][k]))
        pc = z["points_count"][k]
        clusters.append(H.local_cluster(sp, meta["total_dim"], int(pc[0]), int(pc[1]), int(pc[2])))
    group = {"model_hyperparams": mh, "labels": np.array(z["labels"]), "labels_subcluster": np.array(z["labels_subcluster"]),
             "local_clusters": clusters, "weights": np.array(z["weights"], F32), "outlier_weight": ow,
             "outlier_params": op}
    return group, mh, meta["iter"], meta["total_time"], meta["global_params"]
