"""GpuSweep: thin Python mirror of the C ABI (one object = one dpmm_ctx = one GPU shard).

Method names follow the boundary table of SURVEY.md 8b; the oracle's `OracleSweep`
(oracle/dpmm_oracle.py, test infrastructure) exposes the same methods so that host code and parity
tests can drive either with identical calls.  All labels / cluster indices are 1-based, as in the
reference (Julia).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L

NIW = L.PRIOR_NIW
MULTINOMIAL = L.PRIOR_MULTINOMIAL


def _ptr(a, ctype):
    return None if a is None else a.ctypes.data_as(C.POINTER(ctype))


def _i64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.int64))


class GpuSweep:
    """The worker side of the sampler on one B200 (src/local_clusters_actions.jl *_worker!)."""

    def __init__(self, x, prior_kind, seed=0, global_offset=0, device=0):
        self.lib = L.load()
        x = np.asarray(x, dtype=np.float32)
        if x.ndim != 2:
            raise ValueError("x must be D x N")
        self.D, self.n = int(x.shape[0]), int(x.shape[1])
        self.prior_kind = int(prior_kind)
        self.K = 0
        # D x N column-major (Julia, numpy order="F") == N x D row-major: every point is D contiguous floats.
        # A column-major array goes up as it is; a row-major (numpy default) one is transposed once.
        xt = np.ascontiguousarray(x.T)
        h = C.c_void_p()
        rc = self.lib.dpmm_create(C.byref(h), _ptr(xt, C.c_float), self.n, self.D, self.prior_kind, int(device),
                                  C.c_uint64(int(seed) & (2 ** 64 - 1)), int(global_offset))
        L.check(rc, None)
        self.h = h

    # ---- lifetime ----
    def close(self):
        if getattr(self, "h", None):
            self.lib.dpmm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        L.check(rc, self.h)

    def sync(self):
        self._ck(self.lib.dpmm_sync(self.h))

    def set_stream(self, cuda_stream_ptr):
        self._ck(self.lib.dpmm_set_stream(self.h, C.c_void_p(int(cuda_stream_ptr))))

    def set_sampler(self, sampler):
        self._ck(self.lib.dpmm_set_sampler(self.h, int(sampler)))

    # ---- labels ----
    def init_labels(self, init_clusters, outlier=False):
        self._ck(self.lib.dpmm_init_labels(self.h, int(init_clusters), 1 if outlier else 0))

    def randomize_sublabels(self, indices=None):
        if indices is None:
            self._ck(self.lib.dpmm_randomize_sublabels(self.h, None, 0))
        else:
            idx = _i64(indices)
            self._ck(self.lib.dpmm_randomize_sublabels(self.h, _ptr(idx, C.c_int64), len(idx)))

    def get_labels(self):
        out = np.empty(self.n, np.int64)
        self._ck(self.lib.dpmm_get_labels(self.h, _ptr(out, C.c_int64)))
        return out

    def get_sublabels(self):
        out = np.empty(self.n, np.int64)
        self._ck(self.lib.dpmm_get_sublabels(self.h, _ptr(out, C.c_int64)))
        return out

    def set_labels(self, labels):
        a = _i64(labels)
        assert a.shape == (self.n,)
        self._ck(self.lib.dpmm_set_labels(self.h, _ptr(a, C.c_int64)))

    def set_sublabels(self, sublabels):
        a = _i64(sublabels)
        assert a.shape == (self.n,)
        self._ck(self.lib.dpmm_set_sublabels(self.h, _ptr(a, C.c_int64)))

    # ---- parameters ----
    def set_params_niw(self, mu, inv_sigma, logdet, weights, lr_weights):
        """mu [K,3,D], inv_sigma [K,3,D,D], logdet [K,3], weights [K], lr_weights [K,2] (Float32)."""
        mu = np.ascontiguousarray(mu, np.float32)
        K = mu.shape[0]
        inv_sigma = np.ascontiguousarray(inv_sigma, np.float32)
        logdet = np.ascontiguousarray(logdet, np.float32)
        weights = np.ascontiguousarray(weights, np.float32)
        lr_weights = np.ascontiguousarray(lr_weights, np.float32)
        assert mu.shape == (K, 3, self.D) and inv_sigma.shape == (K, 3, self.D, self.D)
        assert logdet.shape == (K, 3) and weights.shape == (K,) and lr_weights.size == 2 * K
        f = C.c_float
        self._ck(self.lib.dpmm_set_params_niw(self.h, K, _ptr(mu, f), _ptr(inv_sigma, f), _ptr(logdet, f),
                                              _ptr(weights, f), _ptr(lr_weights, f)))
        self.K = K

    def set_params_multinomial(self, log_p, weights, lr_weights):
        """log_p [K,3,D] log-probabilities (Float32)."""
        log_p = np.ascontiguousarray(log_p, np.float32)
        K = log_p.shape[0]
        weights = np.ascontiguousarray(weights, np.float32)
        lr_weights = np.ascontiguousarray(lr_weights, np.float32)
        assert log_p.shape == (K, 3, self.D) and weights.shape == (K,) and lr_weights.size == 2 * K
        f = C.c_float
        self._ck(self.lib.dpmm_set_params_multinomial(self.h, K, _ptr(log_p, f), _ptr(weights, f), _ptr(lr_weights, f)))
        self.K = K

    # ---- sweep ----
    def sample_labels(self, final=False):
        self._ck(self.lib.dpmm_sample_labels(self.h, 1 if final else 0))

    def sample_sublabels(self):
        self._ck(self.lib.dpmm_sample_sublabels(self.h))

    def suff_stats(self, indices=None, fetch=True, out=None):
        """Returns (counts [m,3] i64, sum_x [m,3,D] f64, sum_xx [m,3,D,D] f64 or None).
        `out`: an earlier result of the same shape to be overwritten (saves the allocation and the
        first-touch page faults of ~0.5 MB per call in a tight loop)."""
        if indices is None:
            m, idx_p, idx = max(int(self.lib.dpmm_num_clusters(self.h)), 1), None, None
        else:
            idx = _i64(indices)
            m, idx_p = len(idx), _ptr(idx, C.c_int64)
        if not fetch:
            self._ck(self.lib.dpmm_suff_stats(self.h, idx_p, m, None, None, None))
            return None
        if out is not None:
            counts, sum_x, sum_xx = out
            ok = (counts.shape == (m, 3) and counts.dtype == np.int64 and counts.flags.c_contiguous
                  and sum_x.shape == (m, 3, self.D) and sum_x.dtype == np.float64 and sum_x.flags.c_contiguous
                  and (sum_xx is None) == (self.prior_kind != NIW)
                  and (sum_xx is None or (sum_xx.shape == (m, 3, self.D, self.D) and sum_xx.dtype == np.float64
                                          and sum_xx.flags.c_contiguous)))
            if not ok:
                raise ValueError("suff_stats(out=...): arrays of the wrong shape / dtype / layout")
        else:
            counts = np.zeros((m, 3), np.int64)
            sum_x = np.zeros((m, 3, self.D), np.float64)
            sum_xx = np.zeros((m, 3, self.D, self.D), np.float64) if self.prior_kind == NIW else None
        self._ck(self.lib.dpmm_suff_stats(self.h, idx_p, m, _ptr(counts, C.c_int64), _ptr(sum_x, C.c_double),
                                          _ptr(sum_xx, C.c_double)))
        return counts, sum_x, sum_xx

    # ---- device-side parameter step ----
    def set_hyper_niw(self, kappa, m, nu, psi, alpha):
        m = np.ascontiguousarray(m, np.float64).reshape(-1)
        psi = np.ascontiguousarray(psi, np.float64)
        assert m.shape == (self.D,) and psi.shape == (self.D, self.D)
        self._ck(self.lib.dpmm_set_hyper_niw(self.h, float(kappa), _ptr(m, C.c_double), float(nu), _ptr(psi, C.c_double),
                                             float(alpha)))

    def set_hyper_multinomial(self, alpha_prior, alpha):
        a = np.ascontiguousarray(alpha_prior, np.float32).reshape(-1)
        assert a.shape == (self.D,)
        self._ck(self.lib.dpmm_set_hyper_multinomial(self.h, _ptr(a, C.c_float), float(alpha)))

    def posterior_step(self, indices=None, splittable=None, from_table=False, fetch=True):
        """Statistics (unless from_table) -> table -> posteriors.  Returns (counts [m,3] i64, logml [m,3] f64,
        merge [K,K] f64 or None); `splittable` (bool [K]) requests the merge table."""
        if indices is None:
            m, idx_p, idx = max(int(self.lib.dpmm_num_clusters(self.h)), 1), None, None
        else:
            idx = _i64(indices)
            m, idx_p = len(idx), _ptr(idx, C.c_int64)
        if not fetch:
            self._ck(self.lib.dpmm_posterior_step(self.h, idx_p, m, 1 if from_table else 0, None, 0, None, None, None))
            return None
        counts = np.zeros((m, 3), np.int64)
        logml = np.zeros((m, 3), np.float64)
        merge, sp, km = None, None, 0
        if splittable is not None and len(splittable) > 1:
            sp = np.ascontiguousarray(splittable, np.uint8)
            km = len(sp)
            merge = np.empty((km, km), np.float64)
        self._ck(self.lib.dpmm_posterior_step(self.h, idx_p, m, 1 if from_table else 0, _ptr(sp, C.c_uint8), km,
                                              _ptr(counts, C.c_int64), _ptr(logml, C.c_double), _ptr(merge, C.c_double)))
        return counts, logml, merge

    def sample_params(self, K, from_prior=False, unit_weights=False):
        self._ck(self.lib.dpmm_sample_params(self.h, int(K), 1 if from_prior else 0, 1 if unit_weights else 0))
        self.K = int(K)

    def params_merge(self, i, j):
        self._ck(self.lib.dpmm_params_merge(self.h, int(i), int(j)))

    def get_params_niw(self, K):
        """(mu [K,3,D] f32, lfac [K,3,D,D] f64 with invSigma = L L', logdet [K,3] f32, weights [K] f32, lr [K,2] f32)."""
        mu = np.empty((K, 3, self.D), np.float32)
        lf = np.empty((K, 3, self.D, self.D), np.float64)
        ld = np.empty((K, 3), np.float32)
        w = np.empty(K, np.float32)
        lr = np.empty((K, 2), np.float32)
        self._ck(self.lib.dpmm_get_params_niw(self.h, int(K), _ptr(mu, C.c_float), _ptr(lf, C.c_double), _ptr(ld, C.c_float),
                                              _ptr(w, C.c_float), _ptr(lr, C.c_float)))
        return mu, lf, ld, w, lr

    def get_params_multinomial(self, K):
        """(log_p [K,3,D] f32, weights [K] f32, lr [K,2] f32)."""
        lp = np.empty((K, 3, self.D), np.float32)
        w = np.empty(K, np.float32)
        lr = np.empty((K, 2), np.float32)
        self._ck(self.lib.dpmm_get_params_multinomial(self.h, int(K), _ptr(lp, C.c_float), _ptr(w, C.c_float),
                                                      _ptr(lr, C.c_float)))
        return lp, w, lr

    def predict_niw(self, u, mu, tconst, df, want_probs=True):
        """Posterior-predictive labels (and probabilities) of this context's points; see dpmm_predict_niw."""
        u = np.ascontiguousarray(u, np.float32); mu = np.ascontiguousarray(mu, np.float32)
        tconst = np.ascontiguousarray(tconst, np.float32); df = np.ascontiguousarray(df, np.float32)
        K = u.shape[0]
        assert u.shape == (K, self.D, self.D) and mu.shape == (K, self.D) and tconst.shape == (K,) and df.shape == (K,)
        labels = np.empty(self.n, np.int64)
        probs = np.empty((self.n, K), np.float32) if want_probs else None
        self._ck(self.lib.dpmm_predict_niw(self.h, K, _ptr(u, C.c_float), _ptr(mu, C.c_float), _ptr(tconst, C.c_float),
                                           _ptr(df, C.c_float), _ptr(labels, C.c_int64), _ptr(probs, C.c_float)))
        return labels, probs

    def predict_multinomial(self, logp, logw, want_probs=True):
        """Posterior-predictive labels (and probabilities) of this context's points; see dpmm_predict_multinomial."""
        logp = np.ascontiguousarray(logp, np.float64); logw = np.ascontiguousarray(logw, np.float32)
        K = logp.shape[0]
        assert logp.shape == (K, self.D) and logw.shape == (K,)
        labels = np.empty(self.n, np.int64)
        probs = np.empty((self.n, K), np.float32) if want_probs else None
        self._ck(self.lib.dpmm_predict_multinomial(self.h, K, _ptr(logp, C.c_double), _ptr(logw, C.c_float),
                                                   _ptr(labels, C.c_int64), _ptr(probs, C.c_float)))
        return labels, probs

    # ---- smart splits (smart_cluster_init! local_clusters_actions.jl:555-623) ----
    def smart_project(self, cluster, v, mu):
        """tranform_points_worker! on every shard + the master's min / max: returns (lo, hi, count)."""
        v = np.ascontiguousarray(v, np.float64); mu = np.ascontiguousarray(mu, np.float64)
        assert v.shape == (self.D,) and mu.shape == (self.D,)
        lohi = np.empty(2, np.float64)
        cnt = np.zeros(1, np.int64)
        self._ck(self.lib.dpmm_smart_project(self.h, int(cluster), _ptr(v, C.c_double), _ptr(mu, C.c_double),
                                             _ptr(lohi, C.c_double), _ptr(cnt, C.c_int64)))
        return float(lohi[0]), float(lohi[1]), int(cnt[0])

    def smart_kmeans_iter(self, min_mean, max_mean):
        """kmeans_iter_worker! on every shard + the master's sums: returns (sum_1, count_1, sum_2, count_2)."""
        out = np.empty(4, np.float64)
        self._ck(self.lib.dpmm_smart_kmeans_iter(self.h, float(min_mean), float(max_mean), _ptr(out, C.c_double)))
        return tuple(float(o) for o in out)

    def smart_set_sublabels(self, cluster):
        """set_smart_labels_in_worker!."""
        self._ck(self.lib.dpmm_smart_set_sublabels(self.h, int(cluster)))

    # ---- relabel ----
    def apply_split(self, indices, new_indices):
        a, b = _i64(indices), _i64(new_indices)
        assert len(a) == len(b)
        self._ck(self.lib.dpmm_apply_split(self.h, _ptr(a, C.c_int64), _ptr(b, C.c_int64), len(a)))

    def apply_merge(self, indices, new_indices):
        a, b = _i64(indices), _i64(new_indices)
        assert len(a) == len(b)
        self._ck(self.lib.dpmm_apply_merge(self.h, _ptr(a, C.c_int64), _ptr(b, C.c_int64), len(a)))

    def remove_empty(self, pts_count):
        a = _i64(pts_count)
        self._ck(self.lib.dpmm_remove_empty(self.h, _ptr(a, C.c_int64), len(a)))

    # ---- multi-GPU ----
    @staticmethod
    def nccl_unique_id():
        lib = L.load()
        buf = (C.c_char * 128)()
        L.check(lib.dpmm_nccl_unique_id(C.cast(buf, C.c_void_p)), None)
        return bytes(buf)

    def comm_init(self, unique_id: bytes, rank: int, world_size: int):
        buf = C.create_string_buffer(unique_id, 128)
        self._ck(self.lib.dpmm_comm_init(self.h, C.cast(buf, C.c_void_p), int(rank), int(world_size)))

    # ---- parity / measurement hooks ----
    def set_uniforms(self, u_label=None, u_sub=None, r_bits=None):
        ul = None if u_label is None else np.ascontiguousarray(u_label, np.float64)
        us = None if u_sub is None else np.ascontiguousarray(u_sub, np.float64)
        rb = None if r_bits is None else np.ascontiguousarray(r_bits, np.uint8)
        self._ck(self.lib.dpmm_set_uniforms(self.h, _ptr(ul, C.c_double), _ptr(us, C.c_double), _ptr(rb, C.c_uint8)))

    def debug_loglik(self, which=0):
        cols = self.K if which == 0 else 2
        out = np.empty((cols, self.n), np.float32)
        self._ck(self.lib.dpmm_debug_loglik(self.h, int(which), _ptr(out, C.c_float)))
        return np.ascontiguousarray(out.T)  # n x cols, as the reference's parr

    def tc_stats(self, overflow=False):
        """(points drawn, exact cluster evaluations[, points finished by the overflow kernel]) of the last
        sample_labels on the tensor-core path (needs DPMM_TC_STATS=1)."""
        out = np.zeros(3, np.int64)
        self._ck(self.lib.dpmm_debug_tc_stats(self.h, _ptr(out, C.c_int64)))
        return (int(out[0]), int(out[1]), int(out[2])) if overflow else (int(out[0]), int(out[1]))

    def sort_state(self):
        """(perm: point indices in the order of the current label sort, points whose label changed in the last
        tensor-core label call)."""
        perm = np.empty(self.n, np.int32)
        moved = np.zeros(1, np.int64)
        self._ck(self.lib.dpmm_debug_sort(self.h, _ptr(perm, C.c_int32), _ptr(moved, C.c_int64)))
        return perm, int(moved[0])

    def fused_stats(self):
        """(fused sub-label+statistics launches, suff_stats calls served from them, exact recomputations)."""
        out = np.zeros(3, np.int64)
        self._ck(self.lib.dpmm_debug_fused_stats(self.h, _ptr(out, C.c_int64)))
        return int(out[0]), int(out[1]), int(out[2])

    def timing_enable(self, on=True):
        self._ck(self.lib.dpmm_timing_enable(self.h, 1 if on else 0))

    def timing_read(self, reset=True):
        nk = self.lib.dpmm_timing_kinds()
        ms = np.zeros(nk, np.float64)
        cnt = np.zeros(nk, np.int64)
        self._ck(self.lib.dpmm_timing_read(self.h, _ptr(ms, C.c_double), _ptr(cnt, C.c_int64), 1 if reset else 0))
        return {self.lib.dpmm_timing_name(i).decode(): (float(ms[i]), int(cnt[i])) for i in range(nk)}

    def launch_count(self):
        return int(self.lib.dpmm_launch_count(self.h))
