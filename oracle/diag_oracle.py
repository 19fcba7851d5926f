"""CPU ORACLE of the diagonal-covariance Gaussian prior -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The NumPy restatement of what the sweep computes on a DPMM_PRIOR_DIAG_GAUSSIAN context (csrc/kernels_diag.cuh), on
top of dpmm_oracle's sweep (draws, relabelling and randomness are shared): the log-likelihood in the kernels' Float32
order and Float64 statistics [N | sum x | sum x^2 per feature].  Only tests may import this module.
"""
from __future__ import annotations

import numpy as np

from . import dpmm_oracle as O

F32 = np.float32
DIAG = 2


def _fma_f32(a, b, c):
    """Float32 fma: the exact product of two Float32 values fits a Float64, so a Float64 multiply-add rounded to
    Float32 is the single-rounding result except in rare double-rounding cases (far below the parity tolerances)."""
    return (np.asarray(a, np.float64) * np.asarray(b, np.float64) + np.asarray(c, np.float64)).astype(F32)


def diag_images(mu, var):
    """What dpmm_set_params_diag derives per feature: s = 1/sigma and b = -s mu, each rounded once from Float64."""
    s = (1.0 / np.sqrt(np.asarray(var, F32).astype(np.float64))).astype(F32)
    b = (-(s.astype(np.float64)) * np.asarray(mu, F32).astype(np.float64)).astype(F32)
    return s, b


def diag_gaussian_log_likelihood(x, mu, var, logdet):
    """t = fma(s_d, x_d, b_d), acc = fma(t, t, acc) over ascending d, then r = cst - acc / 2 with
    cst = -(D log 2pi + logdetSigma) / 2 rounded once to Float32.  The constant uses D, not mv_gaussian's D^2."""
    x = np.asarray(x, F32)
    s, b = diag_images(mu, var)
    D = s.shape[0]
    acc = np.zeros(x.shape[1], F32)
    for d in range(D):
        t = _fma_f32(s[d], x[d], b[d])
        acc = _fma_f32(t, t, acc)
    cst = F32(-0.5 * (D * np.log(2 * np.pi) + float(F32(logdet))))
    return (np.float64(cst) - 0.5 * acc.astype(np.float64)).astype(F32)


def diag_suff_stats(points):
    """(N, sum_x[D] f64, sum of x_d^2 [D] f64)."""
    pts = np.asarray(points, np.float64)
    return points.shape[1], pts.sum(axis=1), (pts * pts).sum(axis=1)


class DiagDist:
    """One diagonal Gaussian as the sweep sees it (mu, sigma^2, logdetSigma, Float32)."""
    __slots__ = ("mu", "var", "logdet")

    def __init__(self, mu, var, logdet):
        self.mu = np.asarray(mu, F32)
        self.var = np.asarray(var, F32)
        self.logdet = F32(logdet)

    def log_likelihood(self, x):
        return diag_gaussian_log_likelihood(x, self.mu, self.var, self.logdet)


class DiagOracleSweep(O.OracleSweep):
    """OracleSweep of a diagonal Gaussian context: set_params_diag and the [m][3][D] sum of squares."""

    def __init__(self, x, prior_kind=DIAG, seed=0, global_offset=0):
        assert prior_kind == DIAG
        super().__init__(x, DIAG, seed, global_offset)

    def set_params_diag(self, mu, var, logdet, weights, lr_weights):
        """mu [K,3,D], var [K,3,D], logdet [K,3], weights [K], lr_weights [K,2]."""
        mu = np.asarray(mu, F32); var = np.asarray(var, F32); logdet = np.asarray(logdet, F32)
        self.K = mu.shape[0]
        self.dists = [[DiagDist(mu[k, s], var[k, s], logdet[k, s]) for s in range(3)] for k in range(self.K)]
        self.weights = np.asarray(weights, F32)
        self.lr_weights = np.asarray(lr_weights, F32).reshape(self.K, 2)

    def suff_stats(self, indices=None):
        """Returns (counts[m,3] i64, sum_x[m,3,D] f64, sum_xx[m,3,D] f64)."""
        idx = list(range(1, self.K + 1)) if indices is None else [int(i) for i in indices]
        m = len(idx)
        counts = np.zeros((m, 3), np.int64)
        sum_x = np.zeros((m, 3, self.D))
        sum_xx = np.zeros((m, 3, self.D))
        for a, i in enumerate(idx):
            sel = self.labels == i
            sub = self.sublabels[sel]
            pts = self.x[:, sel]
            for s, p in enumerate((pts, pts[:, sub == 1], pts[:, sub == 2])):
                counts[a, s], sum_x[a, s], sum_xx[a, s] = diag_suff_stats(p)
        return counts, sum_x, sum_xx
