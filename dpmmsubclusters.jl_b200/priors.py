"""Host-side prior plugins (the "small K x D^2 work" that stays on the host, north_star).

Python mirror of the reference's plugin API (docs/src/priors.md:22-78): the same type names, the
same generic functions, Float64 host math.
  niw_hyperparams / niw_sufficient_statistics / mv_gaussian     src/priors/niw.jl, src/distributions/mv_gaussian.jl
  multinomial_hyper / multinomial_sufficient_statistics / multinomial_dist
                                                                src/priors/multinomial_prior.jl, src/distributions/multinomial_dist.jl
  diag_niw_hyperparams / diag_niw_sufficient_statistics / diag_gaussian
      a third plugin of the same shape: every feature an independent NIW at D = 1 (shared kappa and nu, per-feature
      m and psi), each function the NIW one at D = 1 summed or multiplied over the features (vectorised)
Random draws use a numpy Generator (the reference uses Distributions.jl on Base.Random; streams are
not reproducible across the two, only distributions are).
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np
import scipy.sparse as sps
from scipy.special import gammaln

F32 = np.float32


# ---------------------------------------------------------------- NIW ----------------------------
@dataclass
class niw_hyperparams:
    """niw.jl:6-11 (kappa, nu Float32; m, psi Float64)."""
    κ: float
    m: np.ndarray
    ν: float
    ψ: np.ndarray

    def __post_init__(self):
        self.κ = float(F32(self.κ))
        self.ν = float(F32(self.ν))
        self.m = np.asarray(self.m, np.float64).reshape(-1)
        self.ψ = np.asarray(self.ψ, np.float64)


@dataclass
class niw_sufficient_statistics:
    """niw.jl:13-17 (N Float32, points_sum / S Float64)."""
    N: float
    points_sum: np.ndarray
    S: np.ndarray


@dataclass
class mv_gaussian:
    """mv_gaussian.jl:12-18: mu, Sigma, invSigma, logdetSigma are Float32; invChol (upper Cholesky
    factor of invSigma, Float64) is carried but unused by the reference."""
    μ: np.ndarray
    Σ: np.ndarray
    invΣ: np.ndarray
    logdetΣ: float
    invChol: np.ndarray | None = None


@dataclass
class multinomial_hyper:
    """multinomial_prior.jl:6-8."""
    α: np.ndarray

    def __post_init__(self):
        self.α = np.asarray(self.α, F32).reshape(-1)


@dataclass
class multinomial_sufficient_statistics:
    """multinomial_prior.jl:10-13."""
    N: float
    points_sum: np.ndarray


@dataclass
class multinomial_dist:
    """multinomial_dist.jl:8-10: alpha holds LOG-probabilities (Float32)."""
    α: np.ndarray


# ---------------------------------------------------------------- diagonal NIW ------------------
@dataclass
class diag_niw_hyperparams:
    """Per-feature NIW at D = 1: kappa, nu Float32 (as niw_hyperparams); m[D], psi[D] Float64.  psi is scaled by nu
    as in the NIW prior: the inverse-Wishart (here inverse-gamma) scale of feature d is nu * psi_d."""
    κ: float
    m: np.ndarray
    ν: float
    ψ: np.ndarray

    def __post_init__(self):
        self.κ = float(F32(self.κ))
        self.ν = float(F32(self.ν))
        self.m = np.asarray(self.m, np.float64).reshape(-1)
        self.ψ = np.asarray(self.ψ, np.float64).reshape(-1)


@dataclass
class diag_niw_sufficient_statistics:
    """N Float32; points_sum[D] and S_diag[D] = sum of x_d^2 per feature, Float64."""
    N: float
    points_sum: np.ndarray
    S_diag: np.ndarray


@dataclass
class diag_gaussian:
    """mu and the per-feature variances sigma^2 (Float32), logdetSigma = sum_d log sigma^2_d (Float32, as
    mv_gaussian.logdetSigma)."""
    μ: np.ndarray
    σ2: np.ndarray
    logdetΣ: float


def log_multivariate_gamma(x, D):
    """utils.jl:66-72 (accumulates in Float32 like the reference)."""
    vals = gammaln(x + (1 - np.arange(1, D + 1)) / 2)       # one vectorised call; accumulation order as the reference
    res = F32(D * (D - 1) / 4 * np.log(np.pi))
    for v in vals:
        res = F32(res + v)
    return float(res)


def empty_suff_stats(hyper):
    """create_sufficient_statistics(dist, pts::Array{Any,1}) utils.jl:34-36."""
    if isinstance(hyper, niw_hyperparams):
        D = hyper.m.shape[0]
        return niw_sufficient_statistics(0.0, np.zeros(D), np.zeros((D, D)))
    if isinstance(hyper, diag_niw_hyperparams):
        D = hyper.m.shape[0]
        return diag_niw_sufficient_statistics(0.0, np.zeros(D), np.zeros(D))
    return multinomial_sufficient_statistics(0.0, np.zeros(hyper.α.shape[0], F32))


def make_suff_stats(hyper, N, points_sum, S=None):
    """Wrap what dpmm_suff_stats returns into the plugin's statistics type (N is Float32 in the
    reference, niw.jl:14)."""
    if isinstance(hyper, niw_hyperparams):
        return niw_sufficient_statistics(float(F32(N)), np.array(points_sum, np.float64), np.array(S, np.float64))
    if isinstance(hyper, diag_niw_hyperparams):
        return diag_niw_sufficient_statistics(float(F32(N)), np.array(points_sum, np.float64), np.array(S, np.float64))
    return multinomial_sufficient_statistics(float(F32(N)), np.asarray(points_sum).astype(F32))


def calc_posterior(prior, ss):
    """niw.jl:20-31 / multinomial_prior.jl:16-21."""
    if ss.N == 0:
        return prior
    if isinstance(prior, niw_hyperparams):
        κ = prior.κ + ss.N
        ν = prior.ν + ss.N
        m = (prior.m * prior.κ + ss.points_sum) / κ
        ψ = (prior.ν * prior.ψ + prior.κ * np.outer(prior.m, prior.m) - κ * np.outer(m, m) + ss.S) / ν
        ψ = np.triu(ψ) + np.triu(ψ, 1).T          # Matrix(Symmetric(psi)) takes the upper triangle
        ψ = (ψ + ψ.T) / 2
        return niw_hyperparams(κ, m, ν, ψ)
    if isinstance(prior, diag_niw_hyperparams):
        κ = prior.κ + ss.N
        ν = prior.ν + ss.N
        m = (prior.m * prior.κ + ss.points_sum) / κ
        ψ = (prior.ν * prior.ψ + prior.κ * prior.m * prior.m - κ * m * m + ss.S_diag) / ν
        return diag_niw_hyperparams(κ, m, ν, ψ)
    return multinomial_hyper(prior.α + np.asarray(ss.points_sum, F32))


def _inverse_wishart(rng, ν, Ψ):
    """One draw of InverseWishart(nu, Psi) via the Bartlett factor of Wishart(nu, Psi^-1)."""
    D = Ψ.shape[0]
    Lp = np.linalg.cholesky(np.linalg.inv(Ψ))
    A = np.tril(rng.standard_normal((D, D)), -1)
    A[np.diag_indices(D)] = np.sqrt(rng.chisquare(ν - np.arange(D)))
    LA = Lp @ A
    return np.linalg.inv(LA @ LA.T)


def sample_distribution(hyper, rng):
    """niw.jl:34-40 / multinomial_prior.jl:23-25."""
    if isinstance(hyper, niw_hyperparams):
        Σ = _inverse_wishart(rng, hyper.ν, hyper.ν * hyper.ψ)
        Σ = (Σ + Σ.T) / 2
        μ = rng.multivariate_normal(hyper.m, Σ / hyper.κ, method="cholesky")
        invΣ = np.linalg.inv(Σ)
        invΣ = (invΣ + invΣ.T) / 2
        try:
            chol = np.linalg.cholesky(invΣ).T      # upper factor, invSigma = U'U
        except np.linalg.LinAlgError:
            chol = None
        return mv_gaussian(μ.astype(F32), Σ.astype(F32), invΣ.astype(F32), float(F32(np.linalg.slogdet(Σ)[1])), chol)
    if isinstance(hyper, diag_niw_hyperparams):
        # _inverse_wishart at D = 1 is nu psi / chi^2_nu; then mu_d ~ N(m_d, sigma^2_d / kappa)
        σ2 = hyper.ν * hyper.ψ / rng.chisquare(hyper.ν, hyper.ψ.shape[0])
        μ = hyper.m + np.sqrt(σ2 / hyper.κ) * rng.standard_normal(hyper.m.shape[0])
        return diag_gaussian(μ.astype(F32), σ2.astype(F32), float(F32(np.log(σ2).sum())))
    p = rng.dirichlet(hyper.α.astype(np.float64))
    with np.errstate(divide="ignore"):
        return multinomial_dist(np.log(p).astype(F32))


def log_marginal_likelihood(hyper, post, ss):
    """niw.jl:53-62 / multinomial_prior.jl:34-39."""
    if isinstance(hyper, niw_hyperparams):
        D = ss.points_sum.shape[0]
        return (-ss.N * D * 0.5 * np.log(np.pi)
                + log_multivariate_gamma(post.ν / 2, D) - log_multivariate_gamma(hyper.ν / 2, D)
                + (hyper.ν / 2) * (D * np.log(hyper.ν) + np.linalg.slogdet(hyper.ψ)[1])
                - (post.ν / 2) * (D * np.log(post.ν) + np.linalg.slogdet(post.ψ)[1])
                + (D / 2) * np.log(hyper.κ / post.κ))
    if isinstance(hyper, diag_niw_hyperparams):
        D = ss.points_sum.shape[0]
        return (-ss.N * D * 0.5 * np.log(np.pi)
                + D * (log_multivariate_gamma(post.ν / 2, 1) - log_multivariate_gamma(hyper.ν / 2, 1))
                + (hyper.ν / 2) * (D * np.log(hyper.ν) + np.log(hyper.ψ).sum())
                - (post.ν / 2) * (D * np.log(post.ν) + np.log(post.ψ).sum())
                + (D / 2) * np.log(hyper.κ / post.κ))
    a0 = hyper.α.astype(np.float64)
    a1 = post.α.astype(np.float64)
    return float(gammaln(a0.sum()) - gammaln(a1.sum()) + (gammaln(a1) - gammaln(a0)).sum())


def aggregate_suff_stats(a, b):
    """niw.jl:64-66 / multinomial_prior.jl:41-43."""
    if isinstance(a, niw_sufficient_statistics):
        return niw_sufficient_statistics(float(F32(a.N + b.N)), a.points_sum + b.points_sum, a.S + b.S)
    if isinstance(a, diag_niw_sufficient_statistics):
        return diag_niw_sufficient_statistics(float(F32(a.N + b.N)), a.points_sum + b.points_sum, a.S_diag + b.S_diag)
    return multinomial_sufficient_statistics(float(F32(a.N + b.N)), (a.points_sum + b.points_sum).astype(F32))


def posterior_predictive(x, post):
    """posterior_predictive! niw.jl:68-76 (multivariate Student-t log-density) and
    multinomial_prior.jl:45-48.  x is D x n; returns Float64[n].  Host-only (predict).  The diagonal prior's
    predictive is the product over features of the D = 1 Student-t densities (df = nu)."""
    if isinstance(post, diag_niw_hyperparams):
        if sps.issparse(x):
            raise ValueError("sparse points are supported for the multinomial prior only")
        df = post.ν
        sig = ((post.κ + 1) / post.κ) * post.ψ                  # ((kappa + 1) / (kappa df)) nu psi at D = 1
        z = np.asarray(x, np.float64) - post.m[:, None]
        q = z * z / sig[:, None]
        return (post.m.shape[0] * (gammaln((df + 1) / 2) - gammaln(df / 2) - 0.5 * np.log(df * np.pi))
                - 0.5 * np.log(sig).sum() - 0.5 * (df + 1) * np.log1p(q / df).sum(axis=0))
    if isinstance(post, niw_hyperparams):
        if sps.issparse(x):
            raise ValueError("sparse points are supported for the multinomial prior only")
        ν, ψ, κ, m = post.ν, post.ψ, post.κ, post.m
        D = m.shape[0]
        df = ν - D + 1
        Sig = ((κ + 1) / (κ * df)) * ν * ψ
        z = np.asarray(x, np.float64) - m[:, None]
        sol = np.linalg.solve(Sig, z)
        q = np.einsum("ij,ij->j", z, sol)
        return (gammaln((df + D) / 2) - gammaln(df / 2) - 0.5 * D * np.log(df * np.pi)
                - 0.5 * np.linalg.slogdet(Sig)[1] - 0.5 * (df + D) * np.log1p(q / df))
    a = post.α.astype(np.float64)
    if sps.issparse(x):   # zero counts contribute nothing (stored or not), as in the sparse device kernels
        xt = sps.csr_matrix(x.T, dtype=np.float64, copy=True)
        xt.eliminate_zeros()
        return np.asarray(xt @ np.log(a / a.sum())).reshape(-1)
    return np.log(a / a.sum()) @ np.asarray(x, np.float64)
