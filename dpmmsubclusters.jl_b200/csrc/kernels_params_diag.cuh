// Device-side parameter step of the diagonal-covariance Gaussian prior (DPMM_PRIOR_DIAG_GAUSSIAN): the counterpart of
// kernels_params.cuh and kernels_params_mnm.cuh.  An iteration needs the same ONE small device->host copy (3K counts +
// 3K log marginal likelihoods + the merge table); the 3K x D draws and their packing for the sweep stay on the device.
// Every formula is the one of priors.py for diag_niw_hyperparams, i.e. the NIW prior at D = 1 per feature:
//
//   calc_posterior            kappa' = kappa + N, nu' = nu + N, m' = (m kappa + sum x) / kappa',
//                             psi' = (nu psi + kappa m^2 - kappa' m'^2 + sum x^2) / nu'        (Float64, per feature)
//   log_marginal_likelihood   -N D/2 log pi + D (fl32(lgamma(nu'/2)) - fl32(lgamma(nu/2)))
//                             + nu/2 (D log nu + sum log psi) - nu'/2 (D log nu' + sum log psi') + D/2 log(kappa/kappa')
//   sample_distribution       sigma^2_d = nu' psi'_d / chi^2_{nu'},  mu_d = m'_d + sqrt(sigma^2_d / kappa') xi_d
//
// diag_niw_hyperparams keeps kappa' and nu' rounded to Float32 while m' and psi' are computed from the unrounded sums;
// the kernels do the same.  m' and psi' are evaluated operation by operation with the _rn intrinsics, so that no
// product is contracted into an FMA: they carry the same bits as the NumPy prior, which matters for psi' when the
// means lie far from the origin relative to sigma (the terms cancel to a small fraction of their size).
//
//   diag_post_kernel   one CTA per (cluster, {c,l,r}): kappa', nu', N and the log marginal likelihood.  The posterior
//                      row is the scalar [kappa', nu', N, logml] (N at slot 2: dpmm_weights_kernel reads it through
//                      its stride); m' and psi' are not stored, the draw recomputes them from the statistics table at
//                      O(1) per feature.
//   diag_merge_kernel  one CTA per candidate pair (i < j): log marginal likelihood of the summed statistics.
//   diag_draw_kernel   one CTA per distribution, features across the threads: Float32 mu and sigma^2 records and
//                      logdet = fl32(sum_d log sigma^2_d) over the Float32 sigma^2.
//   diag_pack_kernel   s = fl32(1/sqrt(sigma^2)), b = fl32(-s mu), cst = fl32(-(D log 2pi + logdet)/2) from those
//                      records; it also serves dpmm_set_params_diag, so the parameter image is defined here only.
// Randomness: ParamRng keyed by (distribution 0..3K-1, feature); the weights kernel keeps 0xFFFFFE / 0xFFFFFF.  Every
// rank of a multi-GPU run draws identical parameters from identical all-reduced statistics.
#pragma once
#include <cfloat>

#include "common.cuh"
#include "kernels_params.cuh"
#include "kernels_params_mnm.cuh"   // mnm_cta_sum

#define DIAG_HYPER_DOUBLES(D) (4 + 2 * (D))   // kappa, nu, sum log psi, fl32(lgamma(nu/2)) | m[D] | psi[D]
#define DIAG_POST_DOUBLES 4                   // kappa', nu', N, logml
#define DIAG_PARAM_THREADS MNM_PARAM_THREADS
#define DIAG_LOG_PI 1.1447298858494002
#define DIAG_LOG_2PI 1.8378770664093453

// m'_d and psi'_d of feature d from the summed statistics (kp = kappa + N, nup = nu + N unrounded), in the operation
// order of priors.calc_posterior
__device__ __forceinline__ void diag_posterior_feature(const double* hyper, int D, int d, double kp, double nup, double sx,
                                                       double sxx, double& mp, double& psip) {
  const double kappa = hyper[0], nu = hyper[1];
  const double m0 = hyper[4 + d], psi0 = hyper[4 + D + d];
  mp = __ddiv_rn(__dadd_rn(__dmul_rn(m0, kappa), sx), kp);
  const double a = __dadd_rn(__dmul_rn(nu, psi0), __dmul_rn(__dmul_rn(kappa, m0), m0));
  psip = __ddiv_rn(__dadd_rn(__dsub_rn(a, __dmul_rn(__dmul_rn(kp, mp), mp)), sxx), nup);
}

// log marginal likelihood of the statistics (N, sum x, sum x^2) given through `stat(d, sx, sxx)`; 0 for N = 0.  All
// threads of the CTA (DIAG_PARAM_THREADS); every thread gets the result, and kappa', nu' as diag_niw_hyperparams holds
// them (Float32).
template <typename Stat>
__device__ inline double diag_logml_cta(const double* hyper, int D, double N, Stat stat, double* red, double& kp32,
                                        double& nup32) {
  const double kappa = hyper[0], nu = hyper[1];
  if (!(N > 0.0)) {
    kp32 = kappa;
    nup32 = nu;
    return 0.0;
  }
  const double kp = kappa + N, nup = nu + N;
  kp32 = (double)(float)kp;
  nup32 = (double)(float)nup;
  double slp = 0.0;
  for (int d = threadIdx.x; d < D; d += DIAG_PARAM_THREADS) {
    double sx, sxx, mp, psip;
    stat(d, sx, sxx);
    diag_posterior_feature(hyper, D, d, kp, nup, sx, sxx, mp, psip);
    slp += log(psip);
  }
  slp = mnm_cta_sum(slp, red);
  const double lg = (double)(float)lgamma(nup32 / 2.0);   // log_multivariate_gamma(x, 1) rounds to Float32
  return -N * D * 0.5 * DIAG_LOG_PI + D * (lg - hyper[3]) + (nu / 2.0) * (D * log(nu) + hyper[2]) -
         (nup32 / 2.0) * (D * log(nup32) + slp) + (D / 2.0) * log(kappa / kp32);
}

struct DiagPostArgs {
  int D, rec;                // rec = 1 + 2D: N | sum x[D] | sum x^2[D]
  const double* hyper;       // [DIAG_HYPER_DOUBLES(D)]
  const double* hyper0;      // prior of cluster 0 (the outlier component's, or == hyper)
  const double* ptab;        // [K][3][rec]
  const int32_t* idx_list;   // [m] or nullptr (a = k)
  double* post;              // [K][3][DIAG_POST_DOUBLES]
  double* out;               // [m][3][2]: (N, logml) for the host
};

__global__ void __launch_bounds__(DIAG_PARAM_THREADS) diag_post_kernel(const DiagPostArgs a) {
  __shared__ double red[DIAG_PARAM_THREADS / 32];
  const int ai = blockIdx.x, s = blockIdx.y, D = a.D;
  const int k = a.idx_list != nullptr ? a.idx_list[ai] : ai;
  const double* src = a.ptab + ((size_t)k * 3 + s) * a.rec;
  const double N = src[0];
  double kp, nup;
  const double lml = diag_logml_cta(
      k == 0 ? a.hyper0 : a.hyper, D, N,
      [&](int d, double& sx, double& sxx) {
        sx = src[1 + d];
        sxx = src[1 + D + d];
      },
      red, kp, nup);
  if (threadIdx.x == 0) {
    double* P = a.post + ((size_t)k * 3 + s) * DIAG_POST_DOUBLES;
    P[0] = kp; P[1] = nup; P[2] = N; P[3] = lml;
    a.out[((size_t)ai * 3 + s) * 2] = N;
    a.out[((size_t)ai * 3 + s) * 2 + 1] = lml;
  }
}

struct DiagMergeArgs {
  int D, rec, K;
  const double* hyper;
  const double* hyper0;        // as in DiagPostArgs (pairs (0, j))
  const double* ptab;
  const uint8_t* splittable;   // [K]
  double* out;                 // [K][K]: entry (i, j), i < j both splittable and non-empty; NaN elsewhere
};
// grid (K, K); CTAs of pairs that are not candidates return at once
__global__ void __launch_bounds__(DIAG_PARAM_THREADS) diag_merge_kernel(const DiagMergeArgs a) {
  __shared__ double red[DIAG_PARAM_THREADS / 32];
  const int i = blockIdx.y, j = blockIdx.x, D = a.D;
  double* o = a.out + (size_t)i * a.K + j;
  const double* si = a.ptab + (size_t)i * 3 * a.rec;
  const double* sj = a.ptab + (size_t)j * 3 * a.rec;
  if (i >= j || !a.splittable[i] || !a.splittable[j] || !(si[0] > 0.0) || !(sj[0] > 0.0)) {
    if (threadIdx.x == 0) *o = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  // aggregate_suff_stats: the sums of the two cluster records
  double kp, nup;
  const double lml = diag_logml_cta(
      i == 0 ? a.hyper0 : a.hyper, D, si[0] + sj[0],
      [&](int d, double& sx, double& sxx) {
        sx = si[1 + d] + sj[1 + d];
        sxx = si[1 + D + d] + sj[1 + D + d];
      },
      red, kp, nup);
  if (threadIdx.x == 0) *o = lml;
}

struct DiagDrawArgs {
  int D, rec;
  const double* hyper;
  const double* hyper0;      // prior of cluster 0 (distributions t < 3)
  const double* ptab;        // [3K][rec]: m' and psi' are recomputed from the statistics
  const double* post;        // [3K][DIAG_POST_DOUBLES]
  float* mu;                 // [3K][D] out
  float* var;                // [3K][D] out (sigma^2)
  float* logdet;             // [3K] out
  uint64_t seed;
  uint32_t call;
  int first;                 // sample from the prior (init_first_clusters!)
};
// One CTA per distribution t = 3k + s.  A sigma^2 outside the normal Float32 range (a chi^2 draw in the far tail of a
// small nu', or a psi' that cancelled to nothing) is clamped into it: the label kernels' tables stay finite.
__global__ void __launch_bounds__(DIAG_PARAM_THREADS) diag_draw_kernel(const DiagDrawArgs a) {
  __shared__ double red[DIAG_PARAM_THREADS / 32];
  const int t = blockIdx.x, D = a.D;
  const double* P = a.post + (size_t)t * DIAG_POST_DOUBLES;
  const double* S = a.ptab + (size_t)t * a.rec;
  const double* hyper = t < 3 ? a.hyper0 : a.hyper;
  const bool prior = a.first != 0 || !(P[2] > 0.0);
  const double N = prior ? 0.0 : P[2];
  const double kp = hyper[0] + N, nup = hyper[1] + N;       // what m' and psi' are computed with
  const double kd = prior ? hyper[0] : P[0], nd = prior ? hyper[1] : P[1];   // the Float32 kappa', nu'
  double lsum = 0.0;
  for (int d = threadIdx.x; d < D; d += DIAG_PARAM_THREADS) {
    double mp, psip;
    if (prior) {
      mp = hyper[4 + d];
      psip = hyper[4 + D + d];
    } else {
      diag_posterior_feature(hyper, D, d, kp, nup, S[1 + d], S[1 + D + d], mp, psip);
    }
    ParamRng rng(a.seed, a.call, (uint32_t)t, (uint32_t)d);
    const double chi2 = 2.0 * rng.gamma(0.5 * nd);
    const double v = fmin(fmax(nd * psip / chi2, (double)FLT_MIN), (double)FLT_MAX);
    const float vf = (float)v;
    const double m = mp + sqrt(v / kd) * rng.normal();
    a.var[(size_t)t * D + d] = vf;
    a.mu[(size_t)t * D + d] = (float)m;
    lsum += log((double)vf);
  }
  lsum = mnm_cta_sum(lsum, red);
  if (threadIdx.x == 0) a.logdet[t] = (float)lsum;
}

struct DiagPackArgs {
  int D, nrec;               // nrec = 3K distributions
  const float* mu;           // [3K][D]
  const float* var;          // [3K][D]
  const float* logdet;       // [3K]
  float* s;                  // [3K][D] out: the s rows of ctx->recs
  float* b;                  // [3K][D] out: the b rows
  float* cst;                // [3K] out
};
// Float64 sqrt and division are correctly rounded; the products and the sum of cst go through the _rn intrinsics, so
// that nothing is contracted into an FMA.
__global__ void diag_pack_kernel(const DiagPackArgs a) {
  const int64_t ne = (int64_t)a.nrec * a.D;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < ne; e += (int64_t)gridDim.x * blockDim.x) {
    const float sv = (float)__ddiv_rn(1.0, __dsqrt_rn((double)a.var[e]));
    a.s[e] = sv;
    a.b[e] = (float)__dmul_rn(-(double)sv, (double)a.mu[e]);
    if (e < a.nrec)
      a.cst[e] = (float)__dmul_rn(-0.5, __dadd_rn(__dmul_rn((double)a.D, DIAG_LOG_2PI), (double)a.logdet[e]));
  }
}
