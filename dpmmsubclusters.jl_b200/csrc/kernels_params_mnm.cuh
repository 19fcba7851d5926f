// Device-side parameter step and predict of the Dirichlet-multinomial model: the multinomial counterpart of
// kernels_params.cuh.  An iteration needs the same ONE small device->host copy (3K counts + 3K log marginal
// likelihoods + the merge table); the K x D parameter draw and its packing for the sweep stay on the device.
//
//   calc_posterior               src/priors/multinomial_prior.jl:16-21  (alpha' = alpha + points_sum, Float32)
//   create_sufficient_statistics src/priors/multinomial_prior.jl:27-32  (points_sum rounded to Float32)
//   sample_distribution          src/priors/multinomial_prior.jl:23-25  (log of a Dirichlet(alpha') draw)
//   log_marginal_likelihood      src/priors/multinomial_prior.jl:34-39
//   aggregate_suff_stats         src/priors/multinomial_prior.jl:41-43
//   posterior_predictive!        src/priors/multinomial_prior.jl:45-48
//   should_merge!                src/shared_actions.jl:21-38
//   predict_points               src/local_clusters_actions.jl:23-40
//
//   mnm_post_kernel   one CTA per (cluster, {c,l,r}): alpha' and the log marginal likelihood.  The posterior row is
//                     [-, -, N, logml | alpha'[D]], so dpmm_weights_kernel reads N at slot 2 through its stride.
//   mnm_merge_kernel  one CTA per candidate pair (i < j): log marginal likelihood of the summed statistics.
//   mnm_draw_kernel   one CTA per distribution: log p ~ log Dirichlet(alpha') in log space, written as the [3K][D]
//                     Float32 records the sweep kernels read.
//   mnm_pack_kernel   derives the transposed table and the TF32 split of the label kernels from those records; it
//                     also serves dpmm_set_params_multinomial, so the packed layout is defined here only.
//   mnm_score_kernel + mnm_predict_finish_kernel   predict: parr[i,k] = fl32(log p_k' x_i) + log w_k, first argmax,
//                     softmax with NaN -> -Inf.
// Randomness: ParamRng keyed by (distribution 0..3K-1, component), the weights kernel keeps 0xFFFFFE / 0xFFFFFF:
// every rank of a multi-GPU run draws identical parameters from identical all-reduced statistics.
#pragma once
#include "common.cuh"
#include "kernels_mnm_tc.cuh"
#include "kernels_params.cuh"

#define MNM_HYPER_DOUBLES(D) (2 + (D))   // sum alpha, lgamma(sum alpha) | alpha[D]
#define MNM_POST_DOUBLES(D) (4 + (D))    // -, -, N, logml | alpha'[D]
#define MNM_PARAM_THREADS 256
// lowest log-probability a draw may take: a Float32 -Inf would turn 0 * log p into NaN in the label kernels, and
// the three-way TF32 split of -FLT_MAX rounds to -Inf
#define MNM_LOGP_MIN (-1e30)

// sum of one double per thread over the CTA (MNM_PARAM_THREADS threads); every thread gets the result
__device__ inline double mnm_cta_sum(double v, double* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  double s = 0.0;
  for (int i = 0; i < MNM_PARAM_THREADS / 32; ++i) s += red[i];
  return s;
}
__device__ inline double mnm_cta_max(double v, double* red) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
  __syncthreads();
  if (lane == 0) red[w] = v;
  __syncthreads();
  double s = red[0];
  for (int i = 1; i < MNM_PARAM_THREADS / 32; ++i) s = fmax(s, red[i]);
  return s;
}

// log marginal likelihood of alpha' = alpha + fl32(sum x), given the Float32 statistics of each component through
// `stat(d)`; 0 for an empty distribution.  Optionally stores alpha'.  All threads; every thread gets the result.
template <typename Stat>
__device__ inline double mnm_logml_cta(const double* hyper, int D, bool empty, Stat stat, double* alpha_out,
                                       double* red) {
  double sa = 0.0, dl = 0.0;
  for (int d = threadIdx.x; d < D; d += MNM_PARAM_THREADS) {
    const float a0 = (float)hyper[2 + d];
    const float ap = empty ? a0 : __fadd_rn(a0, stat(d));
    if (alpha_out != nullptr) alpha_out[d] = (double)ap;
    sa += (double)ap;
    dl += lgamma((double)ap) - lgamma((double)a0);
  }
  sa = mnm_cta_sum(sa, red);
  dl = mnm_cta_sum(dl, red);
  return empty ? 0.0 : hyper[1] - lgamma(sa) + dl;
}

struct MnmPostArgs {
  int D, rec;
  const double* hyper;       // [MNM_HYPER_DOUBLES]
  const double* ptab;        // [K][3][rec]: N | sum x[D]
  const int32_t* idx_list;   // [m] or nullptr (a = k)
  double* post;              // [K][3][MNM_POST_DOUBLES]
  double* out;               // [m][3][2]: (N, logml) for the host
};

__global__ void __launch_bounds__(MNM_PARAM_THREADS) mnm_post_kernel(const MnmPostArgs a) {
  __shared__ double red[MNM_PARAM_THREADS / 32];
  const int ai = blockIdx.x, s = blockIdx.y, D = a.D;
  const int k = a.idx_list != nullptr ? a.idx_list[ai] : ai;
  const double* src = a.ptab + ((size_t)k * 3 + s) * a.rec;
  double* P = a.post + ((size_t)k * 3 + s) * MNM_POST_DOUBLES(D);
  const double N = src[0];
  const double lml = mnm_logml_cta(a.hyper, D, !(N > 0.0), [&](int d) { return (float)src[1 + d]; }, P + 4, red);
  if (threadIdx.x == 0) {
    P[2] = N;
    P[3] = lml;
    a.out[((size_t)ai * 3 + s) * 2] = N;
    a.out[((size_t)ai * 3 + s) * 2 + 1] = lml;
  }
}

struct MnmMergeArgs {
  int D, rec, K;
  const double* hyper;
  const double* ptab;
  const uint8_t* splittable;   // [K]
  double* out;                 // [K][K]: entry (i, j), i < j both splittable and non-empty; NaN elsewhere
};
// grid (K, K); CTAs of pairs that are not candidates return at once
__global__ void __launch_bounds__(MNM_PARAM_THREADS) mnm_merge_kernel(const MnmMergeArgs a) {
  __shared__ double red[MNM_PARAM_THREADS / 32];
  const int i = blockIdx.y, j = blockIdx.x;
  double* o = a.out + (size_t)i * a.K + j;
  const double* si = a.ptab + (size_t)i * 3 * a.rec;
  const double* sj = a.ptab + (size_t)j * 3 * a.rec;
  if (i >= j || !a.splittable[i] || !a.splittable[j] || !(si[0] > 0.0) || !(sj[0] > 0.0)) {
    if (threadIdx.x == 0) *o = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  // aggregate_suff_stats adds the two Float32 statistics in Float32
  const double lml = mnm_logml_cta(a.hyper, a.D, false,
                                   [&](int d) { return __fadd_rn((float)si[1 + d], (float)sj[1 + d]); }, nullptr, red);
  if (threadIdx.x == 0) *o = lml;
}

// log of a Gamma(a, 1) variate; a < 1 through log Gamma(a + 1) + log(U) / a, which stays finite where U^(1/a) would
// underflow
__device__ inline double mnm_log_gamma(ParamRng& rng, double a) {
  if (a >= 1.0) return log(rng.gamma(a));
  const double lu = log(rng.uniform());
  return log(rng.gamma(a + 1.0)) + lu / a;
}

struct MnmDrawArgs {
  int D;
  const double* hyper;
  const double* post;        // [3K][MNM_POST_DOUBLES]
  float* logp;               // [3K][D] out
  uint64_t seed;
  uint32_t call;
  int first;                 // sample from the prior (init_first_clusters!)
};
// One CTA per distribution t = 3k + s.
__global__ void __launch_bounds__(MNM_PARAM_THREADS) mnm_draw_kernel(const MnmDrawArgs a) {
  extern __shared__ double lg[];   // [D]
  __shared__ double red[MNM_PARAM_THREADS / 32];
  const int t = blockIdx.x, D = a.D;
  const double* P = a.post + (size_t)t * MNM_POST_DOUBLES(D);
  const double* alpha = (a.first != 0 || !(P[2] > 0.0)) ? a.hyper + 2 : P + 4;
  double mx = -CUDART_INF;
  for (int d = threadIdx.x; d < D; d += MNM_PARAM_THREADS) {
    ParamRng rng(a.seed, a.call, (uint32_t)t, (uint32_t)d);
    lg[d] = mnm_log_gamma(rng, alpha[d]);
    mx = fmax(mx, lg[d]);
  }
  mx = mnm_cta_max(mx, red);
  double se = 0.0;
  for (int d = threadIdx.x; d < D; d += MNM_PARAM_THREADS) se += exp(lg[d] - mx);
  const double lse = mx + log(mnm_cta_sum(se, red));
  for (int d = threadIdx.x; d < D; d += MNM_PARAM_THREADS)
    a.logp[(size_t)t * D + d] = (float)fmax(lg[d] - lse, MNM_LOGP_MIN);
}

// alpha = hi + lo + lolo with every term exact in TF32 (10 explicit mantissa bits, round to nearest even)
__device__ inline float mnm_tf32(float v) {
  if (!isfinite(v)) return v;
  uint32_t u = __float_as_uint(v);
  u += 0xFFFu + ((u >> 13) & 1u);
  u &= 0xFFFFE000u;
  return __uint_as_float(u);
}

struct MnmPackArgs {
  int D, K, KP;
  const float* logp;   // [3K][D] (ctx->recs)
  float* logp_t;       // [D][KP] cluster distributions transposed, zero past K
  float* mtc_w;        // [3][NP][MTC_N][32] or nullptr: hi / lo / lolo of the cluster distributions, zero padded
};
__global__ void mnm_pack_kernel(const MnmPackArgs a) {
  const int D = a.D, K = a.K, KP = a.KP, NP = (D + 31) / 32;
  const int64_t nt = (int64_t)D * KP;
  const int64_t nw = a.mtc_w != nullptr ? (int64_t)NP * MTC_N * 32 : 0;
  const int64_t ne = nt > nw ? nt : nw;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < ne; e += (int64_t)gridDim.x * blockDim.x) {
    if (e < nt) {
      const int d = (int)(e / KP), k = (int)(e % KP);
      a.logp_t[e] = k < K ? a.logp[(size_t)(3 * k) * D + d] : 0.f;
    }
    if (e < nw) {
      const int c = (int)(e & 31), k = (int)((e >> 5) % MTC_N), p = (int)((e >> 5) / MTC_N), d = p * 32 + c;
      float hi = 0.f, lo = 0.f, lolo = 0.f;
      if (k < K && d < D) {
        const float al = a.logp[(size_t)(3 * k) * D + d];
        hi = mnm_tf32(al);
        const float r1 = isfinite(al) ? __fsub_rn(al, hi) : 0.f;
        lo = mnm_tf32(r1);
        lolo = __fsub_rn(r1, lo);
      }
      a.mtc_w[e] = hi;
      a.mtc_w[nw + e] = lo;
      a.mtc_w[2 * nw + e] = lolo;
    }
  }
}

// ---- predict ----------------------------------------------------------------------------------------------------
struct MnmScoreArgs {
  const float* x;       // [n][D]
  int64_t n;
  int D, K, KC;         // KC clusters per tile (blockIdx.y)
  const double* logp;   // [K][D] log(alpha' / sum alpha') in Float64
  const float* logw;    // [K]
  float* score;         // [n][K] out
};
// One warp per point, lanes over the features: the dot product accumulates in Float64, is rounded to Float32 and
// gets log w in Float32, as the NumPy formula does.  The CTA keeps its tile of KC clusters in shared memory.
__global__ void __launch_bounds__(256) mnm_score_kernel(const MnmScoreArgs a) {
  extern __shared__ double tile[];   // [KC][D]
  const int D = a.D, k0 = blockIdx.y * a.KC, kc = min(a.KC, a.K - k0);
  for (int e = threadIdx.x; e < kc * D; e += blockDim.x) tile[e] = a.logp[(size_t)k0 * D + e];
  __syncthreads();
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
  for (int64_t i = (int64_t)blockIdx.x * 8 + wl; i < a.n; i += (int64_t)gridDim.x * 8) {
    const float* xi = a.x + (size_t)i * D;
    for (int k = 0; k < kc; ++k) {
      const double* lp = tile + (size_t)k * D;
      double s = 0.0;
      for (int d = lane; d < D; d += 32) s = fma((double)__ldg(xi + d), lp[d], s);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) a.score[(size_t)i * a.K + k0 + k] = __fadd_rn((float)s, __ldg(a.logw + k0 + k));
    }
  }
}

// first argmax of each row (NaN counts as maximal), then the row's softmax in place when `probs` is wanted
__global__ void mnm_predict_finish_kernel(float* score, int64_t n, int K, int32_t* labels, int probs) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float* r = score + (size_t)i * K;
    labels[i] = dpmm_draw_argmax(r, 1, K);
    if (!probs) continue;
    float mx = -CUDART_INF_F;
    for (int k = 0; k < K; ++k) {
      if (r[k] != r[k]) r[k] = -CUDART_INF_F;
      mx = fmaxf(mx, r[k]);
    }
    float s = 0.f;
    for (int k = 0; k < K; ++k) {
      r[k] = expf(r[k] - mx);
      s += r[k];
    }
    for (int k = 0; k < K; ++k) r[k] /= s;
  }
}
