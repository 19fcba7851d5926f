// Device-side parameter step of the NIW model (SURVEY.md 8f-1): the per-iteration master work of the
// reference that scales with K D^3 moves next to the statistics it consumes, so an iteration needs ONE
// small device->host copy (3K counts + 3K log marginal likelihoods + the merge table).
//
//   calc_posterior               src/priors/niw.jl:20-31
//   log_marginal_likelihood      src/priors/niw.jl:53-62   (log_multivariate_gamma: src/utils.jl:66-72)
//   sample_distribution          src/priors/niw.jl:34-40
//   sample_cluster_params        src/shared_actions.jl:41-66      (lr_weights: Dirichlet(N_l + a/2, N_r + a/2))
//   sample_clusters!             src/local_clusters_actions.jl:417-437 (weights: Dirichlet(N_1..N_K, a))
//   should_merge!                src/shared_actions.jl:21-38      (posterior + log marginal of the summed statistics)
//
// Designed from the formulas (SURVEY appendix B), not from the host code:
//   niw_post_kernel   one CTA per (cluster, {c,l,r}): posterior (kappa', nu', m', psi'), the Cholesky factor of
//                     psi' in REVERSED index order and the log marginal likelihood.
//   niw_draw_kernel   one CTA per distribution: Sigma ~ InverseWishart(nu', nu' psi') as a Bartlett draw arranged so
//                     that invSigma = L L' comes out with L LOWER triangular directly (no inversion of a sampled
//                     matrix, no second factorisation): with psi' = V V', V upper (that is what the reversed
//                     Cholesky gives), M = V^-T / sqrt(nu') is lower, and for a lower Bartlett factor B
//                     (B_ii^2 ~ chi^2_{nu'-i}, B_ij ~ N(0,1)) invSigma = (M B)(M B)' ~ Wishart(nu', (nu' psi')^-1).
//                     mu = m' + L^-T xi / sqrt(kappa'),  logdet Sigma = -2 sum log L_ii.  niw_pack_kernel then
//                     packs from that factor (its Cholesky step is skipped).
//   niw_merge_kernel  one CTA per candidate pair (i < j): log marginal likelihood of the summed statistics.
//   dpmm_weights_kernel  mixture weights and sub-cluster weights (Gamma draws), written as the Float32 logs
//                     the sweep kernels read.
// Randomness: Philox4x32-10 keyed by (seed, stream PARAMS, parameter-call counter, distribution, variate,
// attempt): every rank of a multi-GPU run draws identical parameters from identical all-reduced statistics.
#pragma once
#include "common.cuh"
#include "kernels_pack.cuh"

#define DPMM_STREAM_PARAMS 5u
#define NIW_HYPER_DOUBLES(D) (4 + (D) + (D) * (D))          // kappa, nu, logdet psi, lmvgamma(nu/2) | m | psi
#define NIW_POST_DOUBLES(D) (8 + (D) + (D) * (D))           // kappa', nu', N, logml, logdet psi', ok, -, - | m' | Lhat

// ---- random variates -----------------------------------------------------------------------------
struct ParamRng {
  uint64_t seed, base;
  uint32_t call, ctr;
  __device__ ParamRng(uint64_t seed_, uint32_t call_, uint32_t dist, uint32_t variate)
      : seed(seed_), base(((uint64_t)dist << 40) | ((uint64_t)variate << 16)), call(call_), ctr(0) {}
  __device__ Philox4 next() { return philox_draw(seed, DPMM_STREAM_PARAMS, call, base + (ctr++)); }
  __device__ double uniform() {   // (0, 1)
    const Philox4 r = next();
    return ((double)(r.x >> 5) * 67108864.0 + (double)(r.y >> 6) + 0.5) * (1.0 / 9007199254740992.0);
  }
  __device__ double normal() {
    const Philox4 r = next();
    // Box-Muller in Float32 on 32-bit uniforms (|z| <= 6.7): the variates feed Float32 parameters anyway, and a
    // CTA draws ~D^2/2 of them on its critical path
    const float u1 = ((float)(r.x >> 8) + 0.5f) * (1.0f / 16777216.0f);
    const float u2 = ((float)(r.z >> 8) + 0.5f) * (1.0f / 16777216.0f);
    return (double)(sqrtf(-2.0f * __logf(u1)) * cospif(2.0f * u2));
  }
  // Gamma(a, 1), Marsaglia & Tsang (2000); a < 1 through Gamma(a + 1) U^(1/a)
  __device__ double gamma(double a) {
    double boost = 1.0;
    if (a < 1.0) {
      boost = exp(log(uniform()) / a);
      a += 1.0;
    }
    const double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    for (int it = 0; it < 64; ++it) {
      const double x = normal();
      double v = 1.0 + c * x;
      if (v <= 0.0) continue;
      v = v * v * v;
      const double u = uniform();
      if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) return d * v * boost;
    }
    return d * boost;   // (probability ~ 1e-30)
  }
};

// log_multivariate_gamma(x, D) with the reference's Float32 accumulation (utils.jl:66-72); one thread
__device__ inline double niw_lmvgamma(double x, int D) {
  float res = (float)((double)D * (D - 1) / 4.0 * 1.1447298858494002);   // log(pi)
  for (int j = 1; j <= D; ++j) res = (float)((double)res + lgamma(x + (1.0 - j) / 2.0));
  return (double)res;
}

// In-place Cholesky A = L L' (lower) of the matrix in shared memory A[D][LD], all threads of the CTA.
// Returns false when a pivot is not positive and finite.
__device__ inline bool cta_cholesky(double* A, int D, int LD) {
  const int tid = threadIdx.x, NT = blockDim.x;
  const int ty = tid >> 4, tx = tid & 15, NY = NT >> 4;   // 16 x (NT / 16) thread tile of the trailing update
  bool ok = true;
  for (int j = 0; j < D; ++j) {
    const double d = A[j * LD + j];
    ok = ok && (d > 0.0) && (d < CUDART_INF);
    const double ljj = sqrt(d), rl = 1.0 / ljj;
    __syncthreads();
    if (tid == 0) A[j * LD + j] = ljj;
    for (int i = j + 1 + tid; i < D; i += NT) A[i * LD + j] *= rl;
    __syncthreads();
    // trailing update of the lower triangle: element (i, k), j < k <= i < D
    for (int i = j + 1 + ty; i < D; i += NY) {
      const double lij = A[i * LD + j];
      for (int k = j + 1 + tx; k <= i; k += 16) A[i * LD + k] -= lij * A[k * LD + j];
    }
    __syncthreads();
  }
  return ok;
}

// Posterior of the statistics (N, sx, S) = sum over `nsrc` source records, written into shared memory:
// A[D][LD] <- psi' (index-reversed when `reversed`), mp[D] <- m'.  Returns kappa', nu' through pointers.
__device__ inline void niw_posterior_to_smem(const double* hyper, int D, int LD, const double* const* src, int nsrc,
                                             bool reversed, double* A, double* mp, double* sxs, double& N,
                                             double& kp, double& nup) {
  const int tid = threadIdx.x, NT = blockDim.x;
  const double kappa = hyper[0], nu = hyper[1];
  const double* m0 = hyper + 4;
  const double* psi = hyper + 4 + D;
  N = 0.0;
  for (int q = 0; q < nsrc; ++q) N += src[q][0];
  kp = kappa + N;
  nup = nu + N;
  for (int i = tid; i < D; i += NT) {
    double sx = 0.0;
    for (int q = 0; q < nsrc; ++q) sx += src[q][1 + i];
    sxs[i] = sx;
    mp[i] = (N > 0.0) ? (kappa * m0[i] + sx) / kp : m0[i];
  }
  __syncthreads();
  for (int e = tid; e < D * D; e += NT) {
    const int i = e / D, j = e - i * D;
    double v;
    if (N > 0.0) {
      double S = 0.0;
      for (int q = 0; q < nsrc; ++q) S += 0.5 * (src[q][1 + D + e] + src[q][1 + D + j * D + i]);
      v = (nu * 0.5 * (psi[e] + psi[j * D + i]) + kappa * m0[i] * m0[j] - kp * mp[i] * mp[j] + S) / nup;
    } else {
      v = 0.5 * (psi[e] + psi[j * D + i]);
    }
    const int ii = reversed ? D - 1 - i : i, jj = reversed ? D - 1 - j : j;
    A[ii * LD + jj] = v;
  }
  __syncthreads();
}

// log marginal likelihood (niw.jl:53-62) from the Cholesky factor in A.  Called by EVERY thread of the CTA (the D
// logarithms and the D log-gamma values are evaluated by D threads, not by one: they are the kernel's critical
// path); thread 0 holds the result.  log_multivariate_gamma keeps the reference's Float32 accumulation order.
__device__ inline double niw_logml_cta(const double* hyper, int D, int LD, const double* A, double N, double kp, double nup,
                                       double* scratch, double& logdet) {
  const int tid = threadIdx.x;
  __syncthreads();
  if (tid < D) scratch[tid] = log(A[tid * LD + tid]);
  __syncthreads();
  logdet = 0.0;
  if (tid == 0)
    for (int i = 0; i < D; ++i) logdet += 2.0 * scratch[i];
  __syncthreads();
  if (tid < D) scratch[tid] = lgamma(nup / 2.0 + (1.0 - (tid + 1)) / 2.0);
  __syncthreads();
  if (tid != 0 || !(N > 0.0)) return 0.0;   // N = 0: posterior == prior, every term cancels
  float lmv = (float)((double)D * (D - 1) / 4.0 * 1.1447298858494002);   // log(pi); utils.jl:66-72
  for (int j = 0; j < D; ++j) lmv = (float)((double)lmv + scratch[j]);
  const double kappa = hyper[0], nu = hyper[1], logdet0 = hyper[2], lmv0 = hyper[3];
  return -N * D * 0.5 * 1.1447298858494002 + (double)lmv - lmv0 + (nu / 2.0) * (D * log(nu) + logdet0) -
         (nup / 2.0) * (D * log(nup) + logdet) + (D / 2.0) * log(kappa / kp);
}

struct NiwPostArgs {
  int D, rec;
  const double* hyper;
  const double* ptab;        // [K][3][rec]
  const int32_t* idx_list;   // [m] or nullptr (a = k)
  double* post;              // [K][3][NIW_POST_DOUBLES]
  double* out;               // [m][3][2]: (N, logml) for the host
};

__global__ void __launch_bounds__(256) niw_post_kernel(const NiwPostArgs a) {
  extern __shared__ double ps[];
  const int D = a.D, LD = D + 1;
  double* A = ps;
  double* mp = A + D * LD;
  double* sxs = mp + D;
  const int ai = blockIdx.x, s = blockIdx.y;
  const int k = a.idx_list != nullptr ? a.idx_list[ai] : ai;
  const double* src[1] = {a.ptab + ((size_t)k * 3 + s) * a.rec};
  double N, kp, nup;
  niw_posterior_to_smem(a.hyper, D, LD, src, 1, true, A, mp, sxs, N, kp, nup);
  const bool ok = cta_cholesky(A, D, LD);
  double* P = a.post + ((size_t)k * 3 + s) * NIW_POST_DOUBLES(D);
  for (int e = threadIdx.x; e < D * D; e += blockDim.x) P[8 + D + e] = A[(e / D) * LD + (e % D)];
  for (int i = threadIdx.x; i < D; i += blockDim.x) P[8 + i] = mp[i];
  double logdet;
  double lml = niw_logml_cta(a.hyper, D, LD, A, N, kp, nup, sxs, logdet);
  if (threadIdx.x == 0) {
    if (!ok) lml = __longlong_as_double(0x7ff8000000000000LL);
    P[0] = kp; P[1] = nup; P[2] = N; P[3] = lml; P[4] = logdet; P[5] = ok ? 1.0 : 0.0;
    a.out[((size_t)ai * 3 + s) * 2] = N;
    a.out[((size_t)ai * 3 + s) * 2 + 1] = lml;
  }
}

struct NiwMergeArgs {
  int D, rec, K;
  const double* hyper;
  const double* ptab;
  const uint8_t* splittable;   // [K]
  double* out;                 // [K][K]: entry (i, j), i < j both splittable and non-empty; NaN elsewhere
};
// grid (K, K); CTAs of pairs that are not candidates return at once
__global__ void __launch_bounds__(256) niw_merge_kernel(const NiwMergeArgs a) {
  extern __shared__ double ps[];
  const int i = blockIdx.y, j = blockIdx.x;
  if (i >= j) {
    if (threadIdx.x == 0) a.out[(size_t)i * a.K + j] = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  const int D = a.D, LD = D + 1;
  const double* si = a.ptab + (size_t)i * 3 * a.rec;
  const double* sj = a.ptab + (size_t)j * 3 * a.rec;
  double* o = a.out + (size_t)i * a.K + j;
  if (!a.splittable[i] || !a.splittable[j] || !(si[0] > 0.0) || !(sj[0] > 0.0)) {
    if (threadIdx.x == 0) *o = __longlong_as_double(0x7ff8000000000000LL);
    return;
  }
  double* A = ps;
  double* mp = A + D * LD;
  double* sxs = mp + D;
  const double* src[2] = {si, sj};
  double N, kp, nup;
  niw_posterior_to_smem(a.hyper, D, LD, src, 2, false, A, mp, sxs, N, kp, nup);
  const bool ok = cta_cholesky(A, D, LD);
  double logdet;
  const double lml = niw_logml_cta(a.hyper, D, LD, A, N, kp, nup, sxs, logdet);
  if (threadIdx.x == 0) *o = ok ? lml : __longlong_as_double(0x7ff8000000000000LL);
}

struct NiwDrawArgs {
  int D;
  float* mu;                 // [3K][D] out
  float* logdet;             // [3K] out
  const double* hyper;
  const double* post;        // [K][3][NIW_POST_DOUBLES]
  double* lfac;              // [3K][D][D] out: L (invSigma = L L'), row-major: input of niw_pack_kernel
  uint64_t seed;
  uint32_t call;
  int first;                 // sample from the prior (init_first_clusters!: sample_clusters!(group, first) semantics)
};

// One CTA of NIW_PACK_THREADS per distribution t = 3k + s.
__global__ void __launch_bounds__(NIW_PACK_THREADS) niw_draw_kernel(const NiwDrawArgs a) {
  extern __shared__ double Ls[];   // [D][LD] L | Wk [D][LD] | Bm [D][LD] | xi [D] | y [D]
  const int D = a.D, LD = D + 1;
  double* Wk = Ls + D * LD;
  double* Bm = Wk + D * LD;
  double* xi = Bm + D * LD;
  double* y = xi + D;
  const int t = blockIdx.x, tid = threadIdx.x, NT = NIW_PACK_THREADS;
  const double* P = a.post + (size_t)t * NIW_POST_DOUBLES(D);
  const bool prior = a.first != 0 || !(P[2] > 0.0);
  double kp, nup;
  const double* mpost;
  if (prior) {
    // factor of the prior psi in reversed order
    kp = a.hyper[0];
    nup = a.hyper[1];
    mpost = a.hyper + 4;
    const double* psi = a.hyper + 4 + D;
    for (int e = tid; e < D * D; e += NT) {
      const int i = e / D, j = e - i * D;
      Wk[(D - 1 - i) * LD + (D - 1 - j)] = 0.5 * (psi[e] + psi[j * D + i]);
    }
    __syncthreads();
    cta_cholesky(Wk, D, LD);
  } else {
    kp = P[0];
    nup = P[1];
    mpost = P + 8;
    for (int e = tid; e < D * D; e += NT) Wk[(e / D) * LD + (e % D)] = P[8 + D + e];
    __syncthreads();
  }
  // ---- Bartlett factor B (lower) and the normals of the mean.  The D chi-square draws (rejection loops in
  //      Float64) go to the lanes of the last warp(s) together, so that no other warp diverges into them ----
  for (int e = tid; e < D * D + D; e += NT) {
    if (e >= D * D) {
      ParamRng rng(a.seed, a.call, (uint32_t)t, (uint32_t)e);
      xi[e - D * D] = rng.normal();
    } else {
      const int i = e / D, j = e - i * D;
      if (i != j) {
        ParamRng rng(a.seed, a.call, (uint32_t)t, (uint32_t)e);
        Bm[i * LD + j] = i > j ? rng.normal() : 0.0;
      }
    }
  }
  for (int i = NT - 1 - tid; i < D; i += NT) {
    ParamRng rng(a.seed, a.call, (uint32_t)t, (uint32_t)(i * D + i));
    Bm[i * LD + i] = sqrt(2.0 * rng.gamma(0.5 * (nup - i)));
  }
  __syncthreads();
  // ---- L = M B with M = V^-T / sqrt(nu'), V = P Lhat P:  Lhat' X = P B / sqrt(nu'),  X = P L.
  //      Back substitution over the rows of the upper-triangular Lhat' in its column-oriented form (once x_i is
  //      final, every row k < i of the right-hand side loses Lhat[i][k] x_i).
  //      Every column j of X is an independent triangular system: a warp takes four of them at a time, lane <->
  //      row (rows k and k + 32), and walks the rows from the last one up; x_i is broadcast with a shuffle, the
  //      updates r_k -= Lhat[i][k] x_i need no barrier.  The rows of X land row-reversed in Ls, i.e. as L. ----
  const double rs = 1.0 / sqrt(nup);
  for (int i = tid; i < D; i += NT) y[i] = 1.0 / Wk[i * LD + i];   // reciprocal pivots (y is free until the mean)
  __syncthreads();
  {
    const int warp = tid >> 5, lane = tid & 31, NW = NT >> 5;
    for (int jb = warp * 4; jb < D; jb += NW * 4) {
      double r0[4], r1[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int j = jb + q;
        r0[q] = (j < D && lane < D) ? Bm[(D - 1 - lane) * LD + j] * rs : 0.0;
        r1[q] = (j < D && lane + 32 < D) ? Bm[(D - 1 - lane - 32) * LD + j] * rs : 0.0;
      }
      for (int i = D - 1; i >= 0; --i) {
        const double rd = y[i];
        const int src = i & 31;
        const double l0 = lane < i ? Wk[i * LD + lane] : 0.0;
        const double l1 = lane + 32 < i ? Wk[i * LD + lane + 32] : 0.0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const double xq = __shfl_sync(0xffffffffu, (i >= 32 ? r1[q] : r0[q]) * rd, src);
          if (lane == src && jb + q < D) Ls[(D - 1 - i) * LD + jb + q] = xq;
          r0[q] -= l0 * xq;
          r1[q] -= l1 * xq;
        }
      }
    }
  }
  __syncthreads();
  __shared__ int ok_s;
  if (tid == 0) ok_s = 1;
  __syncthreads();
  for (int e = tid; e < D * D; e += NT) {
    const int i = e / D, j = e - i * D;
    const double v = j <= i ? Ls[i * LD + j] : 0.0;          // (entries above the diagonal are rounding residue)
    if (!(fabs(v) < CUDART_INF) || (i == j && !(v > 0.0))) ok_s = 0;
    a.lfac[(size_t)t * D * D + e] = v;
  }
  __syncthreads();
  // ---- the mean: L' y = xi, column-oriented back substitution by warp 0 (lane <-> unknowns k, k + 32);
  //      logdet Sigma = -2 sum log L_ii with the D logarithms taken in parallel ----
  if (tid < 32) {
    const int lane = tid;
    double r0 = lane < D ? xi[lane] : 0.0, r1 = lane + 32 < D ? xi[lane + 32] : 0.0;
    double lg = 0.0;
    for (int i = lane; i < D; i += 32) lg += log(Ls[i * LD + i]);
    const double d0 = lane < D ? 1.0 / Ls[lane * LD + lane] : 0.0, d1 = lane + 32 < D ? 1.0 / Ls[(lane + 32) * LD + lane + 32] : 0.0;
    double y0 = 0.0, y1 = 0.0;
    for (int i = D - 1; i >= 0; --i) {
      const double mine = i >= 32 ? r1 * d1 : r0 * d0;
      const double yi = __shfl_sync(0xffffffffu, mine, i & 31);
      if (lane == (i & 31)) {
        if (i >= 32) y1 = yi; else y0 = yi;
      }
      // r_k -= L[i][k] y_i for k < i
      if (lane < i) r0 -= Ls[i * LD + lane] * yi;
      if (lane + 32 < i) r1 -= Ls[i * LD + lane + 32] * yi;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lg += __shfl_xor_sync(0xffffffffu, lg, o);
    __syncwarp();
    const bool okk = ok_s != 0;
    const double rk = 1.0 / sqrt(kp);
    if (lane < D) a.mu[(size_t)t * D + lane] = (float)(mpost[lane] + y0 * rk);
    if (lane + 32 < D) a.mu[(size_t)t * D + lane + 32] = (float)(mpost[lane + 32] + y1 * rk);
    if (lane == 0) a.logdet[t] = okk ? (float)(-2.0 * lg) : __int_as_float(0x7fc00000);
  }
}

struct WeightsArgs {
  int K, D;
  const double* post;     // N of (k, s) at post[(3k+s) * stride + 2]
  int stride;
  double alpha;
  float* logw;            // [K]
  float* loglr;           // [2K]
  float* w_out;           // [K] the Float32 weights themselves (host read-back)
  float* lr_out;          // [2K]
  uint64_t seed;
  uint32_t call;
  int unit;               // 1: weights = 1/K (init_first_clusters!, dp-parallel-sampling.jl:77), lr = (0.5, 0.5)... see host
};
// sample_clusters! :430-436 and sample_cluster_params shared_actions.jl:46-49.  One CTA.
__global__ void __launch_bounds__(256) dpmm_weights_kernel(const WeightsArgs a) {
  extern __shared__ double gs[];   // [K + 1]
  const int K = a.K, tid = threadIdx.x;
  for (int k = tid; k <= K; k += blockDim.x) {
    ParamRng rng(a.seed, a.call, 0xFFFFFFu, (uint32_t)k);
    const double shape = k < K ? fmax(a.post[(size_t)(3 * k) * a.stride + 2], 1e-300) : a.alpha;
    gs[k] = rng.gamma(shape);
  }
  for (int k = tid; k < K; k += blockDim.x) {
    ParamRng rng(a.seed, a.call, 0xFFFFFEu, (uint32_t)k);
    const double gl = rng.gamma(a.post[(size_t)(3 * k + 1) * a.stride + 2] + 0.5 * a.alpha);
    const double gr = rng.gamma(a.post[(size_t)(3 * k + 2) * a.stride + 2] + 0.5 * a.alpha);
    const float l = (float)(gl / (gl + gr)), r = (float)(gr / (gl + gr));
    a.lr_out[2 * k] = l;
    a.lr_out[2 * k + 1] = r;
    a.loglr[2 * k] = (float)log((double)l);
    a.loglr[2 * k + 1] = (float)log((double)r);
  }
  __syncthreads();
  __shared__ double tot;
  if (tid == 0) {
    double s = 0.0;
    for (int k = 0; k <= K; ++k) s += gs[k];
    tot = s;
  }
  __syncthreads();
  for (int k = tid; k < K; k += blockDim.x) {
    const float w = a.unit ? (float)(1.0 / K) : (float)(gs[k] / tot);
    a.w_out[k] = w;
    a.logw[k] = (float)log((double)w);
  }
}

// ptab[idx[a]][s][:] <- outbuf[a][s][:]   (the result of one statistics call into the persistent table)
__global__ void ptab_scatter_kernel(const double* __restrict__ outbuf, const int32_t* __restrict__ idx_list, int m, int rec3,
                                    double* __restrict__ ptab) {
  const int ai = blockIdx.y;
  const int k = idx_list != nullptr ? idx_list[ai] : ai;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < rec3; e += gridDim.x * blockDim.x)
    ptab[(size_t)k * rec3 + e] = outbuf[(size_t)ai * rec3 + e];
}
// dst[new_of[k]] <- src[k] for kept rows (compaction after remove_empty / relabel of tables)
__global__ void table_gather_kernel(const double* __restrict__ src, const int32_t* __restrict__ new_of, int K, int row,
                                    double* __restrict__ dst) {
  const int k = blockIdx.y;
  const int nk = new_of[k];
  if (nk < 0) return;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < row; e += gridDim.x * blockDim.x)
    dst[(size_t)nk * row + e] = src[(size_t)k * row + e];
}
// merge_clusters_to_splittable (shared_actions.jl:12-18) on the tables: cluster i <- {c: c_i + c_j, l: c_i, r: c_j},
// cluster j <- empty.  One CTA.
__global__ void ptab_merge_kernel(double* ptab, int rec, int i, int j) {
  double* pi = ptab + (size_t)i * 3 * rec;
  double* pj = ptab + (size_t)j * 3 * rec;
  for (int e = threadIdx.x; e < rec; e += blockDim.x) {
    const double ci = pi[e], cj = pj[e];
    pi[e] = ci + cj;
    pi[rec + e] = ci;
    pi[2 * rec + e] = cj;
    pj[e] = 0.0;
    pj[rec + e] = 0.0;
    pj[2 * rec + e] = 0.0;
  }
}

// ------------------------------------------------------------------------------------------------
// predict / predict_points (src/dp-parallel-sampling.jl:509-537, src/local_clusters_actions.jl:23-40) with the
// NIW posterior predictive (multivariate Student-t, src/priors/niw.jl:68-76) on the device:
//   parr[i, k] = C_k - (df_k + D)/2 * log1p(q_ik / df_k) + log w_k,   q = |U_k (x_i - m_k)|^2,
// U_k the upper factor of the inverse scale matrix (((kappa+1)/(kappa df)) nu psi)^-1, prepared by the host from
// the K posterior hyper-parameters (K D^3 work); labels = first argmax over k; optional probabilities
// (NaN -> -Inf, softmax over k) as the reference returns them.  One warp per point, lanes <-> clusters.
// ------------------------------------------------------------------------------------------------
struct NiwPredictArgs {
  const float* x;       // [n][D]
  int64_t n;
  int D, K;
  int D_true;           // the caller's feature dimension (D may be zero-padded): the exponent is (df + D_true)/2
  const float* u;       // [K][D][D] rows of U_k (zero below the diagonal)
  const float* mu;      // [K][D]
  const float* tconst;  // [K]  C_k + log w_k
  const float* df;      // [K]
  int32_t* labels;      // [n] out, 0-based
  float* probs;         // [n][K] out (point-major) or nullptr
};

__global__ void __launch_bounds__(256) niw_predict_kernel(const NiwPredictArgs a) {
  extern __shared__ float pr_sm[];   // per warp: x[D] | r[K]
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5, D = a.D, K = a.K;
  float* xs = pr_sm + (size_t)wl * (D + K);
  float* rs = xs + D;
  for (int64_t i = (int64_t)blockIdx.x * 8 + wl; i < a.n; i += (int64_t)gridDim.x * 8) {
    for (int j = lane; j < D; j += 32) xs[j] = a.x[(size_t)i * D + j];
    __syncwarp();
    for (int k = lane; k < K; k += 32) {
      const float* U = a.u + (size_t)k * D * D;
      const float* m = a.mu + (size_t)k * D;
      float q = 0.f;
      for (int r = 0; r < D; ++r) {
        float y = 0.f;
        for (int j = r; j < D; ++j) y = fmaf(__ldg(U + r * D + j), xs[j] - __ldg(m + j), y);
        q = fmaf(y, y, q);
      }
      const float df = __ldg(a.df + k);
      rs[k] = __ldg(a.tconst + k) - 0.5f * (df + (float)a.D_true) * log1pf(q / df);
    }
    __syncwarp();
    if (lane == 0) {
      a.labels[i] = dpmm_draw_argmax(rs, 1, K);
      if (a.probs != nullptr) {
        float mx = -CUDART_INF_F;
        for (int k = 0; k < K; ++k) {
          if (rs[k] != rs[k]) rs[k] = -CUDART_INF_F;
          mx = fmaxf(mx, rs[k]);
        }
        float s = 0.f;
        for (int k = 0; k < K; ++k) {
          rs[k] = expf(rs[k] - mx);
          s += rs[k];
        }
        for (int k = 0; k < K; ++k) a.probs[(size_t)i * K + k] = rs[k] / s;
      }
    }
    __syncwarp();
  }
}
