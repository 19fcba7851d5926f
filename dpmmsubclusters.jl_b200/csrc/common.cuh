// Shared device helpers: the categorical draw (stage 2) and small utilities.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <math_constants.h>

#include "philox.cuh"

#define DPMM_MAX_K 1024
#define DPMM_MNM_MAX_D 16384   // multinomial vocabulary: the device draw keeps one row of D doubles in shared memory

// ---------------------------------------------------------------------------------------------
// Packed FP32 pairs.  On sm_100a the FMA pipe reaches its peak FP32 rate only with the packed
// FFMA2 form (fma.rn.f32x2: two IEEE FP32 FMAs on 64-bit register pairs); measured with
// tools/micro/ffma_bench.cu: scalar outer-product 50.6 TFLOP/s, packed 63-74 TFLOP/s.  Each half is
// an ordinary round-to-nearest FP32 FMA, so results are identical to the scalar form.
// ---------------------------------------------------------------------------------------------
typedef unsigned long long f32x2_t;
__device__ __forceinline__ f32x2_t f2_pack(float lo, float hi) {
  f32x2_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(f32x2_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2_t f2_fma(f32x2_t a, f32x2_t b, f32x2_t c) {
  f32x2_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

// ---------------------------------------------------------------------------------------------
// Stage 2 -- sample_log_cat_array! (src/utils.jl:19-31) for ONE row, in place on `rs`
// (element k at rs[k*stride], Float32 log-probabilities incl. log-weight).  Returns the 0-based
// index.  Order of operations mirrors the reference line by line:
//   :21 NaN -> -Inf        :22 row max        :23 subtract     :24 exp (underflows to 0 far away)
//   :26 row sum (left to right, Float32)      :27 divide
//   :29 StatsBase.sample(ProbabilityWeights(row)):  t = rand() * sum(w)  (Float64 * Float32),
//       i = 1; cw = w[1]; while cw < t && i < n: i += 1; cw += w[i]      (cw Float32)
// exp is CUDA's full-precision expf (<= 2 ulp; Julia's Float32 exp is <= 1 ulp, the oracle's stand-in is
// correctly rounded): a last-ulp difference moves a cumulative boundary by ~1e-7 relative, far inside
// the documented near-tie band (1e-5 in log space).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int dpmm_draw_inverse_cdf(float* rs, int stride, int K, double u) {
  // Every pass is unrolled by 4 with the loads issued together: the passes are serial per point, so
  // instruction-level parallelism is what hides the shared-memory latency here.  Floating-point
  // ORDER is unchanged: the sums run left to right.
  const int K4 = K & ~3;
  // ---- :21-22  NaN -> -Inf, row max ----
  float mx = -CUDART_INF_F;
  for (int k = 0; k < K4; k += 4) {
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = rs[(k + j) * stride];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (v[j] != v[j]) {
        v[j] = -CUDART_INF_F;
        rs[(k + j) * stride] = v[j];
      }
    }
    mx = fmaxf(mx, fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3])));
  }
  for (int k = K4; k < K; ++k) {
    float v = rs[k * stride];
    if (v != v) {
      v = -CUDART_INF_F;
      rs[k * stride] = v;
    }
    mx = fmaxf(mx, v);
  }
  // ---- :23-26  subtract, exp, row sum ----
  float s = 0.f;
  for (int k = 0; k < K4; k += 4) {
    float e[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) e[j] = expf(rs[(k + j) * stride] - mx);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      rs[(k + j) * stride] = e[j];
      s = __fadd_rn(s, e[j]);
    }
  }
  for (int k = K4; k < K; ++k) {
    const float e = expf(rs[k * stride] - mx);
    rs[k * stride] = e;
    s = __fadd_rn(s, e);
  }
  // ---- :27  divide; the running sum cw_k replaces p_k in place (it is all the walk needs) ----
  // The IEEE division takes a ~70-instruction slow path for zero / denormal numerators, which is what
  // most far-away clusters produce (e^d for d < -87.3).  0 / s is exactly 0 for finite s > 0, and a
  // denormal weight (< 1.2e-38) can never decide the walk: the smallest non-zero t is 2^-53 * sum(w)
  // ~ 1e-16 and for t == 0 the walk stops at i = 1 regardless.  Those lanes therefore divide 1 by s,
  // discard the quotient and use p = 0.
  const bool s_regular = (s > 0.f) && (s < CUDART_INF_F);
  float cw = 0.f;
  bool first = true;  // cw starts AT w[1] (not 0 + w[1]): keeps -0 / NaN semantics of the reference
  for (int k = 0; k < K4; k += 4) {
    float p[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float e = rs[(k + j) * stride];
      const bool zero = (e < 1.17549435e-38f) && s_regular;
      const float quo = __fdiv_rn(zero ? 1.f : e, s);
      p[j] = zero ? 0.f : quo;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      cw = first ? p[j] : __fadd_rn(cw, p[j]);
      first = false;
      rs[(k + j) * stride] = cw;
    }
  }
  for (int k = K4; k < K; ++k) {
    const float e = rs[k * stride];
    const bool zero = (e < 1.17549435e-38f) && s_regular;
    const float quo = __fdiv_rn(zero ? 1.f : e, s);
    const float p = zero ? 0.f : quo;
    cw = first ? p : __fadd_rn(cw, p);
    first = false;
    rs[k * stride] = cw;
  }
  // ---- :29  t = rand() * sum(w);  first i with !(cw_i < t), clamped to n ----
  const double t = u * (double)cw;  // sum(w) accumulated left to right == the last running sum
  int i = K - 1;
  for (int k = 0; k < K4; k += 4) {
    float c[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) c[j] = rs[(k + j) * stride];
    int hit = -1;
#pragma unroll
    for (int j = 3; j >= 0; --j)
      if (!((double)c[j] < t)) hit = k + j;
    if (hit >= 0) {
      i = hit;
      break;
    }
  }
  if (i == K - 1) {
    for (int k = K4; k < K - 1; ++k)
      if (!((double)rs[k * stride] < t)) {
        i = k;
        break;
      }
  }
  return i;
}

// The same draw when only the clusters in `mask` (bit k) carry weight and every other entry is
// exactly -Inf (weight exactly 0): identical arithmetic in identical order -- zeros added to the
// left-to-right sums do not change them -- but only the masked entries are touched.  Requires all
// masked entries to be finite or -Inf (callers route NaN rows to the general routine).
__device__ __forceinline__ int dpmm_draw_inverse_cdf_masked(float* rs, int stride, int K, uint64_t mask, double u) {
  float mx = -CUDART_INF_F;
  for (uint64_t m = mask; m; m &= m - 1) mx = fmaxf(mx, rs[(__ffsll((long long)m) - 1) * stride]);
  float s = 0.f;
  for (uint64_t m = mask; m; m &= m - 1) {
    const int k = __ffsll((long long)m) - 1;
    const float e = expf(rs[k * stride] - mx);
    rs[k * stride] = e;
    s = __fadd_rn(s, e);
  }
  const bool s_regular = (s > 0.f) && (s < CUDART_INF_F);
  float cw = 0.f;
  for (uint64_t m = mask; m; m &= m - 1) {
    const int k = __ffsll((long long)m) - 1;
    const float e = rs[k * stride];
    const bool zero = (e < 1.17549435e-38f) && s_regular;
    const float quo = __fdiv_rn(zero ? 1.f : e, s);
    cw = __fadd_rn(cw, zero ? 0.f : quo);
    rs[k * stride] = cw;
  }
  const double t = u * (double)cw;
  if (!(0.0 < t) && !(mask & 1ull)) return 0;   // cw_1 = w_1 = 0 is not < t: the walk stops at i = 1
  for (uint64_t m = mask; m; m &= m - 1) {
    const int k = __ffsll((long long)m) - 1;
    if (k >= K - 1) break;
    if (!((double)rs[k * stride] < t)) return k;
  }
  return K - 1;
}

// Entry point used by the FMA-pipe label kernels: for K <= 64 first find the row maximum and the
// clusters whose weight is not exactly zero (exp(r - max) underflows to +0 in Float32 below -103.98,
// so everything under max - 104 contributes an exact 0 to every sum of the reference), then run the
// masked draw on those few; otherwise (or when the row holds a NaN / has no finite maximum) the
// general routine.  Both produce the same labels.
__device__ __forceinline__ int dpmm_draw_inverse_cdf_screened(float* rs, int stride, int K, double u) {
  if (K > 64) return dpmm_draw_inverse_cdf(rs, stride, K, u);
  float mx = -CUDART_INF_F;
  bool has_nan = false;
  for (int k = 0; k < K; ++k) {
    const float v = rs[k * stride];
    has_nan |= (v != v);
    mx = fmaxf(mx, v);
  }
  if (has_nan || !(mx > -CUDART_INF_F) || !(mx < CUDART_INF_F)) return dpmm_draw_inverse_cdf(rs, stride, K, u);
  const float thr = mx - 104.f;
  uint64_t mask = 0;
  for (int k = 0; k < K; ++k)
    if (rs[k * stride] >= thr) mask |= 1ull << k;
  // with most clusters in play the unrolled general routine is the faster of the two
  if (2 * __popcll(mask) > K) return dpmm_draw_inverse_cdf(rs, stride, K, u);
  return dpmm_draw_inverse_cdf_masked(rs, stride, K, mask, u);
}

// mapslices(argmax, parr, dims=[2]) (local_clusters_actions.jl:130): first maximal element, NaN
// counts as maximal (Julia's argmax); no NaN sanitising on this branch.
__device__ __forceinline__ int dpmm_draw_argmax(const float* rs, int stride, int K) {
  int best = 0;
  float bv = rs[0];
  if (bv != bv) return 0;
  for (int k = 1; k < K; ++k) {
    const float v = rs[k * stride];
    if (v != v) return k;
    if (v > bv) {
      bv = v;
      best = k;
    }
  }
  return best;
}

// Gumbel-max draw (optional fast mode; same categorical distribution as the inverse-CDF walk, but a
// different random stream: one Philox block feeds 4 clusters).
__device__ __forceinline__ int dpmm_draw_gumbel(const float* rs, int stride, int K, uint64_t seed,
                                               uint32_t call, uint64_t gidx) {
  int best = 0;
  float bv = -CUDART_INF_F;
  for (int k0 = 0; k0 < K; k0 += 4) {
    const Philox4 r = philox4x32_10((uint32_t)gidx, (uint32_t)(gidx >> 32), call,
                                    DPMM_STREAM_GUMBEL + 8u * (uint32_t)(k0 >> 2), (uint32_t)seed,
                                    (uint32_t)(seed >> 32));
    const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + j;
      if (k < K) {
        float v = rs[k * stride];
        if (v != v) v = -CUDART_INF_F;
        const float uu = ((float)w[j] + 0.5f) * 2.3283064365386963e-10f;  // (0,1)
        const float g = -__logf(-__logf(uu));
        const float t = v + g;
        if (t > bv || k == 0) {
          bv = t;
          best = k;
        }
      }
    }
  }
  return best;
}

// Two-way draw for sub-labels: sample_log_cat_array! with C = 2 (create_subclusters_labels!,
// local_clusters_actions.jl:83-95).  Returns 0 (left) or 1 (right).
__device__ __forceinline__ int dpmm_draw_two(float rl, float rr, double u) {
  float m[2] = {rl, rr};
  return dpmm_draw_inverse_cdf(m, 1, 2, u);
}

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL).  The sweep's kernels are launched with launch_pdl(): a kernel may start while
// its predecessor on the stream still runs, does only CTA-local set-up (mbarriers, shared-memory tables, tensor memory)
// and then waits in pdl_wait() until the predecessor has completed and its writes are visible.  Every global load or
// store of such a kernel comes after pdl_wait().  pdl_launch_dependents() lets the next kernel be scheduled; the
// kernels here issue it right after their own wait, so at most two grids of the chain overlap.  Both are no-ops in a
// kernel launched without the attribute.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(bool pdl, void (*kern)(KArgs...), dim3 grid, unsigned block, size_t smem,
                              cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(block);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, args...);
}

__device__ __forceinline__ double dpmm_uniform(const double* inj, int64_t local_i, uint64_t seed,
                                               uint32_t stream, uint32_t call, uint64_t gidx) {
  if (inj != nullptr) return inj[local_i];
  return philox_to_uniform(philox_draw(seed, stream, call, gidx));
}

__device__ __forceinline__ int dpmm_randbit(const uint8_t* inj, int64_t local_i, uint64_t seed,
                                            uint32_t call, uint64_t gidx) {
  if (inj != nullptr) return inj[local_i] & 1;
  return (int)(philox_draw(seed, DPMM_STREAM_RANDBITS, call, gidx).x & 1u);
}
