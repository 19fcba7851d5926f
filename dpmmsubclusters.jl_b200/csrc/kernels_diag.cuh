// Stages 1-3 for the diagonal-covariance Gaussian prior (DPMM_PRIOR_DIAG_GAUSSIAN): every feature an independent
// one-dimensional NIW, so a distribution is mu[D], sigma^2[D] and logdetSigma = sum_d log sigma^2_d.
//
//   log-likelihood   r = -(D log 2pi + logdetSigma) / 2 - 1/2 sum_d ((x_d - mu_d) / sigma_d)^2,  then + log w (Float32)
//
// The sweep reads, per distribution, s_d = 1/sigma_d and b_d = -s_d mu_d (both rounded once to Float32 from Float64
// on the host, dpmm_set_params_diag) and the constant cst = -(D log 2pi + logdetSigma) / 2.  Every kernel forms
// t = fmaf(s, x, b) and accumulates fmaf(t, t, acc) over ascending d: the square is never expanded into x^2 and x
// terms, which would cancel catastrophically for points far from the origin relative to sigma.  r = fmaf(-0.5, acc,
// cst) (exactly cst - acc / 2 rounded once), then __fadd_rn(r, log w).  The label kernels of both shapes and the
// sub-label kernel therefore produce the same bits for the same (point, distribution).
//
// Parameter images (ctx->recs, ctx->logp_t):
//   recs    [2][3K][D]   s rows, then b rows, distributions in [cluster k][cluster, left, right] order
//   logp_t  [2][D][KP]   the cluster rows (3k) of s and b transposed and zero padded past K (label kernels)
// A zero s and b contribute t = 0, so padded clusters and ragged feature panels leave every sum unchanged.
#pragma once
#include "common.cuh"
#include "kernels_gauss.cuh"  // SubLabelArgs, sublabel_partition
#include "kernels_stats.cuh"  // StatsArgs, StatsItem, cp.async helpers

struct DiagLabelArgs {
  const float* x;       // [n][D]
  int64_t n;
  int D;
  int DS;               // shared-memory row stride of the point tile (odd; staged kernel)
  int K;
  int KP;               // K rounded up to a multiple of DIAG_KT
  const float* s_t;     // [D][KP]
  const float* b_t;     // [D][KP]
  const float* cst;     // [3K]
  const float* logw;    // [K]
  int32_t* labels;
  int32_t* hist;
  const double* u_inj;
  uint64_t seed;
  uint32_t call;
  int64_t goff;
  int final_iter;
  int sampler;
  float* dump;
  int64_t ntiles;
};

#define DIAG_KT 16

__device__ __forceinline__ float diag_finish(float acc, float cst, float lw) {
  return __fadd_rn(fmaf(-0.5f, acc, cst), lw);
}

// the draw of one point from its column of the [K][stride] slice of parr (+ dump, histogram)
__device__ __forceinline__ void diag_draw_point(const DiagLabelArgs& a, float* col, int stride, int64_t i, int* hs) {
  if (a.dump != nullptr)
    for (int k = 0; k < a.K; ++k) a.dump[(size_t)k * a.n + i] = col[(size_t)k * stride];
  int lab;
  if (a.final_iter) {
    lab = dpmm_draw_argmax(col, stride, a.K);
  } else if (a.sampler == 1) {
    lab = dpmm_draw_gumbel(col, stride, a.K, a.seed, a.call, (uint64_t)(a.goff + i));
  } else {
    const double u = dpmm_uniform(a.u_inj, i, a.seed, DPMM_STREAM_LABEL, a.call, (uint64_t)(a.goff + i));
    lab = dpmm_draw_inverse_cdf_screened(col, stride, a.K, u);
  }
  a.labels[i] = lab;
  atomicAdd(&hs[lab], 1);
}

// Label kernel for shapes whose s / b tables fit shared memory beside a point tile: one thread = one point, tile =
// blockDim.x consecutive points, DIAG_KT clusters per pass as 8 packed pairs (FFMA2).
//   st, bt [D][KP] tables,   xs [T][DS] tile,   rs [K][T] slice of parr,   hs [K]
__global__ void diag_label_kernel(const DiagLabelArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int T = blockDim.x;
  const int tid = threadIdx.x;
  float* st = smem;
  float* bt = st + (size_t)a.D * a.KP;
  float* xs = bt + (size_t)a.D * a.KP;
  float* rs = xs + (size_t)T * a.DS;
  int* hs = reinterpret_cast<int*>(rs + (size_t)a.K * T);
  for (int e = tid; e < a.D * a.KP / 4; e += T) {
    reinterpret_cast<float4*>(st)[e] = __ldg(reinterpret_cast<const float4*>(a.s_t) + e);
    reinterpret_cast<float4*>(bt)[e] = __ldg(reinterpret_cast<const float4*>(a.b_t) + e);
  }
  for (int k = tid; k < a.K; k += T) hs[k] = 0;

  for (int64_t tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
    const int64_t base = tile * T;
    const int npts = (int)min((int64_t)T, a.n - base);
    __syncthreads();
    {
      const float* src = a.x + base * a.D;
      const int nv = npts * a.D;
      for (int e = tid; e < T * a.D; e += T) {
        const int p = e / a.D, c = e - p * a.D;
        xs[(size_t)p * a.DS + c] = (e < nv) ? __ldg(src + e) : 0.f;
      }
    }
    __syncthreads();
    const float* xr = xs + (size_t)tid * a.DS;
    for (int k0 = 0; k0 < a.KP; k0 += DIAG_KT) {
      f32x2_t acc[DIAG_KT / 2];
#pragma unroll
      for (int j = 0; j < DIAG_KT / 2; ++j) acc[j] = 0ull;
      for (int d = 0; d < a.D; ++d) {
        const float xv = xr[d];
        const f32x2_t xx = f2_pack(xv, xv);
        const ulonglong2* sr = reinterpret_cast<const ulonglong2*>(st + (size_t)d * a.KP + k0);
        const ulonglong2* br = reinterpret_cast<const ulonglong2*>(bt + (size_t)d * a.KP + k0);
#pragma unroll
        for (int j4 = 0; j4 < DIAG_KT / 4; ++j4) {
          const ulonglong2 s = sr[j4], b = br[j4];
          const f32x2_t t0 = f2_fma(s.x, xx, b.x), t1 = f2_fma(s.y, xx, b.y);
          acc[2 * j4] = f2_fma(t0, t0, acc[2 * j4]);
          acc[2 * j4 + 1] = f2_fma(t1, t1, acc[2 * j4 + 1]);
        }
      }
#pragma unroll
      for (int j = 0; j < DIAG_KT / 2; ++j) {
        float lo, hi;
        f2_unpack(acc[j], lo, hi);
        const int k = k0 + 2 * j;
        if (k < a.K) rs[(size_t)k * T + tid] = diag_finish(lo, __ldg(a.cst + 3 * k), __ldg(a.logw + k));
        if (k + 1 < a.K) rs[(size_t)(k + 1) * T + tid] = diag_finish(hi, __ldg(a.cst + 3 * (k + 1)), __ldg(a.logw + k + 1));
      }
    }
    if (tid < npts) diag_draw_point(a, rs + tid, T, base + tid, hs);
  }
  __syncthreads();
  for (int k = tid; k < a.K; k += T)
    if (hs[k] != 0) atomicAdd(&a.hist[k], hs[k]);
}

// Label kernel for the shapes whose tables do not fit shared memory (large D and / or K): the blocking of
// mnm_label_stream_kernel.  A persistent CTA of 256 threads owns tiles of TP points; clusters go in chunks of
// KC = 16384 / TP and the features in panels of DIAG_SP, double-buffered with cp.async (s and b panels [DIAG_SP][KC]
// straight from the transposed tables, the X panel transposed to [DIAG_SP][TP + 4]).  Every thread owns an 8 x 8
// block of (point, cluster) sums as 8 x 4 packed pairs.  The panel is half as deep as the multinomial kernel's because
// two tables travel: with K = 1024 the 32-point tile still fits.
#define DIAG_SP 8
template <int TP>
struct DiagStreamCfg {
  static constexpr int KC = 16384 / TP;
  static constexpr int XS = TP + 4;
  static constexpr int WY = TP / 32;
  static constexpr int WX = 8 / WY;
  static constexpr size_t stage_floats = (size_t)DIAG_SP * (2 * KC + XS);
  static size_t smem_bytes(int K) { return (2 * stage_floats + (size_t)K * TP) * 4 + (size_t)K * 4; }
};

template <int TP>
__global__ void __launch_bounds__(256) diag_label_stream_kernel(const DiagLabelArgs a) {
  using C = DiagStreamCfg<TP>;
  constexpr int KC = C::KC, XS = C::XS;
  extern __shared__ __align__(16) float smem[];
  float* stage = smem;                          // 2 x ([DIAG_SP][KC] s | [DIAG_SP][KC] b | [DIAG_SP][XS] X)
  float* rs = smem + 2 * C::stage_floats;       // [K][TP]
  int* hs = reinterpret_cast<int*>(rs + (size_t)a.K * TP);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tx = (warp % C::WX) * 8 + (lane & 7);   // clusters k0 + 4 tx + {0..3} and k0 + KC/2 + 4 tx + {0..3}
  const int ty = (warp / C::WX) * 4 + (lane >> 3);  // points 4 ty + {0..3} and TP/2 + 4 ty + {0..3}
  const int D = a.D;
  const int npan = (D + DIAG_SP - 1) / DIAG_SP;
  const int nsteps = npan * ((a.K + KC - 1) / KC);
  for (int k = tid; k < a.K; k += 256) hs[k] = 0;

  for (int64_t tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
    const int64_t base = tile * TP;
    const int npts = (int)min((int64_t)TP, a.n - base);
    auto issue = [&](int s) {
      float* ss = stage + (size_t)(s & 1) * C::stage_floats;
      float* bs = ss + DIAG_SP * KC;
      float* xs = bs + DIAG_SP * KC;
      const int d0 = (s % npan) * DIAG_SP, k0 = (s / npan) * KC;
#pragma unroll
      for (int r = 0; r < DIAG_SP * KC / 4 / 256; ++r) {
        const int e = tid + 256 * r;
        const int d = e / (KC / 4), k = k0 + 4 * (e % (KC / 4));
        const bool ok = d0 + d < D && k < a.KP;
        const size_t off = ok ? (size_t)(d0 + d) * a.KP + k : 0;
        cp_async16(ss + d * KC + 4 * (e % (KC / 4)), a.s_t + off, ok ? 16 : 0);
        cp_async16(bs + d * KC + 4 * (e % (KC / 4)), a.b_t + off, ok ? 16 : 0);
      }
#pragma unroll
      for (int r = 0; r < TP * DIAG_SP / 256; ++r) {
        const int d = lane & 7;
        const int p = (r * 8 + warp) * 4 + (lane >> 3);
        const bool ok = p < npts && d0 + d < D;
        cp_async4(xs + d * XS + p, ok ? a.x + (base + p) * D + d0 + d : a.x, ok ? 4 : 0);
      }
      cp_async_commit();
    };
    f32x2_t acc[8][4];
    issue(0);
    for (int s = 0; s < nsteps; ++s) {
      if (s % npan == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = 0ull;
      }
      if (s + 1 < nsteps) {
        issue(s + 1);
        cp_async_wait_group<1>();
      } else {
        cp_async_wait_all();
      }
      __syncthreads();
      const float* ss = stage + (size_t)(s & 1) * C::stage_floats;
      const float* bs = ss + DIAG_SP * KC;
      const float* xs = bs + DIAG_SP * KC;
#pragma unroll
      for (int d = 0; d < DIAG_SP; ++d) {
        const float4 x0 = *reinterpret_cast<const float4*>(xs + d * XS + 4 * ty);
        const float4 x1 = *reinterpret_cast<const float4*>(xs + d * XS + TP / 2 + 4 * ty);
        const ulonglong2 s0 = *reinterpret_cast<const ulonglong2*>(ss + d * KC + 4 * tx);
        const ulonglong2 s1 = *reinterpret_cast<const ulonglong2*>(ss + d * KC + KC / 2 + 4 * tx);
        const ulonglong2 b0 = *reinterpret_cast<const ulonglong2*>(bs + d * KC + 4 * tx);
        const ulonglong2 b1 = *reinterpret_cast<const ulonglong2*>(bs + d * KC + KC / 2 + 4 * tx);
        const float xv[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
        const f32x2_t sv[4] = {s0.x, s0.y, s1.x, s1.y};
        const f32x2_t bv[4] = {b0.x, b0.y, b1.x, b1.y};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const f32x2_t xx = f2_pack(xv[i], xv[i]);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const f32x2_t t = f2_fma(sv[j], xx, bv[j]);
            acc[i][j] = f2_fma(t, t, acc[i][j]);
          }
        }
      }
      if (s % npan == npan - 1) {
        const int k0 = (s / npan) * KC;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const int k = k0 + (j < 2 ? 4 * tx + 2 * j + h : KC / 2 + 4 * tx + 2 * (j - 2) + h);
            if (k < a.K) {
              const float c = __ldg(a.cst + 3 * k), lw = __ldg(a.logw + k);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float lo, hi;
                f2_unpack(acc[i][j], lo, hi);
                const int p = i < 4 ? 4 * ty + i : TP / 2 + 4 * ty + i - 4;
                rs[(size_t)k * TP + p] = diag_finish(h ? hi : lo, c, lw);
              }
            }
          }
        }
      }
      __syncthreads();   // the buffer just read is the next issue's target
    }
    if (tid < npts) diag_draw_point(a, rs + tid, TP, base + tid, hs);
    __syncthreads();   // rs is rewritten by the next tile
  }
  for (int k = tid; k < a.K; k += 256)
    if (hs[k] != 0) atomicAdd(&a.hist[k], hs[k]);
}

// Sub-label draw over the label-sorted permutation (+ left / right partition).  128 label-sorted positions per CTA;
// the rows go through a [128][65] shared-memory tile 64 features at a time (every row segment read by a whole warp
// as two 128-byte lines), and each thread runs the chains of its point under the l / r distributions of its label
// (warp-uniform broadcast loads of s and b: the positions are sorted by label).  a.recs = the s rows [3K][D], followed
// by the b rows [3K][D].
#define DIAG_SLS_T 128
__global__ void __launch_bounds__(DIAG_SLS_T) diag_sublabel_kernel(const SubLabelArgs a) {
  __shared__ float xs[DIAG_SLS_T][65];
  __shared__ int32_t s_idx[DIAG_SLS_T];
  __shared__ int s_cnt[2 * DIAG_SLS_T];
  __shared__ int s_base[2 * DIAG_SLS_T];
  __shared__ int s_first[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int D = a.D;
  const int64_t pos = (int64_t)blockIdx.x * DIAG_SLS_T + tid;
  const bool active = pos < a.n;
  int32_t idx = active ? a.perm[pos] : -1;
  const int k = active ? a.labels[idx] : 0;
  s_idx[tid] = idx;
  const float* sl_ = a.recs + (size_t)(3 * k + 1) * D;
  const float* sr_ = a.recs + (size_t)(3 * k + 2) * D;
  const size_t boff = (size_t)3 * a.K * D;
  float sl = 0.f, sr = 0.f;
  for (int d0 = 0; d0 < D; d0 += 64) {
    __syncthreads();   // s_idx written / the previous panel consumed
    const bool ok0 = d0 + lane < D, ok1 = d0 + 32 + lane < D;
#pragma unroll 8
    for (int p = warp; p < DIAG_SLS_T; p += DIAG_SLS_T / 32) {
      const int32_t q = s_idx[p];
      const float* xr = a.x + (size_t)max(q, 0) * D + d0 + lane;
      xs[p][lane] = (q >= 0 && ok0) ? __ldg(xr) : 0.f;
      xs[p][32 + lane] = (q >= 0 && ok1) ? __ldg(xr + 32) : 0.f;
    }
    __syncthreads();
    const int dn = min(64, D - d0);
    for (int d = 0; d < dn; ++d) {
      const float xv = xs[tid][d];
      const float tl = fmaf(__ldg(sl_ + d0 + d), xv, __ldg(sl_ + boff + d0 + d));
      const float tr = fmaf(__ldg(sr_ + d0 + d), xv, __ldg(sr_ + boff + d0 + d));
      sl = fmaf(tl, tl, sl);
      sr = fmaf(tr, tr, sr);
    }
  }
  int side = 0;
  if (active) {
    const float rl = diag_finish(sl, __ldg(a.cst + 3 * k + 1), __ldg(a.loglr + 2 * k));
    const float rr = diag_finish(sr, __ldg(a.cst + 3 * k + 2), __ldg(a.loglr + 2 * k + 1));
    if (a.dump != nullptr) {
      a.dump[idx] = rl;
      a.dump[a.n + idx] = rr;
    }
    const double u = dpmm_uniform(a.u_inj, idx, a.seed, DPMM_STREAM_SUBLABEL, a.call, (uint64_t)(a.goff + idx));
    side = dpmm_draw_two(rl, rr, u);
    a.sub[idx] = (uint8_t)side;
  }
  sublabel_partition(a, active, k, side, active ? idx : 0, s_cnt, s_base, s_first);
}

// Statistics: N (from the partition), sum x and sum x^2 per feature for every (label, side) run of perm2.  One warp
// per (work item, slice of 32 x DIAG_STATS_NREG features); lane l owns the features l, l + 32, ... of its slice, so
// every point is read as coalesced 128-byte segments, and accumulates them in Float64: Gaussian sums, unlike
// multinomial counts, are not exact in Float32, and a Float64 x^2 of a Float32 x is exact, so sum x^2 keeps its
// digits for means far from the origin relative to sigma.  The per-lane sums go to the key's Float64 accumulator
// [2K][1 + 2D] (count slot | sum x | sum x^2) once per unit; stats_finalize_kernel adds left and right.
#define DIAG_STATS_NREG 8
#define DIAG_STATS_UNROLL 4
__global__ void __launch_bounds__(256) diag_stats_kernel(const StatsArgs a) {
  const int lane = threadIdx.x & 31;
  const int nslices = (a.D + 32 * DIAG_STATS_NREG - 1) / (32 * DIAG_STATS_NREG);
  const int n_units = *a.n_items * nslices;
  for (;;) {
    int u = 0;
    if (lane == 0) u = atomicAdd(a.next_item, 1);
    u = __shfl_sync(0xffffffffu, u, 0);
    if (u >= n_units) break;
    const StatsItem item = a.items[u / nslices];
    const int d0 = (u % nslices) * 32 * DIAG_STATS_NREG;
    const int Ds = min(a.D - d0, 32 * DIAG_STATS_NREG);
    const float* x = a.x + d0;
    double s1[DIAG_STATS_NREG], s2[DIAG_STATS_NREG];
#pragma unroll
    for (int r = 0; r < DIAG_STATS_NREG; ++r) s1[r] = s2[r] = 0.0;
    for (int p0 = item.begin; p0 < item.end; p0 += DIAG_STATS_UNROLL) {
      int idx[DIAG_STATS_UNROLL];
#pragma unroll
      for (int j = 0; j < DIAG_STATS_UNROLL; ++j) idx[j] = (p0 + j < item.end) ? __ldg(a.perm2 + p0 + j) : -1;
      float v[DIAG_STATS_UNROLL][DIAG_STATS_NREG];
#pragma unroll
      for (int j = 0; j < DIAG_STATS_UNROLL; ++j)
#pragma unroll
        for (int r = 0; r < DIAG_STATS_NREG; ++r) {
          const int d = lane + 32 * r;
          v[j][r] = (idx[j] >= 0 && d < Ds) ? __ldg(x + (size_t)idx[j] * a.D + d) : 0.f;
        }
#pragma unroll
      for (int j = 0; j < DIAG_STATS_UNROLL; ++j)
#pragma unroll
        for (int r = 0; r < DIAG_STATS_NREG; ++r) {
          const double xv = (double)v[j][r];
          s1[r] += xv;
          s2[r] = fma(xv, xv, s2[r]);
        }
    }
    double* dst = a.acc + (size_t)item.key * a.rec + 1 + d0;
#pragma unroll
    for (int r = 0; r < DIAG_STATS_NREG; ++r) {
      const int d = lane + 32 * r;
      if (d < Ds && s2[r] != 0.0) {
        atomicAdd(dst + d, s1[r]);
        atomicAdd(dst + a.D + d, s2[r]);
      }
    }
  }
}
