// Stage 1+2 for the Dirichlet-multinomial prior.
//
//   log_likelihood!(r, x, ::multinomial_dist)   src/distributions/multinomial_dist.jl:13-15
//       r_j = sum_d alpha_d * x[d,j]   (alpha = log-probabilities, no multinomial coefficient)
//   sample_labels_worker! / create_subclusters_labels!  (as in kernels_gauss.cuh)
//
// The n x K product is a skinny GEMM (counts x log-probabilities) that is HBM-bound once X is
// streamed once: every thread owns one point, keeps KT running dot products in registers and reads
// the log-probability table from shared memory as float4 broadcasts.  D and K are runtime values.
#pragma once
#include "common.cuh"
#include "kernels_gauss.cuh"  // SubLabelArgs, sublabel_partition

struct MnmLabelArgs {
  const float* x;       // [n][D] counts
  int64_t n;
  int D;
  int DS;               // shared-memory row stride (odd)
  int K;
  int KP;               // K rounded up to a multiple of MNM_KT
  const float* logp_t;  // [D][KP] cluster log-probabilities, transposed + zero padded
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

#define MNM_KT 16

// K3: one thread = one point, tile = blockDim.x consecutive points.
//   xs [T][DS]  tile,   as [D][KP] log-probability table,   rs [K][T] slice of parr,   hs [K]
__global__ void mnm_label_kernel(const MnmLabelArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int T = blockDim.x;
  const int tid = threadIdx.x;
  float* as = smem;
  float* xs = as + (size_t)a.D * a.KP;
  float* rs = xs + (size_t)T * a.DS;
  int* hs = reinterpret_cast<int*>(rs + (size_t)a.K * T);
  for (int e = tid; e < a.D * a.KP / 4; e += T)
    reinterpret_cast<float4*>(as)[e] = __ldg(reinterpret_cast<const float4*>(a.logp_t) + e);
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
    for (int k0 = 0; k0 < a.KP; k0 += MNM_KT) {
      float acc[MNM_KT];
#pragma unroll
      for (int j = 0; j < MNM_KT; ++j) acc[j] = 0.f;
      for (int d = 0; d < a.D; ++d) {
        const float xv = xr[d];
        const float4* ar = reinterpret_cast<const float4*>(as + (size_t)d * a.KP + k0);
#pragma unroll
        for (int j4 = 0; j4 < MNM_KT / 4; ++j4) {
          const float4 w = ar[j4];
          acc[4 * j4 + 0] = fmaf(w.x, xv, acc[4 * j4 + 0]);
          acc[4 * j4 + 1] = fmaf(w.y, xv, acc[4 * j4 + 1]);
          acc[4 * j4 + 2] = fmaf(w.z, xv, acc[4 * j4 + 2]);
          acc[4 * j4 + 3] = fmaf(w.w, xv, acc[4 * j4 + 3]);
        }
      }
#pragma unroll
      for (int j = 0; j < MNM_KT; ++j)
        if (k0 + j < a.K) rs[(size_t)(k0 + j) * T + tid] = __fadd_rn(acc[j], __ldg(a.logw + k0 + j));
    }
    if (tid < npts) {
      const int64_t i = base + tid;
      float* col = rs + tid;
      if (a.dump != nullptr)
        for (int k = 0; k < a.K; ++k) a.dump[(size_t)k * a.n + i] = col[(size_t)k * T];
      int lab;
      if (a.final_iter) {
        lab = dpmm_draw_argmax(col, T, a.K);
      } else if (a.sampler == 1) {
        lab = dpmm_draw_gumbel(col, T, a.K, a.seed, a.call, (uint64_t)(a.goff + i));
      } else {
        const double u = dpmm_uniform(a.u_inj, i, a.seed, DPMM_STREAM_LABEL, a.call, (uint64_t)(a.goff + i));
        lab = dpmm_draw_inverse_cdf_screened(col, T, a.K, u);
      }
      a.labels[i] = lab;
      atomicAdd(&hs[lab], 1);
    }
  }
  __syncthreads();
  for (int k = tid; k < a.K; k += T)
    if (hs[k] != 0) atomicAdd(&a.hist[k], hs[k]);
}

// K3 for the shapes whose [D][KP] table does not fit shared memory beside a 32-point tile (large D and / or
// large K).  A persistent CTA of 256 threads owns tiles of TP points; clusters go in chunks of KC = 16384 / TP,
// and D in panels of MNM_SP features, double-buffered with cp.async: the table panel [MNM_SP][KC] straight
// from logp_t, the X panel transposed to [MNM_SP][TP + 4] by 4-byte copies (a warp reads 8 features of 4 points:
// whole 32-byte sectors, conflict-free stores).  Every thread owns an 8 x 8 block of (point, cluster) dot
// products, and each one is the same sequential fmaf chain over ascending d as in mnm_label_kernel, then
// __fadd_rn(acc, logw[k]), so both kernels produce identical bits.  Ragged panels load zeros for both operands
// (fmaf(0, 0, acc) == acc: acc starts at +0 and never holds -0).  The [K][TP] slice of parr stays in shared
// memory, and each point's draw runs on its column with the same helpers and stream keys.
#define MNM_SP 16
template <int TP>
struct MnmStreamCfg {
  static constexpr int KC = 16384 / TP;      // clusters per chunk: TP x KC = 256 threads x 64 products
  static constexpr int XS = TP + 4;          // X panel row stride
  static constexpr int WY = TP / 32;         // warps along the point axis (4 lanes x 4 points x 2 halves each)
  static constexpr int WX = 8 / WY;
  static constexpr size_t stage_floats = (size_t)MNM_SP * (KC + XS);
  static size_t smem_bytes(int K) { return (2 * stage_floats + (size_t)K * TP) * 4 + (size_t)K * 4; }
};

template <int TP>
__global__ void __launch_bounds__(256) mnm_label_stream_kernel(const MnmLabelArgs a) {
  using C = MnmStreamCfg<TP>;
  constexpr int KC = C::KC, XS = C::XS;
  extern __shared__ __align__(16) float smem[];
  float* stage = smem;                          // 2 x ([MNM_SP][KC] table | [MNM_SP][XS] X)
  float* rs = smem + 2 * C::stage_floats;       // [K][TP]
  int* hs = reinterpret_cast<int*>(rs + (size_t)a.K * TP);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tx = (warp % C::WX) * 8 + (lane & 7);   // cluster group: k0 + 4 tx + {0..3} and k0 + KC/2 + 4 tx + {0..3}
  const int ty = (warp / C::WX) * 4 + (lane >> 3);  // point group:   4 ty + {0..3} and TP/2 + 4 ty + {0..3}
  const int D = a.D;
  const int npan = (D + MNM_SP - 1) / MNM_SP;
  const int nsteps = npan * ((a.K + KC - 1) / KC);
  for (int k = tid; k < a.K; k += 256) hs[k] = 0;

  for (int64_t tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
    const int64_t base = tile * TP;
    const int npts = (int)min((int64_t)TP, a.n - base);
    auto issue = [&](int s) {
      float* ts = stage + (size_t)(s & 1) * C::stage_floats;
      float* xs = ts + MNM_SP * KC;
      const int d0 = (s % npan) * MNM_SP, k0 = (s / npan) * KC;
#pragma unroll
      for (int r = 0; r < MNM_SP * KC / 4 / 256; ++r) {
        const int e = tid + 256 * r;
        const int d = e / (KC / 4), k = k0 + 4 * (e % (KC / 4));
        const bool ok = d0 + d < D && k < a.KP;
        cp_async16(ts + d * KC + 4 * (e % (KC / 4)), ok ? a.logp_t + (size_t)(d0 + d) * a.KP + k : a.logp_t, ok ? 16 : 0);
      }
#pragma unroll
      for (int r = 0; r < TP * MNM_SP / 256; ++r) {
        const int d = (r & 1) * 8 + (lane & 7);
        const int p = ((r >> 1) * 8 + warp) * 4 + (lane >> 3);
        const bool ok = p < npts && d0 + d < D;
        cp_async4(xs + d * XS + p, ok ? a.x + (base + p) * D + d0 + d : a.x, ok ? 4 : 0);
      }
      cp_async_commit();
    };
    float acc[8][8];
    issue(0);
    for (int s = 0; s < nsteps; ++s) {
      if (s % npan == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
      }
      if (s + 1 < nsteps) {
        issue(s + 1);
        cp_async_wait_group<1>();
      } else {
        cp_async_wait_all();
      }
      __syncthreads();
      const float* ts = stage + (size_t)(s & 1) * C::stage_floats;
      const float* xs = ts + MNM_SP * KC;
#pragma unroll
      for (int d = 0; d < MNM_SP; ++d) {
        const float4 x0 = *reinterpret_cast<const float4*>(xs + d * XS + 4 * ty);
        const float4 x1 = *reinterpret_cast<const float4*>(xs + d * XS + TP / 2 + 4 * ty);
        const float4 t0 = *reinterpret_cast<const float4*>(ts + d * KC + 4 * tx);
        const float4 t1 = *reinterpret_cast<const float4*>(ts + d * KC + KC / 2 + 4 * tx);
        const float xv[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
        const float tv[8] = {t0.x, t0.y, t0.z, t0.w, t1.x, t1.y, t1.z, t1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(tv[j], xv[i], acc[i][j]);
      }
      if (s % npan == npan - 1) {
        const int k0 = (s / npan) * KC;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int k = k0 + (j < 4 ? 4 * tx + j : KC / 2 + 4 * tx + j - 4);
          if (k < a.K) {
            const float lw = __ldg(a.logw + k);
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int p = i < 4 ? 4 * ty + i : TP / 2 + 4 * ty + i - 4;
              rs[(size_t)k * TP + p] = __fadd_rn(acc[i][j], lw);
            }
          }
        }
      }
      __syncthreads();   // the buffer just read is the next issue's target
    }
    if (tid < npts) {
      const int64_t i = base + tid;
      float* col = rs + tid;
      if (a.dump != nullptr)
        for (int k = 0; k < a.K; ++k) a.dump[(size_t)k * a.n + i] = col[(size_t)k * TP];
      int lab;
      if (a.final_iter) {
        lab = dpmm_draw_argmax(col, TP, a.K);
      } else if (a.sampler == 1) {
        lab = dpmm_draw_gumbel(col, TP, a.K, a.seed, a.call, (uint64_t)(a.goff + i));
      } else {
        const double u = dpmm_uniform(a.u_inj, i, a.seed, DPMM_STREAM_LABEL, a.call, (uint64_t)(a.goff + i));
        lab = dpmm_draw_inverse_cdf_screened(col, TP, a.K, u);
      }
      a.labels[i] = lab;
      atomicAdd(&hs[lab], 1);
    }
    __syncthreads();   // rs is rewritten by the next tile
  }
  for (int k = tid; k < a.K; k += 256)
    if (hs[k] != 0) atomicAdd(&a.hist[k], hs[k]);
}

// Sub-label draw over the label-sorted permutation (+ left/right partition); a.recs = log_p [3K][D].
template <bool SAMPLE>
__global__ void mnm_sublabel_kernel(const SubLabelArgs a) {
  __shared__ int s_cnt[2 * 256];
  __shared__ int s_base[2 * 256];
  __shared__ int s_first[2];
  const int tid = threadIdx.x;
  const int64_t pos = (int64_t)blockIdx.x * blockDim.x + tid;
  const bool active = pos < a.n;
  int32_t idx = 0;
  int k = 0, side = 0;
  if (active) {
    idx = a.perm[pos];
    k = a.labels[idx];
    if constexpr (SAMPLE) {
      const float* xp = a.x + (size_t)idx * a.D;
      const float* al = a.recs + (size_t)(3 * k + 1) * a.D;
      const float* ar = a.recs + (size_t)(3 * k + 2) * a.D;
      float sl = 0.f, sr = 0.f;
      for (int d = 0; d < a.D; ++d) {
        const float xv = __ldg(xp + d);
        sl = fmaf(__ldg(al + d), xv, sl);
        sr = fmaf(__ldg(ar + d), xv, sr);
      }
      const float rl = __fadd_rn(sl, __ldg(a.loglr + 2 * k));
      const float rr = __fadd_rn(sr, __ldg(a.loglr + 2 * k + 1));
      if (a.dump != nullptr) {
        a.dump[idx] = rl;
        a.dump[a.n + idx] = rr;
      }
      const double u = dpmm_uniform(a.u_inj, idx, a.seed, DPMM_STREAM_SUBLABEL, a.call, (uint64_t)(a.goff + idx));
      side = dpmm_draw_two(rl, rr, u);
      a.sub[idx] = (uint8_t)side;
    } else {
      side = a.sub[idx];
    }
  }
  sublabel_partition(a, active, k, side, idx, s_cnt, s_base, s_first);
}

// Sub-label draw, D > 1024: the positions and the per-point arithmetic of mnm_sublabel_kernel<true> (128
// label-sorted positions per CTA, sl / sr sequential fmaf over ascending d), but the 128 rows go through a
// [128][65] shared-memory tile 64 features at a time, every row segment read by a whole warp as two 128-byte
// lines, instead of each thread walking its own row.
#define MNM_SLS_T 128
__global__ void __launch_bounds__(MNM_SLS_T) mnm_sublabel_staged_kernel(const SubLabelArgs a) {
  __shared__ float xs[MNM_SLS_T][65];
  __shared__ int32_t s_idx[MNM_SLS_T];
  __shared__ int s_cnt[2 * MNM_SLS_T];
  __shared__ int s_base[2 * MNM_SLS_T];
  __shared__ int s_first[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int D = a.D;
  const int64_t pos = (int64_t)blockIdx.x * MNM_SLS_T + tid;
  const bool active = pos < a.n;
  int32_t idx = active ? a.perm[pos] : -1;
  const int k = active ? a.labels[idx] : 0;
  s_idx[tid] = idx;
  const float* al = a.recs + (size_t)(3 * k + 1) * D;
  const float* ar = a.recs + (size_t)(3 * k + 2) * D;
  float sl = 0.f, sr = 0.f;
  for (int d0 = 0; d0 < D; d0 += 64) {
    __syncthreads();   // s_idx written / the previous panel consumed
    const bool ok0 = d0 + lane < D, ok1 = d0 + 32 + lane < D;
#pragma unroll 8
    for (int p = warp; p < MNM_SLS_T; p += MNM_SLS_T / 32) {
      const int32_t q = s_idx[p];
      const float* xr = a.x + (size_t)max(q, 0) * D + d0 + lane;
      xs[p][lane] = (q >= 0 && ok0) ? __ldg(xr) : 0.f;
      xs[p][32 + lane] = (q >= 0 && ok1) ? __ldg(xr + 32) : 0.f;
    }
    __syncthreads();
    const int dn = min(64, D - d0);
    for (int d = 0; d < dn; ++d) {
      const float xv = xs[tid][d];
      sl = fmaf(__ldg(al + d0 + d), xv, sl);
      sr = fmaf(__ldg(ar + d0 + d), xv, sr);
    }
  }
  int side = 0;
  if (active) {
    const float rl = __fadd_rn(sl, __ldg(a.loglr + 2 * k));
    const float rr = __fadd_rn(sr, __ldg(a.loglr + 2 * k + 1));
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

// Sub-label draw, D <= 128: a warp evaluates its 32 label-sorted positions one point at a time with
// lanes <-> features (each point is read as coalesced 128-byte segments; the l/r log-probability
// vectors of the current label sit in registers and are reloaded only when the label changes), then
// every lane draws and partitions its own point.
__global__ void __launch_bounds__(128) mnm_sublabel2_kernel(const SubLabelArgs a) {
  __shared__ int s_cnt[2 * 128];
  __shared__ int s_base[2 * 128];
  __shared__ int s_first[2];
  const int tid = threadIdx.x, lane = tid & 31;
  const int D = a.D;
  const int64_t pos = (int64_t)blockIdx.x * blockDim.x + tid;
  const bool active = pos < a.n;
  int32_t idx = -1;
  int k = 0, side = 0;
  if (active) {
    idx = a.perm[pos];
    k = a.labels[idx];
  }
  float my_sl = 0.f, my_sr = 0.f;
  float al[4], ar[4];
  int cur = -1;
#pragma unroll 1
  for (int j0 = 0; j0 < 32; j0 += 4) {
    int pi[4], pk[4];
    float xv[4][4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      pi[j] = __shfl_sync(0xffffffffu, idx, j0 + j);
      pk[j] = __shfl_sync(0xffffffffu, k, j0 + j);
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int d = lane + 32 * r;
        xv[j][r] = (pi[j] >= 0 && d < D) ? __ldg(a.x + (size_t)pi[j] * D + d) : 0.f;
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (pi[j] < 0) continue;                       // warp-uniform
      if (pk[j] != cur) {
        cur = pk[j];
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int d = lane + 32 * r;
          al[r] = d < D ? __ldg(a.recs + (size_t)(3 * cur + 1) * D + d) : 0.f;
          ar[r] = d < D ? __ldg(a.recs + (size_t)(3 * cur + 2) * D + d) : 0.f;
        }
      }
      float sl = 0.f, sr = 0.f;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        sl = fmaf(al[r], xv[j][r], sl);
        sr = fmaf(ar[r], xv[j][r], sr);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sl += __shfl_xor_sync(0xffffffffu, sl, o);
        sr += __shfl_xor_sync(0xffffffffu, sr, o);
      }
      if (lane == j0 + j) {
        my_sl = sl;
        my_sr = sr;
      }
    }
  }
  if (active) {
    const float rl = __fadd_rn(my_sl, __ldg(a.loglr + 2 * k));
    const float rr = __fadd_rn(my_sr, __ldg(a.loglr + 2 * k + 1));
    if (a.dump != nullptr) {
      a.dump[idx] = rl;
      a.dump[a.n + idx] = rr;
    }
    const double u = dpmm_uniform(a.u_inj, idx, a.seed, DPMM_STREAM_SUBLABEL, a.call, (uint64_t)(a.goff + idx));
    side = dpmm_draw_two(rl, rr, u);
    a.sub[idx] = (uint8_t)side;
  }
  sublabel_partition(a, active, k, side, idx, s_cnt, s_base, s_first);
}
