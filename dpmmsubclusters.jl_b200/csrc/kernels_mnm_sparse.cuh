// Multinomial sweep on sparse counts (dpmm_create_sparse): the points are compressed rows, one row per point,
//   ptr int64 [n + 1] (0-based offsets), idx int32 [nnz] (feature, strictly increasing within a row), val float32 [nnz].
//
// Every log-likelihood here is the sequential fmaf chain over the point's stored entries in ascending d, the chain
// the dense kernels (mnm_label_kernel, mnm_label_stream_kernel, mnm_sublabel_kernel, mnm_sublabel_staged_kernel) run
// over all D features.  An absent feature contributes fmaf(lp, 0, acc) == acc there (acc starts at +0 and never holds
// -0), so with finite log-probabilities both produce the same bits.  Stored zeros are skipped as well: a -Inf
// log-probability against a zero count contributes nothing here, where the dense product gives NaN (0 * -Inf).
#pragma once
#include "common.cuh"
#include "kernels_gauss.cuh"  // SubLabelArgs, sublabel_partition
#include "kernels_params_mnm.cuh"  // MnmScoreArgs
#include "kernels_stats.cuh"  // StatsItem, StatsArgs

struct MnmSparse {
  const int64_t* ptr;   // [n + 1]
  const int32_t* idx;   // [nnz]
  const float* val;     // [nnz]
};

// ---- dpmm_create_sparse: validate the caller's 1-based CSC arrays and convert them to the layout above ----------
// One thread per column.  bad = min over invalid columns j of 4 j + reason (0: colptr decreasing or outside
// [1, nnz + 1], 1: row index outside [1, d], 2: row indices not strictly increasing: unsorted or duplicate).
__global__ void mnm_sparse_convert_kernel(const int64_t* __restrict__ colptr, const int64_t* __restrict__ rowval,
                                          int64_t n, int64_t nnz, int d, int64_t* __restrict__ ptr,
                                          int32_t* __restrict__ idx, unsigned long long* bad) {
  for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = colptr[j] - 1, e = colptr[j + 1] - 1;
    ptr[j + 1] = e;
    if (j == 0) ptr[0] = 0;
    if (b < 0 || e < b || e > nnz) {
      atomicMin(bad, (unsigned long long)(4 * j));
      continue;
    }
    int64_t prev = 0;
    for (int64_t q = b; q < e; ++q) {
      const int64_t r = rowval[q];
      if (r < 1 || r > d) {
        atomicMin(bad, (unsigned long long)(4 * j + 1));
        break;
      }
      if (r <= prev) {
        atomicMin(bad, (unsigned long long)(4 * j + 2));
        break;
      }
      prev = r;
      idx[q] = (int32_t)(r - 1);
    }
  }
}

// ---- label draw ------------------------------------------------------------------------------------------------
// A CTA of 256 threads owns tiles of TP consecutive points and keeps their [K][TP] slice of parr in shared memory.
// Groups of W lanes (W = 32, or 16 / 8 / 4 when K is that small) take points; a group reads its point's (d, c) pairs
// W at a time, coalesced, and broadcasts them by shuffle in ascending order, while every lane owns the clusters
// k0 + lane + W j (j < KR) of the current chunk, so each entry is one coalesced read of a logp_t row.  The table
// is read from shared memory when `tab_smem` (it and the slice fit), else from global memory (L2).  Each point's draw
// then runs thread-per-point on its parr column with the helpers and stream keys of the dense kernels.
struct MnmSparseLabelArgs {
  MnmSparse sp;
  int64_t n;
  int D, K, KP, TP;
  const float* logp_t;  // [D][KP]
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
  int tab_smem;
};

#define MNM_SP_THREADS 256
#define MNM_SP_U 4

template <int W, int KR>
__global__ void __launch_bounds__(MNM_SP_THREADS, 4) mnm_sparse_label_kernel(const MnmSparseLabelArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int TP = a.TP, K = a.K;
  float* rs = smem;                                          // [K][TP]
  int* hs = reinterpret_cast<int*>(rs + (size_t)K * TP);     // [K]
  float* ts = reinterpret_cast<float*>(hs + K);              // [D][KP] when tab_smem
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int g = lane / W, sl = lane % W;
  constexpr int NPW = 32 / W;                                // points per warp step
  const float* tab = a.logp_t;
  if (a.tab_smem) {
    for (int e = tid; e < a.D * a.KP; e += MNM_SP_THREADS) ts[e] = __ldg(a.logp_t + e);
    tab = ts;
  }
  for (int k = tid; k < K; k += MNM_SP_THREADS) hs[k] = 0;

  for (int64_t tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
    const int64_t base = tile * TP;
    const int npts = (int)min((int64_t)TP, a.n - base);
    __syncthreads();   // the table / hs are staged; rs of the previous tile has been drawn from
    for (int p0 = warp * NPW; p0 < npts; p0 += (MNM_SP_THREADS / 32) * NPW) {
      const int p = p0 + g;
      const bool act = p < npts;
      const int64_t b = act ? __ldg(a.sp.ptr + base + p) : 0;
      const int len = act ? (int)(__ldg(a.sp.ptr + base + p + 1) - b) : 0;
      const int maxlen = (int)__reduce_max_sync(0xffffffffu, (unsigned)len);
      for (int k0 = 0; k0 < K; k0 += W * KR) {
        float acc[KR];
#pragma unroll
        for (int j = 0; j < KR; ++j) acc[j] = 0.f;
        for (int t0 = 0; t0 < maxlen; t0 += W) {
          const int q = t0 + sl;
          const int dv = q < len ? __ldg(a.sp.idx + b + q) : 0;
          const float cv = q < len ? __ldg(a.sp.val + b + q) : 0.f;
          // MNM_SP_U entries per step: their table rows are loaded before the chain consumes them (entries past the
          // point's end, and stored zeros, have c = 0 and leave acc unchanged)
          const int nt = min(W, maxlen - t0);
          for (int t = 0; t < nt; t += MNM_SP_U) {
            int d[MNM_SP_U];
            float c[MNM_SP_U], v[MNM_SP_U][KR];
#pragma unroll
            for (int u = 0; u < MNM_SP_U; ++u) {
              d[u] = __shfl_sync(0xffffffffu, dv, (t + u) % W, W);
              c[u] = t + u < W ? __shfl_sync(0xffffffffu, cv, (t + u) % W, W) : 0.f;
              const float* row = tab + (size_t)d[u] * a.KP + k0 + sl;
#pragma unroll
              for (int j = 0; j < KR; ++j) v[u][j] = k0 + sl + W * j < K ? row[W * j] : 0.f;
            }
#pragma unroll
            for (int u = 0; u < MNM_SP_U; ++u)
#pragma unroll
              for (int j = 0; j < KR; ++j) acc[j] = c[u] != 0.f ? fmaf(v[u][j], c[u], acc[j]) : acc[j];
          }
        }
        if (act) {
#pragma unroll
          for (int j = 0; j < KR; ++j) {
            const int k = k0 + sl + W * j;
            if (k < K) rs[(size_t)k * TP + p] = __fadd_rn(acc[j], __ldg(a.logw + k));
          }
        }
      }
    }
    __syncthreads();
    if (tid < npts) {
      const int64_t i = base + tid;
      float* col = rs + tid;
      if (a.dump != nullptr)
        for (int k = 0; k < K; ++k) a.dump[(size_t)k * a.n + i] = col[(size_t)k * TP];
      int lab;
      if (a.final_iter) {
        lab = dpmm_draw_argmax(col, TP, K);
      } else if (a.sampler == 1) {
        lab = dpmm_draw_gumbel(col, TP, K, a.seed, a.call, (uint64_t)(a.goff + i));
      } else {
        const double u = dpmm_uniform(a.u_inj, i, a.seed, DPMM_STREAM_LABEL, a.call, (uint64_t)(a.goff + i));
        lab = dpmm_draw_inverse_cdf_screened(col, TP, K, u);
      }
      a.labels[i] = lab;
      atomicAdd(&hs[lab], 1);
    }
  }
  __syncthreads();
  for (int k = tid; k < K; k += MNM_SP_THREADS)
    if (hs[k] != 0) atomicAdd(&a.hist[k], hs[k]);
}

// ---- sub-label draw ------------------------------------------------------------------------------------------------
// The positions of mnm_sublabel_kernel (128 label-sorted positions per CTA, then sublabel_partition).  Every thread
// runs sl / sr as sequential fmaf chains over its point's entries against rows 3k+1 / 3k+2 of recs; the entries reach
// it through a per-warp shared-memory stage: in each round the warp copies the next MNM_SPS_R entries of all its 32
// points (16 lanes per point, consecutive addresses), then each lane walks its own point's row of the stage.
#define MNM_SPS_T 128
#define MNM_SPS_R 16
__global__ void __launch_bounds__(MNM_SPS_T) mnm_sparse_sublabel_kernel(const SubLabelArgs a, const MnmSparse sp) {
  __shared__ int32_t s_d[MNM_SPS_T][MNM_SPS_R + 1];
  __shared__ float s_c[MNM_SPS_T][MNM_SPS_R + 1];
  __shared__ int s_cnt[2 * MNM_SPS_T];
  __shared__ int s_base[2 * MNM_SPS_T];
  __shared__ int s_first[2];
  const int tid = threadIdx.x, lane = tid & 31, wbase = tid & ~31;
  const int64_t pos = (int64_t)blockIdx.x * MNM_SPS_T + tid;
  const bool active = pos < a.n;
  const int32_t idx = active ? a.perm[pos] : 0;
  const int k = active ? a.labels[idx] : 0;
  const int64_t b = active ? __ldg(sp.ptr + idx) : 0;
  const int len = active ? (int)(__ldg(sp.ptr + idx + 1) - b) : 0;
  const int maxlen = (int)__reduce_max_sync(0xffffffffu, (unsigned)len);
  const float* al = a.recs + (size_t)(3 * k + 1) * a.D;
  const float* ar = a.recs + (size_t)(3 * k + 2) * a.D;
  float sl = 0.f, sr = 0.f;
  const int half = lane >> 4, hl = lane & 15;
  for (int r0 = 0; r0 < maxlen; r0 += MNM_SPS_R) {
#pragma unroll 4
    for (int j = 0; j < 32; j += 2) {
      const int src = j + half;                          // the warp lane whose point this half-warp copies
      const int64_t pb = __shfl_sync(0xffffffffu, b, src);
      const int pl = __shfl_sync(0xffffffffu, len, src);
      const int q = r0 + hl;
      const bool ok = q < pl;
      s_d[wbase + src][hl] = ok ? __ldg(sp.idx + pb + q) : 0;
      s_c[wbase + src][hl] = ok ? __ldg(sp.val + pb + q) : 0.f;
    }
    __syncwarp();
    // the stage is zero past the point's end: all MNM_SPS_R loads issue before the chain, c = 0 leaves it unchanged
    float vl[MNM_SPS_R], vr[MNM_SPS_R];
#pragma unroll
    for (int t = 0; t < MNM_SPS_R; ++t) {
      const int d = s_d[tid][t];
      vl[t] = __ldg(al + d);
      vr[t] = __ldg(ar + d);
    }
#pragma unroll
    for (int t = 0; t < MNM_SPS_R; ++t) {
      const float c = s_c[tid][t];
      sl = c != 0.f ? fmaf(vl[t], c, sl) : sl;
      sr = c != 0.f ? fmaf(vr[t], c, sr) : sr;
    }
    __syncwarp();
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
  sublabel_partition(a, active, k, side, idx, s_cnt, s_base, s_first);
}

// ---- statistics ----------------------------------------------------------------------------------------------------
// sum x per (cluster, side) key on the work list of stats_worklist_kernel.  A CTA takes one item (a run of <= chunk
// points of one key) at a time and adds its entries into a Float32 shared-memory copy of the key's D-vector, which it
// then adds, entry by non-zero entry, to the key's Float64 accumulator and clears.  With integral counts every partial
// stays an integer below 2^24 (as the dense kernel's per-item partials), so the result is exact in any order.
__global__ void __launch_bounds__(256) mnm_sparse_stats_kernel(const StatsArgs a, const MnmSparse sp) {
  extern __shared__ float s_acc[];   // [D]
  __shared__ int s_item;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int d = tid; d < a.D; d += 256) s_acc[d] = 0.f;
  const int n_items = *a.n_items;
  for (;;) {
    __syncthreads();   // s_acc cleared, s_item consumed
    if (tid == 0) s_item = atomicAdd(a.next_item, 1);
    __syncthreads();
    const int u = s_item;
    if (u >= n_items) break;
    const StatsItem item = a.items[u];
    for (int p = item.begin + warp; p < item.end; p += 8) {
      const int32_t i = __ldg(a.perm2 + p);
      const int64_t b = __ldg(sp.ptr + i), e = __ldg(sp.ptr + i + 1);
      for (int64_t q = b + lane; q < e; q += 32) atomicAdd(&s_acc[__ldg(sp.idx + q)], __ldg(sp.val + q));
    }
    __syncthreads();
    double* dst = a.acc + (size_t)item.key * a.rec + 1;
    for (int d = tid; d < a.D; d += 256) {
      const float v = s_acc[d];
      if (v != 0.f) {
        atomicAdd(dst + d, (double)v);
        s_acc[d] = 0.f;
      }
    }
  }
}

// ---- predict -------------------------------------------------------------------------------------------------------
// mnm_score_kernel on sparse points: one warp per point, lanes over the stored entries; the dot product accumulates in
// Float64, is rounded to Float32 and gets log w in Float32.  The CTA keeps its tile of KC clusters in shared memory.
__global__ void __launch_bounds__(256) mnm_sparse_score_kernel(const MnmScoreArgs a, const MnmSparse sp) {
  extern __shared__ double tile[];   // [KC][D]
  const int D = a.D, k0 = blockIdx.y * a.KC, kc = min(a.KC, a.K - k0);
  for (int e = threadIdx.x; e < kc * D; e += blockDim.x) tile[e] = a.logp[(size_t)k0 * D + e];
  __syncthreads();
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
  for (int64_t i = (int64_t)blockIdx.x * 8 + wl; i < a.n; i += (int64_t)gridDim.x * 8) {
    const int64_t b = __ldg(sp.ptr + i), e = __ldg(sp.ptr + i + 1);
    for (int k = 0; k < kc; ++k) {
      const double* lp = tile + (size_t)k * D;
      double s = 0.0;
      for (int64_t q = b + lane; q < e; q += 32) {
        const float c = __ldg(sp.val + q);
        if (c != 0.f) s = fma((double)c, lp[__ldg(sp.idx + q)], s);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) a.score[(size_t)i * a.K + k0 + k] = __fadd_rn((float)s, __ldg(a.logw + k0 + k));
    }
  }
}
