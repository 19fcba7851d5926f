// Label grouping (device counting sort) and stage 4 (integer relabelling).
//
// The reference finds the members of a cluster with a boolean scan `labels .== i` over all points,
// once per cluster and per operation (local_clusters_actions.jl:77-78, 159-160, 270-272, 298-302),
// i.e. O(n*K) traffic.  Here the point indices are bucketed once per label change (histogram ->
// exclusive scan -> scatter), and every per-cluster consumer (sub-label draw, statistics) walks the
// sorted permutation instead.
#pragma once
#include "common.cuh"

// hist[k] = #points with label k (used when the labels changed outside sample_labels).
__global__ void label_hist_kernel(const int32_t* __restrict__ labels, int64_t n, int K, int32_t* hist) {
  extern __shared__ int hs[];
  for (int k = threadIdx.x; k < K; k += blockDim.x) hs[k] = 0;
  __syncthreads();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int l = labels[i];
    if (l >= 0 && l < K) atomicAdd(&hs[l], 1);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < K; k += blockDim.x)
    if (hs[k] != 0) atomicAdd(&hist[k], hs[k]);
}

// Single CTA: seg_off = exclusive scan of hist (K+1 entries), scatter cursors, and the left/right
// cursors consumed by the sub-label kernel.
__global__ void label_scan_kernel(const int32_t* __restrict__ hist, int K, int32_t* seg_off,
                                  int32_t* scat_cursor, int32_t* lr_cursor) {
  __shared__ int warp_tot[32];
  __shared__ int carry;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int k0 = 0; k0 < K; k0 += blockDim.x) {
    const int k = k0 + tid;
    const int v = (k < K) ? hist[k] : 0;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      int w = (lane < (blockDim.x >> 5)) ? warp_tot[lane] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, w, o);
        if (lane >= o) w += t;
      }
      warp_tot[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const int excl = carry + (wid ? warp_tot[wid - 1] : 0) + inc - v;
    if (k < K) {
      seg_off[k] = excl;
      scat_cursor[k] = excl;
      lr_cursor[2 * k] = excl;
      lr_cursor[2 * k + 1] = excl + v;
    }
    __syncthreads();
    if (tid == 0) carry += warp_tot[(blockDim.x >> 5) - 1];
    __syncthreads();
  }
  if (tid == 0) seg_off[K] = carry;
}

// perm <- point indices bucketed by label.  Each CTA ranks its points with shared-memory counters
// and reserves one contiguous range per (CTA, label) with a single global atomic.
#define SCATTER_PPT 8
// `zero` / `zero2` (optional): buffers the NEXT kernel expects cleared (the statistics accumulators and left
// counts of the fused sub-label + statistics kernel) -- cleared here instead of by two memset launches; `zero3`
// (optional): one more double, the risk counter of the statistics finalise that follows the fused kernel.
// `moved` (optional): the number of points whose label changed since `perm` was last sorted.  When it is 0, perm
// is still a valid sort of the labels (the order inside a bucket is arbitrary anyway: ranks come from atomics) and
// the cursors, which only the scatter consumes, keep their scan: the kernel only clears the buffers above.
__global__ void label_scatter_kernel(const int32_t* __restrict__ labels, int64_t n, int K,
                                     int32_t* cursor, int32_t* perm, double* zero, int64_t nzero,
                                     int32_t* zero2, int nzero2, double* zero3, const int32_t* moved) {
  extern __shared__ int sm[];
  pdl_wait();
  pdl_launch_dependents();
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < nzero; e += (int64_t)gridDim.x * blockDim.x) zero[e] = 0.0;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nzero2; e += gridDim.x * blockDim.x) zero2[e] = 0;
  if (zero3 != nullptr && blockIdx.x == 0 && threadIdx.x == 0) *zero3 = 0.0;
  if (moved != nullptr && *moved == 0) return;
  int* cnt = sm;
  int* basev = sm + K;
  const int T = blockDim.x, tid = threadIdx.x;
  for (int k = tid; k < K; k += T) cnt[k] = 0;
  __syncthreads();
  const int64_t base = (int64_t)blockIdx.x * T * SCATTER_PPT;
  int lab[SCATTER_PPT], rank[SCATTER_PPT];
#pragma unroll
  for (int j = 0; j < SCATTER_PPT; ++j) {
    const int64_t i = base + (int64_t)j * T + tid;
    lab[j] = (i < n) ? labels[i] : -1;   // all eight loads in flight before the (branchy) ranking below
  }
#pragma unroll
  for (int j = 0; j < SCATTER_PPT; ++j) {
    // A warp whose 32 points share their label (label-sorted or blocked data) reserves its ranks with
    // ONE shared-memory atomic instead of serialising 32 on the same counter; mixed warps rank per lane.
    const int lane = tid & 31;
    const int lab0 = __shfl_sync(0xffffffffu, lab[j], 0);
    if (__all_sync(0xffffffffu, lab[j] == lab0)) {
      int b0 = 0;
      if (lane == 0 && lab0 >= 0) b0 = atomicAdd(&cnt[lab0], 32);
      rank[j] = __shfl_sync(0xffffffffu, b0, 0) + lane;
    } else if (lab[j] >= 0) {
      rank[j] = atomicAdd(&cnt[lab[j]], 1);
    }
  }
  __syncthreads();
  for (int k = tid; k < K; k += T) {
    const int c = cnt[k];
    basev[k] = c ? atomicAdd(&cursor[k], c) : 0;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < SCATTER_PPT; ++j) {
    const int64_t i = base + (int64_t)j * T + tid;
    if (lab[j] >= 0) perm[basev[lab[j]] + rank[j]] = (int32_t)i;
  }
}

// ---------------------------------------------------------------------------------------------
// Stage 4: every relabel operation of the reference is a per-point function of (label, sub-label)
// and one random bit, so the host composes each operation into small lookup tables and one pass
// applies them:
//   split_cluster_local_worker!    local_clusters_actions.jl:265-278
//   merge_clusters_worker!         :293-304
//   remove_empty_clusters_worker!  :446-455
//   reset_bad_clusters_worker! / rand_subclusters_labels! / split_first_cluster_worker!  :257-261, 474-488
//     lut_l[k], lut_r[k] : new label of a point with old label k and sub-label left / right
//     rule[k]            : 0 keep sub-label, 1 set left, 2 set right, 3 fresh rand(1:2)
// ---------------------------------------------------------------------------------------------
__global__ void relabel_kernel(int32_t* labels, uint8_t* sub, int64_t n, int K,
                               const int32_t* __restrict__ lut_l, const int32_t* __restrict__ lut_r,
                               const uint8_t* __restrict__ rule, const uint8_t* r_inj, uint64_t seed,
                               uint32_t call, int64_t goff) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int k = labels[i];
    if (k < 0 || k >= K) continue;
    const int s = sub[i];
    const int nk = s ? lut_r[k] : lut_l[k];
    if (nk != k) labels[i] = nk;
    const int r = rule[k];
    if (r == 1) sub[i] = 0;
    else if (r == 2) sub[i] = 1;
    else if (r == 3) sub[i] = (uint8_t)dpmm_randbit(r_inj, i, seed, call, (uint64_t)(goff + i));
  }
}

// labels = rand(1:init_clusters) (+1 with the outlier component), dp-parallel-sampling.jl:49.
__global__ void init_labels_kernel(int32_t* labels, int64_t n, int init_clusters, int shift,
                                   uint64_t seed, uint32_t call, int64_t goff) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const double u = philox_to_uniform(philox_draw(seed, DPMM_STREAM_INIT, call, (uint64_t)(goff + i)));
    int l = (int)(u * (double)init_clusters);
    if (l > init_clusters - 1) l = init_clusters - 1;
    labels[i] = l + shift;
  }
}

// ---------------------------------------------------------------------------------------------
// Label gather / restore at the boundary (Array(group.labels), dp-parallel-sampling.jl:218,276,371; resume
// :437-438): the widening to 1-based Int64, the narrowing and the range check run on the device, so the host
// side of dpmm_get/set_labels is one copy of the caller's own array, not a scalar loop over n points.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void widen_labels_kernel(const T* __restrict__ in, int64_t n, int64_t* __restrict__ out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (int64_t)in[i] + 1;
}
// out[i] = in[i] - 1; status[0] = max label seen, status[1] = 1 if any label is outside [1, hi]
template <typename T>
__global__ void narrow_labels_kernel(const int64_t* __restrict__ in, int64_t n, int64_t hi, T* __restrict__ out,
                                     int32_t* __restrict__ status) {
  int mx = 0, bad = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t v = in[i];
    if (v < 1 || v > hi) bad = 1;
    else {
      out[i] = (T)(v - 1);
      mx = max(mx, (int)v);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    bad |= __shfl_xor_sync(0xffffffffu, bad, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (mx) atomicMax(&status[0], mx);
    if (bad) atomicOr(&status[1], 1);
  }
}
// multinomial create: are all counts integral and below 2^11 in magnitude (exact in TF32)?  flag[0] |= 1 if not
__global__ void tf32_exact_scan_kernel(const float* __restrict__ x, int64_t n, int32_t* __restrict__ flag) {
  int bad = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = x[i];
    if (!(v == truncf(v) && v > -2048.f && v < 2048.f)) bad = 1;
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(flag, 1);
}

// x_pad[i][0..Dp) = (x[i][0..D), 0, ...): the one-time widening of the points of a context whose feature dimension
// has no instantiated kernels (zero features with unit precision change no likelihood and no statistic)
__global__ void pad_points_kernel(const float* __restrict__ x, int64_t n, int D, int Dp, float* __restrict__ xp) {
  const int64_t tot = n * Dp;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t i = e / Dp;
    const int j = (int)(e - i * Dp);
    xp[e] = j < D ? x[i * D + j] : 0.f;
  }
}
