// K2: tensor-core form of the fused Gaussian log-likelihood + label draw (D = 32).
//
//   sample_labels_worker!        src/local_clusters_actions.jl:112-134
//   log_likelihood!(mv_gaussian) src/distributions/mv_gaussian.jl:21-25
//   sample_log_cat_array!        src/utils.jl:19-31
//
// TF32 screen + FP32 refine (the "error-compensated TF32/FP32 split" of the north star, organised so
// that every value that can influence a draw is an exact-FP32 reference value):
//
//  1. SCREEN on tcgen05: for a tile of 128 points (TMA, 128B-swizzled) and 8 clusters at a time,
//     Y[128 x 256] = X[128 x 32] . W^T with W = the 8 upper-triangular factors U_k stacked K-major in
//     shared memory, accumulated in TMEM (kind::tf32, 4 k-steps).  The epilogue warps read the
//     accumulator with tcgen05.ld and form q~_k = |U_k x - U_k mu_k|^2 per (point, cluster).
//     TF32 keeps 10 mantissa bits of x, so q~ carries an error that is BOUNDED per point:
//       |y~ - y|_2 <= e_k := 2^-9 |U_k|_F |x|_2   =>   |q~_k - q_k| <= 2 sqrt(q~_k) e_k + e_k^2.
//  2. REFINE on the FMA pipe: cluster k is a candidate of the point iff its upper bound reaches
//     within DELTA = 30 of the best lower bound.  Only candidates (typically 1-2 of K) are evaluated
//     exactly -- z = x - mu in Float32, |U z|^2 with packed FFMA2, r = -c - q/2 + log w, the
//     reference's own operations -- and only they enter the draw.  A non-candidate has
//     p_k < e^-30 ~ 1e-13 of the largest term; dropping it moves no cumulative boundary by more
//     than 1e-13, eight orders of magnitude inside the documented near-tie band.
//     Points with a NaN/Inf screen value fall back to "all clusters are candidates".
//
// Warp roles (one persistent CTA per SM, 320 threads): warps 0/1 = control warp of point-group
// 0/1 (TMA producer + tcgen05.mma issuer), warps 2-5 / 6-9 = epilogue+refine+draw warps of group
// 0/1 (thread = TMEM lane = point).  The two groups work on alternating tiles so that the tensor
// pipe, the TMEM loads and the FMA-bound refinement of different tiles overlap.
#pragma once
#include <cuda.h>

#include "common.cuh"
#include "kernels_gauss.cuh"
#include "tcgen05.cuh"

#define TC_D 32
#define TC_TILE 128                 // points per tile = TMEM lanes
#define TC_NCL 4                    // clusters per MMA chunk (4 * 32 = 128 accumulator columns)
#define TC_CHUNK_BYTES (TC_NCL * TC_D * TC_D * 4)
#define TC_STAGE_BYTES (TC_TILE * TC_D * 4)
#define TC_THREADS 320
#define TC_MAX_K 23
#define TC_DELTA 30.0f

struct GaussTcArgs {
  int64_t n;
  int K;
  const float* wmat;   // [K padded to a multiple of 4][32][32] factors U_k, rows (k, i), zero padded
  const float* bvec;   // [K][32]  U_k mu_k
  const float* mu;     // [K][32]
  const float* cst;    // [3K]   c of every distribution (cluster dist = 3k)
  const float* logw;   // [K]
  const float* fro;    // [K]    |U_k|_F
  int32_t* labels;
  int32_t* hist;
  const double* u_inj;
  uint64_t seed;
  uint32_t call;
  int64_t goff;
  int final_iter;
  int64_t ntiles;
  int32_t* stats;      // optional [2]: #points, #candidate evaluations (diagnostics)
};

// shared-memory carve-up (bytes), shared by host and device
struct GaussTcSmem {
  int nch;
  size_t w, stages, bvec, mu, consts, rs, pairs, cnt, hist, bars, total;
  __host__ __device__ explicit GaussTcSmem(int K) {
    nch = (K + TC_NCL - 1) / TC_NCL;
    size_t o = 0;
    w = o;       o += (size_t)nch * TC_CHUNK_BYTES;          // factors (1024-aligned chunks)
    stages = o;  o += 4 * (size_t)TC_STAGE_BYTES;            // X stages, 2 per group
    bvec = o;    o += 4096 + (size_t)nch * 4096;            // bias k-step: A_aug [128 x 8], B_aug [nch][128 x 8]
    mu = o;      o += (size_t)K * TC_D * 4;
    consts = o;  o += (size_t)4 * K * 4;                     // c, log w, |U|_F, pad
    rs = o;      o += 2 * (size_t)K * TC_TILE * 4;           // per group [K][128]
    pairs = o;   o += 2 * (size_t)K * TC_TILE * 2;           // per group candidate (row, k) list, uint16
    o = (o + 15) & ~(size_t)15;
    cnt = o;     o += 2 * 2 * 32 * 4;                        // per group: counts[32], offsets[32]
    hist = o;    o += (size_t)((K + 3) & ~3) * 4;
    o = (o + 15) & ~(size_t)15;
    bars = o;    o += 16 * 8 + 16;
    total = o;
  }
};

// exact q = |U_k (x - mu_k)|^2 from the K-major (row = i) swizzled factor rows in shared memory
__device__ __forceinline__ float gauss_tc_exact_q(const float* wk, const float* mu, const float (&x)[TC_D]) {
  f32x2_t z2[TC_D / 2];
#pragma unroll
  for (int c = 0; c < TC_D / 4; ++c) {
    const float4 m = *reinterpret_cast<const float4*>(mu + 4 * c);
    z2[2 * c] = f2_pack(x[4 * c] - m.x, x[4 * c + 1] - m.y);
    z2[2 * c + 1] = f2_pack(x[4 * c + 2] - m.z, x[4 * c + 3] - m.w);
  }
  float q0 = 0.f, q1 = 0.f;
#pragma unroll
  for (int i = 0; i < TC_D; ++i) {
    const float* row = wk + i * TC_D;
    f32x2_t acc = 0ull;
#pragma unroll
    for (int c = i >> 2; c < TC_D / 4; ++c) {
      const ulonglong2 u = *reinterpret_cast<const ulonglong2*>(row + ((c ^ (i & 7)) << 2));
      acc = f2_fma(u.x, z2[2 * c], acc);
      acc = f2_fma(u.y, z2[2 * c + 1], acc);
    }
    float lo, hi;
    f2_unpack(acc, lo, hi);
    const float y = lo + hi;
    if (i & 1) q1 = fmaf(y, y, q1); else q0 = fmaf(y, y, q0);
  }
  return q0 + q1;
}

__device__ __forceinline__ void group_barrier(int g) { asm volatile("bar.sync %0, 128;" ::"r"(g + 1) : "memory"); }
// barrier of the 128 threads of a point-group that also ORs a predicate across them
__device__ __forceinline__ bool group_any(int g, bool pred) {
  int r;
  asm volatile(
      "{\n\t"
      ".reg .pred p, q;\n\t"
      "setp.ne.b32 q, %1, 0;\n\t"
      "bar.red.or.pred p, %2, 128, q;\n\t"
      "selp.s32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(r)
      : "r"((int)pred), "r"(g + 1)
      : "memory");
  return r != 0;
}

__global__ void __launch_bounds__(TC_THREADS, 1)
gauss_label_tc_kernel(const __grid_constant__ CUtensorMap tmap_x, const GaussTcArgs a) {
  extern __shared__ __align__(1024) uint8_t tc_smem[];
  uint8_t* const smem = tc_smem;
  const int K = a.K;
  const GaussTcSmem L(K);
  const int nch = L.nch;
  float* wsm = reinterpret_cast<float*>(smem + L.w);
  uint8_t* stage0 = smem + L.stages;
  float* aaug = reinterpret_cast<float*>(smem + L.bvec);            // [128 rows][8]: (1, 1, 0, ...)
  float* baug = aaug + 1024;                                        // [nch][128 rows][8]: (-b_hi, -b_lo, 0, ...)
  float* musm = reinterpret_cast<float*>(smem + L.mu);
  float* csm = reinterpret_cast<float*>(smem + L.consts);  // c_k
  float* lwsm = csm + K;                                   // log w_k
  float* frosm = lwsm + K;                                 // |U_k|_F
  float* ccsm = frosm + K;                                 // log w_k - c_k
  float* rs_all = reinterpret_cast<float*>(smem + L.rs);
  uint16_t* pairs_all = reinterpret_cast<uint16_t*>(smem + L.pairs);
  int* cnt_all = reinterpret_cast<int*>(smem + L.cnt);
  int* hs = reinterpret_cast<int*>(smem + L.hist);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
  uint64_t* full = bars;              // [4]     TMA landed in stage s
  uint64_t* empty = bars + 4;         // [4]     stage s released by its 128 consumers
  uint64_t* tfull = bars + 8;         // [2][2]  accumulator buffer (group, b) ready
  uint64_t* tempty = bars + 12;       // [2][2]  accumulator buffer (group, b) drained
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 16);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0) {
    for (int i = 0; i < 4; ++i) {
      tc::mbar_init(&full[i], 1);
      tc::mbar_init(&empty[i], 128);
      tc::mbar_init(&tfull[i], 1);
      tc::mbar_init(&tempty[i], 128);
    }
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc(tmem_ptr, 512);
  // ---- stage the factors once per CTA, applying the 128B swizzle the MMA descriptor expects ----
  for (int e = tid; e < nch * TC_NCL * TC_D * (TC_D / 4); e += TC_THREADS) {
    const int r = e >> 3, c = e & 7;  // row (k * 32 + i), 16-byte chunk
    const float4 v = __ldg(reinterpret_cast<const float4*>(a.wmat) + e);
    *reinterpret_cast<float4*>(wsm + (size_t)r * TC_D + ((c ^ (r & 7)) << 2)) = v;
  }
  // bias k-step: Y -= U mu is folded into the MMA as one more k-step whose A operand is the constant
  // (1, 1, 0, ..) and whose B operand holds -b split into a TF32-exact high part and the remainder
  for (int e = tid; e < 1024 + nch * 1024; e += TC_THREADS) aaug[e] = 0.f;
  __syncthreads();
  for (int r = tid; r < TC_TILE; r += TC_THREADS) {
    float* p = aaug + (r >> 3) * 64 + (r & 7) * 4;   // (r/8)*256 B + (r%8)*16 B
    p[0] = 1.f;
    p[1] = 1.f;
  }
  for (int e = tid; e < K * TC_D; e += TC_THREADS) {
    musm[e] = __ldg(a.mu + e);
    const float b = __ldg(a.bvec + e);
    uint32_t ub = __float_as_uint(b);
    ub += 0xFFFu + ((ub >> 13) & 1u);
    ub &= 0xFFFFE000u;                                // round to TF32 (10 explicit mantissa bits)
    const float bhi = (b == b && fabsf(b) < CUDART_INF_F) ? __uint_as_float(ub) : b;
    const float blo = b - bhi;
    const int c = e / (TC_NCL * TC_D), rl = e - c * (TC_NCL * TC_D);   // chunk, row within the chunk
    float* p = baug + c * 1024 + (rl >> 3) * 64 + (rl & 7) * 4;
    p[0] = -bhi;
    p[1] = -blo;
  }
  for (int k = tid; k < K; k += TC_THREADS) {
    csm[k] = __ldg(a.cst + 3 * k);
    lwsm[k] = __ldg(a.logw + k);
    frosm[k] = __ldg(a.fro + k);
    ccsm[k] = __ldg(a.logw + k) - __ldg(a.cst + 3 * k);
    hs[k] = 0;
  }
  tc::fence_proxy_async();  // generic-proxy writes of W must be visible to the tensor core's async proxy
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp < 2) {
    // =============================== control warp of group g ===============================
    const int g = warp;
    {   // all 32 lanes run the loop (warp-uniform control flow), one elected lane issues: see umma_tf32_*_w
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      int li = 0;
      uint32_t cc = 0;  // chunk counter of this group
      int64_t tile = (int64_t)blockIdx.x + (int64_t)g * gridDim.x;
      const int64_t tstep = 2 * (int64_t)gridDim.x;
      if (tile < a.ntiles && lane == 0) {  // prologue: first tile of this group
        tc::mbar_arrive_expect_tx(&full[g * 2], TC_STAGE_BYTES);
        tc::tma_load_2d(stage0 + (size_t)(g * 2) * TC_STAGE_BYTES, &tmap_x, &full[g * 2], 0, (int)(tile * TC_TILE));
      }
      const uint64_t aaug_desc = tc::smem_desc_k_noswz(tc::smem_u32(aaug));
      for (; tile < a.ntiles; tile += tstep, ++li) {
        const int s = g * 2 + (li & 1);
        tc::mbar_wait(&full[s], (li >> 1) & 1);
        tc::tc_fence_after();
        const uint64_t adesc = tc::smem_desc_k128(tc::smem_u32(stage0 + (size_t)s * TC_STAGE_BYTES));
        for (int c = 0; c < nch; ++c, ++cc) {
          const int b = cc & 1;
          tc::mbar_wait(&tempty[g * 2 + b], ((cc >> 1) & 1) ^ 1);   // epilogue drained this buffer
          tc::tc_fence_after();
          const int ncl = min(TC_NCL, K - c * TC_NCL);
          const uint64_t bdesc = tc::smem_desc_k128(tc::smem_u32(wsm) + c * TC_CHUNK_BYTES);
          const uint32_t idesc = tc::idesc_tf32(ncl * TC_D);
          const uint32_t tmem_d = tmem_u + g * 256 + b * 128;
          tc::umma_tf32_first_w(tmem_d, adesc, bdesc, idesc);
#pragma unroll
          for (int ks = 1; ks < TC_D / 8; ++ks)   // 32-byte k-steps inside the 128-byte swizzled rows
            tc::umma_tf32_acc_w(tmem_d, adesc + ks * 2, bdesc + ks * 2, idesc);
          tc::umma_tf32_acc_w(tmem_d, aaug_desc, tc::smem_desc_k_noswz(tc::smem_u32(baug) + c * 4096), idesc);   // Y -= U mu
          tc::umma_commit_w(&tfull[g * 2 + b]);
        }
        // prefetch this group's next tile into its other stage (freed when tile li-1 was finished)
        const int64_t nt = tile + tstep;
        if (nt < a.ntiles) {
          const int ns = g * 2 + ((li + 1) & 1);
          tc::mbar_wait(&empty[ns], (((li + 1) >> 1) & 1) ^ 1);
          if (lane == 0) {
            tc::mbar_arrive_expect_tx(&full[ns], TC_STAGE_BYTES);
            tc::tma_load_2d(stage0 + (size_t)ns * TC_STAGE_BYTES, &tmap_x, &full[ns], 0, (int)(nt * TC_TILE));
          }
          __syncwarp();
        }
      }
    }
  } else {
    // ======================= epilogue + refine + draw warps of group g =======================
    const int g = (warp - 2) >> 2;
    const int gt = tid - 64 - g * 128;                     // thread index within the group
    const int row = ((warp & 3) << 5) | lane;              // TMEM lane == point within the tile
    const uint32_t tmem_row = tmem_base + ((uint32_t)((warp & 3) << 5) << 16) + g * 256;
    float* rsg = rs_all + (size_t)g * K * TC_TILE;         // [K][128]
    float* rs = rsg + row;                                 // this point's column: element k at rs[k * 128]
    uint16_t* pairs = pairs_all + (size_t)g * K * TC_TILE;
    int* cnt = cnt_all + g * 64;                           // [0..31] counts -> cursors, [32] total
    int li = 0;
    uint32_t cc = 0;
    int ncand_total = 0, npts_total = 0;
    for (int64_t tile = (int64_t)blockIdx.x + (int64_t)g * gridDim.x; tile < a.ntiles; tile += 2 * (int64_t)gridDim.x, ++li) {
      const int s = g * 2 + (li & 1);
      // ---- screen: q~_k for every cluster from the TMEM accumulators (kept in registers: the
      //      chunk / cluster loops are fully unrolled so that qt[] is indexed at compile time) ----
      float qt[TC_MAX_K + 1];
#pragma unroll
      for (int c = 0; c < (TC_MAX_K + TC_NCL) / TC_NCL; ++c) {
        if (c < nch) {
          const int b = cc & 1;
          tc::mbar_wait(&tfull[g * 2 + b], (cc >> 1) & 1);
          tc::tc_fence_after();
          const int ncl = min(TC_NCL, K - c * TC_NCL);
          const uint32_t taddr = tmem_row + b * 128;
#pragma unroll
          for (int kl = 0; kl < TC_NCL; kl += 2) {
            if (kl < ncl) {
              uint32_t v0[32], v1[32];
              tc::tmem_ld32(taddr + kl * TC_D, v0);
              if (kl + 1 < ncl) tc::tmem_ld32(taddr + (kl + 1) * TC_D, v1);
              tc::tmem_ld_wait();
              qt[c * TC_NCL + kl] = gauss_tc_screen_q(v0);
              if (kl + 1 < ncl) qt[c * TC_NCL + kl + 1] = gauss_tc_screen_q(v1);
            }
          }
          tc::tc_fence_before();
          tc::mbar_arrive(&tempty[g * 2 + b]);
          ++cc;
        }
      }
      // ---- the point itself (the TMA wrote it with the 128B swizzle) ----
      tc::mbar_wait(&full[s], (li >> 1) & 1);
      const float* stage = reinterpret_cast<const float*>(stage0 + (size_t)s * TC_STAGE_BYTES);
      const int64_t i = tile * TC_TILE + row;
      const bool valid = i < a.n;
      uint32_t mask = 0;
      bool weird = false;   // a NaN / Inf screen value: every cluster is refined, general draw
      {
        const float* xrow = stage + row * TC_D;
        float xn = 0.f;
#pragma unroll
        for (int c = 0; c < TC_D / 4; ++c) {
          const float4 v = *reinterpret_cast<const float4*>(xrow + ((c ^ (row & 7)) << 2));
          xn = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, xn))));
        }
        // ---- candidates: upper bound of r_k within DELTA of the best lower bound ----
        const float xnorm = sqrtf(xn) * (1.f / 512.f);   // 2^-9 |x|
        float best_lo = -CUDART_INF_F;
#pragma unroll
        for (int k = 0; k < TC_MAX_K; ++k) {
          if (k < K) {
            const float e = xnorm * frosm[k];
            float sq;
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(fmaxf(qt[k], 0.f)));
            const float dr = fmaf(1.01f * sq, e, fmaf(0.5f * e, e, 0.01f));   // |r~ - r| <= sqrt(q~) e + e^2/2
            const float rt = fmaf(-0.5f, qt[k], ccsm[k]);
            weird |= !(fabsf(rt) < CUDART_INF_F) || !(dr < CUDART_INF_F);
            best_lo = fmaxf(best_lo, rt - dr);
            qt[k] = rt + dr;                               // upper bound of r_k
          }
        }
        const float thr = best_lo - TC_DELTA;
#pragma unroll
        for (int k = 0; k < TC_MAX_K; ++k)
          if (k < K && valid && (weird || qt[k] >= thr)) mask |= 1u << k;
      }
      // A point with a single candidate is decided: every other cluster has weight exactly 0 in the
      // draw, so its label is that cluster whatever the exact value is -- no refinement needed.
      const bool multi = __popc(mask) > 1;
      const uint32_t rmask = multi ? mask : 0u;
      // ---- refine only if some point of the group has several candidates (rare once clusters separate) ----
      int npairs = 0;
      if (group_any(g, multi)) {
        // ---- regroup the (point, cluster) candidates by cluster so that a warp refines one cluster ----
        // (counting sort over <= 24 keys in shared memory: count, prefix, scatter)
        if (gt < 32) cnt[gt] = 0;
        group_barrier(g);
        for (uint32_t m = rmask; m; m &= m - 1) atomicAdd(&cnt[__ffs(m) - 1], 1);
        group_barrier(g);
        if (gt == 0) {
          int run = 0;
          for (int k = 0; k < K; ++k) {
            const int c = cnt[k];
            cnt[k] = run;        // becomes the scatter cursor of cluster k
            run += c;
          }
          cnt[32] = run;
        }
        group_barrier(g);
        for (uint32_t m = rmask; m; m &= m - 1) {
          const int k = __ffs(m) - 1;
          pairs[atomicAdd(&cnt[k], 1)] = (uint16_t)((row << 5) | k);
        }
        group_barrier(g);
        npairs = cnt[32];
        for (int idx = gt; idx < npairs; idx += 128) {
          const uint32_t pr = pairs[idx];
          const int prow = pr >> 5, k = pr & 31;
          float x[TC_D];
          const float* xrow = stage + prow * TC_D;
#pragma unroll
          for (int c = 0; c < TC_D / 4; ++c) {
            const float4 v = *reinterpret_cast<const float4*>(xrow + ((c ^ (prow & 7)) << 2));
            x[4 * c] = v.x; x[4 * c + 1] = v.y; x[4 * c + 2] = v.z; x[4 * c + 3] = v.w;
          }
          const float q = gauss_tc_exact_q(wsm + (size_t)k * TC_D * TC_D, musm + k * TC_D, x);
          rsg[k * TC_TILE + prow] = gauss_finish(csm[k], q, lwsm[k]);
          ++ncand_total;
        }
        group_barrier(g);
      }
      // the stage can be refilled now
      tc::mbar_arrive(&empty[s]);
      // ---- draw ----
      if (valid) {
        int lab;
        if (!multi) {
          lab = __ffs(mask) - 1;
          // The walk of utils.jl:29 stops at i = 1 when t = u * sum(w) is 0, i.e. for the uniform u == 0.
          // Injected uniforms are checked.  A Philox uniform is 0 with probability 2^-53 per draw (once in
          // ~10^7 runs of 10^3 iterations over 10^6 points); evaluating the generator for every decided
          // point only to test for it costs ~100 instructions per point, so that case is not reproduced.
          if (a.u_inj != nullptr && lab > 0 && !a.final_iter && a.u_inj[i] == 0.0) lab = 0;
        } else if (a.final_iter) {
          if (weird) {
            lab = dpmm_draw_argmax(rs, TC_TILE, K);
          } else {   // first maximum among the candidates (a non-candidate is > 30 below the maximum)
            lab = 0;
            float bv = -CUDART_INF_F;
            for (uint32_t m = mask; m; m &= m - 1) {
              const int k = __ffs(m) - 1;
              const float v = rs[k * TC_TILE];
              if (v > bv) {
                bv = v;
                lab = k;
              }
            }
          }
        } else {
          const double u = dpmm_uniform(a.u_inj, i, a.seed, DPMM_STREAM_LABEL, a.call, (uint64_t)(a.goff + i));
          lab = weird ? dpmm_draw_inverse_cdf(rs, TC_TILE, K, u) : dpmm_draw_inverse_cdf_masked(rs, TC_TILE, K, mask, u);
        }
        a.labels[i] = lab;
        atomicAdd(&hs[lab], 1);
        ++npts_total;
      }
    }
    if (a.stats != nullptr) {
      atomicAdd(&a.stats[0], npts_total);
      atomicAdd(&a.stats[1], ncand_total);
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc(tmem_base, 512);
  for (int k = tid; k < K; k += TC_THREADS)
    if (hs[k] != 0) atomicAdd(&a.hist[k], hs[k]);
}
