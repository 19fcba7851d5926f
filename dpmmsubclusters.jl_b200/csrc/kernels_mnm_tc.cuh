// K3 on tensor cores: fused multinomial log-likelihood + label draw (D % 4 == 0, D <= 128, K <= 32).
//
//   log_likelihood!(r, x, ::multinomial_dist)   src/distributions/multinomial_dist.jl:13-15
//       r[j] = sum_d alpha_d x[d, j]      -- "a GEMM of counts against log-probabilities"
//   sample_labels_worker! / sample_log_cat_array!   (as in kernels_mnm.cuh)
//
// R[128 x K] = X[128 x D] . A^T on tcgen05 (kind::tf32, FP32 accumulation in TMEM).  The counts are
// small integers (checked on upload: |x| < 2^11, integral), hence exact in TF32, and every Float32
// log-probability is split on the host into three TF32-exact terms alpha = a_hi + a_lo + a_lolo
// (11 + 11 + 2 significant bits), so all 3*D products per (point, cluster) are exact in Float32 and
// the result differs from the reference's SGEMV only by Float32 summation order -- no screening or
// refinement is needed here.  X streams through a 2-stage TMA ring (128B-swizzled 32-column panels),
// which makes the kernel HBM-bound: one pass over X, K log-likelihoods per point straight out of TMEM.
//
// Warp roles (persistent CTA per SM, 576 threads): warp 0 = TMA producer, warp 1 = tcgen05.mma issuer,
// warps 2-17 = four draw groups, group g on the tiles t = g (mod 4) and the accumulator buffer g (thread = TMEM
// lane = point).  The draw is what the kernel spends its instructions on (62 % of them in the reference-exact
// softmax + inverse-CDF walk over K entries, call-site profile of capture r2k), so the number of draw warps sets
// the pace until HBM does.
#pragma once
#include "common.cuh"
#include "tcgen05.cuh"

#define MTC_TILE 128
#define MTC_N 32                  // accumulator columns per tile (clusters, zero padded)
#define MTC_MAX_K 32
#define MTC_MAX_D 128
#define MTC_PANEL_BYTES (MTC_TILE * 128)   // one 32-column panel of a tile
#define MTC_NG 4                  // draw groups (4 warps each) when their parr slices fit shared memory, else 2
#define MTC_THREADS(ng) (64 + (ng) * 128)

struct MnmTcArgs {
  int64_t n;
  int D, K, NP;          // NP = ceil(D / 32) panels
  const float* wsplit;   // [3][NP][MTC_N][32]  TF32-exact split of the cluster log-probabilities
  const float* logw;     // [K]
  int32_t* labels;
  int32_t* hist;
  const double* u_inj;
  uint64_t seed;
  uint32_t call;
  int64_t goff;
  int final_iter;
  int sampler;
  int64_t ntiles;
  int NG;                // draw groups: 4 or 2; tile t -> group t % NG (accumulator buffer t % 4)
};

struct MnmTcSmem {
  size_t w, stages, rs, logw, hist, bars, total;
  __host__ __device__ MnmTcSmem(int K, int NP, int NG) {
    size_t o = 0;
    w = o;      o += (size_t)3 * NP * MTC_N * 128;
    stages = o; o += (size_t)2 * NP * MTC_PANEL_BYTES;
    rs = o;     o += (size_t)NG * K * MTC_TILE * 4;
    logw = o;   o += (size_t)((K + 3) & ~3) * 4;
    hist = o;   o += (size_t)((K + 3) & ~3) * 4;
    o = (o + 15) & ~(size_t)15;
    bars = o;   o += 16 * 8 + 16;
    total = o;
  }
};

__global__ void __launch_bounds__(MTC_THREADS(MTC_NG), 1)
mnm_label_tc_kernel(const __grid_constant__ CUtensorMap tmap_x, const MnmTcArgs a) {
  extern __shared__ __align__(1024) uint8_t mtc_smem[];
  uint8_t* const smem = mtc_smem;
  const int K = a.K, NP = a.NP;
  const MnmTcSmem L(K, NP, a.NG);
  const int NT = (int)blockDim.x;
  float* wsm = reinterpret_cast<float*>(smem + L.w);
  uint8_t* stage0 = smem + L.stages;
  float* rs_all = reinterpret_cast<float*>(smem + L.rs);
  float* lwsm = reinterpret_cast<float*>(smem + L.logw);
  int* hs = reinterpret_cast<int*>(smem + L.hist);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
  uint64_t* full = bars;          // [2] TMA landed in stage s
  uint64_t* empty = bars + 2;     // [2] stage s consumed by the tensor core
  uint64_t* tfull = bars + 4;     // [4] accumulator buffer ready
  uint64_t* tempty = bars + 8;    // [4] accumulator buffer drained by its 128 readers
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 12);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t stage_bytes = (uint32_t)NP * MTC_PANEL_BYTES;

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      tc::mbar_init(&full[i], 1);
      tc::mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 4; ++i) {
      tc::mbar_init(&tfull[i], 1);
      tc::mbar_init(&tempty[i], 128);
    }
    tc::fence_barrier_init();
  }
  if (warp == 1) tc::tmem_alloc(tmem_ptr, 128);   // 4 buffers x 32 columns
  // log-probability splits, 128B-swizzled rows of 32 floats: [split][panel][cluster row][32]
  for (int e = tid; e < 3 * NP * MTC_N * 8; e += NT) {
    const int r = e >> 3, c = e & 7;
    const float4 v = __ldg(reinterpret_cast<const float4*>(a.wsplit) + e);
    *reinterpret_cast<float4*>(wsm + (size_t)r * 32 + ((c ^ (r & 7)) << 2)) = v;
  }
  for (int k = tid; k < K; k += NT) {
    lwsm[k] = __ldg(a.logw + k);
    hs[k] = 0;
  }
  tc::fence_proxy_async();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (lane == 0) {
      int t = 0;
      for (int64_t tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x, ++t) {
        const int s = t & 1;
        tc::mbar_wait(&empty[s], ((t >> 1) & 1) ^ 1);
        tc::mbar_arrive_expect_tx(&full[s], stage_bytes);
        for (int p = 0; p < NP; ++p)
          tc::tma_load_2d(stage0 + (size_t)s * stage_bytes + (size_t)p * MTC_PANEL_BYTES, &tmap_x, &full[s], 32 * p,
                          (int)(tile * MTC_TILE));
      }
    }
  } else if (warp == 1) {
    // ===================================== MMA issuer =====================================
    // (warp-uniform loop, one elected lane issues inside the instruction: issued from an `if (lane == 0)` branch every
    //  tcgen05.mma costs ~100 cycles of R2UR / ELECT preamble, and 3 x ceil(D / 8) of them per tile paced the kernel)
    {
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc = tc::idesc_tf32(MTC_N);
      const int ksteps = (a.D + 7) >> 3;
      const uint64_t a0 = tc::smem_desc_k128(tc::smem_u32(stage0)), w0 = tc::smem_desc_k128(tc::smem_u32(wsm));
      int t = 0;
      for (int64_t tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x, ++t) {
        const int s = t & 1, b = t & 3;
        tc::mbar_wait(&full[s], (t >> 1) & 1);
        tc::mbar_wait(&tempty[b], ((t >> 2) & 1) ^ 1);
        tc::tc_fence_after();
        const uint64_t ad = a0 + (uint64_t)(s * (stage_bytes >> 4));
        const uint32_t tmem_d = tmem_u + b * MTC_N;
        for (int ks = 0; ks < ksteps; ++ks) {
          const int p = ks >> 2, kk = ks & 3;   // panel, 32-byte k-step inside the 128-byte rows
          const uint64_t adesc = ad + (uint64_t)(p * (MTC_PANEL_BYTES >> 4) + kk * 2);
#pragma unroll
          for (int sp = 0; sp < 3; ++sp) {
            const uint64_t bdesc = w0 + (uint64_t)((sp * NP + p) * ((MTC_N * 128) >> 4) + kk * 2);
            if (ks == 0 && sp == 0) tc::umma_tf32_first_w(tmem_d, adesc, bdesc, idesc);
            else tc::umma_tf32_acc_w(tmem_d, adesc, bdesc, idesc);
          }
        }
        tc::umma_commit_w(&empty[s]);    // the stage may be refilled once these MMAs have read it
        tc::umma_commit_w(&tfull[b]);
      }
    }
  } else {
    // ===================================== draw warps =====================================
    const int g = (warp - 2) >> 2;
    const int row = ((warp & 3) << 5) | lane;
    const uint32_t tmem_row = tmem_base + ((uint32_t)((warp & 3) << 5) << 16);
    float* rs = rs_all + (size_t)g * K * MTC_TILE + row;
    int t = 0;
    for (int64_t tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x, ++t) {
      if ((t & (a.NG - 1)) != g) continue;
      const int b = t & 3;
      tc::mbar_wait(&tfull[b], (t >> 2) & 1);
      tc::tc_fence_after();
      uint32_t v[32];
      tc::tmem_ld32(tmem_row + b * MTC_N, v);
      tc::tmem_ld_wait();
      tc::tc_fence_before();
      tc::mbar_arrive(&tempty[b]);
      const int64_t i = tile * MTC_TILE + row;
      if (i < a.n) {
#pragma unroll
        for (int k = 0; k < MTC_N; ++k)
          if (k < K) rs[k * MTC_TILE] = __fadd_rn(__uint_as_float(v[k]), lwsm[k]);   // parr[:,k] .+= log(w_k)
        int lab;
        if (a.final_iter) {
          lab = dpmm_draw_argmax(rs, MTC_TILE, K);
        } else if (a.sampler == 1) {
          lab = dpmm_draw_gumbel(rs, MTC_TILE, K, a.seed, a.call, (uint64_t)(a.goff + i));
        } else {
          const double u = dpmm_uniform(a.u_inj, i, a.seed, DPMM_STREAM_LABEL, a.call, (uint64_t)(a.goff + i));
          lab = dpmm_draw_inverse_cdf_screened(rs, MTC_TILE, K, u);
        }
        a.labels[i] = lab;
        atomicAdd(&hs[lab], 1);
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc(tmem_base, 128);
  for (int k = tid; k < K; k += NT)
    if (hs[k] != 0) atomicAdd(&a.hist[k], hs[k]);
}
