// Stage 3 on the tensor cores (NIW, D = 32, all clusters): S = X X' of every (cluster, side) run as a
// tcgen05 GEMM whose contraction index is the POINT.
//
//   create_suff_stats_dict_worker            src/local_clusters_actions.jl:149-169
//   create_sufficient_statistics (NIW)       src/priors/niw.jl:42-51      N, sum x, S = X X' (Float64)
//
// The label-sorted, left/right-partitioned permutation perm2 makes every key (2k + side) one
// contiguous run of positions.  A tile = 128 consecutive positions of ONE key.  Its points are
// gathered with cp.async into a swizzled [point][feature] panel, which is exactly the canonical MN-major
// operand layout of 32-bit data (feature = M/N index, contiguous; point = K index, rows of 128 bytes;
// SWIZZLE_128B with 32-byte atomicity).  Every value is split x = h + l with h = tf32(x) (exact
// difference), and ONE instruction shape does the rank-8 update
//        D[64 x 32] += [h | l]'[64 x 8 points] . h[8 points x 32]        (kind::tf32, M = 64, N = 32)
// so that TMEM rows 0-31 hold sum h h' and rows 32-63 hold sum l h'.  The epilogue forms
//        S_ij = (hh')_ij + (lh')_ij + (lh')_ji
// which drops only the l l' term (<= 2^-22 relative per product) and the truncation of l to TF32
// (2^-21), far inside the 1e-4 parity band of the statistics, and adds the Float32 partial of at most
// STC_FLUSH tiles (512 points) to the key's Float64 accumulator.  sum x is accumulated by the gather
// warps while they split the tile.  All sums are taken about a centre c of the key (y = x - c; c = mean
// of the run's first 32 points, stats_centers_kernel) and shifted back in Float64 by the finalise
// kernel: S = sum y y' + c s' + s c' + N c c', s = sum y.  The tensor core accumulates round-toward-
// zero (about 1 ulp per k-step), so without the shift the bias would scale with |mean|^2, not the variance.
//
// Warp roles (288 threads, 2 CTAs per SM): warps 0-3 gather + split (thread = one 16-byte column chunk
// of 8 rows), warp 4 issues the MMAs, warps 5-8 drain the accumulator.  Every CTA owns a contiguous
// range of the tile sequence, so there is no work list and no atomically fetched item; all roles walk
// the same deterministic tile sequence.
#pragma once
#include "tcgen05.cuh"
#include "kernels_stats.cuh"

#define STC_D 32
#define STC_TILE 128
#define STC_STAGES 3
#define STC_FLUSH 4
#define STC_THREADS 288
#define STC_PANEL_BYTES (STC_TILE * STC_D * 4)   // 16 KB: one [128][32] panel
#define STC_STAGE_BYTES (2 * STC_PANEL_BYTES)    // h panel | l panel
#define STC_TMEM_COLS 64                         // two accumulators of 32 columns

struct StatsTcArgs {
  const float* x;
  const int32_t* perm2;
  const int32_t* seg_off;    // [K+1]
  const int32_t* lr_cursor;  // [2K]  lr_cursor[2k] = first right-side position of cluster k
  int K;
  double* acc;               // [2K][rec]
  int rec;
  const float* centers;      // [2K][32] shift of every run (stats_centers_kernel)
};

struct StatsTcSmem {
  size_t stages, tbuf, tri, bnd, pre, bars, slot, total;
  __host__ __device__ explicit StatsTcSmem(int K) {
    size_t o = 0;
    stages = o; o += (size_t)STC_STAGES * STC_STAGE_BYTES;
    tbuf = o;   o += 64 * 33 * 4;
    tri = o;    o += 528 * 2;
    o = (o + 15) & ~(size_t)15;
    bnd = o;    o += (size_t)(2 * K + 1) * 4;
    pre = o;    o += (size_t)(2 * K + 1) * 4;
    o = (o + 15) & ~(size_t)15;
    bars = o;   o += 16 * 8;
    slot = o;   o += 16;
    total = o;
  }
};

namespace tc {
// MN-major TF32 operand.  The only layout tcgen05 accepts for 32-bit MN-major data is SWIZZLE_128B with
// 32-byte atomicity (layout type 1): rows of 128 bytes (32 consecutive M/N elements of one K index), 4-row
// atoms, byte-address bits [5,7) ^= bits [7,9).  `saddr` = first row of the k-step (8 rows), LBO = distance
// between 32-element atoms along M/N, SBO = distance between the 4-row groups along K (512 B).
__device__ __forceinline__ uint64_t smem_desc_mn128(uint32_t saddr, uint32_t lbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) | ((uint64_t)(512 >> 4) << 32) |
         ((uint64_t)1 << 46) | ((uint64_t)1 << 61);
}
// FP32 accumulator, TF32 A and B, both MN-major, M = 64, N = n.
__device__ __forceinline__ uint32_t idesc_tf32_mn_m64(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(64 >> 4) << 24);
}
__device__ __forceinline__ uint32_t idesc_tf32_mn_m128(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ float to_tf32(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}
// the TF32 bits of v: what the tensor core reads of an FP32 word (it ignores the low 13 mantissa bits)
__device__ __forceinline__ float trunc_tf32(float v) { return __uint_as_float(__float_as_uint(v) & 0xFFFFE000u); }
}  // namespace tc

// The tile sequence of a CTA: tiles of <= 128 positions that never straddle a key boundary.
struct StcWalk {
  int key, pos, end, tleft, gcount;
};
__device__ __forceinline__ void stc_walk_init(StcWalk& w, const int32_t* B, const int32_t* P, int nkeys, int t0, int t1) {
  int lo = 0, hi = nkeys - 1;   // first key with P[key + 1] > t0
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (P[mid + 1] > t0) hi = mid;
    else lo = mid + 1;
  }
  w.key = lo;
  w.pos = B[lo] + (t0 - P[lo]) * STC_TILE;
  w.end = B[lo + 1];
  w.tleft = t1 - t0;
  w.gcount = 0;
}
// the current tile closes its flush group (last tile of the key, of the CTA's range, or STC_FLUSH-th)
template <int FL = STC_FLUSH>
__device__ __forceinline__ bool stc_is_last(const StcWalk& w) {
  return w.pos + STC_TILE >= w.end || w.gcount == FL - 1 || w.tleft == 1;
}
template <int FL = STC_FLUSH>
__device__ __forceinline__ void stc_advance(StcWalk& w, const int32_t* B) {
  w.gcount = stc_is_last<FL>(w) ? 0 : w.gcount + 1;
  --w.tleft;
  w.pos += STC_TILE;
  if (w.pos >= w.end && w.tleft > 0) {
    do ++w.key; while (B[w.key + 1] == B[w.key]);
    w.pos = B[w.key];
    w.end = B[w.key + 1];
  }
}

// Centre of every run = mean of its first <= 32 points (any fixed vector is exact in the algebra; one
// near the mean keeps |y| ~ the spread of the run).  One CTA per key, 256 threads = 32 points x 8 chunks.
__global__ void __launch_bounds__(256) stats_centers_kernel(const float* __restrict__ x, const int32_t* __restrict__ perm2,
                                                            const int32_t* __restrict__ seg_off,
                                                            const int32_t* __restrict__ lr_cursor, float* __restrict__ centers) {
  __shared__ float4 sm[32][8];
  const int key = blockIdx.x, k = key >> 1;
  const int mid = lr_cursor[2 * k];
  const int beg = (key & 1) ? mid : seg_off[k];
  const int end = (key & 1) ? seg_off[k + 1] : mid;
  const int cnt = min(32, end - beg);
  const int p = threadIdx.x >> 3, c = threadIdx.x & 7;
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (p < cnt) v = __ldg(reinterpret_cast<const float4*>(x + (size_t)perm2[beg + p] * STC_D) + c);
  sm[p][c] = v;
  __syncthreads();
  if (threadIdx.x < STC_D) {
    const float* col = reinterpret_cast<const float*>(&sm[0][0]) + threadIdx.x;
    float sacc = 0.f;
    for (int q = 0; q < 32; ++q) sacc += col[q * STC_D];
    centers[(size_t)key * STC_D + threadIdx.x] = cnt > 0 ? sacc / (float)cnt : 0.f;
  }
}

__global__ void __launch_bounds__(STC_THREADS, 2) niw_stats_tc_kernel(const StatsTcArgs a) {
  extern __shared__ __align__(1024) uint8_t stc_smem[];
  const StatsTcSmem L(a.K);
  uint8_t* stage0 = stc_smem + L.stages;
  float* T = reinterpret_cast<float*>(stc_smem + L.tbuf);
  uint16_t* tri = reinterpret_cast<uint16_t*>(stc_smem + L.tri);
  int32_t* B = reinterpret_cast<int32_t*>(stc_smem + L.bnd);
  int32_t* P = reinterpret_cast<int32_t*>(stc_smem + L.pre);
  uint64_t* ready = reinterpret_cast<uint64_t*>(stc_smem + L.bars);   // [3] tile split and visible to the MMA
  uint64_t* empty = ready + STC_STAGES;                               // [3] MMAs of the stage retired
  uint64_t* accfull = empty + STC_STAGES;                             // [2]
  uint64_t* accempty = accfull + 2;                                   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(stc_smem + L.slot);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nkeys = 2 * a.K;

  // ---- key boundaries B[0..2K] and the exclusive prefix P of tiles per key ----
  for (int j = tid; j <= nkeys; j += STC_THREADS)
    B[j] = (j & 1) ? __ldg(a.lr_cursor + (j - 1)) : __ldg(a.seg_off + (j >> 1));
  for (int e = tid; e < 1024; e += STC_THREADS) {
    const int i = e >> 5, j = e & 31;
    if (j >= i) tri[i * 32 - (i * (i - 1)) / 2 + (j - i)] = (uint16_t)((i << 8) | j);
  }
  if (tid == 0) {
    for (int s = 0; s < STC_STAGES; ++s) {
      tc::mbar_init(&ready[s], 128);
      tc::mbar_init(&empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      tc::mbar_init(&accfull[b], 1);
      tc::mbar_init(&accempty[b], 128);
    }
    tc::fence_barrier_init();
  }
  __syncthreads();
  if (warp == 0) {
    int carry = 0;
    if (lane == 0) P[0] = 0;
    for (int base = 0; base < nkeys; base += 32) {
      const int j = base + lane;
      int v = j < nkeys ? (B[j + 1] - B[j] + STC_TILE - 1) / STC_TILE : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
      }
      if (j < nkeys) P[j + 1] = carry + v;
      carry += __shfl_sync(0xffffffffu, v, 31);
    }
  }
  if (warp == 4) tc::tmem_alloc(tmem_slot, STC_TMEM_COLS);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int ntot = P[nkeys];
  const int t0 = (int)(((int64_t)ntot * blockIdx.x) / gridDim.x);
  const int t1 = (int)(((int64_t)ntot * (blockIdx.x + 1)) / gridDim.x);
  const int nt = t1 - t0;

  if (nt > 0) {
    if (warp < 4) {
      // ======================= gather + split warps =======================
      const int c = tid & 7, r0 = tid >> 3;                 // 16-byte chunk, first row; rows r0 + 16 j
      // 128B swizzle with 32-byte atomicity: the 32-byte chunk index is XORed with (row & 3); (r0 + 16 j) & 3 == r0 & 3
      const uint32_t off0 = (uint32_t)(r0 * 128 + (((((c >> 1) ^ (r0 & 3)) << 1) | (c & 1)) << 4));
      StcWalk wl, wc;
      stc_walk_init(wl, B, P, nkeys, t0, t1);
      wc = wl;
      int idx[8];
      auto load_idx = [&]() {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int p = wl.pos + r0 + 16 * j;
          idx[j] = p < wl.end ? __ldg(a.perm2 + p) : -1;
        }
      };
      auto issue = [&](int s) {
        uint8_t* h = stage0 + (size_t)s * STC_STAGE_BYTES + off0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const bool ok = idx[j] >= 0;
          cp_async16(h + j * 2048, a.x + (size_t)(ok ? idx[j] : 0) * STC_D + 4 * c, ok ? 16 : 0);
        }
      };
      // tiles 0 and 1 in flight, indices of tile 2 in registers
#pragma unroll
      for (int li = 0; li < STC_STAGES - 1; ++li) {
        if (li < nt) {
          load_idx();
          issue(li);
          stc_advance(wl, B);
        }
        cp_async_commit();
      }
      if (STC_STAGES - 1 < nt) load_idx();
      float sx[4] = {0.f, 0.f, 0.f, 0.f};
      // every key is accumulated about a centre near its mean (shifted-data form): the TF32 / Float32
      // rounding then scales with the spread of the run instead of its distance from the origin
      auto load_center = [&](int key) { return __ldg(reinterpret_cast<const float4*>(a.centers + (size_t)key * STC_D) + c); };
      int ckey = wc.key;
      float4 cen = load_center(ckey);
      for (int li = 0; li < nt; ++li) {
        const int s = li % STC_STAGES;
        if (wc.key != ckey) {
          ckey = wc.key;
          cen = load_center(ckey);
        }
        const int npts = wc.end - wc.pos;                    // rows >= npts are zero padding
        cp_async_wait_group<STC_STAGES - 2>();               // this thread's chunks of tile li have landed
        uint8_t* h = stage0 + (size_t)s * STC_STAGE_BYTES + off0;
        float4 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = *reinterpret_cast<const float4*>(h + j * 2048);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (r0 + 16 * j < npts) {
            v[j].x -= cen.x; v[j].y -= cen.y; v[j].z -= cen.z; v[j].w -= cen.w;
          }
          float4 hi, lo;
          hi.x = tc::to_tf32(v[j].x); hi.y = tc::to_tf32(v[j].y); hi.z = tc::to_tf32(v[j].z); hi.w = tc::to_tf32(v[j].w);
          lo.x = v[j].x - hi.x; lo.y = v[j].y - hi.y; lo.z = v[j].z - hi.z; lo.w = v[j].w - hi.w;
          *reinterpret_cast<float4*>(h + j * 2048) = hi;
          *reinterpret_cast<float4*>(h + STC_PANEL_BYTES + j * 2048) = lo;
          sx[0] += v[j].x; sx[1] += v[j].y; sx[2] += v[j].z; sx[3] += v[j].w;
        }
        tc::fence_proxy_async();
        tc::mbar_arrive(&ready[s]);
        // next gather: tile li + 2 goes into the stage tile li - 1 used, once its MMAs have retired
        const int ln = li + STC_STAGES - 1;
        if (ln < nt) {
          const int sn = ln % STC_STAGES;
          tc::mbar_wait(&empty[sn], ((ln / STC_STAGES) & 1) ^ 1);
          issue(sn);
          stc_advance(wl, B);
          if (ln + 1 < nt) load_idx();
        }
        cp_async_commit();
        if (stc_is_last(wc)) {   // sum x of the flush group -> Float64 accumulator
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            sx[q] += __shfl_xor_sync(0xffffffffu, sx[q], 8);
            sx[q] += __shfl_xor_sync(0xffffffffu, sx[q], 16);
          }
          if (lane < 8) {
            double* dst = a.acc + (size_t)wc.key * a.rec + 1 + 4 * lane;   // lane == c for lanes 0-7
#pragma unroll
            for (int q = 0; q < 4; ++q) atomicAdd(dst + q, (double)sx[q]);
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) sx[q] = 0.f;
        }
        stc_advance(wc, B);
      }
    } else if (warp == 4) {
      // ======================= MMA issuer =======================
      if (lane == 0) {
        StcWalk wm;
        stc_walk_init(wm, B, P, nkeys, t0, t1);
        const uint32_t idesc = tc::idesc_tf32_mn_m64(STC_D);
        int buf = 0;
        uint32_t uses[2] = {0u, 0u};
        for (int li = 0; li < nt; ++li) {
          const int s = li % STC_STAGES;
          const bool first = wm.gcount == 0, last = stc_is_last(wm);
          if (first) {
            tc::mbar_wait(&accempty[buf], (uses[buf] & 1) ^ 1);   // the drain of this accumulator's previous group
            ++uses[buf];
          }
          tc::mbar_wait(&ready[s], (li / STC_STAGES) & 1);
          tc::tc_fence_after();
          const uint32_t hs = tc::smem_u32(stage0 + (size_t)s * STC_STAGE_BYTES);
          // A = [h panel | l panel] (two 32-row atoms, LBO apart), B = h panel; one k-step = 8 points = 1024 bytes
          const uint64_t desc = tc::smem_desc_mn128(hs, STC_PANEL_BYTES);
          const uint32_t tmem_d = tmem_base + buf * 32;
          const int npts = min(STC_TILE, wm.end - wm.pos);
          if (npts == STC_TILE) {
            tc::umma_tf32(tmem_d, desc, desc, idesc, first ? 0u : 1u);
#pragma unroll
            for (int ks = 1; ks < STC_TILE / 8; ++ks) tc::umma_tf32(tmem_d, desc + ks * 64, desc + ks * 64, idesc, 1u);
          } else {
            const int nks = (npts + 7) >> 3;
            for (int ks = 0; ks < nks; ++ks)
              tc::umma_tf32(tmem_d, desc + ks * 64, desc + ks * 64, idesc, (first && ks == 0) ? 0u : 1u);
          }
          tc::umma_commit(&empty[s]);
          if (last) {
            tc::umma_commit(&accfull[buf]);
            buf ^= 1;
          }
          stc_advance(wm, B);
        }
      }
    } else {
      // ======================= accumulator drain =======================
      const int sub = warp & 3;                 // TMEM sub-partition of this warp
      const int gt = tid - 160;                 // 0..127
      StcWalk we;
      stc_walk_init(we, B, P, nkeys, t0, t1);
      int buf = 0;
      uint32_t uses[2] = {0u, 0u};
      for (int li = 0; li < nt; ++li) {
        if (stc_is_last(we)) {
          tc::mbar_wait(&accfull[buf], uses[buf] & 1);
          ++uses[buf];
          tc::tc_fence_after();
          uint32_t v[32];
          tc::tmem_ld32(tmem_base + buf * 32 + ((uint32_t)(sub * 32) << 16), v);
          tc::tmem_ld_wait();
          tc::tc_fence_before();
          tc::mbar_arrive(&accempty[buf]);
          // M = 64: accumulator row m lives in lane (m % 16) of sub-partition m / 16
          if (lane < 16) {
            float* trow = T + (16 * sub + lane) * 33;
#pragma unroll
            for (int j = 0; j < 32; ++j) trow[j] = __uint_as_float(v[j]);
          }
          asm volatile("bar.sync 1, 128;" ::: "memory");
          double* dst = a.acc + (size_t)we.key * a.rec + 1 + STC_D;
          for (int e = gt; e < 528; e += 128) {
            const int ij = tri[e], i = ij >> 8, j = ij & 255;
            const float sv = (T[i * 33 + j] + T[(32 + i) * 33 + j]) + T[(32 + j) * 33 + i];
            atomicAdd(dst + i * STC_D + j, (double)sv);
          }
          asm volatile("bar.sync 1, 128;" ::: "memory");
          buf ^= 1;
        }
        stc_advance(we, B);
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 4) tc::tmem_dealloc(tmem_base, STC_TMEM_COLS);
}
