// Stage 3: segmented sufficient statistics.
//
//   create_suff_stats_dict_worker            src/local_clusters_actions.jl:149-169
//   create_sufficient_statistics (NIW)       src/priors/niw.jl:42-51      N, sum x, S = X X' (Float64)
//   create_sufficient_statistics (multinom.) src/priors/multinomial_prior.jl:27-32   N, sum x
//   aggregate_suff_stats                     niw.jl:64-66, multinomial_prior.jl:41-43
//
// The reference masks + gathers + widens the points of every cluster three times (cluster, left,
// right) and runs three DGEMMs.  Here the points are already bucketed by (label, side) in `perm2`
// (kernels_gauss.cuh: sublabel_partition), so each work item is a run of points with ONE key; the
// rank-1 updates are accumulated per key for left and right only (cluster = left + right in the
// finalise kernel), upper-triangular blocks only, in Float32 registers over <= `chunk` points and
// then added in Float64 (atomicAdd(double)) to the per-key accumulator, which is what crosses NVLink.
#pragma once
#include "common.cuh"

struct StatsItem {
  int32_t key;    // 2*k + side
  int32_t begin;  // range in perm2
  int32_t end;
};

#ifndef DPMM_TEMPLATES_ONLY
// Builds the work list: for every wanted cluster k, its left run [seg_off[k], lr_cursor[2k]) and
// right run [lr_cursor[2k], seg_off[k+1]) cut into chunks of `chunk` points.  Single CTA.
__global__ void stats_worklist_kernel(const int32_t* __restrict__ seg_off, const int32_t* __restrict__ lr_cursor,
                                      const uint8_t* __restrict__ wanted, int K, int chunk, StatsItem* items,
                                      int32_t* n_items, int32_t* next_item) {
  extern __shared__ int sc[];  // [2K] chunk counts -> exclusive offsets
  const int tid = threadIdx.x;
  for (int key = tid; key < 2 * K; key += blockDim.x) {
    const int k = key >> 1;
    int len = 0;
    if (wanted == nullptr || wanted[k]) {
      const int mid = lr_cursor[2 * k];
      len = (key & 1) ? seg_off[k + 1] - mid : mid - seg_off[k];
    }
    sc[key] = (len + chunk - 1) / chunk;
  }
  __syncthreads();
  if (tid == 0) {
    int run = 0;
    for (int key = 0; key < 2 * K; ++key) {
      const int c = sc[key];
      sc[key] = run;
      run += c;
    }
    *n_items = run;
    *next_item = 0;
  }
  __syncthreads();
  for (int key = tid; key < 2 * K; key += blockDim.x) {
    const int k = key >> 1;
    if (wanted != nullptr && !wanted[k]) continue;
    const int mid = lr_cursor[2 * k];
    const int b = (key & 1) ? mid : seg_off[k];
    const int e = (key & 1) ? seg_off[k + 1] : mid;
    int o = sc[key];
    for (int s = b; s < e; s += chunk) items[o++] = StatsItem{key, s, min(e, s + chunk)};
  }
}

#endif  // DPMM_TEMPLATES_ONLY

// Transposed warp reduction: on entry every lane holds EP partial sums v[0..EP); on exit lane l
// holds in v[0..EP/32) the warp totals of entries  e = (bits of l, MSB first) * (EP/2, EP/4, ...) + j.
// 2*(EP - EP/32) selects + (EP - EP/32) shuffles instead of 5*EP shuffles.
template <int EP>
__device__ __forceinline__ void warp_transpose_reduce(float (&v)[EP], int lane) {
  static_assert(EP % 32 == 0, "EP must be a multiple of 32");
  int h = EP / 2;
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    const int off = 16 >> s;
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int e = 0; e < EP / 2; ++e) {
      if (e < h) {
        const float send = up ? v[e] : v[e + h];
        const float keep = up ? v[e + h] : v[e];
        v[e] = keep + __shfl_xor_sync(0xffffffffu, send, off);
      }
    }
    h >>= 1;
  }
}
// entry index owned by `lane` in slot j after warp_transpose_reduce<EP>
template <int EP>
__device__ __forceinline__ int warp_transpose_entry(int lane, int j) {
  int e = j, h = EP / 2;
#pragma unroll
  for (int s = 0; s < 5; ++s) {
    if (lane & (16 >> s)) e += h;
    h >>= 1;
  }
  return e;
}

template <int D>
struct StatsCfg {
  static constexpr int BS = (D <= 8) ? D : 8;            // register block edge (rows)
  static constexpr int BSQ = (BS + 1) & ~1;              // block columns, padded to whole FFMA2 pairs
  static constexpr int NB = (D + BS - 1) / BS;           // blocks per matrix edge
  static constexpr int NU = NB * (NB + 1) / 2;           // upper-triangular blocks
  static constexpr int DPAD = NB * BS + (BSQ - BS);
  static constexpr bool VEC = (BS % 4 == 0);
  static constexpr int DS = VEC ? 4 * ((DPAD / 4) | 1) : ((DPAD & 1) ? DPAD : DPAD + 1);
  static constexpr int E = BS * BSQ;
  static constexpr int EP = (E + 31) / 32 * 32;
  static constexpr int G = (NU + 15) / 16;               // block groups: a CTA covers NU/G blocks (<= 16 warps)
  static constexpr int WPG = (NU + G - 1) / G;           // warps (= blocks) per group
  static constexpr int NS = (WPG >= 8) ? 1 : (8 / WPG);  // point slices so that a CTA has ~8+ warps
  static constexpr int WARPS = WPG * NS;
  static constexpr int R = (NS >= 8) ? 2 : 4;            // points per lane per tile
  static constexpr int TPTS = 32 * NS * R;               // points per shared-memory tile
  static constexpr int STAGES = 4;                       // cp.async ring depth (tiles in flight)
  static constexpr int MAX_CHUNK = 2048;                 // longest run (points) of one work item
  static constexpr int SMEM_BYTES = STAGES * TPTS * DS * 4 + MAX_CHUNK * 4;
  static constexpr int MIN_CTAS = (WARPS * 32 <= 320) ? 2 : 1;
};

struct StatsArgs {
  const float* x;
  int D;                    // runtime D (== template D for NIW)
  const int32_t* perm2;
  const StatsItem* items;
  const int32_t* n_items;
  int32_t* next_item;
  double* acc;              // [2K][rec]  rec = 1 + D + D*D (NIW), 1 + 2D (diagonal) or 1 + D (multinomial); count slot unused
  int rec;
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src, int src_bytes) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src, int src_bytes) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(d), "l"(gmem_src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
// 16 bytes of read-only global memory into registers, not allocated in L1 (as cp.async.cg); zeros when !ok, as
// cp_async16 with src_bytes = 0.  Volatile so that it is issued where it is written: the loads of a tile are made
// a tile or two ahead of their use, and the compiler must not sink them to it.
__device__ __forceinline__ float4 ldg_nc16(const void* gmem_src, bool ok) {
  float4 v;
  asm volatile("{\n .reg .pred p;\n setp.ne.b32 p, %5, 0;\n"
               " mov.f32 %0, 0f00000000; mov.f32 %1, 0f00000000; mov.f32 %2, 0f00000000; mov.f32 %3, 0f00000000;\n"
               " @p ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];\n}"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(gmem_src), "r"((int)ok));
  return v;
}

// K5: NIW.  Warp w of a CTA owns upper block u = g*WPG + w % WPG of S (g = block group of the work
// unit; G > 1 only when S has more than 16 upper blocks, i.e. D > 40) and point slice w / WPG; lane l
// owns the points l, l+32, ... of its slice, so the warp's 32 lanes read 32 different staged points
// at the same column offset (conflict-free LDS.128) and the 32 partial blocks are combined once per
// item.  The gathered rows of tile t+1 stream in with cp.async (zero-filled past the end of the run)
// while tile t is accumulated; the rank-1 updates are packed FFMA2 (two columns per instruction).
template <int D>
__global__ void __launch_bounds__(StatsCfg<D>::WARPS * 32, StatsCfg<D>::MIN_CTAS)
niw_stats_kernel(const StatsArgs a) {
  using C = StatsCfg<D>;
  constexpr int BS = C::BS, BSQ = C::BSQ, NQ = C::BSQ / 2;
  extern __shared__ __align__(16) float xs_all[];  // [STAGES][TPTS][DS] | sidx [MAX_CHUNK]
  int32_t* sidx = reinterpret_cast<int32_t*>(xs_all + C::STAGES * C::TPTS * C::DS);
  __shared__ int s_item;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slice = warp / C::WPG;
  for (int e = tid; e < C::STAGES * C::TPTS * C::DS; e += blockDim.x) xs_all[e] = 0.f;  // padding columns stay 0

  // gather tile [t0, t0 + TPTS) of the run into ring slot `buf`; the run's point indices were staged
  // in sidx when the item was fetched, so issuing the copies never waits on a global load
  auto prefetch = [&](const StatsItem& item, int t0, int buf) {
    float* xs = xs_all + buf * C::TPTS * C::DS;
    const int tn = min(C::TPTS, item.end - t0);
    const int32_t* ix = sidx + (t0 - item.begin);
    if constexpr (D % 4 == 0) {
      for (int e = tid; e < C::TPTS * (D / 4); e += blockDim.x) {
        const int p = e / (D / 4), c = e - p * (D / 4);
        const bool ok = p < tn;
        const int idx = ok ? ix[p] : 0;
        cp_async16(xs + p * C::DS + 4 * c, a.x + (size_t)idx * D + 4 * c, ok ? 16 : 0);
      }
    } else {
      for (int e = tid; e < C::TPTS * D; e += blockDim.x) {
        const int p = e / D, c = e - p * D;
        const bool ok = p < tn;
        const int idx = ok ? ix[p] : 0;
        cp_async4(xs + p * C::DS + c, a.x + (size_t)idx * D + c, ok ? 4 : 0);
      }
    }
    cp_async_commit();
  };

  for (;;) {
    __syncthreads();
    if (tid == 0) s_item = atomicAdd(a.next_item, 1);
    __syncthreads();
    const int it = s_item;
    if (it >= *a.n_items * C::G) break;
    const StatsItem item = a.items[it / C::G];
    for (int e = tid; e < item.end - item.begin; e += blockDim.x) sidx[e] = __ldg(a.perm2 + item.begin + e);
    __syncthreads();
    const int u = (it % C::G) * C::WPG + warp % C::WPG;
    const bool live = u < C::NU;
    int bi = 0, bj = 0;
    if (live) {
      int r = u;
      while (r >= C::NB - bi) {
        r -= C::NB - bi;
        ++bi;
      }
      bj = bi + r;
    }
    const bool diag = live && (bi == bj);
    f32x2_t acc[BS][NQ];
    float sx[BS];
#pragma unroll
    for (int p = 0; p < BS; ++p) {
      sx[p] = 0.f;
#pragma unroll
      for (int q = 0; q < NQ; ++q) acc[p][q] = 0ull;
    }

    // cp.async ring: STAGES-1 tiles in flight ahead of the one being accumulated (a commit group is
    // issued every step, empty past the end of the run, so that wait_group<STAGES-2> always means
    // "the tile of this step has landed")
    const int ntl = (item.end - item.begin + C::TPTS - 1) / C::TPTS;
#pragma unroll
    for (int j = 0; j < C::STAGES - 1; ++j) {
      if (j < ntl) prefetch(item, item.begin + j * C::TPTS, j);
      else cp_async_commit();
    }
    for (int t = 0; t < ntl; ++t) {
      const int buf = t % C::STAGES;
      cp_async_wait_group<C::STAGES - 2>();
      __syncthreads();  // tile t has landed for everyone; everyone is done with tile t-1's buffer
      if (t + C::STAGES - 1 < ntl) prefetch(item, item.begin + (t + C::STAGES - 1) * C::TPTS, (t + C::STAGES - 1) % C::STAGES);
      else cp_async_commit();
      if (live) {
        const float* xs = xs_all + buf * C::TPTS * C::DS;
#pragma unroll
        for (int r = 0; r < C::R; ++r) {
          const float* row = xs + (slice * 32 * C::R + r * 32 + lane) * C::DS;
          float xi[BS];
          f32x2_t xj[NQ];
          if constexpr (C::VEC) {
#pragma unroll
            for (int q4 = 0; q4 < BS / 4; ++q4) {
              const float4 vi = *reinterpret_cast<const float4*>(row + bi * BS + 4 * q4);
              const ulonglong2 vj = *reinterpret_cast<const ulonglong2*>(row + bj * BS + 4 * q4);
              xi[4 * q4] = vi.x; xi[4 * q4 + 1] = vi.y; xi[4 * q4 + 2] = vi.z; xi[4 * q4 + 3] = vi.w;
              xj[2 * q4] = vj.x; xj[2 * q4 + 1] = vj.y;
            }
          } else {
#pragma unroll
            for (int q = 0; q < BS; ++q) xi[q] = row[bi * BS + q];
#pragma unroll
            for (int q = 0; q < NQ; ++q) xj[q] = f2_pack(row[bj * BS + 2 * q], row[bj * BS + 2 * q + 1]);
          }
#pragma unroll
          for (int p = 0; p < BS; ++p) {
            const f32x2_t xip = f2_pack(xi[p], xi[p]);
#pragma unroll
            for (int q = 0; q < NQ; ++q) acc[p][q] = f2_fma(xip, xj[q], acc[p][q]);
          }
          if (diag) {
#pragma unroll
            for (int p = 0; p < BS; ++p) sx[p] += xi[p];
          }
        }
      }
    }
    // ---- combine the 32 lanes and add to the key's Float64 accumulator ----
    if (!live) continue;
    float accf[C::EP];
#pragma unroll
    for (int e = 0; e < C::EP; ++e) accf[e] = 0.f;
#pragma unroll
    for (int p = 0; p < BS; ++p)
#pragma unroll
      for (int q = 0; q < NQ; ++q) f2_unpack(acc[p][q], accf[p * BSQ + 2 * q], accf[p * BSQ + 2 * q + 1]);
    warp_transpose_reduce<C::EP>(accf, lane);
    double* dst = a.acc + (size_t)item.key * a.rec;
#pragma unroll
    for (int j = 0; j < C::EP / 32; ++j) {
      const int e = warp_transpose_entry<C::EP>(lane, j);
      if (e < C::E) {
        const int gi = bi * BS + e / BSQ, gj = bj * BS + e % BSQ;
        if (e % BSQ < BS && gi < D && gj < D && gi <= gj) atomicAdd(dst + 1 + D + (size_t)gi * D + gj, (double)accf[j]);
      }
    }
    if (diag) {
#pragma unroll
      for (int p = 0; p < BS; ++p) {
        float v = sx[p];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == p && bi * BS + p < D) atomicAdd(dst + 1 + bi * BS + p, (double)v);
      }
    }
  }
}

// K5 for small D (<= 8): one WARP per work item, lane <-> point.  A row is D scalars (20 bytes at D = 5: not
// worth staging through shared memory, and cp.async would need one 4-byte copy per scalar); each lane keeps
// sum x and the upper triangle of sum x x' of its <= 32 points in Float32 registers, one transposed warp
// reduction combines the lanes, and the totals go to the Float64 accumulator.
template <int D>
__global__ void __launch_bounds__(256) niw_stats_small_kernel(const StatsArgs a) {
  constexpr int NV = D + D * (D + 1) / 2;          // sum x | upper triangle of S, row by row
  constexpr int NVP = (NV + 31) / 32 * 32;
  const int lane = threadIdx.x & 31;
  const int n_items = *a.n_items;
  for (;;) {
    int it = 0;
    if (lane == 0) it = atomicAdd(a.next_item, 1);
    it = __shfl_sync(0xffffffffu, it, 0);
    if (it >= n_items) break;
    const StatsItem item = a.items[it];
    float v[NVP];
#pragma unroll
    for (int e = 0; e < NVP; ++e) v[e] = 0.f;
    for (int p = item.begin + lane; p < item.end; p += 32) {
      const float* xp = a.x + (size_t)__ldg(a.perm2 + p) * D;
      float x[D];
#pragma unroll
      for (int i = 0; i < D; ++i) x[i] = __ldg(xp + i);
      int e = D;
#pragma unroll
      for (int i = 0; i < D; ++i) {
        v[i] += x[i];
#pragma unroll
        for (int j = i; j < D; ++j) {
          v[e] = fmaf(x[i], x[j], v[e]);
          ++e;
        }
      }
    }
    warp_transpose_reduce<NVP>(v, lane);
    double* dst = a.acc + (size_t)item.key * a.rec + 1;
#pragma unroll
    for (int s = 0; s < NVP / 32; ++s) {
      const int e = warp_transpose_entry<NVP>(lane, s);
      if (e < D) {
        if (v[s] != 0.f) atomicAdd(dst + e, (double)v[s]);
      } else if (e < NV) {
        int t = e - D, i = 0;
        while (t >= D - i) {   // row i of the upper triangle holds D - i entries
          t -= D - i;
          ++i;
        }
        if (v[s] != 0.f) atomicAdd(dst + D + (size_t)i * D + (i + t), (double)v[s]);
      }
    }
  }
}

#ifndef DPMM_TEMPLATES_ONLY
// K6: multinomial.  sum x per key.  One warp per work item (a run of points with one (label, side)
// key); lane l owns the features l, l+32, ... so every point is read as fully coalesced 128-byte
// segments straight from global memory (no staging), with MNM_STATS_UNROLL points in flight per
// warp, and the per-lane Float32 partial sums (exact: small integer counts) are added to the key's
// Float64 accumulator once per item.
#define MNM_STATS_NREG 32      // features per lane: slices of 1024 features
#define MNM_STATS_UNROLL 8
template <bool SLICED>
__global__ void __launch_bounds__(256) mnm_stats_kernel(const StatsArgs a) {
  const int lane = threadIdx.x & 31;
  // SLICED (D > 1024): a work unit is (item, slice of 32 x MNM_STATS_NREG features)
  const int nslices = SLICED ? (a.D + 32 * MNM_STATS_NREG - 1) / (32 * MNM_STATS_NREG) : 1;
  const int n_units = *a.n_items * nslices;
  for (;;) {
    int u = 0;
    if (lane == 0) u = atomicAdd(a.next_item, 1);
    u = __shfl_sync(0xffffffffu, u, 0);
    if (u >= n_units) break;
    const StatsItem item = a.items[u / nslices];
    {
      const int d0 = (u % nslices) * 32 * MNM_STATS_NREG;
      const int D = SLICED ? min(a.D - d0, 32 * MNM_STATS_NREG) : a.D;
      const float* x = a.x + d0;
      const int nreg = (D + 31) >> 5;
      float acc[MNM_STATS_NREG];
#pragma unroll
      for (int r = 0; r < MNM_STATS_NREG; ++r) acc[r] = 0.f;
      int idx_n[MNM_STATS_UNROLL];
#pragma unroll
      for (int j = 0; j < MNM_STATS_UNROLL; ++j) idx_n[j] = (item.begin + j < item.end) ? __ldg(a.perm2 + item.begin + j) : -1;
      for (int p0 = item.begin; p0 < item.end; p0 += MNM_STATS_UNROLL) {
        int idx[MNM_STATS_UNROLL];
#pragma unroll
        for (int j = 0; j < MNM_STATS_UNROLL; ++j) {
          idx[j] = idx_n[j];                                   // indices were fetched one batch ahead
          const int pn = p0 + MNM_STATS_UNROLL + j;
          idx_n[j] = (pn < item.end) ? __ldg(a.perm2 + pn) : -1;
        }
        if (nreg <= 4) {  // common case (D <= 128): all loads of the batch in flight at once
          float v[MNM_STATS_UNROLL][4];
#pragma unroll
          for (int j = 0; j < MNM_STATS_UNROLL; ++j)
#pragma unroll
            for (int r = 0; r < 4; ++r) {
              const int d = lane + 32 * r;
              v[j][r] = (idx[j] >= 0 && d < D) ? __ldg(x + (size_t)idx[j] * a.D + d) : 0.f;
            }
#pragma unroll
          for (int j = 0; j < MNM_STATS_UNROLL; ++j)
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[r] += v[j][r];
        } else {
#pragma unroll
          for (int j = 0; j < MNM_STATS_UNROLL; ++j)
            if (idx[j] >= 0) {
#pragma unroll
              for (int r = 0; r < MNM_STATS_NREG; ++r) {
                const int d = lane + 32 * r;
                if (r < nreg && d < D) acc[r] += __ldg(x + (size_t)idx[j] * a.D + d);
              }
            }
        }
      }
      double* dst = a.acc + (size_t)item.key * a.rec + 1 + d0;
#pragma unroll
      for (int r = 0; r < MNM_STATS_NREG; ++r) {
        const int d = lane + 32 * r;
        if (r < nreg && d < D && acc[r] != 0.f) atomicAdd(dst + d, (double)acc[r]);
      }
    }
  }
}

// K8: finalise + pack.  out[m][3][rec] for the m requested clusters: cluster = left + right, S
// mirrored from its upper triangle (niw != 0), counts from the partition cursors.  With niw == 0 every other entry is
// a plain sum and is added as it is: [N | sum x] (multinomial), [N | sum x | sum x^2] (diagonal Gaussian).  When `xc` is given the
// accumulators hold sums of y = x - c about a centre c of every run (centers [2K][D], see
// kernels_stats_tc.cuh) and are shifted back here in Float64: sum x = s + N c,  S = sum y y' + c s' + s c' + N c c'.
// `risk` (optional) counts the diagonal entries whose centred sum exceeds 32 x the un-centred one: the
// centre was far from the run relative to the run's own magnitude (only tiny or degenerate runs), so the
// tensor core's ~2e-6 |y_i||y_j| accumulation error (round-toward-zero over the k-steps of a flush group) is not small against sqrt(S_ii S_jj); the caller then recomputes
// the statistics with the FP32/FP64 kernel.
__global__ void stats_finalize_kernel(const double* __restrict__ acc, const int32_t* __restrict__ seg_off,
                                      const int32_t* __restrict__ lr_cursor, const int32_t* __restrict__ idx_list,
                                      int m, int D, int rec, int niw, double* out, const float* __restrict__ centers,
                                      const int32_t* __restrict__ lcount, double* risk) {
  pdl_wait();
  pdl_launch_dependents();
  const int a = blockIdx.y;
  if (a >= m) return;
  const int k = idx_list != nullptr ? idx_list[a] : a;   // no list: every cluster in order
  const double* L = acc + (size_t)(2 * k) * rec;
  const double* R = acc + (size_t)(2 * k + 1) * rec;
  // left count: from the partition cursors, or as counted by the fused sub-label + statistics kernel
  const int beg = seg_off[k], end = seg_off[k + 1];
  const int mid = lcount != nullptr ? beg + lcount[k] : lr_cursor[2 * k];
  const double nl = (double)(mid - beg), nr = (double)(end - mid);
  const float* cl = centers != nullptr ? centers + (size_t)(2 * k) * D : nullptr;
  const float* cr = centers != nullptr ? centers + (size_t)(2 * k + 1) * D : nullptr;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < rec; e += gridDim.x * blockDim.x) {
    double l, r;
    if (e == 0) {
      l = nl;
      r = nr;
    } else if (e <= D || !niw) {
      l = L[e];
      r = R[e];
      if (cl != nullptr) l += nl * (double)cl[e - 1];
      if (cr != nullptr) r += nr * (double)cr[e - 1];
    } else {
      const int q = e - 1 - D;
      int i = q / D, j = q - i * D;
      if (i > j) {
        const int t = i;
        i = j;
        j = t;
      }
      l = L[1 + D + (size_t)i * D + j];
      r = R[1 + D + (size_t)i * D + j];
      if (cl != nullptr) {
        const double ci = cl[i], cj = cl[j], l0 = l;
        l += ci * L[1 + j] + L[1 + i] * cj + nl * ci * cj;
        if (risk != nullptr && i == j && nl > 0 && l0 > 32.0 * l) atomicAdd(risk, 1.0);
      }
      if (cr != nullptr) {
        const double ci = cr[i], cj = cr[j], r0 = r;
        r += ci * R[1 + j] + R[1 + i] * cj + nr * ci * cj;
        if (risk != nullptr && i == j && nr > 0 && r0 > 32.0 * r) atomicAdd(risk, 1.0);
      }
    }
    double* o = out + (size_t)a * 3 * rec;
    o[e] = l + r;
    o[rec + e] = l;
    o[2 * rec + e] = r;
  }
}

#endif  // DPMM_TEMPLATES_ONLY
