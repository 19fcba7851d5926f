// Stages 2b + 3 fused on the tensor cores (NIW, D = 32): ONE pass over the label-sorted points draws every
// sub-label and accumulates the left / right sufficient statistics of every cluster.
//
//   sample_sub_clusters_worker! / create_subclusters_labels!   src/local_clusters_actions.jl:70-95
//   log_likelihood!(mv_gaussian)                               src/distributions/mv_gaussian.jl:21-25
//   sample_log_cat_array! (C = 2)                              src/utils.jl:19-31
//   create_suff_stats_dict_worker                              src/local_clusters_actions.jl:149-169
//   create_sufficient_statistics (NIW)                         src/priors/niw.jl:42-51
//
// A tile = 128 consecutive positions of ONE cluster k in the label-sorted permutation `perm`.  Its rows
// are loaded into registers (two tiles ahead), shifted there by the cluster's centre c_k (x - c_k is exact
// in Float32, see niw_pack_center), split z = h + l with h = tf32(z), and stored once: z into the raw ring,
// l into the split panel.
//
//   GEMM1 (contraction over FEATURES; h | l as K-major A operands, 128B swizzle, M = 128 points, N = 64):
//       Y = h Wh' + l Wh' + h Wl' - b,   W = [U_left; U_right] = Wh + Wl,   b = U_s (mu_s - c_k)
//     a 3-term error-compensated TF32 product (only l Wl', <= 2^-22 relative, is dropped) whose
//     accumulator row p holds U_l (x_p - mu_l) | U_r (x_p - mu_r).  The epilogue warps read it with
//     tcgen05.ld, form q = |y|^2, r = -c - q/2 + log w (the reference's Float32 final operations) and
//     draw the sub-label with the reference's inverse-CDF rule.
//   GEMM2 (contraction over POINTS; MN-major operands, M = 64, N = 32): once the sub-labels are known the
//     epilogue warps copy the rows of h | l into a second pair of panels PERMUTED so that the left rows
//     come first and the right rows start at a multiple of 8 (zero rows pad both runs), in the MN-major
//     layout (128B swizzle with 32-byte atoms, the only one tcgen05 takes for 32-bit MN-major data).
//     Every 8-row k-step then belongs to one side:   D_side += [h | l]' h   (rows 0-31 sum h h',
//     rows 32-63 sum l h'),  S = hh' + lh' + (lh')' as in kernels_stats_tc.cuh, flushed to the Float64
//     accumulators every SS_FLUSH tiles.  No masked copies, no left/right partition of the permutation.
//   sum y and the left count come from the permuting pass.  Everything is shifted back by c_k in
//   Float64 by stats_finalize_kernel.
//
// Warp roles (896 threads, one CTA per SM; every CTA owns a contiguous range of the tile sequence):
//   warps 0-3, 19-22  gather + shift + split         warps 5-8 / 9-12 / 24-27  GEMM1 epilogue of the tiles
//   warp  4    GEMM1 issuer                                      li = 0 / 1 / 2 (mod 3): draw, permute, sum y
//   warp  17   stages the next cluster's       warps 13-16       GEMM2 accumulator drain
//              factors                         warps 18, 23      GEMM2 issuers (left / right k-steps)
// (the epilogue is a long dependent instruction chain per tile -- a single warp per scheduler issues one
// instruction every ~7-10 cycles -- so three groups work on tiles li mod 3; GEMM1 has six accumulator buffers so
// that its issuer runs ahead of them.)
//
// What bounds it (ncu, round 2, profiles/r2j_ncu_summary.md): the shared-memory data pipe, then at lsu 54 % +
// tc 33 % of its peak.  Per 128-point tile the CUDA cores move ~1150 wavefronts (centre/split stores 128 + 128,
// permuting copy 128 + 272, drain; before the register-path gather also a cp.async landing of 128 and its
// read-back of 128) and the tensor core reads ~1030 (GEMM1: 13 k-steps x (4 KB + 2 KB); GEMM2: 17 x (2 KB + 1 KB)).
// The register-path gather took C2 from 86.9 to 84.1 us (B200, 1000 W).  Measured on the way and rejected:
// suspend-time hints and nanosleep back-off in the waits of the non-critical warps (+2..+14 us), Philox on the
// gather warps (+15 us), three tiles of gather in flight with a 5-slot ring (+9 us).
#pragma once
#include "kernels_gauss.cuh"   // gauss_finish
#include "kernels_stats_tc.cuh"

#define SS_D 32
#define SS_TILE 128
#define SS_RAW 5                         // ring of raw (centred) tiles: split -> GEMM1 and permuting pass
#define SS_PF 2                          // tiles of gather in flight (one register set each)
#define SS_NG 3                          // GEMM1 epilogue groups (4 warps each), tile li -> group li % SS_NG
#define SS_FLUSH 8                       // tiles per GEMM2 flush group (TMEM accumulates 1024 points between drains)
#define SS_NTB 6                         // GEMM1 accumulator buffers (64 TMEM columns each), tile li -> buffer li % SS_NTB
#define SS_THREADS 896
#define SS_GATHER 256                    // gather threads: warps 0-3 and 19-22, 4 rows each
#define SS_PANEL 16384                   // one [128][32] Float32 panel
#define SS_PROWS 136                     // rows of a permuted panel: both runs padded to a multiple of 8
#define SS_PPANEL (SS_PROWS * 128)
#define SS_WSLOT (8192 + 8192 + 2048)    // Wh | Wl | bias k-step operand
#define SS_TMEM_COLS 512                 // GEMM1: SS_NTB x 64 columns, GEMM2: 2 x 64 columns
#define SS_TMEM_G2 (SS_NTB * 64)         // first column of the GEMM2 accumulators
#define SS_TLD 65

struct SubStatsArgs {
  const float* x;
  int64_t n;
  int K;
  const int32_t* perm;     // [n] point indices sorted by label
  const int32_t* seg_off;  // [K+1]
  const float* w;          // [K][2][32][32] rows of U_left, U_right
  const float* bias;       // [K][2][32]     U_s (mu_s - c_k)
  const float* cen;        // [K][32]        c_k
  const float* cst;        // [3K]
  const float* loglr;      // [2K]
  uint8_t* sub;            // [n] out
  double* acc;             // [2K][rec] (zeroed by the caller)
  int rec;
  int32_t* lcount;         // [K] out: number of left points (zeroed by the caller)
  float* centers;          // [2K][32] out: the shift of every (cluster, side) accumulator
  const double* u_inj;
  uint64_t seed;
  uint32_t call;
  int64_t goff;
  float* dump;             // optional [2][n]
};

struct SubStatsSmem {
  size_t raw, split, perm, wslot, aaug, tbuf, tri, dest, cnt, kcnt, bnd, pre, bars, slot, total;
  __host__ __device__ explicit SubStatsSmem(int K) {
    size_t o = 0;
    raw = o;    o += (size_t)SS_RAW * SS_PANEL;
    split = o;  o += (size_t)2 * SS_PANEL;           // 2 x l panel, K-major (lives from the split to the end of GEMM1)
    perm = o;   o += (size_t)2 * 2 * SS_PPANEL;      // 2 x (h | l), permuted, MN-major
    wslot = o;  o += (size_t)SS_WSLOT;
    aaug = o;   o += 4096;
    tbuf = o;   o += 64 * SS_TLD * 4;
    tri = o;    o += 528 * 2;
    o = (o + 15) & ~(size_t)15;
    dest = o;   o += SS_NG * SS_TILE;
    cnt = o;    o += SS_NG * 4 * 4;
    kcnt = o;   o += 4 * 4;
    bnd = o;    o += (size_t)(K + 1) * 4;
    pre = o;    o += (size_t)(K + 1) * 4;
    o = (o + 15) & ~(size_t)15;
    bars = o;   o += 40 * 8;
    slot = o;   o += 16;
    total = o;
  }
};

__global__ void __launch_bounds__(SS_THREADS, 1) niw_substats_tc_kernel(const SubStatsArgs a) {
  extern __shared__ __align__(1024) uint8_t ss_smem[];
  const SubStatsSmem L(a.K);
  uint8_t* raw0 = ss_smem + L.raw;
  uint8_t* split0 = ss_smem + L.split;
  uint8_t* perm0 = ss_smem + L.perm;
  uint8_t* wslot = ss_smem + L.wslot;
  float* aaug = reinterpret_cast<float*>(ss_smem + L.aaug);
  float* T = reinterpret_cast<float*>(ss_smem + L.tbuf);
  uint16_t* tri = reinterpret_cast<uint16_t*>(ss_smem + L.tri);
  uint8_t* dest_s = ss_smem + L.dest;
  volatile int32_t* cnt_s = reinterpret_cast<int32_t*>(ss_smem + L.cnt);
  volatile int32_t* kcnt = reinterpret_cast<int32_t*>(ss_smem + L.kcnt);
  int32_t* B = reinterpret_cast<int32_t*>(ss_smem + L.bnd);
  int32_t* P = reinterpret_cast<int32_t*>(ss_smem + L.pre);
  uint64_t* bars = reinterpret_cast<uint64_t*>(ss_smem + L.bars);
  uint64_t* ready = bars;            // [2] z (in its raw slot) and l of the tile written and visible
  uint64_t* sfree = bars + 2;        // [2] l panel read by GEMM1
  uint64_t* landed = bars + 18;      // [5] raw tile in shared memory
  uint64_t* rfree = bars + 23;       // [5] ... consumed by the permuting pass
  uint64_t* d1full = bars + 28;      // [SS_NTB] GEMM1 accumulator complete
  uint64_t* d1empty = bars + 34;     // [SS_NTB] ... read by the epilogue
  uint64_t* permd = bars + 8;        // [2] permuted panels written
  // [4] GEMM2 of tile li retired: indexed li & 3, NOT by the panel slot li & 1.  With three epilogue groups the group
  // of tile li can run up to four tiles ahead of the slowest one, so a barrier that turns over every two tiles could
  // be two phases behind the waiter -- which a parity wait cannot tell from "complete".  Four tiles per turn-over
  // puts that case (eight tiles of skew) beyond what the raw ring (5) and the accumulator buffers (6) allow.
  uint64_t* pfree = bars + 4;
  uint64_t* d2full = bars + 12;      // [2] flush group complete
  uint64_t* d2empty = bars + 14;     // [2] ... drained
  uint64_t* wfull = bars + 16;       // factors of a cluster staged
  uint64_t* wempty = bars + 17;      // last GEMM1 of the cluster retired
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(ss_smem + L.slot);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nkeys = a.K;

  // ---- triangle index table, constant operands, barriers, tensor memory: CTA-local, before the grid dependency ----
  for (int e = tid; e < 1024; e += SS_THREADS) {
    const int i = e >> 5, j = e & 31;
    if (j >= i) tri[i * 32 - (i * (i - 1)) / 2 + (j - i)] = (uint16_t)((i << 8) | j);
  }
  for (int e = tid; e < 1024; e += SS_THREADS) aaug[e] = 0.f;
  {
    float* baug = reinterpret_cast<float*>(wslot + 16384);
    for (int e = tid; e < 512; e += SS_THREADS) baug[e] = 0.f;
  }
  if (tid == 0) {
    for (int b = 0; b < SS_NTB; ++b) {
      tc::mbar_init(&d1full[b], 1);
      tc::mbar_init(&d1empty[b], 128);
    }
    for (int b = 0; b < 2; ++b) {
      tc::mbar_init(&permd[b], 128);
      tc::mbar_init(&d2full[b], 2);
      tc::mbar_init(&d2empty[b], 128);
    }
    for (int b = 0; b < 4; ++b) tc::mbar_init(&pfree[b], 2);   // one commit per GEMM2 issuer
    for (int r = 0; r < SS_RAW; ++r) {
      tc::mbar_init(&landed[r], SS_GATHER);
      tc::mbar_init(&rfree[r], 128);
    }
    for (int b = 0; b < 2; ++b) {
      tc::mbar_init(&ready[b], SS_GATHER);
      tc::mbar_init(&sfree[b], 1);
    }
    tc::mbar_init(wfull, 32);
    tc::mbar_init(wempty, 1);
    tc::fence_barrier_init();
  }
  // Allocated before the grid dependency, possibly while CTAs of the previous kernel still run: safe because no CTA
  // that holds tensor memory can share an SM with this one (896 threads use nearly the whole register file; checked
  // on the host by sweep_pdl_ok, which otherwise launches this kernel without PDL).
  if (warp == 4) tc::tmem_alloc(tmem_slot, SS_TMEM_COLS);
  pdl_wait();
  pdl_launch_dependents();   // (the finalise kernel's CTAs cannot share an SM with this one: they queue behind it)
  // ---- cluster boundaries, centres ----
  for (int j = tid; j <= nkeys; j += SS_THREADS) B[j] = __ldg(a.seg_off + j);
  if (blockIdx.x == 0)
    for (int e = tid; e < 2 * nkeys * SS_D; e += SS_THREADS)
      a.centers[e] = __ldg(a.cen + (size_t)(e >> 6) * SS_D + (e & 31));
  __syncthreads();
  for (int r = tid; r < SS_TILE; r += SS_THREADS) {   // bias k-step A operand: (1, 1, 0, ...) per row
    float* p = aaug + (r >> 3) * 64 + (r & 7) * 4;
    p[0] = 1.f;
    p[1] = 1.f;
  }
  if (warp == 0) {   // exclusive prefix of tiles per cluster
    int carry = 0;
    if (lane == 0) P[0] = 0;
    for (int base = 0; base < nkeys; base += 32) {
      const int j = base + lane;
      int v = j < nkeys ? (B[j + 1] - B[j] + SS_TILE - 1) / SS_TILE : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
      }
      if (j < nkeys) P[j + 1] = carry + v;
      carry += __shfl_sync(0xffffffffu, v, 31);
    }
  }
  tc::fence_proxy_async();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int ntot = P[nkeys];
  const int t0 = (int)(((int64_t)ntot * blockIdx.x) / gridDim.x);
  const int t1 = (int)(((int64_t)ntot * (blockIdx.x + 1)) / gridDim.x);
  const int nt = t1 - t0;

  if (nt > 0) {
    if (warp < 4 || (warp >= 19 && warp < 23)) {
      // ======================= gather + shift + split =======================
      const int gtid = warp < 4 ? tid : tid - 608 + 128;   // 0..255
      const int c = gtid & 7, r0 = gtid >> 3;   // 16-byte chunk, first row; rows r0 + 32 j
      // raw ring and l panels: K-major rows of 128 bytes with the 128B swizzle.  The raw slot holds z and IS the
      // h operand of GEMM1: the tensor core reads the TF32 bits of z, i.e. h = trunc(z).
      const uint32_t offk = (uint32_t)(r0 * 128 + ((c ^ (r0 & 7)) << 4));
      const uint32_t offr = offk;
      StcWalk wl, wc;
      stc_walk_init(wl, B, P, nkeys, t0, t1);
      wc = wl;
      // The rows go straight into registers (no landing copy in shared memory): tile li + SS_PF is loaded into the
      // register set that tile li has just been stored from, and the indices of a tile are loaded one tile ahead
      // of its rows.  Rows past the end of the cluster load as exact zeros.
      int idx[4];
      auto load_idx = [&]() {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int p = wl.pos + r0 + 32 * j;
          idx[j] = p < wl.end ? __ldg(a.perm + p) : -1;
        }
      };
      auto load_rows = [&](float4 (&v)[4]) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const bool ok = idx[j] >= 0;
          v[j] = ldg_nc16(a.x + (size_t)(ok ? idx[j] : 0) * SS_D + 4 * c, ok);
        }
      };
      float4 va[4], vb[4];
      load_idx();   // (nt > 0 here)
      load_rows(va);
      stc_advance<SS_FLUSH>(wl, B);
      if (1 < nt) {
        load_idx();
        load_rows(vb);
        stc_advance<SS_FLUSH>(wl, B);
      }
      if (SS_PF < nt) load_idx();
      auto load_center = [&](int key) { return __ldg(reinterpret_cast<const float4*>(a.cen + (size_t)key * SS_D) + c); };
      int ckey = wc.key;
      float4 cen = load_center(ckey);
      auto tile = [&](int li, float4 (&v)[4]) {
        const int b = li & 1;
        if (wc.key != ckey) {
          ckey = wc.key;
          cen = load_center(ckey);
        }
        const int npts = wc.end - wc.pos;   // rows >= npts are zero padding
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (r0 + 32 * j < npts) {
            v[j].x -= cen.x; v[j].y -= cen.y; v[j].z -= cen.z; v[j].w -= cen.w;
          }
        }
        tc::mbar_wait(&rfree[li % SS_RAW], ((li / SS_RAW) & 1) ^ 1);   // the permuting pass of tile li - SS_RAW is done
        uint8_t* zk = raw0 + (size_t)(li % SS_RAW) * SS_PANEL + offr;
#pragma unroll
        for (int j = 0; j < 4; ++j) *reinterpret_cast<float4*>(zk + j * 4096) = v[j];
        tc::mbar_arrive(&landed[li % SS_RAW]);             // this thread's chunks of z are in shared memory
        tc::mbar_wait(&sfree[b], ((li >> 1) & 1) ^ 1);     // GEMM1 of tile li - 2 has read the l panel
        uint8_t* lk = split0 + (size_t)b * SS_PANEL + offk;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float4 lo;
          lo.x = v[j].x - tc::trunc_tf32(v[j].x); lo.y = v[j].y - tc::trunc_tf32(v[j].y);
          lo.z = v[j].z - tc::trunc_tf32(v[j].z); lo.w = v[j].w - tc::trunc_tf32(v[j].w);
          *reinterpret_cast<float4*>(lk + j * 4096) = lo;
        }
        tc::fence_proxy_async();
        tc::mbar_arrive(&ready[b]);
        const int ln = li + SS_PF;
        if (ln < nt) {
          load_rows(v);
          stc_advance<SS_FLUSH>(wl, B);
          if (ln + 1 < nt) load_idx();
        }
        stc_advance<SS_FLUSH>(wc, B);
      };
      static_assert(SS_PF == 2, "one register set per tile in flight: va, vb");
      for (int li = 0; li < nt; li += 2) {
        tile(li, va);
        if (li + 1 < nt) tile(li + 1, vb);
      }
    } else if (warp == 4) {
      // ======================= GEMM1 issuer =======================
      // (one thread; its instruction stream is a serial chain, so everything that does not change from
      //  tile to tile -- all thirteen descriptor pairs -- is computed once, and GEMM2 has its own issuer)
      {   // all 32 lanes run the loop (warp-uniform), one elected lane issues: see umma_tf32_*_w
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        StcWalk wm;
        stc_walk_init(wm, B, P, nkeys, t0, t1);
        const uint32_t idesc1 = tc::idesc_tf32(64);
        const uint64_t aaug_desc = tc::smem_desc_k_noswz(tc::smem_u32(aaug));
        const uint32_t ws = tc::smem_u32(wslot);
        const uint64_t baug_desc = tc::smem_desc_k_noswz(ws + 16384);
        const uint64_t raw_desc = tc::smem_desc_k128(tc::smem_u32(raw0)), l_desc = tc::smem_desc_k128(tc::smem_u32(split0));
        uint64_t whd[4], wld[4];
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          whd[ks] = tc::smem_desc_k128(ws) + ks * 2;
          wld[ks] = tc::smem_desc_k128(ws + 8192) + ks * 2;
        }
        int kj = -1, prevkey = -1;
        for (int li = 0; li < nt; ++li) {
          const int b = li & 1;
          if (wm.key != prevkey) {
            prevkey = wm.key;
            ++kj;
            tc::mbar_wait(wfull, kj & 1);
          }
          const int tb = li % SS_NTB, tph = (li / SS_NTB) & 1;
          tc::mbar_wait(&ready[b], (li >> 1) & 1);
          tc::mbar_wait(&d1empty[tb], tph ^ 1);
          tc::tc_fence_after();
          uint64_t hd[4], ld[4];
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            hd[ks] = raw_desc + (uint64_t)((li % SS_RAW) * (SS_PANEL >> 4) + ks * 2);   // z: h = its TF32 bits
            ld[ks] = l_desc + (uint64_t)(b * (SS_PANEL >> 4) + ks * 2);
          }
          const uint32_t tmem_d = tmem_u + tb * 64;
          tc::umma_tf32_first_w(tmem_d, hd[0], whd[0], idesc1);
#pragma unroll
          for (int ks = 1; ks < 4; ++ks) tc::umma_tf32_acc_w(tmem_d, hd[ks], whd[ks], idesc1);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) tc::umma_tf32_acc_w(tmem_d, ld[ks], whd[ks], idesc1);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) tc::umma_tf32_acc_w(tmem_d, hd[ks], wld[ks], idesc1);
          tc::umma_tf32_acc_w(tmem_d, aaug_desc, baug_desc, idesc1);   // Y -= b
          tc::umma_commit_w(&sfree[b]);
          tc::umma_commit_w(&d1full[tb]);
          if (wm.pos + SS_TILE >= wm.end) tc::umma_commit_w(wempty);   // last tile of the cluster
          stc_advance<SS_FLUSH>(wm, B);
        }
      }
    } else if (warp == 18 || warp == 23) {
      // ======================= GEMM2 issuers: warp 18 the left k-steps, warp 23 the right ones =======================
      // (the issue loop costs ~30 instructions per MMA in one dependent chain; each side's accumulator is
      //  written by exactly one issuer, in order)
      {
        const int right = warp == 23 ? 1 : 0;
        const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
        StcWalk wm;
        stc_walk_init(wm, B, P, nkeys, t0, t1);
        // M = 64.  (M = 128 with two garbage atoms after the panels, whose products land in accumulator rows
        // 64-127 that nobody reads, was measured 4 % slower, not faster.)
        const uint32_t idesc2 = tc::idesc_tf32_mn_m64(32);
        // A = [h | l] (two 32-row atoms, one panel apart), B = h: the same descriptor, one k-step = 8 rows = 1024 B
        const uint64_t pd0 = tc::smem_desc_mn128(tc::smem_u32(perm0), SS_PPANEL);
        const uint64_t pd1 = tc::smem_desc_mn128(tc::smem_u32(perm0 + 2 * SS_PPANEL), SS_PPANEL);
        int g2 = 0;
        for (int li = 0; li < nt; ++li) {
          const int b = li & 1;
          const bool first = wm.gcount == 0, last = stc_is_last<SS_FLUSH>(wm);
          tc::mbar_wait(&permd[b], (li >> 1) & 1);
          if (first) tc::mbar_wait(&d2empty[g2 & 1], ((g2 >> 1) & 1) ^ 1);
          tc::tc_fence_after();
          const int nkl = __shfl_sync(0xffffffffu, kcnt[b * 2], 0), nkr = __shfl_sync(0xffffffffu, kcnt[b * 2 + 1], 0);
          const int k0 = right ? nkl : 0, nk = right ? nkr : nkl;
          const uint32_t tm = tmem_u + SS_TMEM_G2 + (g2 & 1) * 64 + right * 32;
          uint64_t pd = (b ? pd1 : pd0) + (uint64_t)(k0 * 64);
          int ks = 0;
          if (first && nk > 0) {
            tc::umma_tf32_first_w(tm, pd, pd, idesc2);
            pd += 64;
            ks = 1;
          }
          for (; ks < nk; ++ks, pd += 64) tc::umma_tf32_acc_w(tm, pd, pd, idesc2);
          tc::umma_commit_w(&pfree[li & 3]);
          if (last) {
            tc::umma_commit_w(&d2full[g2 & 1]);
            ++g2;
          }
          stc_advance<SS_FLUSH>(wm, B);
        }
      }
    } else if (warp < 13 || warp >= 24) {
      // ======================= GEMM1 epilogue: draw, permute, sum y =======================
      const int g = warp >= 24 ? 2 + ((warp - 24) >> 2) : (warp - 5) >> 2;   // group g owns the tiles li = g (mod SS_NG)
      const int sub = warp & 3;                       // TMEM sub-partition of this warp
      const int row = (sub << 5) | lane;              // TMEM lane == row of the tile
      const int gt = warp >= 24 ? (tid - 768) & 127 : (tid - 160) & 127;   // 0..127 within the group
      uint8_t* const dest_g = dest_s + g * SS_TILE;
      volatile int32_t* const cnt_g = cnt_s + g * 4;
      int nacc = 0;
      const int c = gt & 7, r0 = gt >> 3;
      const uint32_t offr = (uint32_t)(r0 * 128 + ((c ^ (r0 & 7)) << 4));   // the gather warps' swizzled rows
      const uint32_t lt_mask = (1u << lane) - 1u;
      StcWalk we;
      stc_walk_init(we, B, P, nkeys, t0, t1);
      float sxl[4] = {0.f, 0.f, 0.f, 0.f}, sxr[4] = {0.f, 0.f, 0.f, 0.f};
      int ckey = -1;
      float cl = 0.f, cr = 0.f, lwl = 0.f, lwr = 0.f;
      for (int li = 0; li < nt; ++li) {
        if (li % SS_NG != g) {
          stc_advance<SS_FLUSH>(we, B);
          continue;
        }
        const int b = li & 1;                          // permuted-panel slot
        const int key = we.key;
        const int npts = min(SS_TILE, we.end - we.pos);
        const bool valid = row < npts;
        // everything that does not depend on the accumulator comes first: index, constants, uniform
        const int32_t idx = valid ? __ldg(a.perm + we.pos + row) : 0;
        if (key != ckey) {
          ckey = key;
          cl = __ldg(a.cst + 3 * key + 1); cr = __ldg(a.cst + 3 * key + 2);
          lwl = __ldg(a.loglr + 2 * key); lwr = __ldg(a.loglr + 2 * key + 1);

        }
        double u = 0.0;
        if (valid) u = dpmm_uniform(a.u_inj, idx, a.seed, DPMM_STREAM_SUBLABEL, a.call, (uint64_t)(a.goff + idx));
        const int tb = li % SS_NTB;
        tc::mbar_wait(&d1full[tb], (li / SS_NTB) & 1);
        tc::tc_fence_after();
        uint32_t v0[32], v1[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(sub * 32) << 16) + tb * 64;
        tc::tmem_ld32(taddr, v0);
        tc::tmem_ld32(taddr + 32, v1);
        tc::tmem_ld_wait();
        const float ql = gauss_tc_screen_q(v0), qr = gauss_tc_screen_q(v1);
        tc::tc_fence_before();
        tc::mbar_arrive(&d1empty[tb]);
        int side = 2;
        if (valid) {
          const float rl = gauss_finish(cl, ql, lwl), rr = gauss_finish(cr, qr, lwr);
          if (a.dump != nullptr) {
            a.dump[idx] = rl;
            a.dump[a.n + idx] = rr;
          }
          side = dpmm_draw_two(rl, rr, u);
          a.sub[idx] = (uint8_t)side;
        }
        // ---- destination row of every point: left run first, right run from a multiple of 8 ----
        const uint32_t bl = __ballot_sync(0xffffffffu, side == 0), br = __ballot_sync(0xffffffffu, side == 1);
        if (lane == 0) cnt_g[sub] = __popc(bl) | (__popc(br) << 8);
        asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
        int nl = 0, nr = 0, offl = 0, offr_ = 0;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const int cw = cnt_g[w];
          if (w < sub) {
            offl += cw & 255;
            offr_ += cw >> 8;
          }
          nl += cw & 255;
          nr += cw >> 8;
        }
        const int nl8 = max(8, (nl + 7) & ~7), nr8 = max(8, (nr + 7) & ~7);
        // rows beyond the end of the cluster hold exact zeros (zero-filled gather, not centred): they go to a
        // zero pad row of a run, or to a row no k-step reads, so that the copy below needs no branch
        const int dinv = nr8 > nr ? nl8 + nr8 - 1 : (nl8 > nl ? nl8 - 1 : nl8 + nr8);
        dest_g[row] = side == 0 ? (uint8_t)(offl + __popc(bl & lt_mask))
                                : (side == 1 ? (uint8_t)(nl8 + offr_ + __popc(br & lt_mask)) : (uint8_t)dinv);
        if (gt == 0 && nl > 0) atomicAdd(a.lcount + key, nl);
        tc::mbar_wait(&landed[li % SS_RAW], (li / SS_RAW) & 1);   // z of the tile (gathered and centred by the gather warps)
        if (li >= 2) tc::mbar_wait(&pfree[(li - 2) & 3], ((li - 2) >> 2) & 1);   // the GEMM2 that read this slot two tiles ago
        asm volatile("bar.sync %0, 128;" ::"r"(1 + g) : "memory");
        if (gt == 0) {
          kcnt[b * 2] = nl8 >> 3;
          kcnt[b * 2 + 1] = nr8 >> 3;
        }
        const uint8_t* rp = raw0 + (size_t)(li % SS_RAW) * SS_PANEL + offr;
        uint8_t* pp = perm0 + (size_t)b * 2 * SS_PPANEL;
        // z = x - c (centred in place).  The h panel takes z itself: the tensor core reads its TF32 bits,
        // h = trunc(z), the same split as GEMM1's; l = z - trunc(z) (|l| <= 2^-10 |z|, l l' is dropped).
        // Loads first, in two batches of four rows: the copies are independent but alias in the compiler's eyes.
        int dd[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) dd[j] = dest_g[r0 + 16 * j];
#pragma unroll
        for (int hb = 0; hb < 2; ++hb) {
          float4 y[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) y[j] = *reinterpret_cast<const float4*>(rp + (4 * hb + j) * 2048);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int d = dd[4 * hb + j];
            const float4 y4 = y[j];
            float4 l4;
            l4.x = y4.x - tc::trunc_tf32(y4.x); l4.y = y4.y - tc::trunc_tf32(y4.y);
            l4.z = y4.z - tc::trunc_tf32(y4.z); l4.w = y4.w - tc::trunc_tf32(y4.w);
            uint8_t* q = pp + d * 128 + (((((c >> 1) ^ (d & 3)) << 1) | (c & 1)) << 4);
            *reinterpret_cast<float4*>(q) = y4;
            *reinterpret_cast<float4*>(q + SS_PPANEL) = l4;
            const bool left = d < nl8;
            sxl[0] += left ? y4.x : 0.f; sxl[1] += left ? y4.y : 0.f; sxl[2] += left ? y4.z : 0.f; sxl[3] += left ? y4.w : 0.f;
            sxr[0] += left ? 0.f : y4.x; sxr[1] += left ? 0.f : y4.y; sxr[2] += left ? 0.f : y4.z; sxr[3] += left ? 0.f : y4.w;
          }
        }
        {   // zero rows that pad the two runs to a multiple of 8 (at most 8 + 8): thread = (row, chunk)
          const int z = gt >> 3, padl = nl8 - nl, padr = nr8 - nr;
          int d = -1;
          if (z < padl) d = nl + z;
          else if (z - padl < padr) d = nl8 + nr + (z - padl);
          if (d >= 0) {
            uint8_t* q = pp + d * 128 + (((((c >> 1) ^ (d & 3)) << 1) | (c & 1)) << 4);
            *reinterpret_cast<float4*>(q) = make_float4(0.f, 0.f, 0.f, 0.f);
            *reinterpret_cast<float4*>(q + SS_PPANEL) = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
        tc::fence_proxy_async();
        tc::mbar_arrive(&permd[b]);
        tc::mbar_arrive(&rfree[li % SS_RAW]);
        // sum y -> Float64 accumulators when this group's next tile (li + SS_NG) belongs to another cluster,
        // after 4 own tiles, or at the end of the range
        bool flush = we.tleft <= SS_NG || ++nacc == 4;
        if (!flush) {
          StcWalk w2 = we;
#pragma unroll
          for (int q = 0; q < SS_NG; ++q) stc_advance<SS_FLUSH>(w2, B);
          flush = w2.key != key;
        }
        if (flush) {
          nacc = 0;
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            sxl[q] += __shfl_xor_sync(0xffffffffu, sxl[q], 8);
            sxl[q] += __shfl_xor_sync(0xffffffffu, sxl[q], 16);
            sxr[q] += __shfl_xor_sync(0xffffffffu, sxr[q], 8);
            sxr[q] += __shfl_xor_sync(0xffffffffu, sxr[q], 16);
          }
          if (lane < 8) {   // lane == c for lanes 0-7
            double* dl = a.acc + (size_t)(2 * key) * a.rec + 1 + 4 * lane;
            double* dr = dl + a.rec;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              if (sxl[q] != 0.f) atomicAdd(dl + q, (double)sxl[q]);
              if (sxr[q] != 0.f) atomicAdd(dr + q, (double)sxr[q]);
            }
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) sxl[q] = sxr[q] = 0.f;
        }
        stc_advance<SS_FLUSH>(we, B);
      }
    } else if (warp < 17) {
      // ======================= GEMM2 accumulator drain =======================
      const int sub = warp & 3;
      const int gt = tid - 416;   // 0..127
      StcWalk wd;
      stc_walk_init(wd, B, P, nkeys, t0, t1);
      int g2 = 0;
      for (int li = 0; li < nt; ++li) {
        if (stc_is_last<SS_FLUSH>(wd)) {
          const int buf = g2 & 1;
          tc::mbar_wait(&d2full[buf], (g2 >> 1) & 1);
          ++g2;
          tc::tc_fence_after();
          uint32_t v0[32], v1[32];
          const uint32_t taddr = tmem_base + SS_TMEM_G2 + buf * 64 + ((uint32_t)(sub * 32) << 16);
          tc::tmem_ld32(taddr, v0);
          tc::tmem_ld32(taddr + 32, v1);
          tc::tmem_ld_wait();
          tc::tc_fence_before();
          tc::mbar_arrive(&d2empty[buf]);
          // M = 64: accumulator row m lives in lane (m % 16) of sub-partition m / 16
          if (lane < 16) {
            float* trow = T + (16 * sub + lane) * SS_TLD;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              trow[j] = __uint_as_float(v0[j]);
              trow[32 + j] = __uint_as_float(v1[j]);
            }
          }
          asm volatile("bar.sync 6, 128;" ::: "memory");
          for (int e = gt; e < 2 * 528; e += 128) {
            const int sd = e >= 528 ? 1 : 0;
            const int ij = tri[e - sd * 528], i = ij >> 8, j = ij & 255;
            const int co = 32 * sd;
            const float sv = (T[i * SS_TLD + co + j] + T[(32 + i) * SS_TLD + co + j]) + T[(32 + j) * SS_TLD + co + i];
            if (sv != 0.f) atomicAdd(a.acc + (size_t)(2 * wd.key + sd) * a.rec + 1 + SS_D + i * SS_D + j, (double)sv);
          }
          asm volatile("bar.sync 6, 128;" ::: "memory");
        }
        stc_advance<SS_FLUSH>(wd, B);
      }
    } else if (warp == 17) {
      // ======================= factor staging (warp 17) =======================
      StcWalk wp;
      stc_walk_init(wp, B, P, nkeys, t0, t1);
      int kj = 0, prevkey = -1;
      float* wh = reinterpret_cast<float*>(wslot);
      float* wlo = wh + 2048;
      float* baug = wh + 4096;
      for (int li = 0; li < nt; ++li) {
        if (wp.key != prevkey) {
          prevkey = wp.key;
          tc::mbar_wait(wempty, (kj & 1) ^ 1);   // every GEMM1 of the previous cluster has retired
          const float4* src = reinterpret_cast<const float4*>(a.w + (size_t)wp.key * 2 * SS_D * SS_D);
          for (int e = lane; e < 512; e += 32) {
            const int r = e >> 3, cc = e & 7;   // row (side, i), 16-byte chunk
            const float4 v = __ldg(src + e);
            float4 hi, lo;
            hi.x = tc::to_tf32(v.x); hi.y = tc::to_tf32(v.y); hi.z = tc::to_tf32(v.z); hi.w = tc::to_tf32(v.w);
            lo.x = v.x - hi.x; lo.y = v.y - hi.y; lo.z = v.z - hi.z; lo.w = v.w - hi.w;
            const int o = r * SS_D + ((cc ^ (r & 7)) << 2);
            *reinterpret_cast<float4*>(wh + o) = hi;
            *reinterpret_cast<float4*>(wlo + o) = lo;
          }
          for (int r = lane; r < 64; r += 32) {
            const float bv = __ldg(a.bias + (size_t)wp.key * 64 + r);
            const float bhi = tc::to_tf32(bv), blo = bv - bhi;
            float* p = baug + (r >> 3) * 64 + (r & 7) * 4;
            p[0] = -bhi;
            p[1] = -blo;
          }
          tc::fence_proxy_async();
          tc::mbar_arrive(wfull);
          ++kj;
        }
        stc_advance<SS_FLUSH>(wp, B);
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 4) tc::tmem_dealloc(tmem_base, SS_TMEM_COLS);
}
