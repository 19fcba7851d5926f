// K2 (second generation): fused Gaussian log-likelihood + label draw on tcgen05 for D = 32 and D = 64,
// any K that fits the shared-memory images (K <= ~250 at D = 32, ~110 at D = 64).
//
//   sample_labels_worker!        src/local_clusters_actions.jl:112-134
//   log_likelihood!(mv_gaussian) src/distributions/mv_gaussian.jl:21-25
//   sample_log_cat_array!        src/utils.jl:19-31
//
// The points are visited in the order of the CURRENT label sort (perm / seg_off of kernels_sort.cuh), so a
// tile = 128 consecutive positions of ONE old cluster p, the tile's PIVOT.  At every iteration but the first
// few almost every point keeps its label, so the pivot is the cluster that decides the draw, and because it
// is uniform over the tile everything below is warp-uniform:
//
//  0. CENTRE: the gather warps shift the tile by the pivot's mean, z = x - mu_p.  The TF32
//     error of everything below is proportional to |z| (the spread of a cluster), not to |x|.
//  1. PIVOT (tcgen05, kind::tf32): Y_p = Z U_p' for the full factor of the pivot (D columns).
//     q~_p = |y|^2 carries a bounded TF32 error, so it yields a LOWER bound of r_p (see kernels_gauss_tc.cuh).
//  2. SCREEN (tcgen05): for EVERY cluster k only R = 8 rows of its factor:  q_k >= |rows of U_k (x - mu_k)|^2.
//     Either the first 8 rows of U_k over all features (KS = D) or the last 8 rows, which only involve the
//     last 8 features (KS = 8: the marginal Mahalanobis distance in those features; 1 k-step instead of D/8).
//     Y = Z U_k[rows]' - U_k[rows] (mu_k - mu_p), the second term from a per-pivot bias table (niw_t2_bias_kernel)
//     folded in as one more k-step.  That gives an UPPER bound of r_k from 8 accumulator columns instead of D.
//     Cluster k is a candidate of the point iff that upper bound reaches within DELTA = 30 of the pivot's
//     lower bound.
//  3. A point without candidates keeps the pivot: every other weight is < e^-30 of the pivot's, and no
//     uniform is drawn.  Otherwise the pivot and the <= 7 candidates are evaluated EXACTLY on the FMA pipe
//     (z = x - mu in Float32, |U z|^2, the reference's final operations) and drawn with the reference's
//     inverse-CDF walk over those entries (all others contribute exact zeros to every sum).
//  4. Points with a NaN / Inf screen value or more than 7 candidates go to an overflow list that
//     gauss_label_list_kernel finishes with the full K-cluster evaluation (one warp per point).
//
// Per tile the tensor core therefore produces D + 8K accumulator columns (C2: 192 instead of 640) and the
// epilogue reads exactly those.  The factor images live in shared memory in the un-swizzled K-major core
// matrix layout (8 rows x 16 bytes), written in that layout by niw_pack_kernel, so any K is a matter of
// more 16-cluster chunks, not of a resident K x D x D block.
//
// Warp roles (384 threads, one CTA per SM, contiguous range of the tile sequence per CTA):
//   warps 0/1   control of point-group 0/1 (pivot image staging + tcgen05.mma issue)
//   warps 2-5 / 6-9  epilogue (TMEM lane = point) of group 0/1, alternate tiles
//   warps 10-13 gather: the 128 rows of a tile into a 128B-swizzled K-major stage ring, centred -- at D = 32 through
//               registers (one store per row chunk), at D = 64 (warps 10-11) by cp.async and centring in place
#pragma once
#include "tcgen05.cuh"
#include "kernels_gauss.cuh"   // gauss_finish
#include "kernels_stats.cuh"   // cp_async16 / commit / wait_group

#define T2_TILE 128
// per-call counter set: [0] points, [1] exact evaluations, [2] overflow points, [3] scan ticket, [4] moved points
#define T2_CTR_SET 8
#define T2_PRODUCERS(D) ((D) == 32 ? 128 : 64)   // gather threads (warps 10-13 / 10-11): D = 64 needs the registers
#define T2_THREADS(D) (320 + T2_PRODUCERS(D))
#define T2_CMAX 8          // exact evaluations per point handled in the kernel (pivot included)
#define T2_R 8             // screen rows per cluster
#define T2_DELTA 30.0f
#define T2_MAX_K 256        // bias tables are K x K
#define T2_COOP_MAX 12      // candidate pairs in a warp up to which they are evaluated one at a time by all lanes
// (measured and rejected: sending the candidate points of a warp with more pairs than that to the overflow list --
//  the all-K list kernel then costs 6 ms on the overlapping-clusters state of C2, against 1 ms evaluated in place)
#define T2_NS32 4          // stage ring at D = 32 (D = 64: 3)

struct GaussTc2Args {
  const float* x;          // [n][D]
  int64_t n;
  int K, KS, nch, n0;      // KS = features of the screen (8 or D); nch chunks; n0 clusters in chunk 0
  const int32_t* perm;     // [n] point indices sorted by the labels at call time
  const int32_t* seg_off;  // [nkeys + 1]
  int nkeys;
  const float* wpiv;       // [K][D*D]  pivot image: D/8 k-step slabs
  const float* wscr;       // [nch][(KS/8) * 1024] screen images
  const float* wbias;      // [K pivots][nch * 512 + 32] bias tables (compact B operand of the bias k-step)
  const float* urows;      // [K][D][D] rows of U_k (zero below the diagonal)
  const float* mu;         // [K][D]
  const float* cst;        // [3K]
  const float* logw;       // [K]
  const float* fro;        // [K] |U_k|_F
  const float* fro8;       // [K] |screen rows of U_k|_F
  int32_t* labels;
  int32_t* hist;
  int32_t* ovf_list;       // [n]
  int32_t* ovf_count;      // [1]
  const double* u_inj;
  uint64_t seed;
  uint32_t call;
  int64_t goff;
  int final_iter;
  int32_t* stats;          // optional [2]: points, exact evaluations
  int32_t* moved;          // [1] += points whose new label differs from their old one (the pivot)
};

struct GaussTc2Smem {
  int ns, pf;
  size_t stage_bytes, piv_bytes, scr_bytes, bias_bytes;
  size_t stages, piv, scr, bias, aaug, ccfro, scrc, cfin, lists, rlists, pairs, misc, bnd, pre, hist, bars, total;
  __host__ __device__ GaussTc2Smem(int D, int K, int KS, int nch, int nkeys) {
    ns = D == 32 ? T2_NS32 : 3;
    pf = ns - 2;
    stage_bytes = (size_t)T2_TILE * D * 4;
    piv_bytes = (size_t)(D * D) * 4;
    scr_bytes = (size_t)(KS / 8) * 4096;
    bias_bytes = (size_t)nch * 2048 + 128;
    size_t o = 0;
    stages = o;  o += ns * stage_bytes;
    piv = o;     o += 2 * piv_bytes;
    scr = o;     o += (size_t)nch * scr_bytes;
    bias = o;    o += 2 * bias_bytes;
    aaug = o;    o += 4096;
    ccfro = o;   o += (size_t)K * 8;
    o = (o + 15) & ~(size_t)15;
    scrc = o;    o += (size_t)(nch * 8 + 8) * 16;
    cfin = o;    o += (size_t)K * 8;
    o = (o + 15) & ~(size_t)15;
    lists = o;   o += 2 * T2_TILE * T2_CMAX * 2;
    rlists = o;  o += 2 * T2_TILE * T2_CMAX * 4;
    pairs = o;   o += 2 * T2_TILE * T2_CMAX * 2;
    misc = o;    o += 2 * 16 * 4;
    bnd = o;     o += (size_t)(nkeys + 1) * 4;
    pre = o;     o += (size_t)(nkeys + 1) * 4;
    hist = o;    o += (size_t)((K + 3) & ~3) * 4;
    o = (o + 15) & ~(size_t)15;
    bars = o;    o += 32 * 8 + 16;
    total = o;
  }
};
__host__ __device__ inline int gauss_tc2_n0(int D) { return (128 - D) / T2_R; }
__host__ __device__ inline int gauss_tc2_nch(int D, int K) {
  const int n0 = gauss_tc2_n0(D);
  return K <= n0 ? 1 : 1 + (K - n0 + 15) / 16;
}

// The tile sequence (tiles of <= 128 positions that never straddle a key boundary) is cut into G * T2_ROUNDS segments of
// equal length (+-1) and segment i goes to CTA i mod G: every CTA gets the same number of tiles (+-T2_ROUNDS) and
// still sees runs of one pivot (its image is staged once per run), but a cluster whose tiles are expensive -- every
// point carrying candidates because a neighbour overlaps it -- is spread over many CTAs instead of making the one CTA
// that owned its contiguous range the straggler of the launch (C5 with freshly sampled parameters: 6.0 -> 2.4 ms).
// Every new run re-stages the pivot image behind a drained MMA pipeline (~1.5 us), so the number of rounds adapts:
// segments of at least T2_SEG_MIN tiles, at most T2_ROUNDS rounds (C2, 53 tiles per CTA: one contiguous range as
// before; 8 rounds of 6.6 tiles cost it 76.6 -> 88 us).
#define T2_ROUNDS 8
#define T2_SEG_MIN 32
struct T2Seq {
  const int32_t* B;   // [nkeys + 1] key boundaries (positions)
  const int32_t* P;   // [nkeys + 1] exclusive prefix of tiles per key
  int nkeys, ntot, G, cta, R;   // R rounds: min(T2_ROUNDS, max(1, ntot / (G * T2_SEG_MIN)))
};
struct T2Walk {
  int key, pos, end, tleft;
  int t, send, seg;   // global tile index, end of the current segment, its index
};
__device__ __forceinline__ int t2_seg_begin(const T2Seq& q, int seg) {
  return (int)(((int64_t)q.ntot * seg) / ((int64_t)q.G * q.R));
}
// tiles CTA `cta` owns: segments cta, cta + G, ...
__device__ __forceinline__ int t2_cta_tiles(const T2Seq& q) {
  int n = 0;
  for (int r = 0; r < q.R; ++r) n += t2_seg_begin(q, q.cta + r * q.G + 1) - t2_seg_begin(q, q.cta + r * q.G);
  return n;
}
__device__ __forceinline__ void t2_seek(T2Walk& w, const T2Seq& q, int t) {
  int lo = 0, hi = q.nkeys - 1;   // first key with P[key + 1] > t
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (q.P[mid + 1] > t) hi = mid;
    else lo = mid + 1;
  }
  w.key = lo;
  w.pos = q.B[lo] + (t - q.P[lo]) * T2_TILE;
  w.end = q.B[lo + 1];
  w.t = t;
}
// first non-empty segment of this CTA at or after `seg`
__device__ __forceinline__ void t2_enter(T2Walk& w, const T2Seq& q, int seg) {
  int b = t2_seg_begin(q, seg), e = t2_seg_begin(q, seg + 1);
  while (e <= b) {
    seg += q.G;
    b = t2_seg_begin(q, seg);
    e = t2_seg_begin(q, seg + 1);
  }
  w.seg = seg;
  w.send = e;
  t2_seek(w, q, b);
}
__device__ __forceinline__ void t2_walk_init(T2Walk& w, const T2Seq& q) {
  w.tleft = t2_cta_tiles(q);
  w.key = 0; w.pos = 0; w.end = 0; w.t = 0; w.send = 0; w.seg = q.cta;
  if (w.tleft > 0) t2_enter(w, q, q.cta);
}
__device__ __forceinline__ void t2_advance(T2Walk& w, const T2Seq& q) {
  --w.tleft;
  if (w.tleft <= 0) return;
  ++w.t;
  if (w.t >= w.send) {                       // next segment of this CTA
    t2_enter(w, q, w.seg + q.G);
    return;
  }
  w.pos += T2_TILE;
  if (w.pos >= w.end) {
    do ++w.key; while (q.B[w.key + 1] == q.B[w.key]);
    w.pos = q.B[w.key];
    w.end = q.B[w.key + 1];
  }
}

// exact q = |U_k (x - mu_k)|^2, rows of U_k and mu_k read through the read-only path; the point is supplied
// as 16-byte chunks by `ld4(c)`.  Same arithmetic and order as gauss_tc_exact_q.
template <int D, typename LD4>
__device__ __forceinline__ float gauss_tc2_exact_q_impl(const float* __restrict__ U, const float* __restrict__ mu, LD4 ld4) {
  f32x2_t z2[D / 2];
#pragma unroll
  for (int c = 0; c < D / 4; ++c) {
    const float4 v = ld4(c);
    const float4 m = __ldg(reinterpret_cast<const float4*>(mu) + c);
    z2[2 * c] = f2_pack(v.x - m.x, v.y - m.y);
    z2[2 * c + 1] = f2_pack(v.z - m.z, v.w - m.w);
  }
  float q0 = 0.f, q1 = 0.f;
#pragma unroll
  for (int i = 0; i < D; ++i) {
    const float* row = U + i * D;
    f32x2_t acc = 0ull;
    float4 uf[D / 4];   // the whole row first: the loads are independent, the FMA chain is not
#pragma unroll
    for (int c = i >> 2; c < D / 4; ++c) uf[c] = __ldg(reinterpret_cast<const float4*>(row) + c);
#pragma unroll
    for (int c = i >> 2; c < D / 4; ++c) {
      acc = f2_fma(f2_pack(uf[c].x, uf[c].y), z2[2 * c], acc);
      acc = f2_fma(f2_pack(uf[c].z, uf[c].w), z2[2 * c + 1], acc);
    }
    float lo, hi;
    f2_unpack(acc, lo, hi);
    const float y = lo + hi;
    if (i & 1) q1 = fmaf(y, y, q1); else q0 = fmaf(y, y, q0);
  }
  return q0 + q1;
}
// the point = a row of X in global memory (the staged tile holds z = x - mu_pivot, not x)
template <int D>
__device__ __noinline__ float gauss_tc2_exact_q_row(const float* __restrict__ U, const float* __restrict__ mu,
                                                    const float* __restrict__ xr) {
  return gauss_tc2_exact_q_impl<D>(U, mu, [&](int c) { return __ldg(reinterpret_cast<const float4*>(xr) + c); });
}

// The same quadratic form evaluated by a whole warp for ONE (point, cluster) pair: lane <-> rows lane, lane + 32, ... of
// U_k (all of a row's loads are independent, rows run in parallel across lanes), then a butterfly sum.  One pair
// costs about two L2 round trips instead of D dependent ones, which is what matters when a tile has only a few
// candidate pairs: with one pair per lane such a tile waited ~20 us for a single lane (D = 64), and a cluster whose
// points all carry a candidate made its CTA the straggler of the whole launch (C5: 4.3 ms, of which 1.9 ms work).
// Rows hold exact zeros below the diagonal, so the full-row dot equals the triangular one; the sum over rows is
// taken in a different order than gauss_tc2_exact_q_impl (last-ulp freedom, as the reference's @fastmath dot has).
template <int D>
__device__ __noinline__ float gauss_tc2_exact_q_coop(const float* __restrict__ U, const float* __restrict__ mu,
                                                     const float* __restrict__ xr, int lane) {
  f32x2_t z2[D / 2];
#pragma unroll
  for (int c = 0; c < D / 4; ++c) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(xr) + c);
    const float4 m = __ldg(reinterpret_cast<const float4*>(mu) + c);
    z2[2 * c] = f2_pack(v.x - m.x, v.y - m.y);
    z2[2 * c + 1] = f2_pack(v.z - m.z, v.w - m.w);
  }
  float q = 0.f;
#pragma unroll
  for (int r = 0; r < D / 32; ++r) {
    const float4* row = reinterpret_cast<const float4*>(U + (size_t)(lane + 32 * r) * D);
    float4 uf[D / 4];
#pragma unroll
    for (int c = 0; c < D / 4; ++c) uf[c] = __ldg(row + c);
    f32x2_t acc = 0ull;
#pragma unroll
    for (int c = 0; c < D / 4; ++c) {
      acc = f2_fma(f2_pack(uf[c].x, uf[c].y), z2[2 * c], acc);
      acc = f2_fma(f2_pack(uf[c].z, uf[c].w), z2[2 * c + 1], acc);
    }
    float lo, hi;
    f2_unpack(acc, lo, hi);
    const float y = lo + hi;
    q = fmaf(y, y, q);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  return q;
}

// sample_log_cat_array! (utils.jl:19-31) over the m listed clusters (ascending indices ks[], values rs[]);
// every unlisted cluster has weight exactly 0.  Mirrors dpmm_draw_inverse_cdf_masked.
__device__ __forceinline__ int gauss_tc2_draw_list(const uint16_t* ks, float* rs, int m, int K, double u) {
  float mx = -CUDART_INF_F;
  for (int j = 0; j < m; ++j) mx = fmaxf(mx, rs[j]);
  float s = 0.f;
  for (int j = 0; j < m; ++j) {
    const float e = expf(rs[j] - mx);
    rs[j] = e;
    s = __fadd_rn(s, e);
  }
  const bool s_regular = (s > 0.f) && (s < CUDART_INF_F);
  float cw = 0.f;
  for (int j = 0; j < m; ++j) {
    const float e = rs[j];
    const bool zero = (e < 1.17549435e-38f) && s_regular;
    const float quo = __fdiv_rn(zero ? 1.f : e, s);
    cw = __fadd_rn(cw, zero ? 0.f : quo);
    rs[j] = cw;
  }
  const double t = u * (double)cw;
  if (!(0.0 < t) && ks[0] != 0) return 0;   // cw_1 = w_1 = 0 is not < t: the walk stops at i = 1
  for (int j = 0; j < m; ++j) {
    const int k = ks[j];
    if (k >= K - 1) break;
    if (!((double)rs[j] < t)) return k;
  }
  return K - 1;
}

__device__ __forceinline__ float t2_sum8(const uint32_t* v) {
  const f32x2_t p0 = f2_pack(__uint_as_float(v[0]), __uint_as_float(v[1]));
  const f32x2_t p1 = f2_pack(__uint_as_float(v[2]), __uint_as_float(v[3]));
  const f32x2_t p2 = f2_pack(__uint_as_float(v[4]), __uint_as_float(v[5]));
  const f32x2_t p3 = f2_pack(__uint_as_float(v[6]), __uint_as_float(v[7]));
  f32x2_t a0 = f2_fma(p0, p0, 0ull), a1 = f2_fma(p1, p1, 0ull);
  a0 = f2_fma(p2, p2, a0);
  a1 = f2_fma(p3, p3, a1);
  float x0, x1, y0, y1;
  f2_unpack(a0, x0, x1);
  f2_unpack(a1, y0, y1);
  return (x0 + x1) + (y0 + y1);
}

template <int D>
__global__ void __launch_bounds__(T2_THREADS(D), 1) gauss_label_tc2_kernel(const GaussTc2Args a) {
  extern __shared__ __align__(1024) uint8_t t2_smem[];
  uint8_t* const smem = t2_smem;
  const int K = a.K, KS = a.KS, nch = a.nch, n0 = a.n0, nkeys = a.nkeys;
  const GaussTc2Smem L(D, K, KS, nch, nkeys);
  constexpr int NS = D == 32 ? T2_NS32 : 3;
  constexpr int PF = NS - 2;
  constexpr int PIVF = D * D;                     // floats of a pivot image
  uint8_t* stage0 = smem + L.stages;
  float* pivsm = reinterpret_cast<float*>(smem + L.piv);
  float* scrsm = reinterpret_cast<float*>(smem + L.scr);
  float* aaug = reinterpret_cast<float*>(smem + L.aaug);
  float2* ccfro = reinterpret_cast<float2*>(smem + L.ccfro);    // (log w_k - c_k, |U_k|_F)
  float4* scrc = reinterpret_cast<float4*>(smem + L.scrc);      // by slot pair (A, B): (4.0816 cc_A, 4.0816 cc_B, |rows_A|_F, |rows_B|_F); pad: (-inf, 0)
  uint8_t* biassm = smem + L.bias;
  float2* cfin = reinterpret_cast<float2*>(smem + L.cfin);      // (c_k, log w_k)
  uint16_t* lists_all = reinterpret_cast<uint16_t*>(smem + L.lists);
  float* rl_all = reinterpret_cast<float*>(smem + L.rlists);
  uint16_t* pairs_all = reinterpret_cast<uint16_t*>(smem + L.pairs);
  int32_t* B = reinterpret_cast<int32_t*>(smem + L.bnd);
  int32_t* P = reinterpret_cast<int32_t*>(smem + L.pre);
  int* hs = reinterpret_cast<int*>(smem + L.hist);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L.bars);
  uint64_t* full = bars;              // [NS]    tile gathered into stage s
  uint64_t* empty = bars + 8;         // [NS]    stage s released by the 128 epilogue threads of its tile
  uint64_t* tfull = bars + 16;        // [2][2]  accumulator buffer (group, b) ready
  uint64_t* tempty = bars + 20;       // [2][2]  ... drained
  uint64_t* wdone = bars + 24;        // [2]     all MMAs of the group's previous tile retired
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 32);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0) {
    for (int i = 0; i < NS; ++i) {
      tc::mbar_init(&full[i], T2_PRODUCERS(D));
      tc::mbar_init(&empty[i], 128);
    }
    for (int i = 0; i < 4; ++i) {
      tc::mbar_init(&tfull[i], 1);
      tc::mbar_init(&tempty[i], 128);
    }
    tc::mbar_init(&wdone[0], 1);
    tc::mbar_init(&wdone[1], 1);
    tc::fence_barrier_init();
  }
  // Tensor memory is allocated before the grid dependency, possibly while CTAs of the previous kernel still run: safe
  // because no CTA that holds tensor memory can share an SM with this one (their register files do not fit together;
  // checked on the host by sweep_pdl_ok, which otherwise launches this kernel without PDL).
  if (warp == 1) tc::tmem_alloc(tmem_ptr, 512);
  pdl_wait();
  pdl_launch_dependents();   // (the overflow kernel's CTAs cannot share an SM with this one: they queue behind it)
  for (int j = tid; j <= nkeys; j += T2_THREADS(D)) B[j] = __ldg(a.seg_off + j);
  {   // screen images: already in the shared-memory layout
    const int nf4 = nch * (KS / 8) * 256;
    const float4* src = reinterpret_cast<const float4*>(a.wscr);
    float4* dst = reinterpret_cast<float4*>(scrsm);
    for (int e = tid; e < nf4; e += T2_THREADS(D)) dst[e] = __ldg(src + e);
  }
  for (int e = tid; e < 1024; e += T2_THREADS(D)) aaug[e] = 0.f;
  for (int k = tid; k < K; k += T2_THREADS(D)) {
    const float c = __ldg(a.cst + 3 * k), lw = __ldg(a.logw + k);
    ccfro[k] = make_float2(lw - c, __ldg(a.fro + k));
    cfin[k] = make_float2(c, lw);
    hs[k] = 0;
  }
  for (int e = tid; e < nch * 16 + 16; e += T2_THREADS(D)) {   // screen slot e: chunk 0 holds n0 clusters, the others 16
    const int ch = e >> 4, j = e & 15;
    const int k = ch == 0 ? (j < n0 ? j : K) : n0 + (ch - 1) * 16 + j;
    float* q = reinterpret_cast<float*>(scrc + (e >> 1)) + (e & 1);
    q[0] = k < K ? 4.0816f * (__ldg(a.logw + k) - __ldg(a.cst + 3 * k)) : -CUDART_INF_F;
    q[2] = k < K ? __ldg(a.fro8 + k) : 0.f;
  }
  __syncthreads();
  for (int r = tid; r < T2_TILE; r += T2_THREADS(D)) {   // bias k-step A operand: (1, 1, 0, ...) per row
    float* p = aaug + (r >> 3) * 64 + (r & 7) * 4;
    p[0] = 1.f;
    p[1] = 1.f;
  }
  if (warp == 0) {   // exclusive prefix of tiles per key
    int carry = 0;
    if (lane == 0) P[0] = 0;
    for (int base = 0; base < nkeys; base += 32) {
      const int j = base + lane;
      int v = j < nkeys ? (B[j + 1] - B[j] + T2_TILE - 1) / T2_TILE : 0;
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
  const uint32_t tmem_base = *tmem_ptr;
  const int ntot = P[nkeys];
  const T2Seq seq{B, P, nkeys, ntot, (int)gridDim.x, (int)blockIdx.x,
                  min(T2_ROUNDS, max(1, ntot / ((int)gridDim.x * T2_SEG_MIN)))};
  const int nt = t2_cta_tiles(seq);

  if (nt > 0) {
    if (warp < 2) {
      // =============================== control warp of group g ===============================
      const int g = warp;
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      float* pivs = pivsm + (size_t)g * PIVF;
      float* biasg = reinterpret_cast<float*>(biassm + (size_t)g * L.bias_bytes);
      const int bias_f4 = (int)(L.bias_bytes / 16);
      const uint32_t pivs_a = tc::smem_u32(pivs), scr_a = tc::smem_u32(scrsm), bias_a = tc::smem_u32(biasg);
      const uint64_t aaug_desc = tc::smem_desc_k_noswz(tc::smem_u32(aaug));
      const uint32_t scr_stride = (uint32_t)L.scr_bytes;
      T2Walk w;
      t2_walk_init(w, seq);
      uint32_t cc = 0;
      int prevkey = -1, ntile_g = 0;
      for (int li = 0; li < nt; ++li, t2_advance(w, seq)) {
        if ((li & 1) != g) continue;
        const int s = li % NS;
        const int key = min(w.key, K - 1);
        tc::mbar_wait(&full[s], (li / NS) & 1);
        tc::tc_fence_after();
        const uint32_t st_a = tc::smem_u32(stage0 + (size_t)s * L.stage_bytes);
        for (int c = 0; c < nch; ++c, ++cc) {
          const int b = cc & 1;
          tc::mbar_wait(&tempty[g * 2 + b], ((cc >> 1) & 1) ^ 1);   // epilogue drained this buffer
          tc::tc_fence_after();
          const uint32_t tmem_d = tmem_u + g * 256 + b * 128;
          int col = 0;
          if (c == 0) {
            if (key != prevkey) {
              // (at most the previous tile's MMAs are outstanding here: the buffer wait above ordered the rest)
              if (ntile_g > 0) tc::mbar_wait(&wdone[g], (ntile_g - 1) & 1);
              const float4* src = reinterpret_cast<const float4*>(a.wpiv + (size_t)key * PIVF);
              float4* dst = reinterpret_cast<float4*>(pivs);
              for (int e = lane; e < PIVF / 4; e += 32) dst[e] = __ldg(src + e);
              const float4* bsrc = reinterpret_cast<const float4*>(a.wbias + (size_t)key * (bias_f4 * 4));
              float4* bdst = reinterpret_cast<float4*>(biasg);
              for (int e = lane; e < bias_f4; e += 32) bdst[e] = __ldg(bsrc + e);
              tc::fence_proxy_async();
              __syncwarp();
              prevkey = key;
            }
            const uint32_t idp = tc::idesc_tf32(D);
#pragma unroll
            for (int ks = 0; ks < D / 8; ++ks) {
              const uint64_t ad = tc::smem_desc_k128(st_a + (ks >> 2) * 16384) + (uint64_t)((ks & 3) * 2);
              const uint64_t bd = tc::smem_desc_k_noswz(pivs_a + ks * (D * 32));
              if (ks == 0) tc::umma_tf32_first_w(tmem_d, ad, bd, idp);
              else tc::umma_tf32_acc_w(tmem_d, ad, bd, idp);
            }
            col = D;   // (no bias: the tile is centred by the pivot's own mean)
          }
          const int ncl = c == 0 ? min(K, n0) : min(16, K - n0 - (c - 1) * 16);
          const uint32_t ids = tc::idesc_tf32((ncl * T2_R + 15) & ~15);
          const uint32_t sc = scr_a + c * scr_stride;
          const int nks = KS >> 3;
          for (int ks = 0; ks < nks; ++ks) {
            const int ka = (KS == D) ? ks : (D / 8 - 1);   // KS = 8: the last 8 features
            const uint64_t ad = tc::smem_desc_k128(st_a + (ka >> 2) * 16384) + (uint64_t)((ka & 3) * 2);
            const uint64_t bd = tc::smem_desc_k_noswz(sc + ks * 4096);
            if (ks == 0) tc::umma_tf32_first_w(tmem_d + col, ad, bd, ids);
            else tc::umma_tf32_acc_w(tmem_d + col, ad, bd, ids);
          }
          // bias k-step: B = compact [128 rows][4] table; its second k half (LBO = 128 B) aliases the next row
          // group, finite values that meet the zero half of the A operand
          tc::umma_tf32_acc_w(tmem_d + col, aaug_desc, tc::smem_desc_k_noswz2(bias_a + c * 2048, 128, 128), ids);
          tc::umma_commit_w(&tfull[g * 2 + b]);
        }
        tc::umma_commit_w(&wdone[g]);
        ++ntile_g;
      }
    } else if (warp < 10) {
      // ======================= epilogue: bounds, candidates, refine, draw =======================
      const int g = (warp - 2) >> 2;
      const int gt = tid - 64 - g * 128;                     // thread index within the group
      const int wq = gt >> 5;                                // warp within the group
      const int row = ((warp & 3) << 5) | lane;              // TMEM lane == point within the tile
      const uint32_t tmem_row = tmem_base + ((uint32_t)((warp & 3) << 5) << 16) + g * 256;
      uint16_t* lists = lists_all + (size_t)g * T2_TILE * T2_CMAX;
      float* rl = rl_all + (size_t)g * T2_TILE * T2_CMAX;
      uint16_t* pairs = pairs_all + (size_t)g * T2_TILE * T2_CMAX;
      uint16_t* mylist = lists + row * T2_CMAX;
      float* myrl = rl + row * T2_CMAX;
      T2Walk w;
      t2_walk_init(w, seq);
      uint32_t cc = 0;
      int ncand_total = 0, npts_total = 0;
      for (int li = 0; li < nt; ++li, t2_advance(w, seq)) {
        if ((li & 1) != g) continue;
        const int s = li % NS;
        const int key = min(w.key, K - 1);
        const int npts = min(T2_TILE, w.end - w.pos);
        const bool valid = row < npts;
        const int32_t idx = valid ? __ldg(a.perm + w.pos + row) : 0;
        const float* stage = reinterpret_cast<const float*>(stage0 + (size_t)s * L.stage_bytes);
        tc::mbar_wait(&full[s], (li / NS) & 1);
        float xnorm;
        {
          f32x2_t nn0 = 0ull, nn1 = 0ull;
#pragma unroll
          for (int c = 0; c < D / 4; ++c) {
            const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(stage + (c >> 3) * 4096 + row * 32 + (((c & 7) ^ (row & 7)) << 2));
            nn0 = f2_fma(v.x, v.x, nn0);
            nn1 = f2_fma(v.y, v.y, nn1);
          }
          float x0, x1, x2, x3;
          f2_unpack(nn0, x0, x1);
          f2_unpack(nn1, x2, x3);
          float sq;
          asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"((x0 + x1) + (x2 + x3)));
          xnorm = sq * (1.002f / 512.f);   // 2^-9 |z| (the approximate root, rounded up)
        }
        // Candidate test without a square root.  With s = e8 + 0.01 (e8 = 2^-9 |screen rows|_F |z|: the TF32 error
        // of the 8 columns), |rows of U_k (x - mu_k)| >= 0.99 sqrt(q8) - s, and cluster k is NOT a candidate when
        // that exceeds sqrt(T), T = 2 (cc_k + 0.01 - thr); (a + b)^2 <= 2 a^2 + 2 b^2 turns it into
        //   q8 > 4.0816 (cc_k + 0.01 - thr) + 2.0408 s^2     (a NaN on either side keeps the candidate).
        float thr = 0.f, A4 = 0.f;
        bool weird = false;
        int cnt = 0;
        // (the columns of two clusters A, B of a slot pair are interleaved: v[2 i] = A_i, v[2 i + 1] = B_i)
        const f32x2_t xn2 = f2_pack(xnorm, xnorm), c01 = f2_pack(0.01f, 0.01f), c204 = f2_pack(2.0408f, 2.0408f);
        f32x2_t A42 = 0ull;
        // hit bits of the 4 clusters of one 32-column batch, branch-free so that the pairs overlap in the pipe
        auto screen4 = [&](const uint32_t* v, int slot0) -> uint32_t {
          uint32_t hits = 0;
#pragma unroll
          for (int pp = 0; pp < 2; ++pp) {
            const uint32_t* w = v + 16 * pp;
            f32x2_t p[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) p[i] = f2_pack(__uint_as_float(w[2 * i]), __uint_as_float(w[2 * i + 1]));
            f32x2_t a0 = f2_fma(p[0], p[0], 0ull), a1 = f2_fma(p[1], p[1], 0ull);
            a0 = f2_fma(p[2], p[2], a0); a1 = f2_fma(p[3], p[3], a1);
            a0 = f2_fma(p[4], p[4], a0); a1 = f2_fma(p[5], p[5], a1);
            a0 = f2_fma(p[6], p[6], a0); a1 = f2_fma(p[7], p[7], a1);
            const float4 sc = scrc[(slot0 >> 1) + pp];
            const f32x2_t sv = f2_fma(xn2, f2_pack(sc.z, sc.w), c01);
            // q8 > bnd  with  bnd = 2.0408 sv^2 + 4.0816 cc + A4
            const f32x2_t t1 = f2_fma(f2_fma(c204, sv, 0ull), sv, f2_fma(f2_pack(sc.x, sc.y), f2_pack(1.f, 1.f), A42));
            float qa, qb, ba, bb, ra, rb;
            f2_unpack(a0, qa, qb);
            f2_unpack(a1, ra, rb);
            f2_unpack(t1, ba, bb);
            hits |= (!((qa + ra) > ba) ? 1u : 0u) << (2 * pp);
            hits |= (!((qb + rb) > bb) ? 1u : 0u) << (2 * pp + 1);
          }
          return hits;
        };
        auto append = [&](uint32_t hits, int k0) {   // rare: the pivot's own bit is masked out by the caller
          for (; hits; hits &= hits - 1) {
            const int k = k0 + __ffs(hits) - 1;
            if (k < K) {
              if (cnt < T2_CMAX) mylist[cnt] = (uint16_t)k;
              ++cnt;
            }
          }
        };
        for (int c = 0; c < nch; ++c, ++cc) {
          const int b = cc & 1;
          tc::mbar_wait(&tfull[g * 2 + b], (cc >> 1) & 1);
          tc::tc_fence_after();
          const uint32_t taddr = tmem_row + b * 128;
          const int ncl = c == 0 ? min(K, n0) : min(16, K - n0 - (c - 1) * 16);
          const int kbase = c == 0 ? 0 : n0 + (c - 1) * 16;
          const int nb = (ncl + 3) >> 2;          // batches of 4 clusters = 32 accumulator columns
          int col = 0, b0 = 0;
          if (c == 0) {
            uint32_t v[32], v1[32];
            float qp = 0.f;
            if constexpr (D == 64) {
              tc::tmem_ld32(taddr, v);
              tc::tmem_ld32(taddr + 32, v1);
              tc::tmem_ld_wait();
              qp = gauss_tc_screen_q(v) + gauss_tc_screen_q(v1);
            } else {
              tc::tmem_ld32(taddr, v);
              tc::tmem_ld32(taddr + 32, v1);          // first screen batch rides along
              tc::tmem_ld_wait();
              qp = gauss_tc_screen_q(v);
            }
            const float2 cf = ccfro[key];
            const float e = xnorm * cf.y;
            float sq;
            asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(sq) : "f"(fmaxf(qp, 0.f)));
            const float dr = fmaf(1.01f * sq, e, fmaf(0.5f * e, e, 0.01f));   // |r~ - r| <= sqrt(q~) e + e^2/2
            const float rt = fmaf(-0.5f, qp, cf.x);
            weird = !(fabsf(rt) < CUDART_INF_F) || !(dr < CUDART_INF_F);
            thr = (rt - dr) - T2_DELTA;
            A4 = 4.0816f * (0.01f - thr);
            A42 = f2_pack(A4, A4);
            col = D;
            if constexpr (D == 32) {
              uint32_t h = screen4(v1, 0);
              if ((unsigned)key < 4u) h &= ~(1u << key);
              if (h) append(h, 0);
              b0 = 1;
            }
          }
          for (; b0 < nb; b0 += 2) {
            uint32_t v[32], v1[32];
            tc::tmem_ld32(taddr + col + b0 * 32, v);
            if (b0 + 1 < nb) tc::tmem_ld32(taddr + col + b0 * 32 + 32, v1);
            tc::tmem_ld_wait();
            uint32_t h = screen4(v, c * 16 + b0 * 4);
            if (b0 + 1 < nb) h |= screen4(v1, c * 16 + b0 * 4 + 4) << 4;
            const int k0 = kbase + b0 * 4;
            if ((unsigned)(key - k0) < 8u) h &= ~(1u << (key - k0));
            if (h) append(h, k0);
          }
          tc::tc_fence_before();
          tc::mbar_arrive(&tempty[g * 2 + b]);
        }
        bool multi = valid && !weird && cnt > 0 && cnt < T2_CMAX;
        bool ovf = valid && (weird || cnt >= T2_CMAX);
        if (multi) {   // insert the pivot at its place (the list is ascending)
          int j = cnt;
          while (j > 0 && mylist[j - 1] > key) {
            mylist[j] = mylist[j - 1];
            --j;
          }
          mylist[j] = (uint16_t)key;
          ++cnt;
        }
        // ---- exact evaluation of the listed (point, cluster) pairs, spread over the 128 threads ----
        // ---- exact evaluation of the listed (point, cluster) pairs, spread over the lanes of the warp ----
        if (__any_sync(0xffffffffu, multi)) {
          const int mine = multi ? cnt : 0;
          int inc = mine;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
          }
          const int total = __shfl_sync(0xffffffffu, inc, 31), off = inc - mine;
          uint16_t* wpairs = pairs + wq * 32 * T2_CMAX;
          for (int j = 0; j < mine; ++j) wpairs[off + j] = (uint16_t)((row << 3) | j);
          __syncwarp();
          // one pair per lane: 32 independent evaluations in flight per warp hide the L2 latency of the factor rows
          // (measured against a warp-cooperative form, lane <-> row of U_k: 3.6x slower, one pair's latency at a time)
          // (measured against a warp-cooperative form, lane <-> row of U_k: 3.6x slower per pair when the lanes are full)
          // ... but with only a few pairs in the warp the cooperative form wins on latency: one pair at a time, all lanes
          if (total <= T2_COOP_MAX) {
            for (int p = 0; p < total; ++p) {
              const int pr = wpairs[p], prow = pr >> 3, slot = pr & 7;
              const int k = lists[prow * T2_CMAX + slot];
              const int32_t pidx = __ldg(a.perm + w.pos + prow);
              const float q = gauss_tc2_exact_q_coop<D>(a.urows + (size_t)k * D * D, a.mu + (size_t)k * D, a.x + (size_t)pidx * D, lane);
              if (lane == 0) {
                const float2 cf = cfin[k];
                rl[prow * T2_CMAX + slot] = gauss_finish(cf.x, q, cf.y);
                ++ncand_total;
              }
            }
          } else {
            for (int p = lane; p < total; p += 32) {
              const int pr = wpairs[p], prow = pr >> 3, slot = pr & 7;
              const int k = lists[prow * T2_CMAX + slot];
              const int32_t pidx = __ldg(a.perm + w.pos + prow);
              const float q = gauss_tc2_exact_q_row<D>(a.urows + (size_t)k * D * D, a.mu + (size_t)k * D, a.x + (size_t)pidx * D);
              const float2 cf = cfin[k];
              rl[prow * T2_CMAX + slot] = gauss_finish(cf.x, q, cf.y);
              ++ncand_total;
            }
          }
          __syncwarp();
        }
        tc::mbar_arrive(&empty[s]);   // the stage can be refilled now
        // ---- draw ----
        if (valid) {
          int lab = key;
          if (multi) {
            bool bad = false;
            for (int j = 0; j < cnt; ++j) bad |= (myrl[j] != myrl[j]);
            if (bad) {
              ovf = true;
            } else if (a.final_iter) {   // first maximum among the candidates (a non-candidate is > 30 below it)
              float bv = -CUDART_INF_F;
              lab = mylist[0];
              for (int j = 0; j < cnt; ++j)
                if (myrl[j] > bv) {
                  bv = myrl[j];
                  lab = mylist[j];
                }
            } else {
              const double u = dpmm_uniform(a.u_inj, idx, a.seed, DPMM_STREAM_LABEL, a.call, (uint64_t)(a.goff + idx));
              lab = gauss_tc2_draw_list(mylist, myrl, cnt, K, u);
            }
          } else if (!ovf) {
            // utils.jl:29 stops at i = 1 for the uniform u == 0; reproduced for injected uniforms only
            // (a Philox uniform is 0 with probability 2^-53 per draw), see kernels_gauss_tc.cuh
            if (a.u_inj != nullptr && lab > 0 && !a.final_iter && a.u_inj[idx] == 0.0) lab = 0;
          }
          if (ovf) {
            a.ovf_list[atomicAdd(a.ovf_count, 1)] = idx;
          } else {
            a.labels[idx] = lab;
            atomicAdd(&hs[lab], 1);
            // (the tile's sort key is the old label of its points; the compiler aggregates this atomic over the warp,
            // and a counter kept across the tile loop would cost the loop spill traffic)
            if (lab != w.key) atomicAdd(a.moved, 1);
          }
          ++npts_total;
        }
      }
      {   // per-call counters (points, exact evaluations): read back asynchronously by the host's path choice
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          npts_total += __shfl_xor_sync(0xffffffffu, npts_total, o);
          ncand_total += __shfl_xor_sync(0xffffffffu, ncand_total, o);
        }
        if (lane == 0 && a.stats != nullptr) {
          atomicAdd(&a.stats[0], npts_total);
          atomicAdd(&a.stats[1], ncand_total);
        }
      }
    } else {
      // =============================== gather warps ===============================
      const int t64 = tid - 320;               // 0 .. T2_PRODUCERS - 1
      constexpr int CPR = D / 4;            // 16-byte chunks per row
      constexpr int RS = T2_PRODUCERS(D) / CPR; // rows covered by the gather threads per pass
      constexpr int NJ = T2_TILE / RS;      // passes per tile
      const int c = t64 % CPR, r0 = t64 / CPR;
      T2Walk wl, wc;
      t2_walk_init(wl, seq);
      wc = wl;
      int ckey = -1;
      float4 cen = make_float4(0.f, 0.f, 0.f, 0.f);
      // the indices of a tile are loaded one tile ahead of the copies that need them: a perm miss is a DRAM
      // round trip, which must not sit between "stage free" and "gather issued"
      int32_t idx[NJ];
      auto load_idx = [&]() {
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const int p = wl.pos + r0 + RS * j;
          idx[j] = p < wl.end ? __ldg(a.perm + p) : -1;
        }
      };
      if constexpr (D == 32) {
        // The rows go straight into registers and are stored once, centred (no landing copy in shared memory):
        // tile li + 2 is loaded into the register set tile li has just been stored from.  Rows past the end of
        // the tile load as exact zeros and are stored uncentred.
        static_assert(PF == 2, "one register set per tile in flight: va, vb");
        auto load_rows = [&](float4 (&v)[NJ]) {
#pragma unroll
          for (int j = 0; j < NJ; ++j) {
            const bool ok = idx[j] >= 0;
            v[j] = ldg_nc16(a.x + (size_t)(ok ? idx[j] : 0) * D + 4 * c, ok);
          }
        };
        float4 va[NJ], vb[NJ];
        load_idx();
        load_rows(va);
        t2_advance(wl, seq);
        if (1 < nt) {
          load_idx();
          load_rows(vb);
          t2_advance(wl, seq);
        }
        if (2 < nt) load_idx();
        auto tile = [&](int li, float4 (&v)[NJ]) {
          const int key = min(wc.key, K - 1);
          if (key != ckey) {
            ckey = key;
            cen = __ldg(reinterpret_cast<const float4*>(a.mu + (size_t)key * D) + c);
          }
          const int nrow = wc.end - wc.pos;
          t2_advance(wc, seq);
#pragma unroll
          for (int j = 0; j < NJ; ++j) {
            if (r0 + RS * j < nrow) {
              v[j].x -= cen.x; v[j].y -= cen.y; v[j].z -= cen.z; v[j].w -= cen.w;
            }
          }
          tc::mbar_wait(&empty[li % NS], ((li / NS) & 1) ^ 1);
          uint8_t* base = stage0 + (size_t)(li % NS) * L.stage_bytes;
#pragma unroll
          for (int j = 0; j < NJ; ++j) {
            const int r = r0 + RS * j;
            *reinterpret_cast<float4*>(base + r * 128 + ((c ^ (r & 7)) << 4)) = v[j];
          }
          tc::fence_proxy_async();
          tc::mbar_arrive(&full[li % NS]);
          const int nx = li + PF;
          if (nx < nt) {
            load_rows(v);
            t2_advance(wl, seq);
            if (nx + 1 < nt) load_idx();
          }
        };
        for (int li = 0; li < nt; li += 2) {
          tile(li, va);
          if (li + 1 < nt) tile(li + 1, vb);
        }
      } else {
        // D = 64: the registers of two tiles in flight do not fit beside the rest of the kernel; cp.async lands
        // the rows in the stage, where they are centred in place
        auto issue = [&](int s) {
          uint8_t* dst0 = stage0 + (size_t)s * L.stage_bytes + (c >> 3) * 16384;
#pragma unroll
          for (int j = 0; j < NJ; ++j) {
            const int r = r0 + RS * j;
            const bool ok = idx[j] >= 0;
            cp_async16(dst0 + r * 128 + (((c & 7) ^ (r & 7)) << 4), a.x + (size_t)(ok ? idx[j] : 0) * D + 4 * c, ok ? 16 : 0);
          }
        };
        load_idx();
#pragma unroll
        for (int q = 0; q < PF; ++q) {
          if (q < nt) {
            issue(q % NS);
            t2_advance(wl, seq);
            if (q + 1 < nt) load_idx();
          }
          cp_async_commit();
        }
        for (int li = 0; li < nt; ++li) {
          cp_async_wait_group<PF - 1>();
          {   // centre this thread's chunks of the landed tile by the pivot's mean (rows beyond the tile stay zero)
            const int key = min(wc.key, K - 1);
            if (key != ckey) {
              ckey = key;
              cen = __ldg(reinterpret_cast<const float4*>(a.mu + (size_t)key * D) + c);
            }
            uint8_t* base = stage0 + (size_t)(li % NS) * L.stage_bytes + (c >> 3) * 16384;
            const int nrow = wc.end - wc.pos;
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
              const int r = r0 + RS * j;
              float4* q = reinterpret_cast<float4*>(base + r * 128 + (((c & 7) ^ (r & 7)) << 4));
              float4 v = *q;
              if (r < nrow) {
                v.x -= cen.x; v.y -= cen.y; v.z -= cen.z; v.w -= cen.w;
                *q = v;
              }
            }
            t2_advance(wc, seq);
          }
          tc::fence_proxy_async();
          tc::mbar_arrive(&full[li % NS]);
          const int nx = li + PF;
          if (nx < nt) {
            tc::mbar_wait(&empty[nx % NS], ((nx / NS) & 1) ^ 1);
            issue(nx % NS);
            t2_advance(wl, seq);
            if (nx + 1 < nt) load_idx();
          }
          cp_async_commit();
        }
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 1) tc::tmem_dealloc(tmem_base, 512);
  for (int k = tid; k < K; k += T2_THREADS(D))
    if (hs[k] != 0) atomicAdd(&a.hist[k], hs[k]);
}

// ------------------------------------------------------------------------------------------------
// Overflow points of the kernel above (and any list of points): the full K-cluster evaluation, one warp
// per point, lanes <-> clusters, then the reference's draw over the whole row (NaN rules included).
// ------------------------------------------------------------------------------------------------
struct GaussListArgs {
  const float* x;
  int K;
  const int32_t* list;
  const int32_t* count;
  const float* urows;
  const float* mu;
  const float* cst;
  const float* logw;
  int32_t* labels;
  int32_t* hist;
  const double* u_inj;
  uint64_t seed;
  uint32_t call;
  int64_t goff;
  int final_iter;
  int32_t* stats;          // optional [2]: [1] += K per listed point
  int32_t* moved;          // [1] += listed points whose label changed
  int32_t* zero_next;      // optional [T2_CTR_SET]: the counter set of the NEXT call, cleared here (no memset launches)
  int32_t* zero_hist;      // optional [zero_hist_n]: the histogram buffer of the NEXT call, cleared here
  int zero_hist_n;
  int32_t* hstat;          // optional [3]: mapped host memory, receives stats[0], stats[1], *count from the last block
  // optional: the last block to finish turns the completed label histogram into the segment offsets and cursors of the
  // sort (what label_scan_kernel does), saving its launch.  ticket: zero on entry, reset on exit.
  int32_t* ticket;
  int scan_k;
  int32_t* seg_off;
  int32_t* scat_cursor;
  int32_t* lr_cursor;
};

template <int D>
__global__ void __launch_bounds__(256) gauss_label_list_kernel(const GaussListArgs a) {
  extern __shared__ float gl_rs[];   // [8][K]
  const int lane = threadIdx.x & 31, wl = threadIdx.x >> 5;
  pdl_wait();
  pdl_launch_dependents();
  const int nlist = *a.count;
  if (a.zero_next != nullptr && blockIdx.x == 0 && threadIdx.x < T2_CTR_SET) a.zero_next[threadIdx.x] = 0;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < a.zero_hist_n; k += gridDim.x * blockDim.x) a.zero_hist[k] = 0;
  float* rs = gl_rs + (size_t)wl * a.K;
  for (int e = blockIdx.x * 8 + wl; e < nlist; e += gridDim.x * 8) {
    const int32_t idx = a.list[e];
    const float* xr = a.x + (size_t)idx * D;
    for (int k = lane; k < a.K; k += 32) {
      const float q = gauss_tc2_exact_q_impl<D>(a.urows + (size_t)k * D * D, a.mu + (size_t)k * D,
                                                [&](int c) { return __ldg(reinterpret_cast<const float4*>(xr) + c); });
      rs[k] = gauss_finish(__ldg(a.cst + 3 * k), q, __ldg(a.logw + k));
    }
    __syncwarp();
    if (lane == 0) {
      int lab;
      if (a.final_iter) {
        lab = dpmm_draw_argmax(rs, 1, a.K);
      } else {
        const double u = dpmm_uniform(a.u_inj, idx, a.seed, DPMM_STREAM_LABEL, a.call, (uint64_t)(a.goff + idx));
        lab = dpmm_draw_inverse_cdf(rs, 1, a.K, u);
      }
      if (a.moved != nullptr && a.labels[idx] != lab) atomicAdd(a.moved, 1);
      a.labels[idx] = lab;
      atomicAdd(a.hist + lab, 1);
      if (a.stats != nullptr) atomicAdd(&a.stats[1], a.K);
    }
    __syncwarp();
  }
  if (a.ticket != nullptr) {
    __shared__ int last_block;
    __shared__ int wtot[8];
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last_block = atomicAdd(a.ticket, 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (last_block) {   // exclusive scan of hist[0 .. scan_k): 256 threads, chunks of 256
      __threadfence();
      int carry = 0;
      for (int k0 = 0; k0 < a.scan_k; k0 += 256) {
        const int k = k0 + (int)threadIdx.x;
        const int v = k < a.scan_k ? __ldcg(a.hist + k) : 0;
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= o) inc += t;
        }
        if (lane == 31) wtot[wl] = inc;
        __syncthreads();
        int before = 0, total = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
          before += w < wl ? wtot[w] : 0;
          total += wtot[w];
        }
        const int excl = carry + before + inc - v;
        if (k < a.scan_k) {
          a.seg_off[k] = excl;
          a.scat_cursor[k] = excl;
          a.lr_cursor[2 * k] = excl;
          a.lr_cursor[2 * k + 1] = excl + v;
        }
        carry += total;
        __syncthreads();
      }
      if (threadIdx.x == 0) {
        a.seg_off[a.scan_k] = carry;
        *a.ticket = 0;
        if (a.hstat != nullptr) {   // the host's path choice reads these once the event behind this kernel has fired
          a.hstat[0] = __ldcg(a.stats + 0);
          a.hstat[1] = __ldcg(a.stats + 1);
          a.hstat[2] = __ldcg(a.count);
          __threadfence_system();
        }
      }
    }
  }
}
