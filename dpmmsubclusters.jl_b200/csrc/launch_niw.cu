// NIW kernels for one group of feature dimensions (compiled once per DPMM_DIMSET so that the
// groups build in parallel): template instantiation + launch configuration.
#define DPMM_TEMPLATES_ONLY
#include "ctx.cuh"
#include "kernels_gauss.cuh"
#include "kernels_stats.cuh"

#ifndef DPMM_DIMSET
#error "compile with -DDPMM_DIMSET=<0..5>"
#endif
#if DPMM_DIMSET == 0
#define SET_DIMS(X) X(1) X(2) X(3) X(4)
#elif DPMM_DIMSET == 1
#define SET_DIMS(X) X(5) X(6) X(7) X(8)
#elif DPMM_DIMSET == 2
#define SET_DIMS(X) X(12) X(16) X(24)
#elif DPMM_DIMSET == 3
#define SET_DIMS(X) X(32)
#elif DPMM_DIMSET == 4
#define SET_DIMS(X) X(48)
#else
#define SET_DIMS(X) X(64)
#endif
#define CAT2(a, b) a##b
#define CAT(a, b) CAT2(a, b)
#define SETFN(name) CAT(name, DPMM_DIMSET)

template <int D>
struct LabelP {  // points per thread of the label kernel
  static constexpr int P = (D <= 16) ? 4 : (D <= 32 ? 2 : 1);
};

template <int D, int P, bool TILE_ONLY = false>
static int launch_gauss_label_p(dpmm_ctx* ctx, GaussLabelArgs a) {
  using C = GaussCfg<D>;
  if constexpr (!TILE_ONLY) {
    // warp-autonomous form: all K records resident + W private warp buffers
    const size_t fixed = ((size_t)a.K * C::REC + 3 * (size_t)((a.K + 3) & ~3)) * 4;
    const size_t perwarp = ((size_t)32 * P * C::DS + (size_t)a.K * 32 * P) * 4;
    int W = fixed < (size_t)ctx->smem_optin ? (int)(((size_t)ctx->smem_optin - fixed) / perwarp) : 0;
    W = std::min(W, 12);
    if (W >= 6) {
      const size_t sm = fixed + (size_t)W * perwarp;
      auto kern = gauss_label_warp_kernel<D, P>;
      CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
      a.KC = a.K;
      a.ntiles = (a.n + 32 * P - 1) / (32 * P);
      const int64_t grid = std::min<int64_t>((a.ntiles + W - 1) / W, (int64_t)ctx->sm_count);
      KernelTimer kt(ctx, TK_LABEL);
      kern<<<(unsigned)grid, W * 32, sm, ctx->stream>>>(a);
      CK(cudaGetLastError());
      return 0;
    }
  }
  const size_t budget2 = 110 * 1024, budget1 = (size_t)ctx->smem_optin;
  int T = 128, KC = a.K;
  auto bytes = [&](int T_, int KC_) {
    return ((size_t)T_ * P * C::DS + (size_t)a.K * T_ * P + (size_t)KC_ * C::REC) * 4 + (size_t)a.K * 4;
  };
  // prefer two CTAs per SM; shrink the staged-cluster chunk first, then the tile
  bool ok = false;
  for (size_t budget : {budget2, budget1}) {
    for (int T_ : {128, 64, 32}) {
      if (bytes(T_, 1) > budget) continue;
      T = T_;
      KC = a.K;
      while (bytes(T, KC) > budget) KC = (KC + 1) / 2;
      ok = true;
      break;
    }
    if (ok) break;
  }
  if (!ok) return fail(ctx, DPMM_ELIMIT, "K too large for the label kernel's shared-memory slice");
  a.KC = KC;
  const int TP = T * P;
  a.ntiles = (a.n + TP - 1) / TP;
  const size_t sm = bytes(T, KC);
  auto kern = gauss_label_kernel<D, P>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
  int occ = 1;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, T, sm));
  occ = std::max(occ, 1);
  const int64_t grid = std::min<int64_t>(a.ntiles, (int64_t)ctx->sm_count * occ);
  KernelTimer kt(ctx, TK_LABEL);
  kern<<<(unsigned)grid, T, sm, ctx->stream>>>(a);
  CK(cudaGetLastError());
  return 0;
}

template <int D>
static int launch_gauss_label(dpmm_ctx* ctx, GaussLabelArgs a) {
  int rc = launch_gauss_label_p<D, LabelP<D>::P>(ctx, a);
  if constexpr (LabelP<D>::P > 1) {
    // the tile's slice of parr ([K][points]) is what limits K: one point per thread carries K up to DPMM_MAX_K
    if (rc == DPMM_ELIMIT) rc = launch_gauss_label_p<D, 1, true>(ctx, a);
  }
  return rc;
}

template <int D>
static int launch_gauss_sublabel(dpmm_ctx* ctx, const SubLabelArgs& a, bool sample) {
  if constexpr (D % 4 == 0 && D >= 16 && D <= 48) {
    if (sample) {
      using C = GaussCfg<D>;
      const size_t sm = ((size_t)2 * 256 * C::DS + (size_t)SUBLABEL_SPAN * 2 * C::REC + a.K + 4) * 4;
      auto kern = gauss_sublabel2_kernel<D>;
      CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
      int occ = 1;
      CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, 128, sm));
      const int64_t ntiles = (a.n + 255) / 256;
      const unsigned grid = (unsigned)std::min<int64_t>(ntiles, (int64_t)ctx->sm_count * std::max(occ, 1));
      KernelTimer kt(ctx, TK_SUBLABEL);
      kern<<<grid, 128, sm, ctx->stream>>>(a);
      CK(cudaGetLastError());
      return 0;
    }
  }
  const int T = 128;
  const unsigned grid = (unsigned)((a.n + T - 1) / T);
  KernelTimer kt(ctx, TK_SUBLABEL);
  if (sample)
    gauss_sublabel_kernel<D, true><<<grid, T, 0, ctx->stream>>>(a);
  else
    gauss_sublabel_kernel<D, false><<<grid, T, 0, ctx->stream>>>(a);
  CK(cudaGetLastError());
  return 0;
}

template <int D>
static int launch_niw_stats(dpmm_ctx* ctx, const StatsArgs& a) {
  using C = StatsCfg<D>;
  if constexpr (D <= 8) {
    // one warp per run chunk pays off once there are enough chunks to fill the machine (C4: 313 -> 82 us);
    // on small inputs the CTA-cooperative kernel below has the shorter critical path (C1: 10 vs 19 us)
    if (ctx->n >= ((int64_t)1 << 18) && env_int("DPMM_STATS_SMALL", 1) != 0) {
      KernelTimer kt(ctx, TK_STATS);
      niw_stats_small_kernel<D><<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(a);
      CK(cudaGetLastError());
      return 0;
    }
  }
  auto kern = niw_stats_kernel<D>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM_BYTES));
  int occ = 1;
  CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, C::WARPS * 32, C::SMEM_BYTES));
  occ = std::max(occ, 1);
  KernelTimer kt(ctx, TK_STATS);
  kern<<<ctx->sm_count * occ, C::WARPS * 32, C::SMEM_BYTES, ctx->stream>>>(a);
  CK(cudaGetLastError());
  return 0;
}

// returns 1 when D is not in this set
int SETFN(niw_set_label_)(dpmm_ctx* ctx, const GaussLabelArgs& a, int D, int* rc) {
  switch (D) {
#define X(d) case d: *rc = launch_gauss_label<d>(ctx, a); return 0;
    SET_DIMS(X)
#undef X
  }
  return 1;
}
int SETFN(niw_set_sublabel_)(dpmm_ctx* ctx, const SubLabelArgs& a, bool sample, int D, int* rc) {
  switch (D) {
#define X(d) case d: *rc = launch_gauss_sublabel<d>(ctx, a, sample); return 0;
    SET_DIMS(X)
#undef X
  }
  return 1;
}
int SETFN(niw_set_stats_)(dpmm_ctx* ctx, const StatsArgs& a, int D, int* rc) {
  switch (D) {
#define X(d) case d: *rc = launch_niw_stats<d>(ctx, a); return 0;
    SET_DIMS(X)
#undef X
  }
  return 1;
}
